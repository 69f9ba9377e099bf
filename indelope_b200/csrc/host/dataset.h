// indelope_b200/csrc/host/dataset.h -- the in-memory dataset the host stand-in sweeps: a reference and coordinate-sorted
// reads with CIGARs, filled either by the synthetic generator (synth_sweep.cpp) or from FASTA + BAM files (bamio.cpp).
#pragma once
#include <cstdint>
#include <string>
#include <vector>
#include "indelope_host.h"

struct IdlhEvent { int chrom; int64_t pos; std::string ins; int dlen; bool hom; bool tr; };

struct IdlhReadRec {
	int32_t chrom, start, stop; uint8_t mapq; uint16_t flag; int32_t len; int64_t seq_off; int64_t cig_off; int32_t n_cig; uint64_t order;
};

struct idlh_dataset {
	idlh_synth_params P;
	std::vector<std::string> names;
	std::vector<std::vector<uint8_t>> chroms;   // ASCII, as in the FASTA (case preserved)
	std::vector<IdlhEvent> events;              // planted truth (synthetic data only)
	std::vector<IdlhReadRec> reads;             // coordinate sorted per chromosome, chromosomes in header order
	std::vector<uint8_t> bases, quals;          // ASCII bases (soft clips included), raw phred
	std::vector<uint32_t> cigars;               // BAM encoding len<<4|op (M0 I1 D2 N3 S4 H5 P6 =7 X8)
};

// regions of interest with the reads they reference; `view` is what the C ABI hands out.  The whole-file sweep borrows
// bases/quals from the dataset it swept; the streaming sweep (bamio.cpp) owns them per group of regions.
struct idlh_rois {
	std::vector<int32_t> start, stop, len; std::vector<uint8_t> mapq; std::vector<uint16_t> flag; std::vector<int64_t> seq_off;
	const uint8_t *bases = nullptr, *quals = nullptr;
	std::vector<uint8_t> own_bases, own_quals;
	std::vector<int32_t> roi_chrom, roi_start, roi_stop, roi_n_reads; std::vector<int64_t> roi_read_begin, read_idx;
	std::vector<const char*> name_ptrs; std::vector<const uint8_t*> seq_ptrs; std::vector<int64_t> chrom_len;
	idlh_roiset view;
};

// host threads of idlh_pack and of the bgzipped FASTA's inflate (idlh_set_threads; 0 = $IDLH_THREADS, else every core up to 32) (pack_vcf.cpp)
int pack_threads();

// skippable (src/indelope.nim:40-47): the two decoy-contig name tests and the flag tests
inline bool idlh_skippable_chrom(const std::string &name) { return name == "hs37d5" || name.compare(0, 2, "GL") == 0; }
inline bool idlh_skippable_flag(uint16_t f) { return (f & 0x400) || (f & 0x200) || (f & 0x4) || (f & 0x800) || (f & 0x100); }
