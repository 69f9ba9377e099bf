// indelope_b200/csrc/bamdev.h -- inside libindelope_cuda.so: building a batch of regions on the device from a resident BAM (bamdev.cu),
// entered by idl_bam_submit / idl_bam_pack (pipeline.cu), which own the lanes' device buffers the batch is written into.
#pragma once
#include <cstddef>
#include <cstdint>
#include <string>
#include <vector>
#include <cuda_runtime.h>
#include "indelope_cuda.h"

// ---- the BGZF inflate stage (bamdev.cu), shared by idl_bam_open and idl_fasta_open (fastadev.cu) ----
struct BgzfMember { unsigned long long in_off; unsigned long long out_off; uint32_t in_len, out_len, crc, pad; };
// the member walk: header checks (gzip magic, BC subfield, sizes, ISIZE <= 64 KiB) and where each member's deflate data lies and its output goes;
// false with the reason in why
bool bgzf_walk(const uint8_t *file, size_t file_len, std::vector<BgzfMember> &members, std::vector<size_t> &member_at, size_t &total, std::string &why);
// the file goes up to d_comp in chunks of whole members and each chunk's members are inflated and CRC-checked into d_out (bgzf_inflate_kernel, one
// warp per member) as soon as they have arrived, on four streams; returns when every kernel is done.  Expects the member table in d_members, *d_err
// = ~0, d_next[0..64) = 0 and the padding behind the file cleared, all ordered on st.  *d_err: the first bad member << 8 | its decoder error.
cudaError_t bgzf_inflate_chunks(cudaStream_t st, int n_sm, const uint8_t *file, size_t file_len, const std::vector<BgzfMember> &members, uint8_t *d_comp,
                                const BgzfMember *d_members, uint8_t *d_out, unsigned long long *d_err, unsigned *d_next, uint32_t *n_chunks);
// the message for a bad member of *d_err
std::string bgzf_error_text(unsigned long long first_error);
// exclusive 64-bit scan of n uint32 values into out[0..n] (out[n] = total); tot = scratch for (n + 1 + 2047) / 2048 tile totals
cudaError_t scan_u32(const uint32_t *in, size_t n, unsigned long long *out, unsigned long long *tot, cudaStream_t st);
// idl_bam_set_reference_fasta: where a record of a parsed FASTA lies on its device (fastadev.cu)
int fasta_record_on_device(const idl_fasta *fa, int64_t record, const uint8_t **seq, int64_t *len, int *device);

struct BamBatchTotals {            // what the device reports after the records are laid out
	unsigned long long n_seq_bases, n_ref_bases;   // multiples of 64
	unsigned max_trim_len, max_ref_len, max_region_reads, n_small_regions;
	unsigned bad_index;                            // a read index outside the BAM's records, or a region on a target without a reference
	unsigned scratch_set;                          // which of the BAM's scratch sets phase 1 used (phase 2 reads the indices from it)
};

// phase 1: region and read records (quality trim, windows, pool offsets) for the regions given as host arrays; d_region / d_read must
// hold n_regions / n_reads records.  Synchronises the stream once to return the totals.
int bam_batch_records(idl_bam *bam, cudaStream_t st, const idl_params *P, size_t n_regions, const int32_t *roi_chrom, const int32_t *roi_start, const int32_t *roi_end,
                      const int32_t *roi_n_reads, const int64_t *read_idx, size_t n_reads, uint32_t ordinal_base, idl_region *d_region, idl_read *d_read,
                      BamBatchTotals *totals);
// phase 2: the bases of the reads (BAM nibbles -> 2 bits + N plane) and of the reference windows (ASCII -> the same) into the pools
int bam_batch_bases(idl_bam *bam, cudaStream_t st, size_t n_regions, size_t n_reads, idl_region *d_region, const idl_read *d_read, const BamBatchTotals *totals,
                    uint32_t *seq2, uint32_t *seqn, uint32_t *ref2, uint32_t *refn);
int bam_device_of(const idl_bam *bam);
