/* include/indelope_host.h -- C ABI of libindelope_host.so
 *
 * C++ stand-in for the parts of indelope that stay on the host (the reference keeps them in Nim; no Nim
 * toolchain exists in this image, see DESIGN.md / INTEGRATION.md):
 *   - the BAM sweep -> evidence counters -> coverage-gap chunking -> regions of interest
 *     (src/indelope.nim:430-545: event_locations, overlaps, gen_roi_internal, cache_t, gen_roi)
 *   - read quality trim and batch packing for libindelope_cuda.so (src/indelope.nim:23-38,169)
 *   - the filter cascade, genotype likelihoods and VCF text over the device results
 *     (src/indelope.nim:49-116,375-428,598-608; src/genotyper.nim:16-47)
 *   - a seeded synthetic data generator with an aligner model (no aligner / BAM library is installed)
 * This library contains no CUDA and does not link the oracle.
 */
#ifndef INDELOPE_HOST_H
#define INDELOPE_HOST_H
#include <stdint.h>
#include "indelope_cuda.h"

#ifdef __cplusplus
extern "C" {
#endif

/* regions of interest in the shape gen_roi yields them, flattened (`roi = tuple[start, stop, reads]`,
 * src/indelope.nim:21).  Reads are referenced by index so a read shared by two regions is stored once. */
typedef struct idlh_roiset {
	int64_t n_reads;
	const int32_t *start;
	const int32_t *stop;
	const uint8_t *mapq;
	const uint16_t *flag;
	const int32_t *len;
	const int64_t *seq_off;
	const uint8_t *bases;     /* ASCII */
	const uint8_t *quals;
	int64_t n_rois;
	const int32_t *roi_chrom;
	const int32_t *roi_start, *roi_stop;
	const int64_t *roi_read_begin;
	const int32_t *roi_n_reads;
	const int64_t *read_idx;
	int32_t n_chroms;
	const char *const *chrom_name;
	const uint8_t *const *chrom_seq;
	const int64_t *chrom_len;
} idlh_roiset;

typedef struct idlh_synth_params {
	uint64_t seed;
	int32_t n_chroms;
	int64_t chrom_len;
	int32_t n_events;           /* planted events per chromosome */
	int32_t min_indel, max_indel;
	double coverage;
	int32_t read_len;
	double sub_rate;            /* substitution errors per base */
	double tr_fraction;         /* share of events that are tandem-repeat expansions/contractions */
	int32_t tr_max_unit;        /* repeat unit 1..tr_max_unit bp */
	double het_fraction;
	double lowq_tail_fraction;  /* reads with a Q2 tail of 1-15 bases */
	double low_mapq_fraction;   /* reads with MAPQ in {0,5,10,19} */
	double dup_fraction;        /* reads flagged duplicate (skippable) */
	double n_base_rate;         /* read bases replaced by N */
	int32_t locus_only;         /* 1: simulate reads only within locus_flank of planted events */
	int32_t locus_flank;
	int32_t max_cigar_indel;    /* aligner model: longer indels are soft-clipped [30] */
	int32_t min_cigar_flank;    /* aligner model: shorter flanks are soft-clipped [20] */
	int32_t chrom_first;        /* generate chromosomes chrom_first .. chrom_first + n_chroms - 1 of the genome this seed defines (every
	                               chromosome has its own random stream, so a rank can build just its interval shard) [0] */
	int32_t qual_levels;        /* 0/1: every untrimmed base has quality 30; k > 1: k distinct qualities in 15 .. 41 drawn per base from a hash of
	                               (read, position) -- all at or above the trim threshold, so reads, regions and calls stay the same while the BAM
	                               compresses like sequencer output instead of 12:1 [0] */
} idlh_synth_params;

void idlh_default_synth(idlh_synth_params *p);

typedef struct idlh_dataset idlh_dataset;   /* reference + coordinate-sorted reads with CIGARs */
typedef struct idlh_rois idlh_rois;         /* owns the arrays behind an idlh_roiset */

idlh_dataset *idlh_synth(const idlh_synth_params *p);
void idlh_dataset_free(idlh_dataset *d);
/* counts[0]=reads, [1]=bases, [2]=events planted, [3]=chroms */
void idlh_dataset_counts(const idlh_dataset *d, int64_t counts[4]);
/* truth table: chrom, pos, ins_len, del_len, hom, is_tr (6 int64 per event) */
int64_t idlh_dataset_truth(const idlh_dataset *d, int64_t *out, int64_t cap);

/* ---- files (indelope_b200/csrc/host/bamio.cpp, written from the SAM/BAM specification on zlib) ----
 * idlh_load: reference FASTA (hts-nim open_fai / fai.get, src/indelope.nim:583) + coordinate-sorted BAM read front to back,
 * the order `for target in targets: b.querys(target.name)` visits (:527,599-602); `threads` inflate BGZF blocks in
 * parallel (the -t option, :566).  Returns NULL and a message in err on failure.  CRAM is not supported.
 * idlh_write_fasta writes path and path.fai; idlh_write_bam writes a BGZF-compressed BAM (deflate level 0-9) of the reads and its
 * BAI index path.bai (SAM spec 5.2: binning index + 16 kb linear index). */
idlh_dataset *idlh_load(const char *fasta_path, const char *bam_path, int threads, char *err, size_t errlen);
/* idlh_load_region: `b.querys(region)` through the BAI index <bam>.bai (idlh_write_bam writes it next to the BAM; the reference opens its
 * BAM with index=true, src/indelope.nim:595): only the records of `target` that overlap [beg, end) (0-based, half open; end <= 0 = to
 * the end of the target), only their BGZF blocks inflated. */
idlh_dataset *idlh_load_region(const char *fasta_path, const char *bam_path, const char *target, int64_t beg, int64_t end, char *err, size_t errlen);
int idlh_write_fasta(const idlh_dataset *d, const char *path);
int idlh_write_bam(const idlh_dataset *d, const char *path, int level);

/* Streaming twin of idlh_load + idlh_sweep for files that do not fit in memory: the BAM is read front to back, BGZF blocks
 * are inflated by `threads` workers, and gen_roi (src/indelope.nim:515-545) runs incrementally over the records; the
 * regions and their read lists are the same as the whole-file sweep's (bamio.cpp explains why).  idlh_stream_next sweeps
 * on until the regions collected hold at least target_reads reads (or the file ends) and returns them as a self-contained
 * group (regions in emission order; free with idlh_rois_free); NULL after the last group, or on error with a message in
 * err.  idlh_stream_targets gives a view without regions (contig names and lengths, for the VCF header). */
typedef struct idlh_stream idlh_stream;
idlh_stream *idlh_stream_open(const char *fasta_path, const char *bam_path, int threads, int32_t min_event_support, int32_t min_read_coverage,
                              int32_t max_read_coverage, char *err, size_t errlen);
idlh_rois *idlh_stream_next(idlh_stream *s, int64_t target_reads, char *err, size_t errlen);
idlh_rois *idlh_stream_targets(const idlh_stream *s);
void idlh_stream_counts(const idlh_stream *s, int64_t counts[2]);   /* BAM records read, regions emitted so far */
void idlh_stream_close(idlh_stream *s);

/* the records of one chromosome of a dataset as the plain arrays idl_sweep (libindelope_cuda: gen_roi on the GPU) takes: BAM order, CIGARs
 * concatenated.  first_read = index of the chromosome's first record in the dataset (read_idx of idlh_sweep counts from the dataset's
 * first record).  Free with idlh_chrom_free. */
typedef struct idlh_chrom_reads {
	int64_t first_read, n_reads;
	int32_t chrom_len;
	int32_t *start, *stop;
	uint16_t *flag;
	uint32_t *cigar;
	uint64_t *cig_off;   /* n_reads + 1 */
} idlh_chrom_reads;
idlh_chrom_reads *idlh_dataset_chrom(const idlh_dataset *d, int32_t chrom);
void idlh_chrom_free(idlh_chrom_reads *c);
int32_t idlh_dataset_n_chroms(const idlh_dataset *d);
const char *idlh_dataset_chrom_name(const idlh_dataset *d, int32_t chrom);
/* the device reads the BAM (idl_bam_open of indelope_cuda.h); the host keeps the reference sequences and turns what idl_bam_sweep / idl_bam_fetch
 * return into the idlh_rois that idlh_pack and idlh_vcf_records take */
idlh_dataset *idlh_load_fasta(const char *fasta_path, char *err, size_t errlen);
/* a reference (no reads) from n names and sequences found elsewhere -- idl_fasta_open of a bgzipped FASTA on the device; everything is copied.  Every
 * loader here takes <fasta_path> plain or compressed with bgzip (BGZF members inflated on idlh_set_threads' host threads); plain gzip is refused. */
idlh_dataset *idlh_dataset_from_sequences(int32_t n, const char *const *names, const uint8_t *const *seqs, const int64_t *lens);
/* the FASTA's sequences in the order of the BAM header's targets; of the BAM only the header is read */
idlh_dataset *idlh_load_targets(const char *fasta_path, const char *bam_path, char *err, size_t errlen);
/* where one target's records lie in the file, from <bam>.bai: the run of whole BGZF members [*file_begin, *file_end) and the start / end of the record
 * chain inside it as idl_bam_open_slice takes them; 0 ok, 1 the index lists no record for the target, -1 error */
int idlh_bai_target_span(const char *bam_path, int32_t target, uint64_t *file_begin, uint64_t *file_end, uint64_t *first_record, uint64_t *end_member,
                         uint64_t *end_offset, char *err, size_t errlen);
/* the records of one target from the first record of 16 kb window w0 (linear index) to the first record of window w1 + 1, or to the target's end
 * (*to_end = 1): the run of members as idl_bam_open_slice takes it, and *zone_lo, the first position whose evidence, cuts and records are those of the
 * whole file (0 at window 0 or at the target's first record, else (w0 << 14) + 1; DESIGN.md 4a).  0 ok, 1 the run holds no record, -1 error */
int idlh_bai_region_run(const char *bam_path, int32_t target, int64_t w0, int64_t w1, uint64_t *file_begin, uint64_t *file_end, uint64_t *first_record,
                        uint64_t *end_member, uint64_t *end_offset, int64_t *zone_lo, int32_t *to_end, char *err, size_t errlen);
/* -r / -R of the command line: region strings chr[:beg[-end]] (1-based, inclusive, commas allowed in numbers) and a BED file (0-based, half open; '#',
 * 'track', 'browser' and blank lines skipped, CRLF accepted, columns after the third ignored), validated against the targets of the BAM header, as
 * sorted, merged half-open intervals per target.  Intervals are clipped to the target; intervals on a decoy target (hs37d5, GL*, which are never
 * called, src/indelope.nim:41-42) are dropped with a note on stderr.  NULL with the reason in err (the BED line number included). */
typedef struct idlh_regions idlh_regions;
idlh_regions *idlh_regions_parse(int32_t n_ref, const char *const *ref_name, const int64_t *ref_len, int32_t n_region, const char *const *region, const char *bed_path,
                                 char *err, size_t errlen);
int64_t idlh_regions_get(const idlh_regions *r, int32_t target, int64_t *beg, int64_t *end, int64_t cap);   /* intervals of a target (up to cap copied); returns their number */
void idlh_regions_free(idlh_regions *r);
int idlh_dataset_set_targets(idlh_dataset *d, int32_t n_ref, const char *const *ref_name, const int64_t *ref_len, char *err, size_t errlen);
/* the same with the targets of a BAM file's header (only the members that hold the header are read): what idlh_load_targets does after loading the FASTA */
int idlh_dataset_set_bam_targets(idlh_dataset *d, const char *bam_path, char *err, size_t errlen);
idlh_rois *idlh_rois_from_arrays(const idlh_dataset *d, int64_t n_reads, const int32_t *start, const int32_t *stop, const int32_t *len, const uint8_t *mapq, const uint16_t *flag,
                                 const int64_t *seq_off, const uint8_t *bases, const uint8_t *quals, int64_t n_rois, const int32_t *roi_chrom, const int32_t *roi_start,
                                 const int32_t *roi_stop, const int32_t *roi_n_reads, const int64_t *read_idx);

/* gen_roi over every target (src/indelope.nim:515-545,601-602), regions in emission order */
idlh_rois *idlh_sweep(const idlh_dataset *d, int32_t min_event_support, int32_t min_read_coverage, int32_t max_read_coverage);
void idlh_rois_free(idlh_rois *r);
const idlh_roiset *idlh_rois_view(const idlh_rois *r);

/* quality trim of src/indelope.nim:23-38: returns a, *trim_len = kept bases */
int32_t idlh_trim(const uint8_t *quals, int32_t n, int32_t *trim_len);

/* batch sizing / packing of regions [lo, hi).  Packing runs on idlh_set_threads(n) host threads (0 = $IDLH_THREADS, else every core
 * up to 32): 16 bases per SSE2 step into the 2-bit pool + the non-ACGT plane.  Bytes outside {A,C,G,T,N} are folded (acgt -> ACGT,
 * anything else -> N) and the region is flagged IDL_RF_ALPHABET; a read longer than max_read_len is packed empty and the region
 * flagged IDL_RF_READ_TOO_LONG (the device drops that region and reports it) instead of failing the batch.  idlh_pack also fills
 * the batch summary (idl_batch.summary_valid) so that idl_submit does no per-read host work. */
void idlh_set_threads(int n);
void idlh_pack_size(const idlh_roiset *rs, int64_t lo, int64_t hi, const idl_params *p, size_t *n_reads, size_t *n_seq_bases, size_t *n_ref_bases);
int idlh_pack(const idlh_roiset *rs, int64_t lo, int64_t hi, const idl_params *p, idl_batch *out);
/* plain-malloc batch for CPU-only inspection/tests (idl_batch_alloc gives pinned memory) */
idl_batch *idlh_batch_alloc_host(size_t max_regions, size_t max_reads, size_t max_seq_bases, size_t max_ref_bases);
void idlh_batch_free_host(idl_batch *b);
/* unpack one packed record back to ASCII (round-trip tests) */
void idlh_unpack(const uint32_t *pool2, const uint32_t *pooln, uint64_t base_off, int32_t n, char *out);

/* VCF writer: header, then records through the filter cascade with the order-dependent dedup state of
 * src/indelope.nim:598-608 carried across batches */
typedef struct idlh_vcf idlh_vcf;
idlh_vcf *idlh_vcf_new(void);
void idlh_vcf_free(idlh_vcf *w);
char *idlh_vcf_header(const idlh_roiset *rs);   /* malloc'ed; free with idlh_free */
/* records for regions [lo, lo + res->n_regions) of rs; malloc'ed text; dump_level as the oracle's (0 = VCF only) */
char *idlh_vcf_records(idlh_vcf *w, const idlh_roiset *rs, int64_t lo, const idl_params *p, const idl_results *res, int32_t dump_level, char **dump);
/* multi-GPU: shards emit records WITHOUT the dedup (idlh_vcf_set_dedup(w, 0)); after concatenating the shards in region
 * order, idlh_vcf_dedup applies the reference's order-dependent filter (drop a record equal in CHROM, POS, REF, ALT to
 * one of the last two emitted, src/indelope.nim:114-116,604-608) to the merged text.  Returns malloc'ed text. */
void idlh_vcf_set_dedup(idlh_vcf *w, int on);
/* regions seen so far with each idl_region_result.status bit set (index = bit number of IDL_RS_*); every such region also gets a
 * warning on stderr (the first 20): capacity limits and the alphabet fold never change the output silently */
void idlh_vcf_status_counts(const idlh_vcf *w, uint64_t out[8]);
char *idlh_vcf_dedup(const char *records);
char *idlh_vcf_dedup_n(const char *records, size_t n, size_t *out_len);   /* the same over n bytes, not necessarily terminated */
size_t idlh_vcf_dedup_inplace(char *records, size_t n);                   /* the same in place (n + 1 bytes writable); returns the new length */
void idlh_free(void *p);

#ifdef __cplusplus
}
#endif
#endif
