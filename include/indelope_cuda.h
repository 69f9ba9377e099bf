/* include/indelope_cuda.h -- C ABI of libindelope_cuda.so
 *
 * B200 (sm_100a) implementation of indelope's per-region calling path.  The library replaces the
 * body of the reference's `callsemble` iterator (src/indelope.nim:201-428) between "region + reads +
 * reference window in" and "per-event integer records out":
 *
 *   kernel 1  slide-and-vote assembler      <- src/contig.nim:70-281, src/indelope.nim:157-183
 *   kernel 2  ksw2 extension DP + traceback <- src/ksw2/csrc/ksw2_extz2_sse.c:113-388 (the only C ABI the
 *                                              reference itself has: src/ksw2/ksw2_c.nim:53-55)
 *   glue      CIGAR -> events -> k-mers     <- src/ksw2/ksw2.nim:22-33,71-91, src/indelope.nim:229-281
 *   kernel 3  ref/alt 27-mer counting       <- src/indelope.nim:283-311 (+ AL fallback :312-372 via kernel 2)
 *
 * Floating point (genotype likelihoods, src/genotyper.nim) and all text stay on the host.
 * Plain C: pointers and sizes only, no C++/torch types.  Every function returns IDL_OK (0) or a
 * negative idl_status; nothing aborts or throws across the boundary.  A context is not thread-safe;
 * distinct contexts (one per GPU / host thread) are independent.  There is no CPU fallback: without
 * a CUDA device idl_create fails with IDL_E_NO_DEVICE.
 */
#ifndef INDELOPE_CUDA_H
#define INDELOPE_CUDA_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IDL_ABI_VERSION 2

typedef enum {
	IDL_OK = 0,
	IDL_E_NO_DEVICE = -1,   /* no CUDA device / driver: there is no CPU path */
	IDL_E_CUDA = -2,        /* a CUDA call failed; idl_last_cuda_error() has the text */
	IDL_E_ARG = -3,
	IDL_E_NOMEM = -4,
	IDL_E_CAPACITY = -5,    /* batch exceeds what idl_batch_alloc / idl_create sized, or its longest read / window needs more kernel-2
	                           workspace or shared memory than one CTA may have (DESIGN.md 7) */
	IDL_E_TICKET = -6,
	IDL_E_BUSY = -7,
	IDL_E_FORMAT = -8       /* idl_bam_open: not a BGZF / BAM file, corrupt member, unsorted records; the call's message has the detail */
} idl_status;

/* per-region status bits (idl_region_result.status) */
#define IDL_RS_OK              0u
#define IDL_RS_CONTIG_OVERFLOW 1u   /* a contig outgrew idl_params.max_contig_len: region dropped */
#define IDL_RS_CORR_OVERFLOW   2u   /* more than IDL_MAX_CORRECTIONS voting sites in one merge */
#define IDL_RS_DP_OVERFLOW     4u   /* an alignment exceeded the DP workspace (tlen/qlen caps) */
#define IDL_RS_CIGAR_OVERFLOW  8u
#define IDL_RS_READ_TOO_LONG  16u   /* a read longer than idl_params.max_read_len (idl_region.flags IDL_RF_READ_TOO_LONG): region dropped */
#define IDL_RS_ALPHABET       32u   /* WARNING, results are produced: a byte outside {A,C,G,T,N} (lower case, IUPAC codes, '=') was folded
                                       at pack time (acgt -> ACGT, anything else -> N).  The reference compares raw characters
                                       (src/contig.nim:93,122), so its answer may differ for this region */
#define IDL_RS_BAD_INPUT      64u   /* a read record of the batch is malformed (bounds / alignment): region dropped */
/* bits that drop the region (no contigs are returned); the others are warnings */
#define IDL_RS_FATAL (IDL_RS_CONTIG_OVERFLOW | IDL_RS_CORR_OVERFLOW | IDL_RS_READ_TOO_LONG | IDL_RS_BAD_INPUT)

/* idl_region.flags, set by whoever packs the batch */
#define IDL_RF_ALPHABET       1u    /* a base of this region's reads or window was folded (see IDL_RS_ALPHABET) */
#define IDL_RF_READ_TOO_LONG  2u    /* a read of this region exceeds max_read_len and was packed empty */

#define IDL_MAX_CORRECTIONS 128
#define IDL_MAX_EVENTS 4            /* src/indelope.nim:229 */
#define IDL_KMER 27                 /* src/indelope.nim:201 (K); codes must fit 64 bits */

/* Every literal of the reference's path (SURVEY.md section 5 "config"); idl_default_params fills
 * the reference's values. */
typedef struct idl_params {
	int32_t abi_version;
	/* CLI, src/indelope.nim:568-570 */
	int32_t min_reads;            /* -m  [3]  */
	int32_t min_ctg_len;          /* -c  [73] */
	int32_t min_event_len;        /* -e  [4]  */
	/* assembler */
	int32_t asm_min_mapq;         /* 20, src/indelope.nim:157,164 */
	int32_t combine_min_support;  /* 3,  src/indelope.nim:176 */
	int32_t combine_min_overlap;  /* 65, src/contig.nim:224 */
	int32_t max_contigs;          /* 20, src/indelope.nim:209 (pre-combine count gate) */
	/* contig -> reference alignment (call-site A), src/indelope.nim:213-221, src/ksw2/ksw2.nim:142 */
	int32_t stop_min_mapq;        /* reads with MAPQ > 5 extend the window, :215 */
	int32_t window_pad;           /* width + 50 = 63, :218-220 */
	int32_t match, mismatch;      /* 1, -2 */
	int32_t a_gapo, a_gape, a_bw, a_zdrop;   /* 4, 1, 50, 400 */
	/* AL fallback (call-site B), src/indelope.nim:317-318,343-344 */
	int32_t b_gapo, b_gape, b_bw, b_zdrop;   /* 5, 1, -1, -1 */
	/* k-mer genotyping, src/indelope.nim:218,229,294 */
	int32_t max_events;           /* 4 */
	int32_t count_min_mapq;       /* 10 */
	/* capacities of this implementation (not reference semantics) */
	int32_t max_contig_len;       /* bases per contig slot, multiple of 64 [4096] */
	int32_t max_read_len;         /* [512] */
	int32_t max_reads_per_region; /* 600 (src/indelope.nim:515) + 1 */
	int32_t n_streams;            /* copy/compute streams [2] */
	/* what to run / return */
	uint32_t stages;              /* IDL_STAGE_* mask, default all */
	uint32_t out_flags;           /* IDL_OUT_* */
} idl_params;

#define IDL_STAGE_ASSEMBLE 1u
#define IDL_STAGE_ALIGN    2u
#define IDL_STAGE_GENOTYPE 4u
#define IDL_STAGE_ALL      7u
#define IDL_OUT_SUPPORT    1u   /* also return per-base support of every contig (parity tests) */

void idl_default_params(idl_params *p);

/* ---- batch: what the host sweep hands over (SURVEY.md 8b) -------------------------------------
 * One record per region of interest (`roi`, src/indelope.nim:21) and per read (hts-nim Record fields the
 * path uses), in the order gen_roi_internal collected them (BAM order, :480-484).  Sequences are 2 bits per
 * base (A,C,G,T = 0..3 as src/ksw2/ksw2.nim:127; base i of a record at bits 2*(i%16) of word i/16) plus a
 * 1-bit-per-base plane marking non-ACGT bases (their 2-bit code must be 0).  Every record starts on a 64-base
 * boundary of its pool, i.e. 16-byte aligned in the 2-bit pool.  The host computes the quality trim
 * (src/indelope.nim:23-38) and min_overlap = int(0.88*trimmed_len) (:169) so base qualities never cross the bus. */
typedef struct idl_region {
	int32_t chrom_id;
	int32_t roi_start, roi_end;   /* inclusive, as yielded by gen_roi_internal */
	uint32_t read_begin, n_reads; /* into read[] */
	int32_t ref_start;            /* genomic 0-based position of ref window base 0 */
	uint32_t ref_off;             /* base offset of the window in the ref pools (multiple of 64) */
	uint32_t ref_len;             /* window must reach min(chrom_len-1, max(max_stop, max read start+trim)+window_pad) */
	int32_t max_stop;             /* max(read.stop) over reads with MAPQ > stop_min_mapq, or -1 (:213-216) */
	uint32_t ordinal;             /* emission order key of the region (SURVEY.md 8e) */
	uint32_t flags;               /* IDL_RF_* */
	uint32_t reserved;
} idl_region;                     /* 48 bytes */

typedef struct idl_read {
	int32_t start, stop;          /* hts-nim start (0-based) and stop (exclusive end) */
	uint32_t seq_off;             /* base offset in the seq pools (multiple of 64) */
	uint16_t len;                 /* l_qseq, soft clips included (k-mer counting uses the whole read, :300) */
	uint16_t trim_a, trim_len;    /* quality trim: kept bases [trim_a, trim_a+trim_len) */
	uint16_t min_overlap;         /* int(0.88 * trim_len) */
	uint8_t mapq;
	uint8_t flags;                /* bit0: skippable (src/indelope.nim:40-47) */
	uint16_t reserved;
} idl_read;                       /* 24 bytes */

typedef struct idl_batch {
	/* capacities (set by idl_batch_alloc) */
	size_t cap_regions, cap_reads, cap_seq_bases, cap_ref_bases;
	/* fill these */
	size_t n_regions, n_reads, n_seq_bases, n_ref_bases;   /* pool lengths in bases, multiples of 64 */
	idl_region *region;
	idl_read *read;
	uint32_t *seq2;   /* 2-bit pool, cap_seq_bases/16 words */
	uint32_t *seqn;   /* non-ACGT plane, cap_seq_bases/32 words */
	uint32_t *ref2;
	uint32_t *refn;
	void *impl;       /* library private */
	/* optional summary, filled by the packer (idlh_pack does): with summary_valid != 0 idl_submit sizes its workspaces from
	 * these instead of scanning every read and region record on the host */
	uint32_t summary_valid;
	uint32_t max_trim_len;        /* max(read.trim_len), >= 1 */
	uint32_t max_ref_len;         /* max(region.ref_len) */
	uint32_t max_region_reads;    /* max(region.n_reads) */
	size_t n_small_regions;       /* regions with n_reads <= 126 (assembled one per warp) */
} idl_batch;

/* ---- results (library-owned pinned memory, valid until idl_release) -------------------------- */
typedef struct idl_region_result {
	uint32_t status;              /* IDL_RS_* */
	int32_t n_contigs_pre;        /* list length before combine (src/indelope.nim:171) -> INFO NC, gate :209 */
	int32_t n_contigs;            /* after combine */
	uint32_t contig_begin;        /* into contig[] */
} idl_region_result;

typedef struct idl_contig_result {
	int32_t start;                /* genomic position of base 0 */
	int32_t nreads;
	int32_t len;
	uint32_t seq_off;             /* into contig_seq[] (ASCII) and, with IDL_OUT_SUPPORT, contig_support[] */
	int32_t aln;                  /* index into aln[] or -1 if the contig failed the gates of :209-211 */
	uint32_t region;              /* owning region */
} idl_contig_result;

/* the fields of ksw_extz_t (src/ksw2/csrc/ksw2.h:22-30) plus what callsemble derives from them */
typedef struct idl_aln_result {
	uint32_t region, contig;      /* contig = index in contig[] */
	int32_t ref_len;              /* length of the window `reference` (:220) */
	int32_t max, zdropped, max_q, max_t, mqe, mqe_t, mte, mte_q, score;
	int32_t n_cigar;              /* full CIGAR */
	int32_t n_cigar_trunc;        /* ops the truncated iterator yields (src/ksw2/ksw2.nim:22-33) */
	uint32_t cigar_off;           /* into cigar[], BAM encoding len<<4|op, 0=M 1=I 2=D */
	int32_t n_events;             /* I/D ops in the truncated CIGAR (len(qlocs), :222) */
	uint32_t event_begin;         /* into event[]; min(n_events, 4) records when 1 <= n_events <= 4 */
	uint32_t status;
} idl_aln_result;

/* reject codes of idl_event_result.reject */
#define IDL_EV_COUNTED   0
#define IDL_EV_SAME_KMER 1   /* src/indelope.nim:264 */
#define IDL_EV_LOW_CPLX  2   /* :266 */
#define IDL_EV_BUG_SAME  3   /* :268-275 */
#define IDL_EV_SHORT    10   /* :234 */
#define IDL_EV_WINDOW   11   /* reference window or contig shorter than K (the reference would raise) */
#define IDL_EV_DP_ERROR 12   /* the alignment hit a capacity limit (idl_aln_result.status) */
#define IDL_NO_EVENTS 0xffffffffu /* idl_aln_result.event_begin when no event records were written */

typedef struct idl_event_result {
	uint32_t aln;                 /* owning alignment */
	int32_t index;                /* ii, position among all I/D events of the truncated CIGAR */
	int32_t type;                 /* 0 insertion, 1 deletion (src/ksw2/ksw2.nim:63-65) */
	int32_t t_start, t_stop;      /* tloc, genomic (src/ksw2/ksw2.nim:71-80) */
	int32_t q_start, q_stop;      /* qloc, contig coordinates (:82-91) */
	int32_t len;
	int32_t reject;               /* IDL_EV_* */
	int32_t tstart, qstart;       /* offsets of ref_kmer in the window and alt_kmer in the contig (:236-262) */
	int32_t offset;               /* min(qloc.start, ctg.len - qloc.stop - 1), :243 */
	int32_t min_flank;            /* get_min_flank, :118-132 */
	int32_t k_ref, k_alt, k_both; /* k-mer pass: ref_support, alt_support, both_found (:293-311) */
	int32_t aligned;              /* 1 if the AL fallback ran (:313-372) */
	int32_t ref_support, alt_support, both_found;   /* final values fed to the filters (:375-) */
	int32_t n_adist, n_rdist;     /* len(adists), len(rdists) */
	int64_t sum_adist, sum_rdist; /* their sums (means are taken on the host in float64) */
	int32_t amq_median, rmq_median; /* median() of :152-155 over amapqs / rmapqs, -1 if empty */
	uint64_t ref_code, alt_code;  /* canonical 2-bit codes of the two k-mers (~0 if non-ACGT) */
} idl_event_result;

typedef struct idl_results {
	size_t n_regions, n_contigs, n_alns, n_events, n_cigar_ops, n_contig_bases;
	const idl_region_result *region;
	const idl_contig_result *contig;
	const idl_aln_result *aln;
	const idl_event_result *event;
	const uint32_t *cigar;
	const char *contig_seq;          /* ASCII, ACGTN */
	const uint32_t *contig_support;  /* NULL unless IDL_OUT_SUPPORT */
	/* device timings of this ticket, ms, CUDA events on the ticket's stream */
	float ms_h2d, ms_assemble, ms_align, ms_genotype, ms_al, ms_d2h, ms_total;
	/* device-side work counters (algorithmic units, SURVEY.md 8d) */
	uint64_t offsets_tested, dp_cells_a, dp_cells_b, dp_a, dp_b, kmer_reads, kmer_bytes, al_events;
	uint32_t kernel_launches;
	uint32_t pool_retries;           /* times the chain was run again with larger CIGAR / AL item pools (their sizes are estimates) */
} idl_results;

typedef struct idl_ctx idl_ctx;

int idl_create(int device, const idl_params *p, idl_ctx **out);
void idl_destroy(idl_ctx *ctx);
int idl_batch_alloc(idl_ctx *ctx, size_t max_regions, size_t max_reads, size_t max_seq_bases, size_t max_ref_bases, idl_batch **out);
void idl_batch_free(idl_ctx *ctx, idl_batch *b);
/* async: H2D copies + the kernel chain on stream (ticket % n_streams); returns immediately */
int idl_submit(idl_ctx *ctx, idl_batch *b, uint64_t *ticket);
/* same, but the batch arrays are already resident on the device from a previous idl_upload (no H2D, no D2H of
 * anything but counters): used to time the kernels alone */
int idl_upload(idl_ctx *ctx, idl_batch *b);
int idl_run_resident(idl_ctx *ctx, idl_batch *b, uint64_t *ticket);
int idl_wait(idl_ctx *ctx, uint64_t ticket, const idl_results **out);
int idl_release(idl_ctx *ctx, uint64_t ticket);
const char *idl_strerror(int status);
const char *idl_last_cuda_error(idl_ctx *ctx);
int idl_device_count(void);
int idl_device_memory(int device, size_t *free_bytes, size_t *total_bytes);   /* cudaMemGetInfo of the device (callers size their work by it) */

/* ---- unit-level entry point: a batch of independent extension alignments through kernel 2 ------
 * Same contract as the reference's ksw_extz2_sse (src/ksw2/csrc/ksw2.h:54, flag = 0, m = 5 with the matrix of
 * src/ksw2/ksw2.nim:135-140).  query/target are 0..4 codes, concatenated; q_off/t_off have n+1 entries.
 * out[i] receives the ksw_extz_t fields; cigar_off[i] is where task i's out[i].n_cigar ops start in cigar[]
 * (cigar_cap ops in total, handed out in completion order). */
typedef struct idl_ez {
	int32_t max, zdropped, max_q, max_t, mqe, mqe_t, mte, mte_q, score, n_cigar;
	int32_t status;
	int32_t reserved;
	int64_t cells;                /* exact in-band cells over executed diagonals */
} idl_ez;
int idl_ksw2_batch(idl_ctx *ctx, size_t n, const uint8_t *query, const uint64_t *q_off, const uint8_t *target, const uint64_t *t_off,
                   int8_t match, int8_t mismatch, int8_t gapo, int8_t gape, int w, int zdrop,
                   idl_ez *out, uint32_t *cigar, uint64_t *cigar_off, size_t cigar_cap, float *kernel_ms);

/* ---- regions of interest on the GPU (SURVEY.md 8(f)4) -----------------------------------------------------------------
 * One call per target (chromosome): replaces the body of gen_roi (src/indelope.nim:515-545) with gen_roi_internal (:461-499),
 * event_locations (:430-442), overlaps (:449-452) and the flag tests of skippable (:40-47; the two contig-name tests stay with the
 * caller, who simply does not call this for a decoy contig).  Input: the records of the target in BAM order (coordinate sorted) as
 * plain arrays; output: the regions in the order gen_roi yields them, each with the indices of its records (into the input arrays),
 * exactly the (roi_start, roi_end, reads) tuples of src/indelope.nim:21.  min_read_coverage must be >= 1.
 * Synchronous; the arrays of idl_sweep_out belong to the library (idl_sweep_free). */
typedef struct idl_sweep_in {
	int32_t chrom_len;            /* t.length (:522) */
	size_t n_reads;
	const int32_t *start, *stop;  /* hts-nim start (0-based) / stop (exclusive end) */
	const uint16_t *flag;         /* BAM flag */
	const uint32_t *cigar;        /* BAM encoding len<<4|op (M0 I1 D2 N3 S4 H5 P6 =7 X8), all records concatenated */
	const uint64_t *cig_off;      /* n_reads + 1 offsets into cigar[] */
} idl_sweep_in;

#define IDL_SWEEP_EVIDENCE 1u     /* also return the saturating uint8 evidence array (:522,538-543; parity tests) */

typedef struct idl_sweep_out {
	size_t n_rois;
	int32_t *roi_start, *roi_end; /* inclusive, as yielded by gen_roi_internal */
	int64_t *roi_read_begin;      /* into read_idx[] */
	int32_t *roi_n_reads;
	size_t n_read_idx;
	int64_t *read_idx;            /* record indices, BAM order inside a region */
	size_t n_runs;                /* runs of evidence >= min_event_support before the read-count filter of :486 */
	size_t n_evidence; uint8_t *evidence;   /* chrom_len + 1 bytes with IDL_SWEEP_EVIDENCE, else NULL */
	float ms_h2d, ms_kernels, ms_d2h;       /* CUDA events on the call's stream */
	uint64_t algorithmic_bytes;   /* records + CIGARs once, one evidence byte per position written and read once, results */
	uint64_t streamed_bytes;      /* what the passes really move through HBM (memsets, difference array twice, evidence + cuts twice ...) */
} idl_sweep_out;

int idl_sweep(int device, const idl_sweep_in *in, int32_t min_event_support, int32_t min_read_coverage, int32_t max_read_coverage, uint32_t flags, idl_sweep_out **out);
void idl_sweep_free(idl_sweep_out *out);

/* ---------------------------------------------------------------------------------------------------------------
 * 8(f)3: the BAM on the device.  Replaces what stands between the file and gen_roi in the reference: htslib's BGZF reader (one
 * inflate + CRC-32 per <= 64 KiB member, `open(b, path, threads = ..., index = true)`, src/indelope.nim:595) and the record
 * iterator behind `for aln in b.querys(t.name)` (:527) with the accessors the sweep uses (aln.start, aln.stop, aln.flag, aln.cigar:
 * :40-47, :430-452), and the base / quality strings `callsemble` takes from the cached records (:216-222).
 *
 * idl_bam_open: the whole file (bytes as read from disk) -> device: every member inflated and CRC-checked by one warp, record
 * boundaries found per 64 KiB segment and chained exactly (a guessed start is only kept when the previous segment's chain ends
 * on it), one thread per record extracts the fixed fields and the reference span of the CIGAR.  Records without a target (the
 * unplaced tail of a sorted BAM) are not kept; a record without a target BEFORE a placed one, an unsorted file, a malformed
 * record or member give IDL_E_FORMAT with the reason in err.  The file and 4-5x its size must fit in device memory.
 * --------------------------------------------------------------------------------------------------------------- */
typedef struct idl_bam idl_bam;

typedef struct idl_bam_info {
	uint64_t file_bytes, inflated_bytes;
	uint32_t n_members;              /* BGZF members, the empty EOF marker included */
	uint32_t boundary_fixups;        /* segments whose guessed first record was not on the chain (re-walked from the true offset) */
	int32_t n_ref;                   /* targets of the header, in header order (the order gen_roi visits them, :599-601) */
	const char *const *ref_name;     /* library-owned, valid until idl_bam_close */
	const int64_t *ref_len;
	const char *header_text; size_t header_len;
	int64_t n_records;               /* records with a target */
	int64_t n_unplaced;              /* records of the unplaced tail (dropped) */
	const int64_t *ref_first;        /* n_ref + 1 entries: records [ref_first[c], ref_first[c + 1]) belong to target c */
	float ms_h2d, ms_inflate, ms_parse;   /* CUDA events on the call's stream; the file goes up in chunks that are inflated as they arrive: ms_h2d is
	                                         the set-up before the first chunk, ms_inflate the copies and the kernels together */
	uint32_t n_chunks;
} idl_bam_info;

int idl_bam_open(int device, const uint8_t *file, size_t file_len, idl_bam **bam, char *err, size_t errlen);

/* The same for ONE TARGET of a file that does not fit in device memory as a whole: <members> is a run of whole BGZF members from the middle of the
 * file that holds the target's records (the index <bam>.bai says where: libindelope_host's idlh_bai_target_span), the header comes from the caller.
 * The record chain starts at first_record (an offset into the inflated bytes of the run: the low 16 bits of the virtual offset of the target's first
 * record) and ends end_offset bytes into the member that starts end_member bytes into the run (end_member == len, end_offset == 0: at the end of the
 * run) -- what lies in front of and behind them belongs to the neighbouring targets.  Everything else as after idl_bam_open; record indices count
 * from the first record of the run. */
typedef struct idl_bam_slice {
	int32_t n_ref; const char *const *ref_name; const int64_t *ref_len;   /* the targets of the file's header */
	uint64_t first_record;
	uint64_t end_member, end_offset;
} idl_bam_slice;
int idl_bam_open_slice(int device, const uint8_t *members, size_t len, const idl_bam_slice *slice, idl_bam **bam, char *err, size_t errlen);
const idl_bam_info *idl_bam_get_info(const idl_bam *bam);
void idl_bam_close(idl_bam *bam);

/* gen_roi for one target on the resident records: the regions idl_sweep returns for the same records given as host arrays;
 * read_idx[] are indices into the BAM's kept records (0 .. n_records). */
int idl_bam_sweep(idl_bam *bam, int32_t target, int32_t min_event_support, int32_t min_read_coverage, int32_t max_read_coverage, uint32_t flags, idl_sweep_out **out);

#define IDL_BAM_SEQ 1u      /* bases (ASCII, "=ACMGRSVTWYHKDBN") and qualities */
#define IDL_BAM_CIGAR 2u    /* CIGAR operations */

/* records idx[0..n) (idx == NULL: records 0..n) as host arrays, in the order of idx: what callsemble reads of a cached record */
typedef struct idl_bam_reads {
	size_t n;
	int32_t *chrom, *start, *stop, *len; uint8_t *mapq; uint16_t *flag;
	int64_t *seq_off;                /* n + 1 offsets into bases[] / quals[] (IDL_BAM_SEQ) */
	uint8_t *bases, *quals;
	uint64_t *cig_off;               /* n + 1 offsets into cigar[] (IDL_BAM_CIGAR) */
	uint32_t *cigar;                 /* BAM encoding len << 4 | op */
	float ms_kernels, ms_d2h;
} idl_bam_reads;
int idl_bam_fetch(idl_bam *bam, size_t n, const int64_t *idx, uint32_t what, idl_bam_reads **out);
void idl_bam_reads_free(idl_bam_reads *r);

/* The batch built ON THE DEVICE: regions (as idl_bam_sweep returned them: target, bounds, records) -> the quality trim of their records
 * (src/indelope.nim:23-38), the reference windows (:213-220), read and region records and the 2-bit + N-plane pools, written straight into
 * a lane's device buffers from the resident BAM (bases are still BAM nibbles there) and the resident reference -- no record, base or
 * quality crosses the bus.  Byte for byte the batch idlh_pack builds on the host from idl_bam_fetch's arrays.
 *   idl_bam_set_reference: the sequence of one target (ASCII, as in the FASTA; length must equal the header's) -- once per target.
 *   idl_bam_submit:        build + run the calling chain; wait / release with idl_wait / idl_release as after idl_submit.
 *                          roi_n_reads[k] records per region, concatenated in read_idx[] (indices into the BAM's records);
 *                          ordinal_base + k becomes idl_region.ordinal.  IDL_E_ARG for an index outside the BAM or a target without reference.
 *   idl_bam_pack:          build only and copy the batch into <out> (from idl_batch_alloc, large enough: IDL_E_CAPACITY otherwise) -- for
 *                          tests and for callers that want to keep the batch. */
int idl_bam_set_reference(idl_bam *bam, int32_t target, const uint8_t *seq, int64_t len);
int idl_bam_submit(idl_ctx *ctx, idl_bam *bam, size_t n_regions, const int32_t *roi_chrom, const int32_t *roi_start, const int32_t *roi_end,
                   const int32_t *roi_n_reads, const int64_t *read_idx, uint32_t ordinal_base, uint64_t *ticket);
int idl_bam_pack(idl_ctx *ctx, idl_bam *bam, size_t n_regions, const int32_t *roi_chrom, const int32_t *roi_start, const int32_t *roi_end,
                 const int32_t *roi_n_reads, const int64_t *read_idx, uint32_t ordinal_base, idl_batch *out);

#ifdef __cplusplus
}
#endif
#endif
