/* oracle/oracle.h -- TEST INFRASTRUCTURE (CPU oracle).
 *
 * C interface (for ctypes) of the CPU restatement of indelope's per-region calling path.
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
 * load this library; the product (libindelope_cuda.so, libindelope_host.so) never does.
 */
#ifndef ORC_ORACLE_H
#define ORC_ORACLE_H
#include <stdint.h>
#include "ksw2_lane.h"

#ifdef __cplusplus
extern "C" {
#endif

/* A set of regions of interest in the shape the reference's gen_roi yields them
 * (src/indelope.nim:21 `roi = tuple[start, stop, reads: seq[Record]]`), flattened to arrays. */
typedef struct {
	/* read table (hts-nim Record fields used on the path) */
	int64_t n_reads;
	const int32_t *start;     /* 0-based leftmost */
	const int32_t *stop;      /* end, exclusive (bam_endpos) */
	const uint8_t *mapq;
	const uint16_t *flag;
	const int32_t *len;       /* l_qseq, soft clips included */
	const int64_t *seq_off;   /* offset of the read in bases[] / quals[] */
	const uint8_t *bases;     /* ASCII */
	const uint8_t *quals;     /* phred, no offset */
	/* regions */
	int64_t n_rois;
	const int32_t *roi_chrom;
	const int32_t *roi_start, *roi_stop;      /* inclusive bounds as gen_roi_internal yields them */
	const int64_t *roi_read_begin;            /* into read_idx[] */
	const int32_t *roi_n_reads;
	const int64_t *read_idx;                  /* read table indices, BAM order inside a region */
	/* reference */
	int32_t n_chroms;
	const char *const *chrom_name;
	const uint8_t *const *chrom_seq;          /* ASCII */
	const int64_t *chrom_len;
} orc_roiset_t;

typedef struct {
	int32_t min_reads;      /* -m, src/indelope.nim:568 */
	int32_t min_ctg_len;    /* -c, :569 */
	int32_t min_event_len;  /* -e, :570 */
	int32_t use_ref_ksw2;   /* 1: run DPs through oracle/_ref/libksw2_ref.so (must be loaded first) */
	int32_t dump_level;     /* bit0 R/C lines, bit1 supports in C lines, bit2 A lines, bit3 E lines, bit4 V lines, bit5 no dedup, bit6 L lines (capacity limits per region; test only) */
	int32_t n_threads;      /* regions are independent; >1 only parallelises across regions */
} orc_params_t;

typedef struct {
	int64_t regions, reads;             /* callsemble invocations, sum of len(roi.reads) */
	int64_t slide_calls, offsets;       /* slide_align calls, offsets tested (SURVEY 8d) */
	int64_t char_compares;              /* early-abort compares the reference really does */
	int64_t exhaustive_compares;        /* sum over offsets of the overlap length */
	int64_t contigs_pre, contigs_post;
	int64_t dp_a, dp_b;                 /* alignments at call-site A / B */
	int64_t cells_a, cells_b;           /* exact in-band cells over executed diagonals */
	int64_t events, kmer_reads, kmer_windows, kmer_bytes;
	int64_t al_events;
	int64_t variants;
	double seconds;                     /* wall time of the call */
	int64_t corrections;                /* voting sites applied by Contig.insert (src/contig.nim:161-173) */
	int64_t vote_invariant_violations;  /* a correction with q.nreads < 4 or t.nreads < 4: never happens (GPU fast path relies on it) */
	int64_t left_merges, merges;        /* merges with offset < 0 / all merges */
} orc_counters_t;

/* load oracle/_ref/libksw2_ref.so (the compiled reference DP); 0 on success */
int orc_load_ref(const char *path);

/* run the path over a region set. *dump and *vcf are malloc'ed NUL-terminated texts (free with
 * orc_free); vcf holds only record lines (no header), dedup'ed as src/indelope.nim:604-608 does. */
int orc_call(const orc_roiset_t *in, const orc_params_t *p, char **dump, char **vcf, orc_counters_t *cnt);
void orc_free(void *p);

/* VCF header as src/indelope.nim:77-102,548-552,600 prints it (malloc'ed) */
char *orc_vcf_header(int32_t n_chroms, const char *const *names, const int64_t *lens);

/* ---- unit-level entry points used by the known-answer tests ---- */
/* rule: 0 = production allowable_mismatch (src/contig.nim:44-47), 1 = the test-only rule of
 * src/contig.nim:287-290 */
typedef struct { int64_t matches, offset, mismatches; int32_t aligned, n_corr; int32_t corr[3 * 64]; } orc_match_t;
void orc_slide_align(const char *q, const uint32_t *qsup, int64_t qreads,
                     const char *t, const uint32_t *tsup, int64_t treads,
                     int64_t min_overlap, int64_t max_mismatch, int rule, orc_match_t *out);
/* insert q into t with a given match; results written back (buffers must hold qlen+tlen) */
void orc_insert(char *t, uint32_t *tsup, int64_t *tlen, int64_t *treads, int64_t *tstart,
                char *q, uint32_t *qsup, int64_t qlen, int64_t qreads, int64_t qstart,
                const orc_match_t *m);
/* assemble one list of (sequence,start,min_overlap) through list-insert + combine; dumps C lines */
char *orc_assemble_strings(int n, const char *const *seqs, const int64_t *starts, const int64_t *min_overlaps,
                           int do_combine, int64_t *n_pre);
/* genotype text "GT:GQ:GL" and class, src/genotyper.nim:31-47 */
int orc_genotype(int64_t r, int64_t a, double error, char *text, int cap, double *qual);
/* read quality trim, src/indelope.nim:23-38: returns a; *out_len = trimmed length */
int32_t orc_trim(const uint8_t *quals, int32_t n, int32_t *out_len);
/* canonical k-mer code declared in SURVEY appendix D; returns 0 and sets *code, or -1 if non-ACGT */
int orc_mincode(const char *s, int k, uint64_t *code);

#ifdef __cplusplus
}
#endif
#endif
