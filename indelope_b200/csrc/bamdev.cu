// indelope_b200/csrc/bamdev.cu -- SURVEY.md 8(f)3: BGZF inflate and BAM record parse on the GPU (idl_bam_* of include/indelope_cuda.h).
//
// What it replaces in the reference: htslib's BGZF reader and record iterator behind `open(b, path, threads, index = true)` and
// `for aln in b.querys(t.name)` (src/indelope.nim:595, :527) -- the reference's own bottleneck (README.md:5: the whole program runs at
// 1.25x `samtools view -c`, i.e. at the speed of the decoder) -- and the accessors the sweep and callsemble read of a record
// (aln.start / stop / flag / cigar :40-47, :430-452; the base and quality strings :216-222).
//
// Stages, all on one stream:
//   1. host: walk the member headers of the file (18 bytes each + ISIZE), prefix sum of ISIZE = where every member's output goes;
//   2. H2D of the compressed bytes; bgzf_inflate_kernel: ONE WARP PER MEMBER, persistent CTAs pulling members from an atomic counter;
//      the decoder and the CRC-32 are inflate_core.cuh (lanes in lockstep on the serial bit stream, parallel in match copies, table
//      fills and the CRC slices);
//   3. record boundaries.  A BAM record is only found by walking block_size fields from the previous one -- a chain through the whole
//      file.  bam_seg_kernel cuts the inflated stream into 64 KiB segments; one warp per segment GUESSES the first record that starts
//      in it (32 candidate offsets per step, each checked against the necessary conditions of a record and of the two records
//      behind it), walks the chain to the segment's end and reports (first, exit, count).  The host then checks the one thing that
//      makes the result exact instead of plausible: segment k's exit must be segment k+1's first record.  Where it is not (a false
//      positive of the guess), that segment is walked again from the true offset (rare; counted in boundary_fixups);
//   4. bam_offsets_kernel writes the offset of every record, bam_fields_kernel (one thread per record) the fixed fields, the reference
//      span of the CIGAR (bam_endpos) and the positions of CIGAR / bases / qualities inside the inflated stream -- the bases stay where
//      they are, as BAM nibbles, until idl_bam_fetch decodes the ones a region needs;
//   5. a 64-bit exclusive scan of n_cigar + a gather make the contiguous CIGAR array idl_sweep's kernels take; per-target record ranges
//      by binary search.
#include <algorithm>
#include <chrono>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include <cuda_runtime.h>
#include "indelope_cuda.h"
#include "sweep_impl.h"
#include "bamdev.h"
#include "inflate_core.cuh"

namespace {

using namespace idl_inflate;

#ifndef INF_WARPS_
#define INF_WARPS_ 6
#endif
#ifndef INF_CTAS_PER_SM_
#define INF_CTAS_PER_SM_ 5
#endif
constexpr int INF_WARPS = INF_WARPS_;        // warps per CTA of the inflate kernel: 6 x 6.1 KB of tables
constexpr int INF_CTAS_PER_SM = INF_CTAS_PER_SM_;
constexpr unsigned SEG_BYTES = 1u << 16;     // segment of the inflated stream one warp chains
constexpr int SCAN_THREADS = 256, SCAN_ITEMS = 8, SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

using Member = BgzfMember;

// ---- stage 2 ----
__global__ void __launch_bounds__(INF_WARPS * 32, INF_CTAS_PER_SM)
bgzf_inflate_kernel(const uint8_t *comp, const Member *members, uint32_t m_begin, uint32_t n_members, uint8_t *out, unsigned long long *first_error, unsigned *next)
{   // members [m_begin, n_members) of the file: one launch per chunk of the file as its bytes arrive (idl_bam_open)
	__shared__ Tables tables[INF_WARPS];
	__shared__ uint32_t crc_tab[256], xp[32];
	crc_init_tables((int)threadIdx.x, (int)blockDim.x, crc_tab, xp);
	__syncthreads();
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	for (;;) {
		unsigned m = 0;
		if (lane == 0) m = m_begin + atomicAdd(next, 1u);
		m = __shfl_sync(0xffffffffu, m, 0);
		if (m >= n_members) break;
		const Member M = members[m];
		int rc = inflate_member(lane, tables[warp], comp, (size_t)M.in_off, (size_t)M.in_len, out + M.out_off, M.out_len);
		__syncwarp();
		if (rc == INF_OK) {
			uint32_t c = crc_lane_part(lane, 32, crc_tab, xp, out + M.out_off, M.out_len);
#pragma unroll
			for (int d = 16; d >= 1; d >>= 1) c ^= __shfl_xor_sync(0xffffffffu, c, d);
			if (~c != M.crc) rc = INF_E_CRC;
		}
		if (rc != INF_OK && lane == 0) atomicMin(first_error, (unsigned long long)m << 8 | (unsigned)rc);   // the first bad member of the file
	}
}

// ---- stage 3 ----
// unaligned little-endian loads from the inflated stream (padded by 8 bytes): two aligned words and a funnel shift
__device__ __forceinline__ uint32_t ld32u(const uint8_t *u, size_t o)
{
	const uint32_t *w = (const uint32_t*)(u + (o & ~(size_t)3));
	return __funnelshift_r(w[0], w[1], (unsigned)(o & 3) * 8);
}

// necessary conditions of a BAM alignment record at offset o (SAM spec 4.2); true records always pass
__device__ bool bam_plausible(const uint8_t *u, size_t total, size_t o, int32_t n_ref, const int32_t *ref_len, size_t *next)
{
	if (o + 36 > total) return false;
	const uint32_t bs = ld32u(u, o);
	if (bs < 32 || bs > (1u << 28) || o + 4 + bs > total) return false;
	const int32_t ref_id = (int32_t)ld32u(u, o + 4), pos = (int32_t)ld32u(u, o + 8);
	if (ref_id < -1 || ref_id >= n_ref || pos < -1) return false;
	if (ref_id >= 0 && pos > ref_len[ref_id]) return false;
	const uint32_t w3 = ld32u(u, o + 12), w4 = ld32u(u, o + 16);
	const uint32_t l_name = w3 & 0xffu, n_cig = w4 & 0xffffu;
	const int32_t l_seq = (int32_t)ld32u(u, o + 20), next_ref = (int32_t)ld32u(u, o + 24), next_pos = (int32_t)ld32u(u, o + 28);
	if (l_name == 0 || l_seq < 0 || next_ref < -1 || next_ref >= n_ref || next_pos < -1) return false;
	if (32ull + l_name + 4ull * n_cig + ((unsigned long long)l_seq + 1) / 2 + (unsigned long long)l_seq > bs) return false;
	if (u[o + 36 + l_name - 1] != 0) return false;   // read_name is NUL terminated
	*next = o + 4 + bs;
	return true;
}

// one warp per segment [begin + k * SEG, begin + (k + 1) * SEG) of the inflated stream.
//   first[k]: offset of the first record that starts in the segment (given when preset[k] >= 0, guessed otherwise), -1 = none
//   exit[k]:  offset of the first record at or behind the segment's end on that chain (total = clean end of file)
//   count[k]: records that start in the segment;  bad[k]: the chain hit a block_size that cannot be (offset stored in exit[k])
__global__ void __launch_bounds__(256) bam_seg_kernel(const uint8_t *u, size_t total, size_t begin, uint32_t n_seg, const uint32_t *which, uint32_t n_which,
                                                      int32_t n_ref, const int32_t *ref_len, const long long *preset, long long *first, long long *exitp,
                                                      uint32_t *count, uint32_t *bad)
{
	const uint32_t wid = (uint32_t)(((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
	const int lane = threadIdx.x & 31;
	if (wid >= (which ? n_which : n_seg)) return;
	const uint32_t k = which ? which[wid] : wid;
	const size_t s0 = begin + (size_t)k * SEG_BYTES, s1 = s0 + SEG_BYTES < total ? s0 + SEG_BYTES : total;
	long long f = preset ? preset[k] : -2;
	if (f < -1) {
		f = -1;
		for (size_t base = s0; base < s1; base += 32) {
			const size_t o = base + lane;
			size_t nx = 0;
			bool ok = o < s1 && bam_plausible(u, total, o, n_ref, ref_len, &nx);
			for (int hop = 0; ok && hop < 2 && nx < total; ++hop) ok = bam_plausible(u, total, nx, n_ref, ref_len, &nx);
			const unsigned m = __ballot_sync(0xffffffffu, ok);
			if (m) { f = (long long)(base + (size_t)(__ffs(m) - 1)); break; }
		}
	}
	// the chain from f to the end of the segment; every lane walks it (identical loads)
	uint32_t c = 0, b = 0;
	size_t o = f < 0 ? s1 : (size_t)f;
	long long ex = f < 0 ? -1 : 0;
	while (f >= 0 && o < s1) {
		if (o + 4 > total) { b = 1; break; }
		const uint32_t bs = ld32u(u, o);
		if (bs < 32 || o + 4 + (size_t)bs > total) { b = 1; break; }
		o += 4 + (size_t)bs; ++c;
	}
	if (f >= 0) ex = (long long)o;
	if (lane == 0) { first[k] = f; exitp[k] = ex; count[k] = c; bad[k] = b; }
}

// offsets of all records: segment k writes count[k] entries from rec_base[k]
__global__ void __launch_bounds__(256) bam_offsets_kernel(const uint8_t *u, size_t total, size_t begin, uint32_t n_seg, const long long *first, const unsigned long long *rec_base,
                                                          long long *rec_off)
{
	const uint32_t k = (uint32_t)(((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
	const int lane = threadIdx.x & 31;
	if (k >= n_seg || first[k] < 0) return;
	const size_t s0 = begin + (size_t)k * SEG_BYTES, s1 = s0 + SEG_BYTES < total ? s0 + SEG_BYTES : total;
	size_t o = (size_t)first[k];
	unsigned long long at = rec_base[k];
	while (o < s1) {
		if (lane == 0) rec_off[at] = (long long)o;
		++at;
		o += 4 + (size_t)ld32u(u, o);
	}
}

// ---- stage 4: one thread per record ----
struct Rec {
	int32_t *ref_id, *pos, *stop, *l_seq; uint8_t *mapq; uint16_t *flag; uint32_t *n_cig; long long *cig_at, *seq_at;
};
__global__ void __launch_bounds__(256) bam_fields_kernel(const uint8_t *u, const long long *rec_off, size_t n, int32_t n_ref, Rec R, unsigned long long *first_bad)
{
	const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const size_t o = (size_t)rec_off[i];
	const uint32_t bs = ld32u(u, o);
	const int32_t ref_id = (int32_t)ld32u(u, o + 4), pos = (int32_t)ld32u(u, o + 8);
	const uint32_t w3 = ld32u(u, o + 12), w4 = ld32u(u, o + 16);
	const uint32_t l_name = w3 & 0xffu, mapq = (w3 >> 8) & 0xffu, n_cig = w4 & 0xffffu, flag = w4 >> 16;
	const uint32_t l_seq = ld32u(u, o + 20);
	bool bad = 32ull + l_name + 4ull * n_cig + ((unsigned long long)l_seq + 1) / 2 + (unsigned long long)l_seq > bs;   // "malformed BAM record"
	bad |= ref_id >= n_ref;                                                                                              // "unknown reference id"
	long long rlen = 0;
	const size_t cig = o + 36 + l_name;
	if (!bad)
		for (uint32_t k = 0; k < n_cig; ++k) {
			const uint32_t c = ld32u(u, cig + 4 * (size_t)k), op = c & 0xfu;
			if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) rlen += c >> 4;
		}
	if ((flag & 4u) || n_cig == 0 || rlen == 0) rlen = 1;   // bam_endpos
	R.ref_id[i] = ref_id; R.pos[i] = pos; R.stop[i] = (int32_t)(pos + rlen); R.l_seq[i] = (int32_t)l_seq; R.mapq[i] = (uint8_t)mapq; R.flag[i] = (uint16_t)flag;
	R.n_cig[i] = bad ? 0u : n_cig; R.cig_at[i] = (long long)cig; R.seq_at[i] = (long long)(cig + 4 * (size_t)n_cig);
	if (bad) atomicMin(first_bad, (unsigned long long)i);
}
// coordinate order of the placed records, placed records before the unplaced tail; n_placed = index of the first record without a target
__global__ void __launch_bounds__(256) bam_order_kernel(const int32_t *ref_id, const int32_t *pos, size_t n, unsigned long long *first_unsorted, unsigned long long *first_unplaced)
{
	const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const int32_t r = ref_id[i];
	if (r < 0) { atomicMin(first_unplaced, (unsigned long long)i); return; }
	if (i > 0) {
		const int32_t rp = ref_id[i - 1];
		if (rp < 0 || rp > r || (rp == r && pos[i - 1] > pos[i])) atomicMin(first_unsorted, (unsigned long long)i);
	}
}
__global__ void bam_ref_first_kernel(const int32_t *ref_id, size_t n, int32_t n_ref, long long *ref_first)
{
	const int c = blockIdx.x * blockDim.x + threadIdx.x;
	if (c > n_ref) return;
	size_t lo = 0, hi = n;   // first record with ref_id >= c
	while (lo < hi) { const size_t mid = (lo + hi) >> 1; if (ref_id[mid] >= c) hi = mid; else lo = mid + 1; }
	ref_first[c] = (long long)lo;
}

// ---- 64-bit exclusive scan of uint32 values (n + 1 outputs): tile totals, one CTA over the totals, apply ----
__device__ __forceinline__ unsigned long long block_excl_scan(unsigned long long v, unsigned long long *sh, unsigned long long *total)
{
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
	unsigned long long inc = v;
#pragma unroll
	for (int d = 1; d < 32; d <<= 1) { const unsigned long long o = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += o; }
	if (lane == 31) sh[warp] = inc;
	__syncthreads();
	unsigned long long before = 0, tot = 0;
	for (int w = 0; w < nw; ++w) { if (w < warp) before += sh[w]; tot += sh[w]; }
	__syncthreads();
	*total = tot;
	return before + inc - v;
}
__global__ void __launch_bounds__(SCAN_THREADS) scan_tile_totals_kernel(const uint32_t *in, size_t n, unsigned long long *totals)
{
	__shared__ unsigned long long sh[SCAN_THREADS / 32];
	const size_t base = (size_t)blockIdx.x * SCAN_TILE + (size_t)threadIdx.x * SCAN_ITEMS;
	unsigned long long acc = 0;
	for (int k = 0; k < SCAN_ITEMS; ++k) if (base + k < n) acc += in[base + k];
	unsigned long long tot;
	block_excl_scan(acc, sh, &tot);
	if (threadIdx.x == 0) totals[blockIdx.x] = tot;
}
__global__ void __launch_bounds__(1024) scan_totals_kernel(unsigned long long *totals, size_t nt)
{
	__shared__ unsigned long long sh[32];
	const size_t per = (nt + 1023) / 1024, lo = (size_t)threadIdx.x * per, hi = lo + per < nt ? lo + per : nt;
	unsigned long long acc = 0;
	for (size_t i = lo; i < hi; ++i) acc += totals[i];
	unsigned long long tot;
	unsigned long long run = block_excl_scan(acc, sh, &tot);
	for (size_t i = lo; i < hi; ++i) { const unsigned long long t = totals[i]; totals[i] = run; run += t; }
}
__global__ void __launch_bounds__(SCAN_THREADS) scan_apply_kernel(const uint32_t *in, size_t n, const unsigned long long *totals, unsigned long long *out)
{
	__shared__ unsigned long long sh[SCAN_THREADS / 32];
	const size_t base = (size_t)blockIdx.x * SCAN_TILE + (size_t)threadIdx.x * SCAN_ITEMS;
	uint32_t x[SCAN_ITEMS]; unsigned long long acc = 0;
#pragma unroll
	for (int k = 0; k < SCAN_ITEMS; ++k) { x[k] = base + k < n ? in[base + k] : 0u; acc += x[k]; }
	unsigned long long tot;
	unsigned long long run = totals[blockIdx.x] + block_excl_scan(acc, sh, &tot);
#pragma unroll
	for (int k = 0; k < SCAN_ITEMS; ++k) if (base + k <= n) { out[base + k] = run; run += x[k]; }   // out[n] = the grand total
}
__global__ void __launch_bounds__(256) bam_cigar_gather_kernel(const uint8_t *u, const long long *cig_at, const unsigned long long *cig_off, size_t n, uint32_t *cigar)
{
	const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const unsigned long long o0 = cig_off[i], o1 = cig_off[i + 1];
	const size_t at = (size_t)cig_at[i];
	for (unsigned long long k = o0; k < o1; ++k) cigar[k] = ld32u(u, at + 4 * (size_t)(k - o0));
}

// ---- idl_bam_fetch: one warp per requested record ----
__constant__ char SEQ16[17] = "=ACMGRSVTWYHKDBN";
__global__ void __launch_bounds__(256) bam_fetch_fields_kernel(const long long *idx, size_t n, Rec R, int32_t *chrom, int32_t *start, int32_t *stop, int32_t *len, uint8_t *mapq,
                                                               uint16_t *flag, uint32_t *n_cig)
{
	const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (j >= n) return;
	const size_t i = idx ? (size_t)idx[j] : j;
	chrom[j] = R.ref_id[i]; start[j] = R.pos[i]; stop[j] = R.stop[i]; len[j] = R.l_seq[i]; mapq[j] = R.mapq[i]; flag[j] = R.flag[i]; n_cig[j] = R.n_cig[i];
}
__global__ void __launch_bounds__(256) bam_fetch_seq_kernel(const uint8_t *u, const long long *idx, size_t n, Rec R, const long long *seq_off, uint8_t *bases, uint8_t *quals)
{
	const size_t j = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	const int lane = threadIdx.x & 31;
	if (j >= n) return;
	const size_t i = idx ? (size_t)idx[j] : j;
	const uint32_t l = (uint32_t)R.l_seq[i];
	const uint8_t *seq = u + R.seq_at[i], *q = seq + (l + 1) / 2;
	uint8_t *b = bases + seq_off[j], *qo = quals + seq_off[j];
	for (uint32_t t = (uint32_t)lane; t < l; t += 32) {
		const uint8_t by = seq[t >> 1];
		b[t] = (uint8_t)SEQ16[(t & 1) ? (by & 15) : (by >> 4)];
		qo[t] = q[t];
	}
}
__global__ void __launch_bounds__(256) bam_fetch_cigar_kernel(const long long *idx, size_t n, const unsigned long long *src_off, const uint32_t *src, const unsigned long long *dst_off, uint32_t *dst)
{
	const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (j >= n) return;
	const size_t i = idx ? (size_t)idx[j] : j;
	const unsigned long long s = src_off[i], e = src_off[i + 1], d = dst_off[j];
	for (unsigned long long k = s; k < e; ++k) dst[d + (k - s)] = src[k];
}

// ---- the batch builder (idl_bam_submit / idl_bam_pack): what idlh_pack does on the host (pack_vcf.cpp), from the resident records ----
struct BuildCounters { unsigned max_trim_len, max_ref_len, max_region_reads, n_small_regions, bad_index, pad[3]; };

// quality trim, src/indelope.nim:23-38 (the restatement of idlh_trim): first and last base with quality >= 15
__device__ __forceinline__ int bam_trim(const uint8_t *bq, int n, int *trim_len)
{
	const int high = n - 1, min_quality = 15;
	int a = 0;
	while (a < high && bq[a] < min_quality) a += 1;
	if (a == high || n <= 0) { *trim_len = 0; return n <= 0 ? 0 : a; }
	int b = high;
	while (b > a && bq[b] < min_quality) b -= 1;
	*trim_len = b - a + 1;
	return a;
}
// one warp per region: read records (all but seq_off), the window, the region record (all but ref_off), padded lengths for the two scans
__global__ void __launch_bounds__(256) bam_build_records_kernel(const uint8_t *u, Rec R, size_t n_records, const int32_t *ref_len, const uint8_t *const *ref_seq, int32_t n_ref,
                                                                idl_params P, size_t n_regions, const int32_t *roi_chrom, const int32_t *roi_start, const int32_t *roi_end,
                                                                const int32_t *roi_n_reads, const unsigned long long *roi_read_begin, const long long *read_idx,
                                                                uint32_t ordinal_base, idl_region *region, idl_read *read, uint32_t *read_pad, uint32_t *slot_region,
                                                                uint32_t *ref_pad, BuildCounters *cnt)
{
	const size_t k = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	const int lane = threadIdx.x & 31;
	if (k >= n_regions) return;
	const unsigned long long begin = roi_read_begin[k];
	const int nr = roi_n_reads[k];
	long long ws = LLONG_MAX, far = -1, max_stop = -1;
	unsigned flags = 0, max_trim = 1, bad = 0;
	for (int j = lane; j < nr; j += 32) {
		const long long i = read_idx[begin + j];
		idl_read r; memset(&r, 0, sizeof r);
		unsigned pad = 0;
		if (i < 0 || (size_t)i >= n_records) bad = 1;
		else {
			const int len = R.l_seq[i];
			const uint8_t *q = u + R.seq_at[i] + (len + 1) / 2;
			int tl; const int ta = bam_trim(q, len, &tl);
			const int start = R.pos[i], stop = R.stop[i]; const unsigned mapq = R.mapq[i], f = R.flag[i];
			r.start = start; r.stop = stop; r.mapq = (uint8_t)mapq;
			r.flags = ((f & 0x400) || (f & 0x200) || (f & 0x4) || (f & 0x800) || (f & 0x100)) ? 1 : 0;   // :40-47
			if (len > P.max_read_len || len > 65535) flags |= IDL_RF_READ_TOO_LONG;                      // packed empty: the device drops the region and says so
			else {
				r.len = (uint16_t)len; r.trim_a = (uint16_t)ta; r.trim_len = (uint16_t)tl;
				r.min_overlap = (uint16_t)(long long)(0.88 * (double)tl);                                // :169
				pad = ((unsigned)len + 63u) & ~63u;
				max_trim = max(max_trim, (unsigned)tl);
			}
			ws = min(ws, (long long)start + ta); far = max(far, (long long)start + ta + tl);
			if ((int)mapq > P.stop_min_mapq) max_stop = max(max_stop, (long long)stop);
		}
		read[begin + j] = r; read_pad[begin + j] = pad; slot_region[begin + j] = (uint32_t)k;
	}
#pragma unroll
	for (int d = 16; d >= 1; d >>= 1) {
		ws = min(ws, __shfl_xor_sync(0xffffffffu, ws, d)); far = max(far, __shfl_xor_sync(0xffffffffu, far, d)); max_stop = max(max_stop, __shfl_xor_sync(0xffffffffu, max_stop, d));
		flags |= __shfl_xor_sync(0xffffffffu, flags, d); max_trim = max(max_trim, __shfl_xor_sync(0xffffffffu, max_trim, d)); bad |= __shfl_xor_sync(0xffffffffu, bad, d);
	}
	if (lane == 0) {
		const int c = roi_chrom[k];
		if (c < 0 || c >= n_ref || !ref_seq[c]) bad = 1;
		if (ws == LLONG_MAX) ws = 0;
		if (ws < 0) ws = 0;
		const long long clen = bad ? 1 : ref_len[c];
		const long long we = min(clen - 1, max(far, max_stop) + P.window_pad);
		idl_region g; memset(&g, 0, sizeof g);
		g.chrom_id = c; g.roi_start = roi_start[k]; g.roi_end = roi_end[k];
		g.read_begin = (uint32_t)begin; g.n_reads = (uint32_t)nr;
		g.ref_start = (int32_t)ws; g.ref_len = (uint32_t)max(0ll, we - ws + 1);
		g.max_stop = (int32_t)max_stop; g.ordinal = ordinal_base + (uint32_t)k; g.flags = flags;
		region[k] = g;
		ref_pad[k] = (g.ref_len + 63u) & ~63u;
		atomicMax(&cnt->max_trim_len, max_trim); atomicMax(&cnt->max_ref_len, g.ref_len); atomicMax(&cnt->max_region_reads, (unsigned)nr);
		if (nr <= 126) atomicAdd(&cnt->n_small_regions, 1u);
		if (bad) atomicOr(&cnt->bad_index, 1u);
	}
}
__global__ void __launch_bounds__(256) bam_build_offsets_kernel(size_t n_reads, size_t n_regions, const unsigned long long *seq_off, const unsigned long long *ref_off, idl_read *read,
                                                                idl_region *region)
{
	const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i < n_reads) read[i].seq_off = (uint32_t)seq_off[i];
	if (i < n_regions) region[i].ref_off = (uint32_t)ref_off[i];
}
// one warp per read: BAM nibbles -> 2-bit codes + N plane, 16 bases per lane and step; the record is padded to a multiple of 64 bases with zero
// words and every word of it is stored.  Nibbles: 1 A, 2 C, 4 G, 8 T, 15 N; the other codes of "=ACMGRSVTWYHKDBN" fold to N and are reported
// (IDL_RF_ALPHABET), as the host packer does with their letters
__global__ void __launch_bounds__(256) bam_pack_reads_kernel(const uint8_t *u, Rec R, const long long *read_idx, size_t n_reads, const idl_read *read, const uint32_t *slot_region,
                                                             idl_region *region, uint32_t *seq2, uint32_t *seqn)
{
	const size_t s = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	const int lane = threadIdx.x & 31;
	if (s >= n_reads) return;
	const idl_read r = read[s];
	if (r.len == 0) return;
	const uint8_t *seq = u + R.seq_at[read_idx[s]];
	const unsigned len = r.len, words = ((len + 63u) & ~63u) >> 4;
	uint32_t *d2 = seq2 + (r.seq_off >> 4); uint16_t *dn = (uint16_t*)seqn + (r.seq_off >> 4);
	unsigned folded = 0;
	for (unsigned w = (unsigned)lane; w < words; w += 32) {
		uint32_t a = 0, nb = 0;
		const unsigned b0 = 16u * w;
		if (b0 < len) {
			// 16 bases = 8 bytes, two nibbles each, the first base in the high nibble
#pragma unroll
			for (int t = 0; t < 8; ++t) {
				const unsigned base = b0 + 2u * (unsigned)t;
				if (base >= len) break;
				const unsigned by = seq[base >> 1];
#pragma unroll
				for (int h = 0; h < 2; ++h) {
					if (base + (unsigned)h >= len) break;
					const unsigned nib = h ? (by & 15u) : (by >> 4);
					const int i = 2 * t + h;
					if (nib == 1u) { }
					else if (nib == 2u) a |= 1u << (2 * i);
					else if (nib == 4u) a |= 2u << (2 * i);
					else if (nib == 8u) a |= 3u << (2 * i);
					else { nb |= 1u << i; folded |= nib != 15u; }
				}
			}
		}
		d2[w] = a; dn[w] = (uint16_t)nb;
	}
	folded = __any_sync(0xffffffffu, folded != 0);
	if (folded && lane == 0) atomicOr(&region[slot_region[s]].flags, (unsigned)IDL_RF_ALPHABET);
}
// one warp per region: the reference window, ASCII -> 2-bit codes + N plane; lower-case acgt fold to upper case, every other byte to N, both
// reported (IDL_RF_ALPHABET): the reference compares raw characters (src/contig.nim:93,122)
__global__ void __launch_bounds__(256) bam_pack_ref_kernel(const uint8_t *const *ref_seq, size_t n_regions, idl_region *region, uint32_t *ref2, uint32_t *refn)
{
	const size_t k = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	const int lane = threadIdx.x & 31;
	if (k >= n_regions) return;
	const idl_region g = region[k];
	const uint8_t *s = ref_seq[g.chrom_id] + g.ref_start;
	const unsigned len = g.ref_len, words = ((len + 63u) & ~63u) >> 4;
	uint32_t *d2 = ref2 + (g.ref_off >> 4); uint16_t *dn = (uint16_t*)refn + (g.ref_off >> 4);
	unsigned folded = 0;
	for (unsigned w = (unsigned)lane; w < words; w += 32) {
		uint32_t a = 0, nb = 0;
		const unsigned b0 = 16u * w;
#pragma unroll
		for (int i = 0; i < 16; ++i) {
			if (b0 + (unsigned)i >= len) break;
			const unsigned c = s[b0 + i];
			if (c == 'A') { }
			else if (c == 'C') a |= 1u << (2 * i);
			else if (c == 'G') a |= 2u << (2 * i);
			else if (c == 'T') a |= 3u << (2 * i);
			else if (c == 'N') nb |= 1u << i;
			else {
				folded = 1;
				if (c == 'a') { }
				else if (c == 'c') a |= 1u << (2 * i);
				else if (c == 'g') a |= 2u << (2 * i);
				else if (c == 't') a |= 3u << (2 * i);
				else nb |= 1u << i;
			}
		}
		d2[w] = a; dn[w] = (uint16_t)nb;
	}
	folded = __any_sync(0xffffffffu, folded != 0);
	if (folded && lane == 0) region[k].flags = g.flags | region[k].flags | (unsigned)IDL_RF_ALPHABET;
}

inline uint16_t h16(const uint8_t *p) { return (uint16_t)(p[0] | p[1] << 8); }
inline uint32_t h32(const uint8_t *p) { return (uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24; }

void set_err(char *err, size_t n, const std::string &m) { if (err && n) snprintf(err, n, "%s", m.c_str()); }

const char *inf_error_text(int rc)
{
	switch (rc) {
	case INF_E_BTYPE: return "reserved deflate block type";
	case INF_E_STORED: return "stored block length check failed";
	case INF_E_CODE: return "invalid Huffman code";
	case INF_E_SYMBOL: return "invalid symbol";
	case INF_E_DISTANCE: return "match distance before the start of the member";
	case INF_E_OUTPUT: return "inflated size differs from ISIZE";
	case INF_E_INPUT: return "compressed data ends early";
	case INF_E_CRC: return "CRC mismatch";
	}
	return "?";
}

} // namespace

// ---- the BGZF inflate stage (bamdev.h) ----
bool bgzf_walk(const uint8_t *file, size_t file_len, std::vector<BgzfMember> &members, std::vector<size_t> &member_at, size_t &total, std::string &why)
{
	total = 0;
	for (size_t at = 0; at < file_len;) {
		if (file_len - at < 18) { why = "truncated BGZF header"; return false; }
		const uint8_t *h = file + at;
		if (h[0] != 0x1f || h[1] != 0x8b || h[2] != 8 || !(h[3] & 4)) { why = "not a BGZF file (is it BAM? CRAM is not supported)"; return false; }
		const unsigned xlen = h16(h + 10);
		if (file_len - at < 12 + (size_t)xlen) { why = "truncated BGZF extra field"; return false; }
		int bsize = -1;
		for (unsigned x = 0; x + 4 <= xlen;) {
			const uint8_t *e = h + 12 + x; const unsigned slen = h16(e + 2);
			if (e[0] == 'B' && e[1] == 'C' && slen == 2) bsize = h16(e + 4);
			x += 4 + slen;
		}
		if (bsize < 0) { why = "BGZF block without BC subfield"; return false; }
		const size_t csize = (size_t)bsize + 1;
		if (csize < 12 + (size_t)xlen + 8 || file_len - at < csize) { why = "truncated BGZF block"; return false; }
		const uint32_t usize = h32(h + csize - 4);
		if (usize > 65536) { why = "BGZF block larger than 64 KiB"; return false; }
		BgzfMember M; M.in_off = at + 12 + xlen; M.in_len = (uint32_t)(csize - 12 - xlen - 8); M.out_off = total; M.out_len = usize; M.crc = h32(h + csize - 8); M.pad = 0;
		members.push_back(M); member_at.push_back(at);
		total += usize; at += csize;
	}
	return true;
}

cudaError_t bgzf_inflate_chunks(cudaStream_t st, int n_sm, const uint8_t *file, size_t file_len, const std::vector<BgzfMember> &members, uint8_t *d_comp,
                                const BgzfMember *d_members, uint8_t *d_out, unsigned long long *d_err, unsigned *d_next, uint32_t *n_chunks)
{
	// The file goes up in chunks of whole members and every chunk's members are inflated as soon as they have arrived, on one of four
	// streams: the copy of chunk k+1 (a staged copy when the caller's buffer is pageable) overlaps the kernels of chunks k, k-1, ...
	// One member is a serial chain of ~9 ms whatever the chunk's size, so consecutive chunks' kernels have to share the SMs.
	constexpr int NS = 4; constexpr size_t CHUNK = 32u << 20;
	cudaStream_t ks[NS] = {}; cudaEvent_t ce[64] = {}, ke[NS] = {};
	cudaError_t e_ = cudaSuccess;
	for (int k = 0; k < NS && e_ == cudaSuccess; ++k) { e_ = cudaStreamCreateWithFlags(&ks[k], cudaStreamNonBlocking); if (e_ == cudaSuccess) e_ = cudaEventCreateWithFlags(&ke[k], cudaEventDisableTiming); }
	if (e_ == cudaSuccess) e_ = cudaEventCreateWithFlags(&ce[0], cudaEventDisableTiming);
	if (e_ == cudaSuccess) e_ = cudaEventRecord(ce[0], st);   // the member table, the cleared counters
	size_t m0 = 0, byte0 = 0; int chunk = 0;
	while (m0 < members.size() && e_ == cudaSuccess) {
		size_t m1 = m0, byte1 = byte0;
		while (m1 < members.size() && (m1 == m0 || members[m1].in_off + members[m1].in_len + 8 - byte0 <= CHUNK)) { byte1 = (size_t)(members[m1].in_off + members[m1].in_len + 8); ++m1; }
		if (chunk >= 62) { m1 = members.size(); byte1 = file_len; }   // (a file of more than 2 GB: the rest as one chunk)
		const int c = chunk + 1;
		e_ = cudaMemcpyAsync(d_comp + byte0, file + byte0, byte1 - byte0, cudaMemcpyHostToDevice, st);
		if (e_ == cudaSuccess) e_ = cudaEventCreateWithFlags(&ce[c], cudaEventDisableTiming);
		if (e_ == cudaSuccess) e_ = cudaEventRecord(ce[c], st);
		cudaStream_t k_st = ks[chunk % NS];
		if (e_ == cudaSuccess) e_ = cudaStreamWaitEvent(k_st, ce[c], 0);
		if (e_ == cudaSuccess && chunk < NS) e_ = cudaStreamWaitEvent(k_st, ce[0], 0);
		if (e_ == cudaSuccess) {
			const size_t nm = m1 - m0;
			const unsigned ctas = (unsigned)std::min<size_t>((size_t)n_sm * INF_CTAS_PER_SM, (nm + INF_WARPS - 1) / INF_WARPS);
			bgzf_inflate_kernel<<<ctas, INF_WARPS * 32, 0, k_st>>>(d_comp, d_members, (uint32_t)m0, (uint32_t)m1, d_out, d_err, d_next + c);
			e_ = cudaGetLastError();
		}
		m0 = m1; byte0 = byte1; ++chunk;
	}
	// the call's stream continues when every chunk's kernel is done (the padding behind the file was cleared before the first of them started)
	for (int k = 0; k < NS && e_ == cudaSuccess; ++k) { e_ = cudaEventRecord(ke[k], ks[k]); if (e_ == cudaSuccess) e_ = cudaStreamWaitEvent(st, ke[k], 0); }
	const cudaError_t e_sync = cudaStreamSynchronize(st);
	for (auto &e : ce) if (e) cudaEventDestroy(e);
	for (int k = 0; k < NS; ++k) { if (ke[k]) cudaEventDestroy(ke[k]); if (ks[k]) cudaStreamDestroy(ks[k]); }
	if (e_ != cudaSuccess) return e_;
	if (e_sync != cudaSuccess) return e_sync;
	*n_chunks = (uint32_t)chunk;
	return cudaSuccess;
}

std::string bgzf_error_text(unsigned long long first_error)
{
	char msg[160];
	snprintf(msg, sizeof msg, "BGZF block %llu failed to inflate (corrupt data or CRC mismatch: %s)", first_error >> 8, inf_error_text((int)(first_error & 0xff)));
	return msg;
}

struct idl_bam {
	int device = 0;
	cudaStream_t st = nullptr;
	uint8_t *d_comp = nullptr, *d_out = nullptr;
	size_t total = 0;
	Rec R = {};
	long long *d_rec_off = nullptr;
	unsigned long long *d_cig_off = nullptr; uint32_t *d_cigar = nullptr;
	size_t n_all = 0, n_cigar = 0;
	int32_t *d_ref_len = nullptr;
	const uint8_t **d_ref_seq = nullptr;       // per target: its sequence (ASCII) on the device, or null (idl_bam_set_reference)
	std::vector<const uint8_t*> ref_seq;
	// scratch of the batch builder: four sets used in turn (grown on demand); a set is reused only after the kernels of the batch that used it
	// last are done (`done`, recorded on that batch's stream behind its pack kernels): several batches are in flight on different lanes
	struct ScratchSet { void *p[8] = {}; size_t cap[8] = {}; cudaEvent_t done = nullptr; bool used = false; };
	ScratchSet sets[4]; unsigned next_set = 0;
	std::vector<void*> owned;   // every stream-ordered allocation of this object (cudaMallocAsync on `st` from the device's default pool, which keeps
	                            // freed memory: a process that opens BAM after BAM -- one per target -- saw cudaMalloc / cudaFree of the gigabyte
	                            // buffers take 0.3-0.7 s now and then)
	idl_bam_info info = {};
	std::vector<std::string> names; std::vector<const char*> name_ptrs; std::vector<int64_t> ref_len, ref_first;
	std::string header;
};

extern "C" {

void idl_bam_close(idl_bam *b)
{
	if (!b) return;
	cudaSetDevice(b->device);
	cudaDeviceSynchronize();   // nothing on any stream still reads the buffers
	if (b->st) { for (void *p : b->owned) cudaFreeAsync(p, b->st); cudaStreamSynchronize(b->st); }
	else for (void *p : b->owned) cudaFree(p);
	for (auto &S : b->sets) { for (void *p : S.p) if (p) cudaFree(p); if (S.done) cudaEventDestroy(S.done); }
	for (const uint8_t *p : b->ref_seq) if (p) cudaFree((void*)p);
	if (b->st) cudaStreamDestroy(b->st);
	delete b;
}

const idl_bam_info *idl_bam_get_info(const idl_bam *b) { return b ? &b->info : nullptr; }

static int bam_open_impl(int device, const uint8_t *file, size_t file_len, const idl_bam_slice *slice, idl_bam **out, char *err, size_t errlen);

int idl_bam_open(int device, const uint8_t *file, size_t file_len, idl_bam **out, char *err, size_t errlen)
{
	return bam_open_impl(device, file, file_len, nullptr, out, err, errlen);
}

int idl_bam_open_slice(int device, const uint8_t *members, size_t len, const idl_bam_slice *slice, idl_bam **out, char *err, size_t errlen)
{
	if (!slice || slice->n_ref < 0 || (slice->n_ref && (!slice->ref_name || !slice->ref_len))) return IDL_E_ARG;
	return bam_open_impl(device, members, len, slice, out, err, errlen);
}

static int bam_open_impl(int device, const uint8_t *file, size_t file_len, const idl_bam_slice *slice, idl_bam **out, char *err, size_t errlen)
{
	if (!out || (!file && file_len)) return IDL_E_ARG;
	*out = nullptr;
	const double t_enter = std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
	int ndev = 0;
	if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { set_err(err, errlen, "no CUDA device (idl_bam_open has no CPU path)"); return IDL_E_NO_DEVICE; }
	if (device < 0 || device >= ndev) return IDL_E_ARG;
	// 1. members
	std::vector<Member> members; std::vector<size_t> member_at; size_t total = 0;
	{ std::string why; if (!bgzf_walk(file, file_len, members, member_at, total, why)) { set_err(err, errlen, why); return IDL_E_FORMAT; } }
	if (members.empty() || (!slice && total < 12)) { set_err(err, errlen, "not a BAM file"); return IDL_E_FORMAT; }
	if (members.size() >= (1ull << 32)) return IDL_E_CAPACITY;
	// IDL_BAM_TIMING=1: wall-clock phases of the call on stderr (context creation and allocations are not inside the CUDA events)
	const bool timing = getenv("IDL_BAM_TIMING") != nullptr;
	auto now = []() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
	double tw[8] = {now(), 0, 0, 0, 0, 0, 0, 0};
	if (cudaSetDevice(device) != cudaSuccess) return IDL_E_CUDA;
	cudaFree(nullptr);
	tw[1] = now();
	idl_bam *b = new idl_bam();
	b->device = device; b->total = total;
	int rc = IDL_OK;
	cudaEvent_t ev[4] = {};
	std::string why;
#define BCK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { why = std::string(#call) + ": " + cudaGetErrorString(e_); rc = IDL_E_CUDA; goto done; } } while (0)
#define BALLOC(ptr, bytes) do { void *p_ = nullptr; BCK(cudaMallocAsync(&p_, (bytes) ? (bytes) : 16, b->st)); b->owned.push_back(p_); ptr = (decltype(ptr))p_; } while (0)
#define BFAIL(msg) do { why = (msg); rc = IDL_E_FORMAT; goto done; } while (0)
	{
		int n_sm = 0;
		BCK(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device));
		BCK(cudaStreamCreateWithFlags(&b->st, cudaStreamNonBlocking));
		cudaStream_t st = b->st;
		{
			cudaMemPool_t pool;   // freed buffers stay with the pool instead of going back to the driver
			if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) { unsigned long long thr = ~0ULL; cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr); }
		}
		for (auto &e : ev) BCK(cudaEventCreate(&e));
		Member *d_members = nullptr; unsigned long long *d_err = nullptr; unsigned *d_next = nullptr;
		BALLOC(b->d_comp, file_len + 512); BALLOC(b->d_out, total + 64); BALLOC(d_members, members.size() * sizeof(Member)); BALLOC(d_err, 64); BALLOC(d_next, 4 * 64);
		// 2. H2D + inflate
		tw[2] = now();
		BCK(cudaEventRecord(ev[0], st));
		BCK(cudaMemsetAsync(b->d_comp + file_len, 0, 512, st));
		BCK(cudaMemcpyAsync(d_members, members.data(), members.size() * sizeof(Member), cudaMemcpyHostToDevice, st));
		BCK(cudaMemsetAsync(d_err, 0xff, 64, st)); BCK(cudaMemsetAsync(d_next, 0, 4 * 64, st)); BCK(cudaMemsetAsync(b->d_out + total, 0, 64, st));
		BCK(cudaEventRecord(ev[1], st));
		{
			const cudaError_t e_ = bgzf_inflate_chunks(st, n_sm, file, file_len, members, b->d_comp, d_members, b->d_out, d_err, d_next, &b->info.n_chunks);
			if (e_ != cudaSuccess) { why = std::string("inflate: ") + cudaGetErrorString(e_); rc = IDL_E_CUDA; goto done; }
		}
		BCK(cudaEventRecord(ev[2], st));
		unsigned long long herr[8];
		BCK(cudaMemcpyAsync(herr, d_err, 64, cudaMemcpyDeviceToHost, st));
		// header: magic, l_text, text, n_ref, (l_name, name, l_ref) per target
		std::vector<uint8_t> head(std::min<size_t>(total, 1u << 20));
		BCK(cudaMemcpyAsync(head.data(), b->d_out, head.size(), cudaMemcpyDeviceToHost, st));
		BCK(cudaStreamSynchronize(st));
		tw[3] = now();
		if (herr[0] != ~0ULL) BFAIL(bgzf_error_text(herr[0]));
		uint32_t n_ref = 0; std::vector<int32_t> ref_len32; size_t begin = 0, rec_total = total;
		if (!slice) {
			if (memcmp(head.data(), "BAM\1", 4) != 0) BFAIL("not a BAM file");
			size_t at = 4;
			const uint32_t l_text = h32(head.data() + at); at += 4;
			auto need = [&](size_t upto) -> bool {   // make head[0..upto) available
				if (upto > total) return false;
				if (upto <= head.size()) return true;
				const size_t old = head.size(); head.resize(std::min(total, std::max(upto, old * 2)));
				return cudaMemcpy(head.data() + old, b->d_out + old, head.size() - old, cudaMemcpyDeviceToHost) == cudaSuccess;
			};
			if (!need(at + (size_t)l_text + 4)) BFAIL("truncated BAM header");
			b->header.assign((const char*)head.data() + at, l_text); at += l_text;
			n_ref = h32(head.data() + at); at += 4;
			if (n_ref > (1u << 24)) BFAIL("truncated BAM reference list");
			for (uint32_t r = 0; r < n_ref; ++r) {
				if (!need(at + 4)) BFAIL("truncated BAM reference list");
				const uint32_t l_name = h32(head.data() + at); at += 4;
				if (l_name == 0 || !need(at + (size_t)l_name + 4)) BFAIL("truncated BAM reference list");
				b->names.emplace_back((const char*)head.data() + at, l_name - 1); at += l_name;
				const uint32_t l_ref = h32(head.data() + at); at += 4;
				b->ref_len.push_back((int64_t)l_ref); ref_len32.push_back((int32_t)std::min<uint32_t>(l_ref, INT_MAX));
			}
			begin = at;   // the first alignment record
		} else {
			// a run of members from the middle of a file (one target's records, found through the index): the header comes from the caller, the
			// records start at first_record and end at end_offset bytes into the member that starts end_member bytes into the run
			n_ref = (uint32_t)slice->n_ref;
			for (uint32_t r = 0; r < n_ref; ++r) {
				b->names.emplace_back(slice->ref_name[r]); b->ref_len.push_back(slice->ref_len[r]);
				ref_len32.push_back((int32_t)std::min<int64_t>(std::max<int64_t>(slice->ref_len[r], 0), INT_MAX));
			}
			begin = (size_t)slice->first_record;
			if (slice->end_member == file_len && slice->end_offset == 0) rec_total = total;
			else {
				const auto it = std::lower_bound(member_at.begin(), member_at.end(), (size_t)slice->end_member);
				if (it == member_at.end() || *it != (size_t)slice->end_member) BFAIL("the slice's end does not lie on a BGZF member of the run");
				const Member &M = members[(size_t)(it - member_at.begin())];
				if (slice->end_offset > M.out_len) BFAIL("the slice's end lies outside its member");
				rec_total = (size_t)M.out_off + (size_t)slice->end_offset;
			}
			if (begin > rec_total) BFAIL("the slice's first record lies behind its end");
		}
		// 3. record boundaries
		const size_t span = rec_total - begin;
		const uint32_t n_seg = (uint32_t)((span + SEG_BYTES - 1) / SEG_BYTES);
		int32_t *&d_ref_len = b->d_ref_len; long long *d_first = nullptr, *d_exit = nullptr, *d_preset = nullptr; uint32_t *d_count = nullptr, *d_bad = nullptr, *d_which = nullptr;
		unsigned long long *d_rec_base = nullptr;
		BALLOC(d_ref_len, (size_t)n_ref * 4); BALLOC(b->d_ref_seq, (size_t)n_ref * 8); BCK(cudaMemsetAsync(b->d_ref_seq, 0, (size_t)n_ref * 8 + (n_ref ? 0 : 16), st)); b->ref_seq.assign(n_ref, nullptr); BALLOC(d_first, (size_t)n_seg * 8); BALLOC(d_exit, (size_t)n_seg * 8); BALLOC(d_preset, (size_t)n_seg * 8);
		BALLOC(d_count, (size_t)n_seg * 4); BALLOC(d_bad, (size_t)n_seg * 4); BALLOC(d_which, (size_t)n_seg * 4); BALLOC(d_rec_base, (size_t)n_seg * 8 + 8);
		if (n_ref) BCK(cudaMemcpyAsync(d_ref_len, ref_len32.data(), (size_t)n_ref * 4, cudaMemcpyHostToDevice, st));
		std::vector<long long> first(n_seg), exitv(n_seg), preset(n_seg, -2);
		std::vector<uint32_t> count(n_seg), bad(n_seg);
		size_t n_all = 0;
		if (n_seg) {
			preset[0] = (long long)begin;
			BCK(cudaMemcpyAsync(d_preset, preset.data(), (size_t)n_seg * 8, cudaMemcpyHostToDevice, st));
			bam_seg_kernel<<<(n_seg * 32 + 255) / 256, 256, 0, st>>>(b->d_out, rec_total, begin, n_seg, nullptr, 0, (int32_t)n_ref, d_ref_len, d_preset, d_first, d_exit, d_count, d_bad);
			BCK(cudaGetLastError());
			auto fetch = [&]() -> cudaError_t {
				cudaError_t e = cudaMemcpyAsync(first.data(), d_first, (size_t)n_seg * 8, cudaMemcpyDeviceToHost, st);
				if (e == cudaSuccess) e = cudaMemcpyAsync(exitv.data(), d_exit, (size_t)n_seg * 8, cudaMemcpyDeviceToHost, st);
				if (e == cudaSuccess) e = cudaMemcpyAsync(count.data(), d_count, (size_t)n_seg * 4, cudaMemcpyDeviceToHost, st);
				if (e == cudaSuccess) e = cudaMemcpyAsync(bad.data(), d_bad, (size_t)n_seg * 4, cudaMemcpyDeviceToHost, st);
				if (e == cudaSuccess) e = cudaStreamSynchronize(st);
				return e;
			};
			BCK(fetch());
			// the chain: `expect` = offset of the next record on the true chain.  Segments are visited in order; one whose first record is not
			// `expect` is walked again from there (one small launch each; guesses are almost never wrong)
			size_t expect = begin;
			for (uint32_t k = 0; k < n_seg; ++k) {
				const size_t s0 = begin + (size_t)k * SEG_BYTES, s1 = std::min(rec_total, s0 + SEG_BYTES);
				const long long want = expect < s1 ? (long long)expect : -1;   // -1: a record spans the whole segment
				if (first[k] != want) {
					++b->info.boundary_fixups;
					preset[k] = want;
					const uint32_t which = k;
					BCK(cudaMemcpyAsync(d_preset + k, &preset[k], 8, cudaMemcpyHostToDevice, st));
					BCK(cudaMemcpyAsync(d_which, &which, 4, cudaMemcpyHostToDevice, st));
					bam_seg_kernel<<<1, 32, 0, st>>>(b->d_out, rec_total, begin, n_seg, d_which, 1, (int32_t)n_ref, d_ref_len, d_preset, d_first, d_exit, d_count, d_bad);
					BCK(cudaGetLastError());
					BCK(cudaMemcpyAsync(&first[k], d_first + k, 8, cudaMemcpyDeviceToHost, st)); BCK(cudaMemcpyAsync(&exitv[k], d_exit + k, 8, cudaMemcpyDeviceToHost, st));
					BCK(cudaMemcpyAsync(&count[k], d_count + k, 4, cudaMemcpyDeviceToHost, st)); BCK(cudaMemcpyAsync(&bad[k], d_bad + k, 4, cudaMemcpyDeviceToHost, st));
					BCK(cudaStreamSynchronize(st));
				}
				if (want >= 0) {
					if (bad[k]) BFAIL("truncated BAM record");
					expect = (size_t)exitv[k];
				}
				n_all += count[k];
			}
			if (expect != rec_total) BFAIL("truncated BAM record");
		}
		tw[4] = now();
		if (n_all >= (1ull << 31)) { rc = IDL_E_CAPACITY; why = "more than 2^31 records"; goto done; }
		b->n_all = n_all;
		// 4. offsets and fields
		{
			std::vector<unsigned long long> rec_base(n_seg + 1, 0);
			for (uint32_t k = 0; k < n_seg; ++k) rec_base[k + 1] = rec_base[k] + count[k];
			BCK(cudaMemcpyAsync(d_rec_base, rec_base.data(), ((size_t)n_seg + 1) * 8, cudaMemcpyHostToDevice, st));
			BALLOC(b->d_rec_off, n_all * 8);
			BALLOC(b->R.ref_id, n_all * 4); BALLOC(b->R.pos, n_all * 4); BALLOC(b->R.stop, n_all * 4); BALLOC(b->R.l_seq, n_all * 4); BALLOC(b->R.mapq, n_all);
			BALLOC(b->R.flag, n_all * 2); BALLOC(b->R.n_cig, n_all * 4 + 4); BALLOC(b->R.cig_at, n_all * 8); BALLOC(b->R.seq_at, n_all * 8);
			BALLOC(b->d_cig_off, (n_all + 1) * 8);
			long long *d_ref_first = nullptr; unsigned long long *d_tot = nullptr;
			const size_t nt = std::max<size_t>(1, (n_all + 1 + SCAN_TILE - 1) / SCAN_TILE);
			BALLOC(d_ref_first, ((size_t)n_ref + 1) * 8); BALLOC(d_tot, nt * 8);
			BCK(cudaMemsetAsync(d_err, 0xff, 64, st));
			if (n_all) {
				bam_offsets_kernel<<<(n_seg * 32 + 255) / 256, 256, 0, st>>>(b->d_out, rec_total, begin, n_seg, d_first, d_rec_base, b->d_rec_off);
				bam_fields_kernel<<<(unsigned)((n_all + 255) / 256), 256, 0, st>>>(b->d_out, b->d_rec_off, n_all, (int32_t)n_ref, b->R, d_err);
				bam_order_kernel<<<(unsigned)((n_all + 255) / 256), 256, 0, st>>>(b->R.ref_id, b->R.pos, n_all, d_err + 1, d_err + 2);
			}
			// 5. CIGARs as one array
			scan_tile_totals_kernel<<<(unsigned)nt, SCAN_THREADS, 0, st>>>(b->R.n_cig, n_all, d_tot);
			scan_totals_kernel<<<1, 1024, 0, st>>>(d_tot, nt);
			scan_apply_kernel<<<(unsigned)nt, SCAN_THREADS, 0, st>>>(b->R.n_cig, n_all, d_tot, b->d_cig_off);
			BCK(cudaGetLastError());
			unsigned long long n_cigar = 0;
			BCK(cudaMemcpyAsync(&n_cigar, b->d_cig_off + n_all, 8, cudaMemcpyDeviceToHost, st));
			BCK(cudaMemcpyAsync(herr, d_err, 64, cudaMemcpyDeviceToHost, st));
			BCK(cudaStreamSynchronize(st));
			if (herr[0] != ~0ULL) {
				// the host reader's two messages for a record that contradicts itself (bamio.cpp idlh_load)
				BFAIL("malformed BAM record or BAM record with an unknown reference id (record " + std::to_string(herr[0]) + ")");
			}
			const size_t n_placed = herr[2] == ~0ULL ? n_all : (size_t)herr[2];
			if (herr[1] != ~0ULL) {
				if (herr[1] < n_placed) BFAIL("BAM is not coordinate sorted");
				BFAIL("BAM records with a target follow records without one (unplaced records are only supported as the tail of the file)");
			}
			b->n_cigar = (size_t)n_cigar;
			BALLOC(b->d_cigar, (size_t)n_cigar * 4);
			if (n_all) bam_cigar_gather_kernel<<<(unsigned)((n_all + 255) / 256), 256, 0, st>>>(b->d_out, b->R.cig_at, b->d_cig_off, n_all, b->d_cigar);
			b->ref_first.assign((size_t)n_ref + 1, 0);
			bam_ref_first_kernel<<<(n_ref + 1 + 255) / 256, 256, 0, st>>>(b->R.ref_id, n_placed, (int32_t)n_ref, d_ref_first);
			BCK(cudaGetLastError());
			BCK(cudaMemcpyAsync(b->ref_first.data(), d_ref_first, ((size_t)n_ref + 1) * 8, cudaMemcpyDeviceToHost, st));
			BCK(cudaEventRecord(ev[3], st));
			BCK(cudaStreamSynchronize(st));
			b->info.n_records = (int64_t)n_placed; b->info.n_unplaced = (int64_t)(n_all - n_placed);
		}
		cudaEventElapsedTime(&b->info.ms_h2d, ev[0], ev[1]); cudaEventElapsedTime(&b->info.ms_inflate, ev[1], ev[2]); cudaEventElapsedTime(&b->info.ms_parse, ev[2], ev[3]);
		b->info.file_bytes = file_len; b->info.inflated_bytes = total; b->info.n_members = (uint32_t)members.size(); b->info.n_ref = (int32_t)n_ref;
		for (auto &s : b->names) b->name_ptrs.push_back(s.c_str());
		b->info.ref_name = b->name_ptrs.data(); b->info.ref_len = b->ref_len.data(); b->info.ref_first = b->ref_first.data();
		b->info.header_text = b->header.c_str(); b->info.header_len = b->header.size();
		// the compressed bytes are not needed any more: the resident footprint is the inflated stream + ~60 bytes per record
		for (auto it = b->owned.begin(); it != b->owned.end(); ++it) if (*it == (void*)b->d_comp) { b->owned.erase(it); break; }
		cudaFreeAsync(b->d_comp, st); b->d_comp = nullptr;
		tw[5] = now();
		if (timing)
			fprintf(stderr, "idl_bam_open: member index %.1f ms, context %.1f ms, stream + allocations %.1f ms, h2d + inflate + header %.1f ms, boundaries %.1f ms, fields + cigars %.1f ms\n",
			        (tw[0] - t_enter) * 1e3, (tw[1] - tw[0]) * 1e3, (tw[2] - tw[1]) * 1e3, (tw[3] - tw[2]) * 1e3, (tw[4] - tw[3]) * 1e3, (tw[5] - tw[4]) * 1e3);
	}
done:
	for (auto &e : ev) if (e) cudaEventDestroy(e);
	if (rc != IDL_OK) { set_err(err, errlen, why); idl_bam_close(b); return rc; }
	*out = b;
	return IDL_OK;
#undef BFAIL
}

// idl_bam_sweep (n_iv < 0: the whole target) and idl_bam_sweep_window
static int bam_sweep(idl_bam *b, int32_t target, int64_t zone_lo, int64_t zone_hi, long long n_iv, const int32_t *iv_beg, const int32_t *iv_end,
                     int32_t min_event_support, int32_t min_read_coverage, int32_t max_read_coverage, uint32_t flags, idl_sweep_out **out)
{
	if (!b || !out || target < 0 || target >= b->info.n_ref) return IDL_E_ARG;
	const size_t r0 = (size_t)b->ref_first[(size_t)target], r1 = (size_t)b->ref_first[(size_t)target + 1];
	if (b->ref_len[(size_t)target] > INT_MAX) return IDL_E_CAPACITY;
	if (n_iv < 0) zone_hi = b->ref_len[(size_t)target];
	if (zone_lo < 0 || zone_hi < zone_lo || zone_hi > b->ref_len[(size_t)target]) return IDL_E_ARG;
	if (r1 == r0 && !(flags & IDL_SWEEP_EVIDENCE)) {
		// a target without records has no regions (a header with thousands of alt / decoy contigs): nothing to launch
		idl_sweep_out *o = (idl_sweep_out*)calloc(1, sizeof *o);
		if (!o) return IDL_E_NOMEM;
		o->roi_start = (int32_t*)malloc(16); o->roi_end = (int32_t*)malloc(16); o->roi_read_begin = (int64_t*)malloc(16); o->roi_n_reads = (int32_t*)malloc(16);
		o->read_idx = (int64_t*)malloc(16);
		*out = o;
		return IDL_OK;
	}
	idl_sweep_in in; memset(&in, 0, sizeof in);
	in.chrom_len = (int32_t)b->ref_len[(size_t)target]; in.n_reads = r1 - r0;
	in.start = b->R.pos + r0; in.stop = b->R.stop + r0; in.flag = b->R.flag + r0; in.cigar = b->d_cigar; in.cig_off = (const uint64_t*)(b->d_cig_off + r0);
	if (cudaStreamSynchronize(b->st) != cudaSuccess) return IDL_E_CUDA;
	const int rc = idl_sweep_impl(b->device, &in, true, 0, (int32_t)zone_lo, (int32_t)zone_hi, n_iv, iv_beg, iv_end, min_event_support, min_read_coverage, max_read_coverage,
	                              flags, out);
	if (rc != IDL_OK) return rc;
	for (size_t k = 0; k < (*out)->n_read_idx; ++k) (*out)->read_idx[k] += (int64_t)r0;
	return IDL_OK;
}

int idl_bam_sweep(idl_bam *b, int32_t target, int32_t min_event_support, int32_t min_read_coverage, int32_t max_read_coverage, uint32_t flags, idl_sweep_out **out)
{
	return bam_sweep(b, target, 0, 0, -1, nullptr, nullptr, min_event_support, min_read_coverage, max_read_coverage, flags, out);
}

int idl_bam_sweep_window(idl_bam *b, int32_t target, int32_t zone_lo, int32_t zone_hi, size_t n_iv, const int32_t *iv_beg, const int32_t *iv_end,
                         int32_t min_event_support, int32_t min_read_coverage, int32_t max_read_coverage, uint32_t flags, idl_sweep_out **out)
{
	if (n_iv >= (1ull << 31)) return IDL_E_CAPACITY;
	return bam_sweep(b, target, zone_lo, zone_hi, (long long)n_iv, iv_beg, iv_end, min_event_support, min_read_coverage, max_read_coverage, flags, out);
}

void idl_bam_reads_free(idl_bam_reads *r)
{
	if (!r) return;
	free(r->chrom); free(r->start); free(r->stop); free(r->len); free(r->mapq); free(r->flag); free(r->seq_off); free(r->bases); free(r->quals); free(r->cig_off); free(r->cigar);
	free(r);
}

int idl_bam_fetch(idl_bam *b, size_t n, const int64_t *idx, uint32_t what, idl_bam_reads **out)
{
	if (!b || !out) return IDL_E_ARG;
	*out = nullptr;
	const size_t n_rec = (size_t)b->info.n_records;
	if (!idx && n > n_rec) return IDL_E_ARG;
	if (idx) for (size_t j = 0; j < n; ++j) if (idx[j] < 0 || (size_t)idx[j] >= n_rec) return IDL_E_ARG;
	if (cudaSetDevice(b->device) != cudaSuccess) return IDL_E_CUDA;
	idl_bam_reads *r = (idl_bam_reads*)calloc(1, sizeof *r);
	if (!r) return IDL_E_NOMEM;
	r->n = n;
	int rc = IDL_OK;
	cudaStream_t st = b->st;
	std::vector<void*> tmp;
	cudaEvent_t ev[3] = {};
	std::vector<uint32_t> ncig(n);
#undef BCK
#define BCK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { fprintf(stderr, "idl_bam_fetch: %s: %s\n", #call, cudaGetErrorString(e_)); rc = IDL_E_CUDA; goto done; } } while (0)
#define TALLOC(ptr, bytes) do { void *p_ = nullptr; BCK(cudaMalloc(&p_, (bytes) ? (bytes) : 16)); tmp.push_back(p_); ptr = (decltype(ptr))p_; } while (0)
#define HALLOC(ptr, bytes) do { ptr = (decltype(ptr))malloc((bytes) ? (bytes) : 16); if (!ptr) { rc = IDL_E_NOMEM; goto done; } } while (0)
	{
		for (auto &e : ev) BCK(cudaEventCreate(&e));
		long long *d_idx = nullptr; int32_t *d_chrom, *d_start, *d_stop, *d_len; uint8_t *d_mapq; uint16_t *d_flag; uint32_t *d_ncig;
		TALLOC(d_chrom, n * 4); TALLOC(d_start, n * 4); TALLOC(d_stop, n * 4); TALLOC(d_len, n * 4); TALLOC(d_mapq, n); TALLOC(d_flag, n * 2); TALLOC(d_ncig, n * 4);
		if (idx) { TALLOC(d_idx, n * 8); BCK(cudaMemcpyAsync(d_idx, idx, n * 8, cudaMemcpyHostToDevice, st)); }
		HALLOC(r->chrom, n * 4); HALLOC(r->start, n * 4); HALLOC(r->stop, n * 4); HALLOC(r->len, n * 4); HALLOC(r->mapq, n); HALLOC(r->flag, n * 2);
		BCK(cudaEventRecord(ev[0], st));
		if (n) bam_fetch_fields_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_idx, n, b->R, d_chrom, d_start, d_stop, d_len, d_mapq, d_flag, d_ncig);
		BCK(cudaGetLastError());
		BCK(cudaMemcpyAsync(r->chrom, d_chrom, n * 4, cudaMemcpyDeviceToHost, st)); BCK(cudaMemcpyAsync(r->start, d_start, n * 4, cudaMemcpyDeviceToHost, st));
		BCK(cudaMemcpyAsync(r->stop, d_stop, n * 4, cudaMemcpyDeviceToHost, st)); BCK(cudaMemcpyAsync(r->len, d_len, n * 4, cudaMemcpyDeviceToHost, st));
		BCK(cudaMemcpyAsync(r->mapq, d_mapq, n, cudaMemcpyDeviceToHost, st)); BCK(cudaMemcpyAsync(r->flag, d_flag, n * 2, cudaMemcpyDeviceToHost, st));
		BCK(cudaMemcpyAsync(ncig.data(), d_ncig, n * 4, cudaMemcpyDeviceToHost, st));
		BCK(cudaStreamSynchronize(st));
		float ms_k = 0, ms_d = 0;
		if (what & IDL_BAM_SEQ) {
			HALLOC(r->seq_off, (n + 1) * 8);
			r->seq_off[0] = 0;
			for (size_t j = 0; j < n; ++j) r->seq_off[j + 1] = r->seq_off[j] + r->len[j];
			const size_t nb = (size_t)r->seq_off[n];
			long long *d_soff; uint8_t *d_b, *d_q;
			TALLOC(d_soff, (n + 1) * 8); TALLOC(d_b, nb); TALLOC(d_q, nb);
			HALLOC(r->bases, nb); HALLOC(r->quals, nb);
			BCK(cudaMemcpyAsync(d_soff, r->seq_off, (n + 1) * 8, cudaMemcpyHostToDevice, st));
			BCK(cudaEventRecord(ev[0], st));
			if (n) bam_fetch_seq_kernel<<<(unsigned)((n * 32 + 255) / 256), 256, 0, st>>>(b->d_out, d_idx, n, b->R, d_soff, d_b, d_q);
			BCK(cudaGetLastError());
			BCK(cudaEventRecord(ev[1], st));
			BCK(cudaMemcpyAsync(r->bases, d_b, nb, cudaMemcpyDeviceToHost, st)); BCK(cudaMemcpyAsync(r->quals, d_q, nb, cudaMemcpyDeviceToHost, st));
			BCK(cudaEventRecord(ev[2], st));
			BCK(cudaStreamSynchronize(st));
			float a = 0, c = 0; cudaEventElapsedTime(&a, ev[0], ev[1]); cudaEventElapsedTime(&c, ev[1], ev[2]); ms_k += a; ms_d += c;
		}
		if (what & IDL_BAM_CIGAR) {
			HALLOC(r->cig_off, (n + 1) * 8);
			r->cig_off[0] = 0;
			for (size_t j = 0; j < n; ++j) r->cig_off[j + 1] = r->cig_off[j] + ncig[j];
			const size_t nc = (size_t)r->cig_off[n];
			unsigned long long *d_coff; uint32_t *d_c;
			TALLOC(d_coff, (n + 1) * 8); TALLOC(d_c, nc * 4);
			HALLOC(r->cigar, nc * 4);
			BCK(cudaMemcpyAsync(d_coff, r->cig_off, (n + 1) * 8, cudaMemcpyHostToDevice, st));
			BCK(cudaEventRecord(ev[0], st));
			if (n) bam_fetch_cigar_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_idx, n, b->d_cig_off, b->d_cigar, d_coff, d_c);
			BCK(cudaGetLastError());
			BCK(cudaEventRecord(ev[1], st));
			BCK(cudaMemcpyAsync(r->cigar, d_c, nc * 4, cudaMemcpyDeviceToHost, st));
			BCK(cudaEventRecord(ev[2], st));
			BCK(cudaStreamSynchronize(st));
			float a = 0, c = 0; cudaEventElapsedTime(&a, ev[0], ev[1]); cudaEventElapsedTime(&c, ev[1], ev[2]); ms_k += a; ms_d += c;
		}
		r->ms_kernels = ms_k; r->ms_d2h = ms_d;
	}
done:
	for (void *p : tmp) cudaFree(p);
	for (auto &e : ev) if (e) cudaEventDestroy(e);
	if (rc != IDL_OK) { idl_bam_reads_free(r); return rc; }
	*out = r;
	return IDL_OK;
}

} // extern "C"

// ---- batch builder entry points (bamdev.h) ----
namespace {
template <class T> cudaError_t scratch_get(idl_bam::ScratchSet &S, int slot, size_t count, T **out)
{
	const size_t bytes = std::max<size_t>(count * sizeof(T), 16);
	if (S.cap[slot] < bytes) {
		if (S.p[slot]) cudaFree(S.p[slot]);
		S.p[slot] = nullptr; S.cap[slot] = 0;
		const cudaError_t e = cudaMalloc(&S.p[slot], bytes + bytes / 4);
		if (e != cudaSuccess) return e;
		S.cap[slot] = bytes + bytes / 4;
	}
	*out = (T*)S.p[slot];
	return cudaSuccess;
}
} // namespace

cudaError_t scan_u32(const uint32_t *in, size_t n, unsigned long long *out, unsigned long long *tot, cudaStream_t st)
{
	const size_t nt = std::max<size_t>(1, (n + 1 + SCAN_TILE - 1) / SCAN_TILE);
	scan_tile_totals_kernel<<<(unsigned)nt, SCAN_THREADS, 0, st>>>(in, n, tot);
	scan_totals_kernel<<<1, 1024, 0, st>>>(tot, nt);
	scan_apply_kernel<<<(unsigned)nt, SCAN_THREADS, 0, st>>>(in, n, tot, out);
	return cudaGetLastError();
}

int bam_device_of(const idl_bam *b) { return b ? b->device : -1; }

int bam_batch_records(idl_bam *b, cudaStream_t st, const idl_params *P, size_t n_regions, const int32_t *roi_chrom, const int32_t *roi_start, const int32_t *roi_end,
                      const int32_t *roi_n_reads, const int64_t *read_idx, size_t n_reads, uint32_t ordinal_base, idl_region *d_region, idl_read *d_read, BamBatchTotals *T)
{
#define QCK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { fprintf(stderr, "idl_bam batch: %s: %s\n", #call, cudaGetErrorString(e_)); return IDL_E_CUDA; } } while (0)
	memset(T, 0, sizeof *T);
	T->scratch_set = b->next_set++ % 4u;
	idl_bam::ScratchSet &S = b->sets[T->scratch_set];
	if (!S.done) QCK(cudaEventCreateWithFlags(&S.done, cudaEventDisableTiming));
	if (S.used) QCK(cudaEventSynchronize(S.done));   // the batch that used this set last has consumed it
	S.used = true;
	QCK(cudaEventRecord(S.done, st));               // (re-recorded behind the pack kernels in bam_batch_bases; this covers an early return)
	// scratch: 0 roi arrays (4 x int32), 1 read_idx, 2 read_pad + slot_region, 3 ref_pad, 4 scans (n_reads + 1 + n_regions + 1 + tile totals), 5 roi_read_begin + counters
	int32_t *d_roi; long long *d_idx; uint32_t *d_rp; uint32_t *d_refpad; unsigned long long *d_scan; unsigned long long *d_rb;
	QCK(scratch_get(S, 0, 4 * n_regions, &d_roi)); QCK(scratch_get(S, 1, n_reads, &d_idx)); QCK(scratch_get(S, 2, 2 * n_reads + 2, &d_rp));
	QCK(scratch_get(S, 3, n_regions + 1, &d_refpad));
	const size_t nt = (std::max(n_reads, n_regions) + 1 + SCAN_TILE - 1) / SCAN_TILE + 1;
	QCK(scratch_get(S, 4, n_reads + 1 + n_regions + 1 + nt, &d_scan)); QCK(scratch_get(S, 5, n_regions + 1 + 8, &d_rb));
	std::vector<unsigned long long> rb(n_regions + 1, 0);
	for (size_t k = 0; k < n_regions; ++k) { if (roi_n_reads[k] < 0) return IDL_E_ARG; rb[k + 1] = rb[k] + (unsigned long long)roi_n_reads[k]; }
	if (rb[n_regions] != n_reads) return IDL_E_ARG;
	BuildCounters *d_cnt = (BuildCounters*)(d_rb + n_regions + 1);
	uint32_t *d_slot_region = d_rp + n_reads + 1;
	if (n_regions) {
		QCK(cudaMemcpyAsync(d_roi, roi_chrom, n_regions * 4, cudaMemcpyHostToDevice, st)); QCK(cudaMemcpyAsync(d_roi + n_regions, roi_start, n_regions * 4, cudaMemcpyHostToDevice, st));
		QCK(cudaMemcpyAsync(d_roi + 2 * n_regions, roi_end, n_regions * 4, cudaMemcpyHostToDevice, st));
		QCK(cudaMemcpyAsync(d_roi + 3 * n_regions, roi_n_reads, n_regions * 4, cudaMemcpyHostToDevice, st));
	}
	if (n_reads) QCK(cudaMemcpyAsync(d_idx, read_idx, n_reads * 8, cudaMemcpyHostToDevice, st));
	QCK(cudaMemcpyAsync(d_rb, rb.data(), (n_regions + 1) * 8, cudaMemcpyHostToDevice, st));
	QCK(cudaMemsetAsync(d_cnt, 0, sizeof(BuildCounters), st));
	if (n_regions)
		bam_build_records_kernel<<<(unsigned)((n_regions * 32 + 255) / 256), 256, 0, st>>>(b->d_out, b->R, (size_t)b->info.n_records, b->d_ref_len, b->d_ref_seq, b->info.n_ref, *P, n_regions,
		                                                                                  d_roi, d_roi + n_regions, d_roi + 2 * n_regions, d_roi + 3 * n_regions, d_rb, d_idx, ordinal_base,
		                                                                                  d_region, d_read, d_rp, d_slot_region, d_refpad, d_cnt);
	unsigned long long *d_soff = d_scan, *d_roff = d_scan + n_reads + 1, *d_tot = d_roff + n_regions + 1;
	QCK(scan_u32(d_rp, n_reads, d_soff, d_tot, st));
	QCK(scan_u32(d_refpad, n_regions, d_roff, d_tot, st));
	const size_t nmax = std::max(n_reads, n_regions);
	if (nmax) bam_build_offsets_kernel<<<(unsigned)((nmax + 255) / 256), 256, 0, st>>>(n_reads, n_regions, d_soff, d_roff, d_read, d_region);
	QCK(cudaGetLastError());
	BuildCounters hc; unsigned long long tot[2] = {0, 0};
	QCK(cudaMemcpyAsync(&hc, d_cnt, sizeof hc, cudaMemcpyDeviceToHost, st));
	QCK(cudaMemcpyAsync(&tot[0], d_soff + n_reads, 8, cudaMemcpyDeviceToHost, st)); QCK(cudaMemcpyAsync(&tot[1], d_roff + n_regions, 8, cudaMemcpyDeviceToHost, st));
	QCK(cudaStreamSynchronize(st));
	T->n_seq_bases = tot[0]; T->n_ref_bases = tot[1];
	T->max_trim_len = std::max(1u, hc.max_trim_len); T->max_ref_len = hc.max_ref_len; T->max_region_reads = hc.max_region_reads; T->n_small_regions = hc.n_small_regions;
	T->bad_index = hc.bad_index;
	return IDL_OK;
}

int bam_batch_bases(idl_bam *b, cudaStream_t st, size_t n_regions, size_t n_reads, idl_region *d_region, const idl_read *d_read, const BamBatchTotals *T,
                    uint32_t *seq2, uint32_t *seqn, uint32_t *ref2, uint32_t *refn)
{
	idl_bam::ScratchSet &S = b->sets[T->scratch_set & 3u];
	const long long *d_idx = (const long long*)S.p[1];
	const uint32_t *d_slot_region = (const uint32_t*)S.p[2] + n_reads + 1;
	if (n_reads) bam_pack_reads_kernel<<<(unsigned)((n_reads * 32 + 255) / 256), 256, 0, st>>>(b->d_out, b->R, d_idx, n_reads, d_read, d_slot_region, d_region, seq2, seqn);
	if (n_regions) bam_pack_ref_kernel<<<(unsigned)((n_regions * 32 + 255) / 256), 256, 0, st>>>(b->d_ref_seq, n_regions, d_region, ref2, refn);
	QCK(cudaGetLastError());
	// guard words behind the pools (the kernels read up to two words past a record)
	QCK(cudaMemsetAsync(seq2 + T->n_seq_bases / 16, 0, 16, st)); QCK(cudaMemsetAsync(seqn + T->n_seq_bases / 32, 0, 16, st));
	QCK(cudaMemsetAsync(ref2 + T->n_ref_bases / 16, 0, 16, st)); QCK(cudaMemsetAsync(refn + T->n_ref_bases / 32, 0, 16, st));
	QCK(cudaEventRecord(S.done, st));
	return IDL_OK;
#undef QCK
}

extern "C" int idl_bam_set_reference(idl_bam *b, int32_t target, const uint8_t *seq, int64_t len)
{
	if (!b || target < 0 || target >= b->info.n_ref || !seq || len != b->ref_len[(size_t)target]) return IDL_E_ARG;
	if (cudaSetDevice(b->device) != cudaSuccess) return IDL_E_CUDA;
	if (b->ref_seq[(size_t)target]) return IDL_OK;
	uint8_t *d = nullptr;
	if (cudaMalloc((void**)&d, (size_t)len + 64) != cudaSuccess) return IDL_E_NOMEM;
	if (cudaMemcpyAsync(d, seq, (size_t)len, cudaMemcpyHostToDevice, b->st) != cudaSuccess || cudaMemsetAsync(d + len, 0, 64, b->st) != cudaSuccess ||
	    cudaMemcpyAsync(b->d_ref_seq + target, &d, 8, cudaMemcpyHostToDevice, b->st) != cudaSuccess || cudaStreamSynchronize(b->st) != cudaSuccess) { cudaFree(d); return IDL_E_CUDA; }
	b->ref_seq[(size_t)target] = d;
	return IDL_OK;
}

extern "C" int idl_bam_set_reference_fasta(idl_bam *b, int32_t target, const idl_fasta *fa, int64_t record)
{
	const uint8_t *src = nullptr; int64_t len = 0; int dev = -1;
	if (!b || target < 0 || target >= b->info.n_ref || fasta_record_on_device(fa, record, &src, &len, &dev) != IDL_OK) return IDL_E_ARG;
	if (dev != b->device || len != b->ref_len[(size_t)target]) return IDL_E_ARG;
	if (cudaSetDevice(b->device) != cudaSuccess) return IDL_E_CUDA;
	if (b->ref_seq[(size_t)target]) return IDL_OK;
	uint8_t *d = nullptr;
	if (cudaMalloc((void**)&d, (size_t)len + 64) != cudaSuccess) return IDL_E_NOMEM;
	if (cudaMemcpyAsync(d, src, (size_t)len, cudaMemcpyDeviceToDevice, b->st) != cudaSuccess || cudaMemsetAsync(d + len, 0, 64, b->st) != cudaSuccess ||
	    cudaMemcpyAsync(b->d_ref_seq + target, &d, 8, cudaMemcpyHostToDevice, b->st) != cudaSuccess || cudaStreamSynchronize(b->st) != cudaSuccess) { cudaFree(d); return IDL_E_CUDA; }
	b->ref_seq[(size_t)target] = d;
	return IDL_OK;
}
