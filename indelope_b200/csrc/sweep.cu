// indelope_b200/csrc/sweep.cu -- SURVEY.md 8(f)4: the evidence array and the extraction of regions of interest on the GPU.
//
// Replaces, for one target (chromosome), the body of gen_roi (src/indelope.nim:515-545) with gen_roi_internal (:461-499),
// event_locations (:430-442), overlaps (:449-452) and skippable (:40-47): from the coordinate-sorted records of the target (start, stop,
// flag, CIGAR) to the list of regions (roi_start, roi_end) with, for every region, the records that overlap it, in BAM order.
//
// The reference sweeps the records once, keeps a cache of the current coverage-connected chunk and, at every coverage gap, scans the
// chunk's part of a saturating uint8 evidence array for runs >= min_event_support.  Three observations make it data-parallel without
// changing a single region (DESIGN.md "evidence and regions on the GPU" has the proofs):
//   1. the evidence counters are order independent: every event interval [es, ee) adds +1 / -1 to a difference array, one prefix sum
//      gives the counts, min(count, 255) is the saturating add of :541-543;
//   2. a chunk boundary only matters as a CUT of a run of evidence at the start of the record that opens a new chunk, and a record
//      opens a chunk exactly when its start lies beyond the stops of ALL non-skippable records before it (a prefix maximum); cutting
//      at such a record while the cache is empty (the reference does not) falls into evidence-free ground or on the same position;
//   3. the records of a region are all non-skippable records that overlap it -- records of other chunks cannot -- and the 600-record
//      cap of :480-486 drops a region exactly when more than max_reads overlap it.
// So: (A) one thread per record marks events and stops, (B) a prefix maximum over the records marks the cuts, (C) a prefix sum over the
// positions writes the reference's evidence bytes, (D) runs are counted and written in position order, (E) one warp per run finds its
// records by two binary searches (prefix maximum of the stops, starts) and a ballot compaction.  Every pass streams its arrays once with
// 128-bit loads: the stage is HBM-bound (bench: tools/sweep_bench.py reports GB/s against the measured copy bandwidth).
#include <algorithm>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cuda_runtime.h>
#include "indelope_cuda.h"
#include "sweep_impl.h"

namespace {

constexpr int SW_THREADS = 256;
constexpr int SW_ITEMS = 16;                       // elements per thread and pass
constexpr int SW_TILE = SW_THREADS * SW_ITEMS;     // elements per CTA

__device__ __forceinline__ bool sw_skippable(uint16_t f) { return (f & 0x400) || (f & 0x200) || (f & 0x4) || (f & 0x800) || (f & 0x100); } // :40-47

// (A) one thread per record: event intervals into the difference array (event_locations :430-442; every op but M is an event, the
// ones that do not consume the reference are one base wide), stop of a non-skippable record for the prefix maximum.  The position arrays cover the
// zone [zone_lo, zone_hi] only (index = position - zone_lo): a record that starts before the zone or ends behind it is clipped to it before it
// addresses `diff` -- the usual case for a zone cut out of a target, not an edge case
__global__ void sw_mark_kernel(size_t n, const int32_t *start, const int32_t *stop, const uint16_t *flag, const uint32_t *cigar, const unsigned long long *cig_off,
                               int32_t zone_lo, int32_t zone_hi, int *diff, int32_t *stopv)
{
	const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	if (sw_skippable(flag[i])) { stopv[i] = INT_MIN; return; }
	stopv[i] = stop[i];
	long long off = 0;
	const long long s = start[i];
	for (unsigned long long k = cig_off[i]; k < cig_off[i + 1]; ++k) {
		const uint32_t c = cigar[k], op = c & 0xf, len = c >> 4;
		const bool cons = op == 0 || op == 2 || op == 3 || op == 7 || op == 8;
		if (op != 0) {
			const long long es = s + off; long long ee = cons ? es + len : es + 1;
			if (ee > (long long)zone_hi + 1) ee = (long long)zone_hi + 1;   // evidence has tlen + 1 entries (:522); the zone ends at zone_hi <= tlen
			if (es >= 0) {
				const long long a = es > zone_lo ? es : zone_lo;
				if (a < ee) { atomicAdd(diff + (a - zone_lo), 1); atomicAdd(diff + (ee - zone_lo), -1); }
			}
		}
		if (cons) off += len;
	}
}

// ---- three-phase scans over int32 (sum or max): per-CTA totals, a scan of the totals by one CTA, the apply pass of the caller ----
template <bool MAX> __device__ __forceinline__ int sw_op(int a, int b) { return MAX ? (a > b ? a : b) : a + b; }
template <bool MAX> __device__ __forceinline__ int sw_id() { return MAX ? INT_MIN : 0; }

template <bool MAX> __device__ __forceinline__ int sw_block_reduce(int v, int *sh)
{
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
	for (int d = 16; d >= 1; d >>= 1) v = sw_op<MAX>(v, __shfl_xor_sync(0xffffffffu, v, d));
	if (lane == 0) sh[warp] = v;
	__syncthreads();
	int r = sw_id<MAX>();
	for (int w = 0; w < SW_THREADS / 32; ++w) r = sw_op<MAX>(r, sh[w]);
	__syncthreads();
	return r;
}
// exclusive scan of the threads' values inside a CTA; returns the thread's exclusive prefix, *total = the CTA's total
template <bool MAX> __device__ __forceinline__ int sw_block_scan(int v, int *sh, int *total)
{
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	int inc = v;
#pragma unroll
	for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc = sw_op<MAX>(inc, o); }
	if (lane == 31) sh[warp] = inc;
	__syncthreads();
	int before = sw_id<MAX>(), tot = sw_id<MAX>();
	for (int w = 0; w < SW_THREADS / 32; ++w) { if (w < warp) before = sw_op<MAX>(before, sh[w]); tot = sw_op<MAX>(tot, sh[w]); }
	__syncthreads();
	const int excl_in_warp = __shfl_up_sync(0xffffffffu, inc, 1);
	*total = tot;
	return sw_op<MAX>(before, lane ? excl_in_warp : sw_id<MAX>());
}

template <bool MAX> __global__ void __launch_bounds__(SW_THREADS) sw_totals_kernel(const int *in, size_t n, int *totals)
{
	__shared__ int sh[SW_THREADS / 32];
	const size_t base = (size_t)blockIdx.x * SW_TILE + (size_t)threadIdx.x * SW_ITEMS;
	int acc = sw_id<MAX>();
	if (base + SW_ITEMS <= n) {
		const int4 *p = (const int4*)(in + base);
#pragma unroll
		for (int q = 0; q < SW_ITEMS / 4; ++q) { const int4 v = p[q]; acc = sw_op<MAX>(acc, sw_op<MAX>(sw_op<MAX>(v.x, v.y), sw_op<MAX>(v.z, v.w))); }
	} else for (int k = 0; k < SW_ITEMS; ++k) if (base + k < n) acc = sw_op<MAX>(acc, in[base + k]);
	const int t = sw_block_reduce<MAX>(acc, sh);
	if (threadIdx.x == 0) totals[blockIdx.x] = t;
}
// exclusive scan of up to a few hundred thousand totals by ONE CTA of 32 warps (in place); *grand = the total of everything.  Every warp owns
// a contiguous chunk and walks it 32 elements at a time with coalesced loads and a shuffle scan: one pass for its total, one scan of the 32
// warp totals, one pass to write.  (A 256-wide block scan looped over the array took 0.3 ms per call on the 60 k totals of a 248 Mb contig,
// a contiguous chunk per THREAD -- uncoalesced, 60 dependent loads -- 54 us.)
constexpr int SW_SCAN_THREADS = 1024;
template <bool MAX> __global__ void __launch_bounds__(SW_SCAN_THREADS) sw_scan_totals_kernel(int *totals, size_t n, int *grand)
{
	__shared__ int sh[SW_SCAN_THREADS / 32];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const size_t per = ((n + 31) / 32 + 31) / 32 * 32, lo = (size_t)warp * per, hi = lo + per < n ? lo + per : n;
	int acc = sw_id<MAX>();
	for (size_t i = lo + lane; i < hi; i += 32) acc = sw_op<MAX>(acc, totals[i]);
#pragma unroll
	for (int d = 16; d >= 1; d >>= 1) acc = sw_op<MAX>(acc, __shfl_xor_sync(0xffffffffu, acc, d));
	if (lane == 0) sh[warp] = acc;
	__syncthreads();
	int carry = sw_id<MAX>(), tot = sw_id<MAX>();
	for (int w = 0; w < SW_SCAN_THREADS / 32; ++w) { if (w < warp) carry = sw_op<MAX>(carry, sh[w]); tot = sw_op<MAX>(tot, sh[w]); }
	for (size_t i0 = lo; i0 < hi; i0 += 32) {
		const size_t i = i0 + lane;
		const int v = i < hi ? totals[i] : sw_id<MAX>();
		int inc = v;
#pragma unroll
		for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc = sw_op<MAX>(inc, o); }
		const int ex = __shfl_up_sync(0xffffffffu, inc, 1);
		if (i < hi) totals[i] = sw_op<MAX>(carry, lane ? ex : sw_id<MAX>());
		carry = sw_op<MAX>(carry, __shfl_sync(0xffffffffu, inc, 31));
	}
	if (threadIdx.x == 0 && grand) *grand = tot;
}

// (B) apply pass of the prefix maximum over the records: pm[i] = max(stopv[0..i]) and the cuts: a record whose start lies beyond every
// non-skippable stop before it opens a new chunk (:529), runs of evidence are cut at its start (cuts outside the zone are not stored)
__global__ void __launch_bounds__(SW_THREADS) sw_prefmax_apply_kernel(const int32_t *stopv, const int32_t *start, size_t n, const int *totals, int32_t *pm, uint8_t *cut,
                                                                      int32_t zone_lo, int32_t zone_hi)
{
	__shared__ int sh[SW_THREADS / 32];
	const size_t base = (size_t)blockIdx.x * SW_TILE + (size_t)threadIdx.x * SW_ITEMS;
	int v[SW_ITEMS]; int acc = INT_MIN;
#pragma unroll
	for (int k = 0; k < SW_ITEMS; ++k) { v[k] = base + k < n ? stopv[base + k] : INT_MIN; acc = max(acc, v[k]); }
	int tot;
	int run = max(totals[blockIdx.x], sw_block_scan<true>(acc, sh, &tot)); // max over everything before my first record
#pragma unroll
	for (int k = 0; k < SW_ITEMS; ++k) {
		if (base + k < n) {
			const int32_t s = start[base + k];
			if (s > run && s >= zone_lo && s <= zone_hi) cut[s - zone_lo] = 1;
			run = max(run, v[k]);
			pm[base + k] = run;
		}
	}
}

// (C) apply pass of the prefix sum over the positions: the reference's evidence bytes (saturating at 255, :541-543)
__global__ void __launch_bounds__(SW_THREADS) sw_evidence_kernel(const int *diff, size_t n, const int *totals, uint8_t *ev)
{
	__shared__ int sh[SW_THREADS / 32];
	const size_t base = (size_t)blockIdx.x * SW_TILE + (size_t)threadIdx.x * SW_ITEMS;
	int v[SW_ITEMS]; int acc = 0;
	if (base + SW_ITEMS <= n) {
		const int4 *p = (const int4*)(diff + base);
#pragma unroll
		for (int q = 0; q < SW_ITEMS / 4; ++q) { const int4 x = p[q]; v[4 * q] = x.x; v[4 * q + 1] = x.y; v[4 * q + 2] = x.z; v[4 * q + 3] = x.w; }
	} else {
#pragma unroll
		for (int k = 0; k < SW_ITEMS; ++k) v[k] = base + k < n ? diff[base + k] : 0;
	}
#pragma unroll
	for (int k = 0; k < SW_ITEMS; ++k) acc += v[k];
	int tot;
	int run = totals[blockIdx.x] + sw_block_scan<false>(acc, sh, &tot);
	uint32_t out[SW_ITEMS / 4];
#pragma unroll
	for (int k = 0; k < SW_ITEMS; ++k) {
		run += v[k];
		const uint32_t b = run > 255 ? 255u : (run < 0 ? 0u : (uint32_t)run);
		if ((k & 3) == 0) out[k >> 2] = b; else out[k >> 2] |= b << (8 * (k & 3));
	}
	if (base + SW_ITEMS <= n) *(uint4*)(ev + base) = make_uint4(out[0], out[1], out[2], out[3]);
	else for (int k = 0; k < SW_ITEMS; ++k) if (base + k < n) ev[base + k] = (uint8_t)(out[k >> 2] >> (8 * (k & 3)));
}

// (D) runs of evidence >= min_evidence, cut at chunk boundaries (gen_roi_internal :468-476).  WRITE = false counts the run starts and
// run ends of every CTA; WRITE = true writes them in position order at the scanned offsets (the k-th start and the k-th end are one run).
template <bool WRITE>
__global__ void __launch_bounds__(SW_THREADS) sw_runs_kernel(const uint8_t *ev, const uint8_t *cut, size_t n, int min_ev, int *cnt_start, int *cnt_end,
                                                             int32_t *run_start, int32_t *run_end)
{
	__shared__ int sh[SW_THREADS / 32];
	const size_t base = (size_t)blockIdx.x * SW_TILE + (size_t)threadIdx.x * SW_ITEMS;
	uint8_t e[SW_ITEMS + 2], c[SW_ITEMS + 1];   // e[0] = ev[base - 1], e[k + 1] = ev[base + k], e[ITEMS + 1] = ev[base + ITEMS]; c[k] = cut[base + k]
	e[0] = base > 0 && base - 1 < n ? ev[base - 1] : 0;
	if (base + SW_ITEMS <= n) {
		const uint4 x = *(const uint4*)(ev + base), y = *(const uint4*)(cut + base);
		const uint32_t xs[4] = {x.x, x.y, x.z, x.w}, ys[4] = {y.x, y.y, y.z, y.w};
#pragma unroll
		for (int k = 0; k < SW_ITEMS; ++k) { e[k + 1] = (uint8_t)(xs[k >> 2] >> (8 * (k & 3))); c[k] = (uint8_t)(ys[k >> 2] >> (8 * (k & 3))); }
	} else {
#pragma unroll
		for (int k = 0; k < SW_ITEMS; ++k) { e[k + 1] = base + k < n ? ev[base + k] : 0; c[k] = base + k < n ? cut[base + k] : 0; }
	}
	e[SW_ITEMS + 1] = base + SW_ITEMS < n ? ev[base + SW_ITEMS] : 0;
	c[SW_ITEMS] = base + SW_ITEMS < n ? cut[base + SW_ITEMS] : 0;
	unsigned ms = 0, me = 0;
#pragma unroll
	for (int k = 0; k < SW_ITEMS; ++k) {
		const bool f = e[k + 1] >= min_ev;
		if (f && (e[k] < min_ev || c[k])) ms |= 1u << k;            // a run starts here
		if (f && (e[k + 2] < min_ev || c[k + 1])) me |= 1u << k;    // ... and ends here
	}
	int tot_s, tot_e;
	const int ex_s = sw_block_scan<false>(__popc(ms), sh, &tot_s);
	const int ex_e = sw_block_scan<false>(__popc(me), sh, &tot_e);
	if (!WRITE) {
		if (threadIdx.x == 0) { cnt_start[blockIdx.x] = tot_s; cnt_end[blockIdx.x] = tot_e; }
	} else {
		int os = cnt_start[blockIdx.x] + ex_s, oe = cnt_end[blockIdx.x] + ex_e;
		while (ms) { const int k = __ffs(ms) - 1; ms &= ms - 1; run_start[os++] = (int32_t)(base + k); }
		while (me) { const int k = __ffs(me) - 1; me &= me - 1; run_end[oe++] = (int32_t)(base + k); }
	}
}

// (E) one warp per run: the records that overlap it (overlaps :449-452), in order.  Candidates: from the first record whose prefix
// maximum of stops reaches roi_start (nothing before it can overlap) to the first record that starts beyond roi_end (:485).
// WRITE = false: count; a run is a region iff min_reads <= count <= max_reads (:486).  WRITE = true: the lists of the regions.
// Runs are positions relative to zone_lo.  With a selection (sel.n_iv >= 0) only runs that overlap one of the sorted, disjoint intervals
// [iv_beg, iv_end) are regions, and a selected run that touches an edge of the zone that is not the target's (rs == edge_lo, re == edge_hi) is
// not one either: it is counted in n_edge[0] / n_edge[1], because evidence beyond the zone may extend it.
struct SwSelect { int n_iv; const int32_t *iv_beg, *iv_end; int32_t edge_lo, edge_hi; unsigned long long *n_edge; };
template <bool WRITE>
__global__ void __launch_bounds__(SW_THREADS) sw_reads_kernel(const int32_t *run_start, const int32_t *run_end, int n_runs, int32_t zone_lo, SwSelect sel,
                                                              const int32_t *start, const int32_t *stopv,
                                                              const int32_t *pm, size_t n_reads, int min_reads, int max_reads, int *count, const int *slot,
                                                              const int *read_off, int32_t *roi_start, int32_t *roi_end, long long *roi_read_begin,
                                                              int32_t *roi_n_reads, long long *read_idx)
{
	const int warp = (int)(((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
	if (warp >= n_runs) return;
	const int32_t rs = run_start[warp] + zone_lo, re = run_end[warp] + zone_lo;
	if (!WRITE && sel.n_iv >= 0) {
		int a = 0, b = sel.n_iv;                                     // the last interval with iv_beg <= re
		while (a < b) { const int mid = (a + b) >> 1; if (sel.iv_beg[mid] <= re) a = mid + 1; else b = mid; }
		const bool picked = a > 0 && sel.iv_end[a - 1] > rs;
		const bool lo_edge = rs == sel.edge_lo, hi_edge = re == sel.edge_hi;
		if (!picked || lo_edge || hi_edge) {
			if (lane == 0) {
				count[warp] = 0;
				if (picked && lo_edge) atomicAdd(sel.n_edge, 1ull);
				if (picked && hi_edge) atomicAdd(sel.n_edge + 1, 1ull);
			}
			return;
		}
	}
	size_t lo = 0, hi = n_reads;                                   // first i with pm[i] >= rs
	while (lo < hi) { const size_t mid = (lo + hi) >> 1; if (pm[mid] >= rs) hi = mid; else lo = mid + 1; }
	const size_t first = lo;
	lo = first; hi = n_reads;                                      // first i with start[i] > re
	while (lo < hi) { const size_t mid = (lo + hi) >> 1; if (start[mid] > re) hi = mid; else lo = mid + 1; }
	const size_t last = lo;
	if (!WRITE) {
		int c = 0;
		for (size_t i = first + lane; i < last && c <= max_reads; i += 32) c += stopv[i] >= rs;  // stopv = INT_MIN for skippable records
		// (every lane stops once ITS count exceeds the cap; the sum is then over the cap as well)
#pragma unroll
		for (int d = 16; d >= 1; d >>= 1) c += __shfl_xor_sync(0xffffffffu, c, d);
		if (lane == 0) count[warp] = (c >= min_reads && c <= max_reads) ? c : 0;
	} else {
		const int c = count[warp];
		if (c == 0) return;
		const int k = slot[warp]; long long o = read_off[warp];
		if (lane == 0) { roi_start[k] = rs; roi_end[k] = re; roi_read_begin[k] = o; roi_n_reads[k] = c; }
		for (size_t i0 = first; i0 < last; i0 += 32) {
			const size_t i = i0 + lane;
			const bool hit = i < last && stopv[i] >= rs;
			const unsigned m = __ballot_sync(0xffffffffu, hit);
			if (hit) read_idx[o + __popc(m & ((1u << lane) - 1u))] = (long long)i;
			o += __popc(m);
		}
	}
}
// flags of accepted runs -> (region slot, first read slot): two exclusive scans over the runs, fused
__global__ void __launch_bounds__(SW_THREADS) sw_accept_kernel(const int *count, int n_runs, int *is_roi, int *reads)
{
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i < n_runs) { is_roi[i] = count[i] > 0; reads[i] = count[i]; }
}
__global__ void __launch_bounds__(SW_THREADS) sw_apply_sum_kernel(int *v, size_t n, const int *totals)
{
	__shared__ int sh[SW_THREADS / 32];
	const size_t base = (size_t)blockIdx.x * SW_TILE + (size_t)threadIdx.x * SW_ITEMS;
	int x[SW_ITEMS]; int acc = 0;
#pragma unroll
	for (int k = 0; k < SW_ITEMS; ++k) { x[k] = base + k < n ? v[base + k] : 0; acc += x[k]; }
	int tot;
	int run = totals[blockIdx.x] + sw_block_scan<false>(acc, sh, &tot);
#pragma unroll
	for (int k = 0; k < SW_ITEMS; ++k) if (base + k < n) { const int t = x[k]; v[base + k] = run; run += t; } // exclusive
}

// stream-ordered allocations from the device's default pool (kept warm: the release threshold is raised on first use), so that the ten
// buffers whose sizes are only known in the middle of the call do not cost a cudaMalloc each (they were half of the first version's 2.4 ms)
struct Dev {
	void *p = nullptr; cudaStream_t st = nullptr;
	~Dev() { if (p) { if (st) cudaFreeAsync(p, st); else cudaFree(p); } }
	cudaError_t get(size_t bytes, cudaStream_t s) { st = s; return cudaMallocAsync(&p, bytes ? bytes : 16, s); }
	template <class T> T *as() { return (T*)p; }
};

size_t tiles(size_t n) { return (n + SW_TILE - 1) / SW_TILE; }

// exclusive prefix sum of v[0..n) in place; *d_grand = the total (device)
void exclusive_sum(int *v, size_t n, int *totals, int *d_grand, cudaStream_t st)
{
	const size_t nt = std::max<size_t>(1, tiles(n));
	sw_totals_kernel<false><<<(unsigned)nt, SW_THREADS, 0, st>>>(v, n, totals);
	sw_scan_totals_kernel<false><<<1, SW_SCAN_THREADS, 0, st>>>(totals, nt, d_grand);
	sw_apply_sum_kernel<<<(unsigned)nt, SW_THREADS, 0, st>>>(v, n, totals);
}

} // namespace

extern "C" {

void idl_sweep_free(idl_sweep_out *o)
{
	if (!o) return;
	free(o->roi_start); free(o->roi_end); free(o->roi_read_begin); free(o->roi_n_reads); free(o->read_idx); free(o->evidence);
	free(o);
}

int idl_sweep(int device, const idl_sweep_in *in, int32_t min_event_support, int32_t min_read_coverage, int32_t max_read_coverage, uint32_t flags, idl_sweep_out **out)
{
	if (!in || !out) return IDL_E_ARG;
	return idl_sweep_impl(device, in, false, in->n_reads && in->cig_off ? (size_t)in->cig_off[in->n_reads] : 0, 0, in->chrom_len, -1, nullptr, nullptr,
	                      min_event_support, min_read_coverage, max_read_coverage, flags, out);
}

} // extern "C"

// the body of idl_sweep; with dev_in the arrays of `in` already live on `device` (idl_bam_sweep: records parsed there by bamdev.cu)
int idl_sweep_impl(int device, const idl_sweep_in *in, bool dev_in, size_t n_cig, int32_t zone_lo, int32_t zone_hi, long long n_iv, const int32_t *iv_beg,
                   const int32_t *iv_end, int32_t min_event_support, int32_t min_read_coverage, int32_t max_read_coverage, uint32_t flags, idl_sweep_out **out)
{
	if (!in || !out || in->chrom_len < 0 || (in->n_reads && (!in->start || !in->stop || !in->flag || !in->cigar || !in->cig_off))) return IDL_E_ARG;
	*out = nullptr;
	if (min_read_coverage < 1 || max_read_coverage < min_read_coverage || min_event_support < 1 || min_event_support > 255) return IDL_E_ARG;
	if (zone_lo < 0 || zone_hi < zone_lo || zone_hi > in->chrom_len) return IDL_E_ARG;
	if (n_iv > 0 && (!iv_beg || !iv_end)) return IDL_E_ARG;
	if (n_iv >= (1ll << 31)) return IDL_E_CAPACITY;
	for (long long k = 0; k < n_iv; ++k)   // sorted and disjoint: the device finds a run's interval by one binary search
		if (iv_beg[k] >= iv_end[k] || (k && iv_beg[k] < iv_end[k - 1])) return IDL_E_ARG;
	int ndev = 0;
	if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) return IDL_E_NO_DEVICE;
	if (device < 0 || device >= ndev) return IDL_E_ARG;
	if (in->n_reads >= (1ull << 31) || (size_t)in->chrom_len + 2 >= (1ull << 31)) return IDL_E_CAPACITY;
	if (cudaSetDevice(device) != cudaSuccess) return IDL_E_CUDA;
	const size_t n = in->n_reads, np = (size_t)(zone_hi - zone_lo) + 2;   // evidence positions zone_lo .. zone_hi (0 .. chrom_len), one more for the closing -1
	const size_t npad = tiles(np) * SW_TILE, nrpad = std::max<size_t>(1, tiles(n)) * SW_TILE;
	idl_sweep_out *o = (idl_sweep_out*)calloc(1, sizeof *o);
	if (!o) return IDL_E_NOMEM;
	cudaStream_t st = nullptr; cudaEvent_t ev[4] = {};
	Dev d_start, d_stop, d_flag, d_cig, d_coff, d_diff, d_stopv, d_pm, d_cut, d_ev, d_tot, d_tot2, d_grand, d_rs, d_re, d_count, d_slot, d_roff, d_o1, d_o2, d_o3, d_o4, d_o5, d_iv, d_edge;
	int rc = IDL_OK;
	SwSelect sel = {-1, nullptr, nullptr, INT_MIN, INT_MAX, nullptr};
#define SWCK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { fprintf(stderr, "idl_sweep: %s: %s\n", #call, cudaGetErrorString(e_)); rc = IDL_E_CUDA; goto done; } } while (0)
	{
		SWCK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
		{
			cudaMemPool_t pool;
			if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) { unsigned long long thr = ~0ULL; cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr); }
		}
		for (auto &e : ev) SWCK(cudaEventCreate(&e));
		if (!dev_in) { SWCK(d_start.get(nrpad * 4, st)); SWCK(d_stop.get(nrpad * 4, st)); SWCK(d_flag.get(nrpad * 2, st)); SWCK(d_cig.get(n_cig * 4 + 16, st)); SWCK(d_coff.get((n + 1) * 8, st)); }
		SWCK(d_diff.get(npad * 4, st)); SWCK(d_stopv.get(nrpad * 4, st)); SWCK(d_pm.get(nrpad * 4, st)); SWCK(d_cut.get(npad + 16, st)); SWCK(d_ev.get(npad + 16, st));
		const size_t ntp = tiles(np), ntr = std::max<size_t>(1, tiles(n));
		SWCK(d_tot.get(std::max(ntp, ntr) * 4, st)); SWCK(d_tot2.get(std::max(ntp, ntr) * 4, st)); SWCK(d_grand.get(16, st));
		if (n_iv >= 0) {
			SWCK(d_iv.get((size_t)n_iv * 8 + 16, st)); SWCK(d_edge.get(16, st));
			sel.n_iv = (int)n_iv; sel.iv_beg = d_iv.as<int32_t>(); sel.iv_end = d_iv.as<int32_t>() + n_iv; sel.n_edge = d_edge.as<unsigned long long>();
			sel.edge_lo = zone_lo > 0 ? zone_lo : INT_MIN; sel.edge_hi = zone_hi < in->chrom_len ? zone_hi : INT_MAX;
			if (n_iv) { SWCK(cudaMemcpyAsync(d_iv.p, iv_beg, (size_t)n_iv * 4, cudaMemcpyHostToDevice, st)); SWCK(cudaMemcpyAsync(d_iv.as<int32_t>() + n_iv, iv_end, (size_t)n_iv * 4, cudaMemcpyHostToDevice, st)); }
			SWCK(cudaMemsetAsync(d_edge.p, 0, 16, st));
		}
		SWCK(cudaEventRecord(ev[0], st));
		if (n && !dev_in) {
			SWCK(cudaMemcpyAsync(d_start.p, in->start, n * 4, cudaMemcpyHostToDevice, st)); SWCK(cudaMemcpyAsync(d_stop.p, in->stop, n * 4, cudaMemcpyHostToDevice, st));
			SWCK(cudaMemcpyAsync(d_flag.p, in->flag, n * 2, cudaMemcpyHostToDevice, st)); SWCK(cudaMemcpyAsync(d_cig.p, in->cigar, n_cig * 4, cudaMemcpyHostToDevice, st));
			SWCK(cudaMemcpyAsync(d_coff.p, in->cig_off, (n + 1) * 8, cudaMemcpyHostToDevice, st));
		}
		SWCK(cudaEventRecord(ev[1], st));
		const int32_t *p_start = dev_in ? in->start : d_start.as<int32_t>(), *p_stop = dev_in ? in->stop : d_stop.as<int32_t>();
		const uint16_t *p_flag = dev_in ? in->flag : d_flag.as<uint16_t>();
		const uint32_t *p_cig = dev_in ? in->cigar : d_cig.as<uint32_t>();
		const unsigned long long *p_coff = dev_in ? (const unsigned long long*)in->cig_off : d_coff.as<unsigned long long>();
		SWCK(cudaMemsetAsync(d_diff.p, 0, npad * 4, st)); SWCK(cudaMemsetAsync(d_cut.p, 0, npad + 16, st));
		int n_runs = 0, n_runs_e = 0;
		if (n) {
			sw_mark_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n, p_start, p_stop, p_flag, p_cig,
			                                                           p_coff, zone_lo, zone_hi, d_diff.as<int>(), d_stopv.as<int32_t>());
			// (B) prefix maximum of the stops, cuts
			sw_totals_kernel<true><<<(unsigned)ntr, SW_THREADS, 0, st>>>(d_stopv.as<int>(), n, d_tot.as<int>());
			sw_scan_totals_kernel<true><<<1, SW_SCAN_THREADS, 0, st>>>(d_tot.as<int>(), ntr, nullptr);
			sw_prefmax_apply_kernel<<<(unsigned)ntr, SW_THREADS, 0, st>>>(d_stopv.as<int32_t>(), p_start, n, d_tot.as<int>(), d_pm.as<int32_t>(), d_cut.as<uint8_t>(), zone_lo, zone_hi);
		}
		// (C) evidence bytes
		sw_totals_kernel<false><<<(unsigned)ntp, SW_THREADS, 0, st>>>(d_diff.as<int>(), np, d_tot.as<int>());
		sw_scan_totals_kernel<false><<<1, SW_SCAN_THREADS, 0, st>>>(d_tot.as<int>(), ntp, nullptr);
		sw_evidence_kernel<<<(unsigned)ntp, SW_THREADS, 0, st>>>(d_diff.as<int>(), np, d_tot.as<int>(), d_ev.as<uint8_t>());
		// (D) runs: count, scan, write.  Positions 0 .. chrom_len (np - 1 entries: the last diff entry only closes intervals)
		sw_runs_kernel<false><<<(unsigned)ntp, SW_THREADS, 0, st>>>(d_ev.as<uint8_t>(), d_cut.as<uint8_t>(), np - 1, min_event_support, d_tot.as<int>(), d_tot2.as<int>(), nullptr, nullptr);
		sw_scan_totals_kernel<false><<<1, SW_SCAN_THREADS, 0, st>>>(d_tot.as<int>(), ntp, d_grand.as<int>());
		sw_scan_totals_kernel<false><<<1, SW_SCAN_THREADS, 0, st>>>(d_tot2.as<int>(), ntp, d_grand.as<int>() + 1);
		{
			int g[2] = {0, 0};
			SWCK(cudaMemcpyAsync(g, d_grand.p, 8, cudaMemcpyDeviceToHost, st)); SWCK(cudaStreamSynchronize(st));
			n_runs = g[0]; n_runs_e = g[1];
		}
		if (n_runs != n_runs_e) { fprintf(stderr, "idl_sweep: %d run starts, %d run ends\n", n_runs, n_runs_e); rc = IDL_E_CUDA; goto done; }
		o->n_runs = (size_t)n_runs;
		int n_rois = 0, n_idx = 0;
		if (n_runs && n) {
			const size_t nrun_pad = tiles((size_t)n_runs) * SW_TILE;
			SWCK(d_rs.get(nrun_pad * 4, st)); SWCK(d_re.get(nrun_pad * 4, st)); SWCK(d_count.get(nrun_pad * 4, st)); SWCK(d_slot.get(nrun_pad * 4, st)); SWCK(d_roff.get(nrun_pad * 4, st));
			sw_runs_kernel<true><<<(unsigned)ntp, SW_THREADS, 0, st>>>(d_ev.as<uint8_t>(), d_cut.as<uint8_t>(), np - 1, min_event_support, d_tot.as<int>(), d_tot2.as<int>(),
			                                                          d_rs.as<int32_t>(), d_re.as<int32_t>());
			// (E) records of every run: count, accept, scan, write
			const unsigned wb = (unsigned)(((size_t)n_runs * 32 + SW_THREADS - 1) / SW_THREADS);
			sw_reads_kernel<false><<<wb, SW_THREADS, 0, st>>>(d_rs.as<int32_t>(), d_re.as<int32_t>(), n_runs, zone_lo, sel, p_start, d_stopv.as<int32_t>(), d_pm.as<int32_t>(), n,
			                                                 min_read_coverage, max_read_coverage, d_count.as<int>(), nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr);
			sw_accept_kernel<<<(unsigned)((n_runs + 255) / 256), 256, 0, st>>>(d_count.as<int>(), n_runs, d_slot.as<int>(), d_roff.as<int>());
			exclusive_sum(d_slot.as<int>(), (size_t)n_runs, d_tot.as<int>(), d_grand.as<int>() + 2, st);
			exclusive_sum(d_roff.as<int>(), (size_t)n_runs, d_tot2.as<int>(), d_grand.as<int>() + 3, st);
			{
				int g[2] = {0, 0};
				SWCK(cudaMemcpyAsync(g, d_grand.as<int>() + 2, 8, cudaMemcpyDeviceToHost, st)); SWCK(cudaStreamSynchronize(st));
				n_rois = g[0]; n_idx = g[1];
			}
			SWCK(d_o1.get((size_t)n_rois * 4 + 16, st)); SWCK(d_o2.get((size_t)n_rois * 4 + 16, st)); SWCK(d_o3.get((size_t)n_rois * 8 + 16, st)); SWCK(d_o4.get((size_t)n_rois * 4 + 16, st));
			SWCK(d_o5.get((size_t)n_idx * 8 + 16, st));
			if (n_rois)
				sw_reads_kernel<true><<<wb, SW_THREADS, 0, st>>>(d_rs.as<int32_t>(), d_re.as<int32_t>(), n_runs, zone_lo, sel, p_start, d_stopv.as<int32_t>(), d_pm.as<int32_t>(), n,
				                                                min_read_coverage, max_read_coverage, d_count.as<int>(), d_slot.as<int>(), d_roff.as<int>(), d_o1.as<int32_t>(),
				                                                d_o2.as<int32_t>(), d_o3.as<long long>(), d_o4.as<int32_t>(), d_o5.as<long long>());
		}
		SWCK(cudaGetLastError());
		SWCK(cudaEventRecord(ev[2], st));
		o->n_rois = (size_t)n_rois; o->n_read_idx = (size_t)n_idx;
		o->roi_start = (int32_t*)malloc((size_t)n_rois * 4 + 16); o->roi_end = (int32_t*)malloc((size_t)n_rois * 4 + 16);
		o->roi_read_begin = (int64_t*)malloc((size_t)n_rois * 8 + 16); o->roi_n_reads = (int32_t*)malloc((size_t)n_rois * 4 + 16);
		o->read_idx = (int64_t*)malloc((size_t)n_idx * 8 + 16);
		if (!o->roi_start || !o->roi_end || !o->roi_read_begin || !o->roi_n_reads || !o->read_idx) { rc = IDL_E_NOMEM; goto done; }
		if (n_rois) {
			SWCK(cudaMemcpyAsync(o->roi_start, d_o1.p, (size_t)n_rois * 4, cudaMemcpyDeviceToHost, st)); SWCK(cudaMemcpyAsync(o->roi_end, d_o2.p, (size_t)n_rois * 4, cudaMemcpyDeviceToHost, st));
			SWCK(cudaMemcpyAsync(o->roi_read_begin, d_o3.p, (size_t)n_rois * 8, cudaMemcpyDeviceToHost, st)); SWCK(cudaMemcpyAsync(o->roi_n_reads, d_o4.p, (size_t)n_rois * 4, cudaMemcpyDeviceToHost, st));
			SWCK(cudaMemcpyAsync(o->read_idx, d_o5.p, (size_t)n_idx * 8, cudaMemcpyDeviceToHost, st));
		}
		if (flags & IDL_SWEEP_EVIDENCE) { // the reference's evidence array itself (parity tests)
			o->evidence = (uint8_t*)malloc(np);
			if (!o->evidence) { rc = IDL_E_NOMEM; goto done; }
			SWCK(cudaMemcpyAsync(o->evidence, d_ev.p, np - 1, cudaMemcpyDeviceToHost, st));
			o->n_evidence = np - 1;
		}
		SWCK(cudaEventRecord(ev[3], st));
		SWCK(cudaStreamSynchronize(st));
		if (sel.n_edge) {
			unsigned long long e2[2] = {0, 0};
			SWCK(cudaMemcpy(e2, d_edge.p, 16, cudaMemcpyDeviceToHost));
			o->n_edge[0] = (size_t)e2[0]; o->n_edge[1] = (size_t)e2[1];
		}
		cudaEventElapsedTime(&o->ms_h2d, ev[0], ev[1]); cudaEventElapsedTime(&o->ms_kernels, ev[1], ev[2]); cudaEventElapsedTime(&o->ms_d2h, ev[2], ev[3]);
		// algorithmic bytes: every record once (start, stop, flag, CIGAR), every position's evidence byte written and read once, the results
		o->algorithmic_bytes = (uint64_t)n * 10 + (uint64_t)n_cig * 4 + (uint64_t)np * 2 + (uint64_t)n_rois * 20 + (uint64_t)n_idx * 8;
		// bytes the passes really stream: memsets (5 B / position), the difference array twice, evidence written once and read twice with the
		// cut bytes, records by (A), (B) twice and the searches of (E)
		o->streamed_bytes = (uint64_t)np * (5 + 8 + 1 + 4) + (uint64_t)n * (10 + 8 + 4 + 12) + (uint64_t)n_cig * 4 + (uint64_t)n_rois * 20 + (uint64_t)n_idx * 8;
	}
done:
	for (Dev *d : {&d_start, &d_stop, &d_flag, &d_cig, &d_coff, &d_diff, &d_stopv, &d_pm, &d_cut, &d_ev, &d_tot, &d_tot2, &d_grand, &d_rs, &d_re, &d_count, &d_slot, &d_roff,
	               &d_o1, &d_o2, &d_o3, &d_o4, &d_o5, &d_iv, &d_edge})
		if (d->p) { cudaFreeAsync(d->p, st); d->p = nullptr; }
	for (auto &e : ev) if (e) cudaEventDestroy(e);
	if (st) { cudaStreamSynchronize(st); cudaStreamDestroy(st); }
	if (rc != IDL_OK) { idl_sweep_free(o); return rc; }
	*out = o;
	return IDL_OK;
#undef SWCK
}
