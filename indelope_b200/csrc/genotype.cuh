// indelope_b200/csrc/genotype.cuh -- the part of callsemble after assembly (src/indelope.nim:208-372):
//
//   sort_*        bucket sort of alignment tasks by estimated anti-diagonals, longest first: the 32/G alignments that
//                 share a warp run in lockstep, so they should have similar lengths
//   align4_kernel call-site A of kernel 2 (contig -> reference window, bw=50 z=400, :213-221) followed, in the same
//                 group, by the glue: truncated CIGAR (src/ksw2/ksw2.nim:22-33), target/query event locations
//                 (:71-91), ref/alt 27-mer selection and rejects (src/indelope.nim:229-281), get_min_flank (:118-132)
//   kmer_kernel   kernel 3: ref/alt canonical 27-mer counting over the reads of the region (:283-311), one CTA per
//                 event, one read per thread, 128-bit loads of the 2-bit packed reads, rolling forward/reverse codes
//   al_prep / al_kernel / al_vote   AL fallback (:312-372): the per-read window tests, call-site B of kernel 2 (two
//                 unbanded alignments per read) and the vote by count_flanked_cigar (:185-199)
#pragma once
#include "common.cuh"
#include "ksw2.cuh"
#include "ksw2_rows.cuh"

#define DP_WARPS 8
#define DP_THREADS (DP_WARPS * 32)
#define KMER_THREADS 128
#define DP_G 8          // threads per alignment
#define DP_NG (32 / DP_G)
#ifndef KSW_UNB_WARPS
#define KSW_UNB_WARPS 5 /* warps per CTA of the unbanded al_kernel.  Measured on the chr1 workload (ms): 8 warps x 2 CTAs at 124 registers
                           22.0, 8 x 3 at 80 24.7, 10 x 2 at 95 21.8, 6 x 3 at 96 21.2, 7 x 3 at 80 21.8, 5 x 4 at 94 21.0, 2 x 10 at 94 21.0:
                           twenty warps at 94 registers */
#endif
#ifndef KSW_UNB_CTAS
#define KSW_UNB_CTAS 4 /* resident CTAs per SM of the unbanded al_kernel */
#endif

struct AlEntry { unsigned event; unsigned base; unsigned n_reads; unsigned pad; };
struct AlItem { unsigned event; unsigned read; int start; int pad; }; // one read of one AL event: two DP tasks (2*i: reference, 2*i+1: contig)


struct GenoArgs {
	const idl_region *region; const idl_read *read;
	const uint32_t *seq2, *seqn;
	const uint8_t *refcodes; const uint8_t *ctg_codes;
	idl_region_result *rres; idl_contig_result *cres; idl_aln_result *ares; idl_event_result *eres; uint32_t *cigar;
	unsigned cap_events, cap_cigar, cap_al, cap_alns, cap_items;
	AlEntry *al_list; AlItem *al_items; int8_t *al_res; // al_res[task] = count_flanked_cigar, or -1 on a DP error
	SortBufs sortA, sortB;
	idl_params P;
	KswParams kpA, kpB; // call-site A (:221) and B (:315-316) scoring, made on the host
	DevCounters *cnt;
	// kernel 2 geometry of this launch (per group) and its global workspaces (one per resident group)
	int ring_cols, seq_cap;
	uint8_t *pmat; size_t p_cap;
	uint32_t *cig_scratch; int cig_cap;
	uint8_t *seq_spill; int seq_spill_cap;  // global-memory sequence staging for alignments that do not fit seq_cap
};

// exclusive scan of the bucket histogram, longest bucket first: one CTA of 1024 threads walks the histogram in 64 coalesced
// chunks of 1024 buckets (all loads issued up front), a shuffle scan per chunk
__global__ void __launch_bounds__(1024) sort_scan_kernel(SortBufs s)
{
	__shared__ unsigned wsum[32];
	constexpr int CH = SORT_BUCKETS / 1024;
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	unsigned v[CH];
#pragma unroll
	for (int c = 0; c < CH; ++c) v[c] = s.hist[SORT_BUCKETS - 1 - (c * 1024 + tid)];
	unsigned carry = 0;
#pragma unroll 1
	for (int c = 0; c < CH; ++c) {
		unsigned x = 0;
#pragma unroll
		for (int k = 0; k < CH; ++k) if (k == c) x = v[k]; // register array, constant indices only
		unsigned inc = x;
#pragma unroll
		for (int d = 1; d < 32; d <<= 1) { const unsigned o = __shfl_up_sync(FULL_MASK, inc, d); if (lane >= d) inc += o; }
		if (lane == 31) wsum[warp] = inc;
		__syncthreads();
		unsigned ws = wsum[lane], wi = ws;
#pragma unroll
		for (int d = 1; d < 32; d <<= 1) { const unsigned o = __shfl_up_sync(FULL_MASK, wi, d); if (lane >= d) wi += o; }
		const unsigned before = __shfl_sync(FULL_MASK, wi - ws, warp), total = __shfl_sync(FULL_MASK, wi, 31);
		const int b = SORT_BUCKETS - 1 - (c * 1024 + tid);
		s.start[b] = carry + before + inc - x; s.cursor[b] = 0;
		carry += total;
		__syncthreads();
	}
}
__global__ void sort_scatter_kernel(SortBufs s, const unsigned *n_ptr, unsigned mul, unsigned cap)
{
	unsigned n = *n_ptr * mul; if (n > cap) n = cap;
	for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
		const unsigned b = s.keys[i];
		s.order[s.start[b] + atomicAdd(&s.cursor[b], 1u)] = i;
	}
}

// sort key of the assembler's queue: the read count of a region
__global__ void region_key_kernel(SortBufs s, const idl_region *region, unsigned n, DevCounters *cnt)
{
	if (blockIdx.x == 0 && threadIdx.x == 0) cnt->n_regions_in = n;
	for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
		const unsigned k = region[i].n_reads < SORT_BUCKETS - 1 ? region[i].n_reads : SORT_BUCKETS - 1;
		s.keys[i] = (uint16_t)k; atomicAdd(&s.hist[k], 1u);
	}
}

// shared/global memory of the group this thread belongs to
template <int G = DP_G>
__device__ __forceinline__ KswMem dp_mem(const GenoArgs &g, unsigned char *smem, int qlen, int tlen, int warps_per_cta = DP_WARPS)
{
	constexpr int NG = 32 / G;
	const int grp = warp_id() * NG + (lane_id() / G);
	const size_t per = ksw_group_smem(g.ring_cols, g.seq_cap);
	const size_t gg = (size_t)blockIdx.x * (warps_per_cta * NG) + grp;
	KswMem m;
	ksw_group_mem(m, smem + per * grp, lane_id() / G, g.ring_cols); m.region_bytes = (int)per;
	if (ksw_seq_bytes(qlen, tlen) <= (size_t)g.seq_cap) m.seq_cap = g.seq_cap;
	else { m.seq = g.seq_spill + gg * (size_t)g.seq_spill_cap; m.seq_cap = g.seq_spill_cap; }
	m.pmat = g.pmat + gg * g.p_cap; m.p_cap = g.p_cap;
	m.cig = g.cig_scratch + gg * (size_t)g.cig_cap; m.cig_cap = g.cig_cap;
	return m;
}

__device__ __forceinline__ unsigned dp_status_bits(int st)
{
	if (st == KSW_ST_CIGCAP) return IDL_RS_CIGAR_OVERFLOW;
	if (st < 0) return IDL_RS_DP_OVERFLOW;
	return 0;
}

// canonical 2-bit code of K codes (declared semantics of kmer.mincode, SURVEY.md appendix D); ~0 if a base is not ACGT
__device__ uint64_t canon_code(const uint8_t *s, int K)
{
	uint64_t f = 0, rc = 0;
	for (int i = 0; i < K; ++i) {
		const unsigned b = s[i];
		if (b > 3) return ~0ULL;
		f = (f << 2) | b;
		rc |= (uint64_t)(3 - b) << (2 * i);
	}
	return f < rc ? f : rc;
}
__device__ __forceinline__ bool same_k(const uint8_t *a, const uint8_t *b, int K)
{
	for (int i = 0; i < K; ++i) if (a[i] != b[i]) return false;
	return true;
}
__device__ __forceinline__ int distinct_k(const uint8_t *a, int K)
{
	unsigned m = 0;
	for (int i = 0; i < K; ++i) m |= 1u << a[i];
	return __popc(m);
}

// ---------------------------------------------------------------------------------------------------------------
// call-site A + glue: one group of G threads per alignment, 32 / G alignments per warp
// ---------------------------------------------------------------------------------------------------------------
template <int G>
__device__ __forceinline__ void align_body(const GenoArgs &g, unsigned char *smem_raw)
{
	constexpr int NG = 32 / G;
	const int lane = lane_id(), gl = lane & (G - 1), grp = lane / G;
	const unsigned gmask = ((1u << G) - 1u) << (lane & ~(G - 1));
	const idl_params &P = g.P;
	const int K = IDL_KMER, width = (K + 1) / 2 - 1; // :218
	const unsigned n_alns = g.cnt->n_alns < g.cap_alns ? g.cnt->n_alns : g.cap_alns;
	for (;;) {
		unsigned base = 0;
		if (lane == 0) base = atomicAdd(&g.cnt->aln_next, (unsigned)NG);
		base = __shfl_sync(FULL_MASK, base, 0);
		if (base >= n_alns) break;
		const bool valid = base + grp < n_alns;
		unsigned ai = 0; idl_aln_result ar; idl_contig_result cr; idl_region R;
		memset(&ar, 0, sizeof ar); memset(&cr, 0, sizeof cr); memset(&R, 0, sizeof R);
		if (valid) { ai = g.sortA.order[base + grp]; ar = g.ares[ai]; cr = g.cres[ar.contig]; R = g.region[ar.region]; }
		const int tlen = ar.ref_len; // window of :213-220, computed when the task was created
		const uint8_t *tq = g.refcodes + R.ref_off + (cr.start - R.ref_start);
		const uint8_t *qq = g.ctg_codes + cr.seq_off;
		KswQuery kq; kq.codes = qq; kq.seq2 = nullptr; kq.seqn = nullptr; kq.base = 0;
		const KswMem M = dp_mem<G>(g, smem_raw, cr.len, tlen, (int)(blockDim.x >> 5));
		KswOut o;
		ksw2_group<G>(valid, cr.len, kq, tlen, tq, g.kpA, M, o);
		if (valid) {
			const uint32_t *cg = M.cig;
			const int n = o.n_cigar;
			int ntr = 0, nev = 0;
			if (gl == 0) {
				ntr = ksw_trunc_count(cg, n, o.max_q);
				for (int k = 0; k < ntr; ++k) nev += (cg[n - 1 - k] & 0xf) != 0;
			}
			ntr = __shfl_sync(gmask, ntr, 0, G); nev = __shfl_sync(gmask, nev, 0, G);
			unsigned coff = 0, eoff = 0;
			const bool want_events = (P.stages & IDL_STAGE_GENOTYPE) && nev >= 1 && nev <= P.max_events; // :229
			if (gl == 0) {
				coff = atomicAdd(&g.cnt->n_cigar_ops, (unsigned)n);
				if (want_events) eoff = atomicAdd(&g.cnt->n_events, (unsigned)nev);
			}
			coff = __shfl_sync(gmask, coff, 0, G); eoff = __shfl_sync(gmask, eoff, 0, G);
			unsigned st = dp_status_bits(o.status);
			if (coff + (unsigned)n > g.cap_cigar) { st |= IDL_RS_CIGAR_OVERFLOW; if (gl == 0) atomicOr(&g.cnt->overflow, 8u); }
			else for (int k = gl; k < n; k += G) g.cigar[coff + k] = cg[n - 1 - k]; // forward order
			bool ev_ok = want_events;
			if (ev_ok && eoff + (unsigned)nev > g.cap_events) { ev_ok = false; if (gl == 0) atomicOr(&g.cnt->overflow, 16u); }
			if (gl == 0) {
				ar.max = o.max; ar.zdropped = o.zdropped; ar.max_q = o.max_q; ar.max_t = o.max_t; ar.mqe = o.mqe; ar.mqe_t = o.mqe_t;
				ar.mte = o.mte; ar.mte_q = o.mte_q; ar.score = o.score; ar.n_cigar = n; ar.n_cigar_trunc = ntr; ar.cigar_off = coff; ar.n_events = nev;
				ar.event_begin = ev_ok ? eoff : IDL_NO_EVENTS; ar.status = st;
				g.ares[ai] = ar;
				if (st) atomicOr(&g.rres[ar.region].status, st);
				atomicAdd(&g.cnt->dp_a, 1ULL); atomicAdd(&g.cnt->dp_cells_a, (unsigned long long)o.cells);
			}
			// ---- glue: thread e of the group handles event e (at most 4)
			if (ev_ok && gl < nev && st) { // slots were handed out before the DP status was known: mark them unusable
				idl_event_result ev; memset(&ev, 0, sizeof ev);
				ev.aln = ai; ev.index = gl; ev.reject = IDL_EV_DP_ERROR; ev.min_flank = -1; ev.amq_median = ev.rmq_median = -1;
				g.eres[eoff + gl] = ev;
			}
			if (ev_ok && gl < nev && !st) {
				idl_event_result ev; memset(&ev, 0, sizeof ev);
				ev.aln = ai; ev.index = gl; ev.min_flank = -1; ev.amq_median = ev.rmq_median = -1; ev.ref_code = ev.alt_code = ~0ULL;
				int toff = 0, qoff = 0, seen = 0; // target_locations / query_locations, src/ksw2/ksw2.nim:71-91
				for (int k = 0; k < ntr; ++k) {
					const uint32_t c = cg[n - 1 - k]; const int op = c & 0xf, len = (int)(c >> 4);
					if (op != 0) {
						if (seen == gl) {
							ev.len = len;
							if (op == 1) { ev.type = 0; ev.t_start = cr.start + toff; ev.t_stop = ev.t_start + 1; ev.q_start = qoff; ev.q_stop = qoff + len; }
							else { ev.type = 1; ev.t_start = cr.start + toff; ev.t_stop = ev.t_start + len; ev.q_start = qoff; ev.q_stop = qoff + 1; }
						}
						++seen;
					}
					if (op != 1) toff += len;
					if (op != 2) qoff += len;
				}
				const int clen = cr.len;
				do {
					if (ev.len < P.min_event_len) { ev.reject = IDL_EV_SHORT; break; } // :234
					int tstart = ev.t_start - cr.start - width; if (tstart < 0) tstart = 0; // :236-238
					if (tstart + K > tlen) tstart = tlen - K;
					ev.tstart = tstart;
					if (tstart < 0) { ev.reject = IDL_EV_WINDOW; break; }
					int off = clen - ev.q_stop - 1; if (ev.q_start < off) off = ev.q_start; // :243
					ev.offset = off;
					int qstart = ev.q_start - width; if (qstart < 0) qstart = 0;              // :244-246
					if (qstart + K > clen) qstart = clen - K;
					ev.qstart = qstart;
					if (qstart < 0) { ev.reject = IDL_EV_WINDOW; break; }
					bool same = same_k(tq + tstart, qq + qstart, K);
					if (same) { // :255-262
						qstart = ev.q_start - 3; if (qstart < 0) qstart = 0;
						if (qstart + K > clen) { int qend = ev.q_stop + 4; if (qend > clen) qend = clen; qstart = qend - K; }
						ev.qstart = qstart;
						if (qstart < 0) { ev.reject = IDL_EV_WINDOW; break; }
						same = same_k(tq + tstart, qq + qstart, K);
					}
					if (same && (ev.q_start == 0 || distinct_k(qq + qstart, K) == 1)) { ev.reject = IDL_EV_SAME_KMER; break; } // :264
					if (distinct_k(tq + tstart, K) < 3) { ev.reject = IDL_EV_LOW_CPLX; break; }                                 // :266
					if (same) { ev.reject = IDL_EV_BUG_SAME; break; }                                                            // :268-275
					ev.ref_code = canon_code(tq + tstart, K); ev.alt_code = canon_code(qq + qstart, K);
					{ // get_min_flank(qloc, ez), :118-132, over the truncated CIGAR
						long long result = 0x7fffffffffffffffLL; bool found = false; int mf = 0;
						for (int k = 0; k < ntr; ++k) {
							const uint32_t c = cg[n - 1 - k]; const int op = c & 0xf; const long long len = c >> 4;
							if (op == 0) {
								result = found ? (len < result ? len : result) : len;
								if (found) { mf = (int)result; break; }
							} else if (op - 1 == ev.type && len == ev.len) {
								if (result == 0x7fffffffffffffffLL) result = 0;
								found = true;
							}
						}
						ev.min_flank = mf;
					}
				} while (0);
				g.eres[eoff + gl] = ev;
			}
		}
		__syncwarp();
	}
}
#ifndef KSW_A4_WARPS
#define KSW_A4_WARPS 4
#endif
#ifndef KSW_A4_CTAS
#define KSW_A4_CTAS 4
#endif
// the shared-memory rings with FOUR threads per alignment, eight alignments per warp in lockstep: the per-diagonal control code (band,
// exact-score bookkeeping, z-drop, block entry) is issued once for eight alignments and the words of a diagonal fill the rounds
// (eight threads per alignment measured 12.9 against 10.1 ms on chr1, DESIGN.md 4.2)
__global__ void __launch_bounds__(32 * KSW_A4_WARPS, KSW_A4_CTAS) align4_kernel(GenoArgs g)
{
	extern __shared__ __align__(16) unsigned char smem_raw[];
	align_body<4>(g, smem_raw);
}

// ---------------------------------------------------------------------------------------------------------------
// kernel 3: k-mer counting (src/indelope.nim:283-311), one WARP per event, the lanes over the windows of one read
//
// A window matches the event's ref (alt) k-mer when its canonical code equals the k-mer's (kmer.mincode / kmer.dists,
// SURVEY appendix D), i.e. when it spells the k-mer or its reverse complement.  The reads are 2-bit packed with base i at
// bits 2i, so the K bases at position p are a 54-bit field of three 32-bit words; with F the event's canonical code
// (first base in the top bits), that field equals  ~F & mask  when the window spells the reverse complement of F's string
// and  pair-reverse(F)  when it spells the string itself.  So a window costs two funnel shifts and four 64-bit compares --
// no rolling state, every window independent.  The first hit per read (:302-309) is the minimum position, found with one
// sub-warp reduction per read; MAPQ medians (:152-155,408-411) come from per-warp histograms.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t kmer_pair_reverse(uint64_t x, int K) // reverse the order of the K 2-bit groups
{
	uint64_t r = __brevll(x);
	r = ((r & 0x5555555555555555ULL) << 1) | ((r >> 1) & 0x5555555555555555ULL);
	return r >> (64 - 2 * K);
}

// first bin where the running count exceeds nn / 2 (median(): sorted[int(len/2)]), all lanes cooperate; -1 for an empty list
__device__ __forceinline__ int kmer_median(const unsigned *h, unsigned nn, int lane)
{
	if (nn == 0) return -1;
	unsigned mine = 0;
#pragma unroll
	for (int q = 0; q < 8; ++q) mine += h[lane * 8 + q];
	unsigned inc = mine;
#pragma unroll
	for (int d = 1; d < 32; d <<= 1) { const unsigned o = __shfl_up_sync(FULL_MASK, inc, d); if (lane >= d) inc += o; }
	const unsigned target = nn / 2;
	const unsigned owner = __ffs(__ballot_sync(FULL_MASK, inc > target)) - 1; // first lane whose bins cross the target
	int med = 0;
	if ((unsigned)lane == owner) {
		unsigned acc = inc - mine;
		for (int q = 0; q < 8; ++q) { acc += h[lane * 8 + q]; if (acc > target) { med = lane * 8 + q; break; } }
	}
	return __shfl_sync(FULL_MASK, med, owner);
}

// Four reads at a time per warp, eight lanes per read, sixteen consecutive windows per lane: a lane loads the three 32-bit
// words (48 bases) and the 64 N-plane bits its windows span once and shifts the fields out of registers, so a read costs
// one round trip for its record and one for its bases, with four reads in flight per warp.
__global__ void __launch_bounds__(KMER_THREADS) kmer_kernel(GenoArgs g)
{
	__shared__ unsigned hist[KMER_THREADS / 32][2][256];
	const int lane = lane_id(), warp = warp_id(), grp = lane >> 3, gl = lane & 7;
	const idl_params &P = g.P;
	const int K = IDL_KMER;
	const uint64_t kmask = (1ULL << (2 * K)) - 1ULL;
	const unsigned n_events = g.cnt->n_events < g.cap_events ? g.cnt->n_events : g.cap_events;
	unsigned *ha = hist[warp][0], *hr = hist[warp][1];
	unsigned long long tot_reads = 0, tot_bytes = 0;
	for (unsigned e = blockIdx.x * (KMER_THREADS / 32) + warp; e < n_events; e += gridDim.x * (KMER_THREADS / 32)) {
		idl_event_result ev = g.eres[e];
		if (ev.reject != IDL_EV_COUNTED) continue; // warp-uniform
		const idl_aln_result ar = g.ares[ev.aln];
		const idl_region R = g.region[ar.region];
		__syncwarp();
		for (int i = lane; i < 256; i += 32) { ha[i] = 0; hr[i] = 0; }
		__syncwarp();
		// a code of ~0 (a k-mer with a non-ACGT base) matches nothing: its constants cannot equal a 54-bit field
		const bool ref_ok = ev.ref_code != ~0ULL, alt_ok = ev.alt_code != ~0ULL;
		const uint64_t r1 = ref_ok ? (~ev.ref_code & kmask) : ~0ULL, r2 = ref_ok ? kmer_pair_reverse(ev.ref_code, K) : ~0ULL;
		const uint64_t a1 = alt_ok ? (~ev.alt_code & kmask) : ~0ULL, a2 = alt_ok ? kmer_pair_reverse(ev.alt_code, K) : ~0ULL;
		unsigned k_ref = 0, k_alt = 0, k_both = 0, n_reads = 0, sum_r = 0, sum_a = 0, bytes = 0; // per group leader
		for (unsigned j0 = 0; j0 < R.n_reads; j0 += 4) { // :293-311
			const unsigned j = j0 + (unsigned)grp;
			idl_read rd; rd.len = 0; rd.mapq = 0; rd.seq_off = 0;
			if (j < R.n_reads) rd = g.read[R.read_begin + j];
			const bool ok = j < R.n_reads && (int)rd.mapq >= P.count_min_mapq; // :294
			const int L = rd.len;
			const int rec2 = ((L + 63) >> 6) << 2, recn = ((L + 63) >> 6) << 1; // words of this read's records in the two pools
			const uint32_t *w2 = g.seq2 + (rd.seq_off >> 4), *wn = g.seqn + (rd.seq_off >> 5);
			int first_r = 0x7fffffff, first_a = 0x7fffffff;
			if (ok)
				for (int base = 0; base + K <= L; base += 128) {
					const int p0 = base + 16 * gl;
					if (p0 + K > L) continue;
					const int w = p0 >> 4, nwd = p0 >> 5, nsh = p0 & 31;
					const uint32_t x0 = __ldg(w2 + w), x1 = __ldg(w2 + w + 1), x2 = w + 2 < rec2 ? __ldg(w2 + w + 2) : 0u;
					const uint32_t n0 = __ldg(wn + nwd), n1 = nwd + 1 < recn ? __ldg(wn + nwd + 1) : 0u;
					const uint64_t nb = (((uint64_t)n1 << 32) | n0) >> nsh; // N flags of bases p0 .. p0+41 (nsh is 0 or 16)
#pragma unroll
					for (int i = 0; i < 16; ++i) {
						const int p = p0 + i;
						if (p + K > L) break;
						if ((unsigned)(nb >> i) & ((1u << K) - 1u)) continue; // a window holding a non-ACGT base never matches
						const uint64_t c = (((uint64_t)__funnelshift_r(x1, x2, 2 * i) << 32) | __funnelshift_r(x0, x1, 2 * i)) & kmask;
						if (c == r1 || c == r2) first_r = min(first_r, p);
						if (c == a1 || c == a2) first_a = min(first_a, p);
					}
				}
#pragma unroll
			for (int d = 1; d < 8; d <<= 1) { first_r = min(first_r, __shfl_xor_sync(FULL_MASK, first_r, d)); first_a = min(first_a, __shfl_xor_sync(FULL_MASK, first_a, d)); }
			if (ok && gl == 0) {
				const bool rf = first_r != 0x7fffffff, af = first_a != 0x7fffffff;
				n_reads += 1; bytes += (unsigned)((L + 3) / 4 + (L + 7) / 8 + 16);
				if (rf) { k_ref += 1; sum_r += (unsigned)(first_r < (L - K) - first_r ? first_r : (L - K) - first_r); atomicAdd(&hr[rd.mapq], 1u); } // declared kmer.dists distance
				if (af) { k_alt += 1; sum_a += (unsigned)(first_a < (L - K) - first_a ? first_a : (L - K) - first_a); atomicAdd(&ha[rd.mapq], 1u); }
				if (rf && af) k_both += 1;
			}
		}
		k_ref = __reduce_add_sync(FULL_MASK, k_ref); k_alt = __reduce_add_sync(FULL_MASK, k_alt); k_both = __reduce_add_sync(FULL_MASK, k_both);
		sum_r = __reduce_add_sync(FULL_MASK, sum_r); sum_a = __reduce_add_sync(FULL_MASK, sum_a);
		n_reads = __reduce_add_sync(FULL_MASK, n_reads); bytes = __reduce_add_sync(FULL_MASK, bytes);
		__syncwarp();
		const int med_a = kmer_median(ha, k_alt, lane), med_r = kmer_median(hr, k_ref, lane);
		if (lane == 0) {
			ev.k_ref = (int)k_ref; ev.k_alt = (int)k_alt; ev.k_both = (int)k_both;
			ev.n_adist = (int)k_alt; ev.n_rdist = (int)k_ref; ev.sum_adist = (long long)sum_a; ev.sum_rdist = (long long)sum_r;
			ev.amq_median = med_a; ev.rmq_median = med_r;
			if (k_both > 0) { // :313: genotype by alignment instead
				ev.aligned = 1; ev.ref_support = ev.alt_support = ev.both_found = 0;
				const unsigned long long old = atomicAdd(&g.cnt->al_pack, (1ULL << 40) | (unsigned long long)R.n_reads);
				const unsigned slot = (unsigned)(old >> 40);
				if (slot < g.cap_al) { AlEntry a; a.event = e; a.base = (unsigned)(old & ((1ULL << 40) - 1)); a.n_reads = R.n_reads; a.pad = 0; g.al_list[slot] = a; }
				else atomicOr(&g.cnt->overflow, 32u);
				atomicAdd(&g.cnt->al_events, 1ULL);
			} else { ev.aligned = 0; ev.ref_support = ev.k_ref; ev.alt_support = ev.k_alt; ev.both_found = 0; }
			g.eres[e] = ev;
		}
		tot_reads += n_reads; tot_bytes += (unsigned long long)bytes + 64ULL;
	}
	if (lane == 0 && tot_bytes) { atomicAdd(&g.cnt->kmer_reads, tot_reads); atomicAdd(&g.cnt->kmer_bytes, tot_bytes); }
}

// ---------------------------------------------------------------------------------------------------------------
// AL fallback, step 1: one thread per (AL event, read): the window tests of :328-341; survivors become two DP tasks
// ---------------------------------------------------------------------------------------------------------------
__global__ void al_prep_kernel(GenoArgs g)
{
	const idl_params &P = g.P;
	const unsigned long long pack = g.cnt->al_pack;
	unsigned n_al = (unsigned)(pack >> 40); if (n_al > g.cap_al) n_al = g.cap_al;
	const unsigned total = (unsigned)(pack & ((1ULL << 40) - 1));
	if (n_al == 0) return;
	for (unsigned it = blockIdx.x * blockDim.x + threadIdx.x; it < total; it += gridDim.x * blockDim.x) {
		// entries are sorted by base (one packed atomic hands out slot and base together)
		int lo = 0, hi = (int)n_al - 1;
		while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (g.al_list[mid].base <= it) lo = mid; else hi = mid - 1; }
		const AlEntry ae = g.al_list[lo];
		const unsigned j = it - ae.base;
		if (j >= ae.n_reads) continue; // item of an entry dropped by overflow
		const idl_event_result ev = g.eres[ae.event];
		const idl_aln_result ar = g.ares[ev.aln];
		const idl_contig_result cr = g.cres[ar.contig];
		const idl_region R = g.region[ar.region];
		const idl_read rd = g.read[R.read_begin + j];
		if ((int)rd.mapq < P.count_min_mapq) continue;              // :328
		const int rs = rd.start + rd.trim_a;                       // :331
		if (rs > ev.t_stop) continue;                              // :332
		const int Lx = ev.type == 0 ? ev.len : 0;                  // :333-335
		if (rs + (int)rd.trim_len + Lx < ev.t_start) continue;     // :336
		const int start = (rs > cr.start ? rs : cr.start) - cr.start; // :339
		const unsigned slot = atomicAdd(&g.cnt->n_al_items, 1u);
		if (slot >= g.cap_items) { atomicOr(&g.cnt->overflow, 64u); continue; }
		AlItem a; a.event = ae.event; a.read = R.read_begin + j; a.start = start; a.pad = 0;
		g.al_items[slot] = a;
		int rlen = ar.ref_len - start; if (rlen < 0) rlen = 0;
		int clen = cr.len - start; if (clen < 0) clen = 0;
		const int qlen = rd.trim_len, wb = P.b_bw;
		const uint16_t k0 = sort_key_b(est_diagonals(qlen, rlen, wb), qlen), k1 = sort_key_b(est_diagonals(qlen, clen, wb), qlen);
		g.sortB.keys[2 * slot] = k0; g.sortB.keys[2 * slot + 1] = k1;
		atomicAdd(&g.sortB.hist[k0], 1u); atomicAdd(&g.sortB.hist[k1], 1u);
	}
}

// count_flanked_cigar (src/indelope.nim:185-199) over the truncated view of the reversed scratch
__device__ __forceinline__ int count_flanked(const uint32_t *cig_rev, int n, int max_q)
{
	const int ntr = ksw_trunc_count(cig_rev, n, max_q);
	bool matched = false; int cnt = 0, last_op = 0;
	for (int k = 0; k < ntr; ++k) {
		const int op = cig_rev[n - 1 - k] & 0xf;
		if (!matched) { if (op == 0) { cnt += 1; matched = true; } }
		else cnt += 1;
		last_op = op;
	}
	if (last_op != 0) cnt -= 1;
	return cnt;
}

// AL fallback, step 2: call-site B of kernel 2, one group per task (read vs reference suffix / contig suffix), :343-347
template <bool UNB>
__global__ void __launch_bounds__(UNB ? 32 * KSW_UNB_WARPS : DP_THREADS, UNB ? KSW_UNB_CTAS : 3) al_kernel(GenoArgs g)
{
	extern __shared__ __align__(16) unsigned char smem_raw[];
	const int lane = lane_id(), gl = lane & (DP_G - 1), grp = lane / DP_G;
	const idl_params &P = g.P;
	unsigned n_items = g.cnt->n_al_items; if (n_items > g.cap_items) n_items = g.cap_items;
	const unsigned n_tasks = 2 * n_items;
	for (;;) {
		unsigned base = 0;
		if (lane == 0) base = atomicAdd(&g.cnt->al_next, (unsigned)DP_NG);
		base = __shfl_sync(FULL_MASK, base, 0);
		if (base >= n_tasks) break;
		const bool valid = base + grp < n_tasks;
		unsigned task = 0, region = 0; int qlen = 0, tlen = 0; const uint8_t *t = g.refcodes;
		KswQuery kq; kq.codes = nullptr; kq.seq2 = g.seq2; kq.seqn = g.seqn; kq.base = 0;
		if (valid) {
			task = g.sortB.order[base + grp];
			const AlItem it = g.al_items[task >> 1];
			const idl_event_result ev = g.eres[it.event];
			const idl_aln_result ar = g.ares[ev.aln];
			const idl_contig_result cr = g.cres[ar.contig];
			const idl_region R = g.region[ar.region];
			const idl_read rd = g.read[it.read];
			region = ar.region;
			qlen = rd.trim_len; kq.base = rd.seq_off + rd.trim_a;
			if (!(task & 1)) { t = g.refcodes + R.ref_off + (cr.start - R.ref_start) + it.start; tlen = ar.ref_len - it.start; } // ref_sub :340
			else { t = g.ctg_codes + cr.seq_off + it.start; tlen = cr.len - it.start; }                                          // ctg_sub :341
			if (tlen < 0) tlen = 0;
		}
		const KswMem M = dp_mem(g, smem_raw, qlen, tlen, UNB ? KSW_UNB_WARPS : DP_WARPS);
		KswOut o;
		// the whole warp: four alignments in lockstep; reads of up to 160 bases take the row-owned variant (ksw2_rows.cuh)
		const int rw = UNB ? ksw_rows_pick(valid, qlen, tlen, g.kpB, M) : 0;
		if (rw == 5) ksw2_rows<5, false>(valid, qlen, kq, tlen, t, g.kpB, M, o);
		else ksw2_group<DP_G, false, UNB>(valid, qlen, kq, tlen, t, g.kpB, M, o);
		if (valid) {
			if (gl == 0) {
				const unsigned st = dp_status_bits(o.status);
				int c = count_flanked(M.cig, o.n_cigar, o.max_q);
				if (c > 126) c = 126; // only "== 1" and "> 1" are consumed (:353-356)
				if (st) { atomicOr(&g.rres[region].status, st); c = -1; }
				g.al_res[task] = (int8_t)c;
				atomicAdd(&g.cnt->dp_b, 1ULL); atomicAdd(&g.cnt->dp_cells_b, (unsigned long long)o.cells);
			}
		}
		__syncwarp();
	}
}

// AL fallback, step 3: the vote of :353-356
__global__ void al_vote_kernel(GenoArgs g)
{
	unsigned n_items = g.cnt->n_al_items; if (n_items > g.cap_items) n_items = g.cap_items;
	for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n_items; i += gridDim.x * blockDim.x) {
		const int rn = g.al_res[2 * i], an = g.al_res[2 * i + 1];
		if (rn < 0 || an < 0) continue; // DP capacity error, already flagged on the region
		const AlItem it = g.al_items[i];
		if (rn == 1 && an > 1) atomicAdd(&g.eres[it.event].ref_support, 1);
		else if (an == 1 && rn > 1) atomicAdd(&g.eres[it.event].alt_support, 1);
	}
}
