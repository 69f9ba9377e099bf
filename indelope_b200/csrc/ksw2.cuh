// indelope_b200/csrc/ksw2.cuh -- kernel 2: ksw2 extension alignment, a sub-warp GROUP of G threads per alignment.
//
// Replaces ksw_extz2_sse (src/ksw2/csrc/ksw2_extz2_sse.c:113-388, flag == 0) bit for bit: the anti-diagonal
// difference recurrence on wrapping int8 lanes, the 16-lane rounding of the band and the stale lanes it leaves
// behind (SURVEY.md appendix B: they feed real cells), the exact 32-bit max with the SSE 4-accumulator tie
// order, z-drop, and ksw_backtrack (:47-79) to a BAM-style CIGAR.
//
// Mapping.  32/G alignments run side by side in one warp, in lockstep (the per-diagonal control code is issued once
// for all of them).  Inside a group every thread owns W consecutive packed words = 4*W consecutive columns of the
// anti-diagonal: u, v, x, y, s are int8x4 words (the SSE code holds sixteen lanes per register), wrapping add/sub and
// signed/unsigned compares are the byte-SIMD intrinsics, the x[t-1]/v[t-1] neighbour is the thread's previous word or
// comes from the previous thread through __shfl_up_sync + a one-byte funnel shift.  One fused pass per diagonal does
// the 16-lane score blocks (:215-228), the core update (:262-284) and the exact-H update (:312-349) with the columns in
// registers.  The lane arrays live in shared memory as a RING over the live band (columns left of the band are dead;
// the 16-lane block that enters the band is cleared just before, exactly reproducing calloc'ed memory and the stale
// values the SSE code leaves behind), H is a ring of the exact band, the backtrack matrix goes to global memory and is
// walked through a 32x32 shared-memory tile.  All arithmetic is integer; no tensor cores.
#pragma once
#include <climits>
#include "common.cuh"

struct KswOut {
	int max, zdropped, max_q, max_t, mqe, mqe_t, mte, mte_q, score;
	int n_cigar;      // ops left in the scratch buffer, REVERSED (last op first)
	int status;       // 0 ok, 1 early return (:147/:171), negative: capacity
	long long cells;  // exact in-band cells over executed diagonals
};

#define KSW_PSTORE(p, v) __stcs((p), (v)) /* streaming stores: the backtrack matrix is written once and read back once, in part */
#define KSW_BTILE_BYTES 1152 /* backtrack tile: 32 rows of nine aligned words */
#define KSW_BTILE_ROW 36
#define KSW_QR_PAD 32     /* zero bytes in front of the reversed query: lanes left of the exact band index it below 0 */
#define KSW_PMAT_PAD 64   /* bytes in front of every backtrack matrix (the tile prefetch may start before row 0) */
#define KSW_ST_EARLY 1
#define KSW_ST_RCAP (-2)
#define KSW_ST_PCAP (-3)
#define KSW_ST_CIGCAP (-4)
#define KSW_ST_HCAP (-5)
#define KSW_ST_SEQCAP (-6)

__device__ __forceinline__ void ksw_reset(KswOut &o) // ksw_reset_extz :81-86
{
	o.max_q = o.max_t = o.mqe_t = o.mte_q = -1;
	o.max = 0; o.score = o.mqe = o.mte = KSW_NEG_INF;
	o.n_cigar = 0; o.zdropped = 0; o.status = 0; o.cells = 0;
}

// widest rounded band (bytes of one backtrack row) for a query/target/bandwidth, :164-165
__host__ __device__ inline int ksw_ncol(int qlen, int tlen, int w)
{
	if (w < 0) w = tlen > qlen ? tlen : qlen;
	int n = qlen < tlen ? qlen : tlen;
	n = n < w + 1 ? n : w + 1;
	return ((n + 15) / 16 + 1) * 16;
}
// row pitch of the backtrack matrix in global memory: a multiple of 32 bytes, so that the 32 bytes a group stores per round
// are one whole, aligned L2 sector (a half-written sector is first FETCHED from DRAM: with the reference's 16-byte pitch
// every second row straddled sectors and the kernel read more than it wrote)
__host__ __device__ inline int ksw_pitch(int ncol) { return (ncol + 31) & ~31; }
// ring of lane columns: the rounded band, the column left of it, 16 lanes of score overrun and the 16 being cleared
__host__ __device__ inline int ksw_ring_cols(int ncol) { int r = 64; while (r < ncol + 48) r <<= 1; return r; }
// bytes of query staging: KSW_QR_PAD zero bytes, the reversed query, zero padding (:188).  The target is not staged as a
// whole: a ring over the live band is filled from global memory as 16-lane blocks enter.
__host__ __device__ inline size_t ksw_seq_bytes(int qlen, int tlen)
{
	(void)tlen;
	return (size_t)(KSW_QR_PAD + ((qlen + 35) & ~3));
}

// rows of the backtrack matrix an alignment can write: the anti-diagonals it can execute before the band runs out (st0 > en0, :200-203)
__host__ __device__ inline int ksw_rows_bound(int qlen, int tlen, int w)
{
	int d = qlen + tlen - 1;
	if (w >= 0) { if (d > 2 * qlen + w + 1) d = 2 * qlen + w + 1; if (d > 2 * tlen + w + 1) d = 2 * tlen + w + 1; }
	return d > 0 ? d : 0;
}
// off[r] / off_end[r] of the reference are pure functions of r (:196-199,205)
// unb: w >= max(qlen, tlen), where the two w-clamps never bind ((r-w+1)>>1 <= max(0, r-qlen+1) and (r+w)>>1 >= min(r, tlen-1))
__device__ __forceinline__ void ksw_band(int r, int qlen, int tlen, int w, int &st0, int &en0, bool unb = false)
{
	int st = 0, en = tlen - 1;
	if (st < r - qlen + 1) st = r - qlen + 1;
	if (en > r) en = r;
	if (!unb) {
		if (st < ((r - w + 1) >> 1)) st = (r - w + 1) >> 1;
		if (en > ((r + w) >> 1)) en = (r + w) >> 1;
	}
	st0 = st; en0 = en;
}

// ---- four int8 lanes per 32-bit register ----
__device__ __forceinline__ uint32_t sel4(uint32_t m, uint32_t a, uint32_t b) { return (a & m) | (b & ~m); } // m ? a : b, per byte (one LOP3)
__device__ __forceinline__ uint32_t rep4(int v) { return (uint32_t)(v & 0xff) * 0x01010101u; }
// 0xff in every byte whose top bit is set (PRMT with the sign-replicate selector bit; __byte_perm() masks that bit off)
__device__ __forceinline__ uint32_t msb_to_mask4(uint32_t v)
{
	uint32_t r;
	asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(v), "r"(0u), "r"(0xba98u));
	return r;
}
#define KSW_H80 0x80808080u
// 0xff in every byte where a >= b, for bytes a, b in [0,127]: (a | 0x80) - b never borrows across bytes
__device__ __forceinline__ uint32_t ge4_pos(uint32_t a, uint32_t b) { return msb_to_mask4((a | KSW_H80) - b); }

// tie order of the SSE arg-max (:316-348): 4 strided accumulators (lower accumulator, then lower t), then the scalar tail
__device__ __forceinline__ unsigned ksw_tie_rank(int t, int st0, int en1) { return 1u + ((t < en1 ? (unsigned)((t - st0) & 3) : 4u) << 20) + (unsigned)(t - st0); }

// where the query of an alignment comes from: 0..4 codes, or a 2-bit packed read (+ non-ACGT plane) of the batch
struct KswQuery { const uint8_t *codes; const uint32_t *seq2, *seqn; unsigned base; };
__device__ __forceinline__ uint8_t ksw_query_code(const KswQuery &q, int i)
{
	if (q.codes) return q.codes[i];
	const unsigned b = q.base + (unsigned)i;
	return ((q.seqn[b >> 5] >> (b & 31)) & 1u) ? (uint8_t)4 : (uint8_t)((q.seq2[b >> 4] >> (2 * (b & 15))) & 3u);
}

// Memory of one group.  Shared memory, four rings over the live band indexed by ((column word + rot) & mask): xvuy =
// {x, v, u, y} packed words (16 bytes per 4 columns, one 128-bit load and store per word and diagonal), g = the exact
// scores as uint16 (8 bytes per 4 columns), S = score words, T = target codes; then seq = the query staging.  The start
// of the region doubles as the backtrack tile once the DP is over.  Global memory: pmat = backtrack matrix workspace,
// cig = CIGAR scratch.
// Bank staggering: a 128-bit access is served one group (8 threads x 16 contiguous bytes) at a time, so xvuy needs none;
// the 64-bit accesses to g pair two groups and the 32-bit accesses to S and T put all four groups of a warp into one
// wavefront: group k of the warp rotates its rings by 8k words, so that groups at the same relative column fall into
// different banks without any slack bytes.
struct KswMem { uint4 *xvuy; uint2 *g; uint32_t *S, *T; int ring_cols, rot; uint8_t *seq; int seq_cap; uint8_t *pmat; size_t p_cap; uint32_t *cig; int cig_cap;
                int region_bytes; /* shared-memory bytes of the group's region (ksw2_rows.cuh stages its target there) */ };
// layout of a group's region (a multiple of 128 bytes): [xvuy 4R][g 2R][S R][T R][seq]
__host__ __device__ inline size_t ksw_group_seq_off(int ring_cols) { return (size_t)8 * ring_cols; }
__host__ __device__ inline size_t ksw_group_smem(int ring_cols, int seq_cap)
{
	size_t b = ksw_group_seq_off(ring_cols) + (size_t)((seq_cap + 15) & ~15);
	if (b < KSW_BTILE_BYTES) b = KSW_BTILE_BYTES;
	return (b + 127) & ~(size_t)127;
}
__device__ __forceinline__ void ksw_group_mem(KswMem &m, unsigned char *base, int grp_in_warp, int ring_cols)
{
	m.xvuy = (uint4*)base; m.ring_cols = ring_cols; m.rot = 8 * (grp_in_warp & 3);
	m.g = (uint2*)(base + (size_t)4 * ring_cols);
	m.S = (uint32_t*)(base + (size_t)6 * ring_cols);
	m.T = (uint32_t*)(base + (size_t)7 * ring_cols);
	m.seq = base + ksw_group_seq_off(ring_cols);
	m.region_bytes = 0;
}
// four target codes starting at column t, zero beyond the end (:187)
__device__ __forceinline__ uint32_t ksw_target_word(const uint8_t *target, int tlen, int t)
{
	uint32_t w = 0;
#pragma unroll
	for (int c = 0; c < 4; ++c) if (t + c < tlen) w |= (uint32_t)target[t + c] << (8 * c);
	return w;
}
__device__ __forceinline__ bool ksw_has4(uint32_t w) { const uint32_t x = w ^ 0x04040404u; return ((x - 0x01010101u) & ~x & 0x80808080u) != 0u; }

// max / min over the 8 threads of a group with full-warp butterflies (the four groups of a warp reduce side by side)
template <int G = 8> __device__ __forceinline__ unsigned ksw_group_max(unsigned v)
{
#pragma unroll
	for (int d = 1; d < G; d <<= 1) { const unsigned o = __shfl_xor_sync(FULL_MASK, v, d); v = v > o ? v : o; }
	return v;
}
template <int G = 8> __device__ __forceinline__ unsigned ksw_group_min(unsigned v)
{
#pragma unroll
	for (int d = 1; d < G; d <<= 1) { const unsigned o = __shfl_xor_sync(FULL_MASK, v, d); v = v < o ? v : o; }
	return v;
}
template <int G = 8> __device__ __forceinline__ bool ksw_group_any(bool p, int lane) { return ((__ballot_sync(FULL_MASK, p) >> (lane & ~(G - 1))) & ((1u << G) - 1u)) != 0u; }
// wildcard (code 4) lanes score 0 (:219,226); out of line so that the common all-ACGT case pays one branch
__device__ __noinline__ uint32_t ksw_wild_score(uint32_t sq, uint32_t sq2, uint32_t sc, uint32_t qe2)
{
	return sel4(msb_to_mask4(((sq ^ 0x04040404u) + 0x7f7f7f7fu) & ((sq2 ^ 0x04040404u) + 0x7f7f7f7fu)), sc, qe2);
}

// The core update of one packed word, :262-284 (flag 0): in (previous diagonal) xt1, vt1 = x, v of lanes t-1 .. t+2, ut, yt = u, y
// of lanes t .. t+3, z0 = s + 2(q+e); out the new x, v, u, y and the backtrack byte d of the four lanes.
__device__ __forceinline__ void ksw_core_word(const KswParams &P, bool fast_ok, uint32_t z0, uint32_t xt1, uint32_t vt1, uint32_t ut, uint32_t yt,
                                              uint32_t &xn, uint32_t &vn, uint32_t &un, uint32_t &yn, uint32_t &d)
{
	const uint32_t MAXSC = P.maxsc_4, Q4 = P.q_4;
	if (fast_ok && !((xt1 | vt1 | ut | yt) & 0xc0c0c0c0u)) {
		// every byte is in [0,63]: sums stay below 128, signed and unsigned compares agree and nothing carries
		// between bytes, so the core runs on plain 32-bit adds and (a | 0x80) - b compares
		const uint32_t a = xt1 + vt1, b = yt + ut;
		uint32_t m = ge4_pos(z0, a);                    // z >= a
		uint32_t z = sel4(m, z0, a);
		d = ~m & 0x01010101u;
		m = ge4_pos(z, b);                              // z >= b
		d = sel4(m, d, 0x02020202u);
		z = sel4(m, z, b);
		z = sel4(msb_to_mask4(P.maxsc_h80 - z), z, MAXSC); // min(z, max score)
		const uint32_t zh = z | KSW_H80;
		un = (zh - vt1) ^ KSW_H80; vn = (zh - ut) ^ KSW_H80;
		z -= Q4;
		m = ge4_pos(z, a);                              // z >= a: x = 0
		xn = sel4(m, z, a) - z; d |= ~m & 0x08080808u;
		m = ge4_pos(z, b);
		yn = sel4(m, z, b) - z; d |= ~m & 0x10101010u;
	} else { // the lane-exact wrapping int8 form
		uint32_t z = z0;
		uint32_t a = __vadd4(xt1, vt1);
		uint32_t b = __vadd4(yt, ut);
		uint32_t m = __vcmpgts4(a, z);                 // a > z (signed)
		d = m & 0x01010101u;
		z = sel4(m, a, z);                             // signed max
		m = __vcmpgts4(b, z);                          // b > z (signed)
		d = sel4(m, 0x02020202u, d);
		z = sel4(__vcmpgtu4(b, z), b, z);              // unsigned max
		z = sel4(__vcmpgtu4(z, MAXSC), MAXSC, z);      // unsigned min
		vn = __vsub4(z, ut); un = __vsub4(z, vt1);
		z = __vsub4(z, Q4);
		a = __vsub4(a, z);
		b = __vsub4(b, z);
		m = __vcmpgts4(a, 0u);
		xn = a & m; d |= m & 0x08080808u;
		m = __vcmpgts4(b, 0u);
		yn = b & m; d |= m & 0x10101010u;
	}
}

// Prefetch of the backtrack bytes the next 32 diagonals of the walk can touch, by the eight threads of a group (all 32 threads of the warp
// call this together).  Tile row k = diagonal r0 - k; the path can enter it at columns c0 - k .. c0 only, i.e. at the matrix bytes
// e_k - k .. e_k with e_k = `row_end(k)`, the byte offset of (r0 - k, c0) from `pmat` (INT_MIN: no such row).  The tile row holds the nine
// aligned words that end with the word of e_k, so the byte of column c0 - d sits at tile byte 36 k + 32 + (e_k & 3) - d; e_k & 3 is the same
// for every row (row pitches and band offsets are multiples of 4).  The eight lanes read eight consecutive words of ONE row per
// instruction -- one or two 32-byte sectors per row.  (The first version gave every thread four rows and one LDG.32 per word: the L1 does
// not merge requests to a sector that is in flight, so every word cost a sector at the L2 and, the lines being long evicted, in DRAM:
// al_kernel read 31.7 GB back for the 20.4 GB it wrote.)  lo / hi bound the byte offsets that may be touched (the workspace of this
// alignment incl. its padding); a row whose entry bytes lie outside is never read by the walk (its state is forced there).
// one word of the backtrack matrix into the shared-memory tile: an asynchronous copy (LDGSTS), so that the 33 words a thread moves per
// tile are all in flight at once without holding 33 registers -- one DRAM round trip per tile, not one per batch of loads -- and with
// the L2 prefetch size capped at 64 bytes: a plain ld.global pulled 128 bytes around every word it missed, four sectors per row of
// the tile where one or two are needed (al_kernel: 804 M sectors read from L2 per launch against 448 M with the cap)
__device__ __forceinline__ void ksw_tile_cp(uint32_t *dst, const uint32_t *src)
{
	const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst);
	asm volatile("cp.async.ca.shared.global.L2::64B [%0], [%1], 4;" :: "r"(d), "l"(src) : "memory");
}
__device__ __forceinline__ void ksw_tile_wait() { asm volatile("cp.async.wait_all;" ::: "memory"); }
template <int G = 8, class F>
__device__ __forceinline__ void ksw_tile_fetch(bool more, F &&row_end, const uint8_t *pmat, int lo, int hi, uint32_t *tile)
{
	static_assert(G == 8 || G == 4, "groups of 8 or 4 threads");
	const int lane = lane_id(), gl = lane & (G - 1), gbase = lane & ~(G - 1);
	constexpr int Q = 32 / G;                                    // rows per thread: thread gl computes the ends of rows gl, gl + G, ...
	int ev[Q];
#pragma unroll
	for (int q = 0; q < Q; ++q) {
		int e = more ? row_end(gl + G * q) : INT_MIN;
		if (e != INT_MIN) e = e < lo + 35 ? lo + 35 : (e > hi - 4 ? hi - 4 : e);
		ev[q] = e;
	}
#pragma unroll
	for (int q = 0; q < Q; ++q) {
#pragma unroll
		for (int kk = 0; kk < G; ++kk) {
			const int k = G * q + kk;
			const int e = __shfl_sync(FULL_MASK, ev[q], gbase + kk);
#pragma unroll
			for (int h = 0; h < 8 / G; ++h) {
				const int wo = gl + G * h;                           // my word(s) of this row, counted down from the word of e
				const int w = (e >> 2) - wo;
				if (e != INT_MIN && w >= ((e - k) >> 2)) ksw_tile_cp(tile + (k * 9 + 8 - wo), (const uint32_t*)(pmat + 4 * (long long)w));
			}
		}
	}
	{ // rows 29 .. 31 can need a ninth word
		const int k = 29 + gl;
		const int e = __shfl_sync(FULL_MASK, ev[Q - 1], gbase + ((29 + gl) & (G - 1)));
		const int w = (e >> 2) - 8;
		if (gl < 3 && e != INT_MIN && w >= ((e - k) >> 2)) ksw_tile_cp(tile + k * 9, (const uint32_t*)(pmat + 4 * (long long)w));
	}
	ksw_tile_wait();
}

// ALL 32 threads of a warp call this together: 4 groups of G = 8 threads, one alignment per group (valid = 0 for a group
// without one).  The anti-diagonal loop and the rounds inside it run in lockstep over the four alignments, so every
// barrier and shuffle is a plain full-warp one; a group whose alignment is shorter or has stopped idles behind a predicate.
// The threads of a group pass identical arguments; `out` comes back identical in each of them.
// EZ_FULL = false drops the end-of-query / end-of-target scores (mqe, mte, score of ksw_extz_t): the AL fallback reads only
// the CIGAR and max_q (src/indelope.nim:346-347 over the truncated iterator of src/ksw2/ksw2.nim:22-33).
// UNB = true is the unbanded case, P.w < 0 (the AL fallback, src/indelope.nim:317-318,343-344): w = max(qlen, tlen), the
// band is the whole anti-diagonal [max(0, r-qlen+1), min(r, tlen-1)] and neither w-clamp of :196-199 ever binds.  A real
// cell then only reads real cells of the previous diagonal (its left neighbour t-1 was the first in-band lane there; a
// column that enters gets u, y from the :212 patch), so the lanes the SSE code computes beyond the exact band through its
// 16-lane rounding -- which the banded call-site must reproduce because they feed real cells later -- are write-only
// here and nothing reads their backtrack bytes.  The variant therefore computes only the packed words that hold in-band
// lanes, always with fresh scores (no stale-score ring), and stores backtrack rows from the band's first word.
template <int G, bool EZ_FULL = true, bool UNB = false>
__device__ void ksw2_group(bool valid, int qlen, const KswQuery query, int tlen, const uint8_t *target, const KswParams P, const KswMem M, KswOut &out)
{
	static_assert(G == 8 || G == 4, "8 threads per alignment (4 alignments per warp) or 4 (8 per warp: the per-diagonal control code is issued once for twice as many alignments)");
	const int lane = lane_id();
	const int gl = lane & (G - 1);
	ksw_reset(out);
	const int qe = P.q + P.e;
	int min_sc = P.mismatch < 0 ? P.mismatch : 0;
	if (P.match < min_sc) min_sc = P.match;
	int w = P.w;
	if (w < 0) w = tlen > qlen ? tlen : qlen; // :161
	const int n_col = valid ? ksw_ncol(qlen, tlen, w) : 16; // :164-165 (bytes)
	const int pitch = UNB ? ksw_pitch(4 * ((((qlen < tlen ? qlen : tlen) + 3) >> 2) + 1)) : ksw_pitch(n_col);
	// The exact scores H[] (:177-178, int32 in the reference) live as uint16: g[t] = H[t] + (q+e)*(r+1) + gbias, r = the
	// diagonal of the last update.  Every in-band column is updated on every diagonal, so the per-diagonal -(q+e) of
	// :323-348 turns into a common offset, the update into an unsigned byte add, and the band max into a packed 16-bit max.
	const int gbias = 2 * qe;
	bool live = valid;
	if (live) {
		if (qlen <= 0 || tlen <= 0) { out.status = KSW_ST_EARLY; live = false; }     // :147
		else if (UNB && P.w >= 0) { out.status = KSW_ST_RCAP; live = false; }         // the caller picked the wrong variant
		else if (-min_sc > 2 * qe) { out.status = KSW_ST_EARLY; live = false; }      // :171
		else if (ksw_ring_cols(n_col) > M.ring_cols) { out.status = KSW_ST_RCAP; live = false; }
		else if (ksw_seq_bytes(qlen, tlen) > (size_t)M.seq_cap) { out.status = KSW_ST_SEQCAP; live = false; }
		else if ((size_t)ksw_rows_bound(qlen, tlen, P.w) * (size_t)pitch + 2 * KSW_PMAT_PAD > M.p_cap) { out.status = KSW_ST_PCAP; live = false; }
		else if ((long long)(qlen + tlen + 2) * qe + (long long)(qlen < tlen ? qlen : tlen) * (P.match > 0 ? P.match : 0) + gbias >= 0xF000) { out.status = KSW_ST_HCAP; live = false; }
	}
	const bool run = live; // this group has a DP to run (and a CIGAR to walk afterwards)
	uint8_t *pmat = M.pmat + KSW_PMAT_PAD;
	const int rm = M.ring_cols - 1, rmw = (M.ring_cols >> 2) - 1, rotw = M.rot, rotc = M.rot << 2;
	uint4 *XV = M.xvuy; uint2 *GR = M.g; uint32_t *S = M.S, *SF = M.T;
	uint16_t *G16 = (uint16_t*)M.g;
	uint8_t *qrp = M.seq; // KSW_QR_PAD zero bytes, then the reversed query, zero padded
	const uint32_t *QRP = (const uint32_t*)qrp;
	const uint32_t QE2 = P.qe2_4, MAXSC = P.maxsc_4, Q4 = P.q_4, MATQ = P.maxsc_4, MISQ = P.misq_4;
	// the carry-free formulation of the core needs every constant and every input byte small and non-negative
	const bool fast_ok = P.match + 2 * qe <= 63 && P.q >= 0 && P.q + 2 * P.e + min_sc >= 0;
	const int nr = live ? qlen + tlen - 1 : 0; // anti-diagonals of this alignment

	// calloc :173: columns [0,16) of u,v,x,y and [0,32) of s start as zero (later blocks are cleared as they enter);
	// stage the first 32 target codes (zero padded, :187) and qr (reversed query, zero padded, :188)
	bool wild = false; // a code 4 seen so far: only then the score needs the wildcard mask (:219,226)
	if (live) {
		for (int k = gl; k < 4; k += G) XV[(k + rotw) & rmw] = make_uint4(0u, 0u, 0u, 0u);
		for (int k = gl; k < 8; k += G) {
			S[(k + rotw) & rmw] = QE2; // S holds s + 2(q+e) (:117): one add less per word and diagonal
			const uint32_t tw = ksw_target_word(target, tlen, 4 * k); SF[(k + rotw) & rmw] = tw; wild |= ksw_has4(tw);
		}
		const int nq = KSW_QR_PAD + ((qlen + 35) & ~3);
		for (int i = gl; i < nq; i += G) {
			const int k = i - KSW_QR_PAD;
			const uint8_t c = (k >= 0 && k < qlen) ? ksw_query_code(query, qlen - 1 - k) : (uint8_t)0; wild |= c == 4; qrp[i] = c;
		}
	}
	wild = ksw_group_any<G>(wild, lane);
	__syncwarp();

	int last_st = -1, last_en = -1, last_st0 = 0, last_en0 = -1, en_clr = 15;
	unsigned g_high = 0; // sticky: an exact score came close to the uint16 range
	int st0 = 0, en0 = 0; // band of diagonal 0 (:196-199)
	for (int r = 0; ; ++r) {
		bool act = live && r < nr;
		if (act && st0 > en0) { out.zdropped = 1; live = false; act = false; } // :200-203
		if (!__any_sync(FULL_MASK, act)) break;
		const int st = st0 & ~15, en = en0 | 15;    // :205
		if (act) out.cells += en0 - st0 + 1;
		// boundary conditions :207-211 (values of the previous diagonal): the word left of the first one supplies x[st-1], v[st-1]
		const bool keep_prev = st > 0 && st - 1 >= last_st && st - 1 <= last_en;
		const uint32_t v1c = (st == 0 && r) ? ((uint32_t)(P.q & 0xff) << 24) : 0u;
		const int goff = qe * (r + 1) + gbias;
		// H[en0] is built from the OLD H[en0-1] (:318): fetch it before this diagonal's updates
		unsigned gprev = 0;
		if (act && r) {
			const int c = en0 > 0 ? en0 - 1 : 0;
			gprev = G16[(c + rotc) & rm];
			if (c < last_st0 || c > last_en0) { // the column was not part of the previous band: its offset is older (the band left the matrix on the right)
				int rr = r - 1;
				for (; rr > 0; --rr) { int s_, e_; ksw_band(rr, qlen, tlen, w, s_, e_, UNB); if (s_ <= c && c <= e_) break; }
				gprev += (unsigned)(qe * (r - 1 - rr));
			}
		}
		const int bend = st0 + (int)((((unsigned)(en0 - st0) >> 4) + 1u) << 4); // one past the last lane the 16-wide score blocks write (en0 >= st0 here)
		const int ws0 = st0 >> 2, w1 = (bend - 1) >> 2, wend = UNB ? en0 >> 2 : en >> 2;
		const int wfirst = UNB ? ws0 : st >> 2, wlast = UNB ? wend : (wend > w1 ? wend : w1);
		const int en1 = st0 + (((en0 - st0) >> 2) << 2);    // end of the 4-wide vector part of the arg-max (:316)
		const unsigned bandw = (unsigned)(en0 - st0);       // columns st0 .. en0-1 are updated in the loop
		uint32_t *prg = (uint32_t*)(pmat + (size_t)r * pitch) + gl; // backtrack row r; word j of the band goes to [j]
		const int cq = qlen - 1 - r;                         // lane t meets query code qr[cq + t]
		const int qsh = 8 * (cq & 3);
		const uint32_t *QRr = QRP + (KSW_QR_PAD >> 2) + (cq >> 2);
		uint32_t bh2 = 0;                                     // this thread's best g over its in-band columns, two uint16 halves
		// Words are dealt round-robin (word j of the band goes to thread j % G), last round first: every word reads the old
		// x, v of the word to its left, which belongs to the previous thread of the same round or to a round not yet done.
		const int rounds = act ? (wlast - wfirst) / G : -1;
		for (int rd = (int)__reduce_max_sync(FULL_MASK, rounds); rd >= 0; --rd) {
			const int j = rd * G + gl, wi = wfirst + j, t = wi << 2, wm = (wi + rotw) & rmw;
			const bool mine = rd <= rounds;
			const bool core = mine && wi <= wend, sca = mine && wi >= ws0 && wi <= w1;
			const uint4 own = XV[wm]; uint2 prv = *(const uint2*)&XV[(wm - 1) & rmw];
			__syncwarp(); // every load of the round is issued before any store of the round
			if (UNB) {
				// one path for every in-band word: fresh scores, the core, the backtrack word; only the exact-score update
				// looks at the band edges (the word that holds st0 and the one that holds en0)
				if (mine && wi <= wend) {
					const uint32_t sq = SF[wm];
					const uint32_t sq2 = __funnelshift_r(QRr[wi], QRr[wi + 1], qsh);
					uint32_t z0 = sel4(msb_to_mask4((sq ^ sq2) + 0x7f7f7f7fu), MISQ, MATQ);
					if (wild) z0 = ksw_wild_score(sq, sq2, z0, QE2);
					if (wi == 0) { prv.x = 0u; prv.y = v1c; } // :207-211 with st == 0; for wi > 0 the ring holds lane 4 wi - 1 of the previous diagonal
					const uint32_t xt1 = __funnelshift_l(prv.x, own.x, 8), vt1 = __funnelshift_l(prv.y, own.y, 8);
					uint32_t d, un, vn, xn, yn;
					ksw_core_word(P, fast_ok, z0, xt1, vt1, own.z, own.w, xn, vn, un, yn, d);
					XV[wm] = make_uint4(xn, vn, un, yn);
					KSW_PSTORE(prg + rd * G, d);
					const int lo = st0 - t, hi = en0 - t; // exact scores of the in-band columns st0 .. en0-1 of this word (:323-348): g[t] += v8[t]
					if (lo <= 0 && hi >= 4) {
						uint2 g2 = GR[wm];
						g2.x += __byte_perm(vn, 0u, 0x4140); g2.y += __byte_perm(vn, 0u, 0x4342);
						bh2 = __vimax3_u16x2(bh2, g2.x, g2.y);
						GR[wm] = g2;
					} else if (hi > 0 && lo < 4) {
						uint2 g2 = GR[wm];
						uint32_t m = 0xffffffffu;
						if (lo > 0) m <<= 8 * lo;
						if (hi < 4) m &= 0xffffffffu >> (8 * (4 - hi));
						const uint32_t vm = vn & m;
						g2.x += __byte_perm(vm, 0u, 0x4140); g2.y += __byte_perm(vm, 0u, 0x4342);
						bh2 = __vimax3_u16x2(bh2, g2.x & __byte_perm(m, 0u, 0x1100), g2.y & __byte_perm(m, 0u, 0x3322));
						GR[wm] = g2;
					}
				}
				continue;
			}
			if (rd > 0 && __all_sync(FULL_MASK, !mine || t + 4 <= en0)) {
				// every word of this round, in all four alignments, lies inside the exact band (rd > 0 puts it at least 32 lanes
				// right of st, so right of st0 too): fresh scores for all four lanes, no boundary lane, no masks.  A group that
				// has no word in this round (shorter band, or finished) only skips.  s is not stored: such a word lies inside
				// the score blocks of the next diagonal as well (st0 grows by at most one, en0 never shrinks), where its
				// scores are recomputed or, on the boundary path, stored.
				if (mine) {
					const uint32_t sq = SF[wm];
					const uint32_t sq2 = __funnelshift_r(QRr[wi], QRr[wi + 1], qsh);
					uint32_t z0 = sel4(msb_to_mask4((sq ^ sq2) + 0x7f7f7f7fu), MISQ, MATQ);
					if (wild) z0 = ksw_wild_score(sq, sq2, z0, QE2);
					const uint32_t xt1 = __funnelshift_l(prv.x, own.x, 8), vt1 = __funnelshift_l(prv.y, own.y, 8);
					uint32_t d, un, vn, xn, yn;
					ksw_core_word(P, fast_ok, z0, xt1, vt1, own.z, own.w, xn, vn, un, yn, d);
					XV[wm] = make_uint4(xn, vn, un, yn);
					KSW_PSTORE(prg + rd * G, d);
					uint2 g2 = GR[wm];
					g2.x += __byte_perm(vn, 0u, 0x4140); g2.y += __byte_perm(vn, 0u, 0x4342);
					bh2 = __vimax3_u16x2(bh2, g2.x, g2.y);
					GR[wm] = g2;
				}
				continue;
			}
			uint32_t z0 = 0;   // s + 2(q+e)
			if (sca) { // scores :215-228: lanes of this word inside the 16-wide blocks get fresh values, the others keep stale s
				const uint32_t sq = SF[wm];
				const uint32_t sq2 = __funnelshift_r(QRr[wi], QRr[wi + 1], qsh);
				const uint32_t neq = msb_to_mask4((sq ^ sq2) + 0x7f7f7f7fu); // 0xff where the codes differ
				uint32_t sc = sel4(neq, MISQ, MATQ);
				if (wild) sc = ksw_wild_score(sq, sq2, sc, QE2);
				const int lo = st0 - t, hi = bend - t; // lanes [lo, hi) of this word belong to the blocks
				if (lo <= 0 && hi >= 4) z0 = sc;
				else {
					uint32_t m = 0xffffffffu;
					if (lo > 0) m <<= 8 * lo;
					if (hi < 4) m &= 0xffffffffu >> (8 * (4 - hi));
					z0 = sel4(m, sc, S[wm]);
				}
				S[wm] = z0;
			} else if (core) z0 = S[wm];
			if (core) {
				if (j == 0 && !keep_prev) { prv.x = 0u; prv.y = v1c; }
				const uint32_t ut = own.z, yt = own.w; // :212 (y[r] = 0, u[r] = q) was applied to the ring at the end of the previous diagonal
				const uint32_t xt1 = __funnelshift_l(prv.x, own.x, 8), vt1 = __funnelshift_l(prv.y, own.y, 8); // lanes t-1..t+2 of the previous diagonal
				uint32_t d, un, vn, xn, yn;
				ksw_core_word(P, fast_ok, z0, xt1, vt1, ut, yt, xn, vn, un, yn, d);
				XV[wm] = make_uint4(xn, vn, un, yn);
				KSW_PSTORE(prg + rd * G, d);
				const int lo = st0 - t, hi = en0 - t; // exact scores of the in-band columns st0 .. en0-1 of this word (:323-348): g[t] += v8[t]
				if (hi > 0 && lo < 4) {
					uint2 g2 = GR[wm];
					if (lo <= 0 && hi >= 4) {
						g2.x += __byte_perm(vn, 0u, 0x4140); g2.y += __byte_perm(vn, 0u, 0x4342);
						bh2 = __vimax3_u16x2(bh2, g2.x, g2.y);
					} else {
						uint32_t m = 0xffffffffu;
						if (lo > 0) m <<= 8 * lo;
						if (hi < 4) m &= 0xffffffffu >> (8 * (4 - hi));
						const uint32_t vm = vn & m;
						g2.x += __byte_perm(vm, 0u, 0x4140); g2.y += __byte_perm(vm, 0u, 0x4342);
						bh2 = __vimax3_u16x2(bh2, g2.x & __byte_perm(m, 0u, 0x1100), g2.y & __byte_perm(m, 0u, 0x3322));
					}
					GR[wm] = g2;
				}
			}
		}
		__syncwarp(); // this diagonal's lanes and g[st0..en0) are visible to the whole group
		// band max of the updated columns, then the en0 cell (:318 / :349)
		unsigned mg = (bh2 & 0xffffu) > (bh2 >> 16) ? (bh2 & 0xffffu) : (bh2 >> 16);
		mg = ksw_group_max<G>(mg);
		unsigned ghen = 0;
		if (act) {
			if (r == 0) ghen = (unsigned)((int)((const uint8_t*)&XV[rotw & rmw])[4] - qe + gbias); // H[0] = v[0] - 2(q+e)
			else {
				const uint8_t *wb = (const uint8_t*)&XV[((en0 >> 2) + rotw) & rmw];
				ghen = gprev + (unsigned)(en0 > 0 ? wb[8 + (en0 & 3)] : wb[4 + (en0 & 3)]); // + u8[en0] or + v8[en0]
			}
		}
		const int hen = (int)ghen - goff;
		g_high |= (unsigned)(mg >= 0xF000u) | (unsigned)(ghen >= 0xF000u);
		const int mh = (int)mg - goff;
		int max_H = hen, max_t = en0; // the initial candidate (H[en0], en0) wins every tie (:318-321)
		// The position of the band max matters only when it becomes the new overall max or when z-drop can fire
		// (ksw_apply_zdrop :88-104 needs max - H > zdrop at least); only then look it up, in the SSE tie order.
		const bool better = act && mh > hen;
		const bool need_t = better && (mh > out.max || (P.zdrop >= 0 && out.max - mh > P.zdrop));
		if (__any_sync(FULL_MASK, need_t)) {
			unsigned best = 0xffffffffu;
			if (need_t) {
				const uint32_t mg2 = mg * 0x10001u;
				for (int wi = ws0 + gl; wi <= ((en0 - 1) >> 2); wi += G) {
					const uint2 g2 = GR[(wi + rotw) & rmw];
					const uint32_t xa = g2.x ^ mg2, xb = g2.y ^ mg2; // a zero halfword = a column that holds the band max
					if (!((((xa - 0x00010001u) & ~xa) | ((xb - 0x00010001u) & ~xb)) & 0x80008000u)) continue;
					const int t = wi << 2;
#pragma unroll
					for (int c = 0; c < 4; ++c) {
						const unsigned val = ((c < 2 ? g2.x : g2.y) >> (16 * (c & 1))) & 0xffffu;
						if ((unsigned)(t + c - st0) < bandw && val == mg) { const unsigned rk = ksw_tie_rank(t + c, st0, en1); best = rk < best ? rk : best; }
					}
				}
			}
			const unsigned rk = ksw_group_min<G>(best);
			if (need_t) { max_H = mh; max_t = st0 + (int)((rk - 1) & 0xfffffu); }
		}
		// band of the next diagonal (:196-199): its new 16-lane block, if any, and its :212 patch are applied now, so that
		// one barrier covers them together with this diagonal's H[en0]
		int st0n, en0n;
		ksw_band(r + 1, qlen, tlen, w, st0n, en0n, UNB);
		const bool nxt = act && r + 1 < nr && st0n <= en0n;
		if (act) {
			if (EZ_FULL) {
				if (en0 == tlen - 1) {
					if (hen > out.mte) { out.mte = hen; out.mte_q = r - en; }
					if (r == qlen + tlen - 2) out.score = hen; // H[tlen-1]
				}
				if (r - st0 == qlen - 1) {
					const int Hst0 = st0 == en0 ? hen : (int)G16[(st0 + rotc) & rm] - goff;
					if (Hst0 > out.mqe) { out.mqe = Hst0; out.mqe_t = st0; }
				}
			}
			if (gl == 0) G16[(en0 + rotc) & rm] = (uint16_t)ghen;
		}
		bool w4 = false;
		const bool enter = nxt && (en0n | 15) > en_clr; // a 16-lane block enters the band: it must read as never written (calloc); the score overrun zone moves on
		if (enter) {
			const int b = en_clr + 1;
			if (G == 4 || gl < 4) XV[((b >> 2) + (gl & 3) + rotw) & rmw] = make_uint4(0u, 0u, 0u, 0u);
			if (G == 4 || gl >= 4) { // ... and the next 16 target codes are fetched
				const int wn = ((b + 16) >> 2) + (gl & 3);
				const uint32_t tw = ksw_target_word(target, tlen, wn << 2);
				if (!UNB) S[(wn + rotw) & rmw] = QE2;
				SF[(wn + rotw) & rmw] = tw; w4 = ksw_has4(tw);
			}
			en_clr += 16;
		}
		if (__any_sync(FULL_MASK, enter)) { wild |= ksw_group_any<G>(w4, lane); __syncwarp(); }
		if (nxt && (en0n | 15) >= r + 1 && gl == 0) { // :212 of the next diagonal: y[r+1] = 0, u[r+1] = q
			uint8_t *wb = (uint8_t*)&XV[(((r + 1) >> 2) + rotw) & rmw];
			wb[8 + ((r + 1) & 3)] = (uint8_t)P.q; wb[12 + ((r + 1) & 3)] = 0;
		}
		__syncwarp();
		if (act && (better ? need_t : true)) { // ksw_apply_zdrop :88-104 (skipped when the band max can neither raise the max nor trigger z-drop)
			if (max_H > out.max) { out.max = max_H; out.max_t = max_t; out.max_q = r - max_t; }
			else if (max_t >= out.max_t && r - max_t >= out.max_q) {
				const int tl = max_t - out.max_t, ql = (r - max_t) - out.max_q;
				const int l = tl > ql ? tl - ql : ql - tl;
				if (P.zdrop >= 0 && out.max - max_H > P.zdrop + l * P.e) { out.zdropped = 1; live = false; }
			}
		}
		last_st = st; last_en = en; last_st0 = st0; last_en0 = en0;
		st0 = st0n; en0 = en0n;
	}
	if (g_high) out.status = KSW_ST_HCAP;
	__syncwarp();
	// backtrack :380-385 -> ksw_backtrack :47-79 (is_rot = 1, left-aligned gaps).  The four groups of the warp walk in
	// lockstep (full-warp barriers; a group without a path, or whose path has ended, idles): with per-group barriers the
	// walkers drift apart and the warp runs them one after the other.
	int i = -1, j = -1;
	if (run) {
		if (!out.zdropped) { i = tlen - 1; j = qlen - 1; }
		else if (out.max_t >= 0 && out.max_q >= 0) { i = out.max_t; j = out.max_q; }
	}
	int n = 0, ovf = 0;
	{
		// The walk itself is serial (one state machine), but its loads are not: before every stretch of <= 32 diagonals the
		// group prefetches the 32 x 32 tile of p[][] the path can touch (row r0-k can only be entered at columns
		// i0-k .. i0) into shared memory (the sequence staging area is free by now), so the walker runs on shared-memory
		// latency instead of one L2/HBM round trip per step.  The four rows a thread fetches are in flight together.
		uint32_t *tile = (uint32_t*)M.xvuy; // 32 rows of 9 words (ksw_tile_fetch); the rings are dead by now
		uint32_t *cig = M.cig; const int cig_cap = M.cig_cap;
		int state = 0;
		unsigned cur_op = 0xffu, cur_len = 0;
		const int p_hi = ksw_rows_bound(qlen, tlen, P.w) * pitch + KSW_PMAT_PAD;
		while (__any_sync(FULL_MASK, i >= 0 && j >= 0)) {
			const bool more = i >= 0 && j >= 0;
			const int i0 = i, r0 = i + j;
			ksw_tile_fetch<G>(more, [&](int k) -> int {
				const int rr = r0 - k;
				if (rr < 0) return INT_MIN;
				int s0, e0;
				ksw_band(rr, qlen, tlen, w, s0, e0, UNB);
				return rr * pitch + (i0 - (UNB ? (s0 & ~3) : (s0 & ~15))); // byte offset of column i0 in row rr
			}, pmat, -KSW_PMAT_PAD, p_hi, tile);
			__syncwarp();
			if (gl == 0) {
				const uint8_t *tb = (const uint8_t*)tile;
				while (i >= 0 && j >= 0 && i + j > r0 - 32) {
					const int r = i + j;
					int s0, e0;
					ksw_band(r, qlen, tlen, w, s0, e0, UNB);
					const int off = s0 & ~15, off_end = e0 | 15;
					int force_state = -1;
					if (i < off) force_state = 2;
					if (i > off_end) force_state = 1;
					const unsigned tmp = force_state < 0 ? tb[(r0 - r) * KSW_BTILE_ROW + 32 + (i0 & 3) - (i0 - i)] : 0u;
					if (state == 0) state = tmp & 7;
					else if (!((tmp >> (state + 2)) & 1)) state = 0;
					if (state == 0) state = tmp & 7;
					if (force_state >= 0) state = force_state;
					unsigned op;
					if (state == 0) { op = 0; --i; --j; }
					else if (state == 1 || state == 3) { op = 2; --i; }
					else { op = 1; --j; }
					if (op == cur_op) ++cur_len;
					else {
						if (cur_len) { if (n < cig_cap) cig[n++] = cur_len << 4 | cur_op; else ovf = 1; }
						cur_op = op; cur_len = 1;
					}
				}
			}
			i = __shfl_sync(FULL_MASK, i, lane & ~(G - 1)); j = __shfl_sync(FULL_MASK, j, lane & ~(G - 1));
			__syncwarp();
		}
		if (gl == 0) {
			// the two trailing pushes (:73-74) merge with an equal pending op exactly as ksw_push_cigar does
			if (i >= 0) {
				if (cur_op == 2) cur_len += i + 1;
				else { if (cur_len) { if (n < cig_cap) cig[n++] = cur_len << 4 | cur_op; else ovf = 1; } cur_op = 2; cur_len = i + 1; }
			}
			if (j >= 0) {
				if (cur_op == 1) cur_len += j + 1;
				else { if (cur_len) { if (n < cig_cap) cig[n++] = cur_len << 4 | cur_op; else ovf = 1; } cur_op = 1; cur_len = j + 1; }
			}
			if (cur_len) { if (n < cig_cap) cig[n++] = cur_len << 4 | cur_op; else ovf = 1; }
		}
	}
	n = __shfl_sync(FULL_MASK, n, lane & ~(G - 1));
	ovf = __shfl_sync(FULL_MASK, ovf, lane & ~(G - 1));
	out.n_cigar = n;
	if (ovf) out.status = KSW_ST_CIGCAP;
	__syncwarp();
}

// query-offset-limited view of the CIGAR (the `cigar` iterator of src/ksw2/ksw2.nim:22-33) over the REVERSED scratch:
// returns how many leading ops (in forward order) the iterator yields.
__device__ __forceinline__ int ksw_trunc_count(const uint32_t *cig_rev, int n, int max_q)
{
	const unsigned max_off = (unsigned)max_q;
	unsigned off = 0;
	int k = 0;
	for (; k < n; ++k) {
		if (off >= max_off) break;
		const uint32_t c = cig_rev[n - 1 - k];
		if ((c & 0xf) != 2) off += c >> 4;
	}
	return k;
}
