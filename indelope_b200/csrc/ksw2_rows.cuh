// indelope_b200/csrc/ksw2_rows.cuh -- kernel 2, unbanded call-site (the AL fallback, src/indelope.nim:317-318,343-344:
// w = -1, zdrop = -1) with the QUERY ROWS resident in registers.
//
// Same results as ksw_extz2_sse (src/ksw2/csrc/ksw2_extz2_sse.c:113-388, flag 0), bit for bit, for w < 0 and zdrop < 0.
// The SSE code indexes u, v, x, y by target column t; on anti-diagonal r the cell (t, j = r - t) reads x, v of the cell
// (t-1, j) -- same query row, previous diagonal -- and u, y of the cell (t, j-1) -- previous query row, previous diagonal.
// Unbanded, a read of <= 32 W bases has few rows and every row is live for tlen consecutive diagonals, so here a
// thread OWNS query rows: word w of the query (rows 4w .. 4w+3, one int8 lane each) belongs to thread w % 8 of the
// group of eight, slot w / 8.  x, v never move; u, y shift up by one row per diagonal: one PRMT inside a word, one
// shuffle between neighbouring threads.  Nothing of the recurrence touches shared memory: no ring, no addressing, no
// load/store per word and diagonal (the column-owned variant in ksw2.cuh spends 116 instructions per word, 33 of them on
// the recurrence; this one about 55).  The interleaved ownership keeps the eight threads busy on the ramps of the band:
// on diagonal r the live rows max(0, r-tlen+1) .. min(r, qlen-1) are a run of consecutive words, dealt round-robin.
//
// Exact scores (:312-349).  H(t, j) is a potential: u = H(t,j) - H(t-1,j) + (q+e), v = H(t,j) - H(t,j-1) + (q+e) are both
// differences of it (the boundary values v1 = q / 0 and the :212 patch encode H(-1, j) = -(q + e(j+1)), H(t, -1) likewise),
// so H can be carried along a row with u instead of down a column with v: g_j = H + (q+e)(r+1) + bias gets u8 added on
// every diagonal, as uint16 halves in registers.  Rows in flight before t = 0 are held at their boundary state; rows past
// t = tlen-1 and rows >= qlen compute real cells of the problem extended with zero codes (nobody reads them) and are
// masked out of the maximum.  The running maximum needs no exchange per diagonal: every thread keeps the best score of its
// own rows, the FIRST diagonal it was reached on and a snapshot of its scores there; the overall maximum was first
// reached on the smallest such diagonal among the threads that hold it, and the SSE tie order (:316-348: H[en0] first,
// then four strided accumulators, then the scalar tail) is applied to the snapshots once, after the last diagonal.
//
// The backtrack matrix is written p[r][j] (one byte per row, pitch 32 W: each group stores whole 32-byte sectors) and
// walked as ksw_backtrack (:47-79) through a 32 x 32 shared-memory tile, like the column-owned variant.
#pragma once
#include "ksw2.cuh"
#include "ksw2_rows_sched.cuh"

// reads of up to 32 W bases: W = 5 covers 160 bp and fits 80 registers (three CTAs per SM); 0 = not served by this variant
// (W = 8 works -- the tests ran it -- but needs 128 registers; longer reads take the column-owned variant)
__host__ __device__ inline int ksw_rows_w(int qlen) { return qlen <= 160 ? 5 : 0; }
// shared-memory bytes of the reversed, zero-padded target
__host__ __device__ inline size_t ksw_rows_snap_bytes(int W) { return (size_t)128 * ((2 * W + 3) / 4); } // score snapshots: (2 W + 3) / 4 uint4 per thread
__host__ __device__ inline size_t ksw_rows_stage_bytes(int W, int tlen) { return (size_t)((tlen + 64 * W + 8 + 3) & ~3) + 96 + ksw_rows_snap_bytes(W); } // + the bank stagger of the group + the snapshots
// bytes of backtrack matrix
__host__ __device__ inline size_t ksw_rows_p_bytes(int W, int qlen, int tlen) { return (size_t)(qlen + tlen - 1) * (size_t)(32 * W) + 2 * KSW_PMAT_PAD + 64; }
__host__ __device__ inline bool ksw_rows_params_ok(const KswParams &P)
{
	const int qe = P.q + P.e;
	int min_sc = P.mismatch < 0 ? P.mismatch : 0;
	if (P.match < min_sc) min_sc = P.match;
	return P.w < 0 && P.zdrop < 0 && P.match > 0 && P.match + 2 * qe <= 63 && P.q >= 0 && P.e >= 0 && P.q + 2 * P.e + min_sc >= 0 && -min_sc <= 2 * qe;
}

__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t s) { return __byte_perm(a, b, s); }
__device__ __forceinline__ uint32_t lds32(uint32_t addr) { uint32_t v; asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr)); return v; }

#define KSW_ROWS_TPAD 5u /* code of the target padding: matches no query code, so cells past the target end only lose score */
#define KSW_ROWS_QPAD 6u /* code of the query padding (rows >= qlen) */

// One packed word of four query rows on one diagonal: the recurrence of :262-284 in its carry-free form (every byte of a
// real cell is in [0, match + 2(q+e)] <= 63: sums stay below 128 and nothing carries between bytes; `chk` collects the
// inputs so that the caller can prove it after the fact), the backtrack word, and the exact scores g += u.
// FRONT: the word holds lanes outside the target (outside `m`): rows that have not reached t = 0 yet keep their boundary
// state (x = 0, v = q, y = 0, g = its initial value), rows past t = tlen-1 are parked in the same state; both stay out of
// the maximum.  One step from in-range inputs cannot carry between bytes, so a parked lane never disturbs its neighbours.
template <bool FRONT, bool WILD>
__device__ __forceinline__ void ksw_rows_word(const KswParams &P, uint32_t m, uint32_t pc, uint32_t tw, uint32_t qv,
                                              uint32_t &x, uint32_t &v, uint32_t &u, uint32_t &y, uint32_t &gx, uint32_t &gy, uint32_t &dm2, uint32_t &chk, uint32_t *pdst)
{
	const uint32_t Q4 = P.q_4;
	const uint32_t ut = prmt(u, pc, 0x2106), yt = prmt(y, pc, 0x2107); // u, y of rows 4w-1 .. 4w+2 (previous diagonal)
	uint32_t z0 = sel4(msb_to_mask4((tw ^ qv) + 0x7f7f7f7fu), P.misq_4, P.maxsc_4);
	if (WILD) z0 = sel4(msb_to_mask4(((tw ^ 0x04040404u) + 0x7f7f7f7fu) & ((qv ^ 0x04040404u) + 0x7f7f7f7fu)), z0, P.qe2_4); // a code 4 on either side scores 0 (:219,226)
	chk |= x | v; chk |= ut | yt; // the proof after the fact that the carry-free form was exact: 0.51 of 19.3 ms
	const uint32_t a = x + v, b = yt + ut;
	uint32_t mk = ge4_pos(z0, a);                   // z >= a
	uint32_t z = sel4(mk, z0, a);
	uint32_t d = ~mk & 0x01010101u;
	mk = ge4_pos(z, b);                             // z >= b
	d = sel4(mk, d, 0x02020202u);
	z = sel4(mk, z, b);
	// no z = min(z, match + 2(q+e)) of :132: on real cells a diagonal step gains at most the match score, so it never binds (DESIGN.md 4.2b)
	const uint32_t zh = z | KSW_H80;
	uint32_t un = (zh - v) ^ KSW_H80, vn = (zh - ut) ^ KSW_H80;
	z -= Q4;
	mk = ge4_pos(z, a);                             // z >= a: x = 0
	uint32_t xn = sel4(mk, z, a) - z; d |= ~mk & 0x08080808u;
	mk = ge4_pos(z, b);
	uint32_t yn = sel4(mk, z, b) - z; d |= ~mk & 0x10101010u;
	KSW_PSTORE(pdst, d);
	if (FRONT) {
		xn &= m; yn &= m; un &= m; vn = sel4(m, vn, Q4);
		gx += prmt(un, 0u, 0x4140); gy += prmt(un, 0u, 0x4342);
		dm2 = __vimax3_u16x2(dm2, gx & prmt(m, 0u, 0x1100), gy & prmt(m, 0u, 0x3322));
	} else {
		gx += prmt(un, 0u, 0x4140); gy += prmt(un, 0u, 0x4342);
		dm2 = __vimax3_u16x2(dm2, gx, gy);
	}
	x = xn; v = vn; u = un; y = yn;
}

// per-diagonal values shared by the slots of a thread (lq: qlen, 0 for a group without a live alignment)
struct KswRowsDiag { KswRowsAt at; int r, lq, tlen, gl, srcl, tsh; uint32_t bconst, taddr; uint8_t *prow; };

// The slots of one diagonal, unrolled by template recursion: every index into the register arrays is a compile-time
// constant from the start (a `#pragma unroll` loop around warp votes and shuffles is unrolled too late for the arrays to
// be promoted to registers).
template <int W, int S, bool WILD>
struct KswRowsSlots {
	static __device__ __forceinline__ void run(const KswParams &P, const KswRowsDiag &dg, const uint32_t (&C)[W], const uint32_t (&qw)[W], uint32_t (&x)[W], uint32_t (&v)[W],
	                                           uint32_t (&u)[W], uint32_t (&y)[W], uint32_t (&gx)[W], uint32_t (&gy)[W], uint32_t &dm2, uint32_t &chk)
	{
		if (ksw_rows_live(dg.at, S)) {
			uint32_t send = C[S];
			if (S > 0 && dg.gl == 7) send = C[S > 0 ? S - 1 : 0];
			uint32_t pc = __shfl_sync(FULL_MASK, send, dg.srcl);
			if (S == 0 && dg.gl == 0) pc = dg.bconst;
			if (ksw_rows_interior(dg.at, S)) {
				// every thread of the warp has all four lanes of the slot inside the target
				const uint32_t tw = __funnelshift_r(lds32(dg.taddr + 32 * S), lds32(dg.taddr + 32 * S + 4), dg.tsh); // target codes met by rows 4w .. 4w+3
				ksw_rows_word<false, WILD>(P, 0u, pc, tw, qw[S], x[S], v[S], u[S], y[S], gx[S], gy[S], dm2, chk, (uint32_t*)(dg.prow + 32 * S));
			} else if (ksw_rows_lane_on(dg.r, dg.gl, S, dg.lq, dg.tlen)) {
				// the ramps: the word may hold lanes in front of t = 0 (the word of row r) or past t = tlen-1 (the word of row
				// r - tlen); those lanes keep a fixed in-range state and stay out of the maximum.  A word wholly inside the target
				// gets m = all ones here, which makes the masked word the plain one: where groups of different shapes overlap it
				// costs the few mask instructions, never a different result
				const int lo = dg.r - 4 * dg.gl - 32 * S; // t of row 4w on this diagonal; lane c is row 4w + c at t = lo - c
				uint32_t m = lo >= 3 ? 0xffffffffu : (lo < 0 ? 0u : (0xffffffffu >> (8 * (3 - lo)))); // a word wholly in front of t = 0 is parked as a whole
				const int cf = lo - (dg.tlen - 1);
				if (cf > 0) m = cf > 3 ? 0u : (m & (0xffffffffu << (8 * cf)));                            // ... and so is one wholly past the end
				const uint32_t tw = __funnelshift_r(lds32(dg.taddr + 32 * S), lds32(dg.taddr + 32 * S + 4), dg.tsh);
				ksw_rows_word<true, WILD>(P, m, pc, tw, qw[S], x[S], v[S], u[S], y[S], gx[S], gy[S], dm2, chk, (uint32_t*)(dg.prow + 32 * S));
			}
		}
		KswRowsSlots<W, S + 1, WILD>::run(P, dg, C, qw, x, v, u, y, gx, gy, dm2, chk);
	}
};
template <int W, bool WILD>
struct KswRowsSlots<W, W, WILD> {
	static __device__ __forceinline__ void run(const KswParams &, const KswRowsDiag &, const uint32_t (&)[W], const uint32_t (&)[W], uint32_t (&)[W], uint32_t (&)[W],
	                                           uint32_t (&)[W], uint32_t (&)[W], uint32_t (&)[W], uint32_t (&)[W], uint32_t &, uint32_t &) {}
};

// ALL 32 threads of a warp call this together (4 groups of 8 threads, one alignment per group; valid = 0 for a group
// without one).  The caller has checked ksw_rows_params_ok, qlen <= 32 W, ksw_rows_stage_bytes <= M.region_bytes and
// ksw_rows_p_bytes <= M.p_cap for every valid group.
template <int W, bool EZ_FULL>
__device__ void ksw2_rows(bool valid, int qlen, const KswQuery query, int tlen, const uint8_t *target, const KswParams P, const KswMem M, KswOut &out)
{
	constexpr int PITCH = 32 * W, PADL = 32 * W;
	const int lane = lane_id(), gl = lane & 7;
	ksw_reset(out);
	const int qe = P.q + P.e, gbias = 2 * qe;
	bool live = valid;
	if (live) {
		if (qlen <= 0 || tlen <= 0) { out.status = KSW_ST_EARLY; live = false; }                                     // :147
		else if (qlen > 32 * W || ksw_rows_stage_bytes(W, tlen) > (size_t)M.region_bytes) { out.status = KSW_ST_RCAP; live = false; }
		else if (ksw_rows_p_bytes(W, qlen, tlen) > M.p_cap) { out.status = KSW_ST_PCAP; live = false; }
		else if ((long long)(qlen + tlen + 2) * qe + (long long)(qlen < tlen ? qlen : tlen) * P.match + gbias + (long long)P.q * 32 * W >= 0xF000) { out.status = KSW_ST_HCAP; live = false; }
	}
	const bool run = live;
	const int nr = live ? qlen + tlen - 1 : 0;
	uint8_t *pmat = M.pmat + KSW_PMAT_PAD;
	// the reversed target, padded on both sides: byte PADL + k holds target[tlen-1-k].  The four groups of a warp read the same
	// relative words at the same time and their regions are a multiple of 128 bytes apart: group k starts 8 k words in
	uint32_t *TW = (uint32_t*)((unsigned char*)M.xvuy + 32 * ((lane >> 3) & 3));

	bool wild = false;
	if (live) {
		const int total = (int)(ksw_rows_stage_bytes(W, tlen) - 96 - ksw_rows_snap_bytes(W));
		for (int i = gl * 4; i < total; i += 32) {
			uint32_t wv = 0;
#pragma unroll
			for (int c = 0; c < 4; ++c) {
				const int k = i + c - PADL;
				wv |= ((k >= 0 && k < tlen) ? (uint32_t)target[tlen - 1 - k] : KSW_ROWS_TPAD) << (8 * c);
			}
			TW[i >> 2] = wv; wild |= ksw_has4(wv);
		}
	}
	// rows in registers: slot s of this thread is query word 8 s + gl
	uint32_t qw[W], x[W], v[W], u[W], y[W], gx[W], gy[W];
#pragma unroll
	for (int s = 0; s < W; ++s) {
		const int j0 = 4 * (8 * s + gl);
		uint32_t qv = 0;
#pragma unroll
		for (int c = 0; c < 4; ++c) {
			const uint32_t code = (live && j0 + c < qlen) ? (uint32_t)ksw_query_code(query, j0 + c) : KSW_ROWS_QPAD;
			wild |= code == 4u; qv |= code << (8 * c);
		}
		qw[s] = qv;
		x[s] = 0u; y[s] = 0u; u[s] = 0u;
		v[s] = P.q_4;                               // v1 = q for a row that starts on a diagonal r > 0 (:211)
		const int i0 = P.q * (j0 - 1) - P.e + gbias; // g of row j before its first cell: H(-1, j) + (q+e) j + bias
		gx[s] = (uint32_t)(i0 & 0xffff) | ((uint32_t)((i0 + P.q) & 0xffff) << 16);
		gy[s] = (uint32_t)((i0 + 2 * P.q) & 0xffff) | ((uint32_t)((i0 + 3 * P.q) & 0xffff) << 16);
	}
	if (gl == 0) v[0] &= 0xffffff00u;              // ... and 0 for row 0 on diagonal 0
	const bool wild_any = __any_sync(FULL_MASK, wild); // a code 4 anywhere in the four alignments: the scores take the wildcard mask
	__syncwarp();

	// Which diagonals run which slot, and how (ksw2_rows_sched.cuh).  The slots that hold query rows are the same for every thread of a
	// group -- in the last one some threads hold only padding rows (code 6: real cells of the query-extended problem that can only lose
	// score), so that the eight threads always store a whole 32-byte sector.  Per slot and diagonal, three cases, all decided by values
	// the same in every thread of the warp: outside the live window the slot is skipped; inside the interior window every thread runs
	// its word without masks or tests; in between (the ramps) each thread tests its own word and masks the lanes outside the target.
	// A group without a live alignment (valid == false, or an early KSW_ST_* status) counts as qlen = tlen = 0, which empties the
	// interior window of the whole warp: its threads only ever see the ramp path, fail the lane test there (qlen = 0), and so never form
	// a target address or a backtrack-matrix address, exactly as before.  At call-site B such a warp is mostly the last, partly filled one
	// of a launch, or one holding tasks with qlen or tlen 0 (al_kernel clamps a negative tlen to 0): those have no diagonals and get the
	// sort keys 0..15, below every task that has one, so they fill warps of their own, and at most one warp per launch mixes them with
	// live alignments.
	const int lq = live ? qlen : 0;
	KswRowsWarp ws;
	ws.qmin = __reduce_min_sync(FULL_MASK, lq); ws.qmax = __reduce_max_sync(FULL_MASK, lq);
	ws.tmin = __reduce_min_sync(FULL_MASK, live ? tlen : 0); ws.tmax = __reduce_max_sync(FULL_MASK, live ? tlen : 0);
	// score snapshots of this thread (taken when its best score rises): the last bytes of the group's region, 16 bytes per
	// thread and vector, so that a group's store is one conflict-free 128-byte line; only the owner ever reads them back
	constexpr int NSV = (2 * W + 3) / 4;
	uint4 *SNAP = (uint4*)((unsigned char*)M.xvuy + (M.region_bytes - (int)ksw_rows_snap_bytes(W))) + gl;
	const int srcl = (lane & ~7) | ((gl + 7) & 7); // the thread that owns the word below mine
	int tbest = 0, tr = -1;                        // best exact score over my rows so far, the first diagonal it was seen on
	int mte = KSW_NEG_INF, mte_r = -1, mqe = KSW_NEG_INF, mqe_t = -1, score = KSW_NEG_INF;
	const int jl = qlen - 1;                       // the last query row: slot (jl >> 5) of thread ((jl >> 2) & 7), lane jl & 3
	const bool own_last = live && ((jl >> 2) & 7) == gl;
	uint8_t *prow = pmat + 4 * gl;
	const int tb = PADL + tlen - 1 + 4 * gl;       // word 8 s + gl meets the reversed-target bytes tb - r + 32 s ...
	const uint32_t tw_sh = (uint32_t)__cvta_generic_to_shared(TW);
	uint32_t chk = 0;

	const int nr_all = (int)__reduce_max_sync(FULL_MASK, (unsigned)nr); // the warp runs until its longest alignment ends
	for (int r = 0; r < nr_all; ++r, prow += PITCH) {
		const bool act = r < nr;
		const int tbase = tb - r;
		const uint32_t taddr = tw_sh + (uint32_t)(tbase & ~3);
		const int tsh = 8 * (tbase & 3);
		uint32_t C[W];
#pragma unroll
		for (int s = 0; s < W; ++s) C[s] = prmt(u[s], y[s], 0x7300); // byte 2 = u of my top lane, byte 3 = y of it
		const uint32_t bconst = r ? ((uint32_t)(P.q & 0xff) << 16) : 0u; // :212  u[r] = q (0 on diagonal 0), y[r] = 0
		uint32_t dm2 = 0;
		// only threads with a live word run a slot: whole sectors on the band's ramps cut DRAM fill reads but cost 1.2 ms (DESIGN.md 4.2c)
		KswRowsDiag dg;
		dg.at = ksw_rows_at(ws, r); dg.r = r; dg.lq = lq; dg.tlen = tlen; dg.gl = gl; dg.srcl = srcl; dg.bconst = bconst; dg.taddr = taddr; dg.tsh = tsh; dg.prow = prow;
		if (wild_any) KswRowsSlots<W, 0, true>::run(P, dg, C, qw, x, v, u, y, gx, gy, dm2, chk);
		else KswRowsSlots<W, 0, false>::run(P, dg, C, qw, x, v, u, y, gx, gy, dm2, chk);
		const int goff = qe * (r + 1) + gbias;
		{
			const int dm = (int)((dm2 & 0xffffu) > (dm2 >> 16) ? (dm2 & 0xffffu) : (dm2 >> 16)) - goff;
			if (dm > tbest) { // strictly better than anything my rows have seen (:92 of ksw_apply_zdrop, per thread)
				tbest = dm; tr = r;
#pragma unroll
				for (int k = 0; k < NSV; ++k) {
					uint32_t q4[4];
#pragma unroll
					for (int c = 0; c < 4; ++c) { const int e = 4 * k + c; q4[c] = e < 2 * W ? ((e & 1) ? gy[e >> 1] : gx[e >> 1]) : 0u; }
					SNAP[8 * k] = make_uint4(q4[0], q4[1], q4[2], q4[3]);
				}
			}
		}
		if (EZ_FULL) {
			if (act && r >= tlen - 1) { // en0 == tlen-1: H[en0] is the cell of row r - tlen + 1 (:351-352,356-357)
				const int jt = r - tlen + 1;
				if (((jt >> 2) & 7) == gl) {
					uint32_t w2 = 0;
#pragma unroll
					for (int s = 0; s < W; ++s) w2 |= ((jt & 2) ? gy[s] : gx[s]) & (0u - (uint32_t)(s == (jt >> 5))); // constant indices only
					const int hen = (int)((w2 >> (16 * (jt & 1))) & 0xffffu) - goff;
					if (hen > mte) { mte = hen; mte_r = r; }
				}
			}
			if (own_last && act && r >= jl) { // r - st0 == qlen-1: H[st0] is the cell of the last row (:353-354)
				uint32_t w2 = 0;
#pragma unroll
				for (int s = 0; s < W; ++s) w2 |= ((jl & 2) ? gy[s] : gx[s]) & (0u - (uint32_t)(s == (jl >> 5)));
				const int h = (int)((w2 >> (16 * (jl & 1))) & 0xffffu) - goff;
				if (h > mqe) { mqe = h; mqe_t = r - jl; }
				if (r == nr - 1) score = h;
			}
		}
	}
	// every byte the recurrence read was in [0, 63] (the carry-free form is exact): anything else is reported, never returned
	if (ksw_group_any((chk & 0xc0c0c0c0u) != 0u, lane) && run) out.status = KSW_ST_HCAP;
	// the overall maximum: best value, then the first diagonal it was reached on, then the SSE tie order on that diagonal
	{
		const unsigned V = ksw_group_max((unsigned)tbest);
		const unsigned rs = ksw_group_min((run && (unsigned)tbest == V && tr >= 0) ? (unsigned)tr : 0x7fffffffu);
		const bool have = run && V > 0u && rs != 0x7fffffffu;
		const int r = have ? (int)rs : 0;
		int st0 = 0, en0 = 0;
		if (have) ksw_band(r, qlen, tlen, 0, st0, en0, true);
		const int en1 = st0 + (((en0 - st0) >> 2) << 2);
		const unsigned want = V + (unsigned)(qe * (r + 1) + gbias);
		unsigned best = 0xffffffffu;
		if (have && (unsigned)tbest == V && tr == r) {
			uint32_t sn[4 * NSV];
#pragma unroll
			for (int k = 0; k < NSV; ++k) { const uint4 q4 = SNAP[8 * k]; sn[4 * k] = q4.x; sn[4 * k + 1] = q4.y; sn[4 * k + 2] = q4.z; sn[4 * k + 3] = q4.w; }
#pragma unroll
			for (int s = 0; s < W; ++s) {
#pragma unroll
				for (int c = 0; c < 4; ++c) {
					const int j = 4 * (8 * s + gl) + c, t = r - j;
					const unsigned val = (sn[2 * s + (c >> 1)] >> (16 * (c & 1))) & 0xffffu;
					if (j < qlen && t >= st0 && t <= en0 && val == want) {
						const unsigned rk = t == en0 ? 0u : ksw_tie_rank(t, st0, en1);
						best = rk < best ? rk : best;
					}
				}
			}
		}
		const unsigned rk = ksw_group_min(best); // every lane of the warp takes part
		if (have) {
			const int t = rk == 0u ? en0 : st0 + (int)((rk - 1) & 0xfffffu);
			out.max = (int)V; out.max_t = t; out.max_q = r - t;
		}
	}
	if (EZ_FULL) {
		// end-of-target scores: the first diagonal with the best H[tlen-1] (:351-352; mte_q = r - en with the ROUNDED en)
		const unsigned bias = 0x40000000u;
		const unsigned mv = ksw_group_max((unsigned)(mte + (int)bias));
		const unsigned mr = ksw_group_min((mte_r >= 0 && (unsigned)(mte + (int)bias) == mv) ? (unsigned)mte_r : 0x7fffffffu);
		if (run && mr != 0x7fffffffu) { out.mte = (int)(mv - bias); out.mte_q = (int)mr - ((tlen - 1) | 15); }
		const int ol = (lane & ~7) | ((jl >> 2) & 7);
		const int a = __shfl_sync(FULL_MASK, mqe, ol & 31), b = __shfl_sync(FULL_MASK, mqe_t, ol & 31), c = __shfl_sync(FULL_MASK, score, ol & 31);
		if (run) { out.mqe = a; out.mqe_t = b; out.score = c; }
	}
	if (run) out.cells = (long long)qlen * (long long)tlen;
	__syncwarp();
	// ksw_backtrack :47-79 from (tlen-1, qlen-1) (never z-dropped: the band is the whole anti-diagonal), is_rot = 1.  Unbanded,
	// the path never leaves [off, off_end], so no state is forced.  In (r, j) coordinates a step back keeps j or lowers it by
	// one, so the rows r0 .. r0-31 can only be entered at columns j0-k .. j0: the group prefetches that triangle.
	// The four groups of the warp walk in lockstep (full-warp barriers; a group whose path has ended idles): with per-group
	// barriers the four walkers drift apart and the warp runs them one after the other.  (The whole traceback is 3.2 of the
	// 20.0 ms of al_kernel: tile prefetch 1.7, walkers 1.5.)
	int i = run ? tlen - 1 : -1, j = run ? qlen - 1 : -1, n = 0, ovf = 0;
	{
		uint32_t *tile = (uint32_t*)M.xvuy;
		uint32_t *cig = M.cig; const int cig_cap = M.cig_cap;
		int state = 0;
		unsigned cur_op = 0xffu, cur_len = 0;
		const int p_hi = (qlen + tlen - 1) * PITCH + KSW_PMAT_PAD;
		while (__any_sync(FULL_MASK, i >= 0 && j >= 0)) {
			const bool more = i >= 0 && j >= 0;
			const int j0 = j, r0 = i + j;
			ksw_tile_fetch(more, [&](int k) -> int { return r0 - k < 0 ? INT_MIN : (r0 - k) * PITCH + j0; }, pmat, -KSW_PMAT_PAD, p_hi, tile);
			__syncwarp();
			if (gl == 0) {
				const uint8_t *tbp = (const uint8_t*)tile;
				while (i >= 0 && j >= 0 && i + j > r0 - 32) {
					const int r = i + j;
					const unsigned tmp = tbp[(r0 - r) * KSW_BTILE_ROW + 32 + (j0 & 3) - (j0 - j)];
					if (state == 0) state = tmp & 7;
					else if (!((tmp >> (state + 2)) & 1)) state = 0;
					if (state == 0) state = tmp & 7;
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
			i = __shfl_sync(FULL_MASK, i, lane & ~7); j = __shfl_sync(FULL_MASK, j, lane & ~7);
			__syncwarp();
		}
		if (gl == 0) {
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
	n = __shfl_sync(FULL_MASK, n, lane & ~7);
	ovf = __shfl_sync(FULL_MASK, ovf, lane & ~7);
	out.n_cigar = n;
	if (ovf) out.status = KSW_ST_CIGCAP;
	__syncwarp();
}

// which variant a warp takes: every valid group votes the W it needs (0: no alignment, 99: not served), the warp runs the
// widest one if all its groups fit
__device__ __forceinline__ int ksw_rows_pick(bool valid, int qlen, int tlen, const KswParams &P, const KswMem &M)
{
	int need = 0;
	if (valid && qlen > 0 && tlen > 0) { need = ksw_rows_w(qlen); if (need == 0) need = 99; }
	const int w = (int)__reduce_max_sync(FULL_MASK, (unsigned)need);
	if (w == 0) return 5;
	if (w > 5 || !ksw_rows_params_ok(P)) return 0;
	const bool ok = !(valid && qlen > 0 && tlen > 0) || (ksw_rows_stage_bytes(w, tlen) <= (size_t)M.region_bytes && ksw_rows_p_bytes(w, qlen, tlen) <= M.p_cap);
	return __all_sync(FULL_MASK, ok) ? w : 0;
}
