// indelope_b200/csrc/ksw2_rows_sched.cuh -- which diagonals the row-owned variant of kernel 2 (ksw2_rows.cuh) runs a slot on, and
// whether it needs masks there.  Slot S of thread gl of a group holds query rows 32 S + 4 gl .. +3; on diagonal r the first of them
// meets target column lo = r - 32 S - 4 gl.  The word has a lane inside the target when lo is in [0, tlen + 2] (and r < qlen + tlen - 1,
// S < the group's slot count (qlen + 31) / 32), and all four lanes when lo is in [3, tlen - 1].  None of this depends on the data, so
// for a group the answer per slot is two windows of diagonals:
//   live      [32 S, min(32 S + tlen + 31, qlen + tlen - 1))   some thread has a lane of the slot inside the target
//                                                             (thread gl is live on [32 S + 4 gl, 32 S + 4 gl + tlen + 2]: runs
//                                                             four diagonals apart and at least four long, so their union is one run)
//   interior  [32 S + 31, 32 S + tlen)                        every thread has the slot wholly inside it (thread gl on
//                                                             [32 S + 4 gl + 3, 32 S + 4 gl + tlen - 1]; 32 S + tlen <= qlen + tlen - 1)
// both empty when S >= (qlen + 31) / 32.  The windows of one slot start at the same diagonal in every group, and both ends grow with
// qlen and tlen, so for the four groups of a warp
//   - the intersection of the interior windows is the interior window of (min qlen, min tlen), and
//   - the union of the live windows lies inside the live window of (max qlen, max tlen) (the warp's last diagonal caps it).
// Tasks are sorted by length, so the groups of a warp are mostly alike; where they are not, the live window of the extremes holds a
// few diagonals on which no thread has a lane of the slot: the warp shuffles, every thread fails its lane test, and no word runs.
// The warp computes the four extremes once per alignment and tests r against these windows on every diagonal: the operands are the
// same in every thread, so the tests run on the uniform datapath.
//
// The same source compiles as plain C++: tests/ build it with g++ and check it against the per-diagonal rule of every thread.
#pragma once

#ifdef __CUDACC__
#define KSW_ROWS_HD __host__ __device__ __forceinline__
#else
#define KSW_ROWS_HD static inline
#endif

// the extremes of the shapes of a warp's groups; a group without a live alignment counts as qlen = tlen = 0 (the minima of such a
// warp are 0: it has no interior window)
struct KswRowsWarp { int qmin, tmin, qmax, tmax; };

// the warp on diagonal r: r against the ends of its windows.  The differences are taken once per diagonal, so that each slot compares
// them with a constant; a difference per slot would be folded into a bound per slot, held in registers through the whole loop.
struct KswRowsAt { int r, ron, rin, qmin, qmax; };
KSW_ROWS_HD KswRowsAt ksw_rows_at(const KswRowsWarp &w, int r) { KswRowsAt a = {r, r - w.tmax - 31, r - w.tmin, w.qmin, w.qmax}; return a; }
// r is in the live window of slot S of some group
KSW_ROWS_HD bool ksw_rows_live(const KswRowsAt &a, int S) { return a.r >= 32 * S && a.ron < 32 * S && 32 * S < a.qmax; }
// r is in the interior window of slot S of every group
KSW_ROWS_HD bool ksw_rows_interior(const KswRowsAt &a, int S) { return a.r >= 32 * S + 31 && a.rin < 32 * S && 32 * S < a.qmin; }

// the word of slot S of thread gl has a lane inside the target on diagonal r (qlen = 0: no live alignment)
KSW_ROWS_HD bool ksw_rows_lane_on(int r, int gl, int S, int qlen, int tlen)
{
	const int lo = r - 32 * S - 4 * gl;
	return qlen > 0 && tlen > 0 && r < qlen + tlen - 1 && 32 * S < qlen && lo >= 0 && lo <= tlen + 2;
}
