// tests/native/rows_sched_host.cpp -- TEST BUILD of indelope_b200/csrc/ksw2_rows_sched.cuh as plain C++: the slot windows the row-owned
// variant of kernel 2 steers its diagonal loop by, checked against the rule the loop used before them, restated here per thread and
// diagonal.  Not part of the product libraries.
#include <cstdint>
#include "ksw2_rows_sched.cuh"

namespace {

const int W = 5;   // slots per thread of ksw2_rows<5>

// the per-diagonal rule of one thread: onm bit s = slot s has a lane inside the target, pm bit s = it has lanes outside it as well
void old_rule(int r, int gl, int lq, int tlen, unsigned &onm, unsigned &pm)
{
	const int nr = lq ? lq + tlen - 1 : 0, nsq = lq ? (lq + 31) >> 5 : 0;
	const bool act = r < nr;
	const int lo0 = r - 4 * gl;
	int s_hi = lo0 >> 5, s_lo = (lo0 - tlen + 29) >> 5;
	s_hi = s_hi < nsq ? s_hi : nsq - 1; s_lo = s_lo > 0 ? s_lo : 0;
	onm = 0; pm = 0;
	if (act && s_hi >= s_lo) {
		onm = ((2u << s_hi) - 1u) & ~((1u << s_lo) - 1u);
		if (lo0 - 32 * s_hi < 3) pm = 1u << s_hi;
		if (lo0 - 32 * s_lo > tlen - 1) pm |= 1u << s_lo;
	}
}

}  // namespace

extern "C" {

// One warp of four groups (valid[g], qlen[g], tlen[g]), every diagonal it runs.  Counts into out[0..5]:
//   0  a thread's onm bit set outside the warp's live window
//   1  the interior window holding a thread whose onm bit is clear or whose pm bit is set
//   2  ksw_rows_lane_on differing from the onm bit
//   3  (slot, diagonal) pairs in the interior window, 4 pairs in the live window, 5 onm bits set (how much was checked)
void idl_test_rows_warp(const int *valid, const int *qlen, const int *tlen, long long *out)
{
	int lq[4], nr_all = 0;
	KswRowsWarp w = {1 << 30, 1 << 30, 0, 0};
	for (int g = 0; g < 4; ++g) {
		const bool live = valid[g] && qlen[g] > 0 && tlen[g] > 0;   // an early status leaves a group without a live alignment
		lq[g] = live ? qlen[g] : 0;
		const int lt = live ? tlen[g] : 0;
		w.qmin = lq[g] < w.qmin ? lq[g] : w.qmin; w.qmax = lq[g] > w.qmax ? lq[g] : w.qmax;
		w.tmin = lt < w.tmin ? lt : w.tmin; w.tmax = lt > w.tmax ? lt : w.tmax;
		const int nr = live ? qlen[g] + tlen[g] - 1 : 0;
		nr_all = nr > nr_all ? nr : nr_all;
	}
	for (int r = 0; r < nr_all; ++r) {
		const KswRowsAt at = ksw_rows_at(w, r);
		for (int S = 0; S < W; ++S) {
			const bool lv = ksw_rows_live(at, S), in = ksw_rows_interior(at, S);
			out[3] += in; out[4] += lv;
			for (int g = 0; g < 4; ++g) {
				if (g && valid[g] == valid[g - 1] && qlen[g] == qlen[g - 1] && tlen[g] == tlen[g - 1]) continue;   // the same group again
				for (int gl = 0; gl < 8; ++gl) {
					unsigned onm, pm;
					old_rule(r, gl, lq[g], tlen[g], onm, pm);
					const bool on = (onm >> S) & 1u, part = (pm >> S) & 1u;
					out[5] += on;
					if (on && !lv) ++out[0];
					if (in && (!on || part)) ++out[1];
					if (ksw_rows_lane_on(r, gl, S, lq[g], tlen[g]) != on) ++out[2];
				}
			}
		}
	}
}

// every shape qlen 1..qmax, tlen 1..tmax, as a warp of four equal groups and as one group beside three without an alignment
void idl_test_rows_shapes(int qmax, int tmax, long long *out)
{
	for (int q = 1; q <= qmax; ++q)
		for (int t = 1; t <= tmax; ++t) {
			const int v4[4] = {1, 1, 1, 1}, q4[4] = {q, q, q, q}, t4[4] = {t, t, t, t};
			idl_test_rows_warp(v4, q4, t4, out);
			const int v1[4] = {1, 0, 0, 0}, q1[4] = {q, 0, 0, 0}, t1[4] = {t, 0, 0, 0};
			idl_test_rows_warp(v1, q1, t1, out);
		}
}

}
