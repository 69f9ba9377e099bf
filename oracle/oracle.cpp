// oracle/oracle.cpp -- TEST INFRASTRUCTURE (CPU oracle), never linked into the product.
//
// Line-by-line CPU restatement of indelope's per-region calling path:
//   src/contig.nim:27-281          slide-and-vote assembler
//   src/indelope.nim:23-38         read quality trim
//   src/indelope.nim:118-132       get_min_flank
//   src/indelope.nim:157-199       assemble, count_flanked_cigar
//   src/indelope.nim:201-428       callsemble (k-mer selection, counting, AL fallback, filters)
//   src/indelope.nim:49-116,598-608  Variant text and order-dependent dedup
//   src/ksw2/ksw2.nim:17-33,71-91,127-164  CIGAR iterators, encode, align_to
//   src/genotyper.nim:16-47        genotype likelihoods and text
// The DP itself is oracle/ksw2_lane.c (own restatement) or, when orc_params_t.use_ref_ksw2 is
// set, the reference's own C file compiled into oracle/_ref/libksw2_ref.so.
//
// Parity status: the assembler, ksw2 and genotyper parts are pinned by the reference's in-file
// known-answer tests (tests/test_oracle_kat.py) and, for ksw2, by fuzzing against the compiled
// reference.  `kmer.mincode` / `kmer.dists` come from the un-vendored, un-pinned nimble package
// "kmer" (indelope.nimble:10-11): their semantics are DECLARED (SURVEY.md appendix D), so the
// AKE/RKE values and the `mean(adists) < 5` filter are "parity unpinned".  Nothing in the
// reference tests callsemble itself; it is pinned only by the source text cited above.
#include <algorithm>
#include <chrono>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <dlfcn.h>
#include <memory>
#include <set>
#include <string>
#include <thread>
#include <vector>
#include "oracle.h"

namespace {

typedef void (*ref_ksw2_fn)(int, const uint8_t*, int, const uint8_t*, int8_t, int8_t, int8_t, int8_t, int, int, int,
                            orc_ez_t*, uint32_t*, int);
ref_ksw2_fn g_ref_ksw2 = nullptr;

const int64_t UNALIGNED = INT64_MIN; // src/contig.nim:27

struct Counters {
	int64_t slide_calls = 0, offsets = 0, char_compares = 0, exhaustive = 0;
	int64_t contigs_pre = 0, contigs_post = 0, dp_a = 0, dp_b = 0, cells_a = 0, cells_b = 0;
	int64_t events = 0, kmer_reads = 0, kmer_windows = 0, kmer_bytes = 0, al_events = 0;
	int64_t corrections = 0, vote_invariant_violations = 0, left_merges = 0, merges = 0;
};

// ---------------------------------------------------------------------------------------------
// src/contig.nim
// ---------------------------------------------------------------------------------------------
struct Contig { // :7-15
	std::string seq;
	std::vector<uint32_t> sup;
	int64_t nreads = 0;
	int64_t start = 0;
	int64_t len() const { return (int64_t)seq.size(); }
};
typedef std::shared_ptr<Contig> CP;

struct Corr { int64_t qoff, toff; bool qbest; }; // :17
struct Match { // :21
	int64_t matches = 0, offset = 0, mismatches = 0;
	std::vector<Corr> corrections;
	int64_t contig_i = 0;
	bool aligned() const { return offset != UNALIGNED; } // :29-30
};

// :44-47 (uint32 arithmetic for the support products, int for the read counts)
bool allowable_mismatch(uint32_t qsup, uint32_t tsup, int64_t qreads, int64_t treads)
{
	return ((qsup < 3u && tsup > 3u * qsup && qreads > 3 * (int64_t)qsup) ||
	        (tsup < 3u && qsup > 3u * tsup && treads > 3 * (int64_t)tsup));
}
// :287-290, the rule the reference's own unit tests use
bool allow_test(uint32_t qsup, uint32_t tsup, int64_t, int64_t)
{
	return ((qsup < 3u && tsup > 3u * qsup) || (tsup < 3u && qsup > 3u * tsup));
}
typedef bool (*allowed_fn)(uint32_t, uint32_t, int64_t, int64_t);

// :49-68
void trim_contig(Contig &c, int64_t min_support)
{
	int64_t a = 0;
	while (a < c.len() - 1 && c.sup[a] < (uint32_t)min_support) a += 1;
	c.start += a;
	if (a >= c.len() - 1) {
		c.seq.clear(); c.sup.clear(); c.nreads = 0;
		return;
	}
	int64_t b = c.len() - 1;
	while (c.sup[b] < (uint32_t)min_support && b > a) b -= 1;
	// `if a > 0 or b <= c.len - 1` (:66) is always true
	c.sup = std::vector<uint32_t>(c.sup.begin() + a, c.sup.begin() + b + 1);
	c.seq = c.seq.substr(a, b - a + 1);
}

// :70-141
Match slide_align(const Contig &q, const Contig &t, int64_t min_overlap, int64_t max_mismatch, allowed_fn allowed, Counters *cn)
{
	int64_t omin = -(q.len() - min_overlap);
	int64_t omax = t.len() - min_overlap;
	int64_t obest = UNALIGNED;
	int64_t best_ma = min_overlap - 1;
	int64_t best_mm = max_mismatch + 1;
	std::vector<Corr> best_correction, correction;
	int64_t qo, to, mm, ma;
	if (cn) cn->slide_calls++;
	for (int64_t o = 0; o <= omax; ++o) {
		correction.clear();
		qo = 0; to = o; mm = 0; ma = 0;
		if (cn) { cn->offsets++; int64_t ov = std::min(q.len(), t.len() - o); if (ov > 0) cn->exhaustive += ov; }
		while (qo < q.len() && to < t.len()) {
			if (cn) cn->char_compares++;
			if (q.seq[qo] != t.seq[to]) {
				if (!allowed(q.sup[qo], t.sup[to], q.nreads, t.nreads)) {
					mm += 1;
					if (mm > max_mismatch) break;
				} else { correction.push_back(Corr{qo, to, q.sup[qo] > t.sup[to]}); if (cn && !(q.nreads >= 4 && t.nreads >= 4)) cn->vote_invariant_violations++; }
			} else ma += 1;
			qo += 1; to += 1;
		}
		if (mm <= max_mismatch && (ma > best_ma || (ma == best_ma && mm < best_mm))) {
			best_ma = ma; best_mm = mm; obest = o; best_correction = correction;
		}
	}
	int64_t aomin = omin < 0 ? -omin : omin;
	for (int64_t o = 1; o <= aomin; ++o) { // :114
		correction.clear();
		qo = o; to = 0; mm = 0; ma = 0;
		if (cn) { cn->offsets++; int64_t ov = std::min(q.len() - o, t.len()); if (ov > 0) cn->exhaustive += ov; }
		while (qo < q.len() && to < t.len()) {
			if (cn) cn->char_compares++;
			if (q.seq[qo] != t.seq[to]) {
				if (!allowed(q.sup[qo], t.sup[to], q.nreads, t.nreads)) {
					mm += 1;
					if (mm > max_mismatch) break;
				} else { correction.push_back(Corr{qo, to, q.sup[qo] > t.sup[to]}); if (cn && !(q.nreads >= 4 && t.nreads >= 4)) cn->vote_invariant_violations++; }
			} else ma += 1;
			qo += 1; to += 1;
		}
		if (mm <= max_mismatch && (ma > best_ma || (ma == best_ma && mm < best_mm))) {
			best_ma = ma; best_mm = mm; obest = -o; best_correction = correction;
		}
	}
	Match m;
	m.matches = best_ma; m.offset = obest; m.mismatches = best_mm; m.corrections = best_correction; m.contig_i = -1;
	return m;
}

// :143-150
CP make_contig(const std::string &dna, int64_t start, uint32_t support = 1)
{
	CP o = std::make_shared<Contig>();
	o->seq = dna; o->sup.assign(dna.size(), support); o->nreads = (int64_t)support; o->start = start;
	return o;
}

// the capacity limits the device enforces per region (dump bit 64): the longest contig reached at any point of assemble + combine
// (a trimmed read or the product of a merge, against idl_params.max_contig_len) and the most voting sites of one merge (IDL_MAX_CORRECTIONS)
struct Limits { int64_t max_len = 0, max_corr = 0; };
thread_local Limits *g_limits = nullptr;

// :156-222
void insert_contig(Contig &t, Contig &q, const Match &m)
{
	if (!m.aligned()) return;
	struct Track { Contig &t; ~Track() { if (g_limits) g_limits->max_len = std::max(g_limits->max_len, t.len()); } } track{t};
	if (g_limits) g_limits->max_corr = std::max(g_limits->max_corr, (int64_t)m.corrections.size());
	std::set<int64_t> dont_overwrite;
	for (const Corr &c : m.corrections) {
		if (c.qbest) { t.seq[c.toff] = q.seq[c.qoff]; t.sup[c.toff] = q.sup[c.qoff]; }
		else         { q.seq[c.qoff] = t.seq[c.toff]; q.sup[c.qoff] = t.sup[c.toff]; }
		if (m.offset < 0) dont_overwrite.insert(c.qoff);
		else dont_overwrite.insert(c.toff);
	}
	if (m.offset < 0) { // :180-205
		int64_t ao = -m.offset;
		std::string tseq; std::vector<uint32_t> tsup;
		tseq.append(q.seq, 0, ao);
		tsup.insert(tsup.end(), q.sup.begin(), q.sup.begin() + ao);
		tseq.append(t.seq);
		tsup.insert(tsup.end(), t.sup.begin(), t.sup.end());
		if (q.len() > (int64_t)tseq.size()) {
			int64_t d = q.len() - (int64_t)tseq.size();
			tseq.append(q.seq, q.len() - d, d);
			tsup.resize(tseq.size(), 0);
		}
		for (int64_t i = ao; i < q.len(); ++i) {
			if (dont_overwrite.count(i)) continue;
			tsup[i] += q.sup[i];
		}
		t.seq = tseq; t.sup = tsup;
		t.nreads += q.nreads;
		t.start = q.start;
		return;
	}
	int64_t original_len = t.len();
	if (m.offset + q.len() > t.len()) {
		t.seq.resize(m.offset + q.len(), '\0');
		t.sup.resize(m.offset + q.len(), 0);
	}
	for (int64_t i = m.offset; i < std::min(q.len() + m.offset, t.len()); ++i) {
		if (dont_overwrite.count(i)) continue;
		int64_t qoff = i - m.offset;
		t.sup[i] += q.sup[qoff];
		if (i >= original_len) t.seq[i] = q.seq[qoff];
	}
	t.nreads += q.nreads;
}

// :32-36
int64_t match_sort(const Match &a, const Match &b)
{
	if (a.matches == b.matches) return a.mismatches - b.mismatches;
	return b.matches - a.matches;
}

// :224-240
Match best_match(std::vector<CP> &contigs, const CP &q, int64_t min_overlap, int64_t max_mismatch, allowed_fn allowed, Counters *cn)
{
	std::vector<Match> matches;
	for (size_t i = 0; i < contigs.size(); ++i) {
		if (contigs[i] == q) continue; // reference identity
		Match ma = slide_align(*q, *contigs[i], min_overlap, max_mismatch, allowed, cn);
		if (ma.aligned()) { ma.contig_i = (int64_t)i; matches.push_back(ma); }
	}
	if (matches.empty()) { Match ma; ma.offset = UNALIGNED; return ma; }
	// Nim's algorithm.sort is a stable merge sort
	std::stable_sort(matches.begin(), matches.end(), [](const Match &a, const Match &b) { return match_sort(a, b) < 0; });
	return matches[0];
}

// :243-248
void list_insert(std::vector<CP> &contigs, CP &q, int64_t min_overlap, int64_t max_mismatch, allowed_fn allowed, Counters *cn)
{
	Match ma = best_match(contigs, q, min_overlap, max_mismatch, allowed, cn);
	if (ma.aligned()) { if (cn) { cn->merges++; cn->left_merges += ma.offset < 0; cn->corrections += (int64_t)ma.corrections.size(); } insert_contig(*contigs[ma.contig_i], *q, ma); }
	else contigs.push_back(q);
}

// :254-281
std::vector<CP> combine(std::vector<CP> &contigs, int64_t max_mismatch, int64_t min_support, bool again, allowed_fn allowed, Counters *cn)
{
	if (again) contigs = combine(contigs, max_mismatch, 0, false, allowed, cn);
	std::vector<CP> result;
	size_t usedi = 0;
	for (size_t i = 0; i < contigs.size(); ++i) {
		CP &c = contigs[i];
		if (min_support > 0) trim_contig(*c, std::min<int64_t>(c->nreads, min_support));
		if (c->nreads > 0 && result.empty()) { result.push_back(c); usedi = i; }
	}
	if (result.empty()) return result;
	for (size_t i = 0; i < contigs.size(); ++i) {
		if (i == usedi) continue;
		Match ma = best_match(result, contigs[i], 65, max_mismatch, allowed, cn); // default min_overlap (:224)
		if (ma.aligned()) { if (cn) { cn->merges++; cn->left_merges += ma.offset < 0; cn->corrections += (int64_t)ma.corrections.size(); } insert_contig(*result[ma.contig_i], *contigs[i], ma); }
		else if (contigs[i]->nreads > 0) result.push_back(contigs[i]);
	}
	return result;
}

// ---------------------------------------------------------------------------------------------
// src/indelope.nim:23-38
// ---------------------------------------------------------------------------------------------
int32_t trim_read(const uint8_t *bq, int32_t n, int32_t *out_len, int min_quality = 15)
{
	int32_t high = n - 1;
	int32_t a = 0;
	while (a < high && bq[a] < (uint8_t)min_quality) a += 1;
	if (a == high) { *out_len = 0; return a; }
	if (n == 0) { *out_len = 0; return 0; }
	int32_t b = high;
	while (b > a && bq[b] < (uint8_t)min_quality) b -= 1;
	*out_len = b - a + 1;
	return a;
}

// ---------------------------------------------------------------------------------------------
// src/ksw2/ksw2.nim
// ---------------------------------------------------------------------------------------------
struct Ez {
	orc_ez_t c;
	std::vector<uint32_t> cig;
	int8_t match = 1, mismatch = -2, gap_open = 4, gap_ext = 1; // new_ez :142
};
struct CigarPair { uint32_t op, length; };

inline uint8_t encode_base(char ch) // lookup :127
{
	switch (ch) { case 'A': case 'a': return 0; case 'C': case 'c': return 1; case 'G': case 'g': return 2; case 'T': case 't': return 3; default: return 4; }
}

// align_to :151-164
void align_to(const std::string &query, const std::string &target, Ez &ez, int bw, int z, bool use_ref, int64_t *cells)
{
	std::vector<uint8_t> q(query.size()), t(target.size());
	for (size_t i = 0; i < query.size(); ++i) q[i] = encode_base(query[i]);
	for (size_t i = 0; i < target.size(); ++i) t[i] = encode_base(target[i]);
	int cap = (int)(query.size() + target.size() + 8);
	ez.cig.assign(cap, 0);
	if (use_ref && g_ref_ksw2 && !query.empty() && !target.empty()) {
		g_ref_ksw2((int)q.size(), q.data(), (int)t.size(), t.data(), ez.match, ez.mismatch, ez.gap_open, ez.gap_ext, bw, z, 0, &ez.c, ez.cig.data(), cap);
	} else {
		orc_ksw2_lane((int)q.size(), q.data(), (int)t.size(), t.data(), ez.match, ez.mismatch, ez.gap_open, ez.gap_ext, bw, z, &ez.c, ez.cig.data(), cap);
		if (cells) *cells += ez.c.cells;
	}
	ez.cig.resize(ez.c.n_cigar > 0 ? ez.c.n_cigar : 0);
}

// the truncated `cigar` iterator :22-33
std::vector<CigarPair> trunc_cigar(const Ez &e)
{
	std::vector<CigarPair> out;
	uint32_t max_off = (uint32_t)e.c.max_q, off = 0;
	for (int i = 0; i < e.c.n_cigar; ++i) {
		if (off >= max_off) break;
		CigarPair r{e.cig[i] & 0xf, e.cig[i] >> 4};
		if (r.op != 2) off += r.length;
		out.push_back(r);
	}
	return out;
}
std::string cigar_string(const std::vector<CigarPair> &c)
{
	std::string s;
	for (auto &x : c) { s += std::to_string(x.length); s += "MID"[x.op]; }
	return s;
}
std::string full_cigar_string(const Ez &e)
{
	std::string s;
	for (int i = 0; i < e.c.n_cigar; ++i) { s += std::to_string(e.cig[i] >> 4); s += "MID"[e.cig[i] & 0xf]; }
	return s;
}

enum EventType { Insertion = 0, Deletion = 1 };
struct Event { int64_t start, stop; uint32_t len; EventType type; };

// :71-80
std::vector<Event> target_locations(const std::vector<CigarPair> &cig, int64_t start)
{
	std::vector<Event> out; int64_t off = start;
	for (auto &c : cig) {
		if (c.op == 1) out.push_back(Event{off, off + 1, c.length, Insertion});
		else if (c.op == 2) out.push_back(Event{off, off + (int64_t)c.length, c.length, Deletion});
		if (c.op != 1) off += c.length;
	}
	return out;
}
// :82-91
std::vector<Event> query_locations(const std::vector<CigarPair> &cig, int64_t start = 0)
{
	std::vector<Event> out; int64_t off = start;
	for (auto &c : cig) {
		if (c.op == 2) out.push_back(Event{off, off + 1, c.length, Deletion});
		else if (c.op == 1) out.push_back(Event{off, off + (int64_t)c.length, c.length, Insertion});
		if (c.op != 2) off += c.length;
	}
	return out;
}

// src/indelope.nim:118-132
int64_t get_min_flank(const Event &e, const std::vector<CigarPair> &cig)
{
	const int64_t init_len = INT64_MAX;
	int64_t result = init_len;
	bool found_event = false;
	for (auto &c : cig) {
		if (c.op == 0) {
			if (found_event) result = std::min<int64_t>(c.length, result);
			else result = c.length;
			if (found_event) return result;
		} else if ((int)c.op - 1 == (int)e.type && c.length == e.len) {
			if (init_len == result) result = 0;
			found_event = true;
		}
	}
	return 0;
}

// src/indelope.nim:185-199
int64_t count_flanked_cigar(const std::vector<CigarPair> &cig)
{
	bool matched = false; int64_t n = 0; int last_op = 0;
	for (auto &e : cig) {
		if (!matched) { if (e.op == 0) { n += 1; matched = true; } }
		else n += 1;
		last_op = (int)e.op;
	}
	if (last_op != 0) n -= 1;
	return n;
}

// ---------------------------------------------------------------------------------------------
// src/genotyper.nim
// ---------------------------------------------------------------------------------------------
enum GT { HOM_REF = 0, HET = 1, HOM_ALT = 2, UNKNOWN = 3 };
struct Genotype { GT gt; double GL[3]; };

Genotype genotype(int64_t r, int64_t a, double error) // :36-47
{
	const double log2 = std::log(2.0);
	double total = (double)(r + a);
	Genotype g; g.gt = UNKNOWN; g.GL[0] = g.GL[1] = g.GL[2] = 0;
	if (total == 0) return g;
	g.gt = HOM_REF;
	for (int G = 0; G <= 2; ++G) {
		g.GL[G] = -total * log2 + (double)r * std::log((double)G * error + (double)(2 - G) * (1 - error)) +
		          (double)a * std::log((double)G * (1 - error) + (double)(2 - G) * error);
		if (g.GL[G] > g.GL[(int)g.gt]) g.gt = (GT)G;
	}
	return g;
}
double gt_qual(const Genotype &g) // :22-29
{
	if (g.gt == HOM_REF) return g.GL[0] - std::max(g.GL[1], g.GL[2]);
	if (g.gt == HET) return g.GL[1] - std::max(g.GL[0], g.GL[2]);
	if (g.gt == HOM_ALT) return g.GL[2] - std::max(g.GL[0], g.GL[1]);
	return 0;
}
// Nim formatFloat(x, ffDecimal, precision) is C sprintf("%#.*f") (SURVEY appendix C)
std::string fmt_float(double x, int precision)
{
	char buf[2600];
	snprintf(buf, sizeof buf, "%#.*f", precision, x);
	return buf;
}
std::string gt_text(const Genotype &g) // :31-34
{
	static const char *enc[] = {"0/0", "0/1", "1/1", "./."};
	return std::string(enc[(int)g.gt]) + ":" + fmt_float(gt_qual(g), 4) + ":" + fmt_float(g.GL[0], 4) + "," +
	       fmt_float(g.GL[1], 4) + "," + fmt_float(g.GL[2], 4);
}

// ---------------------------------------------------------------------------------------------
// [ext] kmer package -- DECLARED semantics (SURVEY appendix D)
// ---------------------------------------------------------------------------------------------
bool mincode(const char *s, int K, uint64_t *code)
{
	uint64_t f = 0, rc = 0;
	for (int i = 0; i < K; ++i) {
		uint8_t b = encode_base(s[i]);
		if (b > 3) return false;
		f = (f << 2) | b;
		rc |= (uint64_t)(3 - b) << (2 * i);
	}
	*code = f < rc ? f : rc;
	return true;
}

int distinct_chars(const std::string &s) { std::set<char> x(s.begin(), s.end()); return (int)x.size(); }

double mean_int(const std::vector<int64_t> &a) // src/indelope.nim:146-150
{
	volatile double result = 0;
	for (int64_t v : a) result = result + (double)v;
	volatile double n = (double)a.size();
	return result / n; // 0.0/0.0 at run time for an empty list, as the reference computes it
}
int median_u8(std::vector<uint8_t> b) // :152-155
{
	std::sort(b.begin(), b.end());
	return (int)b[(size_t)((double)b.size() / 2)];
}

// ---------------------------------------------------------------------------------------------
// src/indelope.nim:49-116  Variant
// ---------------------------------------------------------------------------------------------
struct Variant {
	std::string chrom; int64_t start = 0; double qual = 0;
	std::string reference, alternate; Genotype gt; std::string ref_kmer, alt_kmer, info_str;
	int64_t AD[2] = {0, 0};
	void info_add(const std::string &kv) { if (info_str.empty()) info_str = kv; else { info_str += ';'; info_str += kv; } } // :70-75
	std::string info() const { // :63-68
		std::string r = "AD=" + std::to_string(AD[0]) + "," + std::to_string(AD[1]) + ";ref_kmer=" + ref_kmer + ";alt_kmer=" + alt_kmer;
		if (!info_str.empty()) r += ";" + info_str;
		return r;
	}
	std::string text() const { // :104-112
		return chrom + "\t" + std::to_string(start) + "\t.\t" + reference + "\t" + alternate + "\t" + fmt_float(qual, 2) +
		       "\tPASS\t" + info() + "\tGT:GQ:GL\t" + gt_text(gt);
	}
	bool same(const Variant &b) const { return start == b.start && chrom == b.chrom && reference == b.reference && alternate == b.alternate; } // :114-116
};

// ---------------------------------------------------------------------------------------------
// region input view
// ---------------------------------------------------------------------------------------------
struct ReadV {
	int64_t start, stop; int mapq; int flag; std::string seq; const uint8_t *qual; int32_t len;
};
struct Roi { int64_t start, stop; int chrom; std::vector<ReadV> reads; int64_t ordinal; };

bool skippable(const ReadV &r) // src/indelope.nim:40-47 (chrom name test is host-side, regions never come from those)
{
	int f = r.flag;
	if ((f & 0x400) || (f & 0x200)) return true;
	if (f & 0x4) return true;
	if ((f & 0x800) || (f & 0x100)) return true;
	return false;
}

struct Fai { // hts-nim Fai.get == faidx_fetch_seq: 0-based, inclusive, clipped (SURVEY appendix D)
	const uint8_t *seq; int64_t len;
	std::string get(int64_t a, int64_t b) const {
		if (a < 0) a = 0;
		if (b >= len) b = len - 1;
		if (a > b) return std::string();
		return std::string((const char*)seq + a, (size_t)(b - a + 1));
	}
};

// src/indelope.nim:157-183
std::vector<CP> assemble(const Roi &r, int64_t *n_contigs, Counters *cn, int min_qual = 20, double min_overlap_pct = 0.88)
{
	std::vector<CP> contigs;
	for (const ReadV &read : r.reads) {
		if (read.mapq < min_qual) continue;
		if (skippable(read)) continue;
		int32_t tl; int32_t o = trim_read(read.qual, read.len, &tl);
		std::string read_seq = tl > 0 ? read.seq.substr(o, tl) : std::string();
		if (g_limits) g_limits->max_len = std::max(g_limits->max_len, (int64_t)read_seq.size());
		CP qc = make_contig(read_seq, read.start + o);
		list_insert(contigs, qc, (int64_t)(min_overlap_pct * (double)read_seq.size()), 0, allowable_mismatch, cn);
	}
	*n_contigs = (int64_t)contigs.size();
	contigs = combine(contigs, 0, 3, true, allowable_mismatch, cn);
	return contigs;
}

struct Out { std::string dump; std::vector<Variant> variants; Counters cn; };

void dump_contig(std::string &d, int64_t ord, size_t ci, const Contig &c, bool with_sup)
{
	d += "C\t" + std::to_string(ord) + "\t" + std::to_string(ci) + "\t" + std::to_string(c.start) + "\t" + std::to_string(c.nreads) +
	     "\t" + std::to_string(c.len()) + "\t" + c.seq;
	if (with_sup) {
		d += "\t";
		for (size_t i = 0; i < c.sup.size(); ++i) { if (i) d += ","; d += std::to_string(c.sup[i]); }
	}
	d += "\n";
}

// src/indelope.nim:201-428
void callsemble(const Roi &r, const Fai &fai, const std::string &chrom, const orc_params_t &P, Out &out)
{
	const int K = 27;
	const int64_t min_ctg_len = P.min_ctg_len, min_reads = P.min_reads, min_event_len = P.min_event_len;
	const bool use_ref = P.use_ref_ksw2 != 0;
	Counters &cn = out.cn;
	std::string &d = out.dump;
	int64_t n_contigs = 0;
	Limits lim;
	g_limits = &lim;
	std::vector<CP> contigs = assemble(r, &n_contigs, &cn);
	g_limits = nullptr;
	cn.contigs_pre += n_contigs; cn.contigs_post += (int64_t)contigs.size();
	if (P.dump_level & 64) d += "L\t" + std::to_string(r.ordinal) + "\tmax_len=" + std::to_string(lim.max_len) + "\tmax_corr=" + std::to_string(lim.max_corr) + "\n";
	if (P.dump_level & 1) {
		d += "R\t" + std::to_string(r.ordinal) + "\tpre=" + std::to_string(n_contigs) + "\tn=" + std::to_string(contigs.size()) + "\n";
		for (size_t ci = 0; ci < contigs.size(); ++ci) dump_contig(d, r.ordinal, ci, *contigs[ci], (P.dump_level & 2) != 0);
	}
	Ez ez; // new_ez() :576
	for (size_t ci = 0; ci < contigs.size(); ++ci) {
		Contig &ctg = *contigs[ci];
		if (n_contigs > 20) continue;
		if (ctg.nreads < min_reads || ctg.len() < min_ctg_len) continue;
		int64_t max_stop = ctg.start;
		for (const ReadV &read : r.reads) {
			if (read.mapq <= 5) continue;
			max_stop = std::max(max_stop, read.stop);
		}
		const int64_t width = (int64_t)((double)(K + 1) / 2 - 1);
		std::string reference = fai.get(ctg.start, max_stop + width + 50);
		align_to(ctg.seq, reference, ez, 50, 400, use_ref, &cn.cells_a);
		cn.dp_a++;
		std::vector<CigarPair> cig = trunc_cigar(ez);
		std::vector<Event> qlocs = query_locations(cig);
		if (P.dump_level & 4) {
			char b[256];
			snprintf(b, sizeof b, "A\t%lld\t%zu\t%lld\t%zu\t%d\t%d\t%d\t%d\t%d\t%d\t%d\t%d\t%d\t", (long long)r.ordinal, ci, (long long)ctg.start,
			         reference.size(), ez.c.max, ez.c.zdropped, ez.c.max_q, ez.c.max_t, ez.c.mqe, ez.c.mqe_t, ez.c.mte, ez.c.mte_q, ez.c.score);
			d += b; d += full_cigar_string(ez) + "\t" + cigar_string(cig) + "\n";
		}
		if (qlocs.empty() || qlocs.size() > 4) continue;
		int64_t ii = -1;
		for (const Event &tloc : target_locations(cig, ctg.start)) {
			ii += 1;
			const Event &qloc = qlocs[ii];
			int reject = 0;
			std::string ref_kmer, alt_kmer;
			int64_t tstart = 0, qstart = 0, offset = 0;
			int64_t ref_support = 0, alt_support = 0, both_found = 0, kref = 0, kalt = 0, kboth = 0;
			std::vector<int64_t> adists, rdists; std::vector<uint8_t> amapqs, rmapqs;
			bool aligned = false;
			int64_t min_flank = -1;
			do {
				if ((int64_t)tloc.len < min_event_len) { reject = 10; break; }
				tstart = std::max<int64_t>(0, tloc.start - ctg.start - width);
				if (tstart + K > (int64_t)reference.size()) tstart = (int64_t)reference.size() - K;
				if (tstart < 0) { reject = 11; break; } // window shorter than K: the reference would raise
				ref_kmer = reference.substr(tstart, K);
				offset = std::min<int64_t>(qloc.start, ctg.len() - qloc.stop - 1);
				qstart = std::max<int64_t>(qloc.start - width, 0);
				if (qstart + K > ctg.len()) qstart = ctg.len() - K;
				// a contig shorter than K (min_ctg_len < K): the reference would raise here as well; no k-mers are reported
				if (qstart < 0) { ref_kmer.clear(); reject = 11; break; }
				alt_kmer = ctg.seq.substr(qstart, K);
				if (alt_kmer == ref_kmer) {
					qstart = std::max<int64_t>(qloc.start - 3, 0);
					if (qstart + K > ctg.len()) {
						int64_t qend = std::min<int64_t>(qloc.stop + 4, ctg.len());
						qstart = qend - K;
						if (qstart < 0) { ref_kmer.clear(); alt_kmer.clear(); reject = 11; break; }
						alt_kmer = ctg.seq.substr(qstart, K);
					} else alt_kmer = ctg.seq.substr(qstart, K);
				}
				if (ref_kmer == alt_kmer && (qloc.start == 0 || distinct_chars(alt_kmer) == 1)) { reject = 1; break; }
				if (distinct_chars(ref_kmer) < 3) { reject = 2; break; }
				if (ref_kmer == alt_kmer) { reject = 3; break; } // the "bug!!!" branch :268-275
				uint64_t refe = 0, alte = 0;
				bool ref_ok = mincode(ref_kmer.c_str(), K, &refe), alt_ok = mincode(alt_kmer.c_str(), K, &alte);
				cn.events++;
				for (const ReadV &read : r.reads) { // :293-311
					if (read.mapq < 10) continue;
					bool ref_found = false, alt_found = false;
					cn.kmer_reads++; cn.kmer_bytes += (read.len + 3) / 4 + (read.len + 7) / 8 + 16;
					int64_t L = read.len;
					if (L >= K) {
						uint64_t f = 0, rc = 0; int valid = 0; const uint64_t mask = (1ULL << (2 * K)) - 1;
						for (int64_t i = 0; i < L; ++i) {
							uint8_t b = encode_base(read.seq[i]);
							if (b > 3) { valid = 0; f = rc = 0; continue; }
							f = ((f << 2) | b) & mask;
							rc = (rc >> 2) | ((uint64_t)(3 - b) << (2 * (K - 1)));
							if (++valid < K) continue;
							cn.kmer_windows++;
							int64_t pos = i - K + 1;
							int64_t dd = std::min<int64_t>(pos, (L - K) - pos);
							uint64_t e = f < rc ? f : rc;
							if (!ref_found && ref_ok && e == refe) { ref_support += 1; ref_found = true; rdists.push_back(dd); rmapqs.push_back((uint8_t)read.mapq); }
							if (!alt_found && alt_ok && e == alte) { alt_support += 1; alt_found = true; adists.push_back(dd); amapqs.push_back((uint8_t)read.mapq); }
						}
					}
					if (ref_found && alt_found) both_found += 1;
				}
				cn.kmer_bytes += 64;
				kref = ref_support; kalt = alt_support; kboth = both_found;
				if (both_found > 0) { // :313-372
					cn.al_events++;
					both_found = 0; ref_support = 0; alt_support = 0;
					Ez ez_ref, ez_alt;
					ez_ref.gap_open = ez_alt.gap_open = 5;
					for (const ReadV &read : r.reads) {
						if (read.mapq < 10) continue;
						int32_t tl; int32_t ta = trim_read(read.qual, read.len, &tl);
						std::string read_seq = tl > 0 ? read.seq.substr(ta, tl) : std::string();
						int64_t rs = read.start + ta;
						if (rs > tloc.stop) continue;
						int64_t L = 0;
						if (tloc.type == Insertion) L = (int64_t)tloc.len;
						if (rs + (int64_t)read_seq.size() + L < tloc.start) continue;
						int64_t start = std::max(rs, ctg.start) - ctg.start;
						std::string ref_sub = start <= (int64_t)reference.size() ? reference.substr(start) : std::string();
						std::string ctg_sub = start <= ctg.len() ? ctg.seq.substr(start) : std::string();
						align_to(read_seq, ref_sub, ez_ref, -1, -1, use_ref, &cn.cells_b);
						align_to(read_seq, ctg_sub, ez_alt, -1, -1, use_ref, &cn.cells_b);
						cn.dp_b += 2;
						int64_t rn = count_flanked_cigar(trunc_cigar(ez_ref));
						int64_t an = count_flanked_cigar(trunc_cigar(ez_alt));
						if (rn == 1 && an > 1) ref_support += 1;
						else if (an == 1 && rn > 1) alt_support += 1;
					}
					aligned = true;
				}
				min_flank = get_min_flank(qloc, cig);
			} while (0);
			if (P.dump_level & 8) {
				char b[512];
				snprintf(b, sizeof b, "E\t%lld\t%zu\t%lld\t%c\t%lld\t%lld\t%u\t%lld\t%lld\t%d\t%lld\t%lld\t", (long long)r.ordinal, ci, (long long)ii,
				         tloc.type == Insertion ? 'I' : 'D', (long long)tloc.start, (long long)tloc.stop, tloc.len, (long long)qloc.start,
				         (long long)qloc.stop, reject, (long long)tstart, (long long)qstart);
				d += b; d += (ref_kmer.empty() ? "." : ref_kmer) + "\t" + (alt_kmer.empty() ? "." : alt_kmer);
				int64_t sa = 0, sr = 0; for (auto v : adists) sa += v; for (auto v : rdists) sr += v;
				snprintf(b, sizeof b, "\t%lld\t%lld\t%lld\t%d\t%lld\t%lld\t%lld\t%zu\t%lld\t%zu\t%lld\t%d\t%d\t%lld\t%lld\n", (long long)kref, (long long)kalt,
				         (long long)kboth, aligned ? 1 : 0, (long long)ref_support, (long long)alt_support, (long long)both_found, adists.size(),
				         (long long)sa, rdists.size(), (long long)sr, amapqs.empty() ? -1 : median_u8(amapqs), rmapqs.empty() ? -1 : median_u8(rmapqs),
				         (long long)min_flank, (long long)offset);
				d += b;
			}
			if (reject) continue;
			// ---- filter cascade :375-428
			if (alt_support < min_reads) continue;
			if ((double)alt_support / (double)r.reads.size() < 0.1) continue;
			Genotype gt = genotype(ref_support, alt_support, 1e-3);
			if (gt.gt == HOM_REF) continue;
			Variant v; v.chrom = chrom; v.start = tloc.start; v.gt = gt; v.ref_kmer = ref_kmer; v.qual = gt_qual(gt); v.alt_kmer = alt_kmer;
			v.AD[0] = ref_support; v.AD[1] = alt_support;
			if (offset == 0 && both_found >= (int64_t)(0.75 * (double)std::min(ref_support, alt_support))) continue;
			v.info_add("DP=" + std::to_string(r.reads.size()));
			if (offset < 5) { v.info_add("LO"); v.qual /= 2.0; }
			if (both_found > 0) { v.info_add("BS=" + std::to_string(both_found)); v.qual /= 1.5; }
			else v.qual *= 2;
			v.info_add("CC=" + cigar_string(cig));
			if (aligned) v.info_add("AL");
			if ((min_flank - 1) < std::max(tloc.stop - tloc.start, qloc.stop - qloc.start)) continue;
			v.info_add("MF=" + std::to_string(min_flank));
			v.info_add("CF=" + std::to_string(offset));
			v.info_add("NC=" + std::to_string(n_contigs));
			if (offset == 0) v.qual /= 4.0;
			v.info_add("AKE=" + fmt_float(mean_int(adists), 2));
			v.info_add("RKE=" + fmt_float(mean_int(rdists), 2));
			if (!amapqs.empty()) v.info_add("AMQ=" + std::to_string(median_u8(amapqs)));
			if (!rmapqs.empty()) v.info_add("RMQ=" + std::to_string(median_u8(rmapqs)));
			if (mean_int(adists) < 5) continue;
			if (tloc.type == Deletion) {
				v.reference = fai.get(tloc.start - 1, tloc.stop - 1);
				v.alternate = v.reference.substr(0, 1);
			} else {
				if (qloc.start < 1) continue; // ctg.sequence[-1..] raises in the reference; unreachable with an M-led CIGAR
				v.reference = fai.get(tloc.start - 1, tloc.start - 1);
				v.alternate = ctg.seq.substr(qloc.start - 1, qloc.stop - (qloc.start - 1));
				v.start = tloc.start;
				std::string tail = v.alternate.substr(1);
				if (distinct_chars(tail) == 1 && distinct_chars(alt_kmer.substr(alt_kmer.size() - 11)) == 1 &&
				    distinct_chars(ref_kmer.substr(ref_kmer.size() - 11)) == 1)
					continue;
			}
			out.variants.push_back(v);
		}
	}
}

Roi make_roi(const orc_roiset_t *in, int64_t k)
{
	Roi r; r.start = in->roi_start[k]; r.stop = in->roi_stop[k]; r.chrom = in->roi_chrom[k]; r.ordinal = k;
	r.reads.reserve(in->roi_n_reads[k]);
	for (int32_t j = 0; j < in->roi_n_reads[k]; ++j) {
		int64_t i = in->read_idx[in->roi_read_begin[k] + j];
		ReadV v; v.start = in->start[i]; v.stop = in->stop[i]; v.mapq = in->mapq[i]; v.flag = in->flag[i]; v.len = in->len[i];
		v.seq.assign((const char*)in->bases + in->seq_off[i], (size_t)v.len); v.qual = in->quals + in->seq_off[i];
		r.reads.push_back(std::move(v));
	}
	return r;
}

char *dup_text(const std::string &s)
{
	char *p = (char*)malloc(s.size() + 1);
	memcpy(p, s.data(), s.size()); p[s.size()] = 0;
	return p;
}

} // namespace

extern "C" {

int orc_load_ref(const char *path)
{
	void *h = dlopen(path, RTLD_NOW | RTLD_LOCAL);
	if (!h) return -1;
	g_ref_ksw2 = (ref_ksw2_fn)dlsym(h, "orc_ksw2_ref");
	return g_ref_ksw2 ? 0 : -2;
}

void orc_free(void *p) { free(p); }

int orc_call(const orc_roiset_t *in, const orc_params_t *p, char **dump, char **vcf, orc_counters_t *cnt)
{
	if (p->use_ref_ksw2 && !g_ref_ksw2) return -1;
	auto t0 = std::chrono::steady_clock::now();
	int64_t n = in->n_rois;
	std::vector<Out> outs((size_t)n);
	int nt = p->n_threads > 1 ? p->n_threads : 1;
	auto work = [&](int tid) {
		for (int64_t k = tid; k < n; k += nt) {
			Roi r = make_roi(in, k);
			Fai fai{in->chrom_seq[r.chrom], in->chrom_len[r.chrom]};
			callsemble(r, fai, in->chrom_name[r.chrom], *p, outs[(size_t)k]);
		}
	};
	if (nt == 1) work(0);
	else {
		std::vector<std::thread> th;
		for (int t = 0; t < nt; ++t) th.emplace_back(work, t);
		for (auto &t : th) t.join();
	}
	// emission order + order-dependent dedup against the last two emitted variants, src/indelope.nim:598-608
	std::string d, v;
	const Variant *last_var = nullptr, *last_var2 = nullptr;
	orc_counters_t c; memset(&c, 0, sizeof c);
	for (int64_t k = 0; k < n; ++k) {
		Out &o = outs[(size_t)k];
		d += o.dump;
		for (const Variant &x : o.variants) {
			const bool dedup = !(p->dump_level & 32); // bit5: raw records (interval shards dedup after merging)
			if (dedup && last_var && x.same(*last_var)) continue;
			if (dedup && last_var2 && x.same(*last_var2)) continue;
			std::string line = x.text();
			v += line + "\n";
			if (p->dump_level & 16) d += "V\t" + line + "\n";
			last_var2 = last_var; last_var = &x;
			c.variants++;
		}
		c.regions++; c.reads += in->roi_n_reads[k];
		c.slide_calls += o.cn.slide_calls; c.offsets += o.cn.offsets; c.char_compares += o.cn.char_compares;
		c.exhaustive_compares += o.cn.exhaustive; c.contigs_pre += o.cn.contigs_pre; c.contigs_post += o.cn.contigs_post;
		c.dp_a += o.cn.dp_a; c.dp_b += o.cn.dp_b; c.cells_a += o.cn.cells_a; c.cells_b += o.cn.cells_b;
		c.events += o.cn.events; c.kmer_reads += o.cn.kmer_reads; c.kmer_windows += o.cn.kmer_windows; c.kmer_bytes += o.cn.kmer_bytes;
		c.al_events += o.cn.al_events;
		c.corrections += o.cn.corrections; c.vote_invariant_violations += o.cn.vote_invariant_violations; c.left_merges += o.cn.left_merges; c.merges += o.cn.merges;
	}
	c.seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
	if (dump) *dump = dup_text(d);
	if (vcf) *vcf = dup_text(v);
	if (cnt) *cnt = c;
	return 0;
}

char *orc_vcf_header(int32_t n_chroms, const char *const *names, const int64_t *lens)
{
	// src/indelope.nim:77-102 with $1 = contig lines (:548-552) and $2 = "sample" (:600)
	std::string h =
	    "##fileformat=VCFv4.2\n"
	    "##FORMAT=<ID=AD,Number=R,Type=Integer,Description=\"Allelic depths for the ref and alt alleles in the order listed\">\n"
	    "##INFO=<ID=AD,Number=R,Type=Integer,Description=\"Allelic depths for the ref and alt alleles in the order listed\">\n"
	    "##INFO=<ID=END,Number=1,Type=Integer,Description=\"End position of the variant described in this record\">\n"
	    "##INFO=<ID=SVLEN,Number=1,Type=Integer,Description=\"Difference in length between REF and ALT alleles\">\n"
	    "##INFO=<ID=DP,Number=1,Type=Integer,Description=\"total reads covering this site\">\n"
	    "##INFO=<ID=AL,Number=0,Type=Flag,Description=\"this was genotyped with alignment, no k-mer counting\">\n"
	    "##INFO=<ID=AMQ,Number=1,Type=Integer,Description=\"median mapping quality of alts\">\n"
	    "##INFO=<ID=RMQ,Number=1,Type=Integer,Description=\"median mapping quality of refs\">\n"
	    "##INFO=<ID=BS,Number=1,Type=Integer,Description=\"number of times there was support for both ref and alt k-mer in a single read\">\n"
	    "##INFO=<ID=MF,Number=1,Type=Integer,Description=\"minimum matching bases around this event when BS > 0. Higher gives more confidence\">\n"
	    "##INFO=<ID=CF,Number=1,Type=Integer,Description=\"minimum flank of the event from either end of the contig. higher is better.\">\n"
	    "##INFO=<ID=NC,Number=1,Type=Integer,Description=\"number of contigs at the site of this variant.\">\n"
	    "##INFO=<ID=CC,Number=1,Type=String,Description=\"contig cigar from alignment to reference\">\n"
	    "##INFO=<ID=LO,Number=0,Type=Flag,Description=\"low-offset: the event occurred near at the start of the contig so we may not have the full variant\">\n"
	    "##INFO=<ID=AKE,Number=1,Type=Float,Description=\"mean alt-kmer distance from end of read\">\n"
	    "##INFO=<ID=RKE,Number=1,Type=Float,Description=\"mean ref-kmer distance from end of read\">\n"
	    "##FORMAT=<ID=DP,Number=1,Type=Integer,Description=\"supporting k-mer depth\">\n"
	    "##FORMAT=<ID=GQ,Number=1,Type=Float,Description=\"Genotype Quality\">\n"
	    "##FORMAT=<ID=GT,Number=1,Type=String,Description=\"Genotype\">\n"
	    "##FORMAT=<ID=GL,Number=G,Type=Float,Description=\"Normalized, Phred-scaled likelihoods for genotypes as defined in the VCF specification\">\n"
	    "##INFO=<ID=DP,Number=1,Type=Integer,Description=\"Approximate read depth; some reads may have been filtered\">\n"
	    "##INFO=<ID=ref_kmer,Number=1,Type=String,Description=\"reference kmer used for genotyping\">\n"
	    "##INFO=<ID=alt_kmer,Number=1,Type=String,Description=\"alternate kmer used for genotyping\">\n";
	for (int i = 0; i < n_chroms; ++i) {
		if (i) h += "\n";
		h += "##contig=<ID=" + std::string(names[i]) + ",length=" + std::to_string(lens[i]) + ">";
	}
	h += "\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tsample\n";
	return dup_text(h);
}

void orc_slide_align(const char *q, const uint32_t *qsup, int64_t qreads, const char *t, const uint32_t *tsup, int64_t treads,
                     int64_t min_overlap, int64_t max_mismatch, int rule, orc_match_t *out)
{
	Contig qc, tc;
	qc.seq = q; qc.sup.assign(qsup, qsup + qc.seq.size()); qc.nreads = qreads;
	tc.seq = t; tc.sup.assign(tsup, tsup + tc.seq.size()); tc.nreads = treads;
	Match m = slide_align(qc, tc, min_overlap, max_mismatch, rule ? allow_test : allowable_mismatch, nullptr);
	out->matches = m.matches; out->offset = m.offset; out->mismatches = m.mismatches; out->aligned = m.aligned() ? 1 : 0;
	out->n_corr = (int32_t)std::min<size_t>(m.corrections.size(), 64);
	for (int i = 0; i < out->n_corr; ++i) {
		out->corr[3 * i] = (int32_t)m.corrections[i].qoff; out->corr[3 * i + 1] = (int32_t)m.corrections[i].toff;
		out->corr[3 * i + 2] = m.corrections[i].qbest ? 1 : 0;
	}
}

void orc_insert(char *t, uint32_t *tsup, int64_t *tlen, int64_t *treads, int64_t *tstart, char *q, uint32_t *qsup, int64_t qlen,
                int64_t qreads, int64_t qstart, const orc_match_t *m)
{
	Contig qc, tc;
	qc.seq.assign(q, (size_t)qlen); qc.sup.assign(qsup, qsup + qlen); qc.nreads = qreads; qc.start = qstart;
	tc.seq.assign(t, (size_t)*tlen); tc.sup.assign(tsup, tsup + *tlen); tc.nreads = *treads; tc.start = *tstart;
	Match mm; mm.matches = m->matches; mm.offset = m->aligned ? m->offset : UNALIGNED; mm.mismatches = m->mismatches;
	for (int i = 0; i < m->n_corr; ++i) mm.corrections.push_back(Corr{m->corr[3 * i], m->corr[3 * i + 1], m->corr[3 * i + 2] != 0});
	insert_contig(tc, qc, mm);
	memcpy(t, tc.seq.data(), tc.seq.size()); t[tc.seq.size()] = 0;
	memcpy(tsup, tc.sup.data(), tc.sup.size() * sizeof(uint32_t));
	*tlen = tc.len(); *treads = tc.nreads; *tstart = tc.start;
}

char *orc_assemble_strings(int n, const char *const *seqs, const int64_t *starts, const int64_t *min_overlaps, int do_combine, int64_t *n_pre)
{
	std::vector<CP> contigs;
	for (int i = 0; i < n; ++i) {
		CP qc = make_contig(seqs[i], starts[i]);
		list_insert(contigs, qc, min_overlaps[i], 0, allowable_mismatch, nullptr);
	}
	if (n_pre) *n_pre = (int64_t)contigs.size();
	if (do_combine) contigs = combine(contigs, 0, 3, true, allowable_mismatch, nullptr);
	std::string d;
	for (size_t ci = 0; ci < contigs.size(); ++ci) dump_contig(d, 0, ci, *contigs[ci], true);
	return dup_text(d);
}

int orc_genotype(int64_t r, int64_t a, double error, char *text, int cap, double *qual)
{
	Genotype g = genotype(r, a, error);
	std::string s = gt_text(g);
	if (text && cap > 0) { strncpy(text, s.c_str(), (size_t)cap - 1); text[cap - 1] = 0; }
	if (qual) *qual = gt_qual(g);
	return (int)g.gt;
}

int32_t orc_trim(const uint8_t *quals, int32_t n, int32_t *out_len) { return trim_read(quals, n, out_len); }

int orc_mincode(const char *s, int k, uint64_t *code) { return mincode(s, k, code) ? 0 : -1; }

} // extern "C"
