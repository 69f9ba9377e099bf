// indelope_b200/csrc/host/pack_vcf.cpp
//
// Host side of the drop-in boundary:
//   * quality trim (src/indelope.nim:23-38), min_overlap (:169), 2-bit packing of reads and of the reference
//     window into an idl_batch (include/indelope_cuda.h)
//   * after the device pass: the filter cascade, genotype likelihoods and VCF text of
//     src/indelope.nim:375-428,49-116 and src/genotyper.nim:16-47, with the order-dependent dedup of
//     src/indelope.nim:598-608.  Float64 maths stays here, exactly as in the reference's host.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <chrono>
#include <string>
#include <thread>
#include <vector>
#if defined(__x86_64__)
#include <immintrin.h>
#endif
#include "indelope_host.h"

namespace {

// ---- 2-bit packing ------------------------------------------------------------------------------------------------
// src/ksw2/ksw2.nim:127 lookup: ACGT -> 0..3, anything else 4.  This implementation's alphabet is {A,C,G,T,N}: lower-case acgt
// are folded to upper case and every other byte to N, and the fold is REPORTED (IDL_RF_ALPHABET on the region), because the
// reference compares raw characters (src/contig.nim:93,122) and may answer differently there.
// LUT entry: bits 0-1 code, bit 2 "not ACGT" (N plane), bit 3 "folded" (a byte outside the upper-case alphabet ACGTN)
struct Lut { uint8_t t[256]; Lut() { for (int i = 0; i < 256; ++i) t[i] = 4 | 8; t['A'] = 0; t['C'] = 1; t['G'] = 2; t['T'] = 3; t['N'] = 4;
                                     t['a'] = 0 | 8; t['c'] = 1 | 8; t['g'] = 2 | 8; t['t'] = 3 | 8; } };
const Lut LUT;

inline uint32_t spread16(uint32_t x) // bit i -> bit 2i
{
	x = (x | (x << 8)) & 0x00FF00FFu; x = (x | (x << 4)) & 0x0F0F0F0Fu; x = (x | (x << 2)) & 0x33333333u; x = (x | (x << 1)) & 0x55555555u;
	return x;
}

// 16 bases -> one 2-bit word + 16 N-plane bits; returns nonzero if a byte was folded.  n < 16: the rest reads as padding (zero)
inline unsigned pack16_scalar(const uint8_t *s, int n, uint32_t *w2, uint16_t *wn)
{
	uint32_t a = 0, b = 0; unsigned bad = 0;
	for (int i = 0; i < n; ++i) { const unsigned c = LUT.t[s[i]]; bad |= c & 8; if (c & 4) b |= 1u << i; else a |= (c & 3) << (2 * i); }
	*w2 = a; *wn = (uint16_t)b;
	return bad;
}

#if defined(__x86_64__)
// 32 bases per step on AVX2 + BMI2 (chosen at run time): five byte compares, three movemasks, two PDEPs for the bit interleave
__attribute__((target("avx2,bmi2"))) int64_t pack_chunks_avx2(const uint8_t *s, int64_t n, uint32_t *d2, uint16_t *dn, unsigned *bad_out)
{
	const __m256i cA = _mm256_set1_epi8('A'), cC = _mm256_set1_epi8('C'), cG = _mm256_set1_epi8('G'), cT = _mm256_set1_epi8('T'), cN = _mm256_set1_epi8('N'),
	              fold = _mm256_set1_epi8((char)0xDF);
	__m256i okv = _mm256_set1_epi8((char)0xFF);
	int64_t c = 0;
	for (; (c + 2) * 16 <= n; c += 2) {
		const __m256i x = _mm256_loadu_si256((const __m256i*)(s + 16 * c));
		const __m256i xf = _mm256_and_si256(x, fold);
		const __m256i eA = _mm256_cmpeq_epi8(xf, cA), eC = _mm256_cmpeq_epi8(xf, cC), eG = _mm256_cmpeq_epi8(xf, cG), eT = _mm256_cmpeq_epi8(xf, cT);
		const __m256i acgt = _mm256_or_si256(_mm256_or_si256(eA, eC), _mm256_or_si256(eG, eT));
		const uint32_t b0 = (uint32_t)_mm256_movemask_epi8(_mm256_or_si256(eC, eT)), b1 = (uint32_t)_mm256_movemask_epi8(_mm256_or_si256(eG, eT));
		const uint64_t w = _pdep_u64(b0, 0x5555555555555555ULL) | _pdep_u64(b1, 0xAAAAAAAAAAAAAAAAULL);
		memcpy(d2 + c, &w, 8);
		const uint32_t nn = ~(uint32_t)_mm256_movemask_epi8(acgt);
		memcpy(dn + c, &nn, 4);
		// exact upper-case ACGTN: the folded compare hit and the byte was not changed by the fold, or it is 'N'
		okv = _mm256_and_si256(okv, _mm256_or_si256(_mm256_and_si256(acgt, _mm256_cmpeq_epi8(x, xf)), _mm256_cmpeq_epi8(x, cN)));
	}
	*bad_out |= ~(unsigned)_mm256_movemask_epi8(okv);
	return c;
}
const bool HAVE_AVX2 = __builtin_cpu_supports("avx2") && __builtin_cpu_supports("bmi2");
#endif

// write one record (n ASCII bases, padded with zero codes to a multiple of 64) at base offset `off` (a multiple of 64).  Every word
// of the record is stored, so the pools need no clearing.  Returns nonzero if a byte was folded.
unsigned pack_record(uint32_t *pool2, uint32_t *pooln, uint64_t off, const uint8_t *s, int64_t n)
{
	uint32_t *d2 = pool2 + (off >> 4); uint16_t *dn = (uint16_t*)pooln + (off >> 4);
	const int64_t chunks = (int64_t)(((uint64_t)n + 63) & ~(uint64_t)63) >> 4;
	unsigned bad = 0;
	int64_t c = 0;
#if defined(__x86_64__)
	if (HAVE_AVX2) c = pack_chunks_avx2(s, n, d2, dn, &bad);
	const __m128i cA = _mm_set1_epi8('A'), cC = _mm_set1_epi8('C'), cG = _mm_set1_epi8('G'), cT = _mm_set1_epi8('T'), cN = _mm_set1_epi8('N'), fold = _mm_set1_epi8((char)0xDF);
	__m128i badv = _mm_setzero_si128();
	for (; (c + 1) * 16 <= n; ++c) {
		const __m128i x = _mm_loadu_si128((const __m128i*)(s + 16 * c));
		const __m128i xf = _mm_and_si128(x, fold); // a-z -> A-Z (other bytes that change are caught by the exact compares below)
		const __m128i eC = _mm_cmpeq_epi8(xf, cC), eG = _mm_cmpeq_epi8(xf, cG), eT = _mm_cmpeq_epi8(xf, cT);
		const __m128i acgt = _mm_or_si128(_mm_or_si128(_mm_cmpeq_epi8(xf, cA), eC), _mm_or_si128(eG, eT));
		const uint32_t b0 = (uint32_t)_mm_movemask_epi8(_mm_or_si128(eC, eT)), b1 = (uint32_t)_mm_movemask_epi8(_mm_or_si128(eG, eT));
		d2[c] = spread16(b0) | (spread16(b1) << 1);
		dn[c] = (uint16_t)(~(uint32_t)_mm_movemask_epi8(acgt));
		// folded: not exactly one of A C G T N in upper case
		const __m128i exact = _mm_or_si128(_mm_or_si128(_mm_cmpeq_epi8(x, cA), _mm_cmpeq_epi8(x, cC)),
		                                   _mm_or_si128(_mm_or_si128(_mm_cmpeq_epi8(x, cG), _mm_cmpeq_epi8(x, cT)), _mm_cmpeq_epi8(x, cN)));
		badv = _mm_or_si128(badv, _mm_andnot_si128(exact, _mm_set1_epi8((char)0xFF)));
	}
	bad |= (unsigned)_mm_movemask_epi8(badv);
#endif
	for (; c < chunks; ++c) {
		const int64_t left = n - 16 * c;
		bad |= pack16_scalar(s + 16 * c, left >= 16 ? 16 : (left > 0 ? (int)left : 0), d2 + c, dn + c);
	}
	return bad;
}

inline uint64_t round64(uint64_t x) { return (x + 63) & ~(uint64_t)63; }

struct Win { int64_t ws, we, max_stop; };

// the reference window a region ships (include/indelope_cuda.h: idl_region.ref_len) and, optionally, the quality trim of its reads
template <class F>
Win region_window(const idlh_roiset *rs, int64_t k, const idl_params *p, F &&per_read)
{
	Win w; w.ws = INT64_MAX; w.max_stop = -1; int64_t far = -1;
	for (int32_t j = 0; j < rs->roi_n_reads[k]; ++j) {
		int64_t i = rs->read_idx[rs->roi_read_begin[k] + j];
		int32_t n; int32_t a = idlh_trim(rs->quals + rs->seq_off[i], rs->len[i], &n);
		per_read(j, i, a, n);
		w.ws = std::min<int64_t>(w.ws, (int64_t)rs->start[i] + a);
		far = std::max<int64_t>(far, (int64_t)rs->start[i] + a + n);
		if (rs->mapq[i] > p->stop_min_mapq) w.max_stop = std::max<int64_t>(w.max_stop, rs->stop[i]);
	}
	if (w.ws == INT64_MAX) w.ws = 0;
	if (w.ws < 0) w.ws = 0;
	w.we = std::min<int64_t>(rs->chrom_len[rs->roi_chrom[k]] - 1, std::max(far, w.max_stop) + p->window_pad);
	return w;
}

// ---- a small fork-join helper: packing a step of the chr1 workload is ~400 Mbases; one core cannot feed the GPU ----
std::atomic<int> g_threads{0};

} // namespace

int pack_threads()
{
	int n = g_threads.load();
	if (n <= 0) { const char *e = getenv("IDLH_THREADS"); n = e ? atoi(e) : 0; }
	if (n <= 0) { n = (int)std::thread::hardware_concurrency(); if (n > 32) n = 32; }
	return n < 1 ? 1 : n;
}

namespace {

// f(begin, end, thread) over [0, n) in blocks handed out dynamically
template <class F>
void parallel_blocks(int64_t n, int64_t block, F &&f)
{
	int nt = pack_threads();
	const int64_t nblocks = (n + block - 1) / block;
	if (nt > nblocks) nt = (int)std::max<int64_t>(1, nblocks);
	if (nt <= 1) { if (n > 0) f((int64_t)0, n, 0); return; }
	std::atomic<int64_t> next{0};
	auto work = [&](int t) { for (;;) { const int64_t b = next.fetch_add(1); if (b >= nblocks) break; f(b * block, std::min(n, (b + 1) * block), t); } };
	std::vector<std::thread> th;
	for (int t = 1; t < nt; ++t) th.emplace_back(work, t);
	work(0);
	for (auto &x : th) x.join();
}

inline bool read_too_long(const idlh_roiset *rs, int64_t i, const idl_params *p) { return rs->len[i] > p->max_read_len || rs->len[i] > 65535; }

} // namespace

extern "C" {

void idlh_set_threads(int n) { g_threads.store(n); }

int32_t idlh_trim(const uint8_t *bq, int32_t n, int32_t *trim_len) // src/indelope.nim:23-38
{
	const int32_t high = n - 1, min_quality = 15;
	int32_t a = 0;
	while (a < high && bq[a] < min_quality) a += 1;
	if (a == high || n <= 0) { *trim_len = 0; return n <= 0 ? 0 : a; }
	int32_t b = high;
	while (b > a && bq[b] < min_quality) b -= 1;
	*trim_len = b - a + 1;
	return a;
}

void idlh_pack_size(const idlh_roiset *rs, int64_t lo, int64_t hi, const idl_params *p, size_t *n_reads, size_t *n_seq_bases, size_t *n_ref_bases)
{
	std::atomic<size_t> nr{0}, sb{0}, rb{0};
	parallel_blocks(hi - lo, 256, [&](int64_t a, int64_t e, int) {
		size_t r = 0, s = 0, w8 = 0;
		for (int64_t k = lo + a; k < lo + e; ++k) {
			r += (size_t)rs->roi_n_reads[k];
			Win w = region_window(rs, k, p, [&](int32_t, int64_t i, int32_t, int32_t) { if (!read_too_long(rs, i, p)) s += round64((uint64_t)rs->len[i]); });
			w8 += round64((uint64_t)std::max<int64_t>(0, w.we - w.ws + 1));
		}
		nr += r; sb += s; rb += w8;
	});
	*n_reads = nr; *n_seq_bases = sb; *n_ref_bases = rb;
}

int idlh_pack(const idlh_roiset *rs, int64_t lo, int64_t hi, const idl_params *p, idl_batch *b)
{
	const int64_t n = hi - lo;
	if (n < 0 || (size_t)n > b->cap_regions) return IDL_E_CAPACITY;
	// read records are laid out region after region: a serial prefix over the regions' read counts
	std::vector<uint64_t> ri0((size_t)n + 1), so((size_t)n + 1), ro((size_t)n + 1);
	ri0[0] = 0;
	for (int64_t k = 0; k < n; ++k) ri0[k + 1] = ri0[k] + (uint64_t)rs->roi_n_reads[lo + k];
	if (ri0[n] > b->cap_reads) return IDL_E_CAPACITY;
	const bool timing = getenv("IDLH_PACK_TIMING") != nullptr;
	auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
	const double t0 = now();
	// pass A: quality trim, read and region records (everything but the pool offsets), sizes
	parallel_blocks(n, 128, [&](int64_t a, int64_t e, int) {
		for (int64_t kk = a; kk < e; ++kk) {
			const int64_t k = lo + kk;
			idl_region &g = b->region[kk];
			memset(&g, 0, sizeof g);
			uint64_t sbases = 0; uint32_t flags = 0;
			idl_read *rd = b->read + ri0[kk];
			Win w = region_window(rs, k, p, [&](int32_t j, int64_t i, int32_t ta, int32_t tl) {
				idl_read &r = rd[j];
				memset(&r, 0, sizeof r);
				r.start = rs->start[i]; r.stop = rs->stop[i]; r.mapq = rs->mapq[i];
				const uint16_t f = rs->flag[i];
				r.flags = ((f & 0x400) || (f & 0x200) || (f & 0x4) || (f & 0x800) || (f & 0x100)) ? 1 : 0; // :40-47
				if (read_too_long(rs, i, p)) { flags |= IDL_RF_READ_TOO_LONG; return; } // packed empty; the device drops the region and says so
				r.len = (uint16_t)rs->len[i]; r.trim_a = (uint16_t)ta; r.trim_len = (uint16_t)tl;
				r.min_overlap = (uint16_t)(int64_t)(0.88 * (double)tl); // :169
				sbases += round64((uint64_t)rs->len[i]);
			});
			g.chrom_id = rs->roi_chrom[k]; g.roi_start = rs->roi_start[k]; g.roi_end = rs->roi_stop[k];
			g.read_begin = (uint32_t)ri0[kk]; g.n_reads = (uint32_t)rs->roi_n_reads[k];
			g.ref_start = (int32_t)w.ws; g.ref_len = (uint32_t)std::max<int64_t>(0, w.we - w.ws + 1);
			g.max_stop = (int32_t)w.max_stop; g.ordinal = (uint32_t)k; g.flags = flags;
			so[kk + 1] = sbases; ro[kk + 1] = round64(g.ref_len);
		}
	});
	so[0] = ro[0] = 0;
	for (int64_t k = 0; k < n; ++k) { so[k + 1] += so[k]; ro[k + 1] += ro[k]; }
	const size_t sb = so[n], rb = ro[n];
	const double t1 = now();
	if (sb > b->cap_seq_bases || rb > b->cap_ref_bases) return IDL_E_CAPACITY;
	// pass B: bases.  Every word of every record is written, so the pools are not cleared first.
	const int nt = pack_threads();
	std::vector<uint32_t> mx_trim((size_t)nt, 1), mx_ref((size_t)nt, 0), mx_reads((size_t)nt, 0); std::vector<size_t> n_small((size_t)nt, 0);
	parallel_blocks(n, 64, [&](int64_t a, int64_t e, int t) {
		for (int64_t kk = a; kk < e; ++kk) {
			const int64_t k = lo + kk;
			idl_region &g = b->region[kk];
			g.ref_off = (uint32_t)ro[kk];
			unsigned bad = pack_record(b->ref2, b->refn, ro[kk], rs->chrom_seq[g.chrom_id] + g.ref_start, g.ref_len);
			uint64_t soff = so[kk];
			idl_read *rd = b->read + ri0[kk];
			for (uint32_t j = 0; j < g.n_reads; ++j) {
				const int64_t i = rs->read_idx[rs->roi_read_begin[k] + j];
				idl_read &r = rd[j];
				r.seq_off = (uint32_t)soff;
				if (r.len == 0 && read_too_long(rs, i, p)) continue;
				bad |= pack_record(b->seq2, b->seqn, soff, rs->bases + rs->seq_off[i], r.len);
				soff += round64((uint64_t)r.len);
				mx_trim[t] = std::max<uint32_t>(mx_trim[t], r.trim_len);
			}
			if (bad) g.flags |= IDL_RF_ALPHABET;
			mx_ref[t] = std::max(mx_ref[t], g.ref_len); mx_reads[t] = std::max(mx_reads[t], g.n_reads);
			n_small[t] += g.n_reads <= 126;
		}
	});
	// guard words behind the pools (the device reads up to two words past a record)
	memset(b->seq2 + sb / 16, 0, 16); memset(b->seqn + sb / 32, 0, 16); memset(b->ref2 + rb / 16, 0, 16); memset(b->refn + rb / 32, 0, 16);
	b->n_regions = (size_t)n; b->n_reads = ri0[n]; b->n_seq_bases = sb; b->n_ref_bases = rb;
	b->max_trim_len = 1; b->max_ref_len = 0; b->max_region_reads = 0; b->n_small_regions = 0;
	for (int t = 0; t < nt; ++t) {
		b->max_trim_len = std::max(b->max_trim_len, mx_trim[t]); b->max_ref_len = std::max(b->max_ref_len, mx_ref[t]);
		b->max_region_reads = std::max(b->max_region_reads, mx_reads[t]); b->n_small_regions += n_small[t];
	}
	b->summary_valid = 1;
	if (timing) fprintf(stderr, "idlh_pack: %lld regions, %d threads: records %.1f ms, bases %.1f ms\n", (long long)n, nt, t1 - t0, now() - t1);
	return IDL_OK;
}

idl_batch *idlh_batch_alloc_host(size_t max_regions, size_t max_reads, size_t max_seq_bases, size_t max_ref_bases)
{
	idl_batch *b = (idl_batch*)calloc(1, sizeof(idl_batch));
	max_seq_bases = round64(max_seq_bases); max_ref_bases = round64(max_ref_bases);
	b->cap_regions = max_regions; b->cap_reads = max_reads; b->cap_seq_bases = max_seq_bases; b->cap_ref_bases = max_ref_bases;
	b->region = (idl_region*)calloc(max_regions + 1, sizeof(idl_region));
	b->read = (idl_read*)calloc(max_reads + 1, sizeof(idl_read));
	b->seq2 = (uint32_t*)calloc(max_seq_bases / 16 + 4, 4); b->seqn = (uint32_t*)calloc(max_seq_bases / 32 + 4, 4);
	b->ref2 = (uint32_t*)calloc(max_ref_bases / 16 + 4, 4); b->refn = (uint32_t*)calloc(max_ref_bases / 32 + 4, 4);
	return b;
}

void idlh_batch_free_host(idl_batch *b)
{
	if (!b) return;
	free(b->region); free(b->read); free(b->seq2); free(b->seqn); free(b->ref2); free(b->refn); free(b);
}

void idlh_unpack(const uint32_t *pool2, const uint32_t *pooln, uint64_t off, int32_t n, char *out)
{
	for (int32_t i = 0; i < n; ++i) {
		uint64_t b = off + (uint64_t)i;
		out[i] = (pooln[b >> 5] >> (b & 31)) & 1 ? 'N' : "ACGT"[(pool2[b >> 4] >> (2 * (b & 15))) & 3];
	}
	out[n] = 0;
}

void idlh_free(void *p) { free(p); }

} // extern "C"

// ------------------------------------------------------------------------------------------------
// VCF: src/indelope.nim:49-116 (Variant), :375-428 (cascade), :598-608 (dedup); src/genotyper.nim
// ------------------------------------------------------------------------------------------------
namespace {

std::string ffmt(double x, int prec) // Nim formatFloat(ffDecimal, precision) == sprintf("%#.*f")
{
	char buf[2600];
	snprintf(buf, sizeof buf, "%#.*f", prec, x);
	return buf;
}

struct Geno { int gt; double gl[3]; double qual; };

Geno genotype(int64_t r, int64_t a, double error) // src/genotyper.nim:36-47, :22-29
{
	Geno g; g.gt = 3; g.gl[0] = g.gl[1] = g.gl[2] = 0; g.qual = 0;
	const double ln2 = std::log(2.0), total = (double)(r + a);
	if (total == 0) return g;
	g.gt = 0;
	for (int G = 0; G < 3; ++G) {
		g.gl[G] = -total * ln2 + (double)r * std::log((double)G * error + (double)(2 - G) * (1 - error)) +
		          (double)a * std::log((double)G * (1 - error) + (double)(2 - G) * error);
		if (g.gl[G] > g.gl[g.gt]) g.gt = G;
	}
	if (g.gt == 0) g.qual = g.gl[0] - std::max(g.gl[1], g.gl[2]);
	else if (g.gt == 1) g.qual = g.gl[1] - std::max(g.gl[0], g.gl[2]);
	else g.qual = g.gl[2] - std::max(g.gl[0], g.gl[1]);
	return g;
}

int distinct(const char *s, size_t n)
{
	bool seen[256] = {false}; int k = 0;
	for (size_t i = 0; i < n; ++i) if (!seen[(uint8_t)s[i]]) { seen[(uint8_t)s[i]] = true; ++k; }
	return k;
}

double mean_of(int64_t sum, int64_t n) // src/indelope.nim:146-150; empty list divides 0.0 by 0.0 at run time
{
	volatile double s = (double)sum, d = (double)n;
	return s / d;
}

std::string fetch(const idlh_roiset *rs, int chrom, int64_t a, int64_t b) // Fai.get: 0-based inclusive, clipped
{
	if (a < 0) a = 0;
	if (b >= rs->chrom_len[chrom]) b = rs->chrom_len[chrom] - 1;
	if (a > b) return std::string();
	return std::string((const char*)rs->chrom_seq[chrom] + a, (size_t)(b - a + 1));
}

std::string cigar_text(const uint32_t *c, int n)
{
	std::string s;
	for (int i = 0; i < n; ++i) { s += std::to_string(c[i] >> 4); s += "MID"[c[i] & 0xf]; }
	return s;
}

struct Rec { std::string chrom, ref, alt, line; int64_t pos; };

} // namespace

struct idlh_vcf { bool have1 = false, have2 = false, dedup = true; Rec last1, last2; uint64_t status_count[8] = {0}; int warned = 0; };

namespace {
const char *const RS_NAMES[8] = {"a contig outgrew max_contig_len (region dropped)", "more than 128 voting sites in one merge (region dropped)",
                                 "an alignment exceeded the DP workspace (its events are not called)", "a CIGAR exceeded the scratch capacity (its events are not called)",
                                 "a read longer than max_read_len (region dropped)", "bases outside {A,C,G,T,N} were folded (acgt -> ACGT, others -> N); the reference compares raw characters",
                                 "malformed read record (region dropped)", "unknown"};
}

extern "C" {

idlh_vcf *idlh_vcf_new(void) { return new idlh_vcf(); }
void idlh_vcf_set_dedup(idlh_vcf *w, int on) { w->dedup = on != 0; }
void idlh_vcf_status_counts(const idlh_vcf *w, uint64_t out[8]) { for (int i = 0; i < 8; ++i) out[i] = w->status_count[i]; }

char *idlh_vcf_dedup(const char *records) { return idlh_vcf_dedup_n(records, strlen(records), nullptr); }

// the same over a buffer of `n` bytes that need not be terminated (the gathered shards of a multi-GPU run: tens of megabytes per
// genome).  In place: lines are compared where they lie and the kept ones are moved down over the dropped ones, so nothing but an
// index of the dropped lines is allocated; returns the new length.
//
// The dedup is a two-key state machine over the lines in order (a line is dropped when its CHROM, POS, REF, ALT equal those of one of
// the last two KEPT lines, src/indelope.nim:604-608) -- sequential by definition.  It is run on all host threads exactly:
//   1. the buffer is cut at line ends into one chunk per thread; every chunk runs the machine from the EMPTY state and notes its drops;
//   2. the chunks are stitched in order: chunk c is run again from the TRUE state the previous chunk ends in, side by side with the
//      empty-state run, until both machines hold the same two lines in the same order -- from there on they agree for ever, so the
//      rest of the chunk's phase-1 decisions stand (usually after two kept lines);
//   3. the dropped lines are squeezed out, run by run.
namespace {
struct DdKey { const char *chrom, *pos, *ref, *alt; size_t lc, lp, lr, la; const char *line; };
inline bool dd_same(const DdKey &x, const DdKey &y)
{
	return x.lp == y.lp && x.lc == y.lc && x.lr == y.lr && x.la == y.la && !memcmp(x.pos, y.pos, x.lp) && !memcmp(x.chrom, y.chrom, x.lc) &&
	       !memcmp(x.ref, y.ref, x.lr) && !memcmp(x.alt, y.alt, x.la);
}
struct DdState { DdKey k1{}, k2{}; bool h1 = false, h2 = false; };
// next line of [p, end): returns false at the end; *line / *le its bounds (no terminator), *key filled when the line has the six leading fields
inline bool dd_next(const char *&p, const char *end, const char *&line, const char *&le, DdKey &k, bool &keyed)
{
	for (;;) {
		if (p >= end) return false;
		const char *e = (const char*)memchr(p, '\n', (size_t)(end - p));
		le = e ? e : end; line = p; p = e ? e + 1 : end;
		if (le == line) continue;   // empty lines vanish
		break;
	}
	const char *f[6]; int nf = 0; f[nf++] = line;
	for (const char *q = line; q < le && nf < 6; ) { const char *t = (const char*)memchr(q, '\t', (size_t)(le - q)); if (!t) break; f[nf++] = t + 1; q = t + 1; }
	keyed = nf == 6;
	if (keyed) {
		k.chrom = f[0]; k.lc = (size_t)(f[1] - 1 - f[0]); k.pos = f[1]; k.lp = (size_t)(f[2] - 1 - f[1]);
		k.ref = f[3]; k.lr = (size_t)(f[4] - 1 - f[3]); k.alt = f[4]; k.la = (size_t)(f[5] - 1 - f[4]); k.line = line;
	}
	return true;
}
// one step of the machine: true = the line is kept
inline bool dd_step(DdState &S, const DdKey &k, bool keyed)
{
	if (!keyed) return true;   // a line without the fields is passed through and leaves the state alone
	if ((S.h1 && dd_same(k, S.k1)) || (S.h2 && dd_same(k, S.k2))) return false;
	S.k2 = S.k1; S.h2 = S.h1; S.k1 = k; S.h1 = true;
	return true;
}
inline bool dd_converged(const DdState &a, const DdState &b) { return a.h1 && a.h2 && b.h1 && b.h2 && a.k1.line == b.k1.line && a.k2.line == b.k2.line; }
} // namespace

size_t idlh_vcf_dedup_inplace(char *records, size_t n)
{
	const char *end = records + n;
	int nt = pack_threads();
	if (n < (1u << 20)) nt = 1;
	// chunk starts at line starts
	std::vector<const char*> cut((size_t)nt + 1, end);
	cut[0] = records;
	for (int c = 1; c < nt; ++c) {
		const char *q = records + n / (size_t)nt * (size_t)c;
		if (q < cut[(size_t)c - 1]) q = cut[(size_t)c - 1];
		const char *e = q < end ? (const char*)memchr(q, '\n', (size_t)(end - q)) : nullptr;
		cut[(size_t)c] = e ? e + 1 : end;
	}
	struct Span { const char *b, *e; };            // a dropped line (with its newline) or an empty line
	std::vector<std::vector<Span>> drops((size_t)nt);
	std::vector<DdState> final_state((size_t)nt);
	auto run_chunk = [&](int c) {
		DdState S; const char *p = cut[(size_t)c], *ce = cut[(size_t)c + 1];
		const char *line, *le; DdKey k{}; bool keyed;
		const char *expect = p;
		while (dd_next(p, ce, line, le, k, keyed)) {
			if (line != expect) drops[(size_t)c].push_back({expect, line});          // empty lines in front of this one
			if (!dd_step(S, k, keyed)) drops[(size_t)c].push_back({line, p});
			expect = p;
		}
		if (expect != ce) drops[(size_t)c].push_back({expect, ce});
		final_state[(size_t)c] = S;
	};
	if (nt > 1) {
		std::vector<std::thread> th;
		for (int c = 1; c < nt; ++c) th.emplace_back(run_chunk, c);
		run_chunk(0);
		for (auto &x : th) x.join();
	} else run_chunk(0);
	// 2. stitch
	DdState T = final_state[0];
	for (int c = 1; c < nt; ++c) {
		DdState L;   // the empty-state machine of phase 1, replayed
		const char *p = cut[(size_t)c], *ce = cut[(size_t)c + 1];
		const char *line, *le; DdKey k{}; bool keyed;
		std::vector<Span> head; const char *expect = p; bool conv = false; const char *conv_at = ce;
		while (dd_next(p, ce, line, le, k, keyed)) {
			if (line != expect) head.push_back({expect, line});
			dd_step(L, k, keyed);
			if (!dd_step(T, k, keyed)) head.push_back({line, p});
			expect = p;
			if (dd_converged(T, L)) { conv = true; conv_at = p; break; }
		}
		if (conv) {
			// phase-1 drops from the convergence point on stand; the ones before it are replaced by the stitched ones
			std::vector<Span> &d = drops[(size_t)c];
			size_t i = 0; while (i < d.size() && d[i].b < conv_at) ++i;
			head.insert(head.end(), d.begin() + (long)i, d.end());
			d.swap(head);
			T = final_state[(size_t)c];
		} else {
			if (expect != ce) head.push_back({expect, ce});
			drops[(size_t)c].swap(head);   // the whole chunk was decided by the stitched run; T already holds its final state
		}
	}
	// 3. squeeze the dropped spans out (they are in address order).  Sequentially that is one pass of memmove over everything behind the first
	// drop -- as long as the whole parse.  With threads: every chunk's kept runs are copied to their final offsets in a scratch buffer (the
	// offsets follow from the drops before the chunk), then copied back, both in parallel.
	size_t n_drops = 0;
	for (auto &d : drops) n_drops += d.size();
	size_t w = 0;
	if (n_drops == 0) w = n;
	else if (nt == 1) {
		const char *src = records;
		auto take = [&](const char *b, const char *e) { if (e > b) { if (records + w != b) memmove(records + w, b, (size_t)(e - b)); w += (size_t)(e - b); } };
		for (const Span &d : drops[0]) { take(src, d.b); src = d.e; }
		take(src, end);
	} else {
		std::vector<size_t> dst((size_t)nt + 1, 0);   // final offset of each chunk's first kept byte
		for (int c = 0; c < nt; ++c) {
			size_t dropped = 0;
			for (const Span &d : drops[(size_t)c]) dropped += (size_t)(d.e - d.b);
			dst[(size_t)c + 1] = dst[(size_t)c] + (size_t)(cut[(size_t)c + 1] - cut[(size_t)c]) - dropped;
		}
		w = dst[(size_t)nt];
		int first = 0;
		while (first < nt && drops[(size_t)first].empty()) ++first;   // chunks in front of the first drop stay where they are
		const size_t base = dst[(size_t)first];
		static thread_local std::vector<char> scratch;
		if (scratch.size() < w - base) scratch.resize(w - base + (w - base) / 8);
		char *const sp = scratch.data();   // (the workers must not name the thread_local themselves: they would see their own, empty one)
		auto squeeze = [&](int c) {
			char *o = sp + (dst[(size_t)c] - base);
			const char *src = cut[(size_t)c];
			for (const Span &d : drops[(size_t)c]) { if (d.b > src) { memcpy(o, src, (size_t)(d.b - src)); o += d.b - src; } src = d.e; }
			if (cut[(size_t)c + 1] > src) memcpy(o, src, (size_t)(cut[(size_t)c + 1] - src));
		};
		auto back = [&](int c) { memcpy(records + dst[(size_t)c], sp + (dst[(size_t)c] - base), dst[(size_t)c + 1] - dst[(size_t)c]); };
		for (int pass = 0; pass < 2; ++pass) {
			std::vector<std::thread> th;
			for (int c = first + 1; c < nt; ++c) { if (pass == 0) th.emplace_back(squeeze, c); else th.emplace_back(back, c); }
			if (pass == 0) squeeze(first); else back(first);
			for (auto &x : th) x.join();
		}
	}
	// a kept last line without a newline gets one, as the sequential version wrote it
	if (w && records[w - 1] != '\n') records[w++] = '\n';
	return w;
}

char *idlh_vcf_dedup_n(const char *records, size_t n, size_t *out_len)
{
	char *o = (char*)malloc(n + 2);
	memcpy(o, records, n);
	const size_t w = idlh_vcf_dedup_inplace(o, n);
	o[w] = 0;
	if (out_len) *out_len = w;
	return o;
}
void idlh_vcf_free(idlh_vcf *w) { delete w; }

char *idlh_vcf_header(const idlh_roiset *rs) // src/indelope.nim:77-102,548-552,600
{
	static const char *fixed[] = {
	    "##fileformat=VCFv4.2",
	    "##FORMAT=<ID=AD,Number=R,Type=Integer,Description=\"Allelic depths for the ref and alt alleles in the order listed\">",
	    "##INFO=<ID=AD,Number=R,Type=Integer,Description=\"Allelic depths for the ref and alt alleles in the order listed\">",
	    "##INFO=<ID=END,Number=1,Type=Integer,Description=\"End position of the variant described in this record\">",
	    "##INFO=<ID=SVLEN,Number=1,Type=Integer,Description=\"Difference in length between REF and ALT alleles\">",
	    "##INFO=<ID=DP,Number=1,Type=Integer,Description=\"total reads covering this site\">",
	    "##INFO=<ID=AL,Number=0,Type=Flag,Description=\"this was genotyped with alignment, no k-mer counting\">",
	    "##INFO=<ID=AMQ,Number=1,Type=Integer,Description=\"median mapping quality of alts\">",
	    "##INFO=<ID=RMQ,Number=1,Type=Integer,Description=\"median mapping quality of refs\">",
	    "##INFO=<ID=BS,Number=1,Type=Integer,Description=\"number of times there was support for both ref and alt k-mer in a single read\">",
	    "##INFO=<ID=MF,Number=1,Type=Integer,Description=\"minimum matching bases around this event when BS > 0. Higher gives more confidence\">",
	    "##INFO=<ID=CF,Number=1,Type=Integer,Description=\"minimum flank of the event from either end of the contig. higher is better.\">",
	    "##INFO=<ID=NC,Number=1,Type=Integer,Description=\"number of contigs at the site of this variant.\">",
	    "##INFO=<ID=CC,Number=1,Type=String,Description=\"contig cigar from alignment to reference\">",
	    "##INFO=<ID=LO,Number=0,Type=Flag,Description=\"low-offset: the event occurred near at the start of the contig so we may not have the full variant\">",
	    "##INFO=<ID=AKE,Number=1,Type=Float,Description=\"mean alt-kmer distance from end of read\">",
	    "##INFO=<ID=RKE,Number=1,Type=Float,Description=\"mean ref-kmer distance from end of read\">",
	    "##FORMAT=<ID=DP,Number=1,Type=Integer,Description=\"supporting k-mer depth\">",
	    "##FORMAT=<ID=GQ,Number=1,Type=Float,Description=\"Genotype Quality\">",
	    "##FORMAT=<ID=GT,Number=1,Type=String,Description=\"Genotype\">",
	    "##FORMAT=<ID=GL,Number=G,Type=Float,Description=\"Normalized, Phred-scaled likelihoods for genotypes as defined in the VCF specification\">",
	    "##INFO=<ID=DP,Number=1,Type=Integer,Description=\"Approximate read depth; some reads may have been filtered\">",
	    "##INFO=<ID=ref_kmer,Number=1,Type=String,Description=\"reference kmer used for genotyping\">",
	    "##INFO=<ID=alt_kmer,Number=1,Type=String,Description=\"alternate kmer used for genotyping\">"};
	std::string h;
	for (const char *l : fixed) { h += l; h += "\n"; }
	std::vector<std::string> cl;
	for (int c = 0; c < rs->n_chroms; ++c) cl.push_back("##contig=<ID=" + std::string(rs->chrom_name[c]) + ",length=" + std::to_string(rs->chrom_len[c]) + ">");
	for (size_t i = 0; i < cl.size(); ++i) { if (i) h += "\n"; h += cl[i]; }
	h += "\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tsample\n";
	char *out = (char*)malloc(h.size() + 1);
	memcpy(out, h.c_str(), h.size() + 1);
	return out;
}

char *idlh_vcf_records(idlh_vcf *w, const idlh_roiset *rs, int64_t lo, const idl_params *P, const idl_results *res, int32_t dump_level, char **dump_out)
{
	const int K = IDL_KMER;
	static const char *gt_enc[] = {"0/0", "0/1", "1/1", "./."};
	// Regions are independent up to the order-dependent dedup: the cascade and the text of every region are made on all host cores (the
	// host cascade of a chr1-sized step, 85 k regions, took 46 ms on one core against 38 ms of GPU time), the dedup then walks the
	// candidate records in region order on one.
	const size_t nreg = res->n_regions;
	std::vector<std::vector<Rec>> cand(nreg);
	std::vector<std::string> dtext(dump_level ? nreg : 0);
	auto do_region = [&](size_t i) {
		const idl_region_result &rr = res->region[i];
		const int64_t k = lo + (int64_t)i;
		const int chrom = rs->roi_chrom[k];
		const int64_t n_region_reads = rs->roi_n_reads[k];
		std::vector<Rec> &out = cand[i];
		std::string dlocal;
		std::string &d = dump_level ? dtext[i] : dlocal;
		if (dump_level & 1) {
			d += "R\t" + std::to_string(k) + "\tpre=" + std::to_string(rr.n_contigs_pre) + "\tn=" + std::to_string(rr.n_contigs) + "\n";
			for (int32_t ci = 0; ci < rr.n_contigs; ++ci) {
				const idl_contig_result &c = res->contig[rr.contig_begin + ci];
				d += "C\t" + std::to_string(k) + "\t" + std::to_string(ci) + "\t" + std::to_string(c.start) + "\t" + std::to_string(c.nreads) + "\t" +
				     std::to_string(c.len) + "\t" + std::string(res->contig_seq + c.seq_off, (size_t)c.len);
				if (dump_level & 2) {
					d += "\t";
					for (int32_t x = 0; x < c.len; ++x) { if (x) d += ","; d += std::to_string(res->contig_support ? res->contig_support[c.seq_off + x] : 0u); }
				}
				d += "\n";
			}
		}
		for (int32_t ci = 0; ci < rr.n_contigs; ++ci) {
			const idl_contig_result &c = res->contig[rr.contig_begin + ci];
			if (c.aln < 0) continue;
			const idl_aln_result &a = res->aln[c.aln];
			const uint32_t *cig = res->cigar + a.cigar_off;
			const char *ctg = res->contig_seq + c.seq_off;
			if (dump_level & 4) {
				char b[256];
				snprintf(b, sizeof b, "A\t%lld\t%d\t%d\t%d\t%d\t%d\t%d\t%d\t%d\t%d\t%d\t%d\t%d\t", (long long)k, ci, c.start, a.ref_len, a.max, a.zdropped,
				         a.max_q, a.max_t, a.mqe, a.mqe_t, a.mte, a.mte_q, a.score);
				d += b; d += cigar_text(cig, a.n_cigar) + "\t" + cigar_text(cig, a.n_cigar_trunc) + "\n";
			}
			if (a.n_events < 1 || a.n_events > P->max_events || a.event_begin == IDL_NO_EVENTS || a.status) continue; // src/indelope.nim:229
			for (int32_t ei = 0; ei < a.n_events; ++ei) {
				const idl_event_result &e = res->event[a.event_begin + ei];
				const bool have_kmers = e.reject != IDL_EV_SHORT && e.reject != IDL_EV_WINDOW;
				std::string ref_kmer, alt_kmer;
				if (have_kmers) {
					ref_kmer = fetch(rs, chrom, (int64_t)c.start + e.tstart, (int64_t)c.start + e.tstart + K - 1);
					alt_kmer = std::string(ctg + e.qstart, (size_t)K);
				}
				if (dump_level & 8) {
					char b[512];
					snprintf(b, sizeof b, "E\t%lld\t%d\t%d\t%c\t%d\t%d\t%d\t%d\t%d\t%d\t%d\t%d\t", (long long)k, ci, e.index, e.type == 0 ? 'I' : 'D', e.t_start, e.t_stop,
					         e.len, e.q_start, e.q_stop, e.reject, e.tstart, e.qstart);
					d += b; d += (have_kmers ? ref_kmer : std::string(".")) + "\t" + (have_kmers ? alt_kmer : std::string("."));
					snprintf(b, sizeof b, "\t%d\t%d\t%d\t%d\t%d\t%d\t%d\t%d\t%lld\t%d\t%lld\t%d\t%d\t%d\t%d\n", e.k_ref, e.k_alt, e.k_both, e.aligned, e.ref_support,
					         e.alt_support, e.both_found, e.n_adist, (long long)e.sum_adist, e.n_rdist, (long long)e.sum_rdist, e.amq_median, e.rmq_median,
					         e.min_flank, e.offset);
					d += b;
				}
				if (e.reject != IDL_EV_COUNTED) continue;
				// ---- cascade, src/indelope.nim:375-428
				const int64_t ref_support = e.ref_support, alt_support = e.alt_support, both_found = e.both_found, offset = e.offset;
				if (alt_support < P->min_reads) continue;
				if ((double)alt_support / (double)n_region_reads < 0.1) continue;
				Geno g = genotype(ref_support, alt_support, 1e-3);
				if (g.gt == 0) continue;
				double qual = g.qual;
				if (offset == 0 && both_found >= (int64_t)(0.75 * (double)std::min(ref_support, alt_support))) continue;
				std::string info = "DP=" + std::to_string(n_region_reads);
				if (offset < 5) { info += ";LO"; qual /= 2.0; }
				if (both_found > 0) { info += ";BS=" + std::to_string(both_found); qual /= 1.5; }
				else qual *= 2;
				info += ";CC=" + cigar_text(cig, a.n_cigar_trunc);
				if (e.aligned) info += ";AL";
				if ((int64_t)(e.min_flank - 1) < std::max<int64_t>(e.t_stop - e.t_start, e.q_stop - e.q_start)) continue;
				info += ";MF=" + std::to_string(e.min_flank);
				info += ";CF=" + std::to_string(offset);
				info += ";NC=" + std::to_string(rr.n_contigs_pre);
				if (offset == 0) qual /= 4.0;
				const double ake = mean_of(e.sum_adist, e.n_adist), rke = mean_of(e.sum_rdist, e.n_rdist);
				info += ";AKE=" + ffmt(ake, 2);
				info += ";RKE=" + ffmt(rke, 2);
				if (e.n_adist > 0) info += ";AMQ=" + std::to_string(e.amq_median);
				if (e.n_rdist > 0) info += ";RMQ=" + std::to_string(e.rmq_median);
				if (ake < 5) continue;
				Rec v; v.chrom = rs->chrom_name[chrom]; v.pos = e.t_start;
				if (e.type == 1) {
					v.ref = fetch(rs, chrom, (int64_t)e.t_start - 1, (int64_t)e.t_stop - 1);
					v.alt = v.ref.substr(0, 1);
				} else {
					if (e.q_start < 1) continue; // the reference indexes ctg.sequence[-1]: unsupported, never reached with an M-led CIGAR
					v.ref = fetch(rs, chrom, (int64_t)e.t_start - 1, (int64_t)e.t_start - 1);
					v.alt = std::string(ctg + e.q_start - 1, (size_t)(e.q_stop - (e.q_start - 1)));
					if (distinct(v.alt.data() + 1, v.alt.size() - 1) == 1 && distinct(alt_kmer.data() + K - 11, 11) == 1 &&
					    distinct(ref_kmer.data() + K - 11, 11) == 1)
						continue;
				}
				v.line = v.chrom + "\t" + std::to_string(v.pos) + "\t.\t" + v.ref + "\t" + v.alt + "\t" + ffmt(qual, 2) + "\tPASS\t" + "AD=" +
				         std::to_string(ref_support) + "," + std::to_string(alt_support) + ";ref_kmer=" + ref_kmer + ";alt_kmer=" + alt_kmer + ";" + info +
				         "\tGT:GQ:GL\t" + gt_enc[g.gt] + ":" + ffmt(g.qual, 4) + ":" + ffmt(g.gl[0], 4) + "," + ffmt(g.gl[1], 4) + "," + ffmt(g.gl[2], 4);
				out.push_back(std::move(v));
			}
		}
	};
	if (nreg < 256) for (size_t i = 0; i < nreg; ++i) do_region(i);
	else parallel_blocks((int64_t)nreg, 256, [&](int64_t a, int64_t e, int) { for (int64_t i = a; i < e; ++i) do_region((size_t)i); });
	std::string vcf, d;
	auto same = [](const Rec &x, const Rec &y) { return x.pos == y.pos && x.chrom == y.chrom && x.ref == y.ref && x.alt == y.alt; };
	for (size_t i = 0; i < nreg; ++i) {
		const idl_region_result &rr = res->region[i];
		if (rr.status) { // never silent: the output for this region may differ from the reference's (include/indelope_cuda.h IDL_RS_*)
			const int64_t k = lo + (int64_t)i;
			for (int bit = 0; bit < 8; ++bit)
				if (rr.status & (1u << bit)) {
					w->status_count[bit] += 1;
					if (w->warned < 20) {
						fprintf(stderr, "indelope: warning: region %s:%d-%d: %s\n", rs->chrom_name[rs->roi_chrom[k]], rs->roi_start[k], rs->roi_stop[k], RS_NAMES[bit]);
						if (++w->warned == 20) fprintf(stderr, "indelope: further region warnings are counted, not printed\n");
					}
				}
		}
		if (dump_level) d += dtext[i];
		for (Rec &v : cand[i]) {
			// order-dependent dedup against the last two emitted records, src/indelope.nim:604-608
			if (w->dedup && w->have1 && same(v, w->last1)) continue;
			if (w->dedup && w->have2 && same(v, w->last2)) continue;
			vcf += v.line; vcf += "\n";
			if (dump_level & 16) { d += "V\t"; d += v.line; d += "\n"; }
			w->last2 = std::move(w->last1); w->have2 = w->have1;
			w->last1 = std::move(v); w->have1 = true;
		}
	}
	if (dump_out) { *dump_out = (char*)malloc(d.size() + 1); memcpy(*dump_out, d.c_str(), d.size() + 1); }
	char *out = (char*)malloc(vcf.size() + 1);
	memcpy(out, vcf.c_str(), vcf.size() + 1);
	return out;
}

} // extern "C"
