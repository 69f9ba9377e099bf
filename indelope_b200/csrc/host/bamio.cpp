// indelope_b200/csrc/host/bamio.cpp -- file I/O of the host stand-in, written from the SAM/BAM specification on zlib
// (no htslib / hts-nim in this image):
//
//   * FASTA + .fai reader  (the reference opens it with hts-nim's open_fai and slices it with fai.get,
//     src/indelope.nim:213-220,414,421,583) and a writer for the synthetic references
//   * BGZF + BAM reader    (the reference iterates `b.querys(target.name)` over a coordinate-sorted, indexed BAM,
//     src/indelope.nim:527,593-602; a sequential pass over a sorted BAM visits the same records in the same order)
//     with multi-threaded block inflation: the `-t/--threads` option of the reference's CLI (:566)
//   * BGZF + BAM writer    so that the synthetic configs exist as real .bam/.fa/.fai files (SURVEY.md 8f rows 1-2)
//
// hts-nim field semantics reproduced here (SURVEY.md appendix D): start = pos (0-based), stop = bam_endpos (pos + reference
// bases consumed, at least pos + 1), sequence() = the 4-bit codes through "=ACMGRSVTWYHKDBN" (soft clips included),
// base_qualities() = raw phred bytes, cigar ops as in the file.
#include <algorithm>
#include <atomic>
#include <map>
#include <memory>
#include <condition_variable>
#include <deque>
#include <mutex>
#include <sys/stat.h>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>
#include <zlib.h>
#include "indelope_host.h"
#include "dataset.h"

namespace {

void set_err(char *err, size_t n, const std::string &msg) { if (err && n) { snprintf(err, n, "%s", msg.c_str()); } }

bool read_file(const char *path, std::vector<uint8_t> &out, std::string &why)
{
	FILE *f = fopen(path, "rb");
	if (!f) { why = std::string("cannot open ") + path; return false; }
	fseek(f, 0, SEEK_END);
	const long n = ftell(f);
	fseek(f, 0, SEEK_SET);
	if (n < 0) { fclose(f); why = std::string("cannot size ") + path; return false; }
	out.resize((size_t)n);
	const size_t got = n ? fread(out.data(), 1, (size_t)n, f) : 0;
	fclose(f);
	if (got != (size_t)n) { why = std::string("short read on ") + path; return false; }
	return true;
}

inline uint16_t le16(const uint8_t *p) { return (uint16_t)(p[0] | p[1] << 8); }
inline uint32_t le32(const uint8_t *p) { return (uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24; }
inline void put16(std::vector<uint8_t> &v, uint16_t x) { v.push_back((uint8_t)x); v.push_back((uint8_t)(x >> 8)); }
inline void put32(std::vector<uint8_t> &v, uint32_t x) { for (int i = 0; i < 4; ++i) v.push_back((uint8_t)(x >> (8 * i))); }

// ---------------------------------------------------------------------------------------------------------------
// BGZF (SAM spec 4.1): gzip members of at most 64 KiB with a 'BC' extra subfield holding the member size
// ---------------------------------------------------------------------------------------------------------------
struct BgzfBlock { size_t off, csize; size_t uoff, usize; };

bool bgzf_index(const std::vector<uint8_t> &file, std::vector<BgzfBlock> &blocks, size_t &total, std::string &why)
{
	size_t at = 0; total = 0;
	while (at < file.size()) {
		if (file.size() - at < 18) { why = "truncated BGZF header"; return false; }
		const uint8_t *h = file.data() + at;
		if (h[0] != 0x1f || h[1] != 0x8b || h[2] != 8 || !(h[3] & 4)) { why = "not a BGZF file (is it BAM? CRAM is not supported by this stand-in)"; return false; }
		const unsigned xlen = le16(h + 10);
		if (file.size() - at < 12 + xlen) { why = "truncated BGZF extra field"; return false; }
		int bsize = -1;
		for (unsigned x = 0; x + 4 <= xlen;) {
			const uint8_t *e = h + 12 + x; const unsigned slen = le16(e + 2);
			if (e[0] == 'B' && e[1] == 'C' && slen == 2) bsize = le16(e + 4);
			x += 4 + slen;
		}
		if (bsize < 0) { why = "BGZF block without BC subfield"; return false; }
		const size_t csize = (size_t)bsize + 1;
		if (csize < 12 + xlen + 8 || file.size() - at < csize) { why = "truncated BGZF block"; return false; }
		const size_t usize = le32(h + csize - 4);
		blocks.push_back({at, csize, total, usize});
		total += usize; at += csize;
	}
	return true;
}

bool bgzf_inflate_block(const std::vector<uint8_t> &file, const BgzfBlock &b, uint8_t *dst)
{
	if (b.usize == 0) return true;
	const uint8_t *h = file.data() + b.off;
	const unsigned xlen = le16(h + 10);
	z_stream zs; memset(&zs, 0, sizeof zs);
	if (inflateInit2(&zs, -15) != Z_OK) return false;
	zs.next_in = const_cast<Bytef*>(h + 12 + xlen); zs.avail_in = (uInt)(b.csize - 12 - xlen - 8);
	zs.next_out = dst; zs.avail_out = (uInt)b.usize;
	const int rc = inflate(&zs, Z_FINISH);
	inflateEnd(&zs);
	if (rc != Z_STREAM_END || zs.avail_out != 0) return false;
	return (uint32_t)crc32(crc32(0L, Z_NULL, 0), dst, (uInt)b.usize) == le32(h + b.csize - 8);
}

// every member of a BGZF file's bytes inflated (and CRC-checked) by `threads` workers
bool bgzf_inflate_all(const std::vector<uint8_t> &file, int threads, std::vector<uint8_t> &out, std::string &why)
{
	std::vector<BgzfBlock> blocks; size_t total = 0;
	if (!bgzf_index(file, blocks, total, why)) return false;
	out.resize(total);
	std::atomic<size_t> next(0); std::atomic<bool> ok(true);
	auto work = [&]() {
		for (;;) {
			const size_t i = next.fetch_add(16);
			if (i >= blocks.size() || !ok.load()) return;
			for (size_t k = i; k < std::min(i + 16, blocks.size()); ++k)
				if (!bgzf_inflate_block(file, blocks[k], out.data() + blocks[k].uoff)) { ok.store(false); return; }
		}
	};
	if (threads < 1) threads = 1;
	std::vector<std::thread> pool;
	for (int t = 1; t < threads; ++t) pool.emplace_back(work);
	work();
	for (auto &t : pool) t.join();
	if (!ok.load()) { why = "BGZF block failed to inflate (corrupt data or CRC mismatch)"; return false; }
	return true;
}

bool bgzf_read_all(const char *path, int threads, std::vector<uint8_t> &out, std::string &why)
{
	std::vector<uint8_t> file;
	if (!read_file(path, file, why)) return false;
	return bgzf_inflate_all(file, threads, out, why);
}

struct BgzfWriter {
	FILE *f = nullptr; std::vector<uint8_t> buf; int level = 1; bool ok = true;
	uint64_t coff = 0; // compressed bytes written so far = file offset of the block being filled
	uint64_t tell() const { return coff << 16 | (uint64_t)buf.size(); } // virtual file offset (SAM spec 4.1.1)
	void flush_block(const uint8_t *p, size_t n)
	{
		std::vector<uint8_t> out(18 + compressBound((uLong)n) + 8);
		z_stream zs; memset(&zs, 0, sizeof zs);
		if (deflateInit2(&zs, level, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY) != Z_OK) { ok = false; return; }
		zs.next_in = const_cast<Bytef*>(p); zs.avail_in = (uInt)n;
		zs.next_out = out.data() + 18; zs.avail_out = (uInt)(out.size() - 18 - 8);
		const int rc = deflate(&zs, Z_FINISH);
		const size_t clen = zs.total_out;
		deflateEnd(&zs);
		if (rc != Z_STREAM_END) { ok = false; return; }
		const size_t bsize = 18 + clen + 8;
		static const uint8_t hdr[16] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0};
		memcpy(out.data(), hdr, 16);
		out[16] = (uint8_t)((bsize - 1) & 0xff); out[17] = (uint8_t)((bsize - 1) >> 8);
		const uint32_t crc = (uint32_t)crc32(crc32(0L, Z_NULL, 0), p, (uInt)n);
		for (int i = 0; i < 4; ++i) { out[18 + clen + i] = (uint8_t)(crc >> (8 * i)); out[18 + clen + 4 + i] = (uint8_t)((uint32_t)n >> (8 * i)); }
		if (fwrite(out.data(), 1, bsize, f) != bsize) ok = false;
		coff += bsize;
	}
	void write(const uint8_t *p, size_t n)
	{
		const size_t CAP = 0xff00; // uncompressed bytes per block, the value htslib uses
		while (n) {
			const size_t take = std::min(n, CAP - buf.size());
			buf.insert(buf.end(), p, p + take); p += take; n -= take;
			if (buf.size() == CAP) { flush_block(buf.data(), buf.size()); buf.clear(); }
		}
	}
	void close()
	{
		if (!buf.empty()) { flush_block(buf.data(), buf.size()); buf.clear(); }
		static const uint8_t eof[28] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
		if (fwrite(eof, 1, 28, f) != 28) ok = false;
		if (fclose(f) != 0) ok = false;
		f = nullptr;
	}
};

int reg2bin(int64_t beg, int64_t end) // SAM spec 5.3
{
	--end;
	if (beg >> 14 == end >> 14) return (int)(((1 << 15) - 1) / 7 + (beg >> 14));
	if (beg >> 17 == end >> 17) return (int)(((1 << 12) - 1) / 7 + (beg >> 17));
	if (beg >> 20 == end >> 20) return (int)(((1 << 9) - 1) / 7 + (beg >> 20));
	if (beg >> 23 == end >> 23) return (int)(((1 << 6) - 1) / 7 + (beg >> 23));
	if (beg >> 26 == end >> 26) return (int)(((1 << 3) - 1) / 7 + (beg >> 26));
	return 0;
}

// BAI index (SAM spec 5.2): per reference the binning index (bin -> chunks of virtual offsets) and the 16 kb linear index
struct BaiRef { std::map<uint32_t, std::vector<std::pair<uint64_t, uint64_t>>> bins; std::vector<uint64_t> lin; };
struct BaiBuilder {
	std::vector<BaiRef> refs;
	void add(int ref, int64_t beg, int64_t end, uint64_t v0, uint64_t v1)
	{
		if (ref < 0 || (size_t)ref >= refs.size()) return;
		if (end <= beg) end = beg + 1;
		BaiRef &R = refs[(size_t)ref];
		auto &ch = R.bins[(uint32_t)reg2bin(beg, end)];
		if (!ch.empty() && ch.back().second == v0) ch.back().second = v1; else ch.push_back({v0, v1}); // records of one bin written back to back are one chunk
		const size_t w0 = (size_t)(beg >> 14), w1 = (size_t)((end - 1) >> 14);
		if (R.lin.size() <= w1) R.lin.resize(w1 + 1, 0);
		for (size_t w = w0; w <= w1; ++w) if (R.lin[w] == 0) R.lin[w] = v0; // first record that overlaps the window (the file is coordinate sorted)
	}
	bool write(const std::string &path) const
	{
		std::vector<uint8_t> b = {'B', 'A', 'I', 1};
		put32(b, (uint32_t)refs.size());
		auto put64 = [&](uint64_t x) { for (int i = 0; i < 8; ++i) b.push_back((uint8_t)(x >> (8 * i))); };
		for (const BaiRef &R : refs) {
			put32(b, (uint32_t)R.bins.size());
			for (const auto &kv : R.bins) {
				put32(b, kv.first); put32(b, (uint32_t)kv.second.size());
				for (const auto &c : kv.second) { put64(c.first); put64(c.second); }
			}
			put32(b, (uint32_t)R.lin.size());
			uint64_t last = 0;
			for (size_t w = 0; w < R.lin.size(); ++w) { if (R.lin[w]) last = R.lin[w]; put64(last); } // empty windows carry the previous offset on, as htslib writes them
		}
		FILE *f = fopen(path.c_str(), "wb");
		if (!f) return false;
		const bool ok = fwrite(b.data(), 1, b.size(), f) == b.size();
		return fclose(f) == 0 && ok;
	}
};

const char SEQ16[] = "=ACMGRSVTWYHKDBN";
// two bases per packed byte (high nibble first)
struct Seq16Pairs { uint8_t t[256][2]; Seq16Pairs() { for (int i = 0; i < 256; ++i) { t[i][0] = (uint8_t)SEQ16[i >> 4]; t[i][1] = (uint8_t)SEQ16[i & 15]; } } };
const Seq16Pairs SEQ16_PAIRS;
inline void decode_seq16(const uint8_t *packed, uint32_t n, uint8_t *out)
{
	uint32_t i = 0;
	for (; i + 2 <= n; i += 2) { const uint8_t *p = SEQ16_PAIRS.t[packed[i >> 1]]; out[i] = p[0]; out[i + 1] = p[1]; }
	if (i < n) out[i] = SEQ16_PAIRS.t[packed[i >> 1]][0];
}
inline uint8_t code16(uint8_t c)
{
	switch (c) {
	case 'A': case 'a': return 1; case 'C': case 'c': return 2; case 'G': case 'g': return 4; case 'T': case 't': return 8;
	case '=': return 0; case 'M': return 3; case 'R': return 5; case 'S': return 6; case 'V': return 7; case 'W': return 9; case 'Y': return 10;
	case 'H': return 11; case 'K': return 12; case 'D': return 13; case 'B': return 14; default: return 15;
	}
}

// ---------------------------------------------------------------------------------------------------------------
// FASTA
// ---------------------------------------------------------------------------------------------------------------
// A FASTA file, plain or compressed with bgzip (ref.fa.gz: what htslib's fai_load opens for the reference's open_fai, src/indelope.nim:593); the
// BGZF members are inflated on pack_threads() threads.  Plain gzip is refused, as fai_load refuses it.
bool load_fasta(const char *path, idlh_dataset &D, std::string &why)
{
	std::vector<uint8_t> file;
	if (!read_file(path, file, why)) return false;
	if (file.size() >= 2 && file[0] == 0x1f && file[1] == 0x8b) {
		std::vector<uint8_t> text;
		if (!bgzf_inflate_all(file, pack_threads(), text, why)) {
			if (why.compare(0, 15, "not a BGZF file") == 0 || why == "BGZF block without BC subfield")
				why = "gzip member without the BGZF BC subfield (plain gzip)";
			why = std::string(path) + ": " + why + "; a compressed FASTA must be compressed with bgzip (recompress it with bgzip)";
			return false;
		}
		file.swap(text);
	}
	size_t i = 0; const size_t n = file.size();
	while (i < n) {
		if (file[i] != '>') { why = std::string("FASTA record does not start with '>' in ") + path; return false; }
		size_t e = i + 1;
		while (e < n && file[e] != '\n') ++e;
		std::string name((const char*)file.data() + i + 1, e - i - 1);
		const size_t ws = name.find_first_of(" \t\r");
		if (ws != std::string::npos) name.resize(ws);
		i = e < n ? e + 1 : n;
		std::vector<uint8_t> seq;
		while (i < n && file[i] != '>') {
			size_t le = i;
			while (le < n && file[le] != '\n') ++le;
			size_t re = le;
			while (re > i && (file[re - 1] == '\r' || file[re - 1] == ' ')) --re;
			seq.insert(seq.end(), file.begin() + (long)i, file.begin() + (long)re);
			i = le < n ? le + 1 : n;
		}
		D.names.push_back(name); D.chroms.push_back(std::move(seq));
	}
	return true;
}

// fixed part of one BAM alignment record (SAM spec 4.2) and pointers to its variable parts
struct BamFields { int32_t ref_id, pos; uint8_t mapq; uint16_t flag; unsigned n_cig; uint32_t l_seq; const uint8_t *cig, *seq, *qual; };
inline bool bam_fields(const uint8_t *b, uint32_t block, BamFields &f)
{
	f.ref_id = (int32_t)le32(b); f.pos = (int32_t)le32(b + 4);
	const unsigned l_name = b[8]; f.mapq = b[9];
	f.n_cig = le16(b + 12); f.flag = le16(b + 14); f.l_seq = le32(b + 16);
	if (32 + (size_t)l_name + 4 * (size_t)f.n_cig + ((size_t)f.l_seq + 1) / 2 + f.l_seq > block) return false;
	f.cig = b + 32 + l_name; f.seq = f.cig + 4 * f.n_cig; f.qual = f.seq + (f.l_seq + 1) / 2;
	return true;
}
// reference bases the record spans, as bam_endpos counts them (hts-nim's `stop`)
inline int64_t bam_ref_span(const BamFields &f)
{
	int64_t rlen = 0;
	for (unsigned k = 0; k < f.n_cig; ++k) {
		const uint32_t c = le32(f.cig + 4 * k); const unsigned op = c & 0xf;
		if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) rlen += c >> 4;
	}
	if ((f.flag & 4) || f.n_cig == 0 || rlen == 0) rlen = 1;
	return rlen;
}

void rois_finish_view(idlh_rois &R, const idlh_dataset &ref);

} // namespace

extern "C" {

int idlh_write_fasta(const idlh_dataset *d, const char *path)
{
	FILE *f = fopen(path, "wb");
	if (!f) return -1;
	const std::string fai_path = std::string(path) + ".fai";
	FILE *fi = fopen(fai_path.c_str(), "wb");
	if (!fi) { fclose(f); return -1; }
	const int W = 60;
	long long off = 0;
	for (size_t c = 0; c < d->chroms.size(); ++c) {
		off += fprintf(f, ">%s\n", d->names[c].c_str());
		const std::vector<uint8_t> &s = d->chroms[c];
		fprintf(fi, "%s\t%zu\t%lld\t%d\t%d\n", d->names[c].c_str(), s.size(), off, W, W + 1);
		for (size_t i = 0; i < s.size(); i += W) {
			const size_t k = std::min<size_t>(W, s.size() - i);
			fwrite(s.data() + i, 1, k, f); fputc('\n', f);
			off += (long long)k + 1;
		}
	}
	const bool ok = fclose(f) == 0;
	return (fclose(fi) == 0 && ok) ? 0 : -1;
}

/* coordinate-sorted BAM of the dataset's reads: @HD SO:coordinate, one @SQ per chromosome, read names r<serial>, no mates, no tags */
int idlh_write_bam(const idlh_dataset *d, const char *path, int level)
{
	BgzfWriter w;
	w.f = fopen(path, "wb");
	if (!w.f) return -1;
	w.level = level < 0 ? 1 : (level > 9 ? 9 : level);
	std::vector<uint8_t> b;
	std::string text = "@HD\tVN:1.6\tSO:coordinate\n";
	for (size_t c = 0; c < d->chroms.size(); ++c) text += "@SQ\tSN:" + d->names[c] + "\tLN:" + std::to_string(d->chroms[c].size()) + "\n";
	text += "@PG\tID:indelope_b200\tPN:indelope_b200\n";
	b.insert(b.end(), {'B', 'A', 'M', 1});
	put32(b, (uint32_t)text.size()); b.insert(b.end(), text.begin(), text.end());
	put32(b, (uint32_t)d->chroms.size());
	for (size_t c = 0; c < d->chroms.size(); ++c) {
		put32(b, (uint32_t)d->names[c].size() + 1); b.insert(b.end(), d->names[c].begin(), d->names[c].end()); b.push_back(0);
		put32(b, (uint32_t)d->chroms[c].size());
	}
	w.write(b.data(), b.size());
	BaiBuilder bai; bai.refs.resize(d->chroms.size());
	for (const IdlhReadRec &r : d->reads) {
		b.clear();
		const uint64_t v0 = w.tell();
		char name[32];
		const int ln = snprintf(name, sizeof name, "r%llu", (unsigned long long)r.order) + 1;
		const uint32_t block = 32 + (uint32_t)ln + 4u * (uint32_t)r.n_cig + (uint32_t)(r.len + 1) / 2 + (uint32_t)r.len;
		put32(b, block); put32(b, (uint32_t)r.chrom); put32(b, (uint32_t)r.start);
		b.push_back((uint8_t)ln); b.push_back(r.mapq); put16(b, (uint16_t)reg2bin(r.start, r.stop > r.start ? r.stop : r.start + 1));
		put16(b, (uint16_t)r.n_cig); put16(b, r.flag); put32(b, (uint32_t)r.len);
		put32(b, 0xffffffffu); put32(b, 0xffffffffu); put32(b, 0);
		b.insert(b.end(), name, name + ln);
		for (int k = 0; k < r.n_cig; ++k) put32(b, d->cigars[(size_t)r.cig_off + k]);
		const uint8_t *s = d->bases.data() + r.seq_off, *q = d->quals.data() + r.seq_off;
		for (int i = 0; i < r.len; i += 2) b.push_back((uint8_t)(code16(s[i]) << 4 | (i + 1 < r.len ? code16(s[i + 1]) : 0)));
		b.insert(b.end(), q, q + r.len);
		w.write(b.data(), b.size());
		bai.add(r.chrom, r.start, r.stop, v0, w.tell());
	}
	w.close();
	if (!w.ok) return -1;
	return bai.write(std::string(path) + ".bai") ? 0 : -1; // the reference opens its BAM with index=true (src/indelope.nim:595)
}

/* reference FASTA + coordinate-sorted BAM -> dataset.  Records without a reference id are dropped (a per-target query never
 * returns them); everything else, flags included, is kept for the sweep's `skippable` test (src/indelope.nim:40-47). */
} // extern "C"

namespace {

// What the region front ends need of <bam>.bai (SAM spec 5.2), per target: the smallest chunk begin and the largest chunk end of its bins (the virtual
// offsets of its first record and of the byte behind its last one) and its 16 kb linear index.  The index read last is kept (a header with thousands of
// targets asks for them one after the other, a region list for one target after the other).
struct BaiSummary { std::vector<std::pair<uint64_t, uint64_t>> span; std::vector<std::vector<uint64_t>> lin; };

bool bai_summary(const char *bam_path, std::shared_ptr<const BaiSummary> &out, std::string &why)
{
	static std::mutex mu; static std::string cached_path; static long long cached_stamp = -1; static std::shared_ptr<const BaiSummary> cached;
	std::lock_guard<std::mutex> lock(mu);
	long long stamp = -1;
	{ struct stat sb; if (stat((std::string(bam_path) + ".bai").c_str(), &sb) == 0) stamp = (long long)sb.st_mtime * 1000003LL + (long long)sb.st_size; }
	if (cached_path != bam_path || stamp != cached_stamp) {
		cached_path.clear(); cached.reset();
		std::vector<uint8_t> bai;
		if (!read_file((std::string(bam_path) + ".bai").c_str(), bai, why)) { why += " (no index: write one with idlh_write_bam or samtools index)"; return false; }
		if (bai.size() < 8 || memcmp(bai.data(), "BAI\1", 4) != 0) { why = "not a BAI index"; return false; }
		size_t ia = 4;
		auto rd32 = [&](uint32_t &x) -> bool { if (ia + 4 > bai.size()) return false; x = le32(bai.data() + ia); ia += 4; return true; };
		auto rd64 = [&](uint64_t &x) -> bool { if (ia + 8 > bai.size()) return false; x = (uint64_t)le32(bai.data() + ia) | (uint64_t)le32(bai.data() + ia + 4) << 32; ia += 8; return true; };
		uint32_t n_ref = 0;
		BaiSummary S;
		if (!rd32(n_ref)) { why = "truncated index"; return false; }
		for (uint32_t r = 0; r < n_ref; ++r) {
			uint64_t lo = ~0ULL, hi = 0;
			uint32_t n_bin = 0;
			if (!rd32(n_bin)) { why = "truncated index"; return false; }
			for (uint32_t b = 0; b < n_bin; ++b) {
				uint32_t bin = 0, n_chunk = 0;
				if (!rd32(bin) || !rd32(n_chunk)) { why = "truncated index"; return false; }
				for (uint32_t c = 0; c < n_chunk; ++c) {
					uint64_t a = 0, z = 0;
					if (!rd64(a) || !rd64(z)) { why = "truncated index"; return false; }
					if (bin != 37450u) { lo = std::min(lo, a); hi = std::max(hi, z); }   // 37450: the metadata pseudo-bin of samtools
				}
			}
			uint32_t n_intv = 0;
			if (!rd32(n_intv) || ia + (size_t)n_intv * 8 > bai.size()) { why = "truncated index"; return false; }
			std::vector<uint64_t> lin(n_intv);
			for (uint32_t w = 0; w < n_intv; ++w) rd64(lin[w]);
			S.span.push_back({lo, hi}); S.lin.push_back(std::move(lin));
		}
		cached = std::make_shared<const BaiSummary>(std::move(S)); cached_path = bam_path; cached_stamp = stamp;
	}
	out = cached;
	return true;
}

// the run of whole BGZF members that holds the records at virtual offsets [vbeg, vend), as idl_bam_open_slice takes it
int member_run(const char *bam_path, uint64_t vbeg, uint64_t vend, uint64_t *file_begin, uint64_t *file_end, uint64_t *first_record, uint64_t *end_member,
               uint64_t *end_offset, char *err, size_t errlen)
{
	*file_begin = vbeg >> 16; *first_record = vbeg & 0xffff;
	const uint64_t ce = vend >> 16, ue = vend & 0xffff;
	*end_member = ce - *file_begin; *end_offset = ue;
	if (ue == 0) { *file_end = ce; return 0; }
	// the member the records end in is part of the run: its size is in its own header
	FILE *f = fopen(bam_path, "rb");
	if (!f) { set_err(err, errlen, std::string("cannot open ") + bam_path); return -1; }
	uint8_t h[18];
	const bool ok = fseek(f, (long)ce, SEEK_SET) == 0 && fread(h, 1, 18, f) == 18 && h[0] == 0x1f && h[1] == 0x8b && h[12] == 'B' && h[13] == 'C';
	fclose(f);
	if (!ok) { set_err(err, errlen, "the index points between BGZF blocks"); return -1; }
	*file_end = ce + (uint64_t)le16(h + 16) + 1;
	return 0;
}

bool is_decoy(const std::string &name) { return name == "hs37d5" || name.compare(0, 2, "GL") == 0; }   // skippable targets, src/indelope.nim:41-42

} // namespace

extern "C" {

/* Where the records of one target lie in the BAM file, from <bam>.bai (SAM spec 5.2): the smallest chunk begin and the largest chunk end of the target's
 * bins are the virtual offsets of its first record and of the byte behind its last one.  [*file_begin, *file_end) is the run of whole BGZF members that
 * holds them, *first_record the offset of the first record inside the inflated bytes of that run, (*end_member, *end_offset) the end as idl_bam_open_slice
 * takes it.  Returns 0, 1 when the index lists no record for the target, -1 on error. */
int idlh_bai_target_span(const char *bam_path, int32_t target, uint64_t *file_begin, uint64_t *file_end, uint64_t *first_record, uint64_t *end_member,
                         uint64_t *end_offset, char *err, size_t errlen)
{
	std::shared_ptr<const BaiSummary> P; std::string why;
	if (!bai_summary(bam_path, P, why)) { set_err(err, errlen, why); return -1; }
	const BaiSummary &S = *P;
	if (target < 0 || (size_t)target >= S.span.size()) { set_err(err, errlen, "the index has no such target"); return -1; }
	const uint64_t vmin = S.span[(size_t)target].first, vmax = S.span[(size_t)target].second;
	if (vmin == ~0ULL || vmax <= vmin) return 1;
	return member_run(bam_path, vmin, vmax, file_begin, file_end, first_record, end_member, end_offset, err, errlen);
}

/* The records of one target from the first record of 16 kb window w0 to the first record of window w1 + 1 (or to the target's last record), by the linear
 * index of <bam>.bai.  Every record in front of the run ends at or before position W0 = w0 << 14 (that is what the linear index records; an empty window
 * holds an earlier offset, which only moves the run's start forward in the file), so the evidence, cuts and record lists of positions >= *zone_lo =
 * W0 + 1 are those of the whole file -- 0 when w0 == 0 or the run starts at the target's first record (DESIGN.md 4a).  *to_end = 1 when the run ends
 * behind the target's last record.  The run as idl_bam_open_slice takes it.  Returns 0, 1 when the run holds no record, -1 on error. */
int idlh_bai_region_run(const char *bam_path, int32_t target, int64_t w0, int64_t w1, uint64_t *file_begin, uint64_t *file_end, uint64_t *first_record,
                        uint64_t *end_member, uint64_t *end_offset, int64_t *zone_lo, int32_t *to_end, char *err, size_t errlen)
{
	std::shared_ptr<const BaiSummary> P; std::string why;
	if (!bai_summary(bam_path, P, why)) { set_err(err, errlen, why); return -1; }
	const BaiSummary &S = *P;
	if (target < 0 || (size_t)target >= S.span.size()) { set_err(err, errlen, "the index has no such target"); return -1; }
	if (w0 < 0 || w1 < w0) { set_err(err, errlen, "bad window range"); return -1; }
	const uint64_t vmin = S.span[(size_t)target].first, vmax = S.span[(size_t)target].second;
	const std::vector<uint64_t> &lin = S.lin[(size_t)target];
	*zone_lo = 0; *to_end = 1;
	if (vmin == ~0ULL || vmax <= vmin) return 1;
	auto first_of = [&](int64_t w) -> uint64_t {   // the first record of window w; the target's end behind its last window
		if ((uint64_t)w >= lin.size()) return vmax;
		const uint64_t o = lin[(size_t)w];
		return o < vmin ? vmin : (o > vmax ? vmax : o);   // 0: no record up to this window (htslib writes empty windows so)
	};
	const uint64_t vb = first_of(w0), ve = std::max(vb, first_of(w1 + 1));
	*to_end = ve >= vmax;
	*zone_lo = (w0 == 0 || vb == vmin) ? 0 : (w0 << 14) + 1;
	if (ve <= vb) return 1;
	return member_run(bam_path, vb, ve, file_begin, file_end, first_record, end_member, end_offset, err, errlen);
}

/* -r / -R: region strings (1-based, inclusive, as samtools takes them) and BED lines (0-based, half open) -> per target sorted, merged half-open intervals */
struct idlh_regions { std::vector<std::vector<std::pair<int64_t, int64_t>>> iv; };

idlh_regions *idlh_regions_parse(int32_t n_ref, const char *const *ref_name, const int64_t *ref_len, int32_t n_region, const char *const *region, const char *bed_path,
                                 char *err, size_t errlen)
{
	auto R = std::unique_ptr<idlh_regions>(new idlh_regions());
	R->iv.resize(n_ref > 0 ? (size_t)n_ref : 0);
	std::map<std::string, int32_t> tid;
	for (int32_t c = 0; c < n_ref; ++c) tid[ref_name[c]] = c;
	std::vector<char> noted((size_t)std::max(n_ref, 0), 0);
	auto add = [&](int32_t c, int64_t b, int64_t e) {
		if (is_decoy(ref_name[c])) {
			if (!noted[(size_t)c]) fprintf(stderr, "indelope: note: %s is a decoy target and is not called\n", ref_name[c]);
			noted[(size_t)c] = 1;
			return;
		}
		b = std::min(b, ref_len[c]); e = std::min(e, ref_len[c]);
		if (b < e) R->iv[(size_t)c].push_back({b, e});
	};
	// a number with optional thousands commas; false if anything else is there
	auto number = [](const std::string &t, int64_t &x) -> bool {
		std::string d;
		for (char ch : t) { if (ch == ',') continue; if (ch < '0' || ch > '9') return false; d += ch; }
		if (d.empty() || d.size() > 15) return false;
		x = std::stoll(d);
		return true;
	};
	for (int32_t k = 0; k < n_region; ++k) {
		const std::string r = region[k];
		auto bad = [&](const std::string &why) -> idlh_regions* { set_err(err, errlen, "region '" + r + "': " + why); return nullptr; };
		auto it = tid.find(r);   // a whole target, also one whose name contains ':'
		if (it != tid.end()) { add(it->second, 0, ref_len[it->second]); continue; }
		const size_t colon = r.rfind(':');
		if (colon == std::string::npos) return bad("no such target in the BAM header");
		const std::string name = r.substr(0, colon), rest = r.substr(colon + 1);
		it = tid.find(name);
		if (it == tid.end()) return bad("no such target in the BAM header");
		const size_t dash = rest.find('-');
		int64_t beg = 0, end = ref_len[it->second];
		if (!number(rest.substr(0, dash), beg)) return bad("expected chr[:beg[-end]] with numbers");
		if (dash != std::string::npos && dash + 1 < rest.size() && !number(rest.substr(dash + 1), end)) return bad("expected chr[:beg[-end]] with numbers");
		if (beg < 1) return bad("beg must be >= 1 (1-based)");
		if (end < beg) return bad("end must be >= beg");
		add(it->second, beg - 1, end);
	}
	if (bed_path && *bed_path) {
		std::vector<uint8_t> f; std::string why;
		if (!read_file(bed_path, f, why)) { set_err(err, errlen, why); return nullptr; }
		size_t at = 0; int64_t line_no = 0;
		while (at < f.size()) {
			size_t e = at;
			while (e < f.size() && f[e] != '\n') ++e;
			std::string line((const char*)f.data() + at, e - at);
			at = e + 1; ++line_no;
			while (!line.empty() && (line.back() == '\r' || line.back() == ' ' || line.back() == '\t')) line.pop_back();
			if (line.empty() || line[0] == '#' || line.compare(0, 5, "track") == 0 || line.compare(0, 7, "browser") == 0) continue;
			std::vector<std::string> col;
			for (size_t p = 0; p <= line.size() && col.size() < 3; ) {
				size_t q = line.find_first_of("\t ", p);
				if (q == std::string::npos) q = line.size();
				if (q > p) col.push_back(line.substr(p, q - p));
				p = q + 1;
			}
			auto bad = [&](const std::string &w) -> idlh_regions* { set_err(err, errlen, std::string(bed_path) + " line " + std::to_string(line_no) + ": " + w); return nullptr; };
			if (col.size() < 3) return bad("expected chrom, start and end");
			const auto it = tid.find(col[0]);
			if (it == tid.end()) return bad("target '" + col[0] + "' is not in the BAM header");
			int64_t b = 0, en = 0;
			if (col[1].find(',') != std::string::npos || col[2].find(',') != std::string::npos || !number(col[1], b) || !number(col[2], en)) return bad("start and end must be non-negative integers");
			if (en < b) return bad("end is smaller than start");
			add(it->second, b, en);
		}
	}
	for (auto &v : R->iv) {   // sorted and merged: overlapping or touching intervals become one
		std::sort(v.begin(), v.end());
		std::vector<std::pair<int64_t, int64_t>> m;
		for (const auto &x : v) { if (!m.empty() && x.first <= m.back().second) m.back().second = std::max(m.back().second, x.second); else m.push_back(x); }
		v.swap(m);
	}
	return R.release();
}

int64_t idlh_regions_get(const idlh_regions *r, int32_t target, int64_t *beg, int64_t *end, int64_t cap)
{
	if (!r || target < 0 || (size_t)target >= r->iv.size()) return 0;
	const auto &v = r->iv[(size_t)target];
	for (size_t k = 0; k < v.size() && (int64_t)k < cap; ++k) { beg[k] = v[k].first; end[k] = v[k].second; }
	return (int64_t)v.size();
}

void idlh_regions_free(idlh_regions *r) { delete r; }

/* The FASTA's sequences ordered as the BAM header lists its targets, WITHOUT reading the BAM's records: only the first members of the file are read and
 * inflated, as far as the header reaches (what `open(b, path)` + `b.hdr.targets` give the reference's main, src/indelope.nim:595-601).  For the path that
 * decodes the records on the device target by target (idl_bam_open_slice).  Same checks and messages as idlh_load. */
idlh_dataset *idlh_load_targets(const char *fasta_path, const char *bam_path, char *err, size_t errlen)
{
	idlh_dataset *D = new idlh_dataset();
	memset(&D->P, 0, sizeof D->P);
	std::string why;
	if (!load_fasta(fasta_path, *D, why)) { set_err(err, errlen, why); delete D; return nullptr; }
	if (idlh_dataset_set_bam_targets(D, bam_path, err, errlen) != 0) { delete D; return nullptr; }
	return D;
}

/* idlh_dataset_set_targets with the targets of <bam_path>'s header: only the first members of the file are read and inflated, as far as the header
 * reaches.  Same checks and messages as idlh_load.  0 = ok. */
int idlh_dataset_set_bam_targets(idlh_dataset *D, const char *bam_path, char *err, size_t errlen)
{
	auto fail = [&](const std::string &m) -> int { set_err(err, errlen, m); return 1; };
	FILE *f = fopen(bam_path, "rb");
	if (!f) return fail(std::string("cannot open ") + bam_path);
	std::vector<uint8_t> file, u; size_t cpos = 0; bool eof = false;
	// inflate members from the front until `bytes` of the stream are there
	auto need = [&](size_t bytes) -> bool {
		while (u.size() < bytes) {
			while (!eof && (file.size() - cpos < 18 || file.size() - cpos < (size_t)le16(file.data() + cpos + 16) + 1)) {
				const size_t o = file.size(); file.resize(o + (1u << 20));
				const size_t got = fread(file.data() + o, 1, 1u << 20, f);
				file.resize(o + got);
				if (got == 0) eof = true;
			}
			if (file.size() - cpos < 18) return false;
			const uint8_t *h = file.data() + cpos;
			if (h[0] != 0x1f || h[1] != 0x8b || h[2] != 8 || !(h[3] & 4) || h[12] != 'B' || h[13] != 'C') return false;
			const size_t csize = (size_t)le16(h + 16) + 1;
			if (file.size() - cpos < csize || csize < 26) return false;
			BgzfBlock b{cpos, csize, u.size(), le32(h + csize - 4)};
			const size_t o = u.size(); u.resize(o + b.usize);
			if (!bgzf_inflate_block(file, b, u.data() + o)) return false;
			cpos += csize;
		}
		return true;
	};
	auto done = [&](int r) { fclose(f); return r; };
	if (!need(12) || memcmp(u.data(), "BAM\1", 4) != 0) return done(fail(std::string(bam_path) + ": not a BAM file"));
	size_t at = 4;
	const uint32_t l_text = le32(u.data() + at); at += 4;
	if (!need(at + l_text + 4)) return done(fail("truncated BAM header"));
	at += l_text;
	const uint32_t n_ref = le32(u.data() + at); at += 4;
	std::vector<std::string> names; std::vector<std::vector<uint8_t>> chroms;
	for (uint32_t r = 0; r < n_ref; ++r) {
		if (!need(at + 4)) return done(fail("truncated BAM reference list"));
		const uint32_t l_name = le32(u.data() + at); at += 4;
		if (l_name == 0 || !need(at + l_name + 4)) return done(fail("truncated BAM reference list"));
		const std::string name((const char*)u.data() + at, l_name - 1); at += l_name;
		const uint32_t l_ref = le32(u.data() + at); at += 4;
		size_t k = 0;
		while (k < D->names.size() && D->names[k] != name) ++k;
		if (k == D->names.size()) return done(fail("BAM target " + name + " is not in the FASTA"));
		if (D->chroms[k].size() != l_ref) return done(fail("BAM target " + name + " has a different length than the FASTA record"));
		names.push_back(name); chroms.push_back(D->chroms[k]);
	}
	D->names.swap(names); D->chroms.swap(chroms);
	return done(0);
}

/* the reference sequences alone (the device reads the BAM: idl_bam_open) */
idlh_dataset *idlh_load_fasta(const char *fasta_path, char *err, size_t errlen)
{
	idlh_dataset *D = new idlh_dataset();
	memset(&D->P, 0, sizeof D->P);
	std::string why;
	if (!load_fasta(fasta_path, *D, why)) { set_err(err, errlen, why); delete D; return nullptr; }
	return D;
}

/* a reference from names and sequences found elsewhere (idl_fasta_open: a bgzipped FASTA parsed on the device); everything is copied */
idlh_dataset *idlh_dataset_from_sequences(int32_t n, const char *const *names, const uint8_t *const *seqs, const int64_t *lens)
{
	idlh_dataset *D = new idlh_dataset();
	memset(&D->P, 0, sizeof D->P);
	for (int32_t k = 0; k < n; ++k) { D->names.emplace_back(names[k]); D->chroms.emplace_back(seqs[k], seqs[k] + lens[k]); }
	return D;
}

/* order the sequences as the BAM header lists its targets (the VCF header and the sweep follow the BAM's target order, src/indelope.nim:599-601);
 * same checks and messages as idlh_load.  0 = ok. */
int idlh_dataset_set_targets(idlh_dataset *D, int32_t n_ref, const char *const *ref_name, const int64_t *ref_len, char *err, size_t errlen)
{
	std::vector<std::string> names; std::vector<std::vector<uint8_t>> chroms;
	for (int32_t r = 0; r < n_ref; ++r) {
		const std::string name(ref_name[r]);
		size_t k = 0;
		while (k < D->names.size() && D->names[k] != name) ++k;
		if (k == D->names.size()) { set_err(err, errlen, "BAM target " + name + " is not in the FASTA"); return 1; }
		if ((int64_t)D->chroms[k].size() != ref_len[r]) { set_err(err, errlen, "BAM target " + name + " has a different length than the FASTA record"); return 1; }
		names.push_back(name); chroms.push_back(D->chroms[k]);
	}
	D->names.swap(names); D->chroms.swap(chroms);
	return 0;
}

/* regions and their records found elsewhere (idl_bam_sweep + idl_bam_fetch: BAM decode and gen_roi on the GPU) as an idlh_rois over the sequences of
 * <d>: the arrays describe n_reads records (seq_off has n_reads + 1 entries), read_idx indexes them.  Everything is copied. */
idlh_rois *idlh_rois_from_arrays(const idlh_dataset *d, int64_t n_reads, const int32_t *start, const int32_t *stop, const int32_t *len, const uint8_t *mapq, const uint16_t *flag,
                                 const int64_t *seq_off, const uint8_t *bases, const uint8_t *quals, int64_t n_rois, const int32_t *roi_chrom, const int32_t *roi_start,
                                 const int32_t *roi_stop, const int32_t *roi_n_reads, const int64_t *read_idx)
{
	idlh_rois *R = new idlh_rois();
	const size_t n = (size_t)n_reads;
	R->start.assign(start, start + n); R->stop.assign(stop, stop + n); R->len.assign(len, len + n); R->mapq.assign(mapq, mapq + n); R->flag.assign(flag, flag + n);
	R->seq_off.assign(seq_off, seq_off + n);
	const size_t nb = n ? (size_t)seq_off[n] : 0;
	R->own_bases.assign(bases, bases + nb); R->own_quals.assign(quals, quals + nb);
	int64_t at = 0;
	for (int64_t k = 0; k < n_rois; ++k) {
		R->roi_chrom.push_back(roi_chrom[k]); R->roi_start.push_back(roi_start[k]); R->roi_stop.push_back(roi_stop[k]);
		R->roi_read_begin.push_back(at); R->roi_n_reads.push_back(roi_n_reads[k]);
		at += roi_n_reads[k];
	}
	R->read_idx.assign(read_idx, read_idx + at);
	rois_finish_view(*R, *d);
	return R;
}

idlh_dataset *idlh_load(const char *fasta_path, const char *bam_path, int threads, char *err, size_t errlen)
{
	idlh_dataset *D = new idlh_dataset();
	memset(&D->P, 0, sizeof D->P);
	std::string why;
	auto fail = [&](const std::string &m) -> idlh_dataset* { set_err(err, errlen, m); delete D; return nullptr; };
	if (!load_fasta(fasta_path, *D, why)) return fail(why);
	std::vector<uint8_t> bam;
	if (!bgzf_read_all(bam_path, threads, bam, why)) return fail(std::string(bam_path) + ": " + why);
	const uint8_t *p = bam.data(); const size_t n = bam.size();
	if (n < 12 || memcmp(p, "BAM\1", 4) != 0) return fail(std::string(bam_path) + ": not a BAM file");
	size_t at = 4;
	const uint32_t l_text = le32(p + at); at += 4;
	if (at + l_text + 4 > n) return fail("truncated BAM header");
	at += l_text;
	const uint32_t n_ref = le32(p + at); at += 4;
	// map BAM reference ids onto FASTA records by name; the VCF header and the sweep follow the BAM's target order (:599-601)
	std::vector<std::string> names; std::vector<std::vector<uint8_t>> chroms;
	for (uint32_t r = 0; r < n_ref; ++r) {
		if (at + 4 > n) return fail("truncated BAM reference list");
		const uint32_t l_name = le32(p + at); at += 4;
		if (at + l_name + 4 > n || l_name == 0) return fail("truncated BAM reference list");
		const std::string name((const char*)p + at, l_name - 1); at += l_name;
		const uint32_t l_ref = le32(p + at); at += 4;
		size_t k = 0;
		while (k < D->names.size() && D->names[k] != name) ++k;
		if (k == D->names.size()) return fail("BAM target " + name + " is not in the FASTA");
		if (D->chroms[k].size() != l_ref) return fail("BAM target " + name + " has a different length than the FASTA record");
		names.push_back(name); chroms.push_back(D->chroms[k]);
	}
	D->names.swap(names); D->chroms.swap(chroms);
	int32_t last_ref = 0, last_pos = -1;
	while (at + 4 <= n) {
		const uint32_t block = le32(p + at); at += 4;
		if (block < 32 || at + block > n) return fail("truncated BAM record");
		const uint8_t *b = p + at; at += block;
		BamFields f;
		if (!bam_fields(b, block, f)) return fail("malformed BAM record");
		if (f.ref_id < 0) continue;
		if ((uint32_t)f.ref_id >= n_ref) return fail("BAM record with an unknown reference id");
		if (f.ref_id < last_ref || (f.ref_id == last_ref && f.pos < last_pos)) return fail("BAM is not coordinate sorted");
		last_ref = f.ref_id; last_pos = f.pos;
		IdlhReadRec r;
		r.chrom = f.ref_id; r.start = f.pos; r.mapq = f.mapq; r.flag = f.flag; r.len = (int32_t)f.l_seq;
		r.seq_off = (int64_t)D->bases.size(); r.cig_off = (int64_t)D->cigars.size(); r.n_cig = (int32_t)f.n_cig; r.order = D->reads.size();
		for (unsigned k = 0; k < f.n_cig; ++k) D->cigars.push_back(le32(f.cig + 4 * k));
		r.stop = (int32_t)(f.pos + bam_ref_span(f));
		{ const size_t o = D->bases.size(); D->bases.resize(o + f.l_seq); decode_seq16(f.seq, f.l_seq, D->bases.data() + o); }
		D->quals.insert(D->quals.end(), f.qual, f.qual + f.l_seq);
		D->reads.push_back(r);
	}
	if (at != n) return fail("trailing bytes after the last BAM record");
	return D;
}

/* `b.querys(region)` (src/indelope.nim:454-459 single_roi, :527 per target): the records of <bam> that overlap target:beg-end (0-based,
 * half open; beg = 0, end <= 0: the whole target) found THROUGH THE INDEX <bam>.bai -- candidate bins of the region (SAM spec 5.3),
 * their chunks, cut below the linear index' offset for the region's first 16 kb window -- and only those BGZF blocks are inflated.
 * Returns a dataset with the FASTA's sequences for the BAM's targets and just those records, in file order. */
idlh_dataset *idlh_load_region(const char *fasta_path, const char *bam_path, const char *target, int64_t beg, int64_t end, char *err, size_t errlen)
{
	idlh_dataset *D = new idlh_dataset();
	memset(&D->P, 0, sizeof D->P);
	std::string why;
	auto fail = [&](const std::string &m) -> idlh_dataset* { set_err(err, errlen, m); delete D; return nullptr; };
	if (!load_fasta(fasta_path, *D, why)) return fail(why);
	std::vector<uint8_t> file, bai;
	if (!read_file(bam_path, file, why)) return fail(why);
	if (!read_file((std::string(bam_path) + ".bai").c_str(), bai, why)) return fail(why + " (no index: write one with idlh_write_bam or samtools index)");
	std::vector<BgzfBlock> blocks; size_t total = 0;
	if (!bgzf_index(file, blocks, total, why)) return fail(std::string(bam_path) + ": " + why);
	auto block_at = [&](uint64_t coff) -> long {
		size_t lo = 0, hi = blocks.size();
		while (lo < hi) { const size_t mid = (lo + hi) / 2; if (blocks[mid].off < coff) lo = mid + 1; else hi = mid; }
		return lo < blocks.size() && blocks[lo].off == coff ? (long)lo : -1;
	};
	// the header: inflate blocks from the start until the reference list is complete
	std::vector<uint8_t> u; size_t nb = 0;
	auto need = [&](size_t bytes) -> bool {
		while (u.size() < bytes && nb < blocks.size()) { const size_t o = u.size(); u.resize(o + blocks[nb].usize); if (!bgzf_inflate_block(file, blocks[nb], u.data() + o)) return false; ++nb; }
		return u.size() >= bytes;
	};
	if (!need(12) || memcmp(u.data(), "BAM\1", 4) != 0) return fail(std::string(bam_path) + ": not a BAM file");
	size_t at = 4;
	const uint32_t l_text = le32(u.data() + at); at += 4;
	if (!need(at + l_text + 4)) return fail("truncated BAM header");
	at += l_text;
	const uint32_t n_ref = le32(u.data() + at); at += 4;
	std::vector<std::string> names; std::vector<std::vector<uint8_t>> chroms; int tid = -1;
	for (uint32_t r = 0; r < n_ref; ++r) {
		if (!need(at + 4)) return fail("truncated BAM reference list");
		const uint32_t l_name = le32(u.data() + at); at += 4;
		if (l_name == 0 || !need(at + l_name + 4)) return fail("truncated BAM reference list");
		const std::string name((const char*)u.data() + at, l_name - 1); at += l_name;
		const uint32_t l_ref = le32(u.data() + at); at += 4;
		size_t k = 0;
		while (k < D->names.size() && D->names[k] != name) ++k;
		if (k == D->names.size()) return fail("BAM target " + name + " is not in the FASTA");
		if (D->chroms[k].size() != l_ref) return fail("BAM target " + name + " has a different length than the FASTA record");
		if (name == target) tid = (int)r;
		names.push_back(name); chroms.push_back(D->chroms[k]);
	}
	D->names.swap(names); D->chroms.swap(chroms);
	if (tid < 0) return fail(std::string("target ") + target + " is not in the BAM header");
	const int64_t tlen = (int64_t)D->chroms[(size_t)tid].size();
	if (beg < 0) beg = 0;
	if (end <= 0 || end > tlen) end = tlen;
	if (beg >= end) return D;
	// the index
	if (bai.size() < 8 || memcmp(bai.data(), "BAI\1", 4) != 0) return fail("not a BAI index");
	size_t ia = 4;
	auto rd32 = [&](uint32_t &x) -> bool { if (ia + 4 > bai.size()) return false; x = le32(bai.data() + ia); ia += 4; return true; };
	auto rd64 = [&](uint64_t &x) -> bool { if (ia + 8 > bai.size()) return false; x = (uint64_t)le32(bai.data() + ia) | (uint64_t)le32(bai.data() + ia + 4) << 32; ia += 8; return true; };
	uint32_t bn_ref = 0;
	if (!rd32(bn_ref) || bn_ref != n_ref) return fail("the index does not belong to this BAM (reference count differs)");
	std::vector<std::pair<uint64_t, uint64_t>> chunks; uint64_t min_off = 0;
	{ // candidate bins of [beg, end), SAM spec 5.3 reg2bins
		std::vector<uint32_t> want = {0};
		const int64_t e1 = end - 1;
		for (int64_t k = 1 + (beg >> 26); k <= 1 + (e1 >> 26); ++k) want.push_back((uint32_t)k);
		for (int64_t k = 9 + (beg >> 23); k <= 9 + (e1 >> 23); ++k) want.push_back((uint32_t)k);
		for (int64_t k = 73 + (beg >> 20); k <= 73 + (e1 >> 20); ++k) want.push_back((uint32_t)k);
		for (int64_t k = 585 + (beg >> 17); k <= 585 + (e1 >> 17); ++k) want.push_back((uint32_t)k);
		for (int64_t k = 4681 + (beg >> 14); k <= 4681 + (e1 >> 14); ++k) want.push_back((uint32_t)k);
		std::sort(want.begin(), want.end());
		for (uint32_t r = 0; r < n_ref; ++r) {
			uint32_t n_bin = 0;
			if (!rd32(n_bin)) return fail("truncated index");
			for (uint32_t b = 0; b < n_bin; ++b) {
				uint32_t bin = 0, n_chunk = 0;
				if (!rd32(bin) || !rd32(n_chunk)) return fail("truncated index");
				const bool take = (int)r == tid && std::binary_search(want.begin(), want.end(), bin);
				for (uint32_t c = 0; c < n_chunk; ++c) { uint64_t a = 0, z = 0; if (!rd64(a) || !rd64(z)) return fail("truncated index"); if (take) chunks.push_back({a, z}); }
			}
			uint32_t n_intv = 0;
			if (!rd32(n_intv)) return fail("truncated index");
			for (uint32_t w = 0; w < n_intv; ++w) { uint64_t o = 0; if (!rd64(o)) return fail("truncated index"); if ((int)r == tid && (int64_t)w == (beg >> 14)) min_off = o; }
		}
	}
	std::sort(chunks.begin(), chunks.end());
	// walk the chunks: records are addressed by virtual offsets; a record may straddle blocks
	uint64_t done_to = 0;
	for (const auto &ch : chunks) {
		uint64_t v = std::max(ch.first, std::max(min_off, done_to));
		if (v >= ch.second) continue;
		long bi = block_at(v >> 16);
		if (bi < 0) return fail("the index points between BGZF blocks");
		std::vector<uint8_t> ub; size_t ub_first = (size_t)bi, ub_next = (size_t)bi; // inflated bytes of blocks [ub_first, ub_next)
		auto fill = [&](size_t bytes) -> bool {
			while (ub.size() < bytes && ub_next < blocks.size()) { const size_t o = ub.size(); ub.resize(o + blocks[ub_next].usize); if (!bgzf_inflate_block(file, blocks[ub_next], ub.data() + o)) return false; ++ub_next; }
			return ub.size() >= bytes;
		};
		size_t pos = (size_t)(v & 0xffff);
		for (;;) {
			// virtual offset of `pos`: find the block it falls into
			size_t acc = 0, k = ub_first;
			if (!fill(pos + 4)) break; // end of file
			while (k < ub_next && pos >= acc + blocks[k].usize) { acc += blocks[k].usize; ++k; }
			const uint64_t vcur = (uint64_t)blocks[k < blocks.size() ? k : blocks.size() - 1].off << 16 | (uint64_t)(pos - acc);
			if (vcur >= ch.second) { done_to = vcur; break; }
			const uint32_t block = le32(ub.data() + pos);
			if (block < 32 || !fill(pos + 4 + block)) return fail("truncated BAM record");
			BamFields f;
			if (!bam_fields(ub.data() + pos + 4, block, f)) return fail("malformed BAM record");
			pos += 4 + block;
			done_to = vcur + 1;
			if (f.ref_id != tid) { if (f.ref_id > tid || f.ref_id < 0) break; continue; }
			if (f.pos >= end) break;                       // sorted: nothing further in this chunk can overlap
			const int64_t stop = f.pos + bam_ref_span(f);
			if (stop <= beg) continue;
			IdlhReadRec r;
			r.chrom = f.ref_id; r.start = f.pos; r.mapq = f.mapq; r.flag = f.flag; r.len = (int32_t)f.l_seq;
			r.seq_off = (int64_t)D->bases.size(); r.cig_off = (int64_t)D->cigars.size(); r.n_cig = (int32_t)f.n_cig; r.order = vcur;
			for (unsigned c = 0; c < f.n_cig; ++c) D->cigars.push_back(le32(f.cig + 4 * c));
			r.stop = (int32_t)stop;
			{ const size_t o = D->bases.size(); D->bases.resize(o + f.l_seq); decode_seq16(f.seq, f.l_seq, D->bases.data() + o); }
			D->quals.insert(D->quals.end(), f.qual, f.qual + f.l_seq);
			D->reads.push_back(r);
		}
	}
	// chunks of different bins interleave in the file: file order = virtual offset order; a record reached through two chunks is kept once
	std::stable_sort(D->reads.begin(), D->reads.end(), [](const IdlhReadRec &a, const IdlhReadRec &b) { return a.order < b.order; });
	{
		std::vector<IdlhReadRec> uniq;
		for (const IdlhReadRec &r : D->reads) if (uniq.empty() || uniq.back().order != r.order) uniq.push_back(r);
		D->reads.swap(uniq);
	}
	return D;
}

} // extern "C"

// ---------------------------------------------------------------------------------------------------------------
// Streaming: the BAM is read front to back in slabs, BGZF blocks are inflated by `threads` workers, and the gen_roi
// sweep (src/indelope.nim:515-545) runs INCREMENTALLY over the records, so that neither the file nor a whole
// coverage-gap chunk has to sit in memory (the reference keeps one chunk of records, README "memory": on a deep
// genome without coverage gaps that is a whole chromosome arm).
//
// Why the incremental sweep yields the reference's regions exactly.  The reference scans evidence[last_start, r.start)
// only when a record starts past the end of everything cached (:529-534) and once more at the end of the target (:544);
// the scanned ranges tile [0, length] in order and a region never crosses from one range into the next (:497-499 flush
// at the end of a range).  Records arrive sorted by start and a record only adds evidence at or after its own start
// (:430-442), so evidence[p] is final as soon as a record with start > p has arrived; scanning positions below the
// current record's start therefore sees the same values, and a region that ends there finds every record with
// start <= roi_end already cached, in the same order.  Only the forced flush at a range end has to be replayed: it
// happens exactly where the reference's gap test fires (cache non-empty and r.start > cache.stop, tested BEFORE
// skippable, :529-536).  Records whose stop lies before the next possible region start are dropped from the front of
// the cache early; they could never pass `overlaps` (:449-452) again.
// ---------------------------------------------------------------------------------------------------------------
struct idlh_stream {
	// reference
	idlh_dataset ref;                       // names / chroms in BAM target order (reads stay empty)
	std::vector<uint8_t> skip_chrom;
	// file
	FILE *f = nullptr; int threads = 1; bool file_eof = false;
	std::vector<uint8_t> cbuf; size_t cpos = 0;      // compressed bytes not yet inflated (reader thread only)
	std::vector<uint8_t> ubuf; size_t upos = 0;      // inflated bytes not yet parsed
	std::string error;
	// the reader thread reads and inflates the next slabs while the caller parses and sweeps the current one
	std::thread reader; std::mutex mu; std::condition_variable cv;
	std::deque<std::vector<uint8_t>> ready; bool reader_done = false, stop = false; std::string reader_error;
	// sweep parameters and state
	int32_t min_evidence = 3, min_reads = 3, max_reads = 600;
	int32_t cur_chrom = -1; int64_t tlen = 0;
	std::vector<uint8_t> evidence;
	int64_t scan_pos = 0; bool in_roi = false; int64_t roi_start = 0, roi_end = 0;
	int32_t last_ref = 0, last_pos = -1;
	struct Cached { int32_t start, stop, len; uint8_t mapq; uint16_t flag; int64_t off; uint64_t epoch; int64_t out_idx; };
	std::vector<Cached> cache; size_t head = 0; int64_t cache_stop = 0;
	int64_t cache_len = 0;                            // the reference's cache.len: records cached since the last clear, dropped ones included
	std::vector<uint8_t> cbases;                      // 4-bit sequence + qualities of the cached records, as in the file
	uint64_t epoch = 1;
	bool done = false;
	int64_t n_records = 0, n_regions = 0;
};

namespace {

const size_t SLAB = 4u << 20; // compressed bytes read per refill

// reader thread: read the next slab of the file and inflate its complete blocks (with `threads` workers) into `out`;
// false at the end of the file or on error (err set)
bool stream_read_slab(idlh_stream &S, std::vector<uint8_t> &out, std::string &err)
{
	for (;;) {
		if (S.cpos == S.cbuf.size() && S.file_eof) return false;
		if (!S.file_eof) { // top up the compressed buffer
			if (S.cpos) { S.cbuf.erase(S.cbuf.begin(), S.cbuf.begin() + (long)S.cpos); S.cpos = 0; }
			const size_t old = S.cbuf.size();
			S.cbuf.resize(old + SLAB);
			const size_t got = fread(S.cbuf.data() + old, 1, SLAB, S.f);
			S.cbuf.resize(old + got);
			if (got < SLAB) { if (ferror(S.f)) { err = "read error on the BAM file"; return false; } S.file_eof = true; }
		}
		std::vector<BgzfBlock> blocks; size_t total = 0, at = S.cpos; // index the complete blocks
		while (S.cbuf.size() - at >= 18) {
			const uint8_t *h = S.cbuf.data() + at;
			if (h[0] != 0x1f || h[1] != 0x8b || h[2] != 8 || !(h[3] & 4)) { err = "not a BGZF file (is it BAM? CRAM is not supported by this stand-in)"; return false; }
			const unsigned xlen = le16(h + 10);
			if (S.cbuf.size() - at < 12 + xlen) break;
			int bsize = -1;
			for (unsigned x = 0; x + 4 <= xlen;) {
				const uint8_t *e = h + 12 + x; const unsigned slen = le16(e + 2);
				if (e[0] == 'B' && e[1] == 'C' && slen == 2) bsize = le16(e + 4);
				x += 4 + slen;
			}
			if (bsize < 0) { err = "BGZF block without BC subfield"; return false; }
			const size_t csize = (size_t)bsize + 1;
			if (csize < 12 + xlen + 8) { err = "truncated BGZF block"; return false; }
			if (S.cbuf.size() - at < csize) break;
			const size_t usize = le32(h + csize - 4);
			blocks.push_back({at, csize, total, usize});
			total += usize; at += csize;
		}
		if (blocks.empty()) {
			if (S.file_eof) { if (at != S.cbuf.size()) err = "truncated BGZF block"; S.cpos = S.cbuf.size(); return false; }
			continue;
		}
		out.resize(total);
		std::atomic<size_t> next(0); std::atomic<bool> ok(true);
		auto work = [&]() {
			for (;;) {
				const size_t i = next.fetch_add(16);
				if (i >= blocks.size() || !ok.load()) return;
				for (size_t k = i; k < std::min(i + 16, blocks.size()); ++k)
					if (!bgzf_inflate_block(S.cbuf, blocks[k], out.data() + blocks[k].uoff)) { ok.store(false); return; }
			}
		};
		std::vector<std::thread> pool;
		for (int t = 1; t < S.threads; ++t) pool.emplace_back(work);
		work();
		for (auto &t : pool) t.join();
		if (!ok.load()) { err = "BGZF block failed to inflate (corrupt data or CRC mismatch)"; return false; }
		S.cpos = at;
		if (total == 0) continue; // only empty blocks (the EOF marker)
		return true;
	}
}

void stream_reader_main(idlh_stream *S)
{
	for (;;) {
		std::vector<uint8_t> slab; std::string err;
		const bool ok = stream_read_slab(*S, slab, err);
		std::unique_lock<std::mutex> lk(S->mu);
		if (!ok) { S->reader_error = err; S->reader_done = true; S->cv.notify_all(); return; }
		S->cv.wait(lk, [&] { return S->ready.size() < 4 || S->stop; });
		if (S->stop) { S->reader_done = true; S->cv.notify_all(); return; }
		S->ready.push_back(std::move(slab));
		S->cv.notify_all();
	}
}

// make at least `need` inflated bytes available at ubuf[upos..]; false at end of file or on error (S.error set)
bool stream_fill(idlh_stream &S, size_t need)
{
	while (S.ubuf.size() - S.upos < need) {
		std::vector<uint8_t> slab;
		{
			std::unique_lock<std::mutex> lk(S.mu);
			S.cv.wait(lk, [&] { return !S.ready.empty() || S.reader_done; });
			if (S.ready.empty()) { if (!S.reader_error.empty()) S.error = S.reader_error; return false; }
			slab = std::move(S.ready.front()); S.ready.pop_front();
			S.cv.notify_all();
		}
		if (S.upos == S.ubuf.size()) { S.ubuf.swap(slab); S.upos = 0; }
		else { // a record straddles two slabs: keep the unparsed tail in front of the new bytes
			S.ubuf.erase(S.ubuf.begin(), S.ubuf.begin() + (long)S.upos); S.upos = 0;
			S.ubuf.insert(S.ubuf.end(), slab.begin(), slab.end());
		}
	}
	return true;
}

// a region ends: collect its records from the cache (:476-486) into the group being built
void stream_flush_roi(idlh_stream &S, idlh_rois &R)
{
	std::vector<size_t> reads;
	for (size_t k = S.head; k < S.cache.size(); ++k) {
		const idlh_stream::Cached &r = S.cache[k];
		if (!(r.start > S.roi_end) && !(r.stop < S.roi_start)) { // overlaps :449-452
			reads.push_back(k);
			if ((int64_t)reads.size() > S.max_reads) break;
		}
		if (r.start > S.roi_end) break;
	}
	if ((int64_t)reads.size() < S.min_reads || (int64_t)reads.size() > S.max_reads) return;
	R.roi_chrom.push_back(S.cur_chrom); R.roi_start.push_back((int32_t)S.roi_start); R.roi_stop.push_back((int32_t)S.roi_end);
	R.roi_read_begin.push_back((int64_t)R.read_idx.size()); R.roi_n_reads.push_back((int32_t)reads.size());
	for (size_t k : reads) {
		idlh_stream::Cached &r = S.cache[k];
		if (r.epoch != S.epoch) { // first use in this group: copy the record over
			r.epoch = S.epoch; r.out_idx = (int64_t)R.start.size();
			R.start.push_back(r.start); R.stop.push_back(r.stop); R.len.push_back(r.len); R.mapq.push_back(r.mapq); R.flag.push_back(r.flag);
			R.seq_off.push_back((int64_t)R.own_bases.size());
			// the cache holds the record's 4-bit sequence and its qualities as they are in the file; only records that
			// reach a region (a few percent on a whole genome) are decoded
			const size_t o = R.own_bases.size(), packed = ((size_t)r.len + 1) / 2;
			R.own_bases.resize(o + (size_t)r.len);
			decode_seq16(S.cbases.data() + r.off, (uint32_t)r.len, R.own_bases.data() + o);
			R.own_quals.insert(R.own_quals.end(), S.cbases.begin() + (long)(r.off + packed), S.cbases.begin() + (long)(r.off + packed + r.len));
		}
		R.read_idx.push_back(r.out_idx);
	}
	++S.n_regions;
}

// gen_roi_internal's loop (:461-499) over positions [scan_pos, end); positions below `end` are final
void stream_scan(idlh_stream &S, idlh_rois &R, int64_t end)
{
	if (end > (int64_t)S.evidence.size()) end = (int64_t)S.evidence.size();
	const uint8_t *ev = S.evidence.data();
	const uint8_t me = (uint8_t)S.min_evidence;
	int64_t i = S.scan_pos;
	while (i < end) {
		if (!S.in_roi && me > 0) { // skip runs without any evidence eight positions at a time
			while (i + 8 <= end) { uint64_t w; memcpy(&w, ev + i, 8); if (w) break; i += 8; }
			if (i >= end) break;
		}
		if (ev[i] >= me) {
			if (!S.in_roi) { S.in_roi = true; S.roi_start = i; }
			S.roi_end = i;
		} else if (S.in_roi) { stream_flush_roi(S, R); S.in_roi = false; }
		++i;
	}
	if (end > S.scan_pos) S.scan_pos = end;
}

void stream_drop_passed(idlh_stream &S)
{
	const int64_t thr = S.in_roi ? S.roi_start : S.scan_pos; // no later region can start before this
	while (S.head < S.cache.size() && S.cache[S.head].stop < thr) ++S.head;
	if (S.head == S.cache.size()) { S.cache.clear(); S.head = 0; S.cbases.clear(); }
	else if (S.head > 4096 && S.head * 2 > S.cache.size()) { // compact
		const int64_t off0 = S.cache[S.head].off;
		S.cache.erase(S.cache.begin(), S.cache.begin() + (long)S.head); S.head = 0;
		S.cbases.erase(S.cbases.begin(), S.cbases.begin() + (long)off0);
		for (auto &c : S.cache) c.off -= off0;
	}
}

void stream_end_target(idlh_stream &S, idlh_rois &R)
{
	if (S.cur_chrom < 0) return;
	stream_scan(S, R, (int64_t)S.evidence.size());          // :544
	if (S.in_roi) { stream_flush_roi(S, R); S.in_roi = false; }
	S.cache.clear(); S.head = 0; S.cbases.clear(); S.cache_stop = 0; S.cache_len = 0;
}

void stream_begin_target(idlh_stream &S, int32_t c)
{
	S.cur_chrom = c; S.tlen = (int64_t)S.ref.chroms[(size_t)c].size();
	S.evidence.assign((size_t)S.tlen + 1, 0);                // :522
	S.scan_pos = 0; S.in_roi = false; S.cache_stop = 0;
}

void stream_record(idlh_stream &S, idlh_rois &R, const BamFields &f)
{
	if (f.ref_id != S.cur_chrom) { stream_end_target(S, R); stream_begin_target(S, f.ref_id); }
	const int64_t start = f.pos, stop = f.pos + bam_ref_span(f);
	if (S.cache_len > 0 && start > S.cache_stop) {             // :529-534: coverage gap, the range ends here
		stream_scan(S, R, start);
		if (S.in_roi) { stream_flush_roi(S, R); S.in_roi = false; }
		S.cache.clear(); S.head = 0; S.cbases.clear(); S.cache_stop = 0; S.cache_len = 0;
	} else {
		stream_scan(S, R, start);                               // positions below this record's start are final
		stream_drop_passed(S);
	}
	if (S.skip_chrom[(size_t)f.ref_id] || idlh_skippable_flag(f.flag)) return; // :536
	idlh_stream::Cached c;
	c.start = (int32_t)start; c.stop = (int32_t)stop; c.len = (int32_t)f.l_seq; c.mapq = f.mapq; c.flag = f.flag; c.off = (int64_t)S.cbases.size();
	c.epoch = 0; c.out_idx = -1;
	S.cbases.insert(S.cbases.end(), f.seq, f.qual + f.l_seq); // packed sequence, then qualities (adjacent in the record)
	S.cache.push_back(c); ++S.cache_len; if (stop > S.cache_stop) S.cache_stop = stop; // :504-506,537
	int64_t off = 0; // event_locations :430-442
	for (unsigned k = 0; k < f.n_cig; ++k) {
		const uint32_t cg = le32(f.cig + 4 * k); const unsigned op = cg & 0xf; const int64_t len = cg >> 4;
		const bool cons = op == 0 || op == 2 || op == 3 || op == 7 || op == 8;
		if (op != 0) {
			const int64_t es = start + off, ee = cons ? es + len : es + 1;
			for (int64_t i = es; i < ee && i <= S.tlen; ++i) { uint8_t &e = S.evidence[(size_t)i]; e += 1; if (e == 0) e = 255; } // :539-543
		}
		if (cons) off += len;
	}
}

void rois_finish_view(idlh_rois &R, const idlh_dataset &ref)
{
	for (size_t c = 0; c < ref.chroms.size(); ++c) {
		R.name_ptrs.push_back(ref.names[c].c_str()); R.seq_ptrs.push_back(ref.chroms[c].data()); R.chrom_len.push_back((int64_t)ref.chroms[c].size());
	}
	R.bases = R.own_bases.data(); R.quals = R.own_quals.data();
	idlh_roiset &v = R.view;
	v.n_reads = (int64_t)R.start.size(); v.start = R.start.data(); v.stop = R.stop.data(); v.mapq = R.mapq.data(); v.flag = R.flag.data(); v.len = R.len.data();
	v.seq_off = R.seq_off.data(); v.bases = R.bases; v.quals = R.quals;
	v.n_rois = (int64_t)R.roi_start.size(); v.roi_chrom = R.roi_chrom.data(); v.roi_start = R.roi_start.data(); v.roi_stop = R.roi_stop.data();
	v.roi_read_begin = R.roi_read_begin.data(); v.roi_n_reads = R.roi_n_reads.data(); v.read_idx = R.read_idx.data();
	v.n_chroms = (int32_t)ref.chroms.size(); v.chrom_name = R.name_ptrs.data(); v.chrom_seq = R.seq_ptrs.data(); v.chrom_len = R.chrom_len.data();
}

} // namespace

extern "C" {

void idlh_stream_close(idlh_stream *S);

idlh_stream *idlh_stream_open(const char *fasta_path, const char *bam_path, int threads, int32_t min_event_support, int32_t min_read_coverage,
                              int32_t max_read_coverage, char *err, size_t errlen)
{
	idlh_stream *S = new idlh_stream();
	memset(&S->ref.P, 0, sizeof S->ref.P);
	auto fail = [&](const std::string &m) -> idlh_stream* { set_err(err, errlen, m); idlh_stream_close(S); return nullptr; };
	std::string why;
	if (!load_fasta(fasta_path, S->ref, why)) return fail(why);
	S->f = fopen(bam_path, "rb");
	if (!S->f) return fail(std::string("cannot open ") + bam_path);
	S->threads = threads < 1 ? 1 : threads;
	S->min_evidence = min_event_support; S->min_reads = min_read_coverage; S->max_reads = max_read_coverage;
	S->reader = std::thread(stream_reader_main, S);
	auto need = [&](size_t n) { return stream_fill(*S, n); };
	const std::string pre = std::string(bam_path) + ": ";
	if (!need(12) || memcmp(S->ubuf.data() + S->upos, "BAM\1", 4) != 0) return fail(pre + (S->error.empty() ? "not a BAM file" : S->error));
	const uint32_t l_text = le32(S->ubuf.data() + S->upos + 4);
	if (!need(12 + (size_t)l_text)) return fail(pre + "truncated BAM header");
	S->upos += 8 + l_text;
	const uint32_t n_ref = le32(S->ubuf.data() + S->upos); S->upos += 4;
	std::vector<std::string> names; std::vector<std::vector<uint8_t>> chroms;
	for (uint32_t r = 0; r < n_ref; ++r) { // BAM reference ids -> FASTA records by name; everything follows the BAM's target order (:599-601)
		if (!need(4)) return fail(pre + "truncated BAM reference list");
		const uint32_t l_name = le32(S->ubuf.data() + S->upos);
		if (l_name == 0 || !need(8 + (size_t)l_name)) return fail(pre + "truncated BAM reference list");
		const std::string name((const char*)S->ubuf.data() + S->upos + 4, l_name - 1);
		const uint32_t l_ref = le32(S->ubuf.data() + S->upos + 4 + l_name);
		S->upos += 8 + l_name;
		size_t k = 0;
		while (k < S->ref.names.size() && S->ref.names[k] != name) ++k;
		if (k == S->ref.names.size()) return fail("BAM target " + name + " is not in the FASTA");
		if (S->ref.chroms[k].size() != l_ref) return fail("BAM target " + name + " has a different length than the FASTA record");
		names.push_back(name); chroms.push_back(std::move(S->ref.chroms[k])); S->ref.chroms[k].clear(); S->ref.names[k] = "\1used";
	}
	S->ref.names.swap(names); S->ref.chroms.swap(chroms);
	for (const std::string &nm : S->ref.names) S->skip_chrom.push_back(idlh_skippable_chrom(nm) ? 1 : 0);
	return S;
}

idlh_rois *idlh_stream_next(idlh_stream *S, int64_t target_reads, char *err, size_t errlen)
{
	if (S->done) return nullptr;
	idlh_rois *R = new idlh_rois();
	++S->epoch;
	auto fail = [&](const std::string &m) -> idlh_rois* { set_err(err, errlen, m); delete R; S->done = true; return nullptr; };
	const uint32_t n_ref = (uint32_t)S->ref.names.size();
	for (;;) {
		if ((int64_t)R->read_idx.size() >= target_reads && !R->roi_start.empty()) break;
		if (!stream_fill(*S, 4)) {
			if (!S->error.empty()) return fail(S->error);
			if (S->ubuf.size() != S->upos) return fail("trailing bytes after the last BAM record");
			stream_end_target(*S, *R); // the remaining targets have no records: gen_roi finds nothing there
			S->done = true;
			break;
		}
		const uint32_t block = le32(S->ubuf.data() + S->upos);
		if (block < 32) return fail("truncated BAM record");
		if (!stream_fill(*S, 4 + (size_t)block)) return fail(S->error.empty() ? "truncated BAM record" : S->error);
		const uint8_t *b = S->ubuf.data() + S->upos + 4; S->upos += 4 + (size_t)block;
		BamFields f;
		if (!bam_fields(b, block, f)) return fail("malformed BAM record");
		if (f.ref_id < 0) continue;
		if ((uint32_t)f.ref_id >= n_ref) return fail("BAM record with an unknown reference id");
		if (f.ref_id < S->last_ref || (f.ref_id == S->last_ref && f.pos < S->last_pos)) return fail("BAM is not coordinate sorted");
		S->last_ref = f.ref_id; S->last_pos = f.pos;
		++S->n_records;
		stream_record(*S, *R, f);
	}
	rois_finish_view(*R, S->ref);
	return R;
}

/* contig names / lengths for the VCF header (a view without regions) */
idlh_rois *idlh_stream_targets(const idlh_stream *S)
{
	idlh_rois *R = new idlh_rois();
	rois_finish_view(*R, S->ref);
	return R;
}

void idlh_stream_counts(const idlh_stream *S, int64_t counts[2]) { counts[0] = S->n_records; counts[1] = S->n_regions; }

void idlh_stream_close(idlh_stream *S)
{
	if (!S) return;
	if (S->reader.joinable()) {
		{ std::lock_guard<std::mutex> lk(S->mu); S->stop = true; }
		S->cv.notify_all();
		S->reader.join();
	}
	if (S->f) fclose(S->f);
	delete S;
}

} // extern "C"
