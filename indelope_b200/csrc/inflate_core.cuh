// indelope_b200/csrc/inflate_core.cuh -- SURVEY.md 8(f)3: the DEFLATE (RFC 1951) decoder and the CRC-32 (RFC 1952) of ONE BGZF member
// (SAM spec 4.1: a gzip member of at most 64 KiB), the unit the reference's BAM reader (hts-nim -> htslib bgzf_read_block, behind
// `open(b, path, threads, index=true)`, src/indelope.nim:595) inflates one after the other on host threads.
//
// One WARP decodes one member.  The bit stream of a member is serial, so the 32 lanes run the decoder in LOCKSTEP on identical state
// (bit buffer, tables, output position: every lane computes the same values, the loads are warp-uniform broadcasts); the lanes split
// only where the work is parallel: filling the decode tables, copying a match (lane i copies byte i, i + 32, ...), copying a stored
// block, and the CRC (32 slices combined by multiplication with x^(8 n) mod P).  No lane waits for an elected decoder, no shuffles.
//
// The same source compiles as plain C++ with ONE lane (IDL_INF_LANES == 1): tests/ build it with g++ and check it against zlib
// streams of every block type without a GPU.  Written from RFC 1951 / RFC 1952; not derived from zlib's inflate.
#pragma once
#include <stdint.h>
#include <stddef.h>

#ifdef __CUDACC__
#define IDL_INF_FN __device__ __forceinline__
#define IDL_INF_LANES 32
#define IDL_INF_SYNC() __syncwarp()
#define IDL_INF_CONST __constant__
#else
#define IDL_INF_FN static inline
#define IDL_INF_LANES 1
#define IDL_INF_SYNC() ((void)0)
#define IDL_INF_CONST static const
#endif

namespace idl_inflate {

#ifndef IDL_INF_RING
#define IDL_INF_RING 0
#endif
enum { LIT_BITS = 10, DIST_BITS = 8, CL_BITS = 7, RING = IDL_INF_RING };   // RING: bytes of recent output kept in shared memory (power of two; 0 = none)
enum {
	INF_OK = 0,
	INF_E_BTYPE = 1,      // reserved block type
	INF_E_STORED = 2,     // LEN / NLEN mismatch
	INF_E_CODE = 3,       // over-subscribed or incomplete Huffman code, bad repeat in the code lengths
	INF_E_SYMBOL = 4,     // a bit pattern no code word of the table matches, or length/distance symbol out of range
	INF_E_DISTANCE = 5,   // distance beyond the start of the member (BGZF members carry no preset window)
	INF_E_OUTPUT = 6,     // more (or fewer) bytes than ISIZE says
	INF_E_INPUT = 7,      // ran past the end of the compressed data
	INF_E_CRC = 8         // CRC-32 of the output differs from the member's trailer
};

// A decode-table ENTRY says everything the symbol loop needs, so that a symbol costs one shared-memory load and no second lookup:
//   bits 0-3   length of the code word (0: the bit pattern is not in the fast table -- a longer code or no code)
//   bits 4-7   number of extra bits that follow (lengths, distances)
//   bits 8-9   kind: 0 literal (or a plain symbol of the code-length alphabet), 1 length / distance, 2 end of block, 3 not a valid symbol
//   bits 16-31 value: the literal byte / symbol, or the base of the length / distance
enum { K_LIT = 0, K_BASE = 1, K_END = 2, K_BAD = 3 };
enum { A_CL = 0, A_LIT = 1, A_DIST = 2 };   // alphabets

// per-warp decode tables (shared memory on the device)
struct Tables {
	uint32_t lit_fast[1 << LIT_BITS];
	uint32_t dist_fast[1 << DIST_BITS];                 // the code-length code's table lives here while the block header is read
	uint16_t lit_sym[288], dist_sym[32], cl_sym[20];   // symbols ordered by (code length, symbol): the canonical order of RFC 1951 3.2.2
	uint16_t lit_count[16], dist_count[16], cl_count[16];
	uint8_t lens[320];                                  // code lengths of the literal/length alphabet followed by the distance alphabet
	uint8_t ring[RING != 0 ? RING : 4];                      // the last RING bytes of the output: matches that reach no further back skip the round trip to L2
};

IDL_INF_CONST uint16_t LEN_BASE[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
IDL_INF_CONST uint8_t LEN_EXTRA[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
IDL_INF_CONST uint16_t DIST_BASE[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
IDL_INF_CONST uint8_t DIST_EXTRA[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
IDL_INF_CONST uint8_t CL_ORDER[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

IDL_INF_FN uint32_t make_entry(int alphabet, int sym, int l)
{
	if (alphabet == A_CL) return (uint32_t)sym << 16 | (uint32_t)l;
	if (alphabet == A_LIT) {
		if (sym < 256) return (uint32_t)sym << 16 | (uint32_t)l;
		if (sym == 256) return (uint32_t)K_END << 8 | (uint32_t)l;
		if (sym < 286) return (uint32_t)LEN_BASE[sym - 257] << 16 | (uint32_t)K_BASE << 8 | (uint32_t)LEN_EXTRA[sym - 257] << 4 | (uint32_t)l;
		return (uint32_t)K_BAD << 8 | (uint32_t)l;
	}
	if (sym < 30) return (uint32_t)DIST_BASE[sym] << 16 | (uint32_t)K_BASE << 8 | (uint32_t)DIST_EXTRA[sym] << 4 | (uint32_t)l;
	return (uint32_t)K_BAD << 8 | (uint32_t)l;
}

// ---- bit reader over 32-bit little-endian words ----
// On the device the next 32 words live one per lane (`win`), the 32 after them are already on their way (`win_next`): a refill is a
// shuffle, and the latency of global memory is paid once per 128 bytes, a window ahead of where the decoder reads.
// No load reaches past the last word that holds a byte of the stream (`wend`): the window loads behind it are not made, and the reader
// takes zero words there.  A stream that needs those bits fails the block-end check (bits_overrun), the ISIZE bound or a symbol check; a
// block without an end-of-block that ran off the member used to read on until its output reached ISIZE, up to ~120 KB behind the file.
// IDL_INF_LOOKAHEAD (tests only): the one-lane build keeps the same 2 x 32-word window and makes the device's loads, so that a checked
// build sees exactly the addresses the warp touches.
#ifndef IDL_INF_LOOKAHEAD
#define IDL_INF_LOOKAHEAD 0
#endif
struct Bits {
	const uint32_t *w;      // word 0 = the aligned word that holds the first byte of the stream
	uint32_t wi;            // next word to take
	uint64_t bb; int bc;    // bit buffer: bc valid bits, the next bit of the stream is bit 0
	uint32_t skip, len_byte;   // bytes of word 0 in front of the stream, length of the stream
	uint32_t wend;          // words w[0 .. wend) hold the stream; nothing behind them is loaded
#ifdef __CUDACC__
	uint32_t win, win_next; // win = w[(wi & ~31) + lane], win_next = the 32 words after those
#elif IDL_INF_LOOKAHEAD
	uint32_t win[32], win_next[32];
#endif
};
IDL_INF_FN uint32_t bits_load(const Bits &B, uint32_t i) { return i < B.wend ? B.w[i] : 0u; }
IDL_INF_FN uint32_t bits_next_word(Bits &B)
{
#ifdef __CUDACC__
	const uint32_t v = __shfl_sync(0xffffffffu, B.win, (int)(B.wi & 31u));
	if ((++B.wi & 31u) == 0) { B.win = B.win_next; B.win_next = bits_load(B, B.wi + 32u + (threadIdx.x & 31u)); }
	return v;
#elif IDL_INF_LOOKAHEAD
	const uint32_t v = B.win[B.wi & 31u];
	if ((++B.wi & 31u) == 0) for (uint32_t l = 0; l < 32; ++l) { B.win[l] = B.win_next[l]; B.win_next[l] = bits_load(B, B.wi + 32u + l); }
	return v;
#else
	return bits_load(B, B.wi++);
#endif
}
IDL_INF_FN void bits_open(Bits &B, const uint8_t *base, size_t off, size_t len)
{
	const size_t a = off + ((uintptr_t)base & 3);
	B.w = (const uint32_t*)(base - ((uintptr_t)base & 3)) + (a >> 2);
	B.wi = 0; B.skip = (uint32_t)(a & 3); B.len_byte = (uint32_t)len;
	B.wend = (uint32_t)((B.skip + len + 3) >> 2);
#ifdef __CUDACC__
	B.win = bits_load(B, threadIdx.x & 31u); B.win_next = bits_load(B, 32u + (threadIdx.x & 31u));
#elif IDL_INF_LOOKAHEAD
	for (uint32_t l = 0; l < 32; ++l) { B.win[l] = bits_load(B, l); B.win_next[l] = bits_load(B, 32u + l); }
#endif
	B.bb = (uint64_t)(bits_next_word(B) >> (B.skip * 8)); B.bc = 32 - (int)B.skip * 8;
}
IDL_INF_FN void bits_refill(Bits &B) { if (B.bc <= 32) { B.bb |= (uint64_t)bits_next_word(B) << B.bc; B.bc += 32; } }   // afterwards bc >= 33
IDL_INF_FN uint32_t bits_peek(const Bits &B, int n) { return (uint32_t)B.bb & ((1u << n) - 1u); }
IDL_INF_FN void bits_drop(Bits &B, int n) { B.bb >>= n; B.bc -= n; }
IDL_INF_FN uint32_t bits_take(Bits &B, int n) { const uint32_t v = bits_peek(B, n); bits_drop(B, n); return v; }
IDL_INF_FN uint32_t bits_byte_pos(const Bits &B) { return B.wi * 4u - (uint32_t)(B.bc >> 3) - B.skip; }   // bytes of the stream consumed; whole bytes left in the buffer not counted
IDL_INF_FN bool bits_overrun(const Bits &B) { return (long long)(B.wi * 4u - B.skip) * 8 - B.bc > (long long)B.len_byte * 8; }

// ---- canonical Huffman code (RFC 1951 3.2.2) from code lengths: fast table for codes up to `fast_bits`, counts + ordered symbols for the rest ----
IDL_INF_FN uint32_t rev_bits(uint32_t c, int n)
{
	uint32_t r = 0;
	for (int i = 0; i < n; ++i) { r = r << 1 | (c & 1u); c >>= 1; }
	return r;
}
// every lane runs this with the same arguments; returns INF_OK or INF_E_CODE
IDL_INF_FN int build_code(int lane, int alphabet, const uint8_t *lens, int n, uint32_t *fast, int fast_bits, uint16_t *sym, uint16_t *count)
{
	for (int i = lane; i < (1 << fast_bits); i += IDL_INF_LANES) fast[i] = 0;
	if (lane == 0) {   // read-modify-write of shared counters: one lane, the others wait at the barrier
		for (int l = 0; l < 16; ++l) count[l] = 0;
		for (int s = 0; s < n; ++s) ++count[lens[s]];
	}
	IDL_INF_SYNC();
	uint32_t offs[16], next[16];
	int left = 1;
	offs[0] = 0; next[0] = 0;
	{
		uint32_t code = 0, o = 0;
		for (int l = 1; l < 16; ++l) {
			left <<= 1; left -= count[l];
			if (left < 0) return INF_E_CODE;                 // over-subscribed
			code = (code + (l > 1 ? count[l - 1] : 0)) << 1; // first code word of length l
			next[l] = code; offs[l] = o; o += count[l];
		}
	}
	// incomplete: as in zlib and libdeflate, only a literal/length or distance code that is empty or is one 1-bit code word (a bit pattern
	// outside the code then decodes to no symbol); never the code-length code
	if (left > 0 && (alphabet == A_CL || (left != 1 << 15 && !(left == 1 << 14 && count[1] == 1)))) return INF_E_CODE;
	for (int s = 0; s < n; ++s) {
		const int l = lens[s];
		if (!l) continue;
		sym[offs[l]++] = (uint16_t)s;
		const uint32_t c = next[l]++;
		if (l <= fast_bits) {
			const uint32_t r = rev_bits(c, l);
			const uint32_t e = make_entry(alphabet, s, l);
			for (uint32_t j = r + ((uint32_t)lane << l); j < (1u << fast_bits); j += (uint32_t)IDL_INF_LANES << l) fast[j] = e;
		}
	}
	IDL_INF_SYNC();
	return INF_OK;
}
// a code word longer than the fast table: walk the canonical ranges bit by bit (rare: such symbols have probability < 2^-fast_bits)
IDL_INF_FN uint32_t decode_slow(const Bits &B, int alphabet, const uint16_t *sym, const uint16_t *count)
{
	int code = 0, first = 0, index = 0;
	uint32_t v = (uint32_t)B.bb;
	for (int l = 1; l < 16; ++l) {
		code |= (int)(v & 1u); v >>= 1;
		const int c = count[l];
		if (code - c < first) return make_entry(alphabet, sym[index + (code - first)], l);
		index += c; first += c; first <<= 1; code <<= 1;
	}
	return 0;   // no code word matches
}
// one symbol: the entry of its code word, the code word consumed.  0 = invalid bit pattern.
IDL_INF_FN uint32_t decode_entry(Bits &B, const uint32_t *fast, int fast_bits, int alphabet, const uint16_t *sym, const uint16_t *count)
{
	uint32_t e = fast[bits_peek(B, fast_bits)];
	if (!(e & 15u)) e = decode_slow(B, alphabet, sym, count);
	bits_drop(B, (int)(e & 15u));
	return e;
}

// ---- one member: `in_len` bytes of raw deflate data at byte offset in_off of `base`, `out` receives exactly out_len bytes ----
IDL_INF_FN int inflate_member(int lane, Tables &T, const uint8_t *base, size_t in_off, size_t in_len, uint8_t *out, uint32_t out_len)
{
	Bits B;
	bits_open(B, base, in_off, in_len);
	uint32_t op = 0;
	for (;;) {
		IDL_INF_SYNC();   // every lane is done with the previous block's tables
		bits_refill(B);
		const uint32_t bfinal = bits_take(B, 1), btype = bits_take(B, 2);
		if (btype == 0) {
			// stored: skip to the byte boundary, LEN, NLEN, LEN bytes
			bits_drop(B, B.bc & 7);
			bits_refill(B);
			const uint32_t len = bits_take(B, 16), nlen = bits_take(B, 16);
			if ((len ^ nlen) != 0xffffu) return INF_E_STORED;
			if (len > out_len - op) return INF_E_OUTPUT;
			const uint32_t at = bits_byte_pos(B);                // bytes consumed so far; whole bytes still buffered are re-read below
			if (at + len > B.len_byte) return INF_E_INPUT;
			const uint8_t *src = (const uint8_t*)B.w + B.skip + at;
			for (uint32_t i = (uint32_t)lane; i < len; i += IDL_INF_LANES) { const uint8_t v = src[i]; out[op + i] = v; if (RING != 0) T.ring[(op + i) & (RING - 1)] = v; }
			op += len;
			bits_open(B, (const uint8_t*)B.w, (size_t)B.skip + at + len, (size_t)(B.len_byte - at - len));   // the reader restarts behind the stored bytes
		} else if (btype == 1 || btype == 2) {
			if (btype == 1) {
				for (int i = lane; i < 288; i += IDL_INF_LANES) T.lens[i] = (uint8_t)(i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : 8);
				for (int i = lane; i < 32; i += IDL_INF_LANES) T.lens[288 + i] = 5;   // all 32 five-bit words (a complete code); 30 and 31 decode to K_BAD
				IDL_INF_SYNC();
				if (build_code(lane, A_LIT, T.lens, 288, T.lit_fast, LIT_BITS, T.lit_sym, T.lit_count)) return INF_E_CODE;
				if (build_code(lane, A_DIST, T.lens + 288, 32, T.dist_fast, DIST_BITS, T.dist_sym, T.dist_count)) return INF_E_CODE;
			} else {
				const int hlit = (int)bits_take(B, 5) + 257, hdist = (int)bits_take(B, 5) + 1, hclen = (int)bits_take(B, 4) + 4;
				if (hlit > 286 || hdist > 30) return INF_E_CODE;
				for (int i = lane; i < 19; i += IDL_INF_LANES) T.lens[i] = 0;
				IDL_INF_SYNC();
				for (int i = 0; i < hclen; ++i) {
					bits_refill(B);
					const uint32_t v = bits_take(B, 3);
					if (lane == 0) T.lens[CL_ORDER[i]] = (uint8_t)v;
				}
				IDL_INF_SYNC();
				uint32_t *cl_fast = T.dist_fast;
				if (build_code(lane, A_CL, T.lens, 19, cl_fast, CL_BITS, T.cl_sym, T.cl_count)) return INF_E_CODE;
				// the code lengths of both alphabets as one sequence (repeats may cross from one into the other)
				int n = 0, prev = 0;
				while (n < hlit + hdist) {
					bits_refill(B);
					const uint32_t e = decode_entry(B, cl_fast, CL_BITS, A_CL, T.cl_sym, T.cl_count);
					if (!e) return INF_E_SYMBOL;
					const int s = (int)(e >> 16);
					int rep = 1, val = s;
					if (s == 16) { if (n == 0) return INF_E_CODE; val = prev; rep = 3 + (int)bits_take(B, 2); }
					else if (s == 17) { val = 0; rep = 3 + (int)bits_take(B, 3); }
					else if (s == 18) { val = 0; rep = 11 + (int)bits_take(B, 7); }
					if (n + rep > hlit + hdist) return INF_E_CODE;
					// the code-length code lives in cl_fast / cl_sym / cl_count by now: lens[] is free to take the decoded lengths
					for (int i = lane; i < rep; i += IDL_INF_LANES) T.lens[n + i] = (uint8_t)val;
					n += rep; prev = val;
				}
				IDL_INF_SYNC();
				if (T.lens[256] == 0) return INF_E_CODE;    // no end-of-block code
				if (build_code(lane, A_LIT, T.lens, hlit, T.lit_fast, LIT_BITS, T.lit_sym, T.lit_count)) return INF_E_CODE;
				if (build_code(lane, A_DIST, T.lens + hlit, hdist, T.dist_fast, DIST_BITS, T.dist_sym, T.dist_count)) return INF_E_CODE;
			}
			// symbols
			for (;;) {
				bits_refill(B);
				const uint32_t e = decode_entry(B, T.lit_fast, LIT_BITS, A_LIT, T.lit_sym, T.lit_count);
				// (bit tests, not a switch on the kind: the compiler turned the switch into a jump table and an indirect branch per symbol)
				if (!(e & 0x300u)) {
					if (!e) return INF_E_SYMBOL;
					if (op >= out_len) return INF_E_OUTPUT;
					if (lane == 0) { out[op] = (uint8_t)(e >> 16); if (RING != 0) T.ring[op & (RING - 1)] = (uint8_t)(e >> 16); }
					++op;
					continue;
				}
				if (e & 0x200u) { if (e & 0x100u) return INF_E_SYMBOL; break; }   // K_BAD : K_END
				const uint32_t len = (e >> 16) + bits_take(B, (int)((e >> 4) & 15u));
				bits_refill(B);
				const uint32_t d = decode_entry(B, T.dist_fast, DIST_BITS, A_DIST, T.dist_sym, T.dist_count);
				if (((d >> 8) & 3u) != K_BASE) return INF_E_SYMBOL;
				const uint32_t dist = (d >> 16) + bits_take(B, (int)((d >> 4) & 15u));
				if (dist > op) return INF_E_DISTANCE;
				if (len > out_len - op) return INF_E_OUTPUT;
				IDL_INF_SYNC();   // the bytes written since the last copy, by lane 0 (literals) and by all lanes (matches)
				// source byte of output byte i: i itself, or i modulo dist where the copy overlaps its own output (the last `dist` bytes repeat);
				// either way it lies in [op - dist, op), so no lane reads what another lane writes in this copy
				uint8_t *dst = out + op; const uint8_t *src = dst - dist;
				if (RING != 0 && dist + len <= RING) {   // (with dist + len <= RING no slot of the ring is source and destination of the same copy)
					for (uint32_t i = (uint32_t)lane; i < len; i += IDL_INF_LANES) {
						const uint8_t v = T.ring[(op - dist + (dist >= len ? i : i % dist)) & (RING - 1)];
						dst[i] = v; T.ring[(op + i) & (RING - 1)] = v;
					}
				} else if (RING != 0) {
					for (uint32_t i = (uint32_t)lane; i < len; i += IDL_INF_LANES) { const uint8_t v = src[dist >= len ? i : i % dist]; dst[i] = v; T.ring[(op + i) & (RING - 1)] = v; }
				} else if (dist >= len) {
					if ((uint32_t)lane < len) dst[lane] = src[lane];
					for (uint32_t i = (uint32_t)lane + IDL_INF_LANES; i < len; i += IDL_INF_LANES) dst[i] = src[i];
				} else if (dist == 1) {
					const uint8_t v = src[0];
					for (uint32_t i = (uint32_t)lane; i < len; i += IDL_INF_LANES) dst[i] = v;
				} else {
					for (uint32_t i = (uint32_t)lane; i < len; i += IDL_INF_LANES) dst[i] = src[i % dist];
				}
				op += len;
			}
			if (bits_overrun(B)) return INF_E_INPUT;
		} else return INF_E_BTYPE;
		if (bfinal) break;
	}
	IDL_INF_SYNC();
	if (op != out_len) return INF_E_OUTPUT;
	if (bits_overrun(B)) return INF_E_INPUT;
	return INF_OK;
}

// ---- CRC-32 (RFC 1952 8, polynomial 0xedb88320 reflected): polynomial arithmetic modulo P in the reflected representation, x^0 = 0x80000000 ----
IDL_INF_FN uint32_t gf2_mulmod(uint32_t a, uint32_t b)
{
	uint32_t p = 0;
	for (uint32_t m = 0x80000000u; m; m >>= 1) {
		if (a & m) p ^= b;
		b = (b >> 1) ^ ((b & 1u) ? 0xedb88320u : 0u);
	}
	return p;
}
// x^(8 n) mod P by square and multiply; xp[k] = x^(2^k) mod P for k = 0..31 (crc_init_tables)
IDL_INF_FN uint32_t gf2_xpow8n(const uint32_t *xp, uint32_t n)
{
	uint32_t p = 0x80000000u;
	for (int k = 3; n; n >>= 1, ++k)
		if (n & 1u) p = gf2_mulmod(xp[k & 31], p);   // x^(2^32 - 1) = 1 mod P would wrap; n < 2^17 here so k <= 19
	return p;
}
// tab[256]: byte table of the reflected CRC; xp[32]: x^(2^k) mod P
IDL_INF_FN void crc_init_tables(int lane, int nlanes, uint32_t *tab, uint32_t *xp)
{
	for (int i = lane; i < 256; i += nlanes) {
		uint32_t c = (uint32_t)i;
		for (int k = 0; k < 8; ++k) c = (c >> 1) ^ ((c & 1u) ? 0xedb88320u : 0u);
		tab[i] = c;
	}
	if (lane == 0) {
		uint32_t p = 0x40000000u;   // x^1
		xp[0] = p;
		for (int k = 1; k < 32; ++k) { p = gf2_mulmod(p, p); xp[k] = p; }
	}
}
// this lane's share of crc32(buf[0..n)): slice `lane` of `nlanes` equal slices, already multiplied by x^(8 * bytes behind the slice);
// the XOR over the lanes, complemented, is the CRC-32 of the buffer (the initial 0xffffffff rides in slice 0)
IDL_INF_FN uint32_t crc_lane_part(int lane, int nlanes, const uint32_t *tab, const uint32_t *xp, const uint8_t *buf, uint32_t n)
{
	const uint32_t per = (n + (uint32_t)nlanes - 1) / (uint32_t)nlanes;
	const uint32_t lo = (uint32_t)lane * per < n ? (uint32_t)lane * per : n;
	const uint32_t hi = lo + per < n ? lo + per : n;
	uint32_t c = lane == 0 ? 0xffffffffu : 0u;
	for (uint32_t i = lo; i < hi; ++i) c = tab[(c ^ buf[i]) & 0xffu] ^ (c >> 8);
	if (lane != 0 && lo == hi) return 0;
	return gf2_mulmod(c, gf2_xpow8n(xp, n - hi));
}

} // namespace idl_inflate
