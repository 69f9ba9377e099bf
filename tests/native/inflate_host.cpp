// tests/native/inflate_host.cpp -- TEST BUILD of indelope_b200/csrc/inflate_core.cuh as plain C++ (one lane): the decoder the GPU runs per
// warp, callable from Python without a GPU so that the CPU suite can check it against zlib streams.  Not part of the product libraries.
#include <cstdlib>
#include <cstring>
#include <vector>
#include "inflate_core.cuh"

extern "C" {

// raw deflate stream -> out (exactly out_len bytes); returns the decoder's status
int idl_test_inflate(const uint8_t *in, size_t in_len, uint8_t *out, uint32_t out_len)
{
	std::vector<uint32_t> padded((in_len + 3) / 4 + 4, 0);
	memcpy(padded.data(), in, in_len);
	idl_inflate::Tables *T = new idl_inflate::Tables();
	const int rc = idl_inflate::inflate_member(0, *T, (const uint8_t*)padded.data(), 0, in_len, out, out_len);
	delete T;
	return rc;
}

// same, from a byte offset that is not word aligned (the deflate data of a BGZF member starts 18 bytes into it)
int idl_test_inflate_at(const uint8_t *in, size_t off, size_t in_len, uint8_t *out, uint32_t out_len)
{
	std::vector<uint32_t> padded((off + in_len + 3) / 4 + 4, 0);
	memcpy((uint8_t*)padded.data() + off, in, in_len);
	idl_inflate::Tables *T = new idl_inflate::Tables();
	const int rc = idl_inflate::inflate_member(0, *T, (const uint8_t*)padded.data(), off, in_len, out, out_len);
	delete T;
	return rc;
}

// the member laid out as the device sees the last one of a file: `off` bytes in front of the stream, then the stream, then `pad` bytes
// (idl_bam_open guarantees the member's 8-byte trailer and 512 zero bytes), in heap blocks of exactly that size; the output goes to a
// heap block of exactly out_len bytes.  Built with -fsanitize=address, any load or store outside them is reported.
int idl_test_inflate_tail(const uint8_t *in, size_t off, size_t in_len, size_t pad, uint8_t *out, uint32_t out_len)
{
	uint8_t *buf = (uint8_t*)malloc(off + in_len + pad);
	memset(buf, 0, off + in_len + pad);
	memcpy(buf + off, in, in_len);
	uint8_t *o = (uint8_t*)malloc(out_len ? out_len : 1);
	idl_inflate::Tables *T = new idl_inflate::Tables();
	const int rc = idl_inflate::inflate_member(0, *T, buf, off, in_len, o, out_len);
	memcpy(out, o, out_len);
	delete T;
	free(o);
	free(buf);
	return rc;
}

// CRC-32 as the warp computes it: `nlanes` slices, each multiplied by x^(8 * bytes behind it), XORed
uint32_t idl_test_crc32(const uint8_t *buf, uint32_t n, int nlanes)
{
	uint32_t tab[256], xp[32];
	idl_inflate::crc_init_tables(0, 1, tab, xp);
	uint32_t c = 0;
	for (int l = 0; l < nlanes; ++l) c ^= idl_inflate::crc_lane_part(l, nlanes, tab, xp, buf, n);
	return ~c;
}

}
