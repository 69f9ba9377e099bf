// indelope_b200/csrc/fastadev.cu -- a bgzip-compressed reference (ref.fa.gz) inflated and parsed on the GPU (idl_fasta_* of include/indelope_cuda.h).
//
// What it replaces: htslib's fai_load of a bgzipped FASTA behind the reference's open_fai (src/indelope.nim:593), and on this project's host the
// BGZF inflate + byte loop of load_fasta (host/bamio.cpp), whose rules are the definition of a FASTA here.
//
// Stages, all on one stream:
//   1. the BGZF inflate stage of idl_bam_open (bamdev.h): member walk, chunked upload on four streams, one warp per member, CRC-32;
//   2. byte-parallel parse of the inflated text, tiles of FA_TILE bytes, 32 consecutive bytes per thread.  Per byte three facts decide everything:
//        - the line it is on: the last line start at or before it (prefix MAX of the key 2p + (text[p] == '>') over line starts p, so the key
//          also says whether that line is a header);
//        - whether a byte other than '\r' / ' ' follows it on its line (suffix MIN of the key 2q + (text[q] == '\n') over bytes q that are
//          not '\r' / ' '; the end of the text counts as a '\n'): a trailing run of '\r' / ' ' is dropped, anything before a solid byte kept;
//        - its record: the number of header starts up to it (prefix SUM);
//      fasta_tile_kernel reduces each tile to the three, fasta_carry_kernel scans the tile values (one CTA), fasta_keep_kernel<false> counts the
//      kept bytes per tile, scan_u32 gives every tile its output offset, and fasta_keep_kernel<true> recomputes the flags and scatters the kept
//      bytes, each record's header position and output offset, and the end of each name (atomicMin of the first ' ', '\t', '\r', '\n' of a
//      header line).  No walk over a line is serial: an unwrapped 250 Mb chromosome is as parallel as a 60-column one;
//   3. the names gathered into one buffer (one warp per record) and copied to the host with the offsets.
#include <algorithm>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include <cuda_runtime.h>
#include "indelope_cuda.h"
#include "bamdev.h"

namespace {

constexpr int FA_THREADS = 256, FA_ITEMS = 32, FA_TILE = FA_THREADS * FA_ITEMS;   // 8 KiB of text per CTA and pass

__device__ __forceinline__ bool fa_soft(unsigned c) { return c == '\r' || c == ' '; }
__device__ __forceinline__ unsigned fa_byte(const uint32_t (&w)[8], int k) { return (w[k >> 2] >> ((k & 3) * 8)) & 0xffu; }

// this thread's 32 bytes (the buffer is padded by 64 zero bytes behind the text, so a thread that starts inside the text may read past its end)
__device__ __forceinline__ void fa_load(const uint8_t *t, size_t base, size_t n, uint32_t (&w)[8])
{
	if (base >= n) {
#pragma unroll
		for (int i = 0; i < 8; ++i) w[i] = 0;
		return;
	}
	const uint4 a = ((const uint4*)(t + base))[0], b = ((const uint4*)(t + base))[1];
	w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
}

// exclusive scan over the threads of the CTA in thread order (REV: in reverse order) with a commutative, associative op; *total = all threads
template <bool REV, class T, class Op> __device__ __forceinline__ T fa_block_scan(T v, T id, Op op, T *sh, T *total)
{
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
	T inc = v;
#pragma unroll
	for (int d = 1; d < 32; d <<= 1) {
		const T o = REV ? __shfl_down_sync(0xffffffffu, inc, d) : __shfl_up_sync(0xffffffffu, inc, d);
		if (REV ? lane + d < 32 : lane >= d) inc = op(inc, o);
	}
	T ex = REV ? __shfl_down_sync(0xffffffffu, inc, 1) : __shfl_up_sync(0xffffffffu, inc, 1);
	if (REV ? lane == 31 : lane == 0) ex = id;
	if (REV ? lane == 0 : lane == 31) sh[warp] = inc;
	__syncthreads();
	T before = id, all = id;
	for (int w = 0; w < nw; ++w) { if (REV ? w > warp : w < warp) before = op(before, sh[w]); all = op(all, sh[w]); }
	__syncthreads();
	*total = all;
	return op(before, ex);
}
struct OpMax { __device__ long long operator()(long long a, long long b) const { return a > b ? a : b; } };
struct OpMin { __device__ long long operator()(long long a, long long b) const { return a < b ? a : b; } };
struct OpAdd { __device__ unsigned operator()(unsigned a, unsigned b) const { return a + b; } };

// the byte in front of this thread's first byte; a virtual '\n' in front of the text
__device__ __forceinline__ unsigned fa_prev(const uint8_t *t, size_t base, size_t n) { return base == 0 ? '\n' : (base <= n ? t[base - 1] : 0u); }

// per thread: last line-start key, first stop key, header starts
__device__ __forceinline__ void fa_thread_facts(const uint32_t (&w)[8], size_t base, size_t n, unsigned prev, long long *ls, long long *stop, unsigned *hdr)
{
	long long l = -1, s = LLONG_MAX; unsigned h = 0;
#pragma unroll
	for (int k = 0; k < FA_ITEMS; ++k) {
		const size_t p = base + (size_t)k;
		const unsigned c = fa_byte(w, k);
		if (p < n) {
			if (prev == '\n') { l = 2 * (long long)p + (c == '>'); h += c == '>'; }
			if (!fa_soft(c) && s == LLONG_MAX) s = 2 * (long long)p + (c == '\n');
		}
		prev = c;
	}
	*ls = l; *stop = s; *hdr = h;
}

__global__ void __launch_bounds__(FA_THREADS) fasta_tile_kernel(const uint8_t *t, size_t n, long long *tile_ls, unsigned *tile_hdr, long long *tile_stop)
{
	__shared__ long long sh[FA_THREADS / 32]; __shared__ unsigned shu[FA_THREADS / 32];
	const size_t base = (size_t)blockIdx.x * FA_TILE + (size_t)threadIdx.x * FA_ITEMS;
	uint32_t w[8];
	fa_load(t, base, n, w);
	long long ls, stop; unsigned hdr;
	fa_thread_facts(w, base, n, fa_prev(t, base, n), &ls, &stop, &hdr);
	long long a, b; unsigned c;
	fa_block_scan<false>(ls, -1ll, OpMax(), sh, &a);
	fa_block_scan<false>(stop, LLONG_MAX, OpMin(), sh, &b);
	fa_block_scan<false>(hdr, 0u, OpAdd(), shu, &c);
	if (threadIdx.x == 0) { tile_ls[blockIdx.x] = a; tile_stop[blockIdx.x] = b; tile_hdr[blockIdx.x] = c; }
}

// one CTA: tile values -> carries.  tile_ls becomes the last line-start key in front of the tile, tile_stop the first stop key behind it (2n + 1 = the
// end of the text), hdr_in[k] the header starts in front of tile k (hdr_in[nt] = all of them)
__global__ void __launch_bounds__(1024) fasta_carry_kernel(size_t nt, size_t n, long long *tile_ls, const unsigned *tile_hdr, unsigned long long *hdr_in,
                                                           long long *tile_stop)
{
	__shared__ long long s_ls[1024], s_stop[1024]; __shared__ unsigned long long s_hdr[1024];
	const size_t per = (nt + 1023) / 1024, lo = (size_t)threadIdx.x * per, hi = lo + per < nt ? lo + per : nt;
	long long ls = -1, stop = LLONG_MAX; unsigned long long hdr = 0;
	for (size_t i = lo; i < hi; ++i) { ls = max(ls, tile_ls[i]); stop = min(stop, tile_stop[i]); hdr += tile_hdr[i]; }
	s_ls[threadIdx.x] = ls; s_stop[threadIdx.x] = stop; s_hdr[threadIdx.x] = hdr;
	__syncthreads();
	if (threadIdx.x == 0) {   // exclusive: prefix max and sum in thread order, suffix min in reverse
		long long m = -1; unsigned long long s = 0;
		for (int k = 0; k < 1024; ++k) { const long long a = s_ls[k]; const unsigned long long b = s_hdr[k]; s_ls[k] = m; s_hdr[k] = s; m = max(m, a); s += b; }
		long long q = 2 * (long long)n + 1;
		for (int k = 1023; k >= 0; --k) { const long long a = s_stop[k]; s_stop[k] = q; q = min(q, a); }
		hdr_in[nt] = s;
	}
	__syncthreads();
	ls = s_ls[threadIdx.x]; hdr = s_hdr[threadIdx.x];
	for (size_t i = lo; i < hi; ++i) { const long long v = tile_ls[i]; tile_ls[i] = ls; ls = max(ls, v); hdr_in[i] = hdr; hdr += tile_hdr[i]; }
	stop = s_stop[threadIdx.x];
	for (size_t i = hi; i > lo; --i) { const long long v = tile_stop[i - 1]; tile_stop[i - 1] = stop; stop = min(stop, v); }
}

// SCATTER = false: kept bytes per tile into keep_tile.  SCATTER = true: the kept bytes to seq + keep_off[tile] ..., per record its header position, its
// output offset and the end of its name
template <bool SCATTER>
__global__ void __launch_bounds__(FA_THREADS, 3) fasta_keep_kernel(const uint8_t *t, size_t n, const long long *tile_ls, const unsigned long long *hdr_in,
                                                                const long long *tile_stop, unsigned *keep_tile, const unsigned long long *keep_off, uint8_t *seq,
                                                                long long *rec_pos, unsigned long long *rec_off, unsigned long long *name_end)
{
	__shared__ long long sh[FA_THREADS / 32]; __shared__ unsigned shu[FA_THREADS / 32];
	const size_t base = (size_t)blockIdx.x * FA_TILE + (size_t)threadIdx.x * FA_ITEMS;
	uint32_t w[8];
	fa_load(t, base, n, w);
	const unsigned prev0 = fa_prev(t, base, n);
	long long ls, stop; unsigned hdr;
	fa_thread_facts(w, base, n, prev0, &ls, &stop, &hdr);
	long long tot;
	const long long ls_in = max(tile_ls[blockIdx.x], fa_block_scan<false>(ls, -1ll, OpMax(), sh, &tot));
	const long long stop_in = min(tile_stop[blockIdx.x], fa_block_scan<true>(stop, LLONG_MAX, OpMin(), sh, &tot));
	unsigned tu;
	unsigned long long rec = hdr_in[blockIdx.x] + fa_block_scan<false>(hdr, 0u, OpAdd(), shu, &tu);   // header starts in front of this thread's bytes
	// backward: is the next byte that is not '\r' / ' ' a solid byte of the same line?
	uint32_t solid_after = 0;
	bool next_nl = stop_in & 1;
#pragma unroll
	for (int k = FA_ITEMS - 1; k >= 0; --k) {
		const unsigned c = fa_byte(w, k);
		if (base + (size_t)k < n && !fa_soft(c)) next_nl = c == '\n';
		if (!next_nl) solid_after |= 1u << k;
	}
	// forward: the line's kind, the keep mask
	uint32_t keep = 0;
	bool hdr_line = ls_in & 1;
	unsigned prev = prev0;
#pragma unroll
	for (int k = 0; k < FA_ITEMS; ++k) {
		const unsigned c = fa_byte(w, k);
		if (base + (size_t)k < n) {
			if (prev == '\n') hdr_line = c == '>';
			if (c != '\n' && !hdr_line && ((solid_after >> k) & 1u)) keep |= 1u << k;
		}
		prev = c;
	}
	unsigned kept_tile;
	const unsigned before = fa_block_scan<false>((unsigned)__popc(keep), 0u, OpAdd(), shu, &kept_tile);
	if (!SCATTER) {
		if (threadIdx.x == 0) keep_tile[blockIdx.x] = kept_tile;
		return;
	}
	const unsigned long long off = keep_off[blockIdx.x] + before;
	hdr_line = ls_in & 1; prev = prev0;
	bool named = false;   // the name end of the header line in effect was sent by this thread
#pragma unroll
	for (int k = 0; k < FA_ITEMS; ++k) {
		const unsigned c = fa_byte(w, k);
		const size_t p = base + (size_t)k;
		if (p < n) {
			if (prev == '\n') {
				hdr_line = c == '>'; named = false;
				if (hdr_line) { rec_pos[rec] = (long long)p; rec_off[rec] = off + (unsigned)__popc(keep & ((1u << k) - 1u)); ++rec; }
			}
			if (hdr_line && !named && (c == ' ' || c == '\t' || c == '\r' || c == '\n')) { atomicMin(name_end + (rec - 1), (unsigned long long)p); named = true; }
			if ((keep >> k) & 1u) seq[off + (unsigned)__popc(keep & ((1u << k) - 1u))] = (uint8_t)c;
		}
		prev = c;
	}
}

// one warp per record: its name, text[rec_pos + 1, name_end), to names + name_off[r]
__global__ void __launch_bounds__(256) fasta_names_kernel(const uint8_t *t, size_t n_rec, const long long *rec_pos, const unsigned long long *name_end,
                                                          const unsigned long long *name_off, uint8_t *names)
{
	const size_t r = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	const int lane = threadIdx.x & 31;
	if (r >= n_rec) return;
	const unsigned long long a = (unsigned long long)rec_pos[r] + 1, len = name_off[r + 1] - name_off[r];
	for (unsigned long long i = (unsigned long long)lane; i < len; i += 32) names[name_off[r] + i] = t[a + i];
}

void set_err(char *err, size_t n, const std::string &m) { if (err && n) snprintf(err, n, "%s", m.c_str()); }

} // namespace

struct idl_fasta {
	int device = 0;
	cudaStream_t st = nullptr;
	uint8_t *d_seq = nullptr;                 // every record's sequence, back to back (+ 64 bytes)
	std::vector<void*> owned;                 // stream-ordered allocations still held
	std::vector<std::string> names; std::vector<const char*> name_ptrs;
	std::vector<int64_t> off, len;            // per record: where its sequence starts in d_seq, its length
	idl_fasta_info info = {};
};

int fasta_record_on_device(const idl_fasta *fa, int64_t record, const uint8_t **seq, int64_t *len, int *device)
{
	if (!fa || record < 0 || record >= fa->info.n_records) return IDL_E_ARG;
	*seq = fa->d_seq + fa->off[(size_t)record]; *len = fa->len[(size_t)record]; *device = fa->device;
	return IDL_OK;
}

extern "C" {

void idl_fasta_close(idl_fasta *fa)
{
	if (!fa) return;
	cudaSetDevice(fa->device);
	if (fa->st) { for (void *p : fa->owned) cudaFreeAsync(p, fa->st); cudaStreamSynchronize(fa->st); cudaStreamDestroy(fa->st); }
	else for (void *p : fa->owned) cudaFree(p);
	delete fa;
}

const idl_fasta_info *idl_fasta_get_info(const idl_fasta *fa) { return fa ? &fa->info : nullptr; }

int idl_fasta_copy(const idl_fasta *fa, int64_t record, uint8_t *dst, size_t dst_len)
{
	if (!fa || record < 0 || record >= fa->info.n_records || (!dst && fa->len[(size_t)record])) return IDL_E_ARG;
	const size_t len = (size_t)fa->len[(size_t)record];
	if (dst_len < len) return IDL_E_ARG;
	if (!len) return IDL_OK;
	if (cudaSetDevice(fa->device) != cudaSuccess) return IDL_E_CUDA;
	if (cudaMemcpyAsync(dst, fa->d_seq + fa->off[(size_t)record], len, cudaMemcpyDeviceToHost, fa->st) != cudaSuccess || cudaStreamSynchronize(fa->st) != cudaSuccess)
		return IDL_E_CUDA;
	return IDL_OK;
}

int idl_fasta_open(int device, const uint8_t *file, size_t file_len, idl_fasta **out, char *err, size_t errlen)
{
	if (!out || (!file && file_len)) return IDL_E_ARG;
	*out = nullptr;
	int ndev = 0;
	if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { set_err(err, errlen, "no CUDA device (idl_fasta_open has no CPU path)"); return IDL_E_NO_DEVICE; }
	if (device < 0 || device >= ndev) return IDL_E_ARG;
	// 1. members
	std::vector<BgzfMember> members; std::vector<size_t> member_at; size_t total = 0;
	{
		std::string why;
		if (file_len < 2 || file[0] != 0x1f || file[1] != 0x8b) { set_err(err, errlen, "not gzip-compressed (idl_fasta_open takes a FASTA compressed with bgzip)"); return IDL_E_FORMAT; }
		if (!bgzf_walk(file, file_len, members, member_at, total, why)) {
			if (why.compare(0, 15, "not a BGZF file") == 0 || why == "BGZF block without BC subfield") why = "gzip member without the BGZF BC subfield (plain gzip): recompress the FASTA with bgzip";
			set_err(err, errlen, why);
			return IDL_E_FORMAT;
		}
	}
	if (members.size() >= (1ull << 32)) return IDL_E_CAPACITY;
	if (cudaSetDevice(device) != cudaSuccess) return IDL_E_CUDA;
	idl_fasta *fa = new idl_fasta();
	fa->device = device;
	int rc = IDL_OK;
	cudaEvent_t ev[4] = {};
	std::string why;
	std::vector<void*> scratch;   // freed before returning
#define FCK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { why = std::string(#call) + ": " + cudaGetErrorString(e_); rc = IDL_E_CUDA; goto done; } } while (0)
#define FALLOC(list, ptr, bytes) do { void *p_ = nullptr; FCK(cudaMallocAsync(&p_, (bytes) ? (bytes) : 16, fa->st)); list.push_back(p_); ptr = (decltype(ptr))p_; } while (0)
	{
		int n_sm = 0;
		FCK(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device));
		FCK(cudaStreamCreateWithFlags(&fa->st, cudaStreamNonBlocking));
		cudaStream_t st = fa->st;
		for (auto &e : ev) FCK(cudaEventCreate(&e));
		uint8_t *d_comp = nullptr, *d_text = nullptr; BgzfMember *d_members = nullptr; unsigned long long *d_err = nullptr; unsigned *d_next = nullptr;
		FALLOC(scratch, d_comp, file_len + 512); FALLOC(scratch, d_text, total + 64); FALLOC(scratch, d_members, members.size() * sizeof(BgzfMember));
		FALLOC(scratch, d_err, 64); FALLOC(scratch, d_next, 4 * 64);
		// 2. H2D + inflate
		FCK(cudaEventRecord(ev[0], st));
		FCK(cudaMemsetAsync(d_comp + file_len, 0, 512, st));
		FCK(cudaMemcpyAsync(d_members, members.data(), members.size() * sizeof(BgzfMember), cudaMemcpyHostToDevice, st));
		FCK(cudaMemsetAsync(d_err, 0xff, 64, st)); FCK(cudaMemsetAsync(d_next, 0, 4 * 64, st)); FCK(cudaMemsetAsync(d_text + total, 0, 64, st));
		FCK(cudaEventRecord(ev[1], st));
		{
			const cudaError_t e_ = bgzf_inflate_chunks(st, n_sm, file, file_len, members, d_comp, d_members, d_text, d_err, d_next, &fa->info.n_chunks);
			if (e_ != cudaSuccess) { why = std::string("inflate: ") + cudaGetErrorString(e_); rc = IDL_E_CUDA; goto done; }
		}
		FCK(cudaEventRecord(ev[2], st));
		unsigned long long herr = 0; uint8_t first = 0;
		FCK(cudaMemcpyAsync(&herr, d_err, 8, cudaMemcpyDeviceToHost, st));
		FCK(cudaMemcpyAsync(&first, d_text, 1, cudaMemcpyDeviceToHost, st));
		FCK(cudaStreamSynchronize(st));
		if (herr != ~0ULL) { why = bgzf_error_text(herr); rc = IDL_E_FORMAT; goto done; }
		if (total > 0 && first != '>') { why = "FASTA record does not start with '>'"; rc = IDL_E_FORMAT; goto done; }
		// 3. the parse
		const size_t n = total, nt = (n + FA_TILE - 1) / FA_TILE;
		size_t n_rec = 0; unsigned long long kept = 0;
		std::vector<long long> rec_pos; std::vector<unsigned long long> rec_off, name_end, name_off(1, 0);
		FALLOC(fa->owned, fa->d_seq, n + 64);   // the sequences are at most the text
		if (nt) {
			long long *d_tile_ls, *d_tile_stop, *d_rec_pos; unsigned *d_tile_hdr, *d_keep_tile; unsigned long long *d_hdr_in, *d_keep_off, *d_scan, *d_rec_off, *d_name_end;
			FALLOC(scratch, d_tile_ls, nt * 8); FALLOC(scratch, d_tile_stop, nt * 8); FALLOC(scratch, d_tile_hdr, nt * 4); FALLOC(scratch, d_keep_tile, nt * 4);
			FALLOC(scratch, d_hdr_in, (nt + 1) * 8); FALLOC(scratch, d_keep_off, (nt + 1) * 8); FALLOC(scratch, d_scan, ((nt + 1) / 2048 + 2) * 8);
			fasta_tile_kernel<<<(unsigned)nt, FA_THREADS, 0, st>>>(d_text, n, d_tile_ls, d_tile_hdr, d_tile_stop);
			fasta_carry_kernel<<<1, 1024, 0, st>>>(nt, n, d_tile_ls, d_tile_hdr, d_hdr_in, d_tile_stop);
			fasta_keep_kernel<false><<<(unsigned)nt, FA_THREADS, 0, st>>>(d_text, n, d_tile_ls, d_hdr_in, d_tile_stop, d_keep_tile, nullptr, nullptr, nullptr, nullptr, nullptr);
			FCK(cudaGetLastError());
			FCK(scan_u32(d_keep_tile, nt, d_keep_off, d_scan, st));
			unsigned long long n_hdr = 0;
			FCK(cudaMemcpyAsync(&n_hdr, d_hdr_in + nt, 8, cudaMemcpyDeviceToHost, st));
			FCK(cudaMemcpyAsync(&kept, d_keep_off + nt, 8, cudaMemcpyDeviceToHost, st));
			FCK(cudaStreamSynchronize(st));
			n_rec = (size_t)n_hdr;
			FCK(cudaMemsetAsync(fa->d_seq + kept, 0, 64, st));
			FALLOC(scratch, d_rec_pos, n_rec * 8); FALLOC(scratch, d_rec_off, n_rec * 8); FALLOC(scratch, d_name_end, n_rec * 8);
			FCK(cudaMemsetAsync(d_name_end, 0x7f, n_rec * 8, st));   // no delimiter: the name runs to the end of the text
			fasta_keep_kernel<true><<<(unsigned)nt, FA_THREADS, 0, st>>>(d_text, n, d_tile_ls, d_hdr_in, d_tile_stop, nullptr, d_keep_off, fa->d_seq, d_rec_pos, d_rec_off,
			                                                             d_name_end);
			FCK(cudaGetLastError());
			rec_pos.resize(n_rec); rec_off.resize(n_rec); name_end.resize(n_rec);
			if (n_rec) {
				FCK(cudaMemcpyAsync(rec_pos.data(), d_rec_pos, n_rec * 8, cudaMemcpyDeviceToHost, st)); FCK(cudaMemcpyAsync(rec_off.data(), d_rec_off, n_rec * 8, cudaMemcpyDeviceToHost, st));
				FCK(cudaMemcpyAsync(name_end.data(), d_name_end, n_rec * 8, cudaMemcpyDeviceToHost, st));
			}
			FCK(cudaStreamSynchronize(st));
			// 4. the names
			for (size_t r = 0; r < n_rec; ++r) name_off.push_back(name_off.back() + (std::min<unsigned long long>(name_end[r], n) - (unsigned long long)rec_pos[r] - 1));
			if (name_off.back()) {
				unsigned long long *d_name_off; uint8_t *d_names;
				FALLOC(scratch, d_name_off, (n_rec + 1) * 8); FALLOC(scratch, d_names, name_off.back());
				FCK(cudaMemcpyAsync(d_name_off, name_off.data(), (n_rec + 1) * 8, cudaMemcpyHostToDevice, st));
				fasta_names_kernel<<<(unsigned)((n_rec * 32 + 255) / 256), 256, 0, st>>>(d_text, n_rec, d_rec_pos, d_name_end, d_name_off, d_names);
				FCK(cudaGetLastError());
				std::string all(name_off.back(), '\0');
				FCK(cudaMemcpyAsync(&all[0], d_names, all.size(), cudaMemcpyDeviceToHost, st));
				FCK(cudaStreamSynchronize(st));
				for (size_t r = 0; r < n_rec; ++r) fa->names.push_back(all.substr(name_off[r], name_off[r + 1] - name_off[r]));
			} else fa->names.assign(n_rec, std::string());
		}
		else FCK(cudaMemsetAsync(fa->d_seq, 0, 64, st));
		FCK(cudaEventRecord(ev[3], st));
		FCK(cudaStreamSynchronize(st));
		for (size_t r = 0; r < n_rec; ++r) { fa->off.push_back((int64_t)rec_off[r]); fa->len.push_back((int64_t)((r + 1 < n_rec ? rec_off[r + 1] : kept) - rec_off[r])); }
		cudaEventElapsedTime(&fa->info.ms_h2d, ev[0], ev[1]); cudaEventElapsedTime(&fa->info.ms_inflate, ev[1], ev[2]); cudaEventElapsedTime(&fa->info.ms_parse, ev[2], ev[3]);
		fa->info.file_bytes = file_len; fa->info.inflated_bytes = total; fa->info.sequence_bytes = kept; fa->info.n_members = (uint32_t)members.size();
		fa->info.n_records = (int64_t)n_rec;
		for (auto &s : fa->names) fa->name_ptrs.push_back(s.c_str());
		fa->info.name = fa->name_ptrs.data(); fa->info.len = fa->len.data();
		fa->info.parse_algorithmic_bytes = (uint64_t)n + kept + 24ull * n_rec;
		fa->info.parse_streamed_bytes = 3ull * n + kept + nt * 64ull + 24ull * n_rec;
	}
done:
	if (fa->st) { for (void *p : scratch) cudaFreeAsync(p, fa->st); cudaStreamSynchronize(fa->st); }
	for (auto &e : ev) if (e) cudaEventDestroy(e);
	if (rc != IDL_OK) { set_err(err, errlen, why); idl_fasta_close(fa); return rc; }
	*out = fa;
	return IDL_OK;
#undef FALLOC
#undef FCK
}

} // extern "C"
