// indelope_b200/csrc/pipeline.cu -- libindelope_cuda.so: the C ABI of include/indelope_cuda.h.
//
// One context per GPU.  A context owns `n_streams` lanes; each lane has its stream, device copies of one batch,
// the result pools, the kernel workspaces and pinned host buffers for the results.  idl_submit issues, on the
// lane's stream: cudaMemcpyAsync H2D of the pinned batch -> assemble_kernel -> align4_kernel (DP + glue) ->
// kmer_kernel -> al_kernel -> D2H of the counters; idl_wait then copies back exactly the used prefix of every
// result pool.  All kernels are persistent (grid sized from the SM count) and pull work from device-side queues,
// so the host never needs the intermediate counts.  No CPU fallback exists.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>
#include "common.cuh"
#include "ksw2.cuh"
#include "assemble.cuh"
#include "genotype.cuh"
#include "bamdev.h"

static_assert(sizeof(idl_region) == 48 && sizeof(idl_read) == 24, "batch records are part of the ABI");
static_assert(sizeof(idl_region_result) == 16 && sizeof(idl_contig_result) == 24 && sizeof(idl_aln_result) == 72 && sizeof(idl_event_result) == 128,
              "result records are part of the ABI");

namespace {

struct DevBuf {
	void *p = nullptr; size_t cap = 0;
	cudaError_t ensure(size_t bytes) {
		if (bytes <= cap && p) return cudaSuccess;
		if (p) cudaFree(p);
		p = nullptr; cap = 0;
		size_t want = bytes + bytes / 4 + 256;
		cudaError_t e = cudaMalloc(&p, want);
		if (e == cudaSuccess) cap = want;
		return e;
	}
	void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};
struct HostBuf {
	void *p = nullptr; size_t cap = 0;
	cudaError_t ensure(size_t bytes) {
		if (bytes <= cap && p) return cudaSuccess;
		if (p) cudaFreeHost(p);
		p = nullptr; cap = 0;
		size_t want = bytes + bytes / 4 + 256;
		cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocDefault);
		if (e == cudaSuccess) cap = want;
		return e;
	}
	void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

enum { EV_START = 0, EV_H2D, EV_K0, EV_ASM, EV_ALN, EV_KMER, EV_AL, EV_END, EV_IN, EV_N };

struct Lane {
	cudaStream_t stream = nullptr;
	cudaEvent_t ev[EV_N] = {};
	// device batch
	DevBuf region, read, seq2, seqn, ref2, refn;
	// device results and intermediates
	DevBuf rres, cres, ares, eres, cigar, ctg_ascii, ctg_codes, ctg_sup, refcodes, al_list, al_items, al_res, sort_misc, keysA, orderA, keysB, orderB, keysR, orderR, cnt;
	// workspaces
	DevBuf planes, sup, planes_small, sup_small, pmat, cig_scratch, seq_spill;
	// pinned host results
	HostBuf h_rres, h_cres, h_ares, h_eres, h_cigar, h_seq, h_sup, h_cnt;
	// state
	uint64_t ticket = 0; int state = 0; // 0 free, 1 in flight, 2 done (results valid)
	bool resident = false;              // device batch uploaded by idl_upload
	bool payload = true;                // fetch result arrays in idl_wait
	size_t n_regions = 0, n_reads = 0, n_seq_bases = 0, n_ref_bases = 0;
	// summary of the batch (from idl_batch.summary_*, or one host scan in check_batch when the packer left it out)
	int max_trim = 1; unsigned max_ref = 16; size_t n_small = 0;
	// pools whose size is an estimate grow on overflow: idl_wait relaunches the chain with larger ones (the batch is still resident)
	unsigned cigar_per_aln = 48, items_per_read = 8, cigar_slack = 4096, items_slack = 1024; int retries = 0;
	cudaEvent_t ev_d2h[2] = {};
	unsigned cap_contigs = 0, cap_bases = 0, cap_alns = 0, cap_events = 0, cap_cigar = 0, cap_items = 0;
	unsigned launches = 0;
	idl_results res;
};

} // namespace

struct idl_ctx {
	int device = 0; idl_params P; int n_sm = 148;
	std::vector<Lane> lanes;
	cudaStream_t compute = nullptr; // every lane's kernels run here, in submission order; the lanes' own streams carry the copies
	uint64_t next_ticket = 1;
	int asm_ctas = 0, dp_ctas = 0, ns = 0, nw = 0;
	int cig_cap = 2048;
	size_t ws_budget = 0; // bytes of kernel-2 workspace (backtrack matrices, CIGAR scratch, sequence spill) one lane may hold
	char err[512] = {0};
};

namespace {

int fail(idl_ctx *c, cudaError_t e, const char *what)
{
	if (c) snprintf(c->err, sizeof c->err, "%s: %s", what, cudaGetErrorString(e));
	return IDL_E_CUDA;
}
#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail(ctx, e_, #call); } while (0)

size_t round_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// persistent kernel-2 grids: as many CTAs as fit on the device at this shared-memory size, at most ctx->dp_ctas (launch_chain caps it further
// to the CTAs whose workspaces it allocated)
int dp_grid(const idl_ctx *ctx, const void *kernel, size_t smem, int threads = 256)
{
	int nb = 0;
	if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, threads, smem) != cudaSuccess || nb < 1) nb = 1;
	return std::min(ctx->dp_ctas * 256 / threads, ctx->n_sm * nb);
}

// Shared memory of one kernel-2 CTA at call-site A (align4_kernel) and B (al_kernel).  launch_chain launches with these sizes, and idl_create
// refuses parameters whose worst case (the longest window any batch can have) does not fit DP_SMEM_LIMIT, so that no batch fails for it.
constexpr size_t DP_SMEM_LIMIT = 200 * 1024;
struct DpSmem { int ring_cols, seq_cap; size_t bytes; };
DpSmem smem_site_a(const idl_params &P, int max_ref)
{
	// contigs up to 448 bases stage their reversed copy in shared memory, longer ones in the global spill area
	// (448 bases keep a group at 1.5 KB, four CTAs of 32 alignments per SM -- 16 warps; at 1024 bases three CTAs
	// fit and the kernel ran 12.4 instead of 10.1 ms.  Five CTAs at 256 bases gave nothing more.)
	const int stage = 448;
	DpSmem s;
	s.ring_cols = ksw_ring_cols(ksw_ncol(P.max_contig_len, max_ref, P.a_bw));
	s.seq_cap = (int)round_up(ksw_seq_bytes(std::min(P.max_contig_len, stage), max_ref), 16);
	s.bytes = (size_t)KSW_A4_WARPS * 8 * ksw_group_smem(s.ring_cols, s.seq_cap);
	return s;
}
DpSmem smem_site_b(const idl_params &P, int max_trim, int max_ref)
{
	DpSmem s;
	// unbanded: room for the row-owned variant's target staging whatever the reads' length
	s.ring_cols = std::max(ksw_ring_cols(ksw_ncol(max_trim, std::max(max_ref, P.max_contig_len), P.b_bw)), P.b_bw < 0 ? 256 : 0);
	s.seq_cap = (int)round_up(ksw_seq_bytes(max_trim, max_ref), 16);
	s.bytes = (size_t)(P.b_bw < 0 ? KSW_UNB_WARPS : DP_WARPS) * DP_NG * ksw_group_smem(s.ring_cols, s.seq_cap);
	return s;
}

} // namespace

extern "C" {

void idl_default_params(idl_params *p)
{
	memset(p, 0, sizeof *p);
	p->abi_version = IDL_ABI_VERSION;
	p->min_reads = 3; p->min_ctg_len = 73; p->min_event_len = 4;
	p->asm_min_mapq = 20; p->combine_min_support = 3; p->combine_min_overlap = 65; p->max_contigs = 20;
	p->stop_min_mapq = 5; p->window_pad = 63; p->match = 1; p->mismatch = -2;
	p->a_gapo = 4; p->a_gape = 1; p->a_bw = 50; p->a_zdrop = 400;
	p->b_gapo = 5; p->b_gape = 1; p->b_bw = -1; p->b_zdrop = -1;
	p->max_events = 4; p->count_min_mapq = 10;
	p->max_contig_len = 4096; p->max_read_len = 512; p->max_reads_per_region = 601; p->n_streams = 2;
	p->stages = IDL_STAGE_ALL; p->out_flags = 0;
}

const char *idl_strerror(int s)
{
	switch (s) {
	case IDL_OK: return "ok";
	case IDL_E_NO_DEVICE: return "no CUDA device (libindelope_cuda has no CPU path)";
	case IDL_E_CUDA: return "CUDA error (see idl_last_cuda_error)";
	case IDL_E_ARG: return "bad argument";
	case IDL_E_NOMEM: return "out of memory";
	case IDL_E_CAPACITY: return "batch exceeds allocated capacity";
	case IDL_E_TICKET: return "unknown ticket";
	case IDL_E_BUSY: return "no free lane: wait for and release an earlier ticket";
	case IDL_E_FORMAT: return "not a valid BGZF / BAM file (the call's message buffer has the detail)";
	default: return "unknown status";
	}
}

const char *idl_last_cuda_error(idl_ctx *ctx) { return ctx ? ctx->err : ""; }

int idl_device_count(void)
{
	int n = 0;
	if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
	return n;
}

int idl_device_memory(int device, size_t *free_bytes, size_t *total_bytes)
{
	int n = 0;
	if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) return IDL_E_NO_DEVICE;
	if (device < 0 || device >= n || !free_bytes || !total_bytes) return IDL_E_ARG;
	if (cudaSetDevice(device) != cudaSuccess || cudaMemGetInfo(free_bytes, total_bytes) != cudaSuccess) return IDL_E_CUDA;
	return IDL_OK;
}

int idl_create(int device, const idl_params *p, idl_ctx **out)
{
	if (!out || !p) return IDL_E_ARG;
	*out = nullptr;
	if (p->abi_version != IDL_ABI_VERSION) return IDL_E_ARG;
	if (p->max_contig_len < 64 || p->max_contig_len % 64 || p->max_contig_len > 32768 || p->max_reads_per_region < 1 || p->max_reads_per_region > 4000 ||
	    p->max_read_len < 1 || p->max_read_len > 4096 || p->n_streams < 1 || p->n_streams > 8 || p->max_events < 1 || p->max_events > IDL_MAX_EVENTS)
		return IDL_E_ARG;
	// the query of call-site B (a trimmed read) is staged in shared memory: with the unbanded default that holds reads of up to 960 bases
	// (DESIGN.md 7).  Longer max_read_len is refused here, so that a longer read drops its region (IDL_RS_READ_TOO_LONG) instead of its batch.
	if (smem_site_a(*p, 1 << 20).bytes > DP_SMEM_LIMIT || smem_site_b(*p, p->max_read_len, 1 << 20).bytes > DP_SMEM_LIMIT) return IDL_E_ARG;
	int n = 0;
	if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) return IDL_E_NO_DEVICE;
	if (device < 0 || device >= n) return IDL_E_ARG;
	idl_ctx *ctx = new (std::nothrow) idl_ctx();
	if (!ctx) return IDL_E_NOMEM;
	ctx->device = device; ctx->P = *p;
	cudaError_t e = cudaSetDevice(device);
	if (e != cudaSuccess) { delete ctx; return IDL_E_CUDA; }
	cudaDeviceProp prop;
	size_t total_mem = 0;
	if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { delete ctx; return IDL_E_CUDA; }
	ctx->n_sm = prop.multiProcessorCount; total_mem = prop.totalGlobalMem;
	{
		// kernel-2 workspace per lane: a quarter of the device shared by the lanes, at most 16 GiB (DESIGN.md 7); IDL_WS_BUDGET_MB overrides it
		const char *eb = getenv("IDL_WS_BUDGET_MB");
		ctx->ws_budget = std::min<size_t>(16ull << 30, total_mem / (4 * (size_t)p->n_streams));
		if (eb && atoll(eb) > 0) ctx->ws_budget = (size_t)atoll(eb) << 20;
	}
	ctx->ns = p->max_reads_per_region + 2;
	ctx->nw = p->max_contig_len / 32 + 2;
	// persistent grids: CTAs per SM (tunable for experiments through the environment)
	const char *ea = getenv("IDL_ASM_CTAS_PER_SM"), *ed = getenv("IDL_DP_CTAS_PER_SM");
	ctx->asm_ctas = ctx->n_sm * (ea && atoi(ea) > 0 ? atoi(ea) : ASM_CTAS); // CTAs of each assembler launch (8 regions per CTA in the warp variant)
	ctx->dp_ctas = ctx->n_sm * (ed && atoi(ed) > 0 ? atoi(ed) : 4); // upper bound; every launch asks the occupancy calculator
	ctx->lanes.resize((size_t)p->n_streams);
	{
		// IDL_OVERLAP_KERNELS=1: the kernels of a batch run on its lane's stream and may share the SMs with another batch's
		const char *eo = getenv("IDL_OVERLAP_KERNELS");
		if (!(eo && *eo == '1') && cudaStreamCreateWithFlags(&ctx->compute, cudaStreamNonBlocking) != cudaSuccess) { idl_destroy(ctx); return IDL_E_CUDA; }
	}
	// initial estimates of the two growable pools (tests shrink them to exercise the relaunch)
	const char *ec = getenv("IDL_CIGAR_PER_ALN"), *ei = getenv("IDL_ITEMS_PER_READ");
	for (Lane &L : ctx->lanes) {
		if (ec && atoi(ec) >= 0) { L.cigar_per_aln = (unsigned)atoi(ec); L.cigar_slack = 16; }
		if (ei && atoi(ei) >= 0) { L.items_per_read = (unsigned)atoi(ei); L.items_slack = 16; }
		if (cudaStreamCreateWithFlags(&L.stream, cudaStreamNonBlocking) != cudaSuccess) { idl_destroy(ctx); return IDL_E_CUDA; }
		for (auto &ev : L.ev) if (cudaEventCreate(&ev) != cudaSuccess) { idl_destroy(ctx); return IDL_E_CUDA; }
		for (auto &ev : L.ev_d2h) if (cudaEventCreate(&ev) != cudaSuccess) { idl_destroy(ctx); return IDL_E_CUDA; }
	}
	// opt in to large dynamic shared memory for the DP kernels
	cudaFuncSetAttribute(align4_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
	cudaFuncSetAttribute(al_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
	cudaFuncSetAttribute(al_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
	cudaFuncSetAttribute(assemble_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
	cudaFuncSetAttribute(assemble_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
	*out = ctx;
	return IDL_OK;
}

void idl_destroy(idl_ctx *ctx)
{
	if (!ctx) return;
	cudaSetDevice(ctx->device);
	if (ctx->compute) { cudaStreamSynchronize(ctx->compute); }
	for (Lane &L : ctx->lanes) {
		if (L.stream) cudaStreamSynchronize(L.stream);
		for (DevBuf *b : {&L.region, &L.read, &L.seq2, &L.seqn, &L.ref2, &L.refn, &L.rres, &L.cres, &L.ares, &L.eres, &L.cigar, &L.ctg_ascii, &L.ctg_codes,
		                  &L.ctg_sup, &L.refcodes, &L.al_list, &L.al_items, &L.al_res, &L.sort_misc, &L.keysA, &L.orderA, &L.keysB, &L.orderB, &L.keysR, &L.orderR, &L.cnt, &L.planes, &L.sup,
		                  &L.planes_small, &L.sup_small, &L.pmat, &L.cig_scratch, &L.seq_spill})
			b->release();
		for (HostBuf *b : {&L.h_rres, &L.h_cres, &L.h_ares, &L.h_eres, &L.h_cigar, &L.h_seq, &L.h_sup, &L.h_cnt}) b->release();
		for (auto &ev : L.ev) if (ev) cudaEventDestroy(ev);
		for (auto &ev : L.ev_d2h) if (ev) cudaEventDestroy(ev);
		if (L.stream) cudaStreamDestroy(L.stream);
	}
	if (ctx->compute) cudaStreamDestroy(ctx->compute);
	delete ctx;
}

int idl_batch_alloc(idl_ctx *ctx, size_t max_regions, size_t max_reads, size_t max_seq_bases, size_t max_ref_bases, idl_batch **out)
{
	if (!ctx || !out) return IDL_E_ARG;
	*out = nullptr;
	cudaSetDevice(ctx->device);
	idl_batch *b = (idl_batch*)calloc(1, sizeof(idl_batch));
	if (!b) return IDL_E_NOMEM;
	max_seq_bases = round_up(max_seq_bases, 64); max_ref_bases = round_up(max_ref_bases, 64);
	b->cap_regions = max_regions; b->cap_reads = max_reads; b->cap_seq_bases = max_seq_bases; b->cap_ref_bases = max_ref_bases;
	// the library owns pinned memory (SURVEY.md 8b): the host language never hands GC memory to CUDA
	cudaError_t e = cudaSuccess;
	auto pin = [&](void **p, size_t bytes) { if (e == cudaSuccess) e = cudaHostAlloc(p, bytes, cudaHostAllocDefault); if (e == cudaSuccess) memset(*p, 0, bytes); };
	pin((void**)&b->region, (max_regions + 1) * sizeof(idl_region));
	pin((void**)&b->read, (max_reads + 1) * sizeof(idl_read));
	pin((void**)&b->seq2, max_seq_bases / 4 + 16); pin((void**)&b->seqn, max_seq_bases / 8 + 16);
	pin((void**)&b->ref2, max_ref_bases / 4 + 16); pin((void**)&b->refn, max_ref_bases / 8 + 16);
	if (e != cudaSuccess) { idl_batch_free(ctx, b); return fail(ctx, e, "cudaHostAlloc(batch)"); }
	*out = b;
	return IDL_OK;
}

void idl_batch_free(idl_ctx *ctx, idl_batch *b)
{
	(void)ctx;
	if (!b) return;
	for (void *p : {(void*)b->region, (void*)b->read, (void*)b->seq2, (void*)b->seqn, (void*)b->ref2, (void*)b->refn}) if (p) cudaFreeHost(p);
	free(b);
}

} // extern "C"

namespace {

struct BatchSummary { int max_trim = 1; unsigned max_ref = 16; size_t n_small = 0; };

// Host-side validation: O(regions).  The read records are validated on the device, by the kernel that first touches them
// (assemble_kernel: bounds, alignment, trim range; a malformed record drops its region with IDL_RS_BAD_INPUT), so a submit does
// no per-read host work when the packer filled the batch summary.
int check_batch(const idl_ctx *ctx, const idl_batch *b, BatchSummary &S)
{
	if (!b || b->n_regions > b->cap_regions || b->n_reads > b->cap_reads || b->n_seq_bases > b->cap_seq_bases || b->n_ref_bases > b->cap_ref_bases) return IDL_E_CAPACITY;
	if (b->n_seq_bases % 64 || b->n_ref_bases % 64) return IDL_E_ARG;
	if (b->n_seq_bases >= (1ull << 32) || b->n_ref_bases >= (1ull << 32) || b->n_reads >= (1ull << 31)) return IDL_E_CAPACITY;
	unsigned max_ref = 16; size_t n_small = 0;
	for (size_t i = 0; i < b->n_regions; ++i) {
		const idl_region &r = b->region[i];
		if ((size_t)r.read_begin + r.n_reads > b->n_reads || (size_t)r.ref_off + r.ref_len > b->n_ref_bases || (r.ref_off & 63u)) return IDL_E_ARG;
		if ((int)r.n_reads + 2 > ctx->ns) return IDL_E_CAPACITY;
		max_ref = std::max(max_ref, r.ref_len); n_small += r.n_reads <= ASM_SMALL_READS;
	}
	S.max_ref = max_ref; S.n_small = n_small;
	if (b->summary_valid) S.max_trim = (int)std::max<uint32_t>(1u, std::min<uint32_t>(b->max_trim_len, (uint32_t)ctx->P.max_read_len));
	else {
		int mt = 1;
		for (size_t i = 0; i < b->n_reads; ++i) mt = std::max<int>(mt, b->read[i].trim_len);
		S.max_trim = std::min(mt, ctx->P.max_read_len);
	}
	return IDL_OK;
}

// device copies of the batch + sizing of every pool (shared by submit and upload)
int stage_batch(idl_ctx *ctx, Lane &L, const idl_batch *b, bool copy)
{
	L.n_regions = b->n_regions; L.n_reads = b->n_reads; L.n_seq_bases = b->n_seq_bases; L.n_ref_bases = b->n_ref_bases;
	const size_t s2 = b->n_seq_bases / 4 + 16, sn = b->n_seq_bases / 8 + 16, r2 = b->n_ref_bases / 4 + 16, rn = b->n_ref_bases / 8 + 16;
	CK(L.region.ensure((b->n_regions + 1) * sizeof(idl_region))); CK(L.read.ensure((b->n_reads + 1) * sizeof(idl_read)));
	CK(L.seq2.ensure(s2)); CK(L.seqn.ensure(sn)); CK(L.ref2.ensure(r2)); CK(L.refn.ensure(rn));
	if (copy) {
		CK(cudaMemcpyAsync(L.region.p, b->region, b->n_regions * sizeof(idl_region), cudaMemcpyHostToDevice, L.stream));
		CK(cudaMemcpyAsync(L.read.p, b->read, b->n_reads * sizeof(idl_read), cudaMemcpyHostToDevice, L.stream));
		CK(cudaMemcpyAsync(L.seq2.p, b->seq2, s2, cudaMemcpyHostToDevice, L.stream));
		CK(cudaMemcpyAsync(L.seqn.p, b->seqn, sn, cudaMemcpyHostToDevice, L.stream));
		CK(cudaMemcpyAsync(L.ref2.p, b->ref2, r2, cudaMemcpyHostToDevice, L.stream));
		CK(cudaMemcpyAsync(L.refn.p, b->refn, rn, cudaMemcpyHostToDevice, L.stream));
	}
	return IDL_OK;
}

// record_start: the device-resident timing leg has no copies to wait for, so its clock starts here, after the host-side sizing
struct LaneSizes { size_t n_regions, n_reads, n_seq_bases, n_ref_bases; };

int launch_chain(idl_ctx *ctx, Lane &L, bool record_start = false)
{
	const idl_params &P = ctx->P;
	const LaneSizes bb = {L.n_regions, L.n_reads, L.n_seq_bases, L.n_ref_bases}; const LaneSizes *b = &bb;
	// pool capacities: every contig holds >= 1 read; an aligned contig holds >= max(1, min_reads) reads and a region aligns <= max_contigs
	const int max_trim = L.max_trim; const unsigned max_ref = L.max_ref;
	L.cap_contigs = (unsigned)b->n_reads + 1;
	L.cap_bases = (unsigned)std::min<size_t>(b->n_seq_bases + 4 * b->n_reads + 64, 0xfffffff0u);
	L.cap_alns = (unsigned)std::min<size_t>(b->n_reads / (size_t)std::max(1, P.min_reads) + 1, (size_t)P.max_contigs * b->n_regions + 1);
	L.cap_events = L.cap_alns * (unsigned)P.max_events;
	L.cap_cigar = (unsigned)std::min<size_t>((size_t)L.cap_alns * L.cigar_per_aln + L.cigar_slack, 0xfffffff0u); // an estimate: grown by idl_wait on overflow
	CK(L.rres.ensure((b->n_regions + 1) * sizeof(idl_region_result)));
	CK(L.cres.ensure((size_t)L.cap_contigs * sizeof(idl_contig_result)));
	CK(L.ares.ensure((size_t)L.cap_alns * sizeof(idl_aln_result)));
	CK(L.eres.ensure((size_t)L.cap_events * sizeof(idl_event_result)));
	CK(L.cigar.ensure((size_t)L.cap_cigar * 4));
	CK(L.ctg_ascii.ensure(L.cap_bases)); CK(L.ctg_codes.ensure(L.cap_bases));
	if (P.out_flags & IDL_OUT_SUPPORT) CK(L.ctg_sup.ensure((size_t)L.cap_bases * 4));
	CK(L.refcodes.ensure(b->n_ref_bases + 64));
	CK(L.al_list.ensure((size_t)L.cap_events * sizeof(AlEntry) + 16));
	CK(L.cnt.ensure(sizeof(DevCounters)));
	L.cap_items = (unsigned)std::min<size_t>((size_t)L.items_per_read * b->n_reads + L.items_slack, 0x3fffffffu); // AL items: a read takes part in few AL events (an estimate: grown by idl_wait on overflow)
	CK(L.al_items.ensure((size_t)L.cap_items * sizeof(AlItem))); CK(L.al_res.ensure((size_t)L.cap_items * 2 + 16));
	CK(L.sort_misc.ensure(9 * SORT_BUCKETS * sizeof(unsigned)));
	CK(L.keysR.ensure((size_t)b->n_regions * 2 + 16)); CK(L.orderR.ensure((size_t)b->n_regions * 4 + 16));
	CK(L.keysA.ensure((size_t)L.cap_alns * 2 + 16)); CK(L.orderA.ensure((size_t)L.cap_alns * 4 + 16));
	CK(L.keysB.ensure((size_t)L.cap_items * 4 + 16)); CK(L.orderB.ensure((size_t)L.cap_items * 8 + 16));
	// workspaces
	const size_t n_small = L.n_small;
	const size_t n_big = b->n_regions - n_small;
	// the assembler addresses its arenas with 32-bit element offsets: at large max_reads_per_region / max_contig_len fewer CTAs are
	// launched (they pull regions from an atomic queue, so any grid computes the same); only an arena of one CTA that does not fit fails
	const size_t per_big = (size_t)ctx->ns * std::max<size_t>(3 * (size_t)ctx->nw, (size_t)P.max_contig_len);
	const size_t per_small = (size_t)8 * ASM_SMALL_NS * std::max<size_t>(3 * (size_t)ctx->nw, (size_t)P.max_contig_len);
	if (per_big >= 0xffffffffULL || per_small >= 0xffffffffULL) return IDL_E_CAPACITY;
	const int big_ctas = (int)std::min<size_t>({n_big, (size_t)ctx->asm_ctas, (size_t)0xfffffffeULL / per_big});
	const int small_ctas = (int)std::min<size_t>({(n_small + 7) / 8, (size_t)ctx->asm_ctas, (size_t)0xfffffffeULL / per_small});
	if (n_big) {
		CK(L.planes.ensure((size_t)big_ctas * ctx->ns * 3 * ctx->nw * 4));
		CK(L.sup.ensure((size_t)big_ctas * ctx->ns * P.max_contig_len * 2));
	}
	if (n_small) {
		CK(L.planes_small.ensure((size_t)small_ctas * 8 * ASM_SMALL_NS * 3 * ctx->nw * 4));
		CK(L.sup_small.ensure((size_t)small_ctas * 8 * ASM_SMALL_NS * P.max_contig_len * 2));
	}
	// kernel 2 geometry: call-site A (contig vs window, banded) and B (read vs suffix, unbanded by default)
	const int ncolA = ksw_ncol(P.max_contig_len, (int)max_ref, P.a_bw), ncolB = ksw_ncol(max_trim, std::max((int)max_ref, P.max_contig_len), P.b_bw);
	const size_t rowsA = (size_t)ksw_rows_bound(P.max_contig_len, (int)max_ref, P.a_bw); // the anti-diagonals an alignment can execute before its band runs out
	const size_t rowsB = (size_t)max_trim + std::max<size_t>(max_ref, 1536);
	const size_t pitchB = std::max<size_t>(ksw_pitch(ncolB), P.b_bw < 0 ? 32 * (size_t)ksw_rows_w(max_trim) : 0); // the row-owned variant stores 32 W bytes per diagonal
	const size_t p_capA = round_up(rowsA * ksw_pitch(ncolA) + 2 * KSW_PMAT_PAD + 64, 256), p_capB = round_up(rowsB * pitchB + 2 * KSW_PMAT_PAD + 64, 256);
	const int seq_spill_cap = (int)round_up(ksw_seq_bytes(std::max(P.max_contig_len, max_trim), std::max((int)max_ref, P.max_contig_len)) + 32, 16);
	// Every group of a kernel-2 grid owns a backtrack matrix, CIGAR scratch and a spill area, addressed by its index in the launched grid.
	// Both grids are persistent and take their tasks from atomic counters, so fewer groups compute the same records: each grid is capped
	// at the CTAs its tasks can keep busy and at the CTAs whose workspaces fit the lane's budget, and the workspaces are sized for that cap.
	const size_t gpc_a = (size_t)KSW_A4_WARPS * 8 /* align4_kernel: eight alignments per warp */, warps_b = P.b_bw < 0 ? KSW_UNB_WARPS : DP_WARPS, gpc_b = warps_b * DP_NG;
	const size_t ws_fixed = (size_t)ctx->cig_cap * 4 + (size_t)seq_spill_cap;
	const size_t ctas_a = std::min<size_t>({(size_t)ctx->n_sm * KSW_A4_CTAS, ((size_t)L.cap_alns + gpc_a - 1) / gpc_a, ctx->ws_budget / (gpc_a * (p_capA + ws_fixed))});
	const size_t ctas_b = std::min<size_t>({(size_t)ctx->dp_ctas * DP_WARPS / warps_b, (2 * (size_t)L.cap_items + gpc_b - 1) / gpc_b, ctx->ws_budget / (gpc_b * (p_capB + ws_fixed))});
	if (ctas_a < 1 || ctas_b < 1) return IDL_E_CAPACITY; // the workspaces of one CTA exceed the budget: reads or windows too long for this device
	const size_t groups_a = ctas_a * gpc_a, groups_b = ctas_b * gpc_b, n_groups = std::max(groups_a, groups_b);
	CK(L.pmat.ensure(std::max(groups_a * p_capA, groups_b * p_capB)));
	CK(L.cig_scratch.ensure(n_groups * (size_t)ctx->cig_cap * 4));
	CK(L.seq_spill.ensure(n_groups * (size_t)seq_spill_cap));
	// copies travel on the lane's stream, kernels on the context's compute stream: batches overlap their transfers with each
	// other's kernels, and the persistent kernels of two batches never compete for the SMs
	cudaStream_t cs = ctx->compute ? ctx->compute : L.stream;
	if (cs != L.stream) { CK(cudaEventRecord(L.ev[EV_IN], L.stream)); CK(cudaStreamWaitEvent(cs, L.ev[EV_IN], 0)); }
	if (record_start) { CK(cudaEventRecord(L.ev[EV_START], cs)); CK(cudaEventRecord(L.ev[EV_H2D], cs)); }
	CK(cudaEventRecord(L.ev[EV_K0], cs)); // the stage times start here, on the compute stream: behind the copies AND behind the kernels of the batch ahead
	CK(cudaMemsetAsync(L.cnt.p, 0, sizeof(DevCounters), cs));
	CK(cudaMemsetAsync(L.sort_misc.p, 0, 9 * SORT_BUCKETS * sizeof(unsigned), cs));
	L.launches = 0;
	SortBufs sA, sB;
	sA.hist = (unsigned*)L.sort_misc.p; sA.start = sA.hist + SORT_BUCKETS; sA.cursor = sA.start + SORT_BUCKETS; sA.keys = (uint16_t*)L.keysA.p; sA.order = (unsigned*)L.orderA.p;
	sB.hist = sA.cursor + SORT_BUCKETS; sB.start = sB.hist + SORT_BUCKETS; sB.cursor = sB.start + SORT_BUCKETS; sB.keys = (uint16_t*)L.keysB.p; sB.order = (unsigned*)L.orderB.p;
	SortBufs sR;
	sR.hist = sB.cursor + SORT_BUCKETS; sR.start = sR.hist + SORT_BUCKETS; sR.cursor = sR.start + SORT_BUCKETS; sR.keys = (uint16_t*)L.keysR.p; sR.order = (unsigned*)L.orderR.p;

	AsmArgs a; memset(&a, 0, sizeof a);
	a.region = (const idl_region*)L.region.p; a.read = (const idl_read*)L.read.p;
	a.seq2 = (const uint32_t*)L.seq2.p; a.seqn = (const uint32_t*)L.seqn.p; a.ref2 = (const uint32_t*)L.ref2.p; a.refn = (const uint32_t*)L.refn.p;
	a.n_regions = (unsigned)b->n_regions; a.n_reads = (unsigned)b->n_reads; a.n_seq_bases = (unsigned)b->n_seq_bases; a.P = P;
	a.planes = (uint32_t*)L.planes.p; a.sup = (uint16_t*)L.sup.p; a.ns = ctx->ns; a.nw = ctx->nw; a.cap = P.max_contig_len;
	a.rres = (idl_region_result*)L.rres.p; a.cres = (idl_contig_result*)L.cres.p; a.ares = (idl_aln_result*)L.ares.p;
	a.ctg_ascii = (char*)L.ctg_ascii.p; a.ctg_codes = (uint8_t*)L.ctg_codes.p; a.ctg_sup = (P.out_flags & IDL_OUT_SUPPORT) ? (uint32_t*)L.ctg_sup.p : nullptr;
	a.refcodes = (uint8_t*)L.refcodes.p;
	a.cap_contigs = L.cap_contigs; a.cap_bases = L.cap_bases; a.cap_alns = L.cap_alns;
	a.sortA = sA;
	a.cnt = (DevCounters*)L.cnt.p;
	a.order = sR.order;
	if (b->n_regions > 0 && (P.stages & IDL_STAGE_ASSEMBLE)) { // the assembler's queue: regions by read count, deepest first
		region_key_kernel<<<ctx->n_sm * 2, 256, 0, cs>>>(sR, a.region, a.n_regions, a.cnt);
		sort_scan_kernel<<<1, 1024, 0, cs>>>(sR);
		sort_scatter_kernel<<<ctx->n_sm * 4, 256, 0, cs>>>(sR, &a.cnt->n_regions_in, 1u, a.n_regions);
		CK(cudaGetLastError()); L.launches += 3;
	}
	if (n_small && (P.stages & IDL_STAGE_ASSEMBLE)) { // one warp per region
		a.small = 1; a.ns = ASM_SMALL_NS; a.planes = (uint32_t*)L.planes_small.p; a.sup = (uint16_t*)L.sup_small.p;
		assemble_kernel<32><<<small_ctas, ASM_THREADS, 8 * asm_smem_bytes(ASM_SMALL_NS, ctx->nw, 32), cs>>>(a);
		CK(cudaGetLastError()); L.launches++;
	}
	if (n_big && (P.stages & IDL_STAGE_ASSEMBLE)) { // one CTA per region
		a.small = 0; a.ns = ctx->ns; a.planes = (uint32_t*)L.planes.p; a.sup = (uint16_t*)L.sup.p;
		assemble_kernel<256><<<big_ctas, ASM_THREADS, asm_smem_bytes(ctx->ns, ctx->nw, 256), cs>>>(a);
		CK(cudaGetLastError()); L.launches++;
	}
	CK(cudaEventRecord(L.ev[EV_ASM], cs));

	GenoArgs g; memset(&g, 0, sizeof g);
	g.region = a.region; g.read = a.read; g.seq2 = a.seq2; g.seqn = a.seqn; g.refcodes = a.refcodes; g.ctg_codes = a.ctg_codes;
	g.rres = a.rres; g.cres = a.cres; g.ares = a.ares; g.eres = (idl_event_result*)L.eres.p; g.cigar = (uint32_t*)L.cigar.p;
	g.cap_events = L.cap_events; g.cap_cigar = L.cap_cigar; g.cap_al = L.cap_events; g.cap_alns = L.cap_alns; g.cap_items = L.cap_items;
	g.al_list = (AlEntry*)L.al_list.p; g.al_items = (AlItem*)L.al_items.p; g.al_res = (int8_t*)L.al_res.p;
	g.sortA = sA; g.sortB = sB;
	g.P = P; g.cnt = a.cnt;
	g.kpA = ksw_make_params(P.match, P.mismatch, P.a_gapo, P.a_gape, P.a_bw, P.a_zdrop);
	g.kpB = ksw_make_params(P.match, P.mismatch, P.b_gapo, P.b_gape, P.b_bw, P.b_zdrop);
	g.pmat = (uint8_t*)L.pmat.p; g.p_cap = p_capA; g.cig_scratch = (uint32_t*)L.cig_scratch.p; g.cig_cap = ctx->cig_cap;
	g.seq_spill = (uint8_t*)L.seq_spill.p; g.seq_spill_cap = seq_spill_cap;
	if (b->n_regions > 0 && (P.stages & IDL_STAGE_ALIGN)) {
		const DpSmem sm = smem_site_a(P, (int)max_ref);
		g.ring_cols = sm.ring_cols; g.seq_cap = sm.seq_cap;
		const size_t smem = sm.bytes;
		if (smem > DP_SMEM_LIMIT) return IDL_E_CAPACITY; // idl_create's check makes this unreachable
		sort_scan_kernel<<<1, 1024, 0, cs>>>(sA);
		sort_scatter_kernel<<<ctx->n_sm * 4, 256, 0, cs>>>(sA, &a.cnt->n_alns, 1u, L.cap_alns);
		int nb = 0;
		if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, (const void*)align4_kernel, 32 * KSW_A4_WARPS, smem) != cudaSuccess || nb < 1) nb = 1;
		align4_kernel<<<(int)std::min((size_t)ctx->n_sm * std::min(nb, KSW_A4_CTAS), ctas_a), 32 * KSW_A4_WARPS, smem, cs>>>(g);
		CK(cudaGetLastError()); L.launches += 3;
	}
	CK(cudaEventRecord(L.ev[EV_ALN], cs));
	g.p_cap = p_capB;
	if (b->n_regions > 0 && (P.stages & IDL_STAGE_GENOTYPE) && (P.stages & IDL_STAGE_ALIGN)) {
		kmer_kernel<<<ctx->n_sm * 8, KMER_THREADS, 0, cs>>>(g);
		CK(cudaGetLastError()); L.launches++;
		CK(cudaEventRecord(L.ev[EV_KMER], cs));
		const DpSmem sm = smem_site_b(P, max_trim, (int)max_ref);
		g.ring_cols = sm.ring_cols; g.seq_cap = sm.seq_cap;
		const int al_warps = P.b_bw < 0 ? KSW_UNB_WARPS : DP_WARPS;
		const size_t smem = sm.bytes;
		if (smem > DP_SMEM_LIMIT) return IDL_E_CAPACITY; // idl_create's check makes this unreachable
		al_prep_kernel<<<ctx->n_sm * 8, 256, 0, cs>>>(g);
		sort_scan_kernel<<<1, 1024, 0, cs>>>(sB);
		sort_scatter_kernel<<<ctx->n_sm * 4, 256, 0, cs>>>(sB, &a.cnt->n_al_items, 2u, 2 * L.cap_items);
		if (P.b_bw < 0) al_kernel<true><<<std::min(dp_grid(ctx, (const void*)al_kernel<true>, smem, 32 * al_warps), (int)ctas_b), 32 * al_warps, smem, cs>>>(g); // unbanded (the reference's setting)
		else al_kernel<false><<<std::min(dp_grid(ctx, (const void*)al_kernel<false>, smem), (int)ctas_b), DP_THREADS, smem, cs>>>(g);
		al_vote_kernel<<<ctx->n_sm * 4, 256, 0, cs>>>(g);
		CK(cudaGetLastError()); L.launches += 5;
	} else CK(cudaEventRecord(L.ev[EV_KMER], cs));
	CK(cudaEventRecord(L.ev[EV_AL], cs));
	if (cs != L.stream) CK(cudaStreamWaitEvent(L.stream, L.ev[EV_AL], 0));
	CK(L.h_cnt.ensure(sizeof(DevCounters)));
	CK(cudaMemcpyAsync(L.h_cnt.p, L.cnt.p, sizeof(DevCounters), cudaMemcpyDeviceToHost, L.stream));
	CK(cudaEventRecord(L.ev[EV_END], L.stream));
	return IDL_OK;
}

Lane *find_lane(idl_ctx *ctx, uint64_t ticket)
{
	for (Lane &L : ctx->lanes) if (L.state != 0 && L.ticket == ticket) return &L;
	return nullptr;
}

} // namespace

extern "C" {

int idl_submit(idl_ctx *ctx, idl_batch *b, uint64_t *ticket)
{
	if (!ctx || !b || !ticket) return IDL_E_ARG;
	BatchSummary S;
	int rc = check_batch(ctx, b, S);
	if (rc) return rc;
	cudaSetDevice(ctx->device);
	Lane *Lp = nullptr;
	for (size_t k = 0; k < ctx->lanes.size(); ++k) { Lane &c = ctx->lanes[(ctx->next_ticket + k) % ctx->lanes.size()]; if (c.state == 0) { Lp = &c; break; } }
	if (!Lp) return IDL_E_BUSY;
	Lane &L = *Lp;
	L.resident = false; L.payload = true; L.retries = 0;
	L.max_trim = S.max_trim; L.max_ref = S.max_ref; L.n_small = S.n_small;
	CK(cudaEventRecord(L.ev[EV_START], L.stream));
	rc = stage_batch(ctx, L, b, true);
	if (rc) return rc;
	CK(cudaEventRecord(L.ev[EV_H2D], L.stream));
	rc = launch_chain(ctx, L);
	if (rc) return rc;
	L.ticket = ctx->next_ticket++; L.state = 1;
	*ticket = L.ticket;
	return IDL_OK;
}

// the batch of <n_regions> regions built by the device from a resident BAM into lane L's buffers (bamdev.cu); sets the lane's sizes and summary
static int build_from_bam(idl_ctx *ctx, Lane &L, idl_bam *bam, size_t n_regions, const int32_t *roi_chrom, const int32_t *roi_start, const int32_t *roi_end,
                          const int32_t *roi_n_reads, const int64_t *read_idx, uint32_t ordinal_base, BamBatchTotals &T)
{
	size_t n_reads = 0;
	for (size_t k = 0; k < n_regions; ++k) { if (roi_n_reads[k] < 0) return IDL_E_ARG; n_reads += (size_t)roi_n_reads[k]; }
	if (n_reads >= (1ull << 31) || n_regions >= (1ull << 31)) return IDL_E_CAPACITY;
	CK(L.region.ensure((n_regions + 1) * sizeof(idl_region))); CK(L.read.ensure((n_reads + 1) * sizeof(idl_read)));
	int rc = bam_batch_records(bam, L.stream, &ctx->P, n_regions, roi_chrom, roi_start, roi_end, roi_n_reads, read_idx, n_reads, ordinal_base,
	                           (idl_region*)L.region.p, (idl_read*)L.read.p, &T);
	if (rc) return rc;
	if (T.bad_index) return IDL_E_ARG;
	if (T.n_seq_bases >= (1ull << 32) || T.n_ref_bases >= (1ull << 32)) return IDL_E_CAPACITY;
	if ((int)T.max_region_reads + 2 > ctx->ns) return IDL_E_CAPACITY;
	L.n_regions = n_regions; L.n_reads = n_reads; L.n_seq_bases = (size_t)T.n_seq_bases; L.n_ref_bases = (size_t)T.n_ref_bases;
	CK(L.seq2.ensure(L.n_seq_bases / 4 + 16)); CK(L.seqn.ensure(L.n_seq_bases / 8 + 16)); CK(L.ref2.ensure(L.n_ref_bases / 4 + 16)); CK(L.refn.ensure(L.n_ref_bases / 8 + 16));
	rc = bam_batch_bases(bam, L.stream, n_regions, n_reads, (idl_region*)L.region.p, (const idl_read*)L.read.p, &T, (uint32_t*)L.seq2.p, (uint32_t*)L.seqn.p,
	                     (uint32_t*)L.ref2.p, (uint32_t*)L.refn.p);
	if (rc) return rc;
	L.max_trim = (int)std::max(1u, std::min(T.max_trim_len, (unsigned)ctx->P.max_read_len)); L.max_ref = std::max(16u, T.max_ref_len); L.n_small = T.n_small_regions;
	return IDL_OK;
}

int idl_bam_submit(idl_ctx *ctx, idl_bam *bam, size_t n_regions, const int32_t *roi_chrom, const int32_t *roi_start, const int32_t *roi_end, const int32_t *roi_n_reads,
                   const int64_t *read_idx, uint32_t ordinal_base, uint64_t *ticket)
{
	if (!ctx || !bam || !ticket || (n_regions && (!roi_chrom || !roi_start || !roi_end || !roi_n_reads))) return IDL_E_ARG;
	if (bam_device_of(bam) != ctx->device) return IDL_E_ARG;
	cudaSetDevice(ctx->device);
	Lane *Lp = nullptr;
	for (size_t k = 0; k < ctx->lanes.size(); ++k) { Lane &c = ctx->lanes[(ctx->next_ticket + k) % ctx->lanes.size()]; if (c.state == 0) { Lp = &c; break; } }
	if (!Lp) return IDL_E_BUSY;
	Lane &L = *Lp;
	L.resident = false; L.payload = true; L.retries = 0;
	CK(cudaEventRecord(L.ev[EV_START], L.stream));
	BamBatchTotals T;
	int rc = build_from_bam(ctx, L, bam, n_regions, roi_chrom, roi_start, roi_end, roi_n_reads, read_idx, ordinal_base, T);
	if (rc) return rc;
	CK(cudaEventRecord(L.ev[EV_H2D], L.stream));
	rc = launch_chain(ctx, L);
	if (rc) return rc;
	L.ticket = ctx->next_ticket++; L.state = 1;
	*ticket = L.ticket;
	return IDL_OK;
}

int idl_bam_pack(idl_ctx *ctx, idl_bam *bam, size_t n_regions, const int32_t *roi_chrom, const int32_t *roi_start, const int32_t *roi_end, const int32_t *roi_n_reads,
                 const int64_t *read_idx, uint32_t ordinal_base, idl_batch *b)
{
	if (!ctx || !bam || !b || (n_regions && (!roi_chrom || !roi_start || !roi_end || !roi_n_reads))) return IDL_E_ARG;
	if (bam_device_of(bam) != ctx->device) return IDL_E_ARG;
	cudaSetDevice(ctx->device);
	Lane *Lp = nullptr;
	for (Lane &c : ctx->lanes) if (c.state == 0) { Lp = &c; break; }
	if (!Lp) return IDL_E_BUSY;
	Lane &L = *Lp;
	BamBatchTotals T;
	int rc = build_from_bam(ctx, L, bam, n_regions, roi_chrom, roi_start, roi_end, roi_n_reads, read_idx, ordinal_base, T);
	L.resident = false;
	if (rc) return rc;
	if (L.n_regions > b->cap_regions || L.n_reads > b->cap_reads || L.n_seq_bases > b->cap_seq_bases || L.n_ref_bases > b->cap_ref_bases) return IDL_E_CAPACITY;
	CK(cudaMemcpyAsync(b->region, L.region.p, L.n_regions * sizeof(idl_region), cudaMemcpyDeviceToHost, L.stream));
	CK(cudaMemcpyAsync(b->read, L.read.p, L.n_reads * sizeof(idl_read), cudaMemcpyDeviceToHost, L.stream));
	CK(cudaMemcpyAsync(b->seq2, L.seq2.p, L.n_seq_bases / 4 + 16, cudaMemcpyDeviceToHost, L.stream)); CK(cudaMemcpyAsync(b->seqn, L.seqn.p, L.n_seq_bases / 8 + 16, cudaMemcpyDeviceToHost, L.stream));
	CK(cudaMemcpyAsync(b->ref2, L.ref2.p, L.n_ref_bases / 4 + 16, cudaMemcpyDeviceToHost, L.stream)); CK(cudaMemcpyAsync(b->refn, L.refn.p, L.n_ref_bases / 8 + 16, cudaMemcpyDeviceToHost, L.stream));
	CK(cudaStreamSynchronize(L.stream));
	b->n_regions = L.n_regions; b->n_reads = L.n_reads; b->n_seq_bases = L.n_seq_bases; b->n_ref_bases = L.n_ref_bases;
	b->max_trim_len = T.max_trim_len; b->max_ref_len = T.max_ref_len; b->max_region_reads = T.max_region_reads; b->n_small_regions = T.n_small_regions; b->summary_valid = 1;
	return IDL_OK;
}

int idl_upload(idl_ctx *ctx, idl_batch *b)
{
	if (!ctx || !b) return IDL_E_ARG;
	BatchSummary S;
	int rc = check_batch(ctx, b, S);
	if (rc) return rc;
	cudaSetDevice(ctx->device);
	Lane &L = ctx->lanes[0];
	if (L.state != 0) return IDL_E_BUSY;
	L.max_trim = S.max_trim; L.max_ref = S.max_ref; L.n_small = S.n_small;
	rc = stage_batch(ctx, L, b, true);
	if (rc) return rc;
	CK(cudaStreamSynchronize(L.stream));
	L.resident = true;
	return IDL_OK;
}

int idl_run_resident(idl_ctx *ctx, idl_batch *b, uint64_t *ticket)
{
	if (!ctx || !b || !ticket) return IDL_E_ARG;
	cudaSetDevice(ctx->device);
	Lane &L = ctx->lanes[0];
	if (L.state != 0) return IDL_E_BUSY;
	if (!L.resident || L.n_regions != b->n_regions || L.n_reads != b->n_reads) return IDL_E_ARG;
	L.payload = false; L.retries = 0;
	int rc = launch_chain(ctx, L, true);
	if (rc) return rc;
	L.ticket = ctx->next_ticket++; L.state = 1;
	*ticket = L.ticket;
	return IDL_OK;
}

int idl_wait(idl_ctx *ctx, uint64_t ticket, const idl_results **out)
{
	if (!ctx || !out) return IDL_E_ARG;
	Lane *Lp = find_lane(ctx, ticket);
	if (!Lp) return IDL_E_TICKET;
	Lane &L = *Lp;
	cudaSetDevice(ctx->device);
	if (L.state == 1) {
		CK(cudaStreamSynchronize(L.stream));
		const DevCounters *c = (const DevCounters*)L.h_cnt.p;
		// The CIGAR pool and the AL item pool are sized from estimates (48 ops per alignment, 8 AL events per read).  A batch that
		// needs more -- noisy contigs, deep regions over tandem repeats -- is run again with pools sized from what the device
		// counted: its inputs are still resident, nothing is returned from the short run, the caller only waits longer.
		while ((c->overflow & (8u | 64u)) && L.retries < 6) {
			if (c->overflow & 8u) L.cigar_per_aln = (unsigned)std::min<unsigned long long>(0xfffffu, std::max<unsigned long long>(2ull * L.cigar_per_aln, (unsigned long long)c->n_cigar_ops / std::max(1u, L.cap_alns) + 16));
			if (c->overflow & 64u) L.items_per_read = (unsigned)std::min<unsigned long long>(0xfffffu, std::max<unsigned long long>(2ull * L.items_per_read, (unsigned long long)c->n_al_items / std::max<size_t>(1, L.n_reads) + 2));
			L.retries += 1;
			int rc = launch_chain(ctx, L, !L.payload);
			if (rc) return rc;
			CK(cudaStreamSynchronize(L.stream));
		}
		idl_results &r = L.res; memset(&r, 0, sizeof r);
		r.n_regions = L.n_regions;
		r.n_contigs = std::min(c->n_contigs, L.cap_contigs);
		r.n_contig_bases = std::min(c->n_contig_bases, L.cap_bases);
		r.n_alns = std::min(c->n_alns, L.cap_alns);
		r.n_events = std::min(c->n_events, L.cap_events);
		r.n_cigar_ops = std::min(c->n_cigar_ops, L.cap_cigar);
		float t_d2h = 0;
		if (L.payload) {
			cudaEvent_t a0 = L.ev_d2h[0], a1 = L.ev_d2h[1]; // the lane's stage events still hold unread timings
			CK(L.h_rres.ensure((r.n_regions + 1) * sizeof(idl_region_result))); CK(L.h_cres.ensure((r.n_contigs + 1) * sizeof(idl_contig_result)));
			CK(L.h_ares.ensure((r.n_alns + 1) * sizeof(idl_aln_result))); CK(L.h_eres.ensure((r.n_events + 1) * sizeof(idl_event_result)));
			CK(L.h_cigar.ensure((r.n_cigar_ops + 1) * 4)); CK(L.h_seq.ensure(r.n_contig_bases + 16));
			CK(cudaEventRecord(a0, L.stream));
			if (r.n_regions) CK(cudaMemcpyAsync(L.h_rres.p, L.rres.p, r.n_regions * sizeof(idl_region_result), cudaMemcpyDeviceToHost, L.stream));
			if (r.n_contigs) CK(cudaMemcpyAsync(L.h_cres.p, L.cres.p, r.n_contigs * sizeof(idl_contig_result), cudaMemcpyDeviceToHost, L.stream));
			if (r.n_alns) CK(cudaMemcpyAsync(L.h_ares.p, L.ares.p, r.n_alns * sizeof(idl_aln_result), cudaMemcpyDeviceToHost, L.stream));
			if (r.n_events) CK(cudaMemcpyAsync(L.h_eres.p, L.eres.p, r.n_events * sizeof(idl_event_result), cudaMemcpyDeviceToHost, L.stream));
			if (r.n_cigar_ops) CK(cudaMemcpyAsync(L.h_cigar.p, L.cigar.p, r.n_cigar_ops * 4, cudaMemcpyDeviceToHost, L.stream));
			if (r.n_contig_bases) CK(cudaMemcpyAsync(L.h_seq.p, L.ctg_ascii.p, r.n_contig_bases, cudaMemcpyDeviceToHost, L.stream));
			if (ctx->P.out_flags & IDL_OUT_SUPPORT) {
				CK(L.h_sup.ensure((r.n_contig_bases + 4) * 4));
				if (r.n_contig_bases) CK(cudaMemcpyAsync(L.h_sup.p, L.ctg_sup.p, r.n_contig_bases * 4, cudaMemcpyDeviceToHost, L.stream));
			}
			CK(cudaEventRecord(a1, L.stream));
			CK(cudaStreamSynchronize(L.stream));
			cudaEventElapsedTime(&t_d2h, a0, a1);
			r.region = (const idl_region_result*)L.h_rres.p; r.contig = (const idl_contig_result*)L.h_cres.p; r.aln = (const idl_aln_result*)L.h_ares.p;
			r.event = (const idl_event_result*)L.h_eres.p; r.cigar = (const uint32_t*)L.h_cigar.p; r.contig_seq = (const char*)L.h_seq.p;
			r.contig_support = (ctx->P.out_flags & IDL_OUT_SUPPORT) ? (const uint32_t*)L.h_sup.p : nullptr;
		}
		cudaEventElapsedTime(&r.ms_h2d, L.ev[EV_START], L.ev[EV_H2D]);
		cudaEventElapsedTime(&r.ms_assemble, L.ev[EV_K0], L.ev[EV_ASM]);
		cudaEventElapsedTime(&r.ms_align, L.ev[EV_ASM], L.ev[EV_ALN]);
		cudaEventElapsedTime(&r.ms_genotype, L.ev[EV_ALN], L.ev[EV_KMER]);
		cudaEventElapsedTime(&r.ms_al, L.ev[EV_KMER], L.ev[EV_AL]);
		cudaEventElapsedTime(&r.ms_total, L.ev[EV_START], L.ev[EV_END]);
		r.ms_d2h = t_d2h; r.ms_total += t_d2h;
		r.offsets_tested = c->offsets_tested; r.dp_cells_a = c->dp_cells_a; r.dp_cells_b = c->dp_cells_b; r.dp_a = c->dp_a; r.dp_b = c->dp_b;
		r.kmer_reads = c->kmer_reads; r.kmer_bytes = c->kmer_bytes; r.al_events = c->al_events;
		r.kernel_launches = L.launches; r.pool_retries = (uint32_t)L.retries;
		if (c->overflow) snprintf(ctx->err, sizeof ctx->err, "result pool overflow mask 0x%x", c->overflow);
		L.state = 2;
		if (c->overflow) { *out = &L.res; return IDL_E_CAPACITY; }
	}
	*out = &L.res;
	return IDL_OK;
}

int idl_release(idl_ctx *ctx, uint64_t ticket)
{
	if (!ctx) return IDL_E_ARG;
	Lane *L = find_lane(ctx, ticket);
	if (!L) return IDL_E_TICKET;
	if (L->state == 1) { cudaSetDevice(ctx->device); cudaStreamSynchronize(L->stream); }
	L->state = 0;
	return IDL_OK;
}

} // extern "C"

// ---------------------------------------------------------------------------------------------------------------
// unit-level entry point: batch of independent alignments through kernel 2
// ---------------------------------------------------------------------------------------------------------------
namespace {

struct KswBatchArgs {
	unsigned n; const uint8_t *query, *target; const unsigned long long *q_off, *t_off;
	KswParams kp; idl_ez *out; uint32_t *cigar; unsigned long long *cigar_off; unsigned cigar_cap;
	unsigned *next; unsigned *cig_used;
	uint8_t *pmat; size_t p_cap; uint32_t *cig_scratch; int cig_cap; int ring_cols, seq_cap;
	int no_rows; // IDL_KSW2_COLUMNS=1: run every alignment on the column-owned ksw2_group<8> (tests compare it with the default variants)
};

// MODE 0: banded, shared-memory rings (any w >= 0), G threads per alignment; 1: unbanded (row-owned variant for reads of up to 160 bases, else the rings)
template <int MODE, int G>
__global__ void __launch_bounds__(G == 4 ? 32 * KSW_A4_WARPS : DP_THREADS, MODE == 1 ? 2 : (G == 4 ? KSW_A4_CTAS : 3)) ksw2_batch_kernel(KswBatchArgs a) // unbanded: 8 warps x 2 CTAs at 122 registers (uniform shapes: 774 GCUPS at 150x700 against 745 with al_kernel's 5 x 4)
{
	extern __shared__ __align__(16) unsigned char smem_raw[];
	constexpr int NG = 32 / G;
	const int lane = lane_id(), gl = lane & (G - 1), grp = lane / G;
	const int cg = warp_id() * NG + grp;
	const size_t per = ksw_group_smem(a.ring_cols, a.seq_cap);
	const size_t gg = (size_t)blockIdx.x * ((blockDim.x >> 5) * NG) + cg;
	KswMem M;
	ksw_group_mem(M, smem_raw + per * cg, grp, a.ring_cols); M.seq_cap = a.seq_cap; M.region_bytes = (int)per;
	M.pmat = a.pmat + gg * a.p_cap; M.p_cap = a.p_cap;
	M.cig = a.cig_scratch + gg * (size_t)a.cig_cap; M.cig_cap = a.cig_cap;
	for (;;) {
		unsigned base = 0;
		if (lane == 0) base = atomicAdd(a.next, (unsigned)NG);
		base = __shfl_sync(FULL_MASK, base, 0);
		if (base >= a.n) break;
		const unsigned i = base + grp;
		const bool valid = i < a.n;
		const int qlen = valid ? (int)(a.q_off[i + 1] - a.q_off[i]) : 0, tlen = valid ? (int)(a.t_off[i + 1] - a.t_off[i]) : 0;
		KswQuery kq; kq.codes = a.query + (valid ? a.q_off[i] : 0); kq.seq2 = nullptr; kq.seqn = nullptr; kq.base = 0;
		KswOut o;
		const uint8_t *tq = a.target + (valid ? a.t_off[i] : 0);
		if constexpr (G == 4) ksw2_group<4, true, false>(valid, qlen, kq, tlen, tq, a.kp, M, o);
		else {
			const int rw = MODE == 1 && !a.no_rows ? ksw_rows_pick(valid, qlen, tlen, a.kp, M) : 0;
			if (rw == 5) ksw2_rows<5, true>(valid, qlen, kq, tlen, tq, a.kp, M, o);
			else ksw2_group<8, true, MODE == 1>(valid, qlen, kq, tlen, tq, a.kp, M, o);
		}
		if (valid) {
			const unsigned gmask = ((1u << G) - 1u) << (lane & ~(G - 1));
			unsigned coff = 0;
			if (gl == 0) coff = atomicAdd(a.cig_used, (unsigned)o.n_cigar);
			coff = __shfl_sync(gmask, coff, 0, G);
			int status = o.status;
			if (coff + (unsigned)o.n_cigar > a.cigar_cap) status = KSW_ST_CIGCAP;
			else for (int k = gl; k < o.n_cigar; k += G) a.cigar[coff + k] = M.cig[o.n_cigar - 1 - k];
			if (gl == 0) {
				idl_ez e; e.max = o.max; e.zdropped = o.zdropped; e.max_q = o.max_q; e.max_t = o.max_t; e.mqe = o.mqe; e.mqe_t = o.mqe_t; e.mte = o.mte;
				e.mte_q = o.mte_q; e.score = o.score; e.n_cigar = o.n_cigar; e.status = status; e.reserved = 0; e.cells = o.cells;
				a.out[i] = e; a.cigar_off[i] = coff;
			}
		}
		__syncwarp();
	}
}

} // namespace

extern "C" int idl_ksw2_batch(idl_ctx *ctx, size_t n, const uint8_t *query, const uint64_t *q_off, const uint8_t *target, const uint64_t *t_off,
                              int8_t match, int8_t mismatch, int8_t gapo, int8_t gape, int w, int zdrop,
                              idl_ez *out, uint32_t *cigar, uint64_t *cigar_off, size_t cigar_cap, float *kernel_ms)
{
	if (!ctx || !query || !target || !q_off || !t_off || !out || !cigar || !cigar_off) return IDL_E_ARG;
	if (n == 0) return IDL_OK;
	if (n >= (1ull << 31) || cigar_cap >= (1ull << 32)) return IDL_E_ARG;
	cudaSetDevice(ctx->device);
	int max_q = 1, max_t = 1, max_ncol = 32; size_t max_p = 0;
	for (size_t i = 0; i < n; ++i) {
		const int ql = (int)(q_off[i + 1] - q_off[i]), tl = (int)(t_off[i + 1] - t_off[i]);
		max_q = std::max(max_q, ql); max_t = std::max(max_t, tl);
		const int nc = ksw_ncol(std::max(ql, 1), std::max(tl, 1), w);
		max_ncol = std::max(max_ncol, nc);
		max_p = std::max(max_p, (size_t)std::max(ql + tl - 1, 0) * std::max<size_t>(ksw_pitch(nc), w < 0 ? 32 * (size_t)ksw_rows_w(ql) : 0));
	}
	KswBatchArgs a; memset(&a, 0, sizeof a);
	a.n = (unsigned)n; a.kp = ksw_make_params(match, mismatch, gapo, gape, w, zdrop);
	{ const char *e = getenv("IDL_KSW2_COLUMNS"); a.no_rows = e && *e == '1'; }
	const bool g4 = w >= 0 && !a.no_rows; // the banded call-site with four threads per alignment, as align4_kernel
	const int ng = g4 ? 8 : DP_NG;
	a.ring_cols = ksw_ring_cols(max_ncol);
	a.p_cap = round_up(max_p + 2 * KSW_PMAT_PAD + 64, 256); a.cig_cap = max_q + max_t + 8; a.cigar_cap = (unsigned)cigar_cap;
	a.seq_cap = (int)round_up(ksw_seq_bytes(max_q, max_t), 16);
	const int wpc = g4 ? KSW_A4_WARPS : DP_WARPS; // warps per CTA
	const size_t smem = (size_t)wpc * ng * ksw_group_smem(a.ring_cols, a.seq_cap);
	if (smem > 200 * 1024) return IDL_E_CAPACITY;
	const void *kfn = w < 0 ? (const void*)ksw2_batch_kernel<1, 8> : g4 ? (const void*)ksw2_batch_kernel<0, 4> : (const void*)ksw2_batch_kernel<0, 8>;
	cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
	const size_t per_cta = (size_t)wpc * ng;
	const int ctas = (int)std::min<size_t>((n + per_cta - 1) / per_cta, (size_t)dp_grid(ctx, kfn, smem, 32 * wpc));
	const size_t nwarps = (size_t)ctas * per_cta; // groups, each with its own workspace
	const size_t qbytes = q_off[n], tbytes = t_off[n];
	DevBuf dq, dt, dqo, dto, dout, dcig, dcoff, dmisc, dp, dscr;
	cudaStream_t st = ctx->lanes[0].stream;
	int rc = IDL_OK;
	cudaEvent_t e0 = nullptr, e1 = nullptr;
	auto body = [&]() -> int {
		CK(dq.ensure(qbytes + 16)); CK(dt.ensure(tbytes + 16)); CK(dqo.ensure((n + 1) * 8)); CK(dto.ensure((n + 1) * 8));
		CK(dout.ensure(n * sizeof(idl_ez))); CK(dcig.ensure(cigar_cap * 4 + 16)); CK(dcoff.ensure(n * 8)); CK(dmisc.ensure(64));
		CK(dp.ensure(nwarps * a.p_cap)); CK(dscr.ensure(nwarps * (size_t)a.cig_cap * 4));
		CK(cudaMemcpyAsync(dq.p, query, qbytes, cudaMemcpyHostToDevice, st)); CK(cudaMemcpyAsync(dt.p, target, tbytes, cudaMemcpyHostToDevice, st));
		CK(cudaMemcpyAsync(dqo.p, q_off, (n + 1) * 8, cudaMemcpyHostToDevice, st)); CK(cudaMemcpyAsync(dto.p, t_off, (n + 1) * 8, cudaMemcpyHostToDevice, st));
		CK(cudaMemsetAsync(dmisc.p, 0, 64, st));
		a.query = (const uint8_t*)dq.p; a.target = (const uint8_t*)dt.p; a.q_off = (const unsigned long long*)dqo.p; a.t_off = (const unsigned long long*)dto.p;
		a.out = (idl_ez*)dout.p; a.cigar = (uint32_t*)dcig.p; a.cigar_off = (unsigned long long*)dcoff.p;
		a.next = (unsigned*)dmisc.p; a.cig_used = (unsigned*)dmisc.p + 1; a.pmat = (uint8_t*)dp.p; a.cig_scratch = (uint32_t*)dscr.p;
		CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
		CK(cudaEventRecord(e0, st));
		if (w < 0) ksw2_batch_kernel<1, 8><<<ctas, 32 * wpc, smem, st>>>(a);
		else if (g4) ksw2_batch_kernel<0, 4><<<ctas, 32 * wpc, smem, st>>>(a);
		else ksw2_batch_kernel<0, 8><<<ctas, DP_THREADS, smem, st>>>(a);
		CK(cudaGetLastError());
		CK(cudaEventRecord(e1, st));
		CK(cudaMemcpyAsync(out, dout.p, n * sizeof(idl_ez), cudaMemcpyDeviceToHost, st));
		CK(cudaMemcpyAsync(cigar, dcig.p, cigar_cap * 4, cudaMemcpyDeviceToHost, st));
		CK(cudaMemcpyAsync(cigar_off, dcoff.p, n * 8, cudaMemcpyDeviceToHost, st));
		CK(cudaStreamSynchronize(st));
		if (kernel_ms) cudaEventElapsedTime(kernel_ms, e0, e1);
		return IDL_OK;
	};
	rc = body();
	if (e0) cudaEventDestroy(e0);
	if (e1) cudaEventDestroy(e1);
	for (DevBuf *b : {&dq, &dt, &dqo, &dto, &dout, &dcig, &dcoff, &dmisc, &dp, &dscr}) b->release();
	return rc;
}
