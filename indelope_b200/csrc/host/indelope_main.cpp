// indelope_b200/csrc/host/indelope_main.cpp -- the `indelope` command line, drop-in for the reference's main module
// (src/indelope.nim:553-608):
//
//     indelope [options] <reference> <BAM>          VCF on stdout
//
// Same options, defaults and output as the reference's docopt block (:556-572).  The host part -- BAM sweep, evidence
// counters, coverage-gap chunking, VCF text -- is the C++ stand-in of libindelope_host.so (the reference keeps it in Nim);
// the BAM is streamed in bounded memory and every region of interest goes through libindelope_cuda.so in batches, two in flight.  There is no CPU path: without a
// CUDA device the program stops with an error.  CRAM input and the undocumented `single-site` debugging mode (:578-586)
// are not provided.
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <deque>
#include <map>
#include <string>
#include <chrono>
#include <thread>
#include <vector>
#include "indelope_cuda.h"
#include "indelope_host.h"

static const char USAGE[] =
	"indelope 0.0.1 (B200)\n"
	"\n"
	"  Usage: indelope [options] <reference> <BAM>\n"
	"\n"
	"Arguments:\n"
	"\n"
	"  <reference>     reference fasta file, plain or compressed with bgzip (with -g, -r or -R it is then inflated and parsed on the GPU).\n"
	"  <BAM>           call variants in this file (coordinate sorted).\n"
	"\n"
	"Options:\n"
	"\n"
	"  -m --min-reads <INT>        minimum number of reads to send for alignment [default: 3]\n"
	"  -c --min-contig-len <INT>   minimum contig length to send for alignment [default: 73]\n"
	"  -e --min-event-len <INT>    minimum size of indel to report [default: 4]\n"
	"  -t --threads <INT>          number of bam decompression threads [default: 1]\n"
	"  -d --device <INT>           CUDA device [default: 0]\n"
	"  -g --gpu-decode             inflate and parse the BAM and find the regions of interest on the GPU as well (idl_bam_open,\n"
	"                              idl_bam_sweep); the file is then read whole instead of streamed, --threads is not used\n"
	"  -r --region <chr[:beg[-end]]>  call only the regions of interest that overlap this region (1-based, inclusive, as samtools; may be\n"
	"                              repeated).  Only the BAM members that hold them are read, through <BAM>.bai; the regions found and called are\n"
	"                              exactly those of the whole-file run that overlap the region\n"
	"  -R --regions-file <BED>     the same for the intervals of a BED file (0-based, half open); -r and -R may be combined (their union)\n"
	"  -h --help                   show help\n";

struct Options {
	std::string fa, bam, bed;
	std::vector<std::string> regions;
	int min_reads = 3, min_ctg_len = 73, min_event_len = 4, threads = 1, device = 0;
	bool gpu_decode = false;
};
struct Lane { idl_batch *batch = nullptr; size_t cap[4] = {0, 0, 0, 0}; };
struct Flight { idlh_rois *rois; uint64_t ticket; };

// INDELOPE_TIMING=1: wall-clock phases on stderr
static const bool timing = getenv("INDELOPE_TIMING") != nullptr;
static double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

static int die(const char *what, const std::string &why) { fprintf(stderr, "indelope: %s: %s\n", what, why.c_str()); return 1; }
static int no_device(int rc) { return die("libindelope_cuda", std::string(idl_strerror(rc)) + " (this program has no CPU path; it needs a CUDA device)"); }

// gen_roi(b, target, min_read_coverage=min_reads, min_event_support=max(3, min_reads-2)), src/indelope.nim:602
static int32_t min_event_support(const Options &o) { return o.min_reads - 2 > 3 ? o.min_reads - 2 : 3; }
static bool is_decoy(const char *name) { return strcmp(name, "hs37d5") == 0 || strncmp(name, "GL", 2) == 0; }   // skippable targets, :41-42

// echo header % [b.contig_header, "sample"], :599
static void print_header(const idlh_rois *targets) { char *h = idlh_vcf_header(idlh_rois_view(targets)); fputs(h, stdout); idlh_free(h); }
// the targets of a dataset (names and sequences) without any region
static idlh_rois *no_regions(const idlh_dataset *d)
{
	return idlh_rois_from_arrays(d, 0, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0, nullptr, nullptr, nullptr, nullptr, nullptr);
}

static int64_t file_size(const std::string &path)   // -1: cannot open
{
	FILE *f = fopen(path.c_str(), "rb");
	if (!f) return -1;
	fseek(f, 0, SEEK_END); const long n = ftell(f);
	fclose(f);
	return n > 0 ? n : 0;
}
// bytes [begin, end) of a file into out; "" or why not
static std::string read_range(const std::string &path, uint64_t begin, uint64_t end, std::vector<uint8_t> &out)
{
	out.resize((size_t)(end - begin));
	FILE *f = fopen(path.c_str(), "rb");
	if (!f) return "cannot open " + path;
	const bool ok = fseek(f, (long)begin, SEEK_SET) == 0 && fread(out.data(), 1, out.size(), f) == out.size();
	fclose(f);
	return ok ? "" : "cannot read " + path;
}

// The calling half of every front end (the twin of api.Caller): one context, batches of regions submitted in emission order with at most n_streams in
// flight, and their records on stdout in the same order (the dedup of :604-608 depends on it).  The front ends that decode on the device give it the
// reference as well (the FASTA's sequences in the BAM header's order): the batches' views and idl_bam_set_reference read it.
struct Calls {
	idl_params P;
	idl_ctx *ctx = nullptr;
	int create_rc = IDL_OK;
	idlh_dataset *ref = nullptr;
	idlh_rois *targets = nullptr;          // ref without regions
	idl_fasta *fa = nullptr;               // a bgzipped reference parsed on the device (open_reference): the batches take its sequences from there
	std::vector<int64_t> fa_record;        // per target of ref: its record in fa
	idlh_vcf *writer = idlh_vcf_new();
	std::vector<Lane> lanes;               // pinned batches of submit_packed, one per stream
	std::deque<Flight> inflight;
	size_t n_regions = 0, n_batches = 0;   // submitted so far: the next region's ordinal is n_regions
	double t_create = 0, t_ref = 0, t_submit = 0, t_wait = 0, t_vcf = 0;
	int status = 0;                        // 1 once an error has been reported

	explicit Calls(const Options &o)
	{
		idl_default_params(&P);
		P.min_reads = o.min_reads; P.min_ctg_len = o.min_ctg_len; P.min_event_len = o.min_event_len;
		lanes.resize((size_t)(P.n_streams > 0 ? P.n_streams : 1));
	}
	Calls(const Calls &) = delete;
	Calls &operator=(const Calls &) = delete;
	~Calls() { close(); }

	void create(int device) { const double t0 = now_s(); create_rc = idl_create(device, &P, &ctx); t_create = now_s() - t0; }

	bool drain()
	{
		const Flight f = inflight.front(); inflight.pop_front();
		const idl_results *res = nullptr;
		double t0 = now_s();
		const int r = idl_wait(ctx, f.ticket, &res);
		t_wait += now_s() - t0; t0 = now_s();
		if (r != IDL_OK) { status = die("idl_wait", std::string(idl_strerror(r)) + " " + idl_last_cuda_error(ctx)); idlh_rois_free(f.rois); return false; }
		char *txt = idlh_vcf_records(writer, idlh_rois_view(f.rois), 0, &P, res, 0, nullptr);
		fputs(txt, stdout); idlh_free(txt);
		idl_release(ctx, f.ticket);
		idlh_rois_free(f.rois);
		t_vcf += now_s() - t0;
		return true;
	}
	bool make_room() { return inflight.size() < lanes.size() || drain(); }
	// every batch in flight written; after an error they are only freed
	int finish()
	{
		while (!inflight.empty() && !status) drain();
		while (!inflight.empty()) { idlh_rois_free(inflight.front().rois); inflight.pop_front(); }
		return status;
	}

	// one self-contained group of regions (takes it), packed on the host into its lane's pinned batch
	bool submit_packed(idlh_rois *grp)
	{
		const idlh_roiset *rs = idlh_rois_view(grp);
		if (!make_room()) { idlh_rois_free(grp); return false; }
		const double t0 = now_s();
		Lane &L = lanes[n_batches % lanes.size()];
		size_t need[4] = {(size_t)rs->n_rois, 0, 0, 0};
		idlh_pack_size(rs, 0, rs->n_rois, &P, &need[1], &need[2], &need[3]);
		bool grow = L.batch == nullptr;
		for (int k = 0; k < 4; ++k) grow |= need[k] > L.cap[k];
		if (grow) {
			if (L.batch) idl_batch_free(ctx, L.batch);
			L.batch = nullptr;
			for (int k = 0; k < 4; ++k) L.cap[k] = need[k] + need[k] / 4 + 64;
			const int rc = idl_batch_alloc(ctx, L.cap[0], L.cap[1], L.cap[2], L.cap[3], &L.batch);
			if (rc != IDL_OK) { status = die("idl_batch_alloc", idl_strerror(rc)); idlh_rois_free(grp); return false; }
		}
		if (idlh_pack(rs, 0, rs->n_rois, &P, L.batch) != 0) { status = die("idlh_pack", "the pinned batch is smaller than idlh_pack_size reported (internal error)"); idlh_rois_free(grp); return false; }
		uint64_t ticket = 0;
		const int rc = idl_submit(ctx, L.batch, &ticket);
		if (rc != IDL_OK) { status = die("idl_submit", std::string(idl_strerror(rc)) + " " + idl_last_cuda_error(ctx)); idlh_rois_free(grp); return false; }
		inflight.push_back({grp, ticket});
		t_submit += now_s() - t0;
		n_regions += (size_t)rs->n_rois; ++n_batches;
		return true;
	}

	// regions [0, n) of a BAM resident on the device (targets in header order, regions in gen_roi's order, read_idx its records), the batches built on the
	// device (idl_bam_submit) from at most 400 000 reads and 20 000 regions each.  Returns once every batch is written, so that the BAM may be closed.
	int call_resident(idl_bam *bam, size_t n, const int32_t *chrom, const int32_t *start, const int32_t *end, const int32_t *n_reads, const int64_t *read_idx)
	{
		const idlh_roiset *all = idlh_rois_view(targets);
		double t0 = now_s();
		for (size_t k = 0; k < n && !status; ++k) {
			if (k > 0 && chrom[k] == chrom[k - 1]) continue;
			const int r = fa ? idl_bam_set_reference_fasta(bam, chrom[k], fa, fa_record[(size_t)chrom[k]])
			                 : idl_bam_set_reference(bam, chrom[k], all->chrom_seq[chrom[k]], all->chrom_len[chrom[k]]);
			if (r != IDL_OK) status = die("idl_bam_set_reference", "could not place the reference on the device");
		}
		t_ref += now_s() - t0;
		size_t at_idx = 0;
		for (size_t lo = 0; lo < n && !status; ) {
			size_t hi = lo; int64_t reads = 0;
			while (hi < n && (hi == lo || (reads + n_reads[hi] <= 400000 && hi - lo < 20000))) reads += n_reads[hi++];
			if (!make_room()) break;
			t0 = now_s();
			// the VCF stage reads only the regions' coordinates and the reference of this group
			idlh_rois *grp = idlh_rois_from_arrays(ref, 0, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, (int64_t)(hi - lo), chrom + lo,
			                                       start + lo, end + lo, n_reads + lo, read_idx + at_idx);
			uint64_t ticket = 0;
			const int r = idl_bam_submit(ctx, bam, hi - lo, chrom + lo, start + lo, end + lo, n_reads + lo, read_idx + at_idx, (uint32_t)(n_regions + lo), &ticket);
			if (r != IDL_OK) { status = die("idl_bam_submit", std::string(idl_strerror(r)) + " " + idl_last_cuda_error(ctx)); idlh_rois_free(grp); break; }
			inflight.push_back({grp, ticket});
			t_submit += now_s() - t0;
			at_idx += (size_t)reads; lo = hi; ++n_batches;
		}
		n_regions += n;
		return finish();
	}

	void close()
	{
		finish();
		for (Lane &L : lanes) if (L.batch) idl_batch_free(ctx, L.batch);
		lanes.clear();
		if (writer) idlh_vcf_free(writer);
		writer = nullptr;
		if (ctx) idl_destroy(ctx);
		ctx = nullptr;
		if (targets) idlh_rois_free(targets);
		targets = nullptr;
		if (ref) idlh_dataset_free(ref);
		ref = nullptr;
		if (fa) idl_fasta_close(fa);
		fa = nullptr;
	}

	// after ref has been ordered as the BAM header lists its targets: each target's record in fa (the first of its name, as idlh_dataset_set_targets
	// takes it)
	void map_fasta_records()
	{
		if (!fa) return;
		const idl_fasta_info *fi = idl_fasta_get_info(fa);
		std::map<std::string, int64_t> first;
		for (int64_t r = fi->n_records - 1; r >= 0; --r) first[fi->name[r]] = r;
		fa_record.clear();
		for (int32_t c = 0; c < idlh_dataset_n_chroms(ref); ++c) fa_record.push_back(first[idlh_dataset_chrom_name(ref, c)]);
	}
};

static bool is_gzip(const std::string &path)
{
	FILE *f = fopen(path.c_str(), "rb");
	if (!f) return false;
	unsigned char m[2] = {0, 0};
	const bool gz = fread(m, 1, 2, f) == 2 && m[0] == 0x1f && m[1] == 0x8b;
	fclose(f);
	return gz;
}

// The reference of the front ends that decode on the device, into calls.ref (the FASTA's records in file order).  A bgzipped FASTA is read here and
// inflated and parsed on the device (idl_fasta_open), where it stays for idl_bam_set_reference_fasta; the host keeps copies of the sequences for the
// VCF writer.  A plain FASTA is loaded on the host as before.  0, or the exit status after the message.
static int open_reference(const Options &o, Calls &calls)
{
	char err[512] = {0};
	if (!is_gzip(o.fa)) {
		calls.ref = idlh_load_fasta(o.fa.c_str(), err, sizeof err);
		return calls.ref ? 0 : die("input", err);
	}
	const double t0 = now_s();
	const int64_t size = file_size(o.fa);
	std::vector<uint8_t> file;
	const std::string why = size < 0 ? "cannot open " + o.fa : read_range(o.fa, 0, (uint64_t)size, file);
	if (!why.empty()) return die("input", why);
	const double t_read = now_s() - t0, t1 = now_s();
	const int rc = idl_fasta_open(o.device, file.data(), file.size(), &calls.fa, err, sizeof err);
	if (rc == IDL_E_NO_DEVICE) return no_device(rc);
	if (rc != IDL_OK) return die("input", o.fa + ": " + (err[0] ? err : idl_strerror(rc)));
	const double t_open = now_s() - t1, t2 = now_s();
	const idl_fasta_info *fi = idl_fasta_get_info(calls.fa);
	std::vector<std::vector<uint8_t>> seqs((size_t)fi->n_records);
	std::vector<const uint8_t*> sp; std::vector<const char*> np;
	for (int64_t r = 0; r < fi->n_records; ++r) {
		seqs[(size_t)r].resize((size_t)fi->len[r]);
		if (idl_fasta_copy(calls.fa, r, seqs[(size_t)r].data(), seqs[(size_t)r].size()) != IDL_OK) return die("idl_fasta_copy", "cannot copy the reference back from the device");
		sp.push_back(seqs[(size_t)r].data()); np.push_back(fi->name[r]);
	}
	calls.ref = idlh_dataset_from_sequences((int32_t)fi->n_records, np.data(), sp.data(), fi->len);
	if (timing)
		fprintf(stderr, "indelope timing (reference on the device): read %.3f s, idl_fasta_open %.3f s (h2d %.1f ms, inflate %.1f ms, parse %.1f ms; %.1f MB -> %.1f MB -> "
		        "%.1f MB of sequence, %lld records), copy back %.3f s\n", t_read, t_open, fi->ms_h2d, fi->ms_inflate, fi->ms_parse, fi->file_bytes / 1e6,
		        fi->inflated_bytes / 1e6, fi->sequence_bytes / 1e6, (long long)fi->n_records, now_s() - t2);
	return 0;
}

// The host reads and sweeps the BAM, a group of regions at a time, in bounded memory (idlh_stream_*); while the GPU works on a batch the host reads and
// sweeps the next stretch of the file.
static int run_streamed(const Options &o)
{
	char err[512] = {0};
	const double t_begin = now_s();
	idlh_stream *in = idlh_stream_open(o.fa.c_str(), o.bam.c_str(), o.threads, min_event_support(o), o.min_reads, 600, err, sizeof err);
	if (!in) return die("input", err);
	Calls calls(o);
	int &status = calls.status;
	// the CUDA context and the library's workspaces come up on a helper thread while this one already reads the BAM; nothing
	// is printed before the context exists (without a device the program fails with empty stdout)
	const double t_open = now_s() - t_begin;
	std::thread creator([&]() { calls.create(o.device); });
	bool have_ctx = false;
	auto need_ctx = [&]() -> bool {
		if (have_ctx) return true;
		creator.join();
		if (calls.create_rc != IDL_OK) { status = no_device(calls.create_rc); return false; }
		idlh_rois *t = idlh_stream_targets(in);
		print_header(t);
		idlh_rois_free(t);
		have_ctx = true;
		return true;
	};
	double t_sweep = 0;
	while (!status) {
		err[0] = 0;
		const double t0 = now_s();
		idlh_rois *grp = idlh_stream_next(in, 400000, err, sizeof err);
		t_sweep += now_s() - t0;
		if (!grp) { if (err[0]) status = die("input", err); break; }
		if (idlh_rois_view(grp)->n_rois == 0) { idlh_rois_free(grp); continue; }
		if (!need_ctx()) { idlh_rois_free(grp); break; }
		calls.submit_packed(grp);
	}
	if (!status) need_ctx(); // a BAM without any region still gets its header
	calls.finish();
	if (creator.joinable()) creator.join();
	const double t0 = now_s();
	calls.close();
	idlh_stream_close(in);
	if (timing)
		fprintf(stderr, "indelope timing: open %.3f s, idl_create %.3f s, read+sweep %.3f s, pack+submit %.3f s, idl_wait %.3f s, vcf %.3f s, teardown %.3f s, total %.3f s, batches %zu\n",
		        t_open, calls.t_create, t_sweep, calls.t_submit, calls.t_wait, calls.t_vcf, now_s() - t0, now_s() - t_begin, calls.n_batches);
	return status;
}

// --gpu-decode: the whole front end on the GPU.  The file's bytes go to the device, idl_bam_open inflates the BGZF members and parses the records there,
// idl_bam_sweep runs gen_roi per target on the resident records, and the batches are built on the device from the resident records and reference:
// nothing but the regions' coordinates and record indices crosses the bus.  The host reads the two files and writes the VCF.
static int run_whole_file(const Options &o)
{
	char err[512] = {0}, bam_err[512] = {0};
	const double t_begin = now_s();
	std::vector<uint8_t> file;
	const int64_t size = file_size(o.bam);
	if (size < 0) return die("input", "cannot open " + o.bam);
	const std::string why = read_range(o.bam, 0, (uint64_t)size, file);
	if (!why.empty()) return die("input", why);
	const double t_read = now_s() - t_begin;
	Calls calls(o);
	int &status = calls.status;
	// the device decodes the BAM and creates the calling context while this thread reads the FASTA
	idl_bam *bam = nullptr; int open_rc = IDL_OK; double t_open = 0;
	std::thread opener([&]() {
		const double t1 = now_s();
		open_rc = idl_bam_open(o.device, file.data(), file.size(), &bam, bam_err, sizeof bam_err);
		t_open = now_s() - t1;
		if (open_rc == IDL_OK) calls.create(o.device);
	});
	double t1 = now_s();
	const int ref_status = open_reference(o, calls);
	const double t_fasta = now_s() - t1;
	opener.join();
	std::vector<uint8_t>().swap(file);
	if (ref_status) status = ref_status;
	else if (open_rc == IDL_E_NO_DEVICE) status = no_device(open_rc);
	else if (open_rc != IDL_OK) status = die("input", o.bam + ": " + (bam_err[0] ? bam_err : idl_strerror(open_rc)));
	else if (calls.create_rc != IDL_OK) status = no_device(calls.create_rc);
	const idl_bam_info *info = bam ? idl_bam_get_info(bam) : nullptr;
	if (!status && idlh_dataset_set_targets(calls.ref, info->n_ref, info->ref_name, info->ref_len, err, sizeof err) != 0) status = die("input", err);
	if (!status) calls.map_fasta_records();
	double t_sweep = 0;
	if (!status) {
		// gen_roi per target, in header order (:599-602)
		std::vector<int32_t> rc_, rs_, re_, rn_; std::vector<int64_t> idx_;
		t1 = now_s();
		for (int32_t c = 0; c < info->n_ref; ++c) {
			if (is_decoy(info->ref_name[c])) continue;
			idl_sweep_out *so = nullptr;
			const int r = idl_bam_sweep(bam, c, min_event_support(o), o.min_reads, 600, 0, &so);
			if (r != IDL_OK) { status = die("idl_bam_sweep", idl_strerror(r)); break; }
			for (size_t k = 0; k < so->n_rois; ++k) { rc_.push_back(c); rs_.push_back(so->roi_start[k]); re_.push_back(so->roi_end[k]); rn_.push_back(so->roi_n_reads[k]); }
			idx_.insert(idx_.end(), so->read_idx, so->read_idx + so->n_read_idx);
			idl_sweep_free(so);
		}
		t_sweep = now_s() - t1;
		if (!status) {
			calls.targets = no_regions(calls.ref);
			print_header(calls.targets);
			calls.call_resident(bam, rs_.size(), rc_.data(), rs_.data(), re_.data(), rn_.data(), idx_.data());
		}
	}
	if (timing && info)
		fprintf(stderr, "indelope timing (gpu decode): read file %.3f s, fasta %.3f s, idl_bam_open %.3f s (h2d %.1f ms, inflate %.1f ms, parse %.1f ms; %.1f MB -> %.1f MB, "
		        "%lld records, %u boundary fixups), idl_create %.3f s, idl_bam_sweep %.3f s, reference %.3f s, build+submit %.3f s, idl_wait %.3f s, vcf %.3f s, total %.3f s, "
		        "batches %zu, regions %zu\n", t_read, t_fasta, t_open, info->ms_h2d, info->ms_inflate, info->ms_parse, info->file_bytes / 1e6, info->inflated_bytes / 1e6,
		        (long long)info->n_records, info->boundary_fixups, calls.t_create, t_sweep, calls.t_ref, calls.t_submit, calls.t_wait, calls.t_vcf, now_s() - t_begin,
		        calls.n_batches, calls.n_regions);
	if (bam) idl_bam_close(bam);
	return status;
}

// -r / -R, and --gpu-decode target by target (every target whole) for a file that does not fit in device memory: only the BAM members that hold the
// intervals are decoded.  Per target the intervals become slices of the file: from the linear-index offset of the 16 kb window in front of an interval to
// that of the window behind it (idlh_bai_region_run); slices of a target whose member runs overlap or touch are merged and decoded once.  Each slice is
// decoded (idl_bam_open_slice) and swept over the zone of positions whose evidence it determines exactly (idl_bam_sweep_window, DESIGN.md 4a); when a
// selected region touches an inner edge of the zone, or the zone does not reach the last interval, the slice grows by one window on that side and is swept
// again.  Every target's slices are planned up front, so that a reader thread reads the next slice's members, of the same target or the next one, while
// the device decodes and calls this one.
static int run_sliced(const Options &o)
{
	char err[512] = {0};
	const double t_begin = now_s();
	Calls calls(o);
	int &status = calls.status;
	std::thread creator([&]() { calls.create(o.device); });
	// one slice: a target's window range [w0, w1], its intervals, where its members lie
	struct Slice { int32_t c = 0; int64_t w0 = 0, w1 = 0; std::vector<int32_t> beg, end; uint64_t fb = 0, fe = 0, first = 0, em = 0, eo = 0; int64_t zone_lo = 0; int32_t to_end = 1; int rr = 1; };
	auto locate = [&](Slice &S) -> bool {
		S.rr = idlh_bai_region_run(o.bam.c_str(), S.c, S.w0, S.w1, &S.fb, &S.fe, &S.first, &S.em, &S.eo, &S.zone_lo, &S.to_end, err, sizeof err);
		if (S.rr < 0) { status = die("input", o.bam + ": " + err); return false; }
		return true;
	};
	std::vector<const char*> names; std::vector<int64_t> lens;
	std::deque<Slice> todo;
	size_t n_intervals = 0;
	// the intervals, targets in header order, and the first slice of each: the window holding the position in front of it to the window behind its last
	// base.  Every error of these comes before a missing device's, and before anything is printed.
	auto plan = [&]() {
		if ((status = open_reference(o, calls))) return;
		if (idlh_dataset_set_bam_targets(calls.ref, o.bam.c_str(), err, sizeof err) != 0) { status = die("input", err); return; }
		calls.map_fasta_records();
		calls.targets = no_regions(calls.ref);
		const idlh_roiset *all = idlh_rois_view(calls.targets);
		for (int32_t c = 0; c < all->n_chroms; ++c) { names.push_back(all->chrom_name[c]); lens.push_back(all->chrom_len[c]); }
		std::vector<int32_t> ic; std::vector<int64_t> ib, ie;
		if (o.regions.empty() && o.bed.empty()) {
			for (int32_t c = 0; c < all->n_chroms; ++c)
				if (!is_decoy(names[(size_t)c])) { ic.push_back(c); ib.push_back(0); ie.push_back(lens[(size_t)c]); }
		} else {
			std::vector<const char*> rv; for (const std::string &r : o.regions) rv.push_back(r.c_str());
			idlh_regions *sel = idlh_regions_parse(all->n_chroms, names.data(), lens.data(), (int32_t)rv.size(), rv.data(), o.bed.empty() ? nullptr : o.bed.c_str(), err, sizeof err);
			if (!sel) { status = die("regions", err); return; }
			for (int32_t c = 0; c < all->n_chroms; ++c) {
				const size_t n = (size_t)idlh_regions_get(sel, c, nullptr, nullptr, 0);
				ic.resize(ic.size() + n, c); ib.resize(ib.size() + n); ie.resize(ie.size() + n);
				idlh_regions_get(sel, c, ib.data() + ib.size() - n, ie.data() + ie.size() - n, (int64_t)n);
			}
			idlh_regions_free(sel);
		}
		uint64_t v[5];
		if (all->n_chroms > 0 && idlh_bai_target_span(o.bam.c_str(), 0, v, v + 1, v + 2, v + 3, v + 4, err, sizeof err) < 0) { status = die("input", o.bam + ": " + err); return; }
		n_intervals = ic.size();
		for (size_t k = 0; k < ic.size(); ++k) {
			Slice S;
			S.c = ic[k]; S.w0 = ib[k] > 0 ? (ib[k] - 1) >> 14 : 0; S.w1 = ((ie[k] - 1) >> 14) + 1;
			S.beg.push_back((int32_t)ib[k]); S.end.push_back((int32_t)ie[k]);
			if (!todo.empty() && todo.back().c == S.c && S.w0 <= todo.back().w1) {   // overlapping window ranges: one slice
				Slice &B = todo.back(); B.w1 = std::max(B.w1, S.w1); B.beg.push_back(S.beg[0]); B.end.push_back(S.end[0]);
			} else todo.push_back(S);
		}
		for (Slice &S : todo) if (!locate(S)) return;
	};
	plan();
	creator.join();
	if (status) return status;
	if (calls.create_rc != IDL_OK) return no_device(calls.create_rc);
	print_header(calls.targets);
	size_t n_slices = 0, n_retries = 0; uint64_t bytes_read = 0, bytes_decoded = 0;
	double t_read = 0, t_open = 0, t_sweep = 0, t_call = 0;
	struct Read { uint64_t fb = 0, fe = 0; std::vector<uint8_t> bytes; std::string error; };
	auto load = [&](uint64_t fb, uint64_t fe, Read *R) { R->fb = fb; R->fe = fe; R->error = read_range(o.bam, fb, fe, R->bytes); };
	Read ahead; std::thread reader;
	int32_t last_c = -1; int64_t last_end = -1;   // the last region called: its target and end
	while (!todo.empty() && !status) {
		Slice S = todo.front(); todo.pop_front();
		const int32_t c = S.c;
		// slices whose member runs overlap or touch are decoded once
		while (!todo.empty() && S.rr == 0 && todo.front().rr == 0 && todo.front().c == c && todo.front().fb <= S.fe) {
			const Slice &N = todo.front();
			S.w1 = std::max(S.w1, N.w1); S.beg.insert(S.beg.end(), N.beg.begin(), N.beg.end()); S.end.insert(S.end.end(), N.end.begin(), N.end.end());
			todo.pop_front();
			if (!locate(S)) break;
		}
		if (status) break;
		if (S.rr == 1) {   // no record in the run
			if (S.to_end) continue;                      // ... up to the target's end: no region
			++S.w1; ++n_retries;
			if (locate(S)) todo.push_front(S);
			continue;
		}
		double t1 = now_s();
		if (reader.joinable()) reader.join();
		Read R;
		if (ahead.fb == S.fb && ahead.fe == S.fe && !ahead.bytes.empty()) R = std::move(ahead); else load(S.fb, S.fe, &R);
		ahead = Read();
		if (!todo.empty() && todo.front().rr == 0) reader = std::thread(load, todo.front().fb, todo.front().fe, &ahead);   // the next slice as it stands
		t_read += now_s() - t1;
		if (!R.error.empty()) { status = die("input", R.error); break; }
		bytes_read += R.bytes.size();
		t1 = now_s();
		idl_bam_slice sl; memset(&sl, 0, sizeof sl);
		sl.n_ref = (int32_t)names.size(); sl.ref_name = names.data(); sl.ref_len = lens.data(); sl.first_record = S.first; sl.end_member = S.em; sl.end_offset = S.eo;
		idl_bam *bam = nullptr; char berr[512] = {0};
		const int orc = idl_bam_open_slice(o.device, R.bytes.data(), R.bytes.size(), &sl, &bam, berr, sizeof berr);
		if (orc != IDL_OK) { status = die("input", o.bam + " (" + names[(size_t)c] + "): " + (berr[0] ? berr : idl_strerror(orc))); break; }
		const idl_bam_info *info = idl_bam_get_info(bam);
		bytes_decoded += info->inflated_bytes; ++n_slices;
		t_open += now_s() - t1; t1 = now_s();
		// the zone: positions below the start of the slice's last record are exact (every record left out on the right starts there or later)
		int64_t zone_hi = lens[(size_t)c];
		if (!S.to_end) {
			const int64_t last = info->n_records - 1;
			idl_bam_reads *rd = nullptr;
			if (last < 0 || idl_bam_fetch(bam, 1, &last, 0, &rd) != IDL_OK) { status = die("idl_bam_fetch", "cannot read the slice's last record"); idl_bam_close(bam); break; }
			zone_hi = (int64_t)rd->start[0] - 1;
			idl_bam_reads_free(rd);
		}
		if (zone_hi < S.zone_lo || zone_hi < (int64_t)S.end.back() - 1) {   // the zone does not reach the last interval's last base yet
			idl_bam_close(bam);
			++S.w1; ++n_retries;
			if (locate(S)) todo.push_front(S);
			t_sweep += now_s() - t1;
			continue;
		}
		idl_sweep_out *so = nullptr;
		const int r = idl_bam_sweep_window(bam, c, (int32_t)S.zone_lo, (int32_t)zone_hi, S.beg.size(), S.beg.data(), S.end.data(), min_event_support(o), o.min_reads, 600, 0, &so);
		if (r != IDL_OK) { status = die("idl_bam_sweep_window", idl_strerror(r)); idl_bam_close(bam); break; }
		t_sweep += now_s() - t1; t1 = now_s();
		if (so->n_edge[0] || so->n_edge[1]) {   // a selected region reaches beyond the zone: grow the slice on that side
			if (so->n_edge[0]) --S.w0;
			if (so->n_edge[1]) ++S.w1;
			++n_retries;
			idl_sweep_free(so); idl_bam_close(bam);
			if (locate(S)) todo.push_front(S);
			continue;
		}
		// a slice grown to the left may share regions with the slice of its target before it: those were called there
		if (c != last_c) { last_c = c; last_end = -1; }
		size_t first = 0;
		while (first < so->n_rois && so->roi_start[first] <= last_end) ++first;
		const size_t n = so->n_rois - first;
		const std::vector<int32_t> chrom(n, c);
		calls.call_resident(bam, n, chrom.data(), so->roi_start + first, so->roi_end + first, so->roi_n_reads + first, so->read_idx + (n ? so->roi_read_begin[first] : 0));
		if (n) last_end = so->roi_end[so->n_rois - 1];
		idl_sweep_free(so);
		idl_bam_close(bam);
		t_call += now_s() - t1;
	}
	if (reader.joinable()) reader.join();
	if (timing)
		fprintf(stderr, "indelope timing (regions): %zu intervals, %.1f MB read, %.1f MB decoded, slices %zu, retries %zu, regions %zu; waited %.3f s for reads, "
		        "idl_bam_open_slice %.3f s, zone + idl_bam_sweep_window %.3f s, build + call + vcf %.3f s, total %.3f s\n", n_intervals, bytes_read / 1e6,
		        bytes_decoded / 1e6, n_slices, n_retries, calls.n_regions, t_read, t_open, t_sweep, t_call, now_s() - t_begin);
	return status;
}

int main(int argc, char **argv)
{
	Options o;
	std::vector<std::string> pos;
	for (int i = 1; i < argc; ++i) {
		const std::string a = argv[i];
		auto int_opt = [&](const char *s, const char *l, int &dst) -> int { // 0 no match, 1 consumed, -1 error
			std::string v;
			if (a == s || a == l) { if (i + 1 >= argc) return -1; v = argv[++i]; }
			else if (a.rfind(std::string(l) + "=", 0) == 0) v = a.substr(strlen(l) + 1);
			else if (a.size() > 2 && a.compare(0, 2, s) == 0 && a[1] != '-') v = a.substr(2);
			else return 0;
			char *end = nullptr; const long x = strtol(v.c_str(), &end, 10);
			if (v.empty() || *end) return -1;
			dst = (int)x; return 1;
		};
		if (a == "-h" || a == "--help") { fputs(USAGE, stdout); return 0; }
		if (a == "--version") { puts("indelope 0.0.1"); return 0; }
		if (a == "-g" || a == "--gpu-decode" || a == "--gpu-sweep") { o.gpu_decode = true; continue; }
		auto str_opt = [&](const char *s, const char *l, std::string &dst) -> int { // 0 no match, 1 consumed, -1 error
			if (a == s || a == l) { if (i + 1 >= argc) return -1; dst = argv[++i]; }
			else if (a.rfind(std::string(l) + "=", 0) == 0) dst = a.substr(strlen(l) + 1);
			else if (a.size() > 2 && a.compare(0, 2, s) == 0 && a[1] != '-') dst = a.substr(2);
			else return 0;
			return dst.empty() ? -1 : 1;
		};
		std::string one;
		int sr;
		if ((sr = str_opt("-r", "--region", one))) { if (sr < 0) { fputs(USAGE, stderr); return 1; } o.regions.push_back(one); continue; }
		if ((sr = str_opt("-R", "--regions-file", o.bed))) { if (sr < 0) { fputs(USAGE, stderr); return 1; } continue; }
		int rc;
		if ((rc = int_opt("-m", "--min-reads", o.min_reads)) || (rc = int_opt("-c", "--min-contig-len", o.min_ctg_len)) ||
		    (rc = int_opt("-e", "--min-event-len", o.min_event_len)) || (rc = int_opt("-t", "--threads", o.threads)) || (rc = int_opt("-d", "--device", o.device))) {
			if (rc < 0) { fputs(USAGE, stderr); return 1; }
			continue;
		}
		if (a.size() > 1 && a[0] == '-') { fputs(USAGE, stderr); return 1; }
		pos.push_back(a);
	}
	if (pos.size() != 2) { fputs(USAGE, stderr); return 1; }
	o.fa = pos[0]; o.bam = pos[1];

	if (!o.regions.empty() || !o.bed.empty()) return run_sliced(o);   // with or without -g
	if (!o.gpu_decode) return run_streamed(o);
	// the whole file on the device when it fits (the file and ~5x its size: inflated stream + record arrays), else target by target through the index
	bool by_target = getenv("INDELOPE_BY_TARGET") != nullptr;
	if (!by_target) {
		size_t free_b = 0, total_b = 0;
		const int64_t n = file_size(o.bam);
		by_target = n > 0 && idl_device_memory(o.device, &free_b, &total_b) == IDL_OK && (size_t)n > free_b / 8;
	}
	return by_target ? run_sliced(o) : run_whole_file(o);
}
