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
	"  <reference>     reference fasta file.\n"
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

struct Lane { idl_batch *batch = nullptr; size_t cap[4] = {0, 0, 0, 0}; };
struct Flight { idlh_rois *rois; uint64_t ticket; };

// INDELOPE_TIMING=1: wall-clock phases on stderr
static double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

static int die(const char *what, const std::string &why) { fprintf(stderr, "indelope: %s: %s\n", what, why.c_str()); return 1; }

// --gpu-decode: the whole front end on the GPU.  The file's bytes go to the device, idl_bam_open inflates the BGZF members and parses the records there,
// idl_bam_sweep runs gen_roi per target on the resident records, idl_bam_fetch returns the bases of the records a batch of regions needs.  The host reads
// the two files, packs the reads of the regions (idlh_pack) and writes the VCF: no inflate, no record parse, no sweep on the host.
static int main_gpu_decode(const std::string &fa, const std::string &bam_path, int min_reads, int min_ctg_len, int min_event_len, int device)
{
	char err[512] = {0};
	const bool timing = getenv("INDELOPE_TIMING") != nullptr;
	const double t_begin = now_s();
	idl_params P;
	idl_default_params(&P);
	P.min_reads = min_reads; P.min_ctg_len = min_ctg_len; P.min_event_len = min_event_len;
	// the BAM's bytes
	std::vector<uint8_t> file;
	{
		FILE *f = fopen(bam_path.c_str(), "rb");
		if (!f) return die("input", "cannot open " + bam_path);
		fseek(f, 0, SEEK_END); const long n = ftell(f); fseek(f, 0, SEEK_SET);
		file.resize(n > 0 ? (size_t)n : 0);
		if (n > 0 && fread(file.data(), 1, (size_t)n, f) != (size_t)n) { fclose(f); return die("input", "cannot read " + bam_path); }
		fclose(f);
	}
	const double t_read = now_s() - t_begin;
	// the device decodes the BAM and creates the calling context while this thread reads the FASTA
	idl_ctx *ctx = nullptr; idl_bam *bam = nullptr; int create_rc = IDL_OK, open_rc = IDL_OK; double t_open = 0, t_create = 0;
	char bam_err[512] = {0};
	std::thread opener([&]() {
		double t1 = now_s();
		open_rc = idl_bam_open(device, file.data(), file.size(), &bam, bam_err, sizeof bam_err);
		t_open = now_s() - t1; t1 = now_s();
		if (open_rc == IDL_OK) create_rc = idl_create(device, &P, &ctx);
		t_create = now_s() - t1;
	});
	double t1 = now_s();
	idlh_dataset *ref = idlh_load_fasta(fa.c_str(), err, sizeof err);
	const double t_fasta = now_s() - t1;
	opener.join();
	std::vector<uint8_t>().swap(file);
	int status = 0;
	if (!ref) status = die("input", err);
	else if (open_rc == IDL_E_NO_DEVICE) status = die("libindelope_cuda", std::string(idl_strerror(open_rc)) + " (this program has no CPU path; it needs a CUDA device)");
	else if (open_rc != IDL_OK) status = die("input", bam_path + ": " + (bam_err[0] ? bam_err : idl_strerror(open_rc)));
	else if (create_rc != IDL_OK) status = die("libindelope_cuda", std::string(idl_strerror(create_rc)) + " (this program has no CPU path; it needs a CUDA device)");
	double t_sweep = 0, t_fetch = 0, t_pack = 0, t_wait = 0, t_vcf = 0;
	size_t nb = 0, n_regions = 0;
	const idl_bam_info *info = bam ? idl_bam_get_info(bam) : nullptr;
	if (!status && idlh_dataset_set_targets(ref, info->n_ref, info->ref_name, info->ref_len, err, sizeof err) != 0) status = die("input", err);
	if (!status) {
		// gen_roi per target, in header order (:599-602)
		std::vector<int32_t> rc_, rs_, re_, rn_; std::vector<int64_t> idx_;
		t1 = now_s();
		for (int32_t c = 0; c < info->n_ref && !status; ++c) {
			const std::string name = info->ref_name[c];
			if (name == "hs37d5" || name.compare(0, 2, "GL") == 0) continue;   // skippable targets, :41-42
			idl_sweep_out *so = nullptr;
			const int r = idl_bam_sweep(bam, c, min_reads - 2 > 3 ? min_reads - 2 : 3, min_reads, 600, 0, &so);
			if (r != IDL_OK) { status = die("idl_bam_sweep", idl_strerror(r)); break; }
			for (size_t k = 0; k < so->n_rois; ++k) { rc_.push_back(c); rs_.push_back(so->roi_start[k]); re_.push_back(so->roi_end[k]); rn_.push_back(so->roi_n_reads[k]); }
			idx_.insert(idx_.end(), so->read_idx, so->read_idx + so->n_read_idx);
			idl_sweep_free(so);
		}
		t_sweep = now_s() - t1;
		n_regions = rs_.size();
		{
			idlh_rois *hdr = idlh_rois_from_arrays(ref, 0, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0, nullptr, nullptr, nullptr, nullptr, nullptr);
			if (!status) { char *h = idlh_vcf_header(idlh_rois_view(hdr)); fputs(h, stdout); idlh_free(h); }   // echo header % [b.contig_header, "sample"], :599
			idlh_rois_free(hdr);
		}
		idlh_vcf *writer = idlh_vcf_new();
		std::vector<Lane> lanes((size_t)(P.n_streams > 0 ? P.n_streams : 1));
		std::deque<Flight> inflight;
		auto drain = [&]() -> bool {
			const Flight f = inflight.front(); inflight.pop_front();
			const idl_results *res = nullptr;
			double t2 = now_s();
			const int r = idl_wait(ctx, f.ticket, &res);
			t_wait += now_s() - t2; t2 = now_s();
			if (r != IDL_OK) { status = die("idl_wait", std::string(idl_strerror(r)) + " " + idl_last_cuda_error(ctx)); idlh_rois_free(f.rois); return false; }
			char *txt = idlh_vcf_records(writer, idlh_rois_view(f.rois), 0, &P, res, 0, nullptr);
			fputs(txt, stdout); idlh_free(txt);
			idl_release(ctx, f.ticket);
			idlh_rois_free(f.rois);
			t_vcf += now_s() - t2;
			return true;
		};
		// batches of regions in emission order (the dedup of :604-608 depends on it).  Default: the batch is BUILT ON THE DEVICE from the resident
		// records and reference (idl_bam_submit) -- nothing but the regions' coordinates and record indices crosses the bus.  INDELOPE_HOST_PACK=1:
		// the records of a batch are fetched (idl_bam_fetch) and packed on the host (idlh_pack), as the streamed path does.
		const bool host_pack = getenv("INDELOPE_HOST_PACK") != nullptr;
		if (!host_pack) {
			std::vector<char> has(info->n_ref > 0 ? (size_t)info->n_ref : 0, 0);
			for (int32_t c : rc_) has[(size_t)c] = 1;
			const idlh_roiset *all = nullptr;
			idlh_rois *seqs = idlh_rois_from_arrays(ref, 0, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0, nullptr, nullptr, nullptr, nullptr, nullptr);
			all = idlh_rois_view(seqs);
			double t2 = now_s();
			for (int32_t c = 0; c < info->n_ref && !status; ++c)
				if (has[(size_t)c] && idl_bam_set_reference(bam, c, all->chrom_seq[c], all->chrom_len[c]) != IDL_OK) status = die("idl_bam_set_reference", "could not place the reference on the device");
			t_fetch += now_s() - t2;
			idlh_rois_free(seqs);
		}
		size_t at_idx = 0;
		std::vector<int64_t> uniq, local;
		for (size_t lo = 0; lo < n_regions && !status; ) {
			size_t hi = lo; int64_t reads = 0;
			while (hi < n_regions && (hi == lo || (reads + rn_[hi] <= 400000 && hi - lo < 20000))) reads += rn_[hi++];
			double t2 = now_s();
			idlh_rois *grp = nullptr;
			if (host_pack) {
				uniq.assign(idx_.begin() + (long)at_idx, idx_.begin() + (long)(at_idx + (size_t)reads));
				std::sort(uniq.begin(), uniq.end()); uniq.erase(std::unique(uniq.begin(), uniq.end()), uniq.end());
				local.resize((size_t)reads);
				for (int64_t k = 0; k < reads; ++k) local[(size_t)k] = std::lower_bound(uniq.begin(), uniq.end(), idx_[at_idx + (size_t)k]) - uniq.begin();
				idl_bam_reads *rd = nullptr;
				const int fr = idl_bam_fetch(bam, uniq.size(), uniq.data(), IDL_BAM_SEQ, &rd);
				if (fr != IDL_OK) { status = die("idl_bam_fetch", idl_strerror(fr)); break; }
				grp = idlh_rois_from_arrays(ref, (int64_t)rd->n, rd->start, rd->stop, rd->len, rd->mapq, rd->flag, rd->seq_off, rd->bases, rd->quals, (int64_t)(hi - lo),
				                            rc_.data() + lo, rs_.data() + lo, re_.data() + lo, rn_.data() + lo, local.data());
				idl_bam_reads_free(rd);
			} else {
				// the VCF stage reads only the regions' coordinates and the reference of this group
				grp = idlh_rois_from_arrays(ref, 0, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, (int64_t)(hi - lo),
				                            rc_.data() + lo, rs_.data() + lo, re_.data() + lo, rn_.data() + lo, idx_.data() + at_idx);
			}
			t_fetch += now_s() - t2;
			const idlh_roiset *rs = idlh_rois_view(grp);
			if (inflight.size() >= lanes.size() && !drain()) { idlh_rois_free(grp); break; }
			t2 = now_s();
			uint64_t ticket = 0;
			if (host_pack) {
				Lane &L = lanes[nb % lanes.size()];
				size_t need[4] = {(size_t)rs->n_rois, 0, 0, 0};
				idlh_pack_size(rs, 0, rs->n_rois, &P, &need[1], &need[2], &need[3]);
				bool grow = L.batch == nullptr;
				for (int k = 0; k < 4; ++k) grow |= need[k] > L.cap[k];
				if (grow) {
					if (L.batch) idl_batch_free(ctx, L.batch);
					for (int k = 0; k < 4; ++k) L.cap[k] = need[k] + need[k] / 4 + 64;
					if (idl_batch_alloc(ctx, L.cap[0], L.cap[1], L.cap[2], L.cap[3], &L.batch) != IDL_OK) { status = die("idl_batch_alloc", "out of pinned memory"); idlh_rois_free(grp); break; }
				}
				if (idlh_pack(rs, 0, rs->n_rois, &P, L.batch) != 0) { status = die("idlh_pack", "the pinned batch is smaller than idlh_pack_size reported (internal error)"); idlh_rois_free(grp); break; }
				const int r = idl_submit(ctx, L.batch, &ticket);
				if (r != IDL_OK) { status = die("idl_submit", std::string(idl_strerror(r)) + " " + idl_last_cuda_error(ctx)); idlh_rois_free(grp); break; }
			} else {
				const int r = idl_bam_submit(ctx, bam, hi - lo, rc_.data() + lo, rs_.data() + lo, re_.data() + lo, rn_.data() + lo, idx_.data() + at_idx, (uint32_t)lo, &ticket);
				if (r != IDL_OK) { status = die("idl_bam_submit", std::string(idl_strerror(r)) + " " + idl_last_cuda_error(ctx)); idlh_rois_free(grp); break; }
			}
			inflight.push_back({grp, ticket});
			t_pack += now_s() - t2;
			at_idx += (size_t)reads; lo = hi; ++nb;
		}
		while (!inflight.empty() && !status) if (!drain()) break;
		while (!inflight.empty()) { idlh_rois_free(inflight.front().rois); inflight.pop_front(); }
		for (Lane &L : lanes) if (L.batch) idl_batch_free(ctx, L.batch);
		idlh_vcf_free(writer);
	}
	if (timing && info)
		fprintf(stderr, "indelope timing (gpu decode): read file %.3f s, fasta %.3f s, idl_bam_open %.3f s (h2d %.1f ms, inflate %.1f ms, parse %.1f ms; %.1f MB -> %.1f MB, "
		        "%lld records, %u boundary fixups), idl_create %.3f s, idl_bam_sweep %.3f s, reference / fetch %.3f s, build+submit %.3f s, idl_wait %.3f s, vcf %.3f s, total %.3f s, "
		        "batches %zu, regions %zu\n", t_read, t_fasta, t_open, info->ms_h2d, info->ms_inflate, info->ms_parse, info->file_bytes / 1e6, info->inflated_bytes / 1e6,
		        (long long)info->n_records, info->boundary_fixups, t_create, t_sweep, t_fetch, t_pack, t_wait, t_vcf, now_s() - t_begin, nb, n_regions);
	if (bam) idl_bam_close(bam);
	if (ctx) idl_destroy(ctx);
	if (ref) idlh_dataset_free(ref);
	return status;
}

// regions [first, n_rois) of one sweep of a decoded slice (targets in header order, regions in gen_roi's order) through idl_bam_submit in batches, two in
// flight, and their records on stdout; n_regions_before is the number of regions of the run emitted before these (the ordinals run on)
static int call_swept(idl_ctx *ctx, idl_bam *bam, int32_t c, const idl_sweep_out *sw, size_t first, const idlh_dataset *ref, const idlh_roiset *all, const idl_params &P,
                      idlh_vcf *writer, size_t n_regions_before)
{
	idl_sweep_out view = *sw, *so = &view;
	view.n_rois -= first; view.roi_start += first; view.roi_end += first; view.roi_n_reads += first; view.read_idx += first < sw->n_rois ? sw->roi_read_begin[first] : 0;
	int status = 0;
	if (so->n_rois && idl_bam_set_reference(bam, c, all->chrom_seq[c], all->chrom_len[c]) != IDL_OK) status = die("idl_bam_set_reference", "could not place the reference on the device");
	std::vector<int32_t> chrom(so->n_rois, c);
	std::deque<Flight> inflight;
	auto drain = [&]() -> bool {
		const Flight fl = inflight.front(); inflight.pop_front();
		const idl_results *res = nullptr;
		const int w = idl_wait(ctx, fl.ticket, &res);
		if (w != IDL_OK) { status = die("idl_wait", std::string(idl_strerror(w)) + " " + idl_last_cuda_error(ctx)); idlh_rois_free(fl.rois); return false; }
		char *txt = idlh_vcf_records(writer, idlh_rois_view(fl.rois), 0, &P, res, 0, nullptr);
		fputs(txt, stdout); idlh_free(txt);
		idl_release(ctx, fl.ticket); idlh_rois_free(fl.rois);
		return true;
	};
	size_t at_idx = 0;
	for (size_t lo = 0; lo < so->n_rois && !status; ) {
		size_t hi = lo; int64_t reads = 0;
		while (hi < so->n_rois && (hi == lo || (reads + so->roi_n_reads[hi] <= 400000 && hi - lo < 20000))) reads += so->roi_n_reads[hi++];
		idlh_rois *grp = idlh_rois_from_arrays(ref, 0, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, (int64_t)(hi - lo), chrom.data() + lo,
		                                       so->roi_start + lo, so->roi_end + lo, so->roi_n_reads + lo, so->read_idx + at_idx);
		if (inflight.size() >= (size_t)(P.n_streams > 0 ? P.n_streams : 1) && !drain()) { idlh_rois_free(grp); break; }
		uint64_t ticket = 0;
		const int r = idl_bam_submit(ctx, bam, hi - lo, chrom.data() + lo, so->roi_start + lo, so->roi_end + lo, so->roi_n_reads + lo, so->read_idx + at_idx,
		                             (uint32_t)(n_regions_before + lo), &ticket);
		if (r != IDL_OK) { status = die("idl_bam_submit", std::string(idl_strerror(r)) + " " + idl_last_cuda_error(ctx)); idlh_rois_free(grp); break; }
		inflight.push_back({grp, ticket});
		at_idx += (size_t)reads; lo = hi;
	}
	while (!inflight.empty() && !status) if (!drain()) break;
	while (!inflight.empty()) { idlh_rois_free(inflight.front().rois); inflight.pop_front(); }
	return status;
}

// --gpu-decode for a file that does not fit in device memory as a whole (or with INDELOPE_BY_TARGET=1): target by target.  For every target the index
// <bam>.bai says which run of BGZF members holds its records; that run is read, decoded on the device (idl_bam_open_slice), swept, called and dropped.
// Regions keep gen_roi's order (targets in header order), so the dedup state carries over from target to target as in the reference's single loop.
static int main_gpu_by_target(const std::string &fa, const std::string &bam_path, int min_reads, int min_ctg_len, int min_event_len, int device)
{
	char err[512] = {0};
	const bool timing = getenv("INDELOPE_TIMING") != nullptr;
	const double t_begin = now_s();
	idl_params P;
	idl_default_params(&P);
	P.min_reads = min_reads; P.min_ctg_len = min_ctg_len; P.min_event_len = min_event_len;
	idl_ctx *ctx = nullptr; int create_rc = IDL_OK;
	std::thread creator([&]() { create_rc = idl_create(device, &P, &ctx); });
	idlh_dataset *ref = idlh_load_targets(fa.c_str(), bam_path.c_str(), err, sizeof err);
	creator.join();
	if (!ref) { if (ctx) idl_destroy(ctx); return die("input", err); }
	if (create_rc != IDL_OK) { idlh_dataset_free(ref); return die("libindelope_cuda", std::string(idl_strerror(create_rc)) + " (this program has no CPU path; it needs a CUDA device)"); }
	idlh_rois *seqs = idlh_rois_from_arrays(ref, 0, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0, nullptr, nullptr, nullptr, nullptr, nullptr);
	const idlh_roiset *all = idlh_rois_view(seqs);
	{ char *h = idlh_vcf_header(all); fputs(h, stdout); idlh_free(h); }   // echo header % [b.contig_header, "sample"], :599
	std::vector<const char*> names((size_t)all->n_chroms); std::vector<int64_t> lens((size_t)all->n_chroms);
	for (int32_t c = 0; c < all->n_chroms; ++c) { names[(size_t)c] = all->chrom_name[c]; lens[(size_t)c] = all->chrom_len[c]; }
	int status = 0;
	idlh_vcf *writer = idlh_vcf_new();
	double t_read = 0, t_open = 0, t_sweep = 0, t_call = 0; size_t n_regions = 0, n_targets = 0; uint64_t bytes = 0;
	// the targets that have records, and a reader one target ahead: while the device decodes and calls target k, a thread reads the run of members of
	// target k + 1 from the file
	struct Run { int32_t c = -1; uint64_t first = 0, em = 0, eo = 0; std::vector<uint8_t> bytes; std::string error; double seconds = 0; };
	std::vector<int32_t> todo;
	for (int32_t c = 0; c < all->n_chroms; ++c) {
		const std::string name = names[(size_t)c];
		if (name == "hs37d5" || name.compare(0, 2, "GL") == 0) continue;   // skippable targets, :41-42
		todo.push_back(c);
	}
	auto load = [&](int32_t c, Run *R) {
		const double t1 = now_s();
		char e2[512] = {0};
		uint64_t fb = 0, fe = 0;
		R->c = c; R->bytes.clear(); R->error.clear();
		const int sr = idlh_bai_target_span(bam_path.c_str(), c, &fb, &fe, &R->first, &R->em, &R->eo, e2, sizeof e2);
		if (sr < 0) { R->error = e2; return; }
		if (sr == 1) { R->c = -2; return; }   // no record on this target
		FILE *f = fopen(bam_path.c_str(), "rb");
		if (!f) { R->error = "cannot open " + bam_path; return; }
		R->bytes.resize((size_t)(fe - fb));
		if (fseek(f, (long)fb, SEEK_SET) != 0 || fread(R->bytes.data(), 1, R->bytes.size(), f) != R->bytes.size()) R->error = "cannot read " + bam_path;
		fclose(f);
		R->seconds = now_s() - t1;
	};
	Run runs[2]; std::thread reader;
	if (!todo.empty()) reader = std::thread(load, todo[0], &runs[0]);
	for (size_t ti = 0; ti < todo.size() && !status; ++ti) {
		const int32_t c = todo[ti];
		const std::string name = names[(size_t)c];
		double t1 = now_s();
		reader.join();                                   // the run of this target
		Run &R = runs[ti & 1];
		if (ti + 1 < todo.size()) reader = std::thread(load, todo[ti + 1], &runs[(ti + 1) & 1]);
		t_read += now_s() - t1;                          // (what the call waited for the reader)
		if (!R.error.empty()) { status = die("input", R.error); break; }
		if (R.c == -2) continue;
		t1 = now_s(); bytes += R.bytes.size();
		const std::vector<uint8_t> &run = R.bytes;
		const uint64_t first = R.first, em = R.em, eo = R.eo;
		idl_bam_slice sl; memset(&sl, 0, sizeof sl);
		sl.n_ref = all->n_chroms; sl.ref_name = names.data(); sl.ref_len = lens.data(); sl.first_record = first; sl.end_member = em; sl.end_offset = eo;
		idl_bam *bam = nullptr; char berr[512] = {0};
		const int orc = idl_bam_open_slice(device, run.data(), run.size(), &sl, &bam, berr, sizeof berr);
		if (orc != IDL_OK) { status = die("input", bam_path + " (" + name + "): " + (berr[0] ? berr : idl_strerror(orc))); break; }
		t_open += now_s() - t1; t1 = now_s();
		idl_sweep_out *so = nullptr;
		int r = idl_bam_sweep(bam, c, min_reads - 2 > 3 ? min_reads - 2 : 3, min_reads, 600, 0, &so);
		if (r != IDL_OK) { status = die("idl_bam_sweep", idl_strerror(r)); idl_bam_close(bam); break; }
		t_sweep += now_s() - t1; t1 = now_s();
		++n_targets;
		status = call_swept(ctx, bam, c, so, 0, ref, all, P, writer, n_regions);
		n_regions += so->n_rois;
		idl_sweep_free(so);
		idl_bam_close(bam);
		t_call += now_s() - t1;
	}
	if (reader.joinable()) reader.join();
	if (timing)
		fprintf(stderr, "indelope timing (gpu decode, target by target): %zu targets with records, %.1f MB read (a reader thread one target ahead; waited %.3f s for it), idl_bam_open_slice %.3f s, idl_bam_sweep %.3f s, "
		        "build + call + vcf %.3f s, total %.3f s, regions %zu\n", n_targets, bytes / 1e6, t_read, t_open, t_sweep, t_call, now_s() - t_begin, n_regions);
	idlh_vcf_free(writer);
	idlh_rois_free(seqs);
	idl_destroy(ctx);
	idlh_dataset_free(ref);
	return status;
}

// -r / -R: only the regions of interest that overlap the given intervals, decoding only the BAM members that hold them.  Per target the intervals become
// slices of the file: from the linear-index offset of the 16 kb window in front of an interval to that of the window behind it (idlh_bai_region_run);
// slices whose member runs overlap or touch are merged and decoded once.  Each slice is decoded (idl_bam_open_slice) and swept over the zone of positions
// whose evidence it determines exactly (idl_bam_sweep_window, DESIGN.md 4a); when a selected region touches an inner edge of the zone, or the zone does not
// reach the last interval, the slice grows by one window on that side and is swept again.  A reader thread reads the next slice's members meanwhile.
static int main_regions(const std::string &fa, const std::string &bam_path, const std::vector<std::string> &regions, const std::string &bed, int min_reads,
                        int min_ctg_len, int min_event_len, int device)
{
	char err[512] = {0};
	const bool timing = getenv("INDELOPE_TIMING") != nullptr;
	const double t_begin = now_s();
	idl_params P;
	idl_default_params(&P);
	P.min_reads = min_reads; P.min_ctg_len = min_ctg_len; P.min_event_len = min_event_len;
	const int32_t min_ev = min_reads - 2 > 3 ? min_reads - 2 : 3;
	idlh_dataset *ref = idlh_load_targets(fa.c_str(), bam_path.c_str(), err, sizeof err);
	if (!ref) return die("input", err);
	idlh_rois *seqs = idlh_rois_from_arrays(ref, 0, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0, nullptr, nullptr, nullptr, nullptr, nullptr);
	const idlh_roiset *all = idlh_rois_view(seqs);
	std::vector<const char*> names((size_t)all->n_chroms); std::vector<int64_t> lens((size_t)all->n_chroms);
	for (int32_t c = 0; c < all->n_chroms; ++c) { names[(size_t)c] = all->chrom_name[c]; lens[(size_t)c] = all->chrom_len[c]; }
	std::vector<const char*> rv; for (const std::string &r : regions) rv.push_back(r.c_str());
	idlh_regions *sel = idlh_regions_parse(all->n_chroms, names.data(), lens.data(), (int32_t)rv.size(), rv.data(), bed.empty() ? nullptr : bed.c_str(), err, sizeof err);
	auto cleanup = [&]() { idlh_regions_free(sel); idlh_rois_free(seqs); idlh_dataset_free(ref); };
	if (!sel) { cleanup(); return die("regions", err); }
	{   // the index must be there before anything is printed
		uint64_t v[5];
		if (all->n_chroms > 0 && idlh_bai_target_span(bam_path.c_str(), 0, v, v + 1, v + 2, v + 3, v + 4, err, sizeof err) < 0) { cleanup(); return die("input", bam_path + ": " + err); }
	}
	idl_ctx *ctx = nullptr;
	const int create_rc = idl_create(device, &P, &ctx);
	if (create_rc != IDL_OK) { cleanup(); return die("libindelope_cuda", std::string(idl_strerror(create_rc)) + " (this program has no CPU path; it needs a CUDA device)"); }
	{ char *h = idlh_vcf_header(all); fputs(h, stdout); idlh_free(h); }   // echo header % [b.contig_header, "sample"], :599
	int status = 0;
	idlh_vcf *writer = idlh_vcf_new();
	size_t n_regions = 0, n_slices = 0, n_retries = 0, n_intervals = 0; uint64_t bytes_read = 0, bytes_decoded = 0;
	double t_read = 0, t_open = 0, t_sweep = 0, t_call = 0;
	// one slice: window range [w0, w1], its intervals, where its members lie
	struct Slice { int64_t w0 = 0, w1 = 0; std::vector<int32_t> beg, end; uint64_t fb = 0, fe = 0, first = 0, em = 0, eo = 0; int64_t zone_lo = 0; int32_t to_end = 1; int rr = 1; };
	struct Read { uint64_t fb = 0, fe = 0; std::vector<uint8_t> bytes; std::string error; };
	auto locate = [&](int32_t c, Slice &S) -> bool {
		S.rr = idlh_bai_region_run(bam_path.c_str(), c, S.w0, S.w1, &S.fb, &S.fe, &S.first, &S.em, &S.eo, &S.zone_lo, &S.to_end, err, sizeof err);
		if (S.rr < 0) { status = die("input", bam_path + ": " + err); return false; }
		return true;
	};
	auto load = [&](uint64_t fb, uint64_t fe, Read *R) {
		R->fb = fb; R->fe = fe; R->error.clear(); R->bytes.resize((size_t)(fe - fb));
		FILE *f = fopen(bam_path.c_str(), "rb");
		if (!f) { R->error = "cannot open " + bam_path; return; }
		if (fseek(f, (long)fb, SEEK_SET) != 0 || fread(R->bytes.data(), 1, R->bytes.size(), f) != R->bytes.size()) R->error = "cannot read " + bam_path;
		fclose(f);
	};
	Read ahead; std::thread reader;
	std::vector<int64_t> ib, ie;
	for (int32_t c = 0; c < all->n_chroms && !status; ++c) {
		const int64_t n_iv = idlh_regions_get(sel, c, nullptr, nullptr, 0);
		if (n_iv == 0) continue;
		ib.resize((size_t)n_iv); ie.resize((size_t)n_iv);
		idlh_regions_get(sel, c, ib.data(), ie.data(), n_iv);
		n_intervals += (size_t)n_iv;
		int64_t last_end = -1;   // of the last region called on this target
		// the first slice of every interval: the window holding the position in front of it to the window behind its last base
		std::deque<Slice> todo;
		for (int64_t k = 0; k < n_iv && !status; ++k) {
			Slice S;
			S.w0 = ib[(size_t)k] > 0 ? (ib[(size_t)k] - 1) >> 14 : 0; S.w1 = ((ie[(size_t)k] - 1) >> 14) + 1;
			S.beg.push_back((int32_t)ib[(size_t)k]); S.end.push_back((int32_t)ie[(size_t)k]);
			if (!todo.empty() && S.w0 <= todo.back().w1) {   // overlapping window ranges: one slice
				Slice &B = todo.back(); B.w1 = std::max(B.w1, S.w1); B.beg.push_back(S.beg[0]); B.end.push_back(S.end[0]);
			} else todo.push_back(S);
		}
		for (Slice &S : todo) if (!locate(c, S)) break;
		while (!todo.empty() && !status) {
			Slice S = todo.front(); todo.pop_front();
			// slices whose member runs overlap or touch are decoded once
			while (!todo.empty() && S.rr == 0 && todo.front().rr == 0 && todo.front().fb <= S.fe) {
				const Slice &N = todo.front();
				S.w1 = std::max(S.w1, N.w1); S.beg.insert(S.beg.end(), N.beg.begin(), N.beg.end()); S.end.insert(S.end.end(), N.end.begin(), N.end.end());
				todo.pop_front();
				if (!locate(c, S)) break;
			}
			if (status) break;
			if (S.rr == 1) {   // no record in the run
				if (S.to_end) continue;                      // ... up to the target's end: no region
				++S.w1; ++n_retries;
				if (locate(c, S)) todo.push_front(S);
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
			sl.n_ref = all->n_chroms; sl.ref_name = names.data(); sl.ref_len = lens.data(); sl.first_record = S.first; sl.end_member = S.em; sl.end_offset = S.eo;
			idl_bam *bam = nullptr; char berr[512] = {0};
			const int orc = idl_bam_open_slice(device, R.bytes.data(), R.bytes.size(), &sl, &bam, berr, sizeof berr);
			if (orc != IDL_OK) { status = die("input", bam_path + " (" + names[(size_t)c] + "): " + (berr[0] ? berr : idl_strerror(orc))); break; }
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
				if (locate(c, S)) todo.push_front(S);
				t_sweep += now_s() - t1;
				continue;
			}
			idl_sweep_out *so = nullptr;
			const int r = idl_bam_sweep_window(bam, c, (int32_t)S.zone_lo, (int32_t)zone_hi, S.beg.size(), S.beg.data(), S.end.data(), min_ev, min_reads, 600, 0, &so);
			if (r != IDL_OK) { status = die("idl_bam_sweep_window", idl_strerror(r)); idl_bam_close(bam); break; }
			t_sweep += now_s() - t1; t1 = now_s();
			if (so->n_edge[0] || so->n_edge[1]) {   // a selected region reaches beyond the zone: grow the slice on that side
				if (so->n_edge[0]) --S.w0;
				if (so->n_edge[1]) ++S.w1;
				++n_retries;
				idl_sweep_free(so); idl_bam_close(bam);
				if (locate(c, S)) todo.push_front(S);
				continue;
			}
			// a slice grown to the left may share regions with the slice before it: those were called there
			size_t first = 0;
			while (first < so->n_rois && so->roi_start[first] <= last_end) ++first;
			status = call_swept(ctx, bam, c, so, first, ref, all, P, writer, n_regions);
			n_regions += so->n_rois - first;
			if (so->n_rois > first) last_end = so->roi_end[so->n_rois - 1];
			idl_sweep_free(so);
			idl_bam_close(bam);
			t_call += now_s() - t1;
		}
	}
	if (reader.joinable()) reader.join();
	if (timing)
		fprintf(stderr, "indelope timing (regions): %zu intervals, %.1f MB read, %.1f MB decoded, slices %zu, retries %zu, regions %zu; waited %.3f s for reads, "
		        "idl_bam_open_slice %.3f s, zone + idl_bam_sweep_window %.3f s, build + call + vcf %.3f s, total %.3f s\n", n_intervals, bytes_read / 1e6,
		        bytes_decoded / 1e6, n_slices, n_retries, n_regions, t_read, t_open, t_sweep, t_call, now_s() - t_begin);
	idlh_vcf_free(writer);
	idl_destroy(ctx);
	cleanup();
	return status;
}

int main(int argc, char **argv)
{
	int min_reads = 3, min_ctg_len = 73, min_event_len = 4, threads = 1, device = 0;
	bool gpu_sweep = false;
	std::vector<std::string> pos, regions; std::string bed;
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
		if (a == "-g" || a == "--gpu-decode" || a == "--gpu-sweep") { gpu_sweep = true; continue; }
		auto str_opt = [&](const char *s, const char *l, std::string &dst) -> int { // 0 no match, 1 consumed, -1 error
			if (a == s || a == l) { if (i + 1 >= argc) return -1; dst = argv[++i]; }
			else if (a.rfind(std::string(l) + "=", 0) == 0) dst = a.substr(strlen(l) + 1);
			else if (a.size() > 2 && a.compare(0, 2, s) == 0 && a[1] != '-') dst = a.substr(2);
			else return 0;
			return dst.empty() ? -1 : 1;
		};
		std::string one;
		int sr;
		if ((sr = str_opt("-r", "--region", one))) { if (sr < 0) { fputs(USAGE, stderr); return 1; } regions.push_back(one); continue; }
		if ((sr = str_opt("-R", "--regions-file", bed))) { if (sr < 0) { fputs(USAGE, stderr); return 1; } continue; }
		int rc;
		if ((rc = int_opt("-m", "--min-reads", min_reads)) || (rc = int_opt("-c", "--min-contig-len", min_ctg_len)) ||
		    (rc = int_opt("-e", "--min-event-len", min_event_len)) || (rc = int_opt("-t", "--threads", threads)) || (rc = int_opt("-d", "--device", device))) {
			if (rc < 0) { fputs(USAGE, stderr); return 1; }
			continue;
		}
		if (a.size() > 1 && a[0] == '-') { fputs(USAGE, stderr); return 1; }
		pos.push_back(a);
	}
	if (pos.size() != 2) { fputs(USAGE, stderr); return 1; }

	char err[512] = {0};
	const bool timing = getenv("INDELOPE_TIMING") != nullptr;
	const double t_begin = now_s(); double t_sweep = 0, t_pack = 0, t_wait = 0, t_vcf = 0, t0;
	if (!regions.empty() || !bed.empty()) return main_regions(pos[0], pos[1], regions, bed, min_reads, min_ctg_len, min_event_len, device);   // with or without -g
	if (gpu_sweep) {
		// the whole file on the device when it fits (the file and ~5x its size: inflated stream + record arrays), else target by target through the index
		bool by_target = getenv("INDELOPE_BY_TARGET") != nullptr;
		if (!by_target) {
			size_t free_b = 0, total_b = 0;
			FILE *bf = fopen(pos[1].c_str(), "rb");
			if (bf && idl_device_memory(device, &free_b, &total_b) == IDL_OK) { fseek(bf, 0, SEEK_END); const long n = ftell(bf); by_target = n > 0 && (size_t)n > free_b / 8; }
			if (bf) fclose(bf);
		}
		return by_target ? main_gpu_by_target(pos[0], pos[1], min_reads, min_ctg_len, min_event_len, device)
		                 : main_gpu_decode(pos[0], pos[1], min_reads, min_ctg_len, min_event_len, device);
	}
	// gen_roi(b, target, min_read_coverage=min_reads, min_event_support=max(3, min_reads-2)), src/indelope.nim:602; the BAM
	// is swept front to back in bounded memory (idlh_stream_*), a group of regions at a time
	idlh_stream *in = idlh_stream_open(pos[0].c_str(), pos[1].c_str(), threads, min_reads - 2 > 3 ? min_reads - 2 : 3, min_reads, 600, err, sizeof err);
	if (!in) return die("input", err);

	idl_params P;
	idl_default_params(&P);
	P.min_reads = min_reads; P.min_ctg_len = min_ctg_len; P.min_event_len = min_event_len;
	// the CUDA context and the library's workspaces come up on a helper thread while this one already reads the BAM; nothing
	// is printed before the context exists (without a device the program fails with empty stdout)
	idl_ctx *ctx = nullptr;
	int create_rc = IDL_OK, rc = IDL_OK, status = 0; double t_create = 0;
	const double t_open = now_s() - t_begin;
	std::thread creator([&]() { const double t1 = now_s(); create_rc = idl_create(device, &P, &ctx); t_create = now_s() - t1; });
	bool have_ctx = false;
	auto need_ctx = [&]() -> bool {
		if (have_ctx) return true;
		creator.join();
		if (create_rc != IDL_OK) { status = die("libindelope_cuda", std::string(idl_strerror(create_rc)) + " (this program has no CPU path; it needs a CUDA device)"); return false; }
		idlh_rois *t = idlh_stream_targets(in); // echo header % [b.contig_header, "sample"], :599
		char *h = idlh_vcf_header(idlh_rois_view(t)); fputs(h, stdout); idlh_free(h);
		idlh_rois_free(t);
		have_ctx = true;
		return true;
	};
	idlh_vcf *writer = idlh_vcf_new();
	std::vector<Lane> lanes((size_t)(P.n_streams > 0 ? P.n_streams : 1));
	std::deque<Flight> inflight;
	auto drain = [&]() -> bool {
		const Flight f = inflight.front(); inflight.pop_front();
		const idl_results *res = nullptr;
		double t1 = now_s();
		const int r = idl_wait(ctx, f.ticket, &res);
		t_wait += now_s() - t1; t1 = now_s();
		if (r != IDL_OK) { status = die("idl_wait", std::string(idl_strerror(r)) + " " + idl_last_cuda_error(ctx)); idlh_rois_free(f.rois); return false; }
		char *dump = nullptr;
		char *txt = idlh_vcf_records(writer, idlh_rois_view(f.rois), 0, &P, res, 0, &dump);
		fputs(txt, stdout);
		idlh_free(txt); idlh_free(dump);
		idl_release(ctx, f.ticket);
		idlh_rois_free(f.rois);
		t_vcf += now_s() - t1;
		return true;
	};
	// one batch per group of regions, in emission order (the dedup of :604-608 depends on it); while the GPU works on a
	// batch the host reads and sweeps the next stretch of the BAM
	const int64_t target_reads = 400000;
	size_t nb = 0;
	while (!status) {
		err[0] = 0;
		t0 = now_s();
		idlh_rois *grp = idlh_stream_next(in, target_reads, err, sizeof err);
		t_sweep += now_s() - t0;
		if (!grp) { if (err[0]) status = die("input", err); break; }
		const idlh_roiset *rs = idlh_rois_view(grp);
		if (rs->n_rois == 0) { idlh_rois_free(grp); continue; }
		if (!need_ctx()) { idlh_rois_free(grp); break; }
		if (inflight.size() >= lanes.size() && !drain()) { idlh_rois_free(grp); break; }
		Lane &L = lanes[nb % lanes.size()];
		t0 = now_s();
		size_t need[4] = {(size_t)rs->n_rois, 0, 0, 0};
		idlh_pack_size(rs, 0, rs->n_rois, &P, &need[1], &need[2], &need[3]);
		bool grow = L.batch == nullptr;
		for (int k = 0; k < 4; ++k) grow |= need[k] > L.cap[k];
		if (grow) {
			if (L.batch) idl_batch_free(ctx, L.batch);
			for (int k = 0; k < 4; ++k) L.cap[k] = need[k] + need[k] / 4 + 64;
			rc = idl_batch_alloc(ctx, L.cap[0], L.cap[1], L.cap[2], L.cap[3], &L.batch);
			if (rc != IDL_OK) { status = die("idl_batch_alloc", idl_strerror(rc)); idlh_rois_free(grp); break; }
		}
		if (idlh_pack(rs, 0, rs->n_rois, &P, L.batch) != 0) { status = die("idlh_pack", "the pinned batch is smaller than idlh_pack_size reported (internal error)"); idlh_rois_free(grp); break; }
		uint64_t ticket = 0;
		rc = idl_submit(ctx, L.batch, &ticket);
		if (rc != IDL_OK) { status = die("idl_submit", std::string(idl_strerror(rc)) + " " + idl_last_cuda_error(ctx)); idlh_rois_free(grp); break; }
		inflight.push_back({grp, ticket});
		t_pack += now_s() - t0;
		++nb;
	}
	if (!status) need_ctx(); // a BAM without any region still gets its header
	while (!inflight.empty() && !status) if (!drain()) break;
	while (!inflight.empty()) { idlh_rois_free(inflight.front().rois); inflight.pop_front(); }
	for (Lane &L : lanes) if (L.batch && ctx) idl_batch_free(ctx, L.batch);
	idlh_vcf_free(writer);
	if (creator.joinable()) creator.join();
	t0 = now_s();
	if (ctx) idl_destroy(ctx);
	idlh_stream_close(in);
	if (timing)
		fprintf(stderr, "indelope timing: open %.3f s, idl_create %.3f s, read+sweep %.3f s, pack+submit %.3f s, idl_wait %.3f s, vcf %.3f s, teardown %.3f s, total %.3f s, batches %zu\n",
		        t_open, t_create, t_sweep, t_pack, t_wait, t_vcf, now_s() - t0, now_s() - t_begin, nb);
	return status;
}
