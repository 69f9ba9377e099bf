// indelope_b200/csrc/sweep_impl.h -- inside libindelope_cuda.so: the body of idl_sweep (sweep.cu), also entered by idl_bam_sweep (bamdev.cu)
// with the records' arrays already resident on the device.
#pragma once
#include <cstddef>
#include <cstdint>
#include "indelope_cuda.h"

// dev_in: start / stop / flag / cigar / cig_off of `in` are device pointers on `device` (n_cig is then only used for the byte statistics).
// Positions zone_lo .. zone_hi are swept (0 .. chrom_len: the whole target).  n_iv < 0: every region; n_iv >= 0: only the regions that overlap one of
// the host intervals [iv_beg, iv_end) and lie strictly inside the zone's inner edges (idl_bam_sweep_window)
int idl_sweep_impl(int device, const idl_sweep_in *in, bool dev_in, size_t n_cig, int32_t zone_lo, int32_t zone_hi, long long n_iv, const int32_t *iv_beg,
                   const int32_t *iv_end, int32_t min_event_support, int32_t min_read_coverage, int32_t max_read_coverage, uint32_t flags, idl_sweep_out **out);
