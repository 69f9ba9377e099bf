## integration/indelope_cuda.nim -- Nim bindings of libindelope_cuda.so (include/indelope_cuda.h, IDL_ABI_VERSION 2).
##
## UNVERIFIED: written against the header field by field, but never compiled -- this build image has no Nim toolchain
## (nim, nimble, hts-nim, htslib are absent and there is no network).  `when isMainModule` below checks the struct sizes the
## C side static_asserts, so a first `nim c -r integration/indelope_cuda.nim` on a box with Nim tells whether the layouts agree.
##
## The library replaces the body of `callsemble` (src/indelope.nim:201-428) between "region + reads + reference window in"
## and "per-event integer records out", and -- optionally -- `gen_roi` (src/indelope.nim:515-545) through idl_sweep.
## It owns all pinned memory; Nim never hands GC memory to CUDA.  Every call returns 0 or a negative idl_status.

const libname = "libindelope_cuda.so"

type
  IdlParams* {.bycopy.} = object           ## idl_params: 26 x int32, 2 x uint32
    abi_version*, min_reads*, min_ctg_len*, min_event_len*, asm_min_mapq*, combine_min_support*,
      combine_min_overlap*, max_contigs*, stop_min_mapq*, window_pad*, match*, mismatch*,
      a_gapo*, a_gape*, a_bw*, a_zdrop*, b_gapo*, b_gape*, b_bw*, b_zdrop*, max_events*, count_min_mapq*,
      max_contig_len*, max_read_len*, max_reads_per_region*, n_streams*: int32
    stages*, out_flags*: uint32

  IdlRegion* {.bycopy.} = object           ## 48 bytes
    chrom_id*, roi_start*, roi_end*: int32
    read_begin*, n_reads*: uint32
    ref_start*: int32
    ref_off*, ref_len*: uint32
    max_stop*: int32
    ordinal*: uint32
    flags*: uint32                         ## IDL_RF_ALPHABET = 1, IDL_RF_READ_TOO_LONG = 2
    reserved*: uint32

  IdlRead* {.bycopy.} = object             ## 24 bytes
    start*, stop*: int32
    seq_off*: uint32
    len*, trim_a*, trim_len*, min_overlap*: uint16
    mapq*, flags*: uint8
    reserved*: uint16

  IdlBatch* {.bycopy.} = object
    cap_regions*, cap_reads*, cap_seq_bases*, cap_ref_bases*: csize_t
    n_regions*, n_reads*, n_seq_bases*, n_ref_bases*: csize_t
    region*: ptr UncheckedArray[IdlRegion]
    read*: ptr UncheckedArray[IdlRead]
    seq2*, seqn*, ref2*, refn*: ptr UncheckedArray[uint32]
    impl*: pointer
    summary_valid*, max_trim_len*, max_ref_len*, max_region_reads*: uint32
    n_small_regions*: csize_t

  IdlRegionResult* {.bycopy.} = object     ## 16 bytes
    status*: uint32
    n_contigs_pre*, n_contigs*: int32
    contig_begin*: uint32

  IdlContigResult* {.bycopy.} = object     ## 24 bytes
    start*, nreads*, len*: int32
    seq_off*: uint32
    aln*: int32
    region*: uint32

  IdlAlnResult* {.bycopy.} = object        ## 72 bytes
    region*, contig*: uint32
    ref_len*: int32
    max*, zdropped*, max_q*, max_t*, mqe*, mqe_t*, mte*, mte_q*, score*: int32
    n_cigar*, n_cigar_trunc*: int32
    cigar_off*: uint32
    n_events*: int32
    event_begin*: uint32
    status*: uint32

  IdlEventResult* {.bycopy.} = object      ## 128 bytes
    aln*: uint32
    index*, typ*, t_start*, t_stop*, q_start*, q_stop*, len*, reject*, tstart*, qstart*, offset*, min_flank*,
      k_ref*, k_alt*, k_both*, aligned*, ref_support*, alt_support*, both_found*, n_adist*, n_rdist*: int32
    sum_adist*, sum_rdist*: int64
    amq_median*, rmq_median*: int32
    ref_code*, alt_code*: uint64

  IdlResults* {.bycopy.} = object
    n_regions*, n_contigs*, n_alns*, n_events*, n_cigar_ops*, n_contig_bases*: csize_t
    region*: ptr UncheckedArray[IdlRegionResult]
    contig*: ptr UncheckedArray[IdlContigResult]
    aln*: ptr UncheckedArray[IdlAlnResult]
    event*: ptr UncheckedArray[IdlEventResult]
    cigar*: ptr UncheckedArray[uint32]
    contig_seq*: ptr UncheckedArray[char]
    contig_support*: ptr UncheckedArray[uint32]
    ms_h2d*, ms_assemble*, ms_align*, ms_genotype*, ms_al*, ms_d2h*, ms_total*: cfloat
    offsets_tested*, dp_cells_a*, dp_cells_b*, dp_a*, dp_b*, kmer_reads*, kmer_bytes*, al_events*: uint64
    kernel_launches*, pool_retries*: uint32

  IdlSweepIn* {.bycopy.} = object
    chrom_len*: int32
    n_reads*: csize_t
    start*, stop*: ptr UncheckedArray[int32]
    flag*: ptr UncheckedArray[uint16]
    cigar*: ptr UncheckedArray[uint32]
    cig_off*: ptr UncheckedArray[uint64]

  IdlSweepOut* {.bycopy.} = object
    n_rois*: csize_t
    roi_start*, roi_end*: ptr UncheckedArray[int32]
    roi_read_begin*: ptr UncheckedArray[int64]
    roi_n_reads*: ptr UncheckedArray[int32]
    n_read_idx*: csize_t
    read_idx*: ptr UncheckedArray[int64]
    n_runs*, n_evidence*: csize_t
    evidence*: ptr UncheckedArray[uint8]
    ms_h2d*, ms_kernels*, ms_d2h*: cfloat
    algorithmic_bytes*, streamed_bytes*: uint64

  IdlCtx* = pointer
  IdlBam* = pointer                        ## a BAM decoded into device memory (idl_bam_open)

  IdlBamInfo* {.bycopy.} = object          ## idl_bam_info
    file_bytes*, inflated_bytes*: uint64
    n_members*, boundary_fixups*: uint32
    n_ref*: int32
    ref_name*: cstringArray
    ref_len*: ptr UncheckedArray[int64]
    header_text*: cstring
    header_len*: csize_t
    n_records*, n_unplaced*: int64
    ref_first*: ptr UncheckedArray[int64]  ## n_ref + 1: records of target c are [ref_first[c], ref_first[c + 1])
    ms_h2d*, ms_inflate*, ms_parse*: cfloat
    n_chunks*: uint32

  IdlFasta* = pointer                      ## a bgzipped FASTA parsed into device memory (idl_fasta_open)

  IdlFastaInfo* {.bycopy.} = object        ## idl_fasta_info
    file_bytes*, inflated_bytes*, sequence_bytes*: uint64
    n_members*, n_chunks*: uint32
    n_records*: int64
    name*: cstringArray
    len*: ptr UncheckedArray[int64]
    ms_h2d*, ms_inflate*, ms_parse*: cfloat
    parse_algorithmic_bytes*, parse_streamed_bytes*: uint64

  IdlBamSlice* {.bycopy.} = object         ## idl_bam_slice: a run of BGZF members holding one target's records (found through the .bai)
    n_ref*: int32
    ref_name*: cstringArray
    ref_len*: ptr UncheckedArray[int64]
    first_record*, end_member*, end_offset*: uint64

  IdlBamReads* {.bycopy.} = object         ## idl_bam_reads: what callsemble reads of a cached Record (src/indelope.nim:216-222)
    n*: csize_t
    chrom*, start*, stop*, len*: ptr UncheckedArray[int32]
    mapq*: ptr UncheckedArray[uint8]
    flag*: ptr UncheckedArray[uint16]
    seq_off*: ptr UncheckedArray[int64]
    bases*, quals*: ptr UncheckedArray[uint8]
    cig_off*: ptr UncheckedArray[uint64]
    cigar*: ptr UncheckedArray[uint32]
    ms_kernels*, ms_d2h*: cfloat

const
  IDL_ABI_VERSION* = 2'i32
  IDL_OK* = 0
  IDL_E_NO_DEVICE* = -1
  IDL_E_CAPACITY* = -5
  IDL_E_BUSY* = -7
  IDL_E_FORMAT* = -8
  IDL_BAM_SEQ* = 1'u32
  IDL_BAM_CIGAR* = 2'u32
  IDL_RS_FATAL* = 1'u32 or 2'u32 or 16'u32 or 64'u32
  IDL_RS_ALPHABET* = 32'u32
  IDL_EV_COUNTED* = 0'i32
  IDL_NO_EVENTS* = 0xffffffff'u32
  IDL_KMER* = 27

{.push cdecl, dynlib: libname.}
proc idl_default_params*(p: ptr IdlParams) {.importc.}
proc idl_create*(device: cint, p: ptr IdlParams, ctx: ptr IdlCtx): cint {.importc.}
proc idl_destroy*(ctx: IdlCtx) {.importc.}
proc idl_batch_alloc*(ctx: IdlCtx, max_regions, max_reads, max_seq_bases, max_ref_bases: csize_t, b: ptr ptr IdlBatch): cint {.importc.}
proc idl_batch_free*(ctx: IdlCtx, b: ptr IdlBatch) {.importc.}
proc idl_submit*(ctx: IdlCtx, b: ptr IdlBatch, ticket: ptr uint64): cint {.importc.}
proc idl_wait*(ctx: IdlCtx, ticket: uint64, res: ptr ptr IdlResults): cint {.importc.}
proc idl_release*(ctx: IdlCtx, ticket: uint64): cint {.importc.}
proc idl_strerror*(status: cint): cstring {.importc.}
proc idl_last_cuda_error*(ctx: IdlCtx): cstring {.importc.}
proc idl_device_count*(): cint {.importc.}
proc idl_sweep*(device: cint, inp: ptr IdlSweepIn, min_event_support, min_read_coverage, max_read_coverage: int32, flags: uint32,
                outp: ptr ptr IdlSweepOut): cint {.importc.}
proc idl_sweep_free*(o: ptr IdlSweepOut) {.importc.}
# the BAM on the device: replaces hts-nim's open / querys / Record accessors for the sweep (src/indelope.nim:595, :527, :40-47, :430-452)
proc idl_bam_open*(device: cint, file: ptr uint8, file_len: csize_t, bam: ptr IdlBam, err: cstring, errlen: csize_t): cint {.importc.}
proc idl_bam_open_slice*(device: cint, members: ptr uint8, len: csize_t, slice: ptr IdlBamSlice, bam: ptr IdlBam, err: cstring, errlen: csize_t): cint {.importc.}
proc idl_device_memory*(device: cint, free_bytes, total_bytes: ptr csize_t): cint {.importc.}
proc idl_bam_get_info*(bam: IdlBam): ptr IdlBamInfo {.importc.}
proc idl_bam_close*(bam: IdlBam) {.importc.}
proc idl_bam_sweep*(bam: IdlBam, target: int32, min_event_support, min_read_coverage, max_read_coverage: int32, flags: uint32,
                    outp: ptr ptr IdlSweepOut): cint {.importc.}
proc idl_bam_fetch*(bam: IdlBam, n: csize_t, idx: ptr int64, what: uint32, outp: ptr ptr IdlBamReads): cint {.importc.}
proc idl_bam_reads_free*(r: ptr IdlBamReads) {.importc.}
proc idl_bam_set_reference*(bam: IdlBam, target: int32, sequence: ptr uint8, len: int64): cint {.importc.}
proc idl_bam_submit*(ctx: IdlCtx, bam: IdlBam, n_regions: csize_t, roi_chrom, roi_start, roi_end, roi_n_reads: ptr int32, read_idx: ptr int64,
                     ordinal_base: uint32, ticket: ptr uint64): cint {.importc.}
proc idl_bam_pack*(ctx: IdlCtx, bam: IdlBam, n_regions: csize_t, roi_chrom, roi_start, roi_end, roi_n_reads: ptr int32, read_idx: ptr int64,
                   ordinal_base: uint32, b: ptr IdlBatch): cint {.importc.}
# a bgzip-compressed reference on the device (ref.fa.gz, what open_fai reads through htslib, src/indelope.nim:593)
proc idl_fasta_open*(device: cint, file: ptr uint8, file_len: csize_t, fa: ptr IdlFasta, err: cstring, errlen: csize_t): cint {.importc.}
proc idl_fasta_get_info*(fa: IdlFasta): ptr IdlFastaInfo {.importc.}
proc idl_fasta_copy*(fa: IdlFasta, record: int64, dst: ptr uint8, dst_len: csize_t): cint {.importc.}
proc idl_fasta_close*(fa: IdlFasta) {.importc.}
proc idl_bam_set_reference_fasta*(bam: IdlBam, target: int32, fa: IdlFasta, record: int64): cint {.importc.}
{.pop.}

when isMainModule:
  # the sizes include/indelope_cuda.h and pipeline.cu static_assert
  doAssert sizeof(IdlRegion) == 48 and sizeof(IdlRead) == 24
  doAssert sizeof(IdlRegionResult) == 16 and sizeof(IdlContigResult) == 24 and sizeof(IdlAlnResult) == 72 and sizeof(IdlEventResult) == 128
  doAssert sizeof(IdlParams) == 28 * 4
  var p: IdlParams
  idl_default_params(addr p)
  doAssert p.abi_version == IDL_ABI_VERSION and p.a_bw == 50 and p.b_bw == -1
  echo "indelope_cuda.nim: layouts agree with libindelope_cuda.so; devices: ", idl_device_count()
