// ctx.cuh -- the context behind the C-ABI (device buffers, streams, state).
#pragma once
#include <cstdio>
#include <cstdlib>
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>
#include "common.cuh"

namespace mcov {

// grow-only device / pinned buffers
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  // what ensure(bytes) allocates when it has to grow (ensure_fits checks this much against the free memory)
  static size_t grown(size_t bytes) { return bytes + bytes / 8 + 256; }
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) { cudaFree(p); p = nullptr; cap = 0; }
    size_t want = grown(bytes);
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

// a site list on the device: n records for the contig table of epoch `epoch` (n = -1: none)
struct SiteList {
  DevBuf list;
  int64_t n = -1, epoch = -1;
};

struct PinBuf {
  void* p = nullptr;
  size_t cap = 0;
  bool pageable = false;            // plain malloc instead of pinned memory (pinning costs 0.6 - 2.4 ms per MB on these boxes)
  cudaError_t ensure(size_t bytes, bool pinned = true) {
    if (bytes <= cap && pageable == !pinned) return cudaSuccess;
    release();
    size_t want = bytes + bytes / 8 + 256;
    if (pinned) {
      cudaError_t e = cudaMallocHost(&p, want);
      if (e != cudaSuccess) { p = nullptr; return e; }
    } else {
      p = std::malloc(want);
      if (!p) return cudaErrorMemoryAllocation;
    }
    cap = want; pageable = !pinned;
    return cudaSuccess;
  }
  void release() { if (p) { if (pageable) std::free(p); else cudaFreeHost(p); } p = nullptr; cap = 0; pageable = false; }
  template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

enum PassState { kIdle = 0, kAccumulating = 1, kDepthReady = 2, kStreaming = 3 };

// kernel ids for the optional per-kernel CUDA-event timing (mcov_profile_*)
enum KernelId {
  kKExpand = 0, kKScan, kKFusedPrep, kKScanCounts, kKFarScatter,
  kKWindowSums, kKIsizeHist, kKGroupCount, kKSortedStats, kKClear, kKRegionStatsSmall, kKCapReplay, kKUnpack, kKKmerHist, kKRegionStatsWarp,
  kKExpPrep, kKExpEntries, kKExpRegion, kKExpRevsum, kKRegionHist, kKHistFinish, kKRunCount, kKRunOffsets, kKRunWrite, kKRunEnds, kKBgzfInflate, kKBamGuess, kKBamWalkCount, kKBamWalkWrite, kKDeltaUnpack, kKStreamAcc, kKFusedPrepTma, kKFusedTileTma, kKStatsStream, kKBlockUnpack, kKBamNamesSeq,
  kKSamNlCount, kKSamNlWrite, kKSamFields, kKSamCigar, kKSamNamesSeq, kKMapCounts,
  kKCapExact, kKSamLineMax,
  kKBcAny,
  kKRefEncode, kKAlleleChunks, kKAlleleCombine, kKAlleleSiteCount, kKAlleleSiteWrite,
  kKAlleleSignature, kKCompareChunks, kKCompareCombine, kKCompareSiteCount, kKCompareSiteWrite,
  kKLinkSites, kKLinkObsCount, kKLinkObsWrite, kKLinkSort, kKLinkUnitCalls, kKLinkSelect, kKLinkPairs, kKLinkPairCount,
  kKLinkPairWrite,
  kKGeneChunks, kKGeneCombine, kKGeneSiteWrite,
  kKernelCount
};

struct ProfRec { int id; cudaEvent_t a, b; };

// cached task table of the last region set (mcov_region_stats_run)
struct RegionPlan {
  bool valid = false;
  int64_t g = 0, n_small = 0;
  int32_t ss_grid = 0, n_split = 0;      // balanced stream over the large regions (k_stats_stream.cuh): CTAs, split regions
  int64_t n_contigs_epoch = -1;
  int64_t id = 0;                        // distinct for every plan the context builds
  int64_t hist_tiles = 0;                // tiles that lie wholly inside a large region (their histograms spare the statistics the depth)
  std::vector<int32_t> tid, start, end, rlen, rpad;
};

struct ReadStage {            // one staging set for host-resident batches
  DevBuf tid, pos, flag, mapq, cig_off, cig;
  DevBuf raw;                       // the narrow host transports land here before they are widened into the columns
  cudaEvent_t consumed = nullptr;   // recorded after the kernel that read this set
  bool in_flight = false;
};

}  // namespace mcov

struct mcov_bam_gpu_stream_info;

namespace mcov {

// One batch of the streamed BAM decode (bam_gpu_chunks): device columns of n records, the first n_carry of them carried
// over from the previous batch (their rec_off points into bytes that are gone); data / rec_off locate the records
// [n_carry, n) in this chunk's inflated stream.
struct BamChunk {
  int64_t n, n_carry, n_ops;
  const int32_t* tid; const int32_t* pos; const uint16_t* flag; const uint8_t* mapq; const int32_t* l_seq;
  const uint32_t* cig_off; const uint32_t* cig;
  const uint8_t* data; const uint64_t* rec_off;
  bool last;
};
// A consumer of the streamed decode: begin() once the file is open, batch() for every chunk.  batch() sets how many of
// the batch's last reads (and their ops) lead the next one.
struct BamChunkSink {
  virtual int begin(mcov_ctx*) { return 0; }
  virtual int batch(mcov_ctx* ctx, const BamChunk& b, int64_t* n_carry, int64_t* carry_ops) = 0;
  virtual ~BamChunkSink() {}
};
// bam_gpu.cu: the chunk loop of mcov_bam_gpu_stream_depth; `who` prefixes the error texts
int bam_gpu_chunks(mcov_ctx* ctx, const char* path, int64_t chunk_bytes, int verify_crc, mcov_bam_gpu_stream_info* info,
                   const char* who, BamChunkSink& sink);

}  // namespace mcov

struct mcov_ctx {
  int device = 0;
  int n_sm = 0;               // multiprocessors of the device (queried in mcov_create); grids are sized from it
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  cudaStream_t copy_stream = nullptr;
  cudaStream_t d2h_stream = nullptr;   // copy-back of pipelined statistics records (overlaps the next pass)
  cudaEvent_t copied = nullptr;
  cudaStream_t unpack_stream = nullptr;   // the transport block's unpack kernel: depends on the block's copy only, so it may
  cudaEvent_t unpacked = nullptr;         // overlap the kernels of the previous pass on the main stream
  bool copy_pending = false;       // a transport block's copy has been enqueued and not yet waited for
  std::string err;

  int32_t n_contigs = 0;
  std::vector<int32_t> len;
  std::vector<int64_t> off;
  int64_t n_slots = 0;        // padded to a multiple of 4
  mcov::DevBuf d_len, d_off;

  int32_t* depth = nullptr;   // difference array, then depth
  mcov::DevBuf depth_own;
  bool depth_bound = false;

  mcov_filter filt;
  uint32_t flag_lut[128] = {0};   // the flag part of the filter as a 4096-bit table (rebuilt by mcov_set_filter)
  bool flag_lut_dirty = true;
  mcov::DevBuf d_flag_lut;        // its device copy
  int state = mcov::kIdle;

  mcov::DevBuf d_pc;          // PassCounters
  mcov::DevBuf d_status;      // scan tile status words
  mcov::ReadStage stage[2];
  int stage_next = 0;
  int64_t n_reads_pushed = 0;
  bool verdict_pending = false;   // an asynchronous fused pass has not been checked for sortedness yet
  bool exact_cap = false;         // the any-order pass counts starts for the exact cap metric (mcov_begin_ex)
  mcov::DevBuf d_starts;          // [n_slots] passing reads that start at each slot (exact_cap passes)
  int64_t contig_epoch = 0;
  mcov::RegionPlan plan;
  int32_t cap_contigs = 0;        // contigs replayed under htslib's max_depth cap in the last fused pass
  uint8_t* cap_flags = nullptr;   // device, [n_contigs]: contigs replayed in the last fused pass (inside d_status)
  std::vector<unsigned char> fused_blob;   // FusedArgs of the last fused pass (k_fused.cuh)

  // GPU-side BAM decode (bam_gpu.cu): compressed image, inflated stream, record-chain scratch, SoA columns
  struct BamDev {
    mcov::DevBuf raw, blocks, data, status, starts, segs, wout, tid, pos, flag, mapq, lseq, isize, cig_off, cig;
    mcov::DevBuf rec_off, name_hash, kmer, win;      // record offsets in `data`; read names / SEQ derived from them on request
    // streamed decode (mcov_bam_gpu_stream_depth): pinned file chunks, the bytes of the record a chunk ended in, the reads
    // carried into the next batch
    mcov::PinBuf pin[2];
    mcov::DevBuf tail, tail2, c_tid, c_pos, c_flag, c_mapq, c_off, c_cig;
    // SAM decode (sam_gpu.cu): `data` holds the text; tile newline counts, line ends, per-record field offsets, op counts,
    // the @SQ name table, CUB scratch
    mcov::DevBuf sam_tiles, sam_lines, sam_aux, sam_ops, sam_ref, sam_tmp;
    int64_t n_rec = -1;                              // records of the last decode (-1: none)
    bool sam = false;                                // the last decode read SAM text (names / SEQ come from the text)
    uint32_t sam_ref_mask = 0;                       // the @SQ table in sam_ref: slot mask, bytes of slots / name offsets, names
    size_t sam_tab_bytes = 0, sam_off_bytes = 0;
    int32_t sam_n_ref = 0;
    bool sam_chunked = false;                        // a chunked SAM decode has begun (mcov_sam_chunk_begin)
    int64_t sam_line0 = 0;                           // lines of that stream in front of the next chunk
    int64_t sam_longest = 0;                         // its longest line so far (LF included)
    void release() {
      n_rec = -1;
      sam = false;
      mcov::DevBuf* b[] = {&raw, &blocks, &data, &status, &starts, &segs, &wout, &tid, &pos, &flag, &mapq, &lseq, &isize, &cig_off, &cig,
                           &rec_off, &name_hash, &kmer, &win, &tail, &tail2, &c_tid, &c_pos, &c_flag, &c_mapq, &c_off, &c_cig,
                           &sam_tiles, &sam_lines, &sam_aux, &sam_ops, &sam_ref, &sam_tmp};
      for (mcov::DevBuf* x : b) x->release();
      pin[0].release(); pin[1].release();
    }
  } bam;

  // A / C / G / T counts of the last mcov_base_counts (basecount.cu): [n_slots][4] uint32, for (bc_qthr, bc_mode) of
  // the contig table of epoch bc_epoch; the error word.  Apart from the depth store and its caches.
  mcov::DevBuf d_bc, d_bc_word;
  bool bc_ready = false;
  int32_t bc_qthr = 0, bc_mode = 0;
  int64_t bc_epoch = -1;

  // Alleles (alleles.cu): the reference store ([n_slots] codes 0-3 A C G T, 4 unknown) of the contig table of epoch
  // ref_epoch and which contigs have been given one.  Comparisons (compare.cu): the (sample a, sample b) signature
  // pointers of each pair.
  mcov::DevBuf d_ref, d_ref_stage, d_pair_sigs;
  std::vector<uint8_t> ref_set;
  int64_t ref_epoch = -1;
  // Scratch of the allele, compare and gene region / site calls, one set for all: every such call synchronises before
  // it returns.  Regions: the chunks (AlChunk; GnChunk), the meta [first[g + 1] | length[g]] (int64; the gene call
  // adds codons[g]), a partial record per chunk,
  // the region records.  Sites: the tile counts followed by their inclusive scan (int64), the scan's temporary storage.
  mcov::DevBuf d_chunks, d_chunk_meta, d_chunk_part, d_region_out, d_site_tiles, d_site_scan;
  // the site lists of the last mcov_allele_sites and mcov_compare_sites (both stay readable)
  mcov::SiteList allele_sites, compare_sites;
  // Linkage (linkage.cu): its own SNV site list and pair list; per site the slot, contig, alleles, partner counts and
  // their scan; per record of a batch its observation count and their scan; the observations (two buffers for the
  // sort); the candidate pairs' counters; CUB scratch and the call / unit totals
  mcov::SiteList link_sites, link_pairs;
  mcov::DevBuf d_lk_slot, d_lk_tid, d_lk_allele, d_lk_partners, d_lk_base, d_lk_rec_n, d_lk_rec_off, d_lk_obs[2], d_lk_cnt,
      d_lk_tmp, d_lk_word;
  // Genes (genes.cu): the site list of the last mcov_gene_run that asked for one (its scratch is the allele calls')
  mcov::SiteList gene_sites;

  // fused (sorted) path scratch
  mcov::DevBuf d_start_slot, d_far_list, d_tile_cnt, d_tile_off, d_far_sorted;
  // per-tile depth histograms of the last one-shot fused pass (FusedArgs::tile_hist), written because of plan
  // tile_hist_plan; tile_hist_valid: they describe the depth store as it is now (cleared by every call that writes the
  // depth otherwise, and by mcov_depth_ptr, which hands the store to the caller)
  mcov::DevBuf d_tile_hist;
  bool tile_hist_valid = false;
  int64_t tile_hist_plan = 0, plan_serial = 0;

  // stats scratch
  mcov::DevBuf d_ss_pieces, d_ss_cta, d_ss_split, d_ss_pool;
  // streamed passes (mcov_stream_begin / mcov_stream_push)
  mcov::DevBuf d_stream_acc;          // StreamAcc + the carried reads' counts of the current batch
  mcov::DevBuf d_cap_scratch;         // per-region replays of the max_depth cap (mcov_region_stats_run)
  const void* ncig_key_ptr = nullptr; // device-resident offset array whose total op count is cached (stage_reads)
  int64_t ncig_key_n = -1, ncig_val = -1;
  int64_t stream_tile_lo = 0;         // tiles below this one hold final depth
  int64_t stream_reads = 0;           // distinct reads pushed so far
  bool stream_started = false;        // (count_del = 0 streams: the difference array has been cleared)
  mcov::DevBuf d_tasks, d_rlen, d_done, d_out, d_win_slot, d_win_n, d_win_out, d_htasks, d_tile_heavy, d_run_tasks, d_run_counts, d_run_out;
  int64_t n_runs = -1;               // records held in d_run_out ([tid | start | end | depth] x n_runs), -1 = none
  mcov::PinBuf h_pin;
  // pipelined statistics (mcov_region_stats_submit / collect): two pinned slots
  struct StatSlot {
    mcov::PinBuf buf;              // [g records | PassCounters]
    mcov::DevBuf d_rec;            // the slot's records on the device (copied back on d2h_stream)
    cudaEvent_t ready = nullptr;   // records written (main stream)
    cudaEvent_t done = nullptr;    // records in `buf` (d2h_stream)
    int64_t g = -1;                // -1 = nothing submitted
    bool has_verdict = false;
    bool has_subregion = false;    // some region starts inside its contig (matters only when the max_depth cap fired)
    int32_t cap_contigs = 0;       // of the pass the slot's records describe (-1: arrives with the verdict)
    int64_t n_reads = 0;
    std::vector<int32_t> len0;     // regions of length 0 (their records are zeroed, like mcov_region_stats_run)
  } slot[2];

  // launch accounting + optional per-kernel event timing
  int64_t n_launches = 0;
  bool profiling = false;
  std::vector<mcov::ProfRec> prof;
  std::vector<cudaEvent_t> ev_pool;
  double prof_ms[mcov::kKernelCount] = {0};
  int64_t prof_n[mcov::kKernelCount] = {0};

  cudaEvent_t ev_get() {
    if (!ev_pool.empty()) { cudaEvent_t e = ev_pool.back(); ev_pool.pop_back(); return e; }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
  }
  void prof_begin(int id) {
    ++n_launches;
    if (!profiling) return;
    mcov::ProfRec r; r.id = id; r.a = ev_get(); r.b = ev_get();
    cudaEventRecord(r.a, stream);
    prof.push_back(r);
  }
  void prof_end() {
    if (!profiling || prof.empty()) return;
    cudaEventRecord(prof.back().b, stream);
  }
  // fold finished records into the per-kernel totals (stream must be synchronised)
  void prof_collect() {
    for (auto& r : prof) {
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) { prof_ms[r.id] += ms; prof_n[r.id] += 1; }
      ev_pool.push_back(r.a); ev_pool.push_back(r.b);
    }
    prof.clear();
  }
};

// wrap one kernel launch (or memset) for accounting / timing
#define MCOV_LAUNCH(ctx, id, ...) do { (ctx)->prof_begin(id); __VA_ARGS__; (ctx)->prof_end(); } while (0)

// Host helpers of the count, allele and compare calls (basecount.cu, alleles.cu, compare.cu).  `who`, the entry point,
// starts every error text.

// return from the enclosing call with MCOV_ERR_CUDA ("who: call: CUDA error text") when a CUDA call fails
#define CTX_CU(who, call)                                                                                  \
  do {                                                                                                     \
    cudaError_t e__ = (call);                                                                              \
    if (e__ != cudaSuccess) return mcov::ctx_fail(ctx, MCOV_ERR_CUDA, std::string(who) + ": " + #call, e__); \
  } while (0)

namespace mcov {

struct AlleleParams;

// ctx->err = what (+ ": " and the CUDA error's text); returns code.
inline int ctx_fail(mcov_ctx* ctx, int code, const std::string& what, cudaError_t e = cudaSuccess) {
  ctx->err = what;
  if (e != cudaSuccess) { ctx->err += ": "; ctx->err += cudaGetErrorString(e); }
  return code;
}

// buf.ensure(need), unless the allocation that takes (DevBuf::grown) exceeds the free device memory plus buf's own:
// then MCOV_ERR_NOMEM, "who: " + msg, a format of (n, bytes wanted, bytes free); ensure_fits gives n_slots as n.  The environment variable
// free_hook, when set, stands in for the free bytes (a test hook).
inline int ensure_fits_n(mcov_ctx* ctx, DevBuf& buf, size_t need, const char* free_hook, const char* who, const char* msg,
                         long long n) {
  if (buf.cap < need) {
    size_t free_b = 0, total_b = 0;
    CTX_CU(who, cudaMemGetInfo(&free_b, &total_b));
    if (const char* h = std::getenv(free_hook)) free_b = (size_t)std::strtoull(h, nullptr, 10);
    const size_t want = DevBuf::grown(need);
    if (want > free_b + buf.cap) {
      char text[256];
      std::snprintf(text, sizeof(text), msg, n, want, free_b + buf.cap);
      return ctx_fail(ctx, MCOV_ERR_NOMEM, std::string(who) + ": " + text);
    }
  }
  CTX_CU(who, buf.ensure(need));
  return MCOV_OK;
}
inline int ensure_fits(mcov_ctx* ctx, DevBuf& buf, size_t need, const char* free_hook, const char* who, const char* msg) {
  return ensure_fits_n(ctx, buf, need, free_hook, who, msg, (long long)ctx->n_slots);
}

// g regions of the contig table, and where their records go
inline int check_regions(mcov_ctx* ctx, int64_t g, const int32_t* tid, const int32_t* start, const int32_t* end,
                         const void* out, const char* who) {
  if (g < 0 || (g > 0 && (!tid || !start || !end || !out))) return ctx_fail(ctx, MCOV_ERR_ARG, std::string(who) + ": bad arguments");
  for (int64_t i = 0; i < g; ++i)
    if (tid[i] < 0 || tid[i] >= ctx->n_contigs || start[i] < 0 || end[i] < start[i])
      return ctx_fail(ctx, MCOV_ERR_ARG, std::string(who) + ": need 0 <= start <= end and a valid tid");
  return MCOV_OK;
}

// Records [first, first + n) of a site list to the host; `builder` is the call that builds the list.
inline int read_site_list(mcov_ctx* ctx, const SiteList& sl, int64_t first, int64_t n, void* host_out, size_t site_bytes,
                          const char* who, const char* builder) {
  if (sl.n < 0 || sl.epoch != ctx->contig_epoch)
    return ctx_fail(ctx, MCOV_ERR_STATE, std::string(who) + ": no site list for this contig table (call " + builder + " first)");
  if (first < 0 || n < 0 || first > sl.n - n || (n > 0 && !host_out))
    return ctx_fail(ctx, MCOV_ERR_ARG, std::string(who) + ": range outside the site list");
  if (n == 0) return MCOV_OK;
  CTX_CU(who, cudaSetDevice(ctx->device));
  CTX_CU(who, cudaMemcpyAsync(host_out, sl.list.as<uint8_t>() + first * site_bytes, (size_t)n * site_bytes,
                              cudaMemcpyDeviceToHost, ctx->stream));
  CTX_CU(who, cudaStreamSynchronize(ctx->stream));
  return MCOV_OK;
}

// alleles.cu: the checked parameters or an error (MCOV_ERR_STATE without counts for the contig table); the grid of a
// grid-stride kernel over `items` work items, `per` of them a CTA.
int al_check(mcov_ctx* ctx, const mcov_allele_params* p, AlleleParams* out, const char* who);
unsigned al_grid(const mcov_ctx* ctx, int64_t items, int per);

// alleles.cu: every region cut into chunks of at most `chunk` positions inside its contig (positions past its end add
// to the length only); chunks to ctx->d_chunks, meta to d_chunk_meta, d_region_out sized to out_bytes, d_chunk_part to
// part_bytes a chunk.
int upload_region_chunks(mcov_ctx* ctx, int64_t g, const int32_t* tid, const int32_t* start, const int32_t* end,
                         int64_t chunk, size_t part_bytes, size_t out_bytes, const char* who, int64_t* n_chunks);

// alleles.cu: between a site list's count launch, which wrote `items` tile counts to ctx->d_site_tiles, and its write
// launch: the counts' inclusive scan into the `items` words behind them, the total read back, sl.list sized for it.
// With free_hook, the scan scratch and the list are checked against the free device memory first (ensure_fits_n, that
// test hook); without, a list that does not fit is MCOV_ERR_NOMEM once its allocation has failed.
int size_site_list(mcov_ctx* ctx, SiteList& sl, int64_t items, size_t site_bytes, const char* who, int64_t* total,
                   const char* free_hook = nullptr);

// alleles.cu: every site of the counts under P (mcov_allele_site records in slot order) into sl; *total their number.
// free_hook as in size_site_list, for the tile counts as well.
int allele_site_list(mcov_ctx* ctx, const AlleleParams& P, SiteList& sl, const char* who, int64_t* total,
                     const char* free_hook = nullptr);

}  // namespace mcov
