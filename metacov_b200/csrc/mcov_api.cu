// mcov_api.cu -- C-ABI entry points of the coverage hot path (include/metacov_b200.h).
//
// No CPU fallback lives here: every compute entry point launches CUDA kernels
// and fails with MCOV_ERR_CUDA when there is no device.
#include <algorithm>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

#include "ctx.cuh"
#include "k_expand.cuh"
#include "k_fused.cuh"
#include "k_prep_tma.cuh"
#include "k_tile_tma.cuh"
#include "k_block.cuh"
#include "k_hist.cuh"
#include "k_scan.cuh"
#include "k_export.cuh"
#include "k_stats.cuh"
#include "k_stats_stream.cuh"

using namespace mcov;

int mcov_order_stats_by_sort(mcov_ctx* ctx, const int32_t* d_region, int64_t n, int64_t pad, int breadth_n,
                             mcov_region_stats* d_stat, mcov::DevBuf& keys_out, mcov::DevBuf& temp);

namespace {

int fail(mcov_ctx* c, int code, const char* what, cudaError_t e = cudaSuccess) {
  if (c) {
    c->err = what;
    if (e != cudaSuccess) { c->err += ": "; c->err += cudaGetErrorString(e); }
  }
  return code;
}

#define CU(call)                                                        \
  do {                                                                  \
    cudaError_t e__ = (call);                                           \
    if (e__ != cudaSuccess) return fail(ctx, MCOV_ERR_CUDA, #call, e__); \
  } while (0)

int grid_for(const mcov_ctx* ctx, int64_t n, int threads, int per_sm) {
  int64_t want = (n + threads - 1) / threads;
  int64_t cap = (int64_t)ctx->n_sm * per_sm;
  if (want < 1) want = 1;
  return (int)std::min<int64_t>(want, cap);
}


// Launch with the programmatic-stream-serialization attribute (see pdl_wait in common.cuh): the kernel
// may start while its predecessor in the stream drains.  Only for kernels that call pdl_wait() before
// they touch anything the predecessor writes.
// `allow`: the overlap pays for short kernels (config C2: 0.209 -> 0.200 ms per step) and costs on long ones
// (C4 at full size: 14.9 -> 16.0 ms), so the callers enable it by problem size.
constexpr int64_t kPdlMaxSlots = (int64_t)1 << 27;     // 134 M slots
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(bool allow, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
  static const bool enabled = std::getenv("MCOV_NO_PDL") == nullptr;        // tuning hook: plain stream order instead
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = (enabled && allow) ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

PassCounters* pc_of(mcov_ctx* ctx) { return ctx->d_pc.as<PassCounters>(); }

// The flag tests of the read filter (pysam __advance_samtools + htslib's UNMAP drop, SURVEY.md Appendix A-2) as one
// bit per flag value below 4096; the prep kernel looks reads up instead of evaluating the masks.
void build_flag_lut(mcov_ctx* ctx) {
  const mcov_filter& f = ctx->filt;
  for (int w = 0; w < 128; ++w) ctx->flag_lut[w] = 0;
  for (uint32_t F = 0; F < 4096; ++F) {
    bool p = !(F & ((uint32_t)f.flag_filter | 0x4u));
    if (f.flag_require && !(F & f.flag_require)) p = false;
    if (f.ignore_orphans && (F & 0x1u) && !(F & 0x2u)) p = false;
    if (p) ctx->flag_lut[F >> 5] |= 1u << (F & 31u);
  }
  ctx->flag_lut_dirty = true;
}

int ensure_depth(mcov_ctx* ctx) {
  if (ctx->n_contigs <= 0) return fail(ctx, MCOV_ERR_STATE, "mcov_set_contigs has not been called");
  if (!ctx->depth_bound) {
    CU(ctx->depth_own.ensure((size_t)ctx->n_slots * sizeof(int32_t)));
    ctx->depth = ctx->depth_own.as<int32_t>();
  }
  CU(ctx->d_pc.ensure(sizeof(PassCounters)));
  return MCOV_OK;
}

// A transport block is copied without the call waiting for the copy (the host goes on to enqueue the statistics and
// to prepare the next batch while the link is busy); the copy is waited for at the start of the NEXT staging call,
// in mcov_sync and in mcov_destroy -- the block must stay unchanged until then.
int wait_pending_copy(mcov_ctx* ctx) {
  if (!ctx->copy_pending) return MCOV_OK;
  ctx->copy_pending = false;
  CU(cudaEventSynchronize(ctx->copied));
  return MCOV_OK;
}

// The next of the two staging sets, once the kernels of the pass that last read it are done.
int acquire_stage(mcov_ctx* ctx, ReadStage** out) {
  int rc = wait_pending_copy(ctx);
  if (rc) return rc;
  ReadStage& s = ctx->stage[ctx->stage_next];
  ctx->stage_next ^= 1;
  if (s.in_flight) { CU(cudaEventSynchronize(s.consumed)); s.in_flight = false; }
  *out = &s;
  return MCOV_OK;
}

// Entries of the 32-bit CIGAR offsets of n reads as the device rebuilds them: scanned in place, so a multiple of 4.
int64_t off_len_of(int64_t n) { return (n + 1 + 3) & ~(int64_t)3; }

// Size a staging set's columns for n reads of n_cig ops in all (32-bit offsets).
int stage_columns(mcov_ctx* ctx, ReadStage& st, int64_t n, int64_t n_cig) {
  const size_t n1 = (size_t)std::max<int64_t>(n, 1);
  CU(st.tid.ensure(n1 * 4)); CU(st.pos.ensure(n1 * 4)); CU(st.flag.ensure(n1 * 2)); CU(st.mapq.ensure(n1));
  CU(st.cig_off.ensure((size_t)off_len_of(n) * 4)); CU(st.cig.ensure((size_t)n_cig * 4 + 16));
  return MCOV_OK;
}

// The context's half of a pass's ExpandArgs: contig table, filter, depth store and pass counters.
void context_args(mcov_ctx* ctx, ExpandArgs& a) {
  a.contig_off = ctx->d_off.as<int64_t>(); a.contig_len = ctx->d_len.as<int32_t>(); a.n_contigs = ctx->n_contigs;
  a.filt = ctx->filt; a.delta = ctx->depth; a.pc = pc_of(ctx);
}

// The ExpandArgs of a batch held in the columns of a staging set (stage_columns).
ExpandArgs columns_of(mcov_ctx* ctx, const ReadStage& st, int64_t n, int64_t n_cig) {
  ExpandArgs a;
  std::memset(&a, 0, sizeof(a));
  a.n = n; a.n_cig = n_cig;
  a.tid = st.tid.as<int32_t>(); a.pos = st.pos.as<int32_t>(); a.flag = st.flag.as<uint16_t>();
  a.mapq = st.mapq.as<uint8_t>(); a.cig_off = st.cig_off.as<uint32_t>(); a.cig = st.cig.as<uint32_t>();
  context_args(ctx, a);
  a.cig_aligned16 = 1;
  return a;
}

bool aligned(const void* p, uintptr_t m) { return (reinterpret_cast<uintptr_t>(p) & (m - 1)) == 0; }

// The columns allow the vector loads of the prep and expand kernels (k_fused.cuh).
int vec_ok(const ExpandArgs& a) {
  return (aligned(a.tid, 16) && aligned(a.pos, 16) && aligned(a.cig_off64 ? (const void*)a.cig_off64 : (const void*)a.cig_off, 16) &&
          aligned(a.flag, 8) && aligned(a.mapq, 4)) ? 1 : 0;
}

// Stage host SoA into device memory on the copy stream (double-buffered), or
// pass device pointers through.  On return `a` holds device pointers and the
// compute stream has been made to wait for the copies.  An empty batch stages
// nothing: `a` then holds only the pass counters.
int stage_reads(mcov_ctx* ctx, int64_t n, const int32_t* tid, const int32_t* pos, const uint16_t* flag,
                const uint8_t* mapq, const void* cig_off, bool off64, const uint32_t* cig, int mem_kind,
                ExpandArgs& a, ReadStage** used) {
  *used = nullptr;
  if (n == 0) {
    std::memset(&a, 0, sizeof(a));
    a.pc = pc_of(ctx);
    return MCOV_OK;
  }
  ReadStage* s = nullptr;
  { int rc = mem_kind == MCOV_MEM_HOST ? acquire_stage(ctx, &s) : wait_pending_copy(ctx); if (rc) return rc; }
  a.n = n;
  a.n_cig = -1;
  a.cig_off = nullptr; a.cig_off64 = nullptr;
  const size_t ow = off64 ? 8 : 4;
  if (mem_kind == MCOV_MEM_DEVICE) {
    a.tid = tid; a.pos = pos; a.flag = flag; a.mapq = mapq; a.cig = cig;
    if (off64) a.cig_off64 = static_cast<const uint64_t*>(cig_off); else a.cig_off = static_cast<const uint32_t*>(cig_off);
    // ops per read decide between the two prep kernels; for device-resident columns the total is read back ONCE per
    // (offset array, n) -- a caller that runs pass after pass over the same arrays pays the round trip the first time only
    if (!off64 && n > 0) {
      if (ctx->ncig_key_ptr != cig_off || ctx->ncig_key_n != n) {
        uint32_t last = 0;
        CU(cudaMemcpyAsync(&last, static_cast<const uint32_t*>(cig_off) + n, 4, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        ctx->ncig_key_ptr = cig_off; ctx->ncig_key_n = n; ctx->ncig_val = (int64_t)last;
      }
      a.n_cig = ctx->ncig_val;
    }
  } else if (mem_kind == MCOV_MEM_HOST) {
    const uint64_t n_cig = off64 ? static_cast<const uint64_t*>(cig_off)[n] : static_cast<const uint32_t*>(cig_off)[n];
    a.n_cig = (int64_t)n_cig;
    CU(s->tid.ensure(n * 4)); CU(s->pos.ensure(n * 4)); CU(s->flag.ensure(n * 2)); CU(s->mapq.ensure(n));
    CU(s->cig_off.ensure((n + 1) * ow)); CU(s->cig.ensure((size_t)n_cig * 4 + 16));
    cudaStream_t cs = ctx->copy_stream;
    CU(cudaMemcpyAsync(s->tid.p, tid, n * 4, cudaMemcpyHostToDevice, cs));
    CU(cudaMemcpyAsync(s->pos.p, pos, n * 4, cudaMemcpyHostToDevice, cs));
    CU(cudaMemcpyAsync(s->flag.p, flag, n * 2, cudaMemcpyHostToDevice, cs));
    CU(cudaMemcpyAsync(s->mapq.p, mapq, n, cudaMemcpyHostToDevice, cs));
    CU(cudaMemcpyAsync(s->cig_off.p, cig_off, (n + 1) * ow, cudaMemcpyHostToDevice, cs));
    if (n_cig) CU(cudaMemcpyAsync(s->cig.p, cig, (size_t)n_cig * 4, cudaMemcpyHostToDevice, cs));
    CU(cudaEventRecord(ctx->copied, cs));
    CU(cudaStreamWaitEvent(ctx->stream, ctx->copied, 0));
    a.tid = s->tid.as<int32_t>(); a.pos = s->pos.as<int32_t>(); a.flag = s->flag.as<uint16_t>();
    a.mapq = s->mapq.as<uint8_t>(); a.cig = s->cig.as<uint32_t>();
    if (off64) a.cig_off64 = s->cig_off.as<uint64_t>(); else a.cig_off = s->cig_off.as<uint32_t>();
    *used = s;
  } else {
    return fail(ctx, MCOV_ERR_ARG, "mem_kind must be MCOV_MEM_HOST or MCOV_MEM_DEVICE");
  }
  context_args(ctx, a);
  a.cig_aligned16 = aligned(a.cig, 16) ? 1 : 0;
  return MCOV_OK;
}

int finish_stage(mcov_ctx* ctx, ReadStage* s, bool wait_copy = true) {
  if (!s) return MCOV_OK;
  CU(cudaEventRecord(s->consumed, ctx->stream));
  s->in_flight = true;
  // the caller may reuse its host arrays once the copies are done
  if (wait_copy) CU(cudaEventSynchronize(ctx->copied));
  else ctx->copy_pending = true;
  return MCOV_OK;
}

// Fused depth path for coordinate-sorted reads (k_fused.cuh).  `a` holds device pointers.
// tile_lo < 0: the pass writes the whole slot space; else only the tiles [tile_lo, tile_hi) (one batch of a streamed file).
int fused_depth_sorted(mcov_ctx* ctx, const ExpandArgs& a, int64_t tile_lo = -1, int64_t tile_hi = -1) {
  const int64_t n = a.n;
  if (n >= (int64_t)0xFFFFFFF0ll) return fail(ctx, MCOV_ERR_RANGE, "mcov_depth_sorted: a batch holds at most 2^32-16 reads (read indices are 32-bit); split it or use mcov_begin/push/finalize");
  const int64_t n_tiles = (ctx->n_slots + kTile - 1) / kTile;
  const int64_t cnt_pad = (n_tiles + 1 + 3) & ~(int64_t)3;             // per-tile arrays, scanned in place as int32
  const int64_t scan_len = 2 * cnt_pad;                                // [tile_agg | tile_cnt]
  const int64_t scan_tiles = (scan_len + kScanTile - 1) / kScanTile;
  const uint32_t far_cap = (uint32_t)std::min<int64_t>(std::max<int64_t>(n, 1), kFarCapDefault);
  // one zeroed scratch block: [tile_agg | tile_cnt | tile_cursor | tile_cap | scan status | per-contig "capped" flags]
  const size_t o_agg = 0, o_cnt = o_agg + (size_t)cnt_pad * 4, o_cur = o_cnt + (size_t)cnt_pad * 4,
               o_cap = o_cur + (size_t)n_tiles * 4, o_st = (o_cap + (size_t)n_tiles * 4 + 7) & ~(size_t)7,
               o_flag = o_st + ((size_t)scan_tiles + 1) * 8 /* + the ticket word */, z_bytes = o_flag + (size_t)ctx->n_contigs;
  CU(ctx->d_status.ensure(z_bytes));
  CU(ctx->d_start_slot.ensure((size_t)(std::max<int64_t>(n, 1) + 8) * sizeof(uint32_t)));   // rec (+ vector-load padding)
  CU(ctx->d_tile_off.ensure((size_t)(n_tiles + 1) * 4));                                 // tile_first
  CU(ctx->d_far_list.ensure((size_t)far_cap * 8));
  CU(ctx->d_far_sorted.ensure((size_t)far_cap * 4));
  cudaStream_t s = ctx->stream;
  char* z = ctx->d_status.as<char>();
  CU(cudaMemsetAsync(z, 0, z_bytes, s));
  FusedArgs f;
  f.e = a;
  f.rec = ctx->d_start_slot.as<uint32_t>();
  f.n_slots = ctx->n_slots;
  f.n_tiles = n_tiles;
  if (ctx->flag_lut_dirty) {                                  // the filter changed: refresh the device copy of its flag table
    CU(ctx->d_flag_lut.ensure(sizeof(ctx->flag_lut)));
    CU(cudaMemcpyAsync(ctx->d_flag_lut.p, ctx->flag_lut, sizeof(ctx->flag_lut), cudaMemcpyHostToDevice, s));
    ctx->flag_lut_dirty = false;
  }
  f.tile_lo = 0; f.tile_hi = n_tiles; f.streaming = 0;
  if (tile_lo >= 0) { f.tile_lo = tile_lo; f.tile_hi = std::min(tile_hi, n_tiles); f.streaming = 1; }
  f.far_end = ctx->d_far_list.as<int64_t>();
  f.far_cap = far_cap;
  f.tile_agg = reinterpret_cast<int32_t*>(z + o_agg);
  f.tile_cnt = reinterpret_cast<uint32_t*>(z + o_cnt);
  f.tile_cursor = reinterpret_cast<uint32_t*>(z + o_cur);
  f.far_sorted = ctx->d_far_sorted.as<uint32_t>();
  f.tile_first = ctx->d_tile_off.as<uint32_t>();
  CU(ctx->d_tile_heavy.ensure((size_t)n_tiles * 4));
  f.tile_heavy = ctx->d_tile_heavy.as<uint32_t>();
  // "heavy" = at least 8x the average tile (and at least 4096 reads): scheduled first by the tile kernel
  f.heavy_min = (uint32_t)std::min<int64_t>(std::max<int64_t>(4096, 8 * n / std::max<int64_t>(n_tiles, 1)), 0x7fffffff);
  f.depth = ctx->depth;
  f.tile_cap = reinterpret_cast<int32_t*>(z + o_cap);
  // per-tile depth histograms for the statistics of large regions: written by a one-shot pass when at least half of the
  // tiles lie wholly inside a large region of the cached region plan, and trusted until the depth is written otherwise.
  // The kernel then counts every tile, and a counted tile costs it about a third of what a used histogram saves the
  // statistics (B200, C2: +6.4 us tile, -18.4 us statistics over 23 417 of 24 416 tiles), so a plan that leaves most
  // tiles outside its large regions gets none (C3, 3 % inside: the tile kernel lost 53 us for 6 us of statistics).
  f.tile_hist = nullptr;
  if (tile_lo < 0 && ctx->plan.valid && ctx->plan.n_contigs_epoch == ctx->contig_epoch && 2 * ctx->plan.hist_tiles >= n_tiles) {
    CU(ctx->d_tile_hist.ensure((size_t)n_tiles * kTileHistWords * 2));
    f.tile_hist = ctx->d_tile_hist.as<uint16_t>();
    ctx->tile_hist_plan = ctx->plan.id;
  }
  ctx->tile_hist_valid = f.tile_hist != nullptr;
  f.max_depth = ctx->filt.max_depth;
  f.flag_lut = ctx->d_flag_lut.as<uint32_t>();
  const bool off64 = a.cig_off64 != nullptr;
  f.vec_ok = n > 0 ? vec_ok(a) : 0;
  if (n > 0) {
    const int64_t groups = (n + kPrepPer - 1) / kPrepPer;
    // short-read hot path: SoA chunks staged by TMA bulk copies behind mbarriers (k_prep_tma.cuh); needs 32-bit
    // offsets and 16-byte aligned columns.  Anything else takes the per-thread loads of k_fused_prep.
    // Long CIGARs (config C5: ~2 700 ops per read) are reduced by whole warps straight from global memory in either
    // kernel, and there the 8 x 4 warps per SM of k_fused_prep keep more loads in flight than the staged kernel's 3 x 8
    // consumer warps (B200, C5 at 1 M reads: 2.4 ms against 4.6 ms): more than kPrepLongOps ops per read on average
    // take k_fused_prep.
    constexpr int64_t kPrepLongOps = 16;
    const bool long_cigars = a.n_cig >= 0 && a.n_cig > kPrepLongOps * n;
    const bool tma = !off64 && !long_cigars && aligned(a.tid, 16) && aligned(a.pos, 16) && aligned(a.cig_off, 16) &&
                     aligned(a.flag, 16) && aligned(a.mapq, 16) && aligned(a.cig, 16);
    if (tma) {
      const int64_t n_chunks = (n + kPtChunk - 1) / kPtChunk;
      const unsigned grid = (unsigned)std::min<int64_t>(n_chunks, (int64_t)ctx->n_sm * MCOV_PREP_CTAS);
      MCOV_LAUNCH(ctx, kKFusedPrepTma, (k_fused_prep_tma<<<grid, kPtThreads, kPtSmemBytes, s>>>(f)));
    } else if (off64) MCOV_LAUNCH(ctx, kKFusedPrep, (k_fused_prep<true><<<grid_for(ctx, groups, kPrepThreads, 8), kPrepThreads, 0, s>>>(f)));
    else MCOV_LAUNCH(ctx, kKFusedPrep, (k_fused_prep<false><<<grid_for(ctx, groups, kPrepThreads, 8), kPrepThreads, 0, s>>>(f)));
    CU(cudaGetLastError());
  } else {
    CU(cudaMemsetAsync(f.tile_first, 0, (size_t)(n_tiles + 1) * 4, s));
  }
  // prep -> scan_counts -> far_scatter -> tile (-> statistics) are chained with programmatic dependent
  // launches: each kernel's CTAs are in place before its predecessor has drained
  const bool pdl = ctx->n_slots <= kPdlMaxSlots;
  // (the look-back scan beat one CTA and an 8-CTA cluster on these counters: DESIGN.md 3.1)
  MCOV_LAUNCH(ctx, kKScanCounts, CU(launch_pdl(pdl, k_scan_inplace<false>, dim3((unsigned)scan_tiles), dim3(kScanThreads), 0, s,
      f.tile_agg, scan_len, reinterpret_cast<unsigned long long*>(z + o_st), pc_of(ctx))));
  MCOV_LAUNCH(ctx, kKFarScatter, CU(launch_pdl(pdl, k_far_scatter, dim3(ctx->n_sm * 2), dim3(256), 0, s, f)));
  ctx->fused_blob.assign(reinterpret_cast<const unsigned char*>(&f), reinterpret_cast<const unsigned char*>(&f) + sizeof(f));
  // (a streamed batch that does not reach a new tile launches no tile kernel: everything it holds is carried into the next one)
  if (f.tile_hi > f.tile_lo) {
    // warp-specialised: producer warp + TMA record ring + 4 consumer warps (k_tile_tma.cuh); persistent
    const unsigned grid = (unsigned)std::min<int64_t>(f.tile_hi - f.tile_lo, (int64_t)ctx->n_sm * MCOV_TT_CTAS);
    if (f.tile_hist) MCOV_LAUNCH(ctx, kKFusedTileTma, CU(launch_pdl(pdl, k_fused_tile_tma<true>, dim3(std::max(grid, 1u)), dim3(kTtThreads), 0, s, f)));
    else MCOV_LAUNCH(ctx, kKFusedTileTma, CU(launch_pdl(pdl, k_fused_tile_tma<false>, dim3(std::max(grid, 1u)), dim3(kTtThreads), 0, s, f)));
  }
  // htslib's max_depth cap: replayed on the device, in stream order, where the tile kernel found that
  // it can fire (k_cap_replay returns after one load otherwise) -- every consumer of the depth that
  // follows on this stream sees the capped values, whether or not the host has looked at the verdict yet
  ctx->cap_flags = reinterpret_cast<uint8_t*>(z + o_flag);
  if (f.max_depth > 0)
    MCOV_LAUNCH(ctx, kKCapReplay, CU(launch_pdl(pdl, k_cap_replay, dim3((unsigned)((ctx->n_contigs + 127) / 128)), dim3(128), 0, s,
                                                f, ctx->cap_flags)));
  return MCOV_OK;
}

// Difference array -> depth in place: the look-back scan over the whole slot space, which also records the pass's
// depth metrics.
int scan_depth(mcov_ctx* ctx) {
  const int64_t n_tiles = (ctx->n_slots + kScanTile - 1) / kScanTile;
  CU(ctx->d_status.ensure(((size_t)n_tiles + 1) * 8));            // status words + the ticket word
  CU(cudaMemsetAsync(ctx->d_status.p, 0, ((size_t)n_tiles + 1) * 8, ctx->stream));
  MCOV_LAUNCH(ctx, kKScan, (k_scan_inplace<true><<<(unsigned)n_tiles, kScanThreads, 0, ctx->stream>>>(
      ctx->depth, ctx->n_slots, ctx->d_status.as<unsigned long long>(), pc_of(ctx))));
  CU(cudaGetLastError());
  return MCOV_OK;
}

// count_del = 0 (only M = X positions count): the any-order formulation -- clear, one +1 / -1 pair per run of M = X ops
// (k_expand_runs), look-back scan.  Reads [i_begin, n) of the batch; `clear` / `finalize` let a stream spread the
// pass over its batches.
int runs_depth(mcov_ctx* ctx, const ExpandArgs& a, int64_t i_begin, bool clear, bool finalize) {
  cudaStream_t s = ctx->stream;
  ctx->tile_hist_valid = false;
  if (clear) MCOV_LAUNCH(ctx, kKClear, CU(cudaMemsetAsync(ctx->depth, 0, (size_t)ctx->n_slots * 4, s)));
  if (a.n > i_begin) {
    FusedArgs f;
    std::memset(&f, 0, sizeof(f));
    f.e = a;
    MCOV_LAUNCH(ctx, kKExpand, (k_expand_runs<<<grid_for(ctx, a.n - i_begin, 256, 8), 256, 0, s>>>(f, i_begin)));
    CU(cudaGetLastError());
  }
  return finalize ? scan_depth(ctx) : MCOV_OK;
}

// per-base depth of a whole sorted batch from device columns: the fused path, or the M-run formulation when the
// filter says count_del = 0
int depth_from_columns(mcov_ctx* ctx, const ExpandArgs& a) {
  if (ctx->filt.count_del) return fused_depth_sorted(ctx, a);
  return runs_depth(ctx, a, 0, true, true);
}

// The verdict of a pass from a host copy of its counters; changes nothing but the error text.  `n_reads` is what the
// pass sized its bucket list of long-span reads for; `who` names the call that reports the failure.
int check_pass(mcov_ctx* ctx, const PassCounters& h, int64_t n_reads, const char* who) {
  auto no = [&](int code, const char* why) { return fail(ctx, code, (std::string(who) + ": " + why).c_str()); };
  if (h.unsorted) return no(MCOV_ERR_UNSORTED, "reads are not sorted by (tid,pos); use mcov_begin/push/finalize");
  if ((int64_t)h.n_far > std::min<int64_t>(std::max<int64_t>(n_reads, 1), kFarCapDefault))
    return no(MCOV_ERR_RANGE, "too many long-span reads for the bucket list; use mcov_begin/push/finalize");
  if (h.far_overflow) return no(MCOV_ERR_RANGE, "a batch held too many long-span reads for the bucket list; use mcov_begin/push/finalize");
  if (h.cap_unreplayed)
    return no(MCOV_ERR_STATE, "htslib's max_depth cap fires in this file (a pile deeper than max_depth); the exact replay needs "
                              "the contig's reads in one batch -- run the file through mcov_depth_sorted, or raise max_depth");
  return MCOV_OK;
}

// Deliver the deferred verdict of an asynchronous fused pass (stream already synchronised,
// `h` = the pass counters just read back).
int fused_verdict(mcov_ctx* ctx, const PassCounters& h, const char* who) {
  if (!ctx->verdict_pending) return MCOV_OK;
  ctx->verdict_pending = false;
  int rc = check_pass(ctx, h, ctx->n_reads_pushed, who);
  if (rc) ctx->state = kIdle;
  else ctx->cap_contigs = (int32_t)h.cap_contigs;        // replayed by k_cap_replay right after the tile kernel
  return rc;
}

// Synchronise the stream behind what the caller has enqueued and deliver a pending verdict.  The counters are read
// back only for the verdict, or into `out` when the caller wants them.
int sync_verdict(mcov_ctx* ctx, const char* who, PassCounters* out = nullptr) {
  PassCounters h;
  PassCounters* hp = out ? out : &h;
  if (out || ctx->verdict_pending) CU(cudaMemcpyAsync(hp, ctx->d_pc.p, sizeof(PassCounters), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return fused_verdict(ctx, *hp, who);
}

// The depth pass of a whole sorted batch once its columns are on the device, and its bookkeeping.  With `wait` the
// verdict is delivered here, else by the next synchronising call.
int run_sorted_pass(mcov_ctx* ctx, const ExpandArgs& a, ReadStage* st, int64_t n_reads, bool wait_copy, bool wait, const char* who) {
  CU(cudaMemsetAsync(ctx->d_pc.p, 0, sizeof(PassCounters), ctx->stream));
  int rc = depth_from_columns(ctx, a);
  if (rc) return rc;
  ctx->n_reads_pushed = n_reads;
  rc = finish_stage(ctx, st, wait_copy);
  if (rc) return rc;
  ctx->state = kDepthReady;
  ctx->verdict_pending = true;
  // sortedness is a property of the data: one small read-back decides
  return wait ? sync_verdict(ctx, who) : MCOV_OK;
}

// Host checks of a narrow transport (a per-contig read-count prefix instead of tid[], op counts instead of offsets):
// the device rebuilds the offsets from the op counts and reads cig[] there, so they must add up to the op array.
template <typename NCig>
int check_narrow(mcov_ctx* ctx, int64_t n, const int64_t* contig_read_start, const NCig* n_cigar, int64_t n_cig_total,
                 const uint8_t* mapq, const char* who) {
  auto bad = [&](const char* why) { return fail(ctx, MCOV_ERR_ARG, (std::string(who) + ": " + why).c_str()); };
  if (!mapq && ctx->filt.min_mapq > 0) return bad("mapq is required when min_mapq > 0");
  if (contig_read_start[0] != 0 || contig_read_start[ctx->n_contigs] > n) return bad("contig_read_start must start at 0 and end <= n");
  uint64_t sum = 0;
  for (int64_t i = 0; i < n; ++i) sum += n_cigar[i];
  if (sum != (uint64_t)n_cig_total) return bad("the op counts do not add up to n_cig_total");
  return MCOV_OK;
}

// Bring a transport block (host memory) to the device with ONE copy and widen it into the columns of a staging
// set (k_block.cuh).  On return `a` describes the batch and the compute stream has the unpack kernels enqueued.
int block_stage(mcov_ctx* ctx, const void* block, int64_t bytes, ExpandArgs& a, ReadStage** used, mcov_block_hdr& h) {
  *used = nullptr;
  if (!block || bytes < (int64_t)sizeof(mcov_block_hdr)) return fail(ctx, MCOV_ERR_ARG, "transport block: null or too short");
  std::memcpy(&h, block, sizeof(h));
  if (h.magic != MCOV_BLOCK_MAGIC || h.version != 4) return fail(ctx, MCOV_ERR_ARG, "transport block: bad magic / version");
  const int64_t n = h.n;
  if (n < 0 || n >= 0xFFFFFFF0ll || h.n_carry < 0 || h.n_carry > n || h.n_exc < 0 || h.n_esc < 0 || h.n_esc > n || h.n_xops < 0 || h.n_cigar < 0 ||
      h.n_cigar > 0xFFFFFFF0ll || h.n_xops > h.n_cigar || h.total_bytes > bytes || h.n_contigs != ctx->n_contigs || h.n_dict < 0 || h.n_dict > 128 ||
      h.n_jt < 0 || h.n_jt > 255 || h.n_dictops < 0 || h.n_dictops > 512 || (h.xop_bytes != 2 && h.xop_bytes != 4) || h.nib > 1 ||
      (h.nib && (h.n_dq < 0 || h.n_dq > n || h.n_fq < 0 || h.n_fq > n)))
    return fail(ctx, MCOV_ERR_ARG, "transport block: inconsistent header (or packed for another contig table)");
  {
    const uint64_t tb = (uint64_t)h.total_bytes, n1 = (uint64_t)std::max<int64_t>(n, 1);
    auto in = [&](uint32_t off, uint64_t len) { return (off & 15u) == 0 && (uint64_t)off + len <= tb; };
    const bool per_read = (h.nib ? in(h.off_nb, n1) && in(h.off_dq, (uint64_t)h.n_dq) && in(h.off_fq, (uint64_t)h.n_fq)
                                 : in(h.off_dpos, n1) && in(h.off_fc, n1)) &&
                          in(h.off_chunk, (uint64_t)((n + MCOV_BLOCK_CHUNK - 1) / MCOV_BLOCK_CHUNK) * sizeof(mcov_block_chunk));
    if (!in(h.off_crs, ((uint64_t)h.n_contigs + 1) * 8) || !per_read || !in(h.off_exc_idx, (uint64_t)h.n_exc * 4) ||
        !in(h.off_exc_val, (uint64_t)h.n_exc * 4) || !in(h.off_jt, 1024) || !in(h.off_esc_idx, (uint64_t)h.n_esc * 4) ||
        !in(h.off_esc_flag, (uint64_t)h.n_esc * 2) || !in(h.off_esc_cls, (uint64_t)h.n_esc) || !in(h.off_dict_off, 129 * 4) ||
        !in(h.off_dict_ops, 2048) || !in(h.off_xops, (uint64_t)h.n_xops * (uint64_t)h.xop_bytes) || (h.has_mapq && !in(h.off_mapq, n1)))
      return fail(ctx, MCOV_ERR_ARG, "transport block: a section lies outside the block");
  }
  if (!h.has_mapq && ctx->filt.min_mapq > 0) return fail(ctx, MCOV_ERR_ARG, "transport block: packed without mapq, but the filter has min_mapq > 0");
  ReadStage* st = nullptr;
  int rc = acquire_stage(ctx, &st);
  if (rc) return rc;
  const int64_t off_len = off_len_of(n);
  CU(st->raw.ensure((size_t)h.total_bytes + 16));
  rc = stage_columns(ctx, *st, n, h.n_cigar);
  if (rc) return rc;
  const int64_t n_chunks = (off_len + kBlkChunk - 1) / kBlkChunk;
  CU(cudaMemcpyAsync(st->raw.p, block, (size_t)h.total_bytes, cudaMemcpyHostToDevice, ctx->copy_stream));
  CU(cudaEventRecord(ctx->copied, ctx->copy_stream));
  BlockArgs b;
  b.blk = st->raw.as<char>(); b.h = h; b.off_len = off_len;
  b.tid = st->tid.as<int32_t>(); b.pos = st->pos.as<int32_t>(); b.flag = st->flag.as<uint16_t>(); b.mapq = st->mapq.as<uint8_t>();
  b.cig_off = st->cig_off.as<uint32_t>(); b.cig = st->cig.as<uint32_t>();
  // The unpack kernel needs the block's copy and nothing else -- it writes the columns of THIS staging set, which no kernel
  // of the previous pass reads -- so it runs on a stream of its own and fills whatever the previous pass leaves idle (the
  // tails of its kernels, the gaps between them) instead of queueing behind it.  (Per-kernel timing keeps it on the main
  // stream: the event pairs are recorded there.)
  if (ctx->profiling) {
    CU(cudaStreamWaitEvent(ctx->stream, ctx->copied, 0));
    MCOV_LAUNCH(ctx, kKBlockUnpack, (k_block_expand<<<(unsigned)n_chunks, kBlkThreads, 0, ctx->stream>>>(b)));
  } else {
    CU(cudaStreamWaitEvent(ctx->unpack_stream, ctx->copied, 0));
    MCOV_LAUNCH(ctx, kKBlockUnpack, (k_block_expand<<<(unsigned)n_chunks, kBlkThreads, 0, ctx->unpack_stream>>>(b)));
    CU(cudaEventRecord(ctx->unpacked, ctx->unpack_stream));
    CU(cudaStreamWaitEvent(ctx->stream, ctx->unpacked, 0));
  }
  CU(cudaGetLastError());
  a = columns_of(ctx, *st, n, h.n_cigar);
  *used = st;
  return MCOV_OK;
}

// tile up to which a batch ending with the read (lt, lp) makes the depth final (reads without a valid contig sort
// after every slot)
int64_t stream_tile_of(const mcov_ctx* ctx, int32_t lt, int32_t lp) {
  const int64_t n_tiles = (ctx->n_slots + kTile - 1) / kTile;
  int64_t slot = ctx->n_slots;
  if (lt >= 0 && lt < ctx->n_contigs) slot = ctx->off[lt] + std::min<int64_t>(std::max<int64_t>(lp, 0), ctx->len[lt]);
  return std::min<int64_t>(slot >> kTileShift, n_tiles);
}

// Regions come from the caller: each needs a valid contig and 0 <= start <= end.
int check_regions(mcov_ctx* ctx, int64_t g, const int32_t* tid, const int32_t* start, const int32_t* end, const char* who) {
  for (int64_t i = 0; i < g; ++i)
    if (tid[i] < 0 || tid[i] >= ctx->n_contigs || start[i] < 0 || end[i] < start[i])
      return fail(ctx, MCOV_ERR_ARG, (std::string(who) + ": need 0 <= start <= end and a valid tid").c_str());
  return MCOV_OK;
}

// A region clipped to its contig: n positions from cs lie inside it.  A region may reach past its contig: the
// reference's vector is end-start long whatever the contig length (pileup.py:10-11) and stays 0 there, so the pad
// positions past the contig's end count as depth 0.
struct Clip { int64_t cs, n; int32_t pad; };
Clip clip_region(const mcov_ctx* ctx, int32_t tid, int32_t start, int32_t end) {
  const int64_t len = ctx->len[tid];
  const int64_t cs = std::min<int64_t>(start, len), n = std::min<int64_t>(end, len) - cs;
  return {cs, n, (int32_t)((int64_t)end - start - n)};
}

// Every kernel of a pass asks for the same shared-memory carve-out (the maximum): consecutive kernels with
// different L1 / shared-memory splits make the SMs reconfigure between launches, which costs a few
// microseconds per kernel on a step of ~180 us.  Also opts the TMA kernels into their dynamic shared memory.
int configure_kernels(mcov_ctx* ctx) {
  const int mx = (int)cudaSharedmemCarveoutMaxShared;           // (function attributes are per device: set for every context)
  CU(cudaFuncSetAttribute(k_fused_prep_tma, cudaFuncAttributeMaxDynamicSharedMemorySize, kPtSmemBytes));
  CU(cudaFuncSetAttribute(k_stats_stream, cudaFuncAttributeMaxDynamicSharedMemorySize, kSsSmemBytes));
  CU(cudaFuncSetAttribute(k_fused_prep_tma, cudaFuncAttributePreferredSharedMemoryCarveout, mx));
  CU(cudaFuncSetAttribute(k_block_expand, cudaFuncAttributePreferredSharedMemoryCarveout, mx));
  CU(cudaFuncSetAttribute(k_fused_prep<false>, cudaFuncAttributePreferredSharedMemoryCarveout, mx));
  CU(cudaFuncSetAttribute(k_scan_inplace<false>, cudaFuncAttributePreferredSharedMemoryCarveout, mx));
  CU(cudaFuncSetAttribute(k_far_scatter, cudaFuncAttributePreferredSharedMemoryCarveout, mx));
  CU(cudaFuncSetAttribute(k_fused_tile_tma<false>, cudaFuncAttributePreferredSharedMemoryCarveout, mx));
  CU(cudaFuncSetAttribute(k_fused_tile_tma<true>, cudaFuncAttributePreferredSharedMemoryCarveout, mx));
  CU(cudaFuncSetAttribute(k_cap_replay, cudaFuncAttributePreferredSharedMemoryCarveout, mx));
  CU(cudaFuncSetAttribute(k_stats_stream, cudaFuncAttributePreferredSharedMemoryCarveout, mx));
  CU(cudaFuncSetAttribute(k_region_stats_warp, cudaFuncAttributePreferredSharedMemoryCarveout, mx));
  CU(cudaFuncSetAttribute(k_region_stats_small, cudaFuncAttributePreferredSharedMemoryCarveout, mx));
  return MCOV_OK;
}

}  // namespace

extern "C" {

int mcov_abi_version(void) { return MCOV_ABI_VERSION; }

void mcov_default_filter(mcov_filter* f) {
  if (!f) return;
  std::memset(f, 0, sizeof(*f));
  f->flag_filter = 0x704;   // UNMAP | SECONDARY | QCFAIL | DUP (pysam pileup default)
  f->flag_require = 0;
  f->min_mapq = 0;
  f->ignore_orphans = 1;
  f->count_del = 1;          // `column.n` counts the reads whose op at the position is D or N (SURVEY.md Appendix A-4)
  f->reflen0_as_one = 0;     // a read that consumes no reference contributes nothing (current htslib)
  f->max_depth = 8000;
}

int mcov_create(mcov_ctx** out, int device, void* stream) {
  if (!out) return MCOV_ERR_ARG;
  *out = nullptr;
  int n_dev = 0;
  cudaError_t e = cudaGetDeviceCount(&n_dev);
  if (e != cudaSuccess || n_dev <= 0 || device < 0 || device >= n_dev) return MCOV_ERR_CUDA;
  mcov_ctx* ctx = new (std::nothrow) mcov_ctx();
  if (!ctx) return MCOV_ERR_NOMEM;
  ctx->device = device;
  if (cudaSetDevice(device) != cudaSuccess) { delete ctx; return MCOV_ERR_CUDA; }
  if (cudaDeviceGetAttribute(&ctx->n_sm, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || ctx->n_sm <= 0) { delete ctx; return MCOV_ERR_CUDA; }
  if (stream) { ctx->stream = reinterpret_cast<cudaStream_t>(stream); ctx->own_stream = false; }
  else {
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return MCOV_ERR_CUDA; }
    ctx->own_stream = true;
  }
  bool ok = cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) == cudaSuccess &&
            cudaStreamCreateWithFlags(&ctx->d2h_stream, cudaStreamNonBlocking) == cudaSuccess &&
            cudaEventCreateWithFlags(&ctx->copied, cudaEventDisableTiming) == cudaSuccess &&
            cudaStreamCreateWithFlags(&ctx->unpack_stream, cudaStreamNonBlocking) == cudaSuccess &&
            cudaEventCreateWithFlags(&ctx->unpacked, cudaEventDisableTiming) == cudaSuccess &&
            cudaEventCreateWithFlags(&ctx->stage[0].consumed, cudaEventDisableTiming) == cudaSuccess &&
            cudaEventCreateWithFlags(&ctx->stage[1].consumed, cudaEventDisableTiming) == cudaSuccess;
  if (!ok) { mcov_destroy(ctx); return MCOV_ERR_CUDA; }
  mcov_default_filter(&ctx->filt);
  build_flag_lut(ctx);
  if (configure_kernels(ctx) != MCOV_OK) { mcov_destroy(ctx); return MCOV_ERR_CUDA; }
  *out = ctx;
  return MCOV_OK;
}

void mcov_destroy(mcov_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  if (ctx->copy_stream) { cudaStreamSynchronize(ctx->copy_stream); cudaStreamDestroy(ctx->copy_stream); }
  if (ctx->d2h_stream) { cudaStreamSynchronize(ctx->d2h_stream); cudaStreamDestroy(ctx->d2h_stream); }
  if (ctx->copied) cudaEventDestroy(ctx->copied);
  if (ctx->unpack_stream) { cudaStreamSynchronize(ctx->unpack_stream); cudaStreamDestroy(ctx->unpack_stream); }
  if (ctx->unpacked) cudaEventDestroy(ctx->unpacked);
  for (auto& s : ctx->stage) {
    if (s.consumed) cudaEventDestroy(s.consumed);
    s.tid.release(); s.pos.release(); s.flag.release(); s.mapq.release(); s.cig_off.release(); s.cig.release(); s.raw.release();
  }
  DevBuf* bufs[] = {&ctx->d_len, &ctx->d_off, &ctx->depth_own, &ctx->d_pc, &ctx->d_status,
                    &ctx->d_start_slot, &ctx->d_far_list, &ctx->d_tile_cnt, &ctx->d_tile_off, &ctx->d_far_sorted, &ctx->d_tile_hist,
                    &ctx->d_tasks, &ctx->d_rlen, &ctx->d_done,
                    &ctx->d_cap_scratch, &ctx->d_flag_lut, &ctx->d_stream_acc, &ctx->d_ss_pieces, &ctx->d_ss_cta, &ctx->d_ss_split, &ctx->d_ss_pool,
                    &ctx->d_out, &ctx->d_win_slot, &ctx->d_win_n, &ctx->d_win_out, &ctx->d_htasks, &ctx->d_tile_heavy, &ctx->d_run_tasks, &ctx->d_run_counts, &ctx->d_run_out,
                    &ctx->d_starts, &ctx->d_bc, &ctx->d_bc_word,
                    &ctx->d_ref, &ctx->d_ref_stage, &ctx->d_pair_sigs, &ctx->d_chunks, &ctx->d_chunk_meta, &ctx->d_chunk_part,
                    &ctx->d_region_out, &ctx->d_site_tiles, &ctx->d_site_scan, &ctx->allele_sites.list, &ctx->compare_sites.list};
  for (DevBuf* b : bufs) b->release();
  ctx->bam.release();
  ctx->h_pin.release();
  for (auto& sl : ctx->slot) {
    sl.buf.release(); sl.d_rec.release();
    if (sl.done) cudaEventDestroy(sl.done);
    if (sl.ready) cudaEventDestroy(sl.ready);
  }
  ctx->prof_collect();
  for (cudaEvent_t e : ctx->ev_pool) cudaEventDestroy(e);
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char* mcov_last_error(const mcov_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int mcov_set_contigs(mcov_ctx* ctx, int32_t n_contigs, const int32_t* len) {
  if (!ctx || n_contigs <= 0 || !len) return fail(ctx, MCOV_ERR_ARG, "mcov_set_contigs: bad arguments");
  CU(cudaSetDevice(ctx->device));
  ctx->len.assign(len, len + n_contigs);
  ctx->off.resize((size_t)n_contigs + 1);
  int64_t o = 0;
  for (int32_t c = 0; c < n_contigs; ++c) {
    if (len[c] < 0) return fail(ctx, MCOV_ERR_ARG, "mcov_set_contigs: negative contig length");
    ctx->off[c] = o;
    o += ((int64_t)len[c] + 1 + 3) & ~(int64_t)3;   // len+1 slots, next contig 16-byte aligned
  }
  ctx->off[n_contigs] = o;
  ctx->n_slots = o;
  ctx->n_contigs = n_contigs;
  CU(ctx->d_len.ensure((size_t)n_contigs * 4));
  CU(ctx->d_off.ensure(((size_t)n_contigs + 1) * 8));
  CU(cudaMemcpyAsync(ctx->d_len.p, ctx->len.data(), (size_t)n_contigs * 4, cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(ctx->d_off.p, ctx->off.data(), ((size_t)n_contigs + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  ctx->state = kIdle;
  ctx->depth_bound = false;
  ctx->depth = nullptr;
  ctx->contig_epoch += 1;
  ctx->plan.valid = false;
  ctx->tile_hist_valid = false;
  return MCOV_OK;
}

int64_t mcov_n_slots(const mcov_ctx* ctx) { return ctx ? ctx->n_slots : 0; }

int64_t mcov_contig_offset(const mcov_ctx* ctx, int32_t tid) {
  if (!ctx || tid < 0 || tid >= ctx->n_contigs) return -1;
  return ctx->off[tid];
}

int mcov_bind_depth(mcov_ctx* ctx, int32_t* dev, int64_t n_slots) {
  if (!ctx) return MCOV_ERR_ARG;
  if (!dev || n_slots < ctx->n_slots || (reinterpret_cast<uintptr_t>(dev) & 15u))
    return fail(ctx, MCOV_ERR_ARG, "mcov_bind_depth: need a 16-byte aligned device buffer of >= mcov_n_slots() int32");
  ctx->depth = dev;
  ctx->depth_bound = true;
  ctx->state = kIdle;
  ctx->tile_hist_valid = false;
  return MCOV_OK;
}

int mcov_set_filter(mcov_ctx* ctx, const mcov_filter* f) {
  if (!ctx || !f) return fail(ctx, MCOV_ERR_ARG, "mcov_set_filter: null argument");
  ctx->filt = *f;
  build_flag_lut(ctx);
  return MCOV_OK;
}

int mcov_depth_sorted_delta(mcov_ctx* ctx, int64_t n, const int64_t* contig_read_start, const uint16_t* dpos,
                            int64_t n_exc, const uint32_t* exc_index, const int32_t* exc_delta, const uint16_t* flag,
                            const uint8_t* mapq, const uint8_t* n_cigar, const uint16_t* cig, int64_t n_cig_total, int wait) {
  if (!ctx) return MCOV_ERR_ARG;
  if (n < 0 || n_exc < 0 || n_cig_total < 0 || n_cig_total > 0xFFFFFFFFll) return fail(ctx, MCOV_ERR_ARG, "mcov_depth_sorted_delta: bad sizes");
  if (!contig_read_start || (n > 0 && (!dpos || !flag || !n_cigar)) || (n_cig_total > 0 && !cig) || (n_exc > 0 && (!exc_index || !exc_delta)))
    return fail(ctx, MCOV_ERR_ARG, "mcov_depth_sorted_delta: null array");
  CU(cudaSetDevice(ctx->device));
  int rc = ensure_depth(ctx);
  if (rc) return rc;
  rc = check_narrow(ctx, n, contig_read_start, n_cigar, n_cig_total, mapq, "mcov_depth_sorted_delta");
  if (rc) return rc;
  ReadStage* pst = nullptr;
  rc = acquire_stage(ctx, &pst);
  if (rc) return rc;
  ReadStage& st = *pst;
  rc = stage_columns(ctx, st, n, n_cig_total);
  if (rc) return rc;
  const int64_t n1 = std::max<int64_t>(n, 1);
  const int64_t off_len = off_len_of(n);
  const size_t crs_bytes = ((size_t)ctx->n_contigs + 1) * 8;
  // staging of the narrow columns: [contig_read_start | dpos u16 | n_cigar u8 | exc_index | exc_delta | cig u16]
  const size_t o_dpos = (crs_bytes + 15) & ~(size_t)15, o_nc = (o_dpos + (size_t)n1 * 2 + 15) & ~(size_t)15,
               o_ei = (o_nc + (size_t)n1 + 15) & ~(size_t)15, o_ed = (o_ei + (size_t)std::max<int64_t>(n_exc, 1) * 4 + 15) & ~(size_t)15,
               o_c16 = (o_ed + (size_t)std::max<int64_t>(n_exc, 1) * 4 + 15) & ~(size_t)15, x_bytes = o_c16 + (size_t)n_cig_total * 2 + 16;
  CU(st.raw.ensure(x_bytes));                                           // (part of the double-buffered stage: the copy of the next
                                                                        //  call must not land on columns this call's kernels still read)
  CU(ctx->d_start_slot.ensure((size_t)(off_len + 8) * 4));              // S (the record buffer of the fused pass: free until k_fused_prep)
  cudaStream_t cs = ctx->copy_stream;
  char* x = st.raw.as<char>();
  CU(cudaMemcpyAsync(x, contig_read_start, crs_bytes, cudaMemcpyHostToDevice, cs));
  if (n > 0) {
    CU(cudaMemcpyAsync(x + o_dpos, dpos, (size_t)n * 2, cudaMemcpyHostToDevice, cs));
    CU(cudaMemcpyAsync(x + o_nc, n_cigar, (size_t)n, cudaMemcpyHostToDevice, cs));
    if (n_exc) {
      CU(cudaMemcpyAsync(x + o_ei, exc_index, (size_t)n_exc * 4, cudaMemcpyHostToDevice, cs));
      CU(cudaMemcpyAsync(x + o_ed, exc_delta, (size_t)n_exc * 4, cudaMemcpyHostToDevice, cs));
    }
    CU(cudaMemcpyAsync(st.flag.p, flag, (size_t)n * 2, cudaMemcpyHostToDevice, cs));
    if (mapq) CU(cudaMemcpyAsync(st.mapq.p, mapq, (size_t)n, cudaMemcpyHostToDevice, cs));
    else CU(cudaMemsetAsync(st.mapq.p, 0xff, (size_t)n, cs));
    if (n_cig_total) CU(cudaMemcpyAsync(x + o_c16, cig, (size_t)n_cig_total * 2, cudaMemcpyHostToDevice, cs));
  }
  CU(cudaEventRecord(ctx->copied, cs));
  CU(cudaStreamWaitEvent(ctx->stream, ctx->copied, 0));
  cudaStream_t s = ctx->stream;
  int32_t* S = ctx->d_start_slot.as<int32_t>();
  const int64_t* d_crs = reinterpret_cast<const int64_t*>(x);
  ctx->prof_begin(kKDeltaUnpack);
  k_delta_seed<<<(unsigned)((off_len + 255) / 256), 256, 0, s>>>(n, d_crs, ctx->n_contigs, reinterpret_cast<const uint16_t*>(x + o_dpos),
                                                               reinterpret_cast<const uint8_t*>(x + o_nc), S, st.tid.as<int32_t>(),
                                                               st.cig_off.as<uint32_t>(), off_len);
  if (n_exc) k_delta_patch<<<(unsigned)((n_exc + 255) / 256), 256, 0, s>>>(n_exc, reinterpret_cast<const uint32_t*>(x + o_ei),
                                                                          reinterpret_cast<const int32_t*>(x + o_ed), n, S);
  ctx->prof_end();
  CU(cudaGetLastError());
  {
    const int64_t tiles = (off_len + kScanTile - 1) / kScanTile;
    CU(ctx->d_tile_cnt.ensure(((size_t)tiles + 1) * 16));             // two scans: status words + a ticket word each
    CU(cudaMemsetAsync(ctx->d_tile_cnt.p, 0, ((size_t)tiles + 1) * 16, s));
    unsigned long long* stw = ctx->d_tile_cnt.as<unsigned long long>();
    MCOV_LAUNCH(ctx, kKScanCounts, (k_scan_inplace<false><<<(unsigned)tiles, kScanThreads, 0, s>>>(st.cig_off.as<int32_t>(), off_len, stw, pc_of(ctx))));
    MCOV_LAUNCH(ctx, kKScanCounts, (k_scan_inplace<false><<<(unsigned)tiles, kScanThreads, 0, s>>>(S, off_len, stw + tiles + 1, pc_of(ctx))));
    CU(cudaGetLastError());
  }
  MCOV_LAUNCH(ctx, kKDeltaUnpack, (k_delta_finish<<<grid_for(ctx, std::max<int64_t>(n1, n_cig_total), 256, 8), 256, 0, s>>>(
      n, d_crs, ctx->n_contigs, st.tid.as<int32_t>(), S, st.pos.as<int32_t>(), reinterpret_cast<const uint16_t*>(x + o_c16),
      st.cig.as<uint32_t>(), n_cig_total)));
  CU(cudaGetLastError());
  return run_sorted_pass(ctx, columns_of(ctx, st, n, n_cig_total), &st, n, true, wait != 0, "mcov_depth_sorted_delta");
}

int mcov_begin_ex(mcov_ctx* ctx, int flags) {
  if (!ctx) return MCOV_ERR_ARG;
  if (flags & ~MCOV_BEGIN_EXACT_CAP) return fail(ctx, MCOV_ERR_ARG, "mcov_begin_ex: unknown flags");
  CU(cudaSetDevice(ctx->device));
  int rc = ensure_depth(ctx);
  if (rc) return rc;
  MCOV_LAUNCH(ctx, kKClear, CU(cudaMemsetAsync(ctx->depth, 0, (size_t)ctx->n_slots * 4, ctx->stream)));
  CU(cudaMemsetAsync(ctx->d_pc.p, 0, sizeof(PassCounters), ctx->stream));
  // the starts array of the exact cap metric: only where a cap exists and k_expand counts (count_del = 0 keeps the bound)
  ctx->exact_cap = (flags & MCOV_BEGIN_EXACT_CAP) && ctx->filt.max_depth > 0 && ctx->filt.count_del;
  if (ctx->exact_cap) {
    CU(ctx->d_starts.ensure((size_t)ctx->n_slots * 4));
    MCOV_LAUNCH(ctx, kKClear, CU(cudaMemsetAsync(ctx->d_starts.p, 0, (size_t)ctx->n_slots * 4, ctx->stream)));
  }
  ctx->n_reads_pushed = 0;
  ctx->verdict_pending = false;
  ctx->tile_hist_valid = false;
  ctx->state = kAccumulating;
  return MCOV_OK;
}

int mcov_begin(mcov_ctx* ctx) { return mcov_begin_ex(ctx, 0); }

static int push_reads_impl(mcov_ctx* ctx, int64_t n, const int32_t* tid, const int32_t* pos, const uint16_t* flag,
                           const uint8_t* mapq, const void* cig_off, bool off64, const uint32_t* cig, int mem_kind) {
  if (!ctx) return MCOV_ERR_ARG;
  if (ctx->state != kAccumulating) return fail(ctx, MCOV_ERR_STATE, "mcov_push_reads: call mcov_begin first");
  if (n < 0) return fail(ctx, MCOV_ERR_ARG, "mcov_push_reads: n < 0");
  if (n == 0) return MCOV_OK;
  if (!tid || !pos || !flag || !mapq || !cig_off) return fail(ctx, MCOV_ERR_ARG, "mcov_push_reads: null array");
  CU(cudaSetDevice(ctx->device));
  ctx->tile_hist_valid = false;
  ExpandArgs a;
  ReadStage* st = nullptr;
  int rc = stage_reads(ctx, n, tid, pos, flag, mapq, cig_off, off64, cig, mem_kind, a, &st);
  if (rc) return rc;
  FusedArgs f;
  std::memset(&f, 0, sizeof(f));
  f.e = a;
  f.vec_ok = vec_ok(a);
  const int grid = grid_for(ctx, (n + kPrepPer - 1) / kPrepPer, kPrepThreads, 8);
  // a filter changed inside the pass so that starts are no longer counted (count_del = 0, or no cap): the pass keeps the
  // scan's bound rather than report a metric over starts that miss these reads
  if (ctx->exact_cap && (!ctx->filt.count_del || ctx->filt.max_depth <= 0)) ctx->exact_cap = false;
  if (!ctx->filt.count_del) MCOV_LAUNCH(ctx, kKExpand, (k_expand_runs<<<grid_for(ctx, n, 256, 8), 256, 0, ctx->stream>>>(f, 0)));
  else if (ctx->exact_cap) {
    f.starts = ctx->d_starts.as<int32_t>();
    if (off64) MCOV_LAUNCH(ctx, kKExpand, (k_expand<true, true><<<grid, kPrepThreads, 0, ctx->stream>>>(f)));
    else MCOV_LAUNCH(ctx, kKExpand, (k_expand<false, true><<<grid, kPrepThreads, 0, ctx->stream>>>(f)));
  } else if (off64) MCOV_LAUNCH(ctx, kKExpand, (k_expand<true, false><<<grid, kPrepThreads, 0, ctx->stream>>>(f)));
  else MCOV_LAUNCH(ctx, kKExpand, (k_expand<false, false><<<grid, kPrepThreads, 0, ctx->stream>>>(f)));
  CU(cudaGetLastError());
  ctx->n_reads_pushed += n;
  return finish_stage(ctx, st);
}

int mcov_push_reads(mcov_ctx* ctx, int64_t n, const int32_t* tid, const int32_t* pos, const uint16_t* flag,
                    const uint8_t* mapq, const uint32_t* cig_off, const uint32_t* cig, int mem_kind) {
  return push_reads_impl(ctx, n, tid, pos, flag, mapq, cig_off, false, cig, mem_kind);
}

int mcov_push_reads_wide(mcov_ctx* ctx, int64_t n, const int32_t* tid, const int32_t* pos, const uint16_t* flag,
                         const uint8_t* mapq, const uint64_t* cig_off, const uint32_t* cig, int mem_kind) {
  return push_reads_impl(ctx, n, tid, pos, flag, mapq, cig_off, true, cig, mem_kind);
}

int mcov_finalize(mcov_ctx* ctx) {
  if (!ctx) return MCOV_ERR_ARG;
  if (ctx->state != kAccumulating) return fail(ctx, MCOV_ERR_STATE, "mcov_finalize: nothing accumulated");
  CU(cudaSetDevice(ctx->device));
  ctx->tile_hist_valid = false;
  int rc = scan_depth(ctx);
  if (rc) return rc;
  if (ctx->exact_cap) {                  // the scan's bound is replaced by the exact value
    CU(cudaMemsetAsync(&pc_of(ctx)->cap_metric, 0, sizeof(int), ctx->stream));
    MCOV_LAUNCH(ctx, kKCapExact, (k_cap_exact<<<grid_for(ctx, ctx->n_slots / 4, 256, 8), 256, 0, ctx->stream>>>(
        ctx->depth, ctx->d_starts.as<int32_t>(), ctx->n_slots, pc_of(ctx))));
    CU(cudaGetLastError());
  }
  ctx->state = kDepthReady;
  return MCOV_OK;
}

static int depth_sorted_impl(mcov_ctx* ctx, int64_t n, const int32_t* tid, const int32_t* pos, const uint16_t* flag,
                             const uint8_t* mapq, const void* cig_off, bool off64, const uint32_t* cig, int mem_kind, bool wait) {
  if (!ctx) return MCOV_ERR_ARG;
  if (n < 0) return fail(ctx, MCOV_ERR_ARG, "mcov_depth_sorted: n < 0");
  if (n > 0 && (!tid || !pos || !flag || !mapq || !cig_off)) return fail(ctx, MCOV_ERR_ARG, "mcov_depth_sorted: null array");
  CU(cudaSetDevice(ctx->device));
  int rc = ensure_depth(ctx);
  if (rc) return rc;
  ExpandArgs a;
  ReadStage* st = nullptr;
  rc = stage_reads(ctx, n, tid, pos, flag, mapq, cig_off, off64, cig, mem_kind, a, &st);
  if (rc) return rc;
  return run_sorted_pass(ctx, a, st, n, true, wait, "mcov_depth_sorted");
}

int mcov_depth_sorted(mcov_ctx* ctx, int64_t n, const int32_t* tid, const int32_t* pos, const uint16_t* flag,
                      const uint8_t* mapq, const uint32_t* cig_off, const uint32_t* cig, int mem_kind) {
  return depth_sorted_impl(ctx, n, tid, pos, flag, mapq, cig_off, false, cig, mem_kind, true);
}

int mcov_depth_sorted_wide(mcov_ctx* ctx, int64_t n, const int32_t* tid, const int32_t* pos, const uint16_t* flag,
                           const uint8_t* mapq, const uint64_t* cig_off, const uint32_t* cig, int mem_kind, int wait) {
  return depth_sorted_impl(ctx, n, tid, pos, flag, mapq, cig_off, true, cig, mem_kind, wait != 0);
}

int mcov_depth_sorted_async(mcov_ctx* ctx, int64_t n, const int32_t* tid, const int32_t* pos, const uint16_t* flag,
                            const uint8_t* mapq, const uint32_t* cig_off, const uint32_t* cig, int mem_kind) {
  return depth_sorted_impl(ctx, n, tid, pos, flag, mapq, cig_off, false, cig, mem_kind, false);
}

// ---- streaming a coordinate-sorted file in batches ------------------------------------------------------------
int mcov_stream_begin(mcov_ctx* ctx) {
  if (!ctx) return MCOV_ERR_ARG;
  CU(cudaSetDevice(ctx->device));
  int rc = ensure_depth(ctx);
  if (rc) return rc;
  CU(ctx->d_stream_acc.ensure(sizeof(StreamAcc) + 16));
  CU(cudaMemsetAsync(ctx->d_stream_acc.p, 0, sizeof(StreamAcc) + 16, ctx->stream));
  ctx->stream_tile_lo = 0;
  ctx->stream_reads = 0;
  ctx->stream_started = false;
  CU(cudaMemsetAsync(ctx->d_pc.p, 0, sizeof(PassCounters), ctx->stream));
  ctx->verdict_pending = false;
  ctx->tile_hist_valid = false;
  ctx->state = kStreaming;
  return MCOV_OK;
}

int mcov_stream_resend_point(const mcov_ctx* ctx, int32_t last_tid, int32_t last_pos, int32_t* resend_tid, int32_t* resend_pos) {
  if (!ctx || !resend_tid || !resend_pos || ctx->n_contigs <= 0) return MCOV_ERR_ARG;
  const int64_t tb = stream_tile_of(ctx, last_tid, last_pos);
  // everything that starts at or after the first slot of tile tb-1, or reaches past it, is needed again
  const int64_t rs = std::max<int64_t>(tb - 1, 0) << kTileShift;
  if (rs >= ctx->n_slots) { *resend_tid = ctx->n_contigs; *resend_pos = 0; return MCOV_OK; }
  const int32_t c = (int32_t)(std::upper_bound(ctx->off.begin(), ctx->off.begin() + ctx->n_contigs, rs) - ctx->off.begin()) - 1;
  *resend_tid = c;
  *resend_pos = (int32_t)std::min<int64_t>(rs - ctx->off[c], ctx->len[c]);
  return MCOV_OK;
}

// the part of a stream push that follows the staging of the batch (`a` = device columns)
static int stream_push_staged(mcov_ctx* ctx, const ExpandArgs& a, ReadStage* st, int64_t n, int64_t n_carry, int32_t lt, int32_t lp,
                              int last, int32_t* resend_tid, int32_t* resend_pos, bool wait_copy = true) {
  ctx->tile_hist_valid = false;
  const int64_t n_tiles = (ctx->n_slots + kTile - 1) / kTile;
  int64_t tile_hi = n_tiles;
  if (!last) {
    tile_hi = n == 0 ? ctx->stream_tile_lo : stream_tile_of(ctx, lt, lp);
    if (tile_hi < ctx->stream_tile_lo) {
      ctx->state = kIdle;
      return fail(ctx, MCOV_ERR_UNSORTED, "mcov_stream_push: the batch ends before the previous one (batches must follow the sorted order)");
    }
  }
  if (resend_tid && resend_pos) {
    if (n > 0) mcov_stream_resend_point(ctx, lt, lp, resend_tid, resend_pos);
    else { *resend_tid = -1; *resend_pos = 0; }                  // (an empty batch changes nothing: keep sending what was being sent)
  }
  if (!ctx->filt.count_del) {
    // M = X positions only: the batches accumulate in the difference array (carried reads skipped), the last one scans
    int rc = runs_depth(ctx, a, n_carry, ctx->stream_reads == 0 && ctx->stream_tile_lo == 0 && !ctx->stream_started, last != 0);
    if (rc) return rc;
    ctx->stream_started = true;
  } else {
    CU(cudaMemsetAsync(ctx->d_pc.p, 0, sizeof(PassCounters), ctx->stream));
    int rc = fused_depth_sorted(ctx, a, ctx->stream_tile_lo, tile_hi);
    if (rc) return rc;
    // pass counters of the stream: this batch minus its carried reads, added to the running totals
    unsigned long long* carry = reinterpret_cast<unsigned long long*>(ctx->d_stream_acc.as<char>() + sizeof(StreamAcc));
    CU(cudaMemsetAsync(carry, 0, 16, ctx->stream));
    FusedArgs f;
    std::memcpy(&f, ctx->fused_blob.data(), sizeof(f));
    if (n_carry > 0) {
      MCOV_LAUNCH(ctx, kKStreamAcc, (k_carry_counts<<<grid_for(ctx, n_carry, 256, 4), 256, 0, ctx->stream>>>(f, n_carry, carry)));
      CU(cudaGetLastError());
    }
    MCOV_LAUNCH(ctx, kKStreamAcc, (k_stream_accumulate<<<1, 1, 0, ctx->stream>>>(pc_of(ctx), ctx->d_stream_acc.as<StreamAcc>(), carry, f.far_cap)));
    CU(cudaGetLastError());
  }
  ctx->stream_reads += n - n_carry;
  ctx->n_reads_pushed = ctx->stream_reads;
  ctx->stream_tile_lo = tile_hi;
  int rc = finish_stage(ctx, st, wait_copy);
  if (rc) return rc;
  if (last) {
    ctx->state = kDepthReady;
    ctx->verdict_pending = true;                                 // delivered by the next synchronising call, like mcov_depth_sorted_async
  }
  return MCOV_OK;
}

int mcov_stream_push(mcov_ctx* ctx, int64_t n, int64_t n_carry, const int32_t* tid, const int32_t* pos, const uint16_t* flag,
                     const uint8_t* mapq, const uint32_t* cig_off, const uint32_t* cig, int mem_kind, int last,
                     int32_t* resend_tid, int32_t* resend_pos) {
  if (!ctx) return MCOV_ERR_ARG;
  if (ctx->state != kStreaming) return fail(ctx, MCOV_ERR_STATE, "mcov_stream_push: call mcov_stream_begin first");
  if (n < 0 || n_carry < 0 || n_carry > n) return fail(ctx, MCOV_ERR_ARG, "mcov_stream_push: need 0 <= n_carry <= n");
  if (n > 0 && (!tid || !pos || !flag || !mapq || !cig_off)) return fail(ctx, MCOV_ERR_ARG, "mcov_stream_push: null array");
  CU(cudaSetDevice(ctx->device));
  // the batch's last read decides how far the depth becomes final
  int32_t lt = -1, lp = 0;
  if (n > 0) {
    if (mem_kind == MCOV_MEM_HOST) { lt = tid[n - 1]; lp = pos[n - 1]; }
    else {
      CU(cudaMemcpyAsync(&lt, tid + n - 1, 4, cudaMemcpyDeviceToHost, ctx->stream));
      CU(cudaMemcpyAsync(&lp, pos + n - 1, 4, cudaMemcpyDeviceToHost, ctx->stream));
      CU(cudaStreamSynchronize(ctx->stream));
    }
  }
  ExpandArgs a;
  ReadStage* st = nullptr;
  int rc = stage_reads(ctx, n, tid, pos, flag, mapq, cig_off, false, cig, mem_kind, a, &st);
  if (rc) return rc;
  return stream_push_staged(ctx, a, st, n, n_carry, lt, lp, last, resend_tid, resend_pos);
}

int mcov_stream_push_block(mcov_ctx* ctx, const void* block, int64_t bytes, int last, int32_t* resend_tid, int32_t* resend_pos) {
  if (!ctx) return MCOV_ERR_ARG;
  if (ctx->state != kStreaming) return fail(ctx, MCOV_ERR_STATE, "mcov_stream_push_block: call mcov_stream_begin first");
  CU(cudaSetDevice(ctx->device));
  ExpandArgs a;
  ReadStage* st = nullptr;
  mcov_block_hdr h;
  int rc = block_stage(ctx, block, bytes, a, &st, h);
  if (rc) return rc;
  return stream_push_staged(ctx, a, st, h.n, h.n_carry, h.last_tid, h.last_pos, last, resend_tid, resend_pos, /*wait_copy=*/false);
}

int mcov_block_unpack(mcov_ctx* ctx, const void* block, int64_t bytes, int32_t* tid, int32_t* pos, uint16_t* flag,
                      uint8_t* mapq, uint32_t* cig_off, uint32_t* cig) {
  if (!ctx) return MCOV_ERR_ARG;
  CU(cudaSetDevice(ctx->device));
  ExpandArgs a;
  ReadStage* st = nullptr;
  mcov_block_hdr h;
  int rc = block_stage(ctx, block, bytes, a, &st, h);
  if (rc) return rc;
  cudaStream_t s = ctx->stream;
  const size_t n = (size_t)h.n;
  if (n) {
    if (tid) CU(cudaMemcpyAsync(tid, a.tid, n * 4, cudaMemcpyDeviceToHost, s));
    if (pos) CU(cudaMemcpyAsync(pos, a.pos, n * 4, cudaMemcpyDeviceToHost, s));
    if (flag) CU(cudaMemcpyAsync(flag, a.flag, n * 2, cudaMemcpyDeviceToHost, s));
    if (mapq) CU(cudaMemcpyAsync(mapq, a.mapq, n, cudaMemcpyDeviceToHost, s));
  }
  if (cig_off) CU(cudaMemcpyAsync(cig_off, a.cig_off, (n + 1) * 4, cudaMemcpyDeviceToHost, s));
  if (cig && h.n_cigar) CU(cudaMemcpyAsync(cig, a.cig, (size_t)h.n_cigar * 4, cudaMemcpyDeviceToHost, s));
  rc = finish_stage(ctx, st, /*wait_copy=*/true);
  if (rc) return rc;
  CU(cudaStreamSynchronize(s));
  return MCOV_OK;
}

int mcov_depth_sorted_block(mcov_ctx* ctx, const void* block, int64_t bytes, int wait) {
  if (!ctx) return MCOV_ERR_ARG;
  CU(cudaSetDevice(ctx->device));
  int rc = ensure_depth(ctx);
  if (rc) return rc;
  ExpandArgs a;
  ReadStage* st = nullptr;
  mcov_block_hdr h;
  rc = block_stage(ctx, block, bytes, a, &st, h);
  if (rc) return rc;
  return run_sorted_pass(ctx, a, st, h.n, /*wait_copy=*/false, wait != 0, "mcov_depth_sorted_block");
}

int mcov_depth_sorted_packed(mcov_ctx* ctx, int64_t n, const int64_t* contig_read_start, const int32_t* pos,
                             const uint16_t* flag, const uint8_t* mapq, const uint16_t* n_cigar, const uint32_t* cig,
                             int64_t n_cig_total, int wait) {
  if (!ctx) return MCOV_ERR_ARG;
  if (n < 0 || n_cig_total < 0 || n_cig_total > 0xFFFFFFFFll) return fail(ctx, MCOV_ERR_ARG, "mcov_depth_sorted_packed: bad sizes");
  if (!contig_read_start || (n > 0 && (!pos || !flag || !n_cigar)) || (n_cig_total > 0 && !cig))
    return fail(ctx, MCOV_ERR_ARG, "mcov_depth_sorted_packed: null array");
  CU(cudaSetDevice(ctx->device));
  int rc = ensure_depth(ctx);
  if (rc) return rc;
  rc = check_narrow(ctx, n, contig_read_start, n_cigar, n_cig_total, mapq, "mcov_depth_sorted_packed");
  if (rc) return rc;
  ReadStage* pst = nullptr;
  rc = acquire_stage(ctx, &pst);
  if (rc) return rc;
  ReadStage& st = *pst;
  rc = stage_columns(ctx, st, n, n_cig_total);
  if (rc) return rc;
  const int64_t off_len = off_len_of(n);
  const size_t crs_bytes = ((size_t)ctx->n_contigs + 1) * 8;
  CU(st.raw.ensure((size_t)std::max<int64_t>(n, 1) * 2 + crs_bytes + 16));     // [contig_read_start | n_cigar]
  cudaStream_t cs = ctx->copy_stream;
  char* extra = st.raw.as<char>();
  CU(cudaMemcpyAsync(extra, contig_read_start, crs_bytes, cudaMemcpyHostToDevice, cs));
  if (n > 0) {
    CU(cudaMemcpyAsync(extra + crs_bytes, n_cigar, (size_t)n * 2, cudaMemcpyHostToDevice, cs));
    CU(cudaMemcpyAsync(st.pos.p, pos, (size_t)n * 4, cudaMemcpyHostToDevice, cs));
    CU(cudaMemcpyAsync(st.flag.p, flag, (size_t)n * 2, cudaMemcpyHostToDevice, cs));
    if (mapq) CU(cudaMemcpyAsync(st.mapq.p, mapq, (size_t)n, cudaMemcpyHostToDevice, cs));
    else CU(cudaMemsetAsync(st.mapq.p, 0xff, (size_t)n, cs));
    if (n_cig_total) CU(cudaMemcpyAsync(st.cig.p, cig, (size_t)n_cig_total * 4, cudaMemcpyHostToDevice, cs));
  }
  CU(cudaEventRecord(ctx->copied, cs));
  CU(cudaStreamWaitEvent(ctx->stream, ctx->copied, 0));
  cudaStream_t s = ctx->stream;
  // rebuild tid[] and cig_off[] on the device
  MCOV_LAUNCH(ctx, kKUnpack, (k_unpack_reads<<<(unsigned)((off_len + 255) / 256), 256, 0, s>>>(
      n, reinterpret_cast<const int64_t*>(extra), ctx->n_contigs, reinterpret_cast<const uint16_t*>(extra + crs_bytes),
      st.tid.as<int32_t>(), st.cig_off.as<uint32_t>(), off_len)));
  CU(cudaGetLastError());
  {
    const int64_t tiles = (off_len + kScanTile - 1) / kScanTile;
    CU(ctx->d_tile_cnt.ensure(((size_t)tiles + 1) * 8));              // status words + the ticket word
    CU(cudaMemsetAsync(ctx->d_tile_cnt.p, 0, ((size_t)tiles + 1) * 8, s));
    MCOV_LAUNCH(ctx, kKScanCounts, (k_scan_inplace<false><<<(unsigned)tiles, kScanThreads, 0, s>>>(
        st.cig_off.as<int32_t>(), off_len, ctx->d_tile_cnt.as<unsigned long long>(), pc_of(ctx))));
    CU(cudaGetLastError());
  }
  return run_sorted_pass(ctx, columns_of(ctx, st, n, n_cig_total), &st, n, true, wait != 0, "mcov_depth_sorted_packed");
}

int mcov_pass_info_get(mcov_ctx* ctx, mcov_pass_info* out) {
  if (!ctx || !out) return fail(ctx, MCOV_ERR_ARG, "mcov_pass_info_get: null argument");
  if (ctx->state == kIdle) return fail(ctx, MCOV_ERR_STATE, "mcov_pass_info_get: no pass has run");
  CU(cudaSetDevice(ctx->device));
  PassCounters h;
  { int vr = sync_verdict(ctx, "mcov_pass_info_get", &h); if (vr) return vr; }
  out->n_reads = ctx->n_reads_pushed;
  out->n_pass = (int64_t)h.n_pass;
  out->aligned_bases = (int64_t)h.aligned_bases;
  out->max_depth_seen = h.max_depth_seen;
  out->cap_metric = h.cap_metric;
  out->sorted = h.unsorted ? 0 : 1;
  out->cap_contigs = ctx->cap_contigs;
  return MCOV_OK;
}

static const char* kKernelNames[kKernelCount] = {
    "k_expand", "k_scan_inplace", "k_fused_prep", "k_scan_counts", "k_far_scatter",
    "k_window_sums", "k_isize_hist", "k_group_count", "k_sorted_stats",
    "memset_depth", "k_region_stats_small", "k_cap_replay", "k_unpack_reads", "k_kmer_hist", "k_region_stats_warp",
    "k_exp_prep", "k_exp_entries", "k_exp_region", "k_exp_revsum", "k_region_hist", "k_hist_finish", "k_run_count", "k_run_offsets", "k_run_write", "k_run_ends",
    "k_bgzf_inflate", "k_bam_guess", "k_bam_walk_count", "k_bam_walk_write", "k_delta_unpack", "k_stream_accumulate",
    "k_fused_prep_tma", "k_fused_tile_tma", "k_stats_stream", "k_block_unpack", "k_bam_names_seq",
    "k_sam_nl_count", "k_sam_nl_write", "k_sam_fields", "k_sam_cigar", "k_sam_names_seq", "k_dev_map_counts",
    "k_cap_exact", "k_sam_line_max",
    "k_bc_any",
    "k_ref_encode", "k_allele_chunks", "k_allele_combine", "k_allele_site_count", "k_allele_site_write",
    "k_allele_signature", "k_compare_chunks", "k_compare_combine", "k_compare_site_count", "k_compare_site_write"};

int mcov_copy_to_host(mcov_ctx* ctx, const void* dev, void* host, int64_t n_bytes) {
  if (!ctx) return MCOV_ERR_ARG;
  if (n_bytes < 0 || (n_bytes > 0 && (!dev || !host))) return fail(ctx, MCOV_ERR_ARG, "mcov_copy_to_host: bad arguments");
  if (n_bytes == 0) return MCOV_OK;
  CU(cudaSetDevice(ctx->device));
  CU(cudaMemcpyAsync(host, dev, (size_t)n_bytes, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return MCOV_OK;
}

int mcov_sync(mcov_ctx* ctx) {
  if (!ctx) return MCOV_ERR_ARG;
  CU(cudaSetDevice(ctx->device));
  { int wrc = wait_pending_copy(ctx); if (wrc) return wrc; }
  CU(cudaStreamSynchronize(ctx->stream));
  return MCOV_OK;
}

int64_t mcov_launch_count(const mcov_ctx* ctx) { return ctx ? ctx->n_launches : 0; }

int mcov_profile_enable(mcov_ctx* ctx, int on) {
  if (!ctx) return MCOV_ERR_ARG;
  CU(cudaSetDevice(ctx->device));
  CU(cudaStreamSynchronize(ctx->stream));
  ctx->prof_collect();
  ctx->profiling = on != 0;
  if (on) for (int k = 0; k < kKernelCount; ++k) { ctx->prof_ms[k] = 0; ctx->prof_n[k] = 0; }
  return MCOV_OK;
}

int mcov_profile_read(mcov_ctx* ctx, mcov_kernel_time* out, int cap) {
  if (!ctx || (cap > 0 && !out)) return MCOV_ERR_ARG;
  CU(cudaSetDevice(ctx->device));
  CU(cudaStreamSynchronize(ctx->stream));
  ctx->prof_collect();
  int n = 0;
  for (int k = 0; k < kKernelCount && n < cap; ++k) {
    if (!ctx->prof_n[k]) continue;
    std::snprintf(out[n].name, sizeof(out[n].name), "%s", kKernelNames[k]);
    out[n].launches = ctx->prof_n[k];
    out[n].total_ms = ctx->prof_ms[k];
    ++n;
  }
  return n;
}

int32_t* mcov_depth_ptr(mcov_ctx* ctx) {
  if (!ctx || ctx->state != kDepthReady) return nullptr;
  ctx->tile_hist_valid = false;           // the caller may write the depth: statistics read it again
  return ctx->depth;
}

int mcov_copy_depth(mcov_ctx* ctx, int32_t tid, int32_t start, int32_t end, int32_t* host_out) {
  if (!ctx) return MCOV_ERR_ARG;
  if (ctx->state != kDepthReady) return fail(ctx, MCOV_ERR_STATE, "mcov_copy_depth: depth not ready (finalize first)");
  if (tid < 0 || tid >= ctx->n_contigs || start < 0 || end < start || end > ctx->len[tid] || (!host_out && end > start))
    return fail(ctx, MCOV_ERR_ARG, "mcov_copy_depth: region out of range");
  if (end == start) return MCOV_OK;
  CU(cudaSetDevice(ctx->device));
  CU(cudaMemcpyAsync(host_out, ctx->depth + ctx->off[tid] + start, (size_t)(end - start) * 4, cudaMemcpyDeviceToHost,
                     ctx->stream));
  return sync_verdict(ctx, "mcov_copy_depth");
}

// Build (or reuse) the plan of a region set and enqueue the statistics kernels writing g
// records to d_out (device memory).
static int stats_launch(mcov_ctx* ctx, int64_t g, const int32_t* tid, const int32_t* start, const int32_t* end,
                        int32_t breadth_n, mcov_region_stats* d_out, const char* who) {
  cudaStream_t s = ctx->stream;
  RegionPlan& rp = ctx->plan;
  // The plan of a region set is cached on the device: a caller that asks for the same
  // regions again (cli.py loops, benchmarks) pays for it once.
  const bool same = rp.valid && rp.g == g && rp.n_contigs_epoch == ctx->contig_epoch && g > 0 &&
                    std::memcmp(rp.tid.data(), tid, (size_t)g * 4) == 0 &&
                    std::memcmp(rp.start.data(), start, (size_t)g * 4) == 0 &&
                    std::memcmp(rp.end.data(), end, (size_t)g * 4) == 0;
  if (!same && g > 0) {
    rp.valid = false;
    int rc = check_regions(ctx, g, tid, start, end, who);
    if (rc) return rc;
    // A region is LARGE (k_stats_stream) when more than kSmallRegion of its slots lie inside the
    // contig, SMALL (k_region_stats_warp) when it has fewer but at least one slot or one padding
    // position; a region with neither is in no list.
    std::vector<StatTask> small;
    rp.rlen.assign((size_t)g, 0); rp.rpad.assign((size_t)g, 0);
    for (int64_t i = 0; i < g; ++i) {
      const Clip c = clip_region(ctx, tid[i], start[i], end[i]);
      rp.rlen[i] = (int32_t)c.n; rp.rpad[i] = c.pad;
      if (c.n <= kSmallRegion && c.n + c.pad > 0) {
        StatTask t;
        t.slot = ctx->off[tid[i]] + c.cs; t.n = (int32_t)c.n; t.region = (int32_t)i;
        small.push_back(t);
      }
    }
    // The balanced stream over the large regions (k_stats_stream.cuh): their concatenation cut into equal slices,
    // one per persistent CTA; a region cut by a slice border becomes a "split" region with a global histogram.
    int64_t total_big = 0;
    for (int64_t i = 0; i < g; ++i) if (rp.rlen[i] > kSmallRegion) total_big += rp.rlen[i];
    std::vector<SsPiece> pieces;
    std::vector<int32_t> cta_start, split_npieces;
    const int32_t grid = (int32_t)std::min<int64_t>((int64_t)ctx->n_sm * MCOV_SS_CTAS, std::max<int64_t>(1, total_big / 16384));
    const int64_t W = std::max<int64_t>(4, ((total_big + grid - 1) / grid + 3) & ~(int64_t)3);
    int64_t room = W;
    cta_start.push_back(0);
    for (int64_t i = 0; i < g && total_big > 0; ++i) {
      if (rp.rlen[i] <= kSmallRegion) continue;
      int64_t rem = rp.rlen[i];
      int64_t slot = ctx->off[tid[i]] + clip_region(ctx, tid[i], start[i], end[i]).cs;
      const size_t first_piece = pieces.size();
      while (rem > 0) {
        const int64_t take = std::min(rem, room);
        SsPiece pc;
        pc.slot = slot; pc.n = (int32_t)take; pc.region = (int32_t)i; pc.pad = pieces.size() == first_piece ? rp.rpad[i] : 0; pc.split = -1;
        pieces.push_back(pc);
        rem -= take; slot += take; room -= take;
        if (room == 0) { cta_start.push_back((int32_t)pieces.size()); room = W; }
      }
      if (pieces.size() - first_piece > 1) {
        const int32_t id = (int32_t)split_npieces.size();
        split_npieces.push_back((int32_t)(pieces.size() - first_piece));
        for (size_t k = first_piece; k < pieces.size(); ++k) pieces[k].split = id;
      }
    }
    if (cta_start.back() != (int32_t)pieces.size()) cta_start.push_back((int32_t)pieces.size());
    rp.ss_grid = total_big > 0 ? (int32_t)cta_start.size() - 1 : 0;
    rp.n_split = (int32_t)split_npieces.size();
    // tiles that lie wholly inside a large region (overlapping regions may count a tile twice): decide whether the fused
    // passes that follow count depth histograms
    rp.hist_tiles = 0;
    for (const SsPiece& pc : pieces) rp.hist_tiles += std::max<int64_t>(0, ((pc.slot + pc.n) >> kTileShift) - ((pc.slot + kTile - 1) >> kTileShift));
    if (rp.ss_grid > 0) {
      CU(ctx->d_ss_pieces.ensure(pieces.size() * sizeof(SsPiece)));
      CU(ctx->d_ss_cta.ensure(cta_start.size() * 4));
      CU(ctx->d_ss_split.ensure(std::max<size_t>(split_npieces.size(), 1) * 4));      // pieces of each split region
      CU(ctx->d_ss_pool.ensure((size_t)std::max(rp.n_split, 1) * (sizeof(RegionScratch) + (size_t)kHistBins * 4)));
      CU(cudaMemcpyAsync(ctx->d_ss_pieces.p, pieces.data(), pieces.size() * sizeof(SsPiece), cudaMemcpyHostToDevice, s));
      CU(cudaMemcpyAsync(ctx->d_ss_cta.p, cta_start.data(), cta_start.size() * 4, cudaMemcpyHostToDevice, s));
      if (rp.n_split) {
        CU(cudaMemcpyAsync(ctx->d_ss_split.p, split_npieces.data(), split_npieces.size() * 4, cudaMemcpyHostToDevice, s));
        CU(cudaMemsetAsync(ctx->d_ss_pool.p, 0, (size_t)rp.n_split * (sizeof(RegionScratch) + (size_t)kHistBins * 4), s));
      }
    }
    // Largest regions first, and neighbours of similar size: a CTA of 8 warps lives as long as its largest
    // region, and with the log-normal contig lengths of config C3 an unsorted CTA keeps its slots for about
    // twice the mean of its regions.
    auto by_size = [](const StatTask& x, const StatTask& y) { return x.n > y.n; };
    if (!std::is_sorted(small.begin(), small.end(), by_size)) std::stable_sort(small.begin(), small.end(), by_size);
    rp.n_small = (int64_t)small.size();
    CU(ctx->d_out.ensure((size_t)g * sizeof(mcov_region_stats)));
    CU(ctx->d_tasks.ensure(std::max<size_t>(small.size(), 1) * sizeof(StatTask)));
    CU(ctx->d_rlen.ensure((size_t)g * 8));
    int32_t* d_rlen = ctx->d_rlen.as<int32_t>();
    if (!small.empty()) CU(cudaMemcpyAsync(ctx->d_tasks.p, small.data(), small.size() * sizeof(StatTask), cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(d_rlen, rp.rlen.data(), (size_t)g * 4, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(d_rlen + g, rp.rpad.data(), (size_t)g * 4, cudaMemcpyHostToDevice, s));
    CU(cudaStreamSynchronize(s));                   // the host vectors above go out of scope
    rp.tid.assign(tid, tid + g); rp.start.assign(start, start + g); rp.end.assign(end, end + g);
    rp.g = g; rp.n_contigs_epoch = ctx->contig_epoch; rp.valid = true; rp.id = ++ctx->plan_serial;
  }
  if (g > 0) {
    if (rp.ss_grid > 0) {
      SsArgs a;
      int32_t* d_rlen = ctx->d_rlen.as<int32_t>();
      a.depth = ctx->depth; a.pieces = ctx->d_ss_pieces.as<SsPiece>(); a.cta_piece_start = ctx->d_ss_cta.as<int32_t>();
      a.region_len = d_rlen; a.region_pad = d_rlen + g;
      a.split_scratch = ctx->d_ss_pool.as<RegionScratch>();
      a.split_hist = reinterpret_cast<uint32_t*>(ctx->d_ss_pool.as<char>() + (size_t)rp.n_split * sizeof(RegionScratch));
      a.split_pieces = ctx->d_ss_split.as<int32_t>();
      // (histograms exist only for the tiles of the plan the pass was run with)
      a.tile_hist = ctx->tile_hist_valid && ctx->tile_hist_plan == rp.id ? ctx->d_tile_hist.as<uint16_t>() : nullptr;
      a.out = d_out; a.breadth_n = breadth_n;
      const bool pdl = ctx->n_slots <= kPdlMaxSlots;
      MCOV_LAUNCH(ctx, kKStatsStream, CU(launch_pdl(pdl, k_stats_stream, dim3((unsigned)rp.ss_grid), dim3(kSsThreads), (size_t)kSsSmemBytes, s, a)));
    }
    if (rp.n_small) {
      StatArgs a;
      int32_t* d_rlen = ctx->d_rlen.as<int32_t>();
      a.depth = ctx->depth; a.tasks = ctx->d_tasks.as<StatTask>(); a.region_len = d_rlen; a.region_pad = d_rlen + g;
      a.out = d_out; a.breadth_n = breadth_n;
      // one warp per region first; regions whose depth range does not fit a warp's window are
      // collected in a retry list (device side) and finished by the CTA-per-region kernel
      CU(ctx->d_done.ensure(((size_t)rp.n_small + 1) * 4));
      uint32_t* retry = ctx->d_done.as<uint32_t>();
      CU(cudaMemsetAsync(retry, 0, 4, s));
      const unsigned wgrid = (unsigned)((rp.n_small + kWarpsPerCta - 1) / kWarpsPerCta);
      MCOV_LAUNCH(ctx, kKRegionStatsWarp, (k_region_stats_warp<<<wgrid, kWarpsPerCta * 32, 0, s>>>(a, rp.n_small, retry)));
      CU(cudaGetLastError());
      const unsigned rgrid = (unsigned)std::min<int64_t>(rp.n_small, (int64_t)ctx->n_sm * 6);
      MCOV_LAUNCH(ctx, kKRegionStatsSmall, (k_region_stats_small<<<rgrid, kSmallThreads, 0, s>>>(a, retry)));
      CU(cudaGetLastError());
    }
  }
  return MCOV_OK;
}

int mcov_region_stats_run(mcov_ctx* ctx, int64_t g, const int32_t* tid, const int32_t* start, const int32_t* end,
                          int32_t breadth_n, mcov_region_stats* host_out) {
  if (!ctx) return MCOV_ERR_ARG;
  if (ctx->state != kDepthReady) return fail(ctx, MCOV_ERR_STATE, "mcov_region_stats_run: depth not ready (finalize first)");
  if (g < 0 || (g > 0 && (!tid || !start || !end || !host_out))) return fail(ctx, MCOV_ERR_ARG, "mcov_region_stats_run: bad arguments");
  if (g > INT32_MAX) return fail(ctx, MCOV_ERR_RANGE, "mcov_region_stats_run: more than 2^31-1 regions");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  // Results and the pending verdict come back through pinned memory (a pageable destination would
  // make the copy synchronous and slow): straight into host_out when the caller's buffer is itself
  // pinned, else through the context's staging buffer.
  const size_t out_bytes = (size_t)g * sizeof(mcov_region_stats);
  bool direct = false;
  if (g > 0) {
    cudaPointerAttributes pa;
    if (cudaPointerGetAttributes(&pa, host_out) == cudaSuccess) direct = (pa.type == cudaMemoryTypeHost);
    else (void)cudaGetLastError();
  }
  CU(ctx->h_pin.ensure((direct ? 0 : out_bytes) + sizeof(PassCounters)));
  char* stage = ctx->h_pin.as<char>();
  if (g > 0) {
    CU(ctx->d_out.ensure(out_bytes));
    int rc = stats_launch(ctx, g, tid, start, end, breadth_n, ctx->d_out.as<mcov_region_stats>(), "mcov_region_stats_run");
    if (rc) return rc;
    CU(cudaMemcpyAsync(direct ? (void*)host_out : (void*)stage, ctx->d_out.p, out_bytes, cudaMemcpyDeviceToHost, s));
  }
  PassCounters* hp = reinterpret_cast<PassCounters*>(stage + (direct ? 0 : out_bytes));
  if (ctx->verdict_pending) CU(cudaMemcpyAsync(hp, ctx->d_pc.p, sizeof(PassCounters), cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  { int vr = fused_verdict(ctx, *hp, "mcov_region_stats_run"); if (vr) return vr; }
  if (g > 0 && !direct) std::memcpy(host_out, stage, out_bytes);
  // htslib's cap fired in this pass (rare: a pile deeper than max_depth).  The depth store holds the replay of the
  // WHOLE-CONTIG iterator; the reference builds one iterator per region (metacov/cli.py:85-95 -> pileup.py:13), which is
  // given only the reads overlapping the region.  For a region that starts at 0 the two agree; every other region of
  // a capped contig is replayed with its own iterator into scratch memory and its record recomputed from that.
  if (ctx->cap_contigs > 0 && g > 0 && ctx->state == kDepthReady && !ctx->fused_blob.empty()) {
    std::vector<uint8_t> capped((size_t)ctx->n_contigs);
    CU(cudaMemcpyAsync(capped.data(), ctx->cap_flags, (size_t)ctx->n_contigs, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    std::vector<int32_t> idx, rt, rs_, re_;
    std::vector<int64_t> soff;
    int64_t tot = 0;
    for (int64_t i = 0; i < g; ++i) {
      if (!capped[(size_t)tid[i]] || start[i] <= 0 || end[i] <= start[i] || start[i] >= ctx->len[tid[i]]) continue;
      idx.push_back((int32_t)i); rt.push_back(tid[i]); rs_.push_back(start[i]); re_.push_back(end[i]);
      soff.push_back(tot);
      tot += ((int64_t)ctx->len[tid[i]] + 1 + 3) & ~(int64_t)3;
    }
    if (!idx.empty()) {
      const size_t k = idx.size();
      FusedArgs f;
      std::memcpy(&f, ctx->fused_blob.data(), sizeof(f));
      CU(ctx->d_cap_scratch.ensure((size_t)tot * 4 + k * 20 + 64));
      char* sb = ctx->d_cap_scratch.as<char>();
      int32_t* d_scr = reinterpret_cast<int32_t*>(sb);
      int64_t* d_soff = reinterpret_cast<int64_t*>(sb + (((size_t)tot * 4 + 7) & ~(size_t)7));
      int32_t* d_rt = reinterpret_cast<int32_t*>(d_soff + k);
      int32_t* d_rs = d_rt + k;
      int32_t* d_re = d_rs + k;
      CU(cudaMemcpyAsync(d_soff, soff.data(), k * 8, cudaMemcpyHostToDevice, s));
      CU(cudaMemcpyAsync(d_rt, rt.data(), k * 4, cudaMemcpyHostToDevice, s));
      CU(cudaMemcpyAsync(d_rs, rs_.data(), k * 4, cudaMemcpyHostToDevice, s));
      CU(cudaMemcpyAsync(d_re, re_.data(), k * 4, cudaMemcpyHostToDevice, s));
      MCOV_LAUNCH(ctx, kKCapReplay, (k_cap_replay_region<<<(unsigned)((k + 31) / 32), 32, 0, s>>>(f, (int)k, d_rt, d_rs, d_re, d_soff, d_scr)));
      CU(cudaGetLastError());
      for (size_t q = 0; q < k; ++q) {
        const int64_t i = idx[q];
        const Clip c = clip_region(ctx, tid[i], start[i], end[i]);
        int rc = mcov_order_stats_by_sort(ctx, d_scr + soff[q] + c.cs, c.n, c.pad, breadth_n,
                                          ctx->d_out.as<mcov_region_stats>() + i, ctx->d_win_slot, ctx->d_win_out);
        if (rc) return fail(ctx, rc, "mcov_region_stats_run: per-region cap replay failed");
        CU(cudaMemcpyAsync(&host_out[i], ctx->d_out.as<mcov_region_stats>() + i, sizeof(mcov_region_stats), cudaMemcpyDeviceToHost, s));
      }
      CU(cudaStreamSynchronize(s));
      for (size_t q = 0; q < k; ++q) host_out[idx[q]].flags &= ~kStatOverflow;     // (the sort path marks its records)
    }
  }
  // regions whose depth left the counting histogram's range: exact statistics by a GPU radix sort
  // of the region (rare: needs max_depth raised above 8190)
  bool redo = false;
  for (int64_t i = 0; i < g; ++i) {
    if (end[i] == start[i]) { std::memset(&host_out[i], 0, sizeof(mcov_region_stats)); continue; }
    if (host_out[i].flags & kStatOverflow) {
      const Clip c = clip_region(ctx, tid[i], start[i], end[i]);
      int rc = mcov_order_stats_by_sort(ctx, ctx->depth + ctx->off[tid[i]] + c.cs, c.n, c.pad, breadth_n,
                                        ctx->d_out.as<mcov_region_stats>() + i, ctx->d_win_slot, ctx->d_win_out);
      if (rc) return fail(ctx, rc, "mcov_region_stats_run: radix statistics failed");
      redo = true;
    }
  }
  if (redo) {
    std::vector<mcov_region_stats> again((size_t)g);
    CU(cudaMemcpyAsync(again.data(), ctx->d_out.p, (size_t)g * sizeof(mcov_region_stats), cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    for (int64_t i = 0; i < g; ++i)
      if (end[i] != start[i] && (host_out[i].flags & kStatOverflow)) host_out[i] = again[i];
  }
  return MCOV_OK;
}

int mcov_region_stats_submit(mcov_ctx* ctx, int64_t g, const int32_t* tid, const int32_t* start, const int32_t* end,
                             int32_t breadth_n, int slot) {
  if (!ctx) return MCOV_ERR_ARG;
  if (ctx->state != kDepthReady) return fail(ctx, MCOV_ERR_STATE, "mcov_region_stats_submit: depth not ready");
  if (slot < 0 || slot > 1 || g < 0 || (g > 0 && (!tid || !start || !end))) return fail(ctx, MCOV_ERR_ARG, "mcov_region_stats_submit: bad arguments");
  if (g > INT32_MAX) return fail(ctx, MCOV_ERR_RANGE, "mcov_region_stats_submit: more than 2^31-1 regions");
  CU(cudaSetDevice(ctx->device));
  mcov_ctx::StatSlot& sl = ctx->slot[slot];
  if (sl.g >= 0) return fail(ctx, MCOV_ERR_STATE, "mcov_region_stats_submit: slot not collected yet");
  cudaStream_t s = ctx->stream;
  const size_t out_bytes = (size_t)g * sizeof(mcov_region_stats);
  CU(sl.buf.ensure(out_bytes + sizeof(PassCounters)));
  if (!sl.done) CU(cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming));
  if (!sl.ready) CU(cudaEventCreateWithFlags(&sl.ready, cudaEventDisableTiming));
  if (g > 0) {
    CU(sl.d_rec.ensure(out_bytes));
    int rc = stats_launch(ctx, g, tid, start, end, breadth_n, sl.d_rec.as<mcov_region_stats>(), "mcov_region_stats_submit");
    if (rc) return rc;
  }
  sl.has_verdict = ctx->verdict_pending;
  if (sl.has_verdict) {
    // (on the main stream: the next pass clears the counters there)
    CU(cudaMemcpyAsync(sl.buf.as<char>() + out_bytes, ctx->d_pc.p, sizeof(PassCounters), cudaMemcpyDeviceToHost, s));
    ctx->verdict_pending = false;                  // the verdict of this pass now travels with the slot
  }
  // The records travel on their own stream, so the kernels of the next pass do not queue behind the
  // copy (32 MB for the 500 k regions of config C3).
  CU(cudaEventRecord(sl.ready, s));
  CU(cudaStreamWaitEvent(ctx->d2h_stream, sl.ready, 0));
  if (g > 0) CU(cudaMemcpyAsync(sl.buf.p, sl.d_rec.p, out_bytes, cudaMemcpyDeviceToHost, ctx->d2h_stream));
  CU(cudaEventRecord(sl.done, ctx->d2h_stream));
  sl.g = g;
  sl.n_reads = ctx->n_reads_pushed;
  sl.len0.clear();
  sl.has_subregion = false;
  for (int64_t i = 0; i < g; ++i) {
    if (end[i] == start[i]) sl.len0.push_back((int32_t)i);
    else if (start[i] > 0) sl.has_subregion = true;
  }
  sl.cap_contigs = sl.has_verdict ? -1 : ctx->cap_contigs;
  return MCOV_OK;
}

// Wait for a submitted slot and vet it; on success *view points at its g records in the slot's
// pinned buffer (valid until the next submit on that slot).
static int stats_collect_common(mcov_ctx* ctx, int slot, mcov_region_stats** view, int64_t* g_out) {
  if (slot < 0 || slot > 1) return fail(ctx, MCOV_ERR_ARG, "mcov_region_stats_collect: bad slot");
  mcov_ctx::StatSlot& sl = ctx->slot[slot];
  if (sl.g < 0) return fail(ctx, MCOV_ERR_STATE, "mcov_region_stats_collect: nothing submitted in this slot");
  CU(cudaSetDevice(ctx->device));
  CU(cudaEventSynchronize(sl.done));
  const int64_t g = sl.g;
  sl.g = -1;
  const size_t out_bytes = (size_t)g * sizeof(mcov_region_stats);
  if (sl.has_verdict) {
    // (the context may hold the next pass by now: its state and pending verdict are not this slot's)
    PassCounters h;
    std::memcpy(&h, sl.buf.as<char>() + out_bytes, sizeof(h));
    int rc = check_pass(ctx, h, sl.n_reads, "mcov_region_stats_collect");
    if (rc) return rc;
    ctx->cap_contigs = (int32_t)h.cap_contigs;      // (the replay ran on the device before the statistics kernels)
    sl.cap_contigs = (int32_t)h.cap_contigs;
  }
  // The device replay is the whole-contig iterator's.  The reference builds one iterator per region, fed the reads that
  // overlap it (pileup.py:13); a region that does not start at 0 can differ once the cap has fired, and the reads of the
  // pass may be gone by now: refuse rather than return the other iterator's numbers.
  if (sl.cap_contigs > 0 && sl.has_subregion)
    return fail(ctx, MCOV_ERR_STATE, "mcov_region_stats_collect: max_depth fired in that pass and a region starts inside its contig; "
                                     "rerun it through mcov_region_stats_run (per-region iterator)");
  mcov_region_stats* rec = sl.buf.as<mcov_region_stats>();
  for (int32_t i : sl.len0) std::memset(&rec[i], 0, sizeof(mcov_region_stats));
  for (int64_t i = 0; i < g; ++i)
    if (rec[i].flags & kStatOverflow)
      return fail(ctx, MCOV_ERR_STATE, "mcov_region_stats_collect: a region's depth left the counting histogram; rerun it through mcov_region_stats_run");
  *view = rec;
  *g_out = g;
  return MCOV_OK;
}

int mcov_region_stats_collect(mcov_ctx* ctx, int slot, mcov_region_stats* host_out) {
  if (!ctx) return MCOV_ERR_ARG;
  if (slot >= 0 && slot <= 1 && ctx->slot[slot].g > 0 && !host_out) return fail(ctx, MCOV_ERR_ARG, "mcov_region_stats_collect: null output");
  mcov_region_stats* rec = nullptr;
  int64_t g = 0;
  int rc = stats_collect_common(ctx, slot, &rec, &g);
  if (rc) return rc;
  if (g > 0) std::memcpy(host_out, rec, (size_t)g * sizeof(mcov_region_stats));
  return MCOV_OK;
}

int mcov_region_stats_collect_view(mcov_ctx* ctx, int slot, const mcov_region_stats** view, int64_t* g_out) {
  if (!ctx) return MCOV_ERR_ARG;
  if (!view || !g_out) return fail(ctx, MCOV_ERR_ARG, "mcov_region_stats_collect_view: null output");
  mcov_region_stats* rec = nullptr;
  int rc = stats_collect_common(ctx, slot, &rec, g_out);
  if (rc) return rc;
  *view = rec;
  return MCOV_OK;
}

int mcov_region_stats_enqueue(mcov_ctx* ctx, int64_t g, const int32_t* tid, const int32_t* start, const int32_t* end,
                              int32_t breadth_n, mcov_region_stats* dev_out) {
  if (!ctx) return MCOV_ERR_ARG;
  if (ctx->state != kDepthReady) return fail(ctx, MCOV_ERR_STATE, "mcov_region_stats_enqueue: depth not ready");
  if (g < 0 || (g > 0 && (!tid || !start || !end || !dev_out))) return fail(ctx, MCOV_ERR_ARG, "mcov_region_stats_enqueue: bad arguments");
  if (g > INT32_MAX) return fail(ctx, MCOV_ERR_RANGE, "mcov_region_stats_enqueue: more than 2^31-1 regions");
  if (g == 0) return MCOV_OK;
  CU(cudaSetDevice(ctx->device));
  return stats_launch(ctx, g, tid, start, end, breadth_n, dev_out, "mcov_region_stats_enqueue");
}

int mcov_region_hist_enqueue(mcov_ctx* ctx, int64_t g, const int32_t* tid, const int32_t* start, const int32_t* end,
                             uint32_t* dev_hist) {
  if (!ctx) return MCOV_ERR_ARG;
  if (ctx->state != kDepthReady) return fail(ctx, MCOV_ERR_STATE, "mcov_region_hist_enqueue: depth not ready");
  if (g < 0 || (g > 0 && (!tid || !start || !end || !dev_hist))) return fail(ctx, MCOV_ERR_ARG, "mcov_region_hist_enqueue: bad arguments");
  if (g > INT32_MAX) return fail(ctx, MCOV_ERR_RANGE, "mcov_region_hist_enqueue: more than 2^31-1 regions");
  if (g == 0) return MCOV_OK;
  CU(cudaSetDevice(ctx->device));
  int rc = check_regions(ctx, g, tid, start, end, "mcov_region_hist_enqueue");
  if (rc) return rc;
  constexpr int64_t kChunk = 65536;
  std::vector<HistTask> tasks;
  for (int64_t i = 0; i < g; ++i) {
    const Clip c = clip_region(ctx, tid[i], start[i], end[i]);
    const int64_t nch = std::max<int64_t>((c.n + kChunk - 1) / kChunk, c.pad > 0 ? 1 : 0);
    for (int64_t k = 0; k < nch; ++k) {
      HistTask t;
      t.slot = ctx->off[tid[i]] + c.cs + k * kChunk;
      t.n = (int32_t)std::max<int64_t>(0, std::min<int64_t>(kChunk, c.n - k * kChunk));
      t.region = (int32_t)i; t.pad = k == 0 ? c.pad : 0; t.reserved = 0;
      tasks.push_back(t);
    }
  }
  if (tasks.empty()) return MCOV_OK;
  cudaStream_t s = ctx->stream;
  CU(ctx->d_htasks.ensure(tasks.size() * sizeof(HistTask)));
  CU(cudaMemcpyAsync(ctx->d_htasks.p, tasks.data(), tasks.size() * sizeof(HistTask), cudaMemcpyHostToDevice, s));
  MCOV_LAUNCH(ctx, kKRegionHist, (k_region_hist<<<(unsigned)tasks.size(), kStatThreads, 0, s>>>(
      ctx->depth, ctx->d_htasks.as<HistTask>(), dev_hist)));
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(s));                    // `tasks` goes out of scope (pageable source)
  return MCOV_OK;
}

int mcov_hist_stats_enqueue(mcov_ctx* ctx, int64_t g, const uint32_t* dev_hist, int32_t breadth_n, mcov_region_stats* dev_out) {
  if (!ctx) return MCOV_ERR_ARG;
  if (g < 0 || (g > 0 && (!dev_hist || !dev_out))) return fail(ctx, MCOV_ERR_ARG, "mcov_hist_stats_enqueue: bad arguments");
  if (g > INT32_MAX) return fail(ctx, MCOV_ERR_RANGE, "mcov_hist_stats_enqueue: more than 2^31-1 regions");
  if (g == 0) return MCOV_OK;
  CU(cudaSetDevice(ctx->device));
  MCOV_LAUNCH(ctx, kKHistFinish, (k_hist_finish<<<(unsigned)g, kStatThreads, 0, ctx->stream>>>(dev_hist, dev_out, breadth_n)));
  CU(cudaGetLastError());
  return MCOV_OK;
}

int mcov_depth_runs(mcov_ctx* ctx, int32_t tid0, int32_t tid1, int64_t* n_runs_out) {
  if (!ctx) return MCOV_ERR_ARG;
  if (ctx->state != kDepthReady) return fail(ctx, MCOV_ERR_STATE, "mcov_depth_runs: depth not ready (finalize first)");
  if (tid0 < 0 || tid1 < tid0 || tid1 > ctx->n_contigs || !n_runs_out) return fail(ctx, MCOV_ERR_ARG, "mcov_depth_runs: bad contig range");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  ctx->n_runs = -1;
  std::vector<RunTask> tasks;
  for (int32_t c = tid0; c < tid1; ++c)
    for (int64_t p = 0; p < ctx->len[c]; p += kRunChunk) {
      RunTask t;
      t.slot = ctx->off[c] + p; t.n = (int32_t)std::min<int64_t>(kRunChunk, ctx->len[c] - p); t.tid = c; t.pos0 = (int32_t)p; t.reserved = 0;
      tasks.push_back(t);
    }
  const int64_t nt = (int64_t)tasks.size();
  *n_runs_out = 0;
  if (nt == 0) { ctx->n_runs = 0; return MCOV_OK; }
  if (nt > INT32_MAX) return fail(ctx, MCOV_ERR_RANGE, "mcov_depth_runs: contig range too large for one call");
  CU(ctx->d_run_tasks.ensure((size_t)nt * sizeof(RunTask)));
  CU(ctx->d_run_counts.ensure(((size_t)nt + 1) * 8));
  CU(cudaMemcpyAsync(ctx->d_run_tasks.p, tasks.data(), (size_t)nt * sizeof(RunTask), cudaMemcpyHostToDevice, s));
  long long* counts = ctx->d_run_counts.as<long long>();
  MCOV_LAUNCH(ctx, kKRunCount, (k_run_count<<<(unsigned)nt, kRunThreads, 0, s>>>(ctx->depth, ctx->d_run_tasks.as<RunTask>(), counts)));
  CU(cudaGetLastError());
  MCOV_LAUNCH(ctx, kKRunOffsets, (k_run_offsets<<<1, 1024, 0, s>>>(counts, nt)));
  CU(cudaGetLastError());
  long long total = 0;
  CU(cudaMemcpyAsync(&total, counts + nt, 8, cudaMemcpyDeviceToHost, s));
  { int vr = sync_verdict(ctx, "mcov_depth_runs"); if (vr) return vr; }     // (the synchronise also: `tasks` has been consumed)
  if (total > 0) {
    CU(ctx->d_run_out.ensure((size_t)total * 16));
    int32_t* o = ctx->d_run_out.as<int32_t>();
    MCOV_LAUNCH(ctx, kKRunWrite, (k_run_write<<<(unsigned)nt, kRunThreads, 0, s>>>(ctx->depth, ctx->d_run_tasks.as<RunTask>(), counts,
                                                                                    o, o + total, o + 3 * total)));
    CU(cudaGetLastError());
    MCOV_LAUNCH(ctx, kKRunEnds, (k_run_ends<<<grid_for(ctx, total, 256, 8), 256, 0, s>>>(o, o + total, ctx->d_len.as<int32_t>(), total, o + 2 * total)));
    CU(cudaGetLastError());
  }
  ctx->n_runs = total;
  *n_runs_out = total;
  return MCOV_OK;
}

int mcov_depth_runs_read(mcov_ctx* ctx, int64_t first, int64_t n, int32_t* tid, int32_t* start, int32_t* end, int32_t* depth) {
  if (!ctx) return MCOV_ERR_ARG;
  if (ctx->n_runs < 0) return fail(ctx, MCOV_ERR_STATE, "mcov_depth_runs_read: call mcov_depth_runs first");
  if (first < 0 || n < 0 || first + n > ctx->n_runs || (n > 0 && (!tid || !start || !end || !depth)))
    return fail(ctx, MCOV_ERR_ARG, "mcov_depth_runs_read: bad range");
  if (n == 0) return MCOV_OK;
  CU(cudaSetDevice(ctx->device));
  const int32_t* o = ctx->d_run_out.as<int32_t>();
  const int64_t total = ctx->n_runs;
  int32_t* dst[4] = {tid, start, end, depth};
  for (int k = 0; k < 4; ++k)
    CU(cudaMemcpyAsync(dst[k], o + (int64_t)k * total + first, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return MCOV_OK;
}

int mcov_window_means(mcov_ctx* ctx, int32_t window, double* host_out, int64_t n_out) {
  if (!ctx) return MCOV_ERR_ARG;
  if (ctx->state != kDepthReady) return fail(ctx, MCOV_ERR_STATE, "mcov_window_means: depth not ready");
  if (window <= 0 || !host_out) return fail(ctx, MCOV_ERR_ARG, "mcov_window_means: bad arguments");
  CU(cudaSetDevice(ctx->device));
  std::vector<int64_t> wslot;
  std::vector<int32_t> wn;
  for (int32_t c = 0; c < ctx->n_contigs; ++c)
    for (int64_t p = 0; p < ctx->len[c]; p += window) {
      wslot.push_back(ctx->off[c] + p);
      wn.push_back((int32_t)std::min<int64_t>(window, ctx->len[c] - p));
    }
  int64_t nw = (int64_t)wslot.size();
  if (nw != n_out) return fail(ctx, MCOV_ERR_ARG, "mcov_window_means: n_out != sum(ceil(len/window))");
  if (nw == 0) return MCOV_OK;
  cudaStream_t s = ctx->stream;
  CU(ctx->d_win_slot.ensure((size_t)nw * 8)); CU(ctx->d_win_n.ensure((size_t)nw * 4)); CU(ctx->d_win_out.ensure((size_t)nw * 8));
  CU(cudaMemcpyAsync(ctx->d_win_slot.p, wslot.data(), (size_t)nw * 8, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(ctx->d_win_n.p, wn.data(), (size_t)nw * 4, cudaMemcpyHostToDevice, s));
  int64_t threads = nw * 32;
  MCOV_LAUNCH(ctx, kKWindowSums, (k_window_sums<<<(unsigned)((threads + 255) / 256), 256, 0, s>>>(
      ctx->depth, ctx->d_win_slot.as<int64_t>(), ctx->d_win_n.as<int32_t>(), nw, ctx->d_win_out.as<long long>())));
  CU(cudaGetLastError());
  std::vector<long long> sums((size_t)nw);
  CU(cudaMemcpyAsync(sums.data(), ctx->d_win_out.p, (size_t)nw * 8, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  for (int64_t i = 0; i < nw; ++i) host_out[i] = (double)sums[i] / (double)wn[i];
  return MCOV_OK;
}

int mcov_isize_hist(mcov_ctx* ctx, int64_t n, const uint16_t* flag, const int32_t* isize, int mem_kind,
                    int32_t n_group_flags, const uint16_t* group_flags, int32_t n_bins, uint32_t* hist_out,
                    uint64_t* group_counts_out, int32_t* max_isize_out) {
  if (!ctx) return MCOV_ERR_ARG;
  if (n < 0 || n_group_flags < 0 || n_group_flags > kMaxGroupFlags || n_bins <= 0 || !hist_out || !group_counts_out ||
      !max_isize_out || (n_group_flags > 0 && !group_flags) || (n > 0 && (!flag || !isize)))
    return fail(ctx, MCOV_ERR_ARG, "mcov_isize_hist: bad arguments");
  CU(cudaSetDevice(ctx->device));
  const int groups = 1 << n_group_flags;
  const size_t hist_bytes = (size_t)groups * n_bins * 4;
  cudaStream_t s = ctx->stream;
  // scratch: [hist][group_cnt u64][max_isize int]
  size_t off_cnt = (hist_bytes + 7) & ~(size_t)7, off_mx = off_cnt + (size_t)groups * 8;
  CU(ctx->d_win_out.ensure(off_mx + 8));
  char* base = ctx->d_win_out.as<char>();
  CU(cudaMemsetAsync(base, 0, off_mx + 8, s));
  IsizeArgs a;
  a.n = n; a.n_group_flags = n_group_flags; a.n_bins = n_bins;
  for (int k = 0; k < kMaxGroupFlags; ++k) a.group_flags[k] = k < n_group_flags ? group_flags[k] : 0;
  a.hist = reinterpret_cast<uint32_t*>(base);
  a.group_cnt = reinterpret_cast<unsigned long long*>(base + off_cnt);
  a.max_isize = reinterpret_cast<int*>(base + off_mx);
  if (n > 0) {
    if (mem_kind == MCOV_MEM_HOST) {
      ReadStage& st = ctx->stage[0];
      if (st.in_flight) { CU(cudaEventSynchronize(st.consumed)); st.in_flight = false; }
      CU(st.flag.ensure((size_t)n * 2)); CU(st.pos.ensure((size_t)n * 4));
      CU(cudaMemcpyAsync(st.flag.p, flag, (size_t)n * 2, cudaMemcpyHostToDevice, s));
      CU(cudaMemcpyAsync(st.pos.p, isize, (size_t)n * 4, cudaMemcpyHostToDevice, s));
      a.flag = st.flag.as<uint16_t>(); a.isize = st.pos.as<int32_t>();
    } else if (mem_kind == MCOV_MEM_DEVICE) {
      a.flag = flag; a.isize = isize;
    } else return fail(ctx, MCOV_ERR_ARG, "mcov_isize_hist: bad mem_kind");
    int use_smem = ((int64_t)groups * n_bins <= kIsizeSmemBins) ? 1 : 0;
    int grid = grid_for(ctx, n, kHistThreads, 4);
    MCOV_LAUNCH(ctx, kKIsizeHist, (k_isize_hist<<<grid, kHistThreads, 0, s>>>(a, use_smem)));
    CU(cudaGetLastError());
    MCOV_LAUNCH(ctx, kKGroupCount, (k_group_count<<<grid, kHistThreads, 0, s>>>(a)));
    CU(cudaGetLastError());
  }
  CU(cudaMemcpyAsync(hist_out, a.hist, hist_bytes, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(group_counts_out, a.group_cnt, (size_t)groups * 8, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(max_isize_out, a.max_isize, 4, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  return MCOV_OK;
}

int mcov_kmer_hist(mcov_ctx* ctx, int64_t n, const uint16_t* flag, const int32_t* l_seq, const uint8_t* seq_win,
                   int32_t win_bytes, int32_t win_bases, int32_t K, int32_t NK, int32_t STEP, int32_t OFFSET,
                   int32_t n_group_flags, const uint16_t* group_flags, uint32_t* hist_out) {
  return mcov_kmer_hist_mem(ctx, n, flag, l_seq, seq_win, MCOV_MEM_HOST, win_bytes, win_bases, K, NK, STEP, OFFSET, n_group_flags,
                            group_flags, hist_out);
}

int mcov_kmer_hist_mem(mcov_ctx* ctx, int64_t n, const uint16_t* flag, const int32_t* l_seq, const uint8_t* seq_win, int mem_kind,
                       int32_t win_bytes, int32_t win_bases, int32_t K, int32_t NK, int32_t STEP, int32_t OFFSET,
                       int32_t n_group_flags, const uint16_t* group_flags, uint32_t* hist_out) {
  if (!ctx) return MCOV_ERR_ARG;
  if (mem_kind != MCOV_MEM_HOST && mem_kind != MCOV_MEM_DEVICE) return fail(ctx, MCOV_ERR_ARG, "mcov_kmer_hist: bad mem_kind");
  if (n < 0 || K < 1 || K > 12 || NK < 1 || STEP < 1 || OFFSET < 0 || n_group_flags < 0 || n_group_flags > kMaxGroupFlags ||
      win_bases < OFFSET + (NK - 1) * STEP + K || win_bytes < (win_bases + 1) / 2 || !hist_out ||
      (n > 0 && (!flag || !l_seq || !seq_win)) || (n_group_flags > 0 && !group_flags))
    return fail(ctx, MCOV_ERR_ARG, "mcov_kmer_hist: bad arguments (K in 1..12, OFFSET >= 0, window must cover OFFSET+(NK-1)*STEP+K bases)");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  const int64_t table = ((int64_t)1 << (2 * K)) + 1;
  const size_t hist_bytes = (size_t)(1 << n_group_flags) * table * NK * 4;
  CU(ctx->d_win_out.ensure(hist_bytes));
  CU(cudaMemsetAsync(ctx->d_win_out.p, 0, hist_bytes, s));
  if (n > 0) {
    KmerArgs a;
    a.n = n;
    if (mem_kind == MCOV_MEM_DEVICE) {                          // (a GPU-decoded file: the columns never leave the device)
      a.flag = flag; a.l_seq = l_seq; a.win = seq_win;
    } else {
      ReadStage& st = ctx->stage[0];
      if (st.in_flight) { CU(cudaEventSynchronize(st.consumed)); st.in_flight = false; }
      CU(st.flag.ensure((size_t)n * 2)); CU(st.pos.ensure((size_t)n * 4)); CU(st.cig.ensure((size_t)n * win_bytes));
      CU(cudaMemcpyAsync(st.flag.p, flag, (size_t)n * 2, cudaMemcpyHostToDevice, s));
      CU(cudaMemcpyAsync(st.pos.p, l_seq, (size_t)n * 4, cudaMemcpyHostToDevice, s));
      CU(cudaMemcpyAsync(st.cig.p, seq_win, (size_t)n * win_bytes, cudaMemcpyHostToDevice, s));
      a.flag = st.flag.as<uint16_t>(); a.l_seq = st.pos.as<int32_t>(); a.win = st.cig.as<uint8_t>();
    }
    a.win_bytes = win_bytes; a.win_bases = win_bases; a.K = K; a.NK = NK; a.STEP = STEP; a.OFFSET = OFFSET;
    a.n_group_flags = n_group_flags;
    for (int k = 0; k < kMaxGroupFlags; ++k) a.group_flags[k] = k < n_group_flags ? group_flags[k] : 0;
    a.hist = ctx->d_win_out.as<uint32_t>();
    MCOV_LAUNCH(ctx, kKKmerHist, (k_kmer_hist<<<grid_for(ctx, n, kHistThreads, 8), kHistThreads, 0, s>>>(a)));
    CU(cudaGetLastError());
  }
  CU(cudaMemcpyAsync(hist_out, ctx->d_win_out.p, hist_bytes, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  return MCOV_OK;
}

}  // extern "C"
