// basecount.cu -- A / C / G / T counts at every reference position (include/metacov_b200.h: mcov_base_counts,
// mcov_copy_base_counts; kernels in k_basecount.cuh).
//
// The counts cover the whole file and live in their own store (mcov_ctx::d_bc): the depth store, its verdict and its
// caches are never touched.  Records come from the last device decode (BAM or SAM), or from a BAM file through the
// streamed decoder chunk by chunk (bam_gpu_chunks), each chunk's records counted while they are resident.
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "ctx.cuh"
#include "k_basecount.cuh"

using namespace mcov;

namespace {

// Count the records [i0, n) of one set of device columns.
int count_records(mcov_ctx* ctx, const BcArgs& a, bool sam) {
  if (a.n <= a.i0) return MCOV_OK;
  const int64_t grid = std::min<int64_t>((a.n - a.i0 + kBcWarps - 1) / kBcWarps, (int64_t)std::max(ctx->n_sm, 1) * 8);
  if (sam) MCOV_LAUNCH(ctx, kKBcAny, (k_bc_any<BcSamRec><<<(unsigned)grid, kBcThreads, 0, ctx->stream>>>(a)));
  else MCOV_LAUNCH(ctx, kKBcAny, (k_bc_any<BcBamRec><<<(unsigned)grid, kBcThreads, 0, ctx->stream>>>(a)));
  CTX_CU("mcov_base_counts", cudaGetLastError());
  return MCOV_OK;
}

// The context's half of BcArgs: contig table, filter, counters, error word.
BcArgs context_bc_args(mcov_ctx* ctx, int32_t qthr, int mode) {
  BcArgs a;
  std::memset(&a, 0, sizeof(a));
  a.contig_off = ctx->d_off.as<int64_t>(); a.contig_len = ctx->d_len.as<int32_t>(); a.n_contigs = ctx->n_contigs;
  a.skip_flags = (mode & MCOV_BC_NOFILTER) ? 0u : kBcSkipAll;
  a.qthr = qthr;
  a.cnt = ctx->d_bc.as<uint32_t>();
  a.err = ctx->d_bc_word.as<unsigned long long>();
  return a;
}

// The streamed decode's consumer: each batch's own records (not the carried ones -- this consumer carries none).
struct CountSink : BamChunkSink {
  int32_t qthr; int mode; int64_t done = 0;
  CountSink(int32_t q, int m) : qthr(q), mode(m) {}
  int batch(mcov_ctx* ctx, const BamChunk& b, int64_t* n_carry, int64_t* carry_ops) override {
    *n_carry = 0; *carry_ops = 0;
    BcArgs a = context_bc_args(ctx, qthr, mode);
    a.tid = b.tid; a.pos = b.pos; a.flag = b.flag; a.l_seq = b.l_seq; a.cig_off = b.cig_off; a.cig = b.cig;
    a.data = b.data; a.rec_off = b.rec_off;
    a.i0 = b.n_carry; a.n = b.n;
    a.rec_base = done - b.n_carry;
    done += b.n - b.n_carry;
    return count_records(ctx, a, false);
  }
};

}  // namespace

extern "C" int mcov_base_counts(mcov_ctx* ctx, const char* path, int64_t chunk_bytes, int32_t quality_threshold, int mode) {
  const char* who = "mcov_base_counts";
  if (!ctx) return MCOV_ERR_ARG;
  if (mode != MCOV_BC_ALL && mode != MCOV_BC_NOFILTER) return ctx_fail(ctx, MCOV_ERR_ARG, "mcov_base_counts: mode must be MCOV_BC_ALL or MCOV_BC_NOFILTER");
  if (ctx->n_contigs <= 0) return ctx_fail(ctx, MCOV_ERR_STATE, "mcov_base_counts: mcov_set_contigs has not been called");
  mcov_ctx::BamDev& B = ctx->bam;
  if (!path && (B.n_rec < 0 || !B.data.p)) return ctx_fail(ctx, MCOV_ERR_STATE, "mcov_base_counts: no file decoded on this context");
  CTX_CU(who, cudaSetDevice(ctx->device));
  ctx->bc_ready = false;
  // the counters: 16 bytes a slot, checked against the free device memory before anything is allocated
  const size_t need = (size_t)ctx->n_slots * 16;
  if (int rc = ensure_fits(ctx, ctx->d_bc, need, "MCOV_BC_FREE_BYTES", who,
                           "the A/C/G/T counters of %lld reference slots need %zu bytes of device memory, %zu are free"))
    return rc;
  CTX_CU(who, ctx->d_bc_word.ensure(8));
  cudaStream_t s = ctx->stream;
  CTX_CU(who, cudaMemsetAsync(ctx->d_bc.p, 0, need, s));
  CTX_CU(who, cudaMemsetAsync(ctx->d_bc_word.p, 0xFF, 8, s));
  if (path) {
    mcov_bam_gpu_stream_info info;
    std::memset(&info, 0, sizeof(info));
    CountSink sink(quality_threshold, mode);
    const int rc = bam_gpu_chunks(ctx, path, chunk_bytes, 1, &info, who, sink);
    if (rc) return rc;
  } else {
    BcArgs a = context_bc_args(ctx, quality_threshold, mode);
    a.tid = B.tid.as<int32_t>(); a.pos = B.pos.as<int32_t>(); a.flag = B.flag.as<uint16_t>(); a.l_seq = B.lseq.as<int32_t>();
    a.cig_off = B.cig_off.as<uint32_t>(); a.cig = B.cig.as<uint32_t>();
    a.data = B.data.as<uint8_t>(); a.rec_off = B.rec_off.as<uint64_t>(); a.aux = B.sam ? B.sam_aux.as<SamAux>() : nullptr;
    a.i0 = 0; a.n = B.n_rec;
    const int rc = count_records(ctx, a, B.sam);
    if (rc) return rc;
  }
  unsigned long long e = 0;
  CTX_CU(who, cudaMemcpyAsync(&e, ctx->d_bc_word.p, 8, cudaMemcpyDeviceToHost, s));
  CTX_CU(who, cudaStreamSynchronize(s));
  if (e != ~0ull) {
    char msg[256];
    std::snprintf(msg, sizeof(msg), (e & 3) == kBcErrQueryLong
                      ? "mcov_base_counts: record %lld (0-based, file order): its CIGAR consumes more query bases than SEQ holds"
                      : "mcov_base_counts: record %lld (0-based, file order): its SEQ / QUAL leave the record",
                  (long long)(e >> 2));
    return ctx_fail(ctx, MCOV_ERR_IO, msg);
  }
  ctx->bc_ready = true;
  ctx->bc_qthr = quality_threshold; ctx->bc_mode = mode;
  ctx->bc_epoch = ctx->contig_epoch;
  return MCOV_OK;
}

extern "C" int mcov_copy_base_counts(mcov_ctx* ctx, int32_t tid, int32_t start, int32_t end, uint32_t* host_out) {
  const char* who = "mcov_copy_base_counts";
  if (!ctx) return MCOV_ERR_ARG;
  if (!ctx->bc_ready || ctx->bc_epoch != ctx->contig_epoch)
    return ctx_fail(ctx, MCOV_ERR_STATE, "mcov_copy_base_counts: no counts for this contig table (call mcov_base_counts first)");
  if (tid < 0 || tid >= ctx->n_contigs || start < 0 || end < start || end > ctx->len[tid] || (end > start && !host_out))
    return ctx_fail(ctx, MCOV_ERR_ARG, "mcov_copy_base_counts: region out of range");
  const int64_t n = (int64_t)end - start;
  if (n == 0) return MCOV_OK;
  CTX_CU(who, cudaSetDevice(ctx->device));
  std::vector<uint32_t> tmp((size_t)n * 4);
  CTX_CU(who, cudaMemcpyAsync(tmp.data(), ctx->d_bc.as<uint32_t>() + (ctx->off[tid] + start) * 4, (size_t)n * 16, cudaMemcpyDeviceToHost, ctx->stream));
  CTX_CU(who, cudaStreamSynchronize(ctx->stream));
  for (int64_t k = 0; k < n; ++k)
    for (int b = 0; b < 4; ++b) host_out[b * n + k] = tmp[(size_t)k * 4 + b];
  return MCOV_OK;
}
