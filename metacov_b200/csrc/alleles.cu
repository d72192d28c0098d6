// alleles.cu -- SNV sites, nucleotide diversity and reference agreement per region from the A / C / G / T counts of
// mcov_base_counts (include/metacov_b200.h: mcov_set_reference, mcov_allele_stats_run, mcov_allele_sites,
// mcov_allele_sites_read; kernels in k_alleles.cuh).
//
// Reads the counters (mcov_ctx::d_bc) and the reference store (d_ref); writes only its own scratch and the site list.
// The depth store, its verdict and caches, and the counters are never written.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include <cub/device/device_scan.cuh>

#include "ctx.cuh"
#include "k_alleles.cuh"

using namespace mcov;

static_assert(sizeof(mcov_allele_stats) == 64, "mcov_allele_stats is 64 bytes");
static_assert(sizeof(mcov_allele_site) == 32, "mcov_allele_site is 32 bytes");
static_assert(sizeof(AlPart) == 64, "AlPart is 64 bytes");

namespace mcov {

int al_check(mcov_ctx* ctx, const mcov_allele_params* p, AlleleParams* out, const char* who) {
  if (!p) return ctx_fail(ctx, MCOV_ERR_ARG, std::string(who) + ": null parameters");
  if (p->min_coverage < 1 || p->min_count < 1 || !(p->min_freq >= 0.0 && p->min_freq <= 1.0) ||
      (p->use_reference != 0 && p->use_reference != 1))
    return ctx_fail(ctx, MCOV_ERR_ARG, std::string(who) + ": need min_coverage >= 1, min_count >= 1, 0 <= min_freq <= 1 and use_reference 0 or 1");
  if (!ctx->bc_ready || ctx->bc_epoch != ctx->contig_epoch)
    return ctx_fail(ctx, MCOV_ERR_STATE, std::string(who) + ": no counts for this contig table (call mcov_base_counts first)");
  if (p->use_reference) {
    if (ctx->ref_epoch != ctx->contig_epoch)
      return ctx_fail(ctx, MCOV_ERR_STATE, std::string(who) + ": use_reference without a reference (mcov_set_reference)");
    for (int32_t c = 0; c < ctx->n_contigs; ++c)
      if (!ctx->ref_set[c]) {
        char msg[200];
        std::snprintf(msg, sizeof(msg), "%s: use_reference, and contig %d has no reference (mcov_set_reference)", who, c);
        return ctx_fail(ctx, MCOV_ERR_STATE, msg);
      }
  }
  out->min_cov = p->min_coverage; out->min_count = p->min_count; out->min_freq = p->min_freq; out->use_ref = p->use_reference;
  return MCOV_OK;
}

unsigned al_grid(const mcov_ctx* ctx, int64_t items, int per) {
  return (unsigned)std::max<int64_t>(1, std::min<int64_t>((items + per - 1) / per, (int64_t)std::max(ctx->n_sm, 1) * 64));
}

int upload_region_chunks(mcov_ctx* ctx, int64_t g, const int32_t* tid, const int32_t* start, const int32_t* end,
                         int64_t chunk, size_t part_bytes, size_t out_bytes, const char* who, int64_t* n_chunks) {
  cudaStream_t s = ctx->stream;
  std::vector<AlChunk> chunks;
  std::vector<int64_t> meta((size_t)(2 * g + 1));
  int64_t* first = meta.data();
  int64_t* length = meta.data() + g + 1;
  for (int64_t i = 0; i < g; ++i) {
    first[i] = (int64_t)chunks.size();
    length[i] = (int64_t)end[i] - start[i];
    const int64_t len = ctx->len[tid[i]];
    const int64_t a = std::min<int64_t>(start[i], len), b = std::min<int64_t>(end[i], len);
    for (int64_t p = a; p < b; p += chunk) chunks.push_back({ctx->off[tid[i]] + p, std::min<int64_t>(chunk, b - p)});
  }
  first[g] = (int64_t)chunks.size();
  const int64_t nc = (int64_t)chunks.size();
  CTX_CU(who, ctx->d_chunk_meta.ensure(meta.size() * 8));
  CTX_CU(who, ctx->d_region_out.ensure(out_bytes));
  CTX_CU(who, cudaMemcpyAsync(ctx->d_chunk_meta.p, meta.data(), meta.size() * 8, cudaMemcpyHostToDevice, s));
  if (nc > 0) {
    CTX_CU(who, ctx->d_chunks.ensure((size_t)nc * sizeof(AlChunk)));
    CTX_CU(who, ctx->d_chunk_part.ensure((size_t)nc * part_bytes));
    CTX_CU(who, cudaMemcpyAsync(ctx->d_chunks.p, chunks.data(), (size_t)nc * sizeof(AlChunk), cudaMemcpyHostToDevice, s));
  }
  *n_chunks = nc;
  return MCOV_OK;
}

int size_site_list(mcov_ctx* ctx, SiteList& sl, int64_t items, size_t site_bytes, const char* who, int64_t* total,
                   const char* free_hook) {
  cudaStream_t s = ctx->stream;
  int64_t* tile_n = ctx->d_site_tiles.as<int64_t>();
  size_t tb = 0;
  CTX_CU(who, cub::DeviceScan::InclusiveSum(nullptr, tb, tile_n, tile_n + items, items, s));
  if (!free_hook) {
    CTX_CU(who, ctx->d_site_scan.ensure(tb));
  } else if (int rc = ensure_fits_n(ctx, ctx->d_site_scan, tb, free_hook, who,
                                    "the scan of %lld tile counts needs %zu bytes of device memory, %zu are free", items)) {
    return rc;
  }
  CTX_CU(who, cub::DeviceScan::InclusiveSum(ctx->d_site_scan.p, tb, tile_n, tile_n + items, items, s));
  CTX_CU(who, cudaMemcpyAsync(total, tile_n + 2 * items - 1, 8, cudaMemcpyDeviceToHost, s));
  CTX_CU(who, cudaStreamSynchronize(s));
  const size_t bytes = (size_t)*total * site_bytes;
  if (*total > 0 && free_hook)
    return ensure_fits_n(ctx, sl.list, bytes, free_hook, who, "a list of %lld records needs %zu bytes of device memory, %zu are free",
                         (long long)*total);
  if (*total > 0 && sl.list.ensure(bytes) != cudaSuccess) {
    (void)cudaGetLastError();
    char msg[200];
    std::snprintf(msg, sizeof(msg), "%s: %lld sites need %zu bytes of device memory", who, (long long)*total, bytes);
    return ctx_fail(ctx, MCOV_ERR_NOMEM, msg);
  }
  return MCOV_OK;
}

}  // namespace mcov

namespace {

constexpr int64_t kRefStageBytes = 64 << 20;      // the reference goes up in pieces of this size

}  // namespace

extern "C" int mcov_set_reference(mcov_ctx* ctx, int32_t tid, const char* ascii, int32_t n) {
  if (!ctx) return MCOV_ERR_ARG;
  if (tid < 0 || tid >= ctx->n_contigs || n != ctx->len[tid] || (n > 0 && !ascii))
    return ctx_fail(ctx, MCOV_ERR_ARG, "mcov_set_reference: need a valid tid and n equal to the contig's length");
  CTX_CU("mcov_set_reference", cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  if (ctx->ref_epoch != ctx->contig_epoch) {
    // a new contig table: every slot unknown until its contig is given
    ctx->ref_epoch = -1;
    const size_t need = (size_t)ctx->n_slots;
    if (int rc = ensure_fits(ctx, ctx->d_ref, need, "MCOV_REF_FREE_BYTES", "mcov_set_reference",
                             "the reference store of %lld reference slots needs %zu bytes of device memory, %zu are free"))
      return rc;
    CTX_CU("mcov_set_reference", cudaMemsetAsync(ctx->d_ref.p, kRefUnknown, need, s));
    ctx->ref_set.assign((size_t)ctx->n_contigs, 0);
    ctx->ref_epoch = ctx->contig_epoch;
  }
  ctx->ref_set[tid] = 0;
  uint8_t* dst = ctx->d_ref.as<uint8_t>() + ctx->off[tid];
  if (n > 0) CTX_CU("mcov_set_reference", ctx->d_ref_stage.ensure((size_t)std::min<int64_t>(n, kRefStageBytes)));
  for (int64_t a = 0; a < n; a += kRefStageBytes) {
    const int64_t m = std::min<int64_t>(kRefStageBytes, n - a);
    CTX_CU("mcov_set_reference", cudaMemcpyAsync(ctx->d_ref_stage.p, ascii + a, (size_t)m, cudaMemcpyHostToDevice, s));
    MCOV_LAUNCH(ctx, kKRefEncode, (k_ref_encode<<<al_grid(ctx, m, 1024), 256, 0, s>>>(ctx->d_ref_stage.as<uint8_t>(), m, dst + a)));
    CTX_CU("mcov_set_reference", cudaGetLastError());
  }
  CTX_CU("mcov_set_reference", cudaStreamSynchronize(s));
  ctx->ref_set[tid] = 1;
  return MCOV_OK;
}

extern "C" int mcov_allele_stats_run(mcov_ctx* ctx, int64_t g, const int32_t* tid, const int32_t* start, const int32_t* end,
                                     const mcov_allele_params* params, mcov_allele_stats* host_out) {
  const char* who = "mcov_allele_stats_run";
  if (!ctx) return MCOV_ERR_ARG;
  if (int rc = check_regions(ctx, g, tid, start, end, host_out, who)) return rc;
  AlleleParams P;
  if (int rc = al_check(ctx, params, &P, who)) return rc;
  if (g == 0) return MCOV_OK;
  CTX_CU(who, cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  int64_t nc = 0;
  if (int rc = upload_region_chunks(ctx, g, tid, start, end, kAlChunk, sizeof(AlPart), (size_t)g * sizeof(mcov_allele_stats), who, &nc))
    return rc;
  if (nc > 0) {
    AlRegionArgs a;
    a.cnt = ctx->d_bc.as<uint4>(); a.ref = ctx->d_ref.as<uint8_t>();
    a.chunks = ctx->d_chunks.as<AlChunk>(); a.n_chunks = nc;
    a.part = ctx->d_chunk_part.as<AlPart>(); a.P = P;
    MCOV_LAUNCH(ctx, kKAlleleChunks, (k_allele_chunks<<<al_grid(ctx, nc, kAlWarps), kAlThreads, 0, s>>>(a)));
    CTX_CU(who, cudaGetLastError());
  }
  const int64_t* d_meta = ctx->d_chunk_meta.as<int64_t>();
  MCOV_LAUNCH(ctx, kKAlleleCombine, (k_allele_combine<<<al_grid(ctx, g, kAlWarps), kAlThreads, 0, s>>>(
                                         ctx->d_chunk_part.as<AlPart>(), d_meta, d_meta + g + 1, g, ctx->d_region_out.as<mcov_allele_stats>())));
  CTX_CU(who, cudaGetLastError());
  CTX_CU(who, cudaMemcpyAsync(host_out, ctx->d_region_out.p, (size_t)g * sizeof(mcov_allele_stats), cudaMemcpyDeviceToHost, s));
  CTX_CU(who, cudaStreamSynchronize(s));
  return MCOV_OK;
}

namespace mcov {

int allele_site_list(mcov_ctx* ctx, const AlleleParams& P, SiteList& sl, const char* who, int64_t* total_out,
                     const char* free_hook) {
  sl.n = -1;
  cudaStream_t s = ctx->stream;
  const int64_t n_tiles = (ctx->n_slots + kAlTile - 1) / kAlTile;
  // [n_tiles] site counts, then [n_tiles] their inclusive scan
  if (!free_hook) {
    CTX_CU(who, ctx->d_site_tiles.ensure((size_t)n_tiles * 16));
  } else if (int rc = ensure_fits_n(ctx, ctx->d_site_tiles, (size_t)n_tiles * 16, free_hook, who,
                                    "the counts of %lld site tiles need %zu bytes of device memory, %zu are free", n_tiles)) {
    return rc;
  }
  AlSiteArgs a;
  a.cnt = ctx->d_bc.as<uint4>(); a.ref = ctx->d_ref.as<uint8_t>();
  a.n_slots = ctx->n_slots; a.n_tiles = n_tiles;
  a.contig_off = ctx->d_off.as<int64_t>(); a.n_contigs = ctx->n_contigs;
  a.tile_n = ctx->d_site_tiles.as<int64_t>(); a.tile_incl = a.tile_n + n_tiles;
  a.sites = nullptr; a.P = P;
  MCOV_LAUNCH(ctx, kKAlleleSiteCount, (k_allele_site_count<<<al_grid(ctx, n_tiles, 1), kAlTileThreads, 0, s>>>(a)));
  CTX_CU(who, cudaGetLastError());
  int64_t total = 0;
  if (int rc = size_site_list(ctx, sl, n_tiles, sizeof(mcov_allele_site), who, &total, free_hook)) return rc;
  if (total > 0) {
    a.sites = sl.list.as<mcov_allele_site>();
    MCOV_LAUNCH(ctx, kKAlleleSiteWrite, (k_allele_site_write<<<al_grid(ctx, n_tiles, 1), kAlTileThreads, 0, s>>>(a)));
    CTX_CU(who, cudaGetLastError());
    CTX_CU(who, cudaStreamSynchronize(s));
  }
  sl.n = total;
  sl.epoch = ctx->contig_epoch;
  *total_out = total;
  return MCOV_OK;
}

}  // namespace mcov

extern "C" int mcov_allele_sites(mcov_ctx* ctx, const mcov_allele_params* params, int64_t* n_sites_out) {
  const char* who = "mcov_allele_sites";
  if (!ctx) return MCOV_ERR_ARG;
  ctx->allele_sites.n = -1;
  if (!n_sites_out) return ctx_fail(ctx, MCOV_ERR_ARG, "mcov_allele_sites: null n_sites_out");
  AlleleParams P;
  if (int rc = al_check(ctx, params, &P, who)) return rc;
  CTX_CU(who, cudaSetDevice(ctx->device));
  return allele_site_list(ctx, P, ctx->allele_sites, who, n_sites_out);
}

extern "C" int mcov_allele_sites_read(mcov_ctx* ctx, int64_t first, int64_t n, mcov_allele_site* host_out) {
  if (!ctx) return MCOV_ERR_ARG;
  return read_site_list(ctx, ctx->allele_sites, first, n, host_out, sizeof(mcov_allele_site), "mcov_allele_sites_read",
                        "mcov_allele_sites");
}
