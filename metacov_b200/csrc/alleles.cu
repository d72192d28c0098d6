// alleles.cu -- SNV sites, nucleotide diversity and reference agreement per region from the A / C / G / T counts of
// mcov_base_counts (include/metacov_b200.h: mcov_set_reference, mcov_allele_stats_run, mcov_allele_sites,
// mcov_allele_sites_read; kernels in k_alleles.cuh).
//
// Reads the counters (mcov_ctx::d_bc) and the reference store (d_ref); writes only its own scratch and the site list.
// The depth store, its verdict and caches, and the counters are never written.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
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

int al_fail(mcov_ctx* ctx, int code, const std::string& what, cudaError_t e) {
  ctx->err = what;
  if (e != cudaSuccess) { ctx->err += ": "; ctx->err += cudaGetErrorString(e); }
  return code;
}

#define ALU(who, call)                                                                                    \
  do {                                                                                                    \
    cudaError_t e__ = (call);                                                                             \
    if (e__ != cudaSuccess) return al_fail(ctx, MCOV_ERR_CUDA, std::string(who) + ": " + #call, e__);     \
  } while (0)

// Parameters and state shared by the region and site calls: the kernel's parameters, or an error.
int al_check(mcov_ctx* ctx, const mcov_allele_params* p, AlleleParams* out, const char* who) {
  if (!p) return al_fail(ctx, MCOV_ERR_ARG, std::string(who) + ": null parameters");
  if (p->min_coverage < 1 || p->min_count < 1 || !(p->min_freq >= 0.0 && p->min_freq <= 1.0) ||
      (p->use_reference != 0 && p->use_reference != 1))
    return al_fail(ctx, MCOV_ERR_ARG, std::string(who) + ": need min_coverage >= 1, min_count >= 1, 0 <= min_freq <= 1 and use_reference 0 or 1");
  if (!ctx->bc_ready || ctx->bc_epoch != ctx->contig_epoch)
    return al_fail(ctx, MCOV_ERR_STATE, std::string(who) + ": no counts for this contig table (call mcov_base_counts first)");
  if (p->use_reference) {
    if (ctx->ref_epoch != ctx->contig_epoch)
      return al_fail(ctx, MCOV_ERR_STATE, std::string(who) + ": use_reference without a reference (mcov_set_reference)");
    for (int32_t c = 0; c < ctx->n_contigs; ++c)
      if (!ctx->ref_set[c]) {
        char msg[200];
        std::snprintf(msg, sizeof(msg), "%s: use_reference, and contig %d has no reference (mcov_set_reference)", who, c);
        return al_fail(ctx, MCOV_ERR_STATE, msg);
      }
  }
  out->min_cov = p->min_coverage; out->min_count = p->min_count; out->min_freq = p->min_freq; out->use_ref = p->use_reference;
  return MCOV_OK;
}

// Grid of a grid-stride kernel over `items` work items, `per` of them a CTA.
unsigned al_grid(const mcov_ctx* ctx, int64_t items, int per) {
  return (unsigned)std::max<int64_t>(1, std::min<int64_t>((items + per - 1) / per, (int64_t)std::max(ctx->n_sm, 1) * 64));
}

}  // namespace mcov

namespace {

constexpr int64_t kRefStageBytes = 64 << 20;      // the reference goes up in pieces of this size

}  // namespace

extern "C" int mcov_set_reference(mcov_ctx* ctx, int32_t tid, const char* ascii, int32_t n) {
  if (!ctx) return MCOV_ERR_ARG;
  if (tid < 0 || tid >= ctx->n_contigs || n != ctx->len[tid] || (n > 0 && !ascii))
    return al_fail(ctx, MCOV_ERR_ARG, "mcov_set_reference: need a valid tid and n equal to the contig's length");
  ALU("mcov_set_reference", cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  if (ctx->ref_epoch != ctx->contig_epoch) {
    // a new contig table: every slot unknown until its contig is given
    ctx->ref_epoch = -1;
    const size_t need = (size_t)ctx->n_slots;
    if (ctx->d_ref.cap < need) {
      size_t free_b = 0, total_b = 0;
      ALU("mcov_set_reference", cudaMemGetInfo(&free_b, &total_b));
      if (const char* h = std::getenv("MCOV_REF_FREE_BYTES")) free_b = (size_t)std::strtoull(h, nullptr, 10);   // test hook
      const size_t want = need + need / 8 + 256;                 // (DevBuf's growth margin)
      if (want > free_b + ctx->d_ref.cap) {
        char msg[256];
        std::snprintf(msg, sizeof(msg), "mcov_set_reference: the reference store of %lld reference slots needs %zu bytes of device memory, %zu are free",
                      (long long)ctx->n_slots, want, free_b + ctx->d_ref.cap);
        return al_fail(ctx, MCOV_ERR_NOMEM, msg);
      }
    }
    ALU("mcov_set_reference", ctx->d_ref.ensure(need));
    ALU("mcov_set_reference", cudaMemsetAsync(ctx->d_ref.p, kRefUnknown, need, s));
    ctx->ref_set.assign((size_t)ctx->n_contigs, 0);
    ctx->ref_epoch = ctx->contig_epoch;
  }
  ctx->ref_set[tid] = 0;
  uint8_t* dst = ctx->d_ref.as<uint8_t>() + ctx->off[tid];
  if (n > 0) ALU("mcov_set_reference", ctx->d_ref_stage.ensure((size_t)std::min<int64_t>(n, kRefStageBytes)));
  for (int64_t a = 0; a < n; a += kRefStageBytes) {
    const int64_t m = std::min<int64_t>(kRefStageBytes, n - a);
    ALU("mcov_set_reference", cudaMemcpyAsync(ctx->d_ref_stage.p, ascii + a, (size_t)m, cudaMemcpyHostToDevice, s));
    MCOV_LAUNCH(ctx, kKRefEncode, (k_ref_encode<<<al_grid(ctx, m, 1024), 256, 0, s>>>(ctx->d_ref_stage.as<uint8_t>(), m, dst + a)));
    ALU("mcov_set_reference", cudaGetLastError());
  }
  ALU("mcov_set_reference", cudaStreamSynchronize(s));
  ctx->ref_set[tid] = 1;
  return MCOV_OK;
}

extern "C" int mcov_allele_stats_run(mcov_ctx* ctx, int64_t g, const int32_t* tid, const int32_t* start, const int32_t* end,
                                     const mcov_allele_params* params, mcov_allele_stats* host_out) {
  const char* who = "mcov_allele_stats_run";
  if (!ctx) return MCOV_ERR_ARG;
  if (g < 0 || (g > 0 && (!tid || !start || !end || !host_out))) return al_fail(ctx, MCOV_ERR_ARG, "mcov_allele_stats_run: bad arguments");
  for (int64_t i = 0; i < g; ++i)
    if (tid[i] < 0 || tid[i] >= ctx->n_contigs || start[i] < 0 || end[i] < start[i])
      return al_fail(ctx, MCOV_ERR_ARG, "mcov_allele_stats_run: need 0 <= start <= end and a valid tid");
  AlleleParams P;
  if (int rc = al_check(ctx, params, &P, who)) return rc;
  if (g == 0) return MCOV_OK;
  ALU(who, cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  // Every region cut into chunks of kAlChunk positions inside its contig (the positions past the contig's end add to
  // its length only); first[g + 1] locates each region's chunks, length[g] follows it.
  std::vector<AlChunk> chunks;
  std::vector<int64_t> meta((size_t)(2 * g + 1));
  int64_t* first = meta.data();
  int64_t* length = meta.data() + g + 1;
  for (int64_t i = 0; i < g; ++i) {
    first[i] = (int64_t)chunks.size();
    length[i] = (int64_t)end[i] - start[i];
    const int64_t len = ctx->len[tid[i]];
    const int64_t a = std::min<int64_t>(start[i], len), b = std::min<int64_t>(end[i], len);
    for (int64_t p = a; p < b; p += kAlChunk) chunks.push_back({ctx->off[tid[i]] + p, std::min<int64_t>(kAlChunk, b - p)});
  }
  first[g] = (int64_t)chunks.size();
  const int64_t nc = (int64_t)chunks.size();
  ALU(who, ctx->d_al_meta.ensure(meta.size() * 8));
  ALU(who, ctx->d_al_out.ensure((size_t)g * sizeof(mcov_allele_stats)));
  ALU(who, cudaMemcpyAsync(ctx->d_al_meta.p, meta.data(), meta.size() * 8, cudaMemcpyHostToDevice, s));
  if (nc > 0) {
    ALU(who, ctx->d_al_chunks.ensure((size_t)nc * sizeof(AlChunk)));
    ALU(who, ctx->d_al_part.ensure((size_t)nc * sizeof(AlPart)));
    ALU(who, cudaMemcpyAsync(ctx->d_al_chunks.p, chunks.data(), (size_t)nc * sizeof(AlChunk), cudaMemcpyHostToDevice, s));
    AlRegionArgs a;
    a.cnt = ctx->d_bc.as<uint4>(); a.ref = ctx->d_ref.as<uint8_t>();
    a.chunks = ctx->d_al_chunks.as<AlChunk>(); a.n_chunks = nc;
    a.part = ctx->d_al_part.as<AlPart>(); a.P = P;
    MCOV_LAUNCH(ctx, kKAlleleChunks, (k_allele_chunks<<<al_grid(ctx, nc, kAlWarps), kAlThreads, 0, s>>>(a)));
    ALU(who, cudaGetLastError());
  }
  const int64_t* d_meta = ctx->d_al_meta.as<int64_t>();
  MCOV_LAUNCH(ctx, kKAlleleCombine, (k_allele_combine<<<al_grid(ctx, g, kAlWarps), kAlThreads, 0, s>>>(
                                         ctx->d_al_part.as<AlPart>(), d_meta, d_meta + g + 1, g, ctx->d_al_out.as<mcov_allele_stats>())));
  ALU(who, cudaGetLastError());
  ALU(who, cudaMemcpyAsync(host_out, ctx->d_al_out.p, (size_t)g * sizeof(mcov_allele_stats), cudaMemcpyDeviceToHost, s));
  ALU(who, cudaStreamSynchronize(s));
  return MCOV_OK;
}

extern "C" int mcov_allele_sites(mcov_ctx* ctx, const mcov_allele_params* params, int64_t* n_sites_out) {
  const char* who = "mcov_allele_sites";
  if (!ctx) return MCOV_ERR_ARG;
  ctx->n_sites = -1;
  if (!n_sites_out) return al_fail(ctx, MCOV_ERR_ARG, "mcov_allele_sites: null n_sites_out");
  AlleleParams P;
  if (int rc = al_check(ctx, params, &P, who)) return rc;
  ALU(who, cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  const int64_t n_tiles = (ctx->n_slots + kAlTile - 1) / kAlTile;
  // [n_tiles] site counts, then [n_tiles] their inclusive scan
  ALU(who, ctx->d_al_tiles.ensure((size_t)n_tiles * 16));
  AlSiteArgs a;
  a.cnt = ctx->d_bc.as<uint4>(); a.ref = ctx->d_ref.as<uint8_t>();
  a.n_slots = ctx->n_slots; a.n_tiles = n_tiles;
  a.contig_off = ctx->d_off.as<int64_t>(); a.n_contigs = ctx->n_contigs;
  a.tile_n = ctx->d_al_tiles.as<int64_t>(); a.tile_incl = a.tile_n + n_tiles;
  a.sites = nullptr; a.P = P;
  MCOV_LAUNCH(ctx, kKAlleleSiteCount, (k_allele_site_count<<<al_grid(ctx, n_tiles, 1), kAlTileThreads, 0, s>>>(a)));
  ALU(who, cudaGetLastError());
  size_t tb = 0;
  ALU(who, cub::DeviceScan::InclusiveSum(nullptr, tb, a.tile_n, a.tile_n + n_tiles, n_tiles, s));
  ALU(who, ctx->d_al_scan.ensure(tb));
  ALU(who, cub::DeviceScan::InclusiveSum(ctx->d_al_scan.p, tb, a.tile_n, a.tile_n + n_tiles, n_tiles, s));
  int64_t total = 0;
  ALU(who, cudaMemcpyAsync(&total, a.tile_n + 2 * n_tiles - 1, 8, cudaMemcpyDeviceToHost, s));
  ALU(who, cudaStreamSynchronize(s));
  if (total > 0) {
    const size_t bytes = (size_t)total * sizeof(mcov_allele_site);
    if (ctx->d_sites.ensure(bytes) != cudaSuccess) {
      (void)cudaGetLastError();
      char msg[200];
      std::snprintf(msg, sizeof(msg), "mcov_allele_sites: %lld sites need %zu bytes of device memory", (long long)total, bytes);
      return al_fail(ctx, MCOV_ERR_NOMEM, msg);
    }
    a.sites = ctx->d_sites.as<mcov_allele_site>();
    MCOV_LAUNCH(ctx, kKAlleleSiteWrite, (k_allele_site_write<<<al_grid(ctx, n_tiles, 1), kAlTileThreads, 0, s>>>(a)));
    ALU(who, cudaGetLastError());
    ALU(who, cudaStreamSynchronize(s));
  }
  ctx->n_sites = total;
  ctx->sites_epoch = ctx->contig_epoch;
  *n_sites_out = total;
  return MCOV_OK;
}

extern "C" int mcov_allele_sites_read(mcov_ctx* ctx, int64_t first, int64_t n, mcov_allele_site* host_out) {
  if (!ctx) return MCOV_ERR_ARG;
  if (ctx->n_sites < 0 || ctx->sites_epoch != ctx->contig_epoch)
    return al_fail(ctx, MCOV_ERR_STATE, "mcov_allele_sites_read: no site list for this contig table (call mcov_allele_sites first)");
  if (first < 0 || n < 0 || first > ctx->n_sites - n || (n > 0 && !host_out))
    return al_fail(ctx, MCOV_ERR_ARG, "mcov_allele_sites_read: range outside the site list");
  if (n == 0) return MCOV_OK;
  ALU("mcov_allele_sites_read", cudaSetDevice(ctx->device));
  ALU("mcov_allele_sites_read", cudaMemcpyAsync(host_out, ctx->d_sites.as<mcov_allele_site>() + first, (size_t)n * sizeof(mcov_allele_site),
                                                cudaMemcpyDeviceToHost, ctx->stream));
  ALU("mcov_allele_sites_read", cudaStreamSynchronize(ctx->stream));
  return MCOV_OK;
}
