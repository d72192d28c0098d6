// compare.cu -- samples compared per region and per site from their allele signatures (include/metacov_b200.h:
// mcov_allele_signature, mcov_compare_run, mcov_compare_sites, mcov_compare_sites_read; kernels in k_compare.cuh).
//
// A signature is one byte a slot made from the counters of the last mcov_base_counts; a comparison keeps nothing else
// of a file, so the files of a comparison can be counted one after the other on the same GPU.  The pair calls read the
// caller's signature arrays and the contig table; they write only their own scratch and the site list.  The depth
// store, its verdict and caches, the counters and the reference store are never written.
#include <algorithm>
#include <cstdio>
#include <string>
#include <vector>

#include "ctx.cuh"
#include "k_compare.cuh"

using namespace mcov;

static_assert(sizeof(mcov_compare_stats) == 48, "mcov_compare_stats is 48 bytes");
static_assert(sizeof(mcov_compare_site) == 16, "mcov_compare_site is 16 bytes");
static_assert(sizeof(CmpPart) == 24, "CmpPart is 24 bytes");

namespace {

// p is 4-byte aligned device memory on ctx's GPU, or an error naming `what`.
int cmp_device_ptr(mcov_ctx* ctx, const void* p, const char* who, const std::string& what) {
  cudaPointerAttributes at;
  const cudaError_t e = p ? cudaPointerGetAttributes(&at, p) : cudaErrorInvalidValue;
  if (e != cudaSuccess) (void)cudaGetLastError();
  if (e != cudaSuccess || at.type != cudaMemoryTypeDevice || at.device != ctx->device || (reinterpret_cast<uintptr_t>(p) & 3))
    return ctx_fail(ctx, MCOV_ERR_ARG, std::string(who) + ": " + what + " is not 4-byte aligned device memory on the context's GPU");
  return MCOV_OK;
}

// The checks the pair calls share; on success the device table [2 * n_pairs] of (sample a, sample b) signature pointers
// is in ctx->d_pair_sigs (copied on ctx->stream).
int cmp_pairs(mcov_ctx* ctx, int32_t n_sig, const uint8_t* const* sig, int32_t n_pairs, const int32_t* pairs, const char* who) {
  if (ctx->n_contigs <= 0) return ctx_fail(ctx, MCOV_ERR_STATE, std::string(who) + ": no contig table (mcov_set_contigs)");
  if (n_sig < 2 || !sig || n_pairs < 1 || !pairs)
    return ctx_fail(ctx, MCOV_ERR_ARG, std::string(who) + ": need at least two signatures and one pair");
  for (int32_t i = 0; i < n_sig; ++i)
    if (int rc = cmp_device_ptr(ctx, sig[i], who, "signature " + std::to_string(i))) return rc;
  std::vector<const uint8_t*> tab((size_t)2 * n_pairs);
  for (int32_t p = 0; p < n_pairs; ++p) {
    const int32_t a = pairs[2 * p], b = pairs[2 * p + 1];
    if (a < 0 || a >= n_sig || b < 0 || b >= n_sig || a == b) {
      char msg[200];
      std::snprintf(msg, sizeof(msg), "%s: pair %d is (%d, %d); need two different signatures of 0 .. %d", who, p, a, b, n_sig - 1);
      return ctx_fail(ctx, MCOV_ERR_ARG, msg);
    }
    tab[2 * (size_t)p] = sig[a]; tab[2 * (size_t)p + 1] = sig[b];
  }
  CTX_CU(who, ctx->d_pair_sigs.ensure(tab.size() * sizeof(void*)));
  CTX_CU(who, cudaMemcpyAsync(ctx->d_pair_sigs.p, tab.data(), tab.size() * sizeof(void*), cudaMemcpyHostToDevice, ctx->stream));
  return MCOV_OK;
}

}  // namespace

extern "C" int mcov_allele_signature(mcov_ctx* ctx, const mcov_allele_params* params, uint8_t* dev_out) {
  const char* who = "mcov_allele_signature";
  if (!ctx) return MCOV_ERR_ARG;
  if (params && params->use_reference != 0) return ctx_fail(ctx, MCOV_ERR_ARG, "mcov_allele_signature: use_reference must be 0");
  AlleleParams P;
  if (int rc = al_check(ctx, params, &P, who)) return rc;
  CTX_CU(who, cudaSetDevice(ctx->device));
  if (int rc = cmp_device_ptr(ctx, dev_out, who, "dev_out")) return rc;
  cudaStream_t s = ctx->stream;
  MCOV_LAUNCH(ctx, kKAlleleSignature, (k_allele_signature<<<al_grid(ctx, ctx->n_slots, kSigThreads * kSigUnroll), kSigThreads, 0, s>>>(
                                          ctx->d_bc.as<uint4>(), ctx->n_slots, P, dev_out)));
  CTX_CU(who, cudaGetLastError());
  CTX_CU(who, cudaStreamSynchronize(s));
  return MCOV_OK;
}

extern "C" int mcov_compare_run(mcov_ctx* ctx, int32_t n_sig, const uint8_t* const* sig, int32_t n_pairs, const int32_t* pairs,
                                int64_t g, const int32_t* tid, const int32_t* start, const int32_t* end,
                                mcov_compare_stats* host_out) {
  const char* who = "mcov_compare_run";
  if (!ctx) return MCOV_ERR_ARG;
  if (int rc = check_regions(ctx, g, tid, start, end, host_out, who)) return rc;
  CTX_CU(who, cudaSetDevice(ctx->device));
  if (int rc = cmp_pairs(ctx, n_sig, sig, n_pairs, pairs, who)) return rc;
  if (g == 0) return MCOV_OK;
  cudaStream_t s = ctx->stream;
  int64_t nc = 0;
  if (int rc = upload_region_chunks(ctx, g, tid, start, end, kCmpChunk, (size_t)n_pairs * sizeof(CmpPart),
                                    (size_t)g * n_pairs * sizeof(mcov_compare_stats), who, &nc))
    return rc;
  if (nc > 0) {
    CmpRegionArgs a;
    a.sig = ctx->d_pair_sigs.as<const uint8_t* const>(); a.n_pairs = n_pairs;
    a.chunks = ctx->d_chunks.as<AlChunk>(); a.n_chunks = nc;
    a.part = ctx->d_chunk_part.as<CmpPart>();
    MCOV_LAUNCH(ctx, kKCompareChunks, (k_compare_chunks<<<al_grid(ctx, nc * n_pairs, kCmpWarps), kCmpThreads, 0, s>>>(a)));
    CTX_CU(who, cudaGetLastError());
  }
  const int64_t* d_meta = ctx->d_chunk_meta.as<int64_t>();
  MCOV_LAUNCH(ctx, kKCompareCombine, (k_compare_combine<<<al_grid(ctx, g * n_pairs, kCmpWarps), kCmpThreads, 0, s>>>(
                                          ctx->d_chunk_part.as<CmpPart>(), n_pairs, d_meta, d_meta + g + 1, g,
                                          ctx->d_region_out.as<mcov_compare_stats>())));
  CTX_CU(who, cudaGetLastError());
  CTX_CU(who, cudaMemcpyAsync(host_out, ctx->d_region_out.p, (size_t)g * n_pairs * sizeof(mcov_compare_stats), cudaMemcpyDeviceToHost, s));
  CTX_CU(who, cudaStreamSynchronize(s));
  return MCOV_OK;
}

extern "C" int mcov_compare_sites(mcov_ctx* ctx, int32_t n_sig, const uint8_t* const* sig, int32_t n_pairs, const int32_t* pairs,
                                  int64_t* n_sites_out) {
  const char* who = "mcov_compare_sites";
  if (!ctx) return MCOV_ERR_ARG;
  ctx->compare_sites.n = -1;
  if (!n_sites_out) return ctx_fail(ctx, MCOV_ERR_ARG, "mcov_compare_sites: null n_sites_out");
  CTX_CU(who, cudaSetDevice(ctx->device));
  if (int rc = cmp_pairs(ctx, n_sig, sig, n_pairs, pairs, who)) return rc;
  cudaStream_t s = ctx->stream;
  const int64_t n_tiles = (ctx->n_slots + kCmpTile - 1) / kCmpTile;
  const int64_t items = n_tiles * n_pairs;
  // [items] site counts (pair-major), then [items] their inclusive scan
  CTX_CU(who, ctx->d_site_tiles.ensure((size_t)items * 16));
  CmpSiteArgs a;
  a.sig = ctx->d_pair_sigs.as<const uint8_t* const>(); a.n_pairs = n_pairs;
  a.n_slots = ctx->n_slots; a.n_tiles = n_tiles;
  a.contig_off = ctx->d_off.as<int64_t>(); a.n_contigs = ctx->n_contigs;
  a.tile_n = ctx->d_site_tiles.as<int64_t>(); a.tile_incl = a.tile_n + items;
  a.sites = nullptr;
  MCOV_LAUNCH(ctx, kKCompareSiteCount, (k_compare_site_count<<<al_grid(ctx, items, 1), kCmpTileThreads, 0, s>>>(a)));
  CTX_CU(who, cudaGetLastError());
  int64_t total = 0;
  if (int rc = size_site_list(ctx, ctx->compare_sites, items, sizeof(mcov_compare_site), who, &total)) return rc;
  if (total > 0) {
    a.sites = ctx->compare_sites.list.as<mcov_compare_site>();
    MCOV_LAUNCH(ctx, kKCompareSiteWrite, (k_compare_site_write<<<al_grid(ctx, items, 1), kCmpTileThreads, 0, s>>>(a)));
    CTX_CU(who, cudaGetLastError());
    CTX_CU(who, cudaStreamSynchronize(s));
  }
  ctx->compare_sites.n = total;
  ctx->compare_sites.epoch = ctx->contig_epoch;
  *n_sites_out = total;
  return MCOV_OK;
}

extern "C" int mcov_compare_sites_read(mcov_ctx* ctx, int64_t first, int64_t n, mcov_compare_site* host_out) {
  if (!ctx) return MCOV_ERR_ARG;
  return read_site_list(ctx, ctx->compare_sites, first, n, host_out, sizeof(mcov_compare_site), "mcov_compare_sites_read",
                        "mcov_compare_sites");
}
