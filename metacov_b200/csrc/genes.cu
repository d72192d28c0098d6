// genes.cu -- codons of genes from the A / C / G / T counts of mcov_base_counts and the reference store
// (include/metacov_b200.h: mcov_gene_run, mcov_gene_sites_read; kernels in k_genes.cuh).
//
// Reads the counters (mcov_ctx::d_bc) and the reference store (d_ref); writes only the allele calls' scratch and its
// own site list.  The depth store, its caches, the counters, the reference store and the allele, compare and linkage
// lists are never written.
#include <algorithm>
#include <cstdio>
#include <string>
#include <vector>

#include "ctx.cuh"
#include "k_genes.cuh"

using namespace mcov;

static_assert(sizeof(mcov_gene_stats) == 96, "mcov_gene_stats is 96 bytes");
static_assert(sizeof(mcov_gene_site) == 32, "mcov_gene_site is 32 bytes");
static_assert(sizeof(GnChunk) == 40, "GnChunk is 40 bytes");

namespace {

constexpr const char* kHook = "MCOV_GENE_FREE_BYTES";

int check_genes(mcov_ctx* ctx, int64_t g, const int32_t* tid, const int32_t* start, const int32_t* end,
                const int32_t* strand, const int32_t* phase, const mcov_gene_stats* out, const char* who) {
  if (g < 0 || (g > 0 && (!tid || !start || !end || !strand || !phase || !out)))
    return ctx_fail(ctx, MCOV_ERR_ARG, std::string(who) + ": bad arguments");
  for (int64_t i = 0; i < g; ++i) {
    if (tid[i] < 0 || tid[i] >= ctx->n_contigs || start[i] < 0 || start[i] >= end[i] || end[i] > ctx->len[tid[i]] ||
        (strand[i] != 1 && strand[i] != -1) || phase[i] < 0 || phase[i] > 2) {
      char msg[240];
      std::snprintf(msg, sizeof(msg), "%s: gene %lld: need a valid tid, 0 <= start < end <= the contig's length, strand "
                    "+1 or -1 and phase 0-2", who, (long long)i);
      return ctx_fail(ctx, MCOV_ERR_ARG, msg);
    }
  }
  return MCOV_OK;
}

// Every gene's codon span cut into chunks of at most kGnChunk codons in genomic order: chunks to ctx->d_chunks, the meta
// [first[g + 1] | length[g] | codons[g]] to d_chunk_meta, d_region_out sized for the records, d_chunk_part for the
// partials.
int upload_gene_chunks(mcov_ctx* ctx, int64_t g, const int32_t* tid, const int32_t* start, const int32_t* end,
                       const int32_t* strand, const int32_t* phase, const char* who, int64_t* n_chunks) {
  cudaStream_t s = ctx->stream;
  std::vector<GnChunk> chunks;
  std::vector<int64_t> meta((size_t)(3 * g + 1));
  int64_t* first = meta.data();
  int64_t* length = first + g + 1;
  int64_t* codons = length + g;
  for (int64_t i = 0; i < g; ++i) {
    first[i] = (int64_t)chunks.size();
    length[i] = (int64_t)end[i] - start[i];
    const int32_t K = (int32_t)(std::max<int64_t>(length[i] - phase[i], 0) / 3);
    codons[i] = K;
    const int32_t cs = strand[i] > 0 ? start[i] + phase[i] : end[i] - phase[i] - 3 * K;   // the span's first position
    for (int32_t c = 0; c < K; c += kGnChunk) {
      GnChunk ch;
      ch.slot = ctx->off[tid[i]] + cs + 3 * (int64_t)c; ch.gene = i;
      ch.tid = tid[i]; ch.pos = cs + 3 * c; ch.n = std::min(kGnChunk, K - c);
      ch.codon0 = strand[i] > 0 ? c : K - 1 - c; ch.dir = strand[i]; ch.pad = 0;
      chunks.push_back(ch);
    }
  }
  first[g] = (int64_t)chunks.size();
  const int64_t nc = (int64_t)chunks.size();
  CTX_CU(who, ctx->d_chunk_meta.ensure(meta.size() * 8));
  CTX_CU(who, ctx->d_region_out.ensure((size_t)g * sizeof(mcov_gene_stats)));
  CTX_CU(who, cudaMemcpyAsync(ctx->d_chunk_meta.p, meta.data(), meta.size() * 8, cudaMemcpyHostToDevice, s));
  if (nc > 0) {
    CTX_CU(who, ctx->d_chunks.ensure((size_t)nc * sizeof(GnChunk)));
    CTX_CU(who, ctx->d_chunk_part.ensure((size_t)nc * sizeof(GnPart)));
    CTX_CU(who, cudaMemcpyAsync(ctx->d_chunks.p, chunks.data(), (size_t)nc * sizeof(GnChunk), cudaMemcpyHostToDevice, s));
  }
  *n_chunks = nc;
  return MCOV_OK;
}

}  // namespace

extern "C" int mcov_gene_run(mcov_ctx* ctx, int64_t g, const int32_t* tid, const int32_t* start, const int32_t* end,
                             const int32_t* strand, const int32_t* phase, const mcov_allele_params* params,
                             mcov_gene_stats* host_out, int64_t* n_sites_out) {
  const char* who = "mcov_gene_run";
  if (!ctx) return MCOV_ERR_ARG;
  const bool with_sites = n_sites_out != nullptr;
  if (with_sites) ctx->gene_sites.n = -1;
  if (int rc = check_genes(ctx, g, tid, start, end, strand, phase, host_out, who)) return rc;
  if (params && params->use_reference != 1)
    return ctx_fail(ctx, MCOV_ERR_ARG, std::string(who) + ": the gene rules need use_reference = 1");
  AlleleParams P;
  if (int rc = al_check(ctx, params, &P, who)) return rc;
  CTX_CU(who, cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  int64_t nc = 0;
  if (int rc = upload_gene_chunks(ctx, g, tid, start, end, strand, phase, who, &nc)) return rc;
  GnArgs a;
  a.cnt = ctx->d_bc.as<uint4>(); a.ref = ctx->d_ref.as<uint8_t>();
  a.chunks = ctx->d_chunks.as<GnChunk>(); a.n_chunks = nc;
  a.part = ctx->d_chunk_part.as<GnPart>();
  a.tile_n = nullptr; a.tile_incl = nullptr; a.sites = nullptr; a.P = P;
  if (with_sites && nc > 0) {
    // [nc] record counts a chunk, then [nc] their inclusive scan
    if (int rc = ensure_fits_n(ctx, ctx->d_site_tiles, (size_t)nc * 16, kHook, who,
                               "the counts of %lld gene chunks need %zu bytes of device memory, %zu are free", nc))
      return rc;
    a.tile_n = ctx->d_site_tiles.as<int64_t>(); a.tile_incl = a.tile_n + nc;
  }
  if (nc > 0) {
    MCOV_LAUNCH(ctx, kKGeneChunks, (k_gene_chunks<<<al_grid(ctx, nc, kGnWarps), kGnThreads, 0, s>>>(a)));
    CTX_CU(who, cudaGetLastError());
  }
  if (g > 0) {
    const int64_t* d_meta = ctx->d_chunk_meta.as<int64_t>();
    MCOV_LAUNCH(ctx, kKGeneCombine, (k_gene_combine<<<al_grid(ctx, g, kGnWarps), kGnThreads, 0, s>>>(
                                         a.part, d_meta, d_meta + g + 1, d_meta + 2 * g + 1, g,
                                         ctx->d_region_out.as<mcov_gene_stats>())));
    CTX_CU(who, cudaGetLastError());
    CTX_CU(who, cudaMemcpyAsync(host_out, ctx->d_region_out.p, (size_t)g * sizeof(mcov_gene_stats), cudaMemcpyDeviceToHost, s));
  }
  int64_t total = 0;
  if (with_sites && nc > 0) {
    if (int rc = size_site_list(ctx, ctx->gene_sites, nc, sizeof(mcov_gene_site), who, &total, kHook)) return rc;
    if (total > 0) {
      a.sites = ctx->gene_sites.list.as<mcov_gene_site>();
      MCOV_LAUNCH(ctx, kKGeneSiteWrite, (k_gene_site_write<<<al_grid(ctx, nc, kGnWarps), kGnThreads, 0, s>>>(a)));
      CTX_CU(who, cudaGetLastError());
    }
  }
  CTX_CU(who, cudaStreamSynchronize(s));
  if (with_sites) {
    ctx->gene_sites.n = total;
    ctx->gene_sites.epoch = ctx->contig_epoch;
    *n_sites_out = total;
  }
  return MCOV_OK;
}

extern "C" int mcov_gene_sites_read(mcov_ctx* ctx, int64_t first, int64_t n, mcov_gene_site* host_out) {
  if (!ctx) return MCOV_ERR_ARG;
  return read_site_list(ctx, ctx->gene_sites, first, n, host_out, sizeof(mcov_gene_site), "mcov_gene_sites_read",
                        "mcov_gene_run with n_sites_out");
}
