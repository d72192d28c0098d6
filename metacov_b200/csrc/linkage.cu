// linkage.cu -- haplotype counts between nearby SNV sites from the reads and their mates (include/metacov_b200.h:
// mcov_linkage, mcov_linkage_read; kernels in k_linkage.cuh, rules restated in oracle/linkage.py).
//
// Reads the counters (mcov_ctx::d_bc) for the sites and the records of the last device decode, or of a BAM file through
// the streamed decoder; writes only its own site list, scratch and pair list.  The depth store and its caches, the
// counters, the reference store and the allele and compare site lists are never written.
//
// Steps: the SNV site list (allele_site_list, use_reference 0) -> per site its slot, alleles and candidate partners,
// scanned into each site's first counter row -> the observations of every record (count, scan, write; in streamed mode
// batch by batch, appended, since mates may lie in different batches) -> one radix sort by (unit, site, base) -> the
// unit calls, compacted -> one atomicAdd per (unit, pair of called sites) -> the pairs with min_reads units (count, scan,
// write).
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <string>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <cuda/std/tuple>

#include "ctx.cuh"
#include "k_linkage.cuh"

using namespace mcov;

static_assert(sizeof(mcov_linkage_pair) == 32, "mcov_linkage_pair is 32 bytes");
static_assert(sizeof(LkObs) == 16, "an observation is 16 bytes");

namespace {

constexpr const char* kWho = "mcov_linkage";
constexpr const char* kHook = "MCOV_LINK_FREE_BYTES";

struct LkObsBits {               // the sort key: name, then sec
  __host__ __device__ ::cuda::std::tuple<uint64_t&, uint64_t&> operator()(LkObs& o) const { return {o.name, o.sec}; }
};

struct LkIsCall {
  int sb;
  __host__ __device__ bool operator()(const LkObs& o) const { return ((o.sec >> (61 - sb)) & 3u) < 2u; }
};

// ensure_fits_n with the linkage's test hook: `what` names the buffer, n its items
int fits(mcov_ctx* ctx, DevBuf& buf, size_t need, const char* what, long long n) {
  const std::string msg = std::string(what) + " need %zu bytes of device memory, %zu are free";
  std::string fmt = "%lld " + msg;
  return ensure_fits_n(ctx, buf, need, kHook, kWho, fmt.c_str(), n);
}

// buf grown to hold `need` bytes with its first `keep` bytes kept (the old allocation lives until the copy is done)
int grow_keep(mcov_ctx* ctx, DevBuf& buf, size_t keep, size_t need, long long n_obs) {
  if (need <= buf.cap) return MCOV_OK;
  if (keep == 0) return fits(ctx, buf, need, "observations:", n_obs);
  size_t free_b = 0, total_b = 0;
  CTX_CU(kWho, cudaMemGetInfo(&free_b, &total_b));
  if (const char* h = std::getenv(kHook)) free_b = (size_t)std::strtoull(h, nullptr, 10);
  const size_t want = DevBuf::grown(need);
  if (want > free_b) {
    char text[200];
    std::snprintf(text, sizeof(text),
                  "mcov_linkage: %lld observations: growing their buffer needs %zu bytes of device memory (%zu held), %zu are free",
                  n_obs, want, buf.cap, free_b);
    return ctx_fail(ctx, MCOV_ERR_NOMEM, text);
  }
  void* p = nullptr;
  CTX_CU(kWho, cudaMalloc(&p, want));
  cudaError_t e = cudaMemcpyAsync(p, buf.p, keep, cudaMemcpyDeviceToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  if (e != cudaSuccess) { cudaFree(p); return ctx_fail(ctx, MCOV_ERR_CUDA, "mcov_linkage: cudaMemcpyAsync", e); }
  buf.release();
  buf.p = p; buf.cap = want;
  return MCOV_OK;
}

BcArgs link_bc_args(mcov_ctx* ctx) {
  BcArgs a;
  std::memset(&a, 0, sizeof(a));
  a.contig_off = ctx->d_off.as<int64_t>(); a.contig_len = ctx->d_len.as<int32_t>(); a.n_contigs = ctx->n_contigs;
  a.skip_flags = (ctx->bc_mode & MCOV_BC_NOFILTER) ? 0u : kBcSkipAll;
  a.qthr = ctx->bc_qthr;
  a.err = ctx->d_lk_word.as<unsigned long long>();
  return a;
}

// The observations of the records [a.bc.i0, a.bc.n) appended to d_lk_obs[0] behind the *total held there.
int observe(mcov_ctx* ctx, LkObsArgs a, bool sam, int64_t* total) {
  const int64_t m = a.bc.n - a.bc.i0;
  if (m <= 0) return MCOV_OK;
  cudaStream_t s = ctx->stream;
  if (int rc = fits(ctx, ctx->d_lk_rec_n, (size_t)(m + 1) * 8, "records:", m)) return rc;
  if (int rc = fits(ctx, ctx->d_lk_rec_off, (size_t)(m + 1) * 8, "records:", m)) return rc;
  a.rec_n = ctx->d_lk_rec_n.as<int64_t>();
  a.rec_off = ctx->d_lk_rec_off.as<int64_t>();
  const unsigned grid = (unsigned)std::min<int64_t>((m + kLkWarps - 1) / kLkWarps, (int64_t)std::max(ctx->n_sm, 1) * 8);
  if (sam) MCOV_LAUNCH(ctx, kKLinkObsCount, (k_link_obs<BcSamRec, false><<<grid, kLkThreads, 0, s>>>(a)));
  else MCOV_LAUNCH(ctx, kKLinkObsCount, (k_link_obs<BcBamRec, false><<<grid, kLkThreads, 0, s>>>(a)));
  CTX_CU(kWho, cudaGetLastError());
  CTX_CU(kWho, cudaMemsetAsync(a.rec_n + m, 0, 8, s));
  size_t tb = 0;
  CTX_CU(kWho, cub::DeviceScan::ExclusiveSum(nullptr, tb, a.rec_n, ctx->d_lk_rec_off.as<int64_t>(), m + 1, s));
  if (int rc = fits(ctx, ctx->d_lk_tmp, tb, "records (scan scratch):", m)) return rc;
  CTX_CU(kWho, cub::DeviceScan::ExclusiveSum(ctx->d_lk_tmp.p, tb, a.rec_n, ctx->d_lk_rec_off.as<int64_t>(), m + 1, s));
  int64_t add = 0;
  CTX_CU(kWho, cudaMemcpyAsync(&add, ctx->d_lk_rec_off.as<int64_t>() + m, 8, cudaMemcpyDeviceToHost, s));
  CTX_CU(kWho, cudaStreamSynchronize(s));
  if (add == 0) return MCOV_OK;
  if (int rc = grow_keep(ctx, ctx->d_lk_obs[0], (size_t)*total * sizeof(LkObs), (size_t)(*total + add) * sizeof(LkObs),
                         (long long)(*total + add)))
    return rc;
  a.obs = ctx->d_lk_obs[0].as<LkObs>() + *total;
  if (sam) MCOV_LAUNCH(ctx, kKLinkObsWrite, (k_link_obs<BcSamRec, true><<<grid, kLkThreads, 0, s>>>(a)));
  else MCOV_LAUNCH(ctx, kKLinkObsWrite, (k_link_obs<BcBamRec, true><<<grid, kLkThreads, 0, s>>>(a)));
  CTX_CU(kWho, cudaGetLastError());
  *total += add;
  return MCOV_OK;
}

// The streamed decode's consumer: each batch's own records (like basecount.cu's CountSink, it carries none).
struct LinkSink : BamChunkSink {
  LkObsArgs base;
  int64_t done = 0, total = 0;
  explicit LinkSink(const LkObsArgs& a) : base(a) {}
  int batch(mcov_ctx* ctx, const BamChunk& b, int64_t* n_carry, int64_t* carry_ops) override {
    *n_carry = 0; *carry_ops = 0;
    LkObsArgs a = base;
    a.bc.tid = b.tid; a.bc.pos = b.pos; a.bc.flag = b.flag; a.bc.l_seq = b.l_seq; a.bc.cig_off = b.cig_off; a.bc.cig = b.cig;
    a.bc.data = b.data; a.bc.rec_off = b.rec_off;
    a.bc.i0 = b.n_carry; a.bc.n = b.n;
    a.bc.rec_base = done - b.n_carry;
    done += b.n - b.n_carry;
    return observe(ctx, a, false, &total);
  }
};

int bits_for(int64_t n) {        // bits that hold every index below n (at least 1)
  int b = 1;
  while (b < 62 && (n - 1) >> b) ++b;
  return b;
}

}  // namespace

extern "C" int mcov_linkage(mcov_ctx* ctx, const char* path, int64_t chunk_bytes, const mcov_linkage_params* params,
                            int64_t* n_pairs_out, mcov_linkage_info* info) {
  const char* who = kWho;
  if (!ctx) return MCOV_ERR_ARG;
  ctx->link_pairs.n = -1;
  if (!params || !n_pairs_out) return ctx_fail(ctx, MCOV_ERR_ARG, "mcov_linkage: null arguments");
  if (params->max_distance < 1 || params->max_distance > 100000 || params->min_reads < 1 || params->sites.use_reference != 0)
    return ctx_fail(ctx, MCOV_ERR_ARG, "mcov_linkage: need 1 <= max_distance <= 100000, min_reads >= 1 and sites.use_reference 0");
  AlleleParams P;
  if (int rc = al_check(ctx, &params->sites, &P, who)) return rc;
  mcov_ctx::BamDev& B = ctx->bam;
  if (!path && (B.n_rec < 0 || !B.data.p)) return ctx_fail(ctx, MCOV_ERR_STATE, "mcov_linkage: no file decoded on this context");
  CTX_CU(who, cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  mcov_linkage_info inf;
  std::memset(&inf, 0, sizeof(inf));

  // 1. the SNV sites; per site its slot, contig, alleles and first counter row
  int64_t ns = 0;
  if (int rc = allele_site_list(ctx, P, ctx->link_sites, who, &ns, kHook)) return rc;
  inf.n_sites = ns;
  int64_t n_pairs = 0;
  if (ns > 0) {
    const int sb = bits_for(ns);
    if (int rc = fits(ctx, ctx->d_lk_slot, (size_t)ns * 8, "sites:", ns)) return rc;
    if (int rc = fits(ctx, ctx->d_lk_tid, (size_t)ns * 4, "sites:", ns)) return rc;
    if (int rc = fits(ctx, ctx->d_lk_allele, (size_t)ns, "sites:", ns)) return rc;
    if (int rc = fits(ctx, ctx->d_lk_partners, (size_t)(ns + 1) * 8, "sites:", ns)) return rc;
    if (int rc = fits(ctx, ctx->d_lk_base, (size_t)(ns + 1) * 8, "sites:", ns)) return rc;
    int64_t* partners = ctx->d_lk_partners.as<int64_t>();
    int64_t* base = ctx->d_lk_base.as<int64_t>();
    MCOV_LAUNCH(ctx, kKLinkSites, (k_link_sites<<<al_grid(ctx, ns, kLkThreads), kLkThreads, 0, s>>>(
                                       ctx->link_sites.list.as<mcov_allele_site>(), ns, ctx->d_off.as<int64_t>(),
                                       params->max_distance, ctx->d_lk_slot.as<int64_t>(), ctx->d_lk_tid.as<int32_t>(),
                                       ctx->d_lk_allele.as<uint8_t>(), partners)));
    CTX_CU(who, cudaGetLastError());
    CTX_CU(who, cudaMemsetAsync(partners + ns, 0, 8, s));
    size_t tb = 0;
    CTX_CU(who, cub::DeviceScan::ExclusiveSum(nullptr, tb, partners, base, ns + 1, s));
    if (int rc = fits(ctx, ctx->d_lk_tmp, tb, "sites (scan scratch):", ns)) return rc;
    CTX_CU(who, cub::DeviceScan::ExclusiveSum(ctx->d_lk_tmp.p, tb, partners, base, ns + 1, s));
    int64_t n_cand = 0;
    CTX_CU(who, cudaMemcpyAsync(&n_cand, base + ns, 8, cudaMemcpyDeviceToHost, s));
    CTX_CU(who, cudaStreamSynchronize(s));
    inf.n_candidates = n_cand;

    // 2. the candidates' counters
    if (n_cand > 0) {
      if (int rc = fits(ctx, ctx->d_lk_cnt, (size_t)n_cand * 16, "candidate pairs:", n_cand)) return rc;
      CTX_CU(who, cudaMemsetAsync(ctx->d_lk_cnt.p, 0, (size_t)n_cand * 16, s));
    }

    // 3. the observations
    if (int rc = fits(ctx, ctx->d_lk_word, 24, "status words:", 3)) return rc;
    CTX_CU(who, cudaMemsetAsync(ctx->d_lk_word.p, 0xFF, 8, s));
    CTX_CU(who, cudaMemsetAsync(ctx->d_lk_word.as<uint8_t>() + 8, 0, 16, s));
    LkObsArgs a;
    std::memset(&a, 0, sizeof(a));
    a.bc = link_bc_args(ctx);
    a.slot = ctx->d_lk_slot.as<int64_t>(); a.n_sites = ns; a.sb = sb;
    int64_t n_obs = 0;
    if (path) {
      mcov_bam_gpu_stream_info sinfo;
      std::memset(&sinfo, 0, sizeof(sinfo));
      LinkSink sink(a);
      const int rc = bam_gpu_chunks(ctx, path, chunk_bytes, 1, &sinfo, who, sink);
      if (rc) return rc;
      n_obs = sink.total;
    } else {
      BcArgs& b = a.bc;
      b.tid = B.tid.as<int32_t>(); b.pos = B.pos.as<int32_t>(); b.flag = B.flag.as<uint16_t>(); b.l_seq = B.lseq.as<int32_t>();
      b.cig_off = B.cig_off.as<uint32_t>(); b.cig = B.cig.as<uint32_t>();
      b.data = B.data.as<uint8_t>(); b.rec_off = B.rec_off.as<uint64_t>(); b.aux = B.sam ? B.sam_aux.as<SamAux>() : nullptr;
      b.i0 = 0; b.n = B.n_rec;
      if (int rc = observe(ctx, a, B.sam, &n_obs)) return rc;
    }
    unsigned long long e = 0;
    CTX_CU(who, cudaMemcpyAsync(&e, ctx->d_lk_word.p, 8, cudaMemcpyDeviceToHost, s));
    CTX_CU(who, cudaStreamSynchronize(s));
    if (e != ~0ull) {
      char msg[256];
      std::snprintf(msg, sizeof(msg), (e & 3) == kBcErrQueryLong
                        ? "mcov_linkage: record %lld (0-based, file order): its CIGAR consumes more query bases than SEQ holds"
                        : "mcov_linkage: record %lld (0-based, file order): its SEQ / QUAL leave the record",
                    (long long)(e >> 2));
      return ctx_fail(ctx, MCOV_ERR_IO, msg);
    }
    inf.n_observations = n_obs;

    if (n_obs > 0) {
      // 4. sort by (unit, site, base); 5. the unit calls, compacted into the other buffer
      if (int rc = fits(ctx, ctx->d_lk_obs[1], (size_t)n_obs * sizeof(LkObs), "observations:", n_obs)) return rc;
      cub::DoubleBuffer<LkObs> keys(ctx->d_lk_obs[0].as<LkObs>(), ctx->d_lk_obs[1].as<LkObs>());
      const int begin_bit = 61 - sb;
      size_t sort_b = 0, sel_b = 0;
      CTX_CU(who, cub::DeviceRadixSort::SortKeys(nullptr, sort_b, keys, n_obs, LkObsBits{}, begin_bit, 128, s));
      CTX_CU(who, cub::DeviceSelect::If(nullptr, sel_b, keys.Current(), keys.Alternate(),
                                         ctx->d_lk_word.as<int64_t>() + 1, n_obs, LkIsCall{sb}, s));
      if (int rc = fits(ctx, ctx->d_lk_tmp, std::max(sort_b, sel_b), "observations (sort scratch):", n_obs)) return rc;
      MCOV_LAUNCH(ctx, kKLinkSort, CTX_CU(who, cub::DeviceRadixSort::SortKeys(ctx->d_lk_tmp.p, sort_b, keys, n_obs, LkObsBits{},
                                                                               begin_bit, 128, s)));
      LkObs* sorted = keys.Current();
      LkObs* other = keys.Alternate();
      MCOV_LAUNCH(ctx, kKLinkUnitCalls, (k_link_unit_calls<<<al_grid(ctx, n_obs, kLkThreads), kLkThreads, 0, s>>>(
                                             sorted, n_obs, ctx->d_lk_allele.as<uint8_t>(), sb, other,
                                             ctx->d_lk_word.as<unsigned long long>() + 2)));
      CTX_CU(who, cudaGetLastError());
      MCOV_LAUNCH(ctx, kKLinkSelect, CTX_CU(who, cub::DeviceSelect::If(ctx->d_lk_tmp.p, sel_b, other, sorted,
                                                                       ctx->d_lk_word.as<int64_t>() + 1, n_obs, LkIsCall{sb}, s)));
      int64_t words[2] = {0, 0};
      CTX_CU(who, cudaMemcpyAsync(words, ctx->d_lk_word.as<int64_t>() + 1, 16, cudaMemcpyDeviceToHost, s));
      CTX_CU(who, cudaStreamSynchronize(s));
      const int64_t n_calls = words[0];
      inf.n_units = words[1];

      LkPairArgs pa;
      std::memset(&pa, 0, sizeof(pa));
      pa.calls = sorted; pa.n_calls = n_calls; pa.sb = sb;
      pa.slot = ctx->d_lk_slot.as<int64_t>(); pa.tid = ctx->d_lk_tid.as<int32_t>(); pa.allele = ctx->d_lk_allele.as<uint8_t>();
      pa.base = base; pa.n_sites = ns; pa.contig_off = ctx->d_off.as<int64_t>();
      pa.max_distance = params->max_distance; pa.min_reads = params->min_reads;
      pa.cnt = ctx->d_lk_cnt.as<uint32_t>(); pa.n_cand = n_cand;
      // 6. the haplotype counts; 7. the pairs with min_reads units
      if (n_cand > 0 && n_calls > 1) {
        MCOV_LAUNCH(ctx, kKLinkPairs, (k_link_pairs<<<al_grid(ctx, n_calls, kLkThreads), kLkThreads, 0, s>>>(pa)));
        CTX_CU(who, cudaGetLastError());
        const int64_t n_tiles = (n_cand + kLkTile - 1) / kLkTile;
        if (int rc = fits(ctx, ctx->d_site_tiles, (size_t)n_tiles * 16, "candidate tiles:", n_tiles)) return rc;
        pa.n_tiles = n_tiles;
        pa.tile_n = ctx->d_site_tiles.as<int64_t>(); pa.tile_incl = pa.tile_n + n_tiles;
        MCOV_LAUNCH(ctx, kKLinkPairCount, (k_link_pair_count<<<al_grid(ctx, n_tiles, 1), kLkTileThreads, 0, s>>>(pa)));
        CTX_CU(who, cudaGetLastError());
        if (int rc = size_site_list(ctx, ctx->link_pairs, n_tiles, sizeof(mcov_linkage_pair), who, &n_pairs, kHook)) return rc;
        if (n_pairs > 0) {
          pa.pairs = ctx->link_pairs.list.as<mcov_linkage_pair>();
          MCOV_LAUNCH(ctx, kKLinkPairWrite, (k_link_pair_write<<<al_grid(ctx, n_tiles, 1), kLkTileThreads, 0, s>>>(pa)));
          CTX_CU(who, cudaGetLastError());
          CTX_CU(who, cudaStreamSynchronize(s));
        }
      }
    }
  }
  ctx->link_pairs.n = n_pairs;
  ctx->link_pairs.epoch = ctx->contig_epoch;
  *n_pairs_out = n_pairs;
  if (info) *info = inf;
  return MCOV_OK;
}

extern "C" int mcov_linkage_read(mcov_ctx* ctx, int64_t first, int64_t n, mcov_linkage_pair* host_out) {
  if (!ctx) return MCOV_ERR_ARG;
  return read_site_list(ctx, ctx->link_pairs, first, n, host_out, sizeof(mcov_linkage_pair), "mcov_linkage_read",
                        "mcov_linkage");
}
