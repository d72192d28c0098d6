/* metacov_b200.h -- C-ABI of the B200-native coverage hot path.
 *
 * Drop-in boundary for the coverage path of epruesse/metacov.  The reference
 * has no FFI of its own for this path: its boundary is the Python surface
 * (metacov/pileup.py:9 `classic`, metacov/scan.pyx:623 `scan_reads`) on top of
 * the pysam object protocol (`AlignmentFile.pileup` pileup.py:13, `.fetch`
 * pileup.py:90, raw `bam1_t` fields scan.pyx:243-294).  Every entry point below
 * names the reference interface it replaces.  Plain C: pointers and sizes only.
 *
 * Conventions
 *   - every function returns MCOV_OK (0) or a negative mcov_status; nothing
 *     throws across the ABI; `mcov_last_error(ctx)` has the message.
 *   - one context per GPU; a context is NOT thread-safe.
 *   - work is enqueued on the context's CUDA stream; calls that hand results
 *     to host memory synchronise that stream before returning.
 *   - the caller owns every array it passes; host arrays passed to
 *     `mcov_push_reads` may be reused as soon as the call returns.
 *   - there is no CPU fallback: without a CUDA device `mcov_create` fails.
 */
#ifndef METACOV_B200_H
#define METACOV_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MCOV_ABI_VERSION 1

typedef enum mcov_status {
  MCOV_OK = 0,
  MCOV_ERR_ARG = -1,      /* bad argument (null pointer, negative size, bad tid ...) */
  MCOV_ERR_STATE = -2,    /* call out of order (e.g. push after finalize)            */
  MCOV_ERR_CUDA = -3,     /* CUDA runtime error, text in mcov_last_error             */
  MCOV_ERR_NOMEM = -4,
  MCOV_ERR_IO = -5,       /* BAM/BGZF/BAI decode error                               */
  MCOV_ERR_RANGE = -6,    /* value outside what the kernels represent exactly        */
  MCOV_ERR_UNSORTED = -7  /* sorted-only entry point fed unsorted reads              */
} mcov_status;

typedef enum mcov_mem_kind {
  MCOV_MEM_HOST = 0,      /* pageable or pinned host memory  */
  MCOV_MEM_DEVICE = 1     /* device memory on the ctx's GPU  */
} mcov_mem_kind;

typedef struct mcov_ctx mcov_ctx;

/* The implicit arguments of `bam.pileup(ref, start, end)` (reference
 * metacov/pileup.py:13 calls it with pysam's defaults) made explicit.
 * Defaults = pysam stepper "samtools": see SURVEY.md Appendix A-1/A-2. */
typedef struct mcov_filter {
  uint16_t flag_filter;    /* drop if (flag & flag_filter)            default 0x704 */
  uint16_t flag_require;   /* if !=0 drop unless (flag & flag_require) default 0    */
  uint8_t  min_mapq;       /* drop if mapq < min_mapq                 default 0     */
  uint8_t  ignore_orphans; /* drop paired && !proper_pair             default 1     */
  uint8_t  count_del;      /* 1: positions under D / N ops count (`column.n`, what the reference reads,
                              pileup.py:16); 0: only M = X positions count (like get_num_aligned()) --
                              additive; computed by the any-order formulation        default 1 */
  uint8_t  reflen0_as_one; /* a passing read whose CIGAR consumes no reference: 0 = contributes nothing
                              (current htslib), 1 = occupies the one position `pos` (older htslib);
                              SURVEY.md Appendix A-4                                 default 0 */
  int32_t  max_depth;      /* htslib maxcnt; <=0 disables the cap     default 8000  */
} mcov_filter;

/* Exact integer statistics of one region [start,end) of one contig; the host
 * finishes `classic`'s seven outputs (reference metacov/pileup.py:18-26) from
 * these without touching the depth again.  64 bytes. */
typedef struct mcov_region_stats {
  int64_t  sum;        /* sum of depth                       -> 'sum', 'avg'           */
  uint64_t sumsq;      /* sum of depth^2                     -> 'std'                  */
  int64_t  iq_sum;     /* sum of sorted depth[n/4 : n-n/4)   -> 'q23'                  */
  int64_t  n_ge1;      /* positions with depth >= 1          (breadth; additive)       */
  int64_t  n_geN;      /* positions with depth >= breadth_n  (breadth; additive)       */
  int32_t  min;        /*                                    -> 'min'                  */
  int32_t  max;        /*                                    -> 'max'                  */
  int32_t  med_lo;     /* sorted depth[(n-1)/2]              -> 'med' = (lo+hi)/2      */
  int32_t  med_hi;     /* sorted depth[n/2]                                            */
  int32_t  reserved;
  int32_t  flags;      /* bit0: order statistics valid; bit1: depth overflowed the
                          histogram range and the radix path was used                 */
} mcov_region_stats;

/* ---- context ------------------------------------------------------------ */

/* device: CUDA ordinal.  stream: a cudaStream_t (e.g. torch's current stream
 * handle) or NULL for a stream owned by the context. */
int  mcov_create(mcov_ctx** out, int device, void* stream);
void mcov_destroy(mcov_ctx* ctx);
const char* mcov_last_error(const mcov_ctx* ctx);
int  mcov_abi_version(void);

/* Replaces `AlignmentFile.references/.lengths` as the shape of the depth
 * store (reference metacov/util.py:64-69 iterates them; pileup.py:10-11
 * allocates one float64 vector per region -- here ONE int32 array holds every
 * contig: contig c owns len[c]+1 slots starting at a 16-byte aligned offset). */
int  mcov_set_contigs(mcov_ctx* ctx, int32_t n_contigs, const int32_t* len);
int64_t mcov_n_slots(const mcov_ctx* ctx);
/* slot offset of contig `tid` inside the depth array */
int64_t mcov_contig_offset(const mcov_ctx* ctx, int32_t tid);

/* Optional: caller-owned device buffer (e.g. a torch.int32 tensor) of at
 * least mcov_n_slots() elements to hold the depth.  The caller must not write
 * it between a depth pass and the statistics of that pass: the statistics of
 * large regions may be taken from per-tile histograms counted by the pass. */
int  mcov_bind_depth(mcov_ctx* ctx, int32_t* dev, int64_t n_slots);

int  mcov_set_filter(mcov_ctx* ctx, const mcov_filter* f);
void mcov_default_filter(mcov_filter* f);

/* Start a new pass: clears the difference array and all counters. */
int  mcov_begin(mcov_ctx* ctx);

/* mcov_begin with flags.  MCOV_BEGIN_EXACT_CAP: the pass also counts, per
 * slot, the passing reads that start there (an int32 array the size of the
 * depth store, allocated on first use), and mcov_finalize reports the exact
 * cap_metric max_p depth[p-1]+starts[p] within each contig (depth[-1] = 0) --
 * the value the fused path reports for the same reads, whatever their order:
 * when it does not exceed max_depth, htslib's cap cannot fire.  Without a cap
 * (max_depth <= 0) nothing is counted, and with count_del = 0 cap_metric stays
 * the upper bound of mcov_begin -- also when mcov_set_filter switches to either
 * inside the pass (the starts would miss the reads pushed after it). */
#define MCOV_BEGIN_EXACT_CAP 1
int  mcov_begin_ex(mcov_ctx* ctx, int flags);

/* Replaces the per-record work of htslib's pileup engine behind
 * `bam.pileup()` (reference metacov/pileup.py:13): filter each record, reduce
 * its CIGAR to a reference length, and add +1 @ pos / -1 @ pos+reflen to the
 * difference array.  SoA layout = the `bam1_t.core` fields the reference reads
 * at scan.pyx:243-294.  cig_off has n+1 entries (offsets into cig); cig holds
 * BAM-encoded ops (len<<4 | op).  Any order of reads is accepted. */
int  mcov_push_reads(mcov_ctx* ctx, int64_t n,
                     const int32_t* tid, const int32_t* pos,
                     const uint16_t* flag, const uint8_t* mapq,
                     const uint32_t* cig_off, const uint32_t* cig,
                     int mem_kind);

/* Prefix-scan the difference array into per-base depth.  Afterwards
 * depth(tid, p) = value of `column.n` at that position (pileup.py:16). */
int  mcov_finalize(mcov_ctx* ctx);

/* One-call variant for coordinate-sorted input: expansion, scan and depth
 * materialisation fused in one pass over the slot space (no separate clear,
 * no atomics to L2).  Returns MCOV_ERR_UNSORTED if the reads are not sorted
 * by (tid,pos); the caller then uses begin/push/finalize. */
int  mcov_depth_sorted(mcov_ctx* ctx, int64_t n,
                       const int32_t* tid, const int32_t* pos,
                       const uint16_t* flag, const uint8_t* mapq,
                       const uint32_t* cig_off, const uint32_t* cig,
                       int mem_kind);

/* Batches of 2^32 or more CIGAR ops (long reads: BASELINE config 5 at full size
 * is 5 M reads with 1.4e10 ops): the same two entry points with 64-bit offsets.
 * wait = 0 defers the verdict like mcov_depth_sorted_async. */
int  mcov_depth_sorted_wide(mcov_ctx* ctx, int64_t n,
                            const int32_t* tid, const int32_t* pos,
                            const uint16_t* flag, const uint8_t* mapq,
                            const uint64_t* cig_off, const uint32_t* cig,
                            int mem_kind, int wait);
int  mcov_push_reads_wide(mcov_ctx* ctx, int64_t n,
                          const int32_t* tid, const int32_t* pos,
                          const uint16_t* flag, const uint8_t* mapq,
                          const uint64_t* cig_off, const uint32_t* cig,
                          int mem_kind);

/* Same, but returns without waiting for the GPU: the sortedness verdict
 * (MCOV_ERR_UNSORTED / MCOV_ERR_RANGE) is delivered by the next call that
 * synchronises -- mcov_region_stats_run, mcov_copy_depth, mcov_pass_info_get. */
int  mcov_depth_sorted_async(mcov_ctx* ctx, int64_t n,
                             const int32_t* tid, const int32_t* pos,
                             const uint16_t* flag, const uint8_t* mapq,
                             const uint32_t* cig_off, const uint32_t* cig,
                             int mem_kind);

/* Streaming a coordinate-sorted file in batches (the reference never holds the file:
 * metacov/scan.pyx:653-667 loops over `cnext()`, pileup.py:13 iterates htslib's
 * streaming pileup).  mcov_stream_begin starts a pass; every mcov_stream_push adds the
 * next batch in file order through the fused sorted path and makes the depth FINAL up
 * to the 2048-slot tile that holds the batch's last read; the last push (last = 1)
 * finishes the slot space.  What crosses a batch border travels as DATA, like the
 * boundary reads of a contig cut between GPUs: each push returns a resend point
 * (resend_tid, resend_pos), and the next batch must BEGIN with a copy of every read of
 * the earlier batches that starts at or after that point or whose interval
 * [pos, pos + reflen) reaches past it, in file order (n_carry = how many such reads
 * lead the batch; they are not counted twice in mcov_pass_info).  Sending more than
 * required is harmless as long as the order is kept.  The final push carries the last
 * resend set too (n may equal n_carry).  The sortedness verdict is delivered by the
 * first synchronising call after the last push.  A file in which htslib's max_depth
 * cap fires is reported (MCOV_ERR_STATE) rather than replayed: the replay needs a
 * contig's reads in one batch.  mcov_stream_resend_point computes the resend point a
 * batch ending with the read (last_tid, last_pos) will return (host arithmetic only). */
int  mcov_stream_begin(mcov_ctx* ctx);
int  mcov_stream_push(mcov_ctx* ctx, int64_t n, int64_t n_carry,
                      const int32_t* tid, const int32_t* pos,
                      const uint16_t* flag, const uint8_t* mapq,
                      const uint32_t* cig_off, const uint32_t* cig,
                      int mem_kind, int last,
                      int32_t* resend_tid, int32_t* resend_pos);
int  mcov_stream_resend_point(const mcov_ctx* ctx, int32_t last_tid, int32_t last_pos,
                              int32_t* resend_tid, int32_t* resend_pos);

/* Compact HOST transport of a coordinate-sorted batch (the PCIe link bounds the
 * end-to-end rate): instead of tid[n] the per-contig read prefix
 * contig_read_start[n_contigs+1] (reads [crs[c], crs[c+1]) belong to contig c,
 * reads from crs[n_contigs] on are unplaced); instead of cig_off[n+1] the u16 op
 * counts n_cigar[n] (BAM's own limit); mapq may be NULL when min_mapq == 0.  The
 * SoA columns are rebuilt on the device (k_unpack_reads + scan).  All arrays are
 * host memory.  wait=0 defers the sortedness verdict like _async. */
int  mcov_depth_sorted_packed(mcov_ctx* ctx, int64_t n,
                              const int64_t* contig_read_start, const int32_t* pos,
                              const uint16_t* flag, const uint8_t* mapq /* nullable */,
                              const uint16_t* n_cigar, const uint32_t* cig, int64_t n_cig_total,
                              int wait);

/* Narrower still (7.3 bytes per read on config C2 instead of 12.6): positions as u16
 * differences to the previous read of the same contig (first read of a contig: to
 * 0; unplaced reads form one more segment), with the differences that do not fit
 * 0..65535 listed as exceptions (exc_index ascending or not, exc_delta = the true
 * 32-bit difference; dpos of those reads is ignored); u8 op counts and u16 ops
 * (len << 4 | op) -- a batch with a CIGAR of more than 255 ops or an op longer than
 * 4095 takes mcov_depth_sorted_packed instead.  Rebuilt on the device
 * (k_delta_seed / k_delta_patch, one int32 prefix sum, k_delta_finish). */
int  mcov_depth_sorted_delta(mcov_ctx* ctx, int64_t n,
                             const int64_t* contig_read_start, const uint16_t* dpos,
                             int64_t n_exc, const uint32_t* exc_index, const int32_t* exc_delta,
                             const uint16_t* flag, const uint8_t* mapq /* may be NULL */,
                             const uint8_t* n_cigar, const uint16_t* cig, int64_t n_cig_total, int wait);

/* ---- the transport block: what the host decoder hands to the GPU ----------------
 * ONE contiguous host buffer per batch of coordinate-sorted reads -> ONE host-to-device
 * copy; the SoA columns are rebuilt on the device.  The end-to-end rate is bound by the
 * PCIe link, so the block is as narrow as the data allows (config C2: 1.4 bytes per
 * read instead of 19.6 for the plain columns):
 *   crs      int64[n_contigs+1]  reads [crs[c], crs[c+1]) belong to contig c, reads from
 *                                crs[n_contigs] on are unplaced (instead of tid[n])
 *   dpos     u8[n]               position - position of the previous read of the same
 *                                contig (first read of a contig: - 0); differences outside
 *                                0..255 are listed as exceptions (exc_idx u32 ASCENDING,
 *                                exc_val i32)
 *   fc       u8[n]               index into the joint table jt[<=255] of the batch's most
 *                                frequent (flag, CIGAR class) pairs (u16 flag, u8 class);
 *                                255 = the pair is listed as an escape (esc_idx u32
 *                                ASCENDING, esc_flag u16, esc_cls u8)
 *   CIGAR class                  < 128: the read's whole CIGAR is dictionary entry `class`
 *                                (dict_off u32[n_dict+1], dict_ops u32[]: the batch's most
 *                                frequent CIGARs of up to four ops); >= 128: class - 128
 *                                explicit ops follow in xops[] in read order: u16
 *                                (len << 4 | op) when every explicit op of the batch is
 *                                shorter than 4096 (xop_bytes = 2), else u32
 *   mapq     u8[n]               only when the filter asks for it (min_mapq > 0)
 * NIBBLE FORM (nib = 1; chosen by the packer when it is the smaller one -- deep short-read
 * data, where most differences are below 15 and a handful of (flag, CIGAR) pairs cover
 * most reads; config C2: 1.4 bytes per read): dpos[] and fc[] are replaced by
 *   nb       u8[n]               low nibble: the position difference 0..14, or 15 = the
 *                                difference (15..255) is the next entry of dq u8[] (reads
 *                                listed as exceptions carry 0); high nibble: the joint-table
 *                                index 0..14, or 15 = the index (15..254, 255 = escape) is
 *                                the next entry of fq u8[]
 * and, in both forms, a CHUNK TABLE (mcov_block_chunk per 2048 reads): where the chunk's
 * entries of dq / fq / xops and of the escape and exception lists begin, the op offset of
 * its first read and the position of the read before it -- all the packer has at hand, and
 * all a CTA needs to rebuild its 2048 reads without looking at any other chunk (ONE unpack
 * kernel, no device-side prefix sums).
 * A batch with a CIGAR of more than 127 ops (long reads) does not qualify
 * (mcov_pack_block returns MCOV_ERR_RANGE): it travels as plain columns or through
 * mcov_depth_sorted_packed.  All sections start on 16-byte boundaries. */
#define MCOV_BLOCK_MAGIC 0x4256434Du   /* "MCVB" */
typedef struct mcov_block_hdr {
  uint32_t magic, version;                     /* version 4 */
  int64_t  n, n_carry, n_cigar, n_exc, n_esc, n_xops, total_bytes;
  int32_t  n_contigs, n_jt, n_dict, n_dictops, has_mapq, xop_bytes;   /* xop_bytes: 2 or 4 (width of an explicit op) */
  int32_t  last_tid, last_pos;                 /* the batch's last read (streams: how far the depth becomes final) */
  uint32_t off_crs, off_dpos, off_exc_idx, off_exc_val, off_fc, off_jt, off_esc_idx, off_esc_flag, off_esc_cls,
           off_dict_off, off_dict_ops, off_xops, off_mapq, nib;         /* nib: 1 = nibble form (off_dpos = off_fc = 0) */
  int64_t  n_dq, n_fq;                         /* nibble form: entries of the two side lists */
  uint32_t off_nb, off_dq, off_fq, off_chunk;
} mcov_block_hdr;
#define MCOV_BLOCK_CHUNK 2048                  /* reads per entry of the chunk table (and per CTA of the unpack kernel) */
typedef struct mcov_block_chunk {
  uint32_t dq_off, fq_off;                     /* nibble form: first entry of dq / fq that belongs to the chunk */
  uint32_t op_off, xop_off;                    /* cig_off of the chunk's first read; first explicit op of the chunk */
  int32_t  pos_carry;                          /* position of the read in front of the chunk (0 for the first chunk) */
  uint32_t esc_first, exc_first;               /* first escape / exception at or after the chunk's first read that lies in the chunk (0xFFFFFFFF: none) */
  uint32_t reserved;
} mcov_block_chunk;
/* Upper bound of the block size for a batch of n reads with n_cigar ops over n_contigs contigs. */
int64_t mcov_block_bound(int64_t n, int64_t n_cigar, int32_t n_contigs);
/* Pack a coordinate-sorted SoA batch (host arrays, grouped by contig with unplaced reads last; the first
 * n_carry reads are repeats of earlier batches, see mcov_stream_push) into `out` (capacity cap bytes, 16-byte
 * aligned; pinned memory makes the copy asynchronous).  mapq may be NULL.  n_threads <= 0: all cores.
 * Returns MCOV_OK and the size in *bytes_out, MCOV_ERR_ARG (not grouped by contig, cap too small) or
 * MCOV_ERR_RANGE (a CIGAR of more than 127 ops). */
int  mcov_pack_block(int64_t n, int64_t n_carry, const int32_t* tid, const int32_t* pos, const uint16_t* flag,
                     const uint8_t* mapq, const uint32_t* cig_off, const uint32_t* cig, int32_t n_contigs,
                     void* out, int64_t cap, int64_t* bytes_out, int n_threads);
/* The fused sorted pass from a transport block in host memory (wait = 0 defers the verdict like
 * mcov_depth_sorted_async), and one batch of a streamed pass (see mcov_stream_push; the block's n_carry
 * leading reads are the repeats).  These two calls do NOT wait for the host-to-device copy of the
 * block (the host goes on preparing the next batch while the link is busy): the block must stay
 * unchanged until the next call on the context that takes reads has returned, or until mcov_sync /
 * a call that delivers results (the streaming reader's two block buffers satisfy this). */
int  mcov_depth_sorted_block(mcov_ctx* ctx, const void* block, int64_t bytes, int wait);
int  mcov_stream_push_block(mcov_ctx* ctx, const void* block, int64_t bytes, int last,
                            int32_t* resend_tid, int32_t* resend_pos);
/* The columns a transport block widens into on the device (k_block.cuh), copied back to host arrays of n
 * (cig_off: n + 1, cig: n_cigar) entries; any output may be NULL.  mapq reads 0xff when the block carries none.
 * What a caller uses to check a block it built itself, and the test suite to pin the unpack kernels column by
 * column.  Synchronises; leaves the depth untouched. */
int  mcov_block_unpack(mcov_ctx* ctx, const void* block, int64_t bytes, int32_t* tid, int32_t* pos, uint16_t* flag,
                       uint8_t* mapq, uint32_t* cig_off, uint32_t* cig);

/* Replaces the seven reductions of `classic` (reference
 * metacov/pileup.py:18-26) for g regions at once (the loop at cli.py:85-95).
 * tid/start/end are host arrays; 0 <= start <= end.  Positions >= len[tid]
 * count as depth 0 (the reference's vector is end-start long, pileup.py:10-11).
 * breadth_n: threshold of n_geN.  host_out: g structs.  Synchronises.
 * When the max_depth cap fired in the pass (mcov_pass_info.cap_contigs > 0), a
 * region that starts inside a replayed contig is replayed again with its own
 * iterator -- only the reads overlapping it, as bam.pileup(ref, start, end)
 * feeds htslib (pileup.py:13) -- and its record computed from that. */
int  mcov_region_stats_run(mcov_ctx* ctx, int64_t g,
                           const int32_t* tid, const int32_t* start, const int32_t* end,
                           int32_t breadth_n, mcov_region_stats* host_out);

/* Pipelined variant of mcov_region_stats_run for callers that process batch
 * after batch: `submit` enqueues the statistics kernels, the copy of the g
 * records into pinned staging slot `slot` (0 or 1) and the copy of the pass
 * verdict, and returns without synchronising -- the caller may enqueue the next
 * depth pass right away (same stream: it runs after these kernels).  `collect`
 * waits for that slot, delivers the verdict of the pass the statistics belong
 * to and copies the records to host_out.  What cannot be done once a later
 * pass may have overwritten the depth is reported instead of approximated:
 * MCOV_ERR_STATE if the max_depth cap fired in that pass and a region of the
 * slot starts inside its contig (it needs its own iterator over reads that may
 * be gone), or a region's depth left the counting histogram (run the batch
 * again through mcov_depth_sorted + mcov_region_stats_run). */
int  mcov_region_stats_submit(mcov_ctx* ctx, int64_t g,
                              const int32_t* tid, const int32_t* start, const int32_t* end,
                              int32_t breadth_n, int slot);
int  mcov_region_stats_collect(mcov_ctx* ctx, int slot, mcov_region_stats* host_out);
/* Same, without the copy: *view points at the g records in the slot's pinned
 * staging buffer (owned by the context, valid until the next submit on that
 * slot).  The records are copied back on a stream of their own, so the kernels
 * of the next pass do not queue behind a large copy (500 k regions = 32 MB). */
int  mcov_region_stats_collect_view(mcov_ctx* ctx, int slot, const mcov_region_stats** view, int64_t* g_out);

/* Asynchronous variant for multi-GPU pipelines: the g records are written to
 * DEVICE memory dev_out on the context's stream and the call returns without
 * synchronising (the records can be handed to a collective on the same
 * stream).  Regions whose flags carry bit1 (depth beyond the counting
 * histogram) need mcov_region_stats_run for exact order statistics; zero-length
 * regions are not zeroed; a pending sortedness verdict is not delivered. */
int  mcov_region_stats_enqueue(mcov_ctx* ctx, int64_t g,
                               const int32_t* tid, const int32_t* start, const int32_t* end,
                               int32_t breadth_n, mcov_region_stats* dev_out);

/* Regions cut across devices (SURVEY.md 8(e): a contig split between ranks at
 * position p; the boundary reads are given to both sides and clipped there, see
 * metacov_b200/sharding.py).  A region that straddles the cut cannot be finished
 * from 64-byte records -- `med` and `q23` (reference pileup.py:21,24) need the
 * merged multiset -- so each rank ADDS the exact counting histogram of its part
 * of every such region to dev_hist[g][MCOV_HIST_BINS] (device memory, zeroed by
 * the caller; last bin = overflow), the tables are summed across ranks (one
 * all-reduce) and mcov_hist_stats_enqueue walks the merged histograms into the
 * same records mcov_region_stats_run produces (flags bit1 set if the overflow
 * bin is populated).  Both are enqueued on the context's stream;
 * mcov_region_hist_enqueue returns after its task table has been consumed. */
#define MCOV_HIST_BINS 8192
int  mcov_region_hist_enqueue(mcov_ctx* ctx, int64_t g,
                              const int32_t* tid, const int32_t* start, const int32_t* end,
                              uint32_t* dev_hist);
int  mcov_hist_stats_enqueue(mcov_ctx* ctx, int64_t g, const uint32_t* dev_hist,
                             int32_t breadth_n, mcov_region_stats* dev_out);

/* Run-length export of the per-base depth of the contigs [tid0, tid1) -- the rows
 * of a bedGraph file (additive feature, SURVEY.md 8(f) row 4; the reference keeps
 * its `columns` vector private, pileup.py:10-26).  A run is a maximal stretch of
 * equal depth inside one contig, zero-depth runs included.  mcov_depth_runs
 * computes the runs on the GPU, keeps them in the context and reports their
 * number; mcov_depth_runs_read copies runs [first, first+n) to host arrays
 * (tid, start, end, depth; 0-based half-open, position order).  The depth must
 * not be recomputed between the two calls. */
int  mcov_depth_runs(mcov_ctx* ctx, int32_t tid0, int32_t tid1, int64_t* n_runs_out);
int  mcov_depth_runs_read(mcov_ctx* ctx, int64_t first, int64_t n,
                          int32_t* tid, int32_t* start, int32_t* end, int32_t* depth);

/* Fixed-window mean depth (additive feature named by north_star; no
 * reference counterpart): for every contig, ceil(len/window) float64 means,
 * concatenated in tid order into host_out (n_out = total windows). */
int  mcov_window_means(mcov_ctx* ctx, int32_t window, double* host_out, int64_t n_out);

/* Replaces reading `column.n` back one column at a time (pileup.py:13-16). */
int  mcov_copy_depth(mcov_ctx* ctx, int32_t tid, int32_t start, int32_t end, int32_t* host_out);
/* Device pointer to the depth array (valid after finalize / depth_sorted).
 * The caller may write through it: later statistics read the depth again. */
int32_t* mcov_depth_ptr(mcov_ctx* ctx);

/* Counters of the last pass. */
typedef struct mcov_pass_info {
  int64_t n_reads;        /* records pushed                                   */
  int64_t n_pass;         /* records that passed the filter with reflen > 0   */
  int64_t aligned_bases;  /* sum of reflen over passing reads (unclipped)     */
  int32_t max_depth_seen; /* max depth over all contigs (before the cap)      */
  int32_t cap_metric;     /* max_p depth[p-1]+starts[p] (fused path, and
                             push passes begun with MCOV_BEGIN_EXACT_CAP) or
                             an upper bound of it (other push passes)         */
  int32_t sorted;         /* 1 if the input was coordinate-sorted             */
  int32_t cap_contigs;    /* contigs whose depth was replayed under the max_depth
                             cap (fused path; 0 = the cap never fired)        */
} mcov_pass_info;
int  mcov_pass_info_get(mcov_ctx* ctx, mcov_pass_info* out);

/* ---- launch accounting and per-kernel timing (bench / profiling support) -- */

typedef struct mcov_kernel_time {
  char    name[32];
  int64_t launches;
  double  total_ms;   /* CUDA-event time summed over the launches, on the ctx's stream */
} mcov_kernel_time;

/* Wait for everything enqueued on the context's stream (for callers that mix the *_enqueue entry
 * points with work on other streams). */
int  mcov_sync(mcov_ctx* ctx);
/* Copy n_bytes of device memory owned by the context (e.g. the columns of mcov_bam_dev) to the host. */
int  mcov_copy_to_host(mcov_ctx* ctx, const void* dev, void* host, int64_t n_bytes);

/* kernels (and clears) enqueued by this context since it was created */
int64_t mcov_launch_count(const mcov_ctx* ctx);
/* The cached statistics plan (the regions of the last mcov_region_stats_* call): CTAs of the large-region stream and
 * regions it splits between CTAs (0 and 0 before any plan). */
int  mcov_region_plan_info(const mcov_ctx* ctx, int32_t* stream_ctas, int32_t* split_regions);
/* on=1: bracket every kernel launch with CUDA events and reset the totals; on=0: stop. */
int  mcov_profile_enable(mcov_ctx* ctx, int on);
/* Synchronises; fills up to cap entries; returns the number written (>=0) or an error. */
int  mcov_profile_read(mcov_ctx* ctx, mcov_kernel_time* out, int cap);

/* ---- read-statistics scan (metacov scan) --------------------------------- */

/* Replaces `ByFlag.process_read` + `IsizeHist.process_read` over every record
 * (reference metacov/scan.pyx:406-420, 590-610; getter semantics
 * scan.pyx:267-271: isize counts only if PROPER_PAIR, else bin 0).
 * group_flags: the user-ordered flag masks of ByFlag (MSB first, scan.pyx:
 * 414-418); n_groups_out = 2^n_group_flags.  hist_out: host u32
 * [2^n_group_flags][n_bins]; |isize| >= n_bins is reported through
 * *max_isize_out so the caller can retry with a larger table.
 * group_counts_out: host u64[2^n_group_flags] reads per group. */
int  mcov_isize_hist(mcov_ctx* ctx, int64_t n,
                     const uint16_t* flag, const int32_t* isize, int mem_kind,
                     int32_t n_group_flags, const uint16_t* group_flags,
                     int32_t n_bins, uint32_t* hist_out,
                     uint64_t* group_counts_out, int32_t* max_isize_out);

/* Replaces `KmerHist.process_read` over every record (reference
 * metacov/scan.pyx:503-522 with the sequence decoding of scan.pyx:240-259): reads
 * shorter than OFFSET+STEP*NK are skipped; for i < NK the k-mer at read position
 * OFFSET+i*STEP (first base in the low bits, any non-ACGT base -> bin 4^K) is
 * counted in hist[group][kmer][i].  seq_win = per-read windows from
 * mcov_bam_seq_windows (win_bases >= OFFSET+(NK-1)*STEP+K).  Host arrays;
 * hist_out: u32[2^n_group_flags][4^K+1][NK].  K <= 12, OFFSET >= 0. */
int  mcov_kmer_hist(mcov_ctx* ctx, int64_t n, const uint16_t* flag, const int32_t* l_seq,
                    const uint8_t* seq_win, int32_t win_bytes, int32_t win_bases,
                    int32_t K, int32_t NK, int32_t STEP, int32_t OFFSET,
                    int32_t n_group_flags, const uint16_t* group_flags, uint32_t* hist_out);
/* The same with flag / l_seq / seq_win in host or DEVICE memory (mem_kind): a file decoded on the GPU
 * (mcov_bam_decode_gpu + mcov_bam_gpu_names_seq into device buffers) is scanned without its columns or its
 * SEQ windows ever crossing the bus -- the `scan` loop of scan.pyx:653-667 with nothing on the host. */
int  mcov_kmer_hist_mem(mcov_ctx* ctx, int64_t n, const uint16_t* flag, const int32_t* l_seq,
                        const uint8_t* seq_win, int mem_kind, int32_t win_bytes, int32_t win_bases,
                        int32_t K, int32_t NK, int32_t STEP, int32_t OFFSET,
                        int32_t n_group_flags, const uint16_t* group_flags, uint32_t* hist_out);

/* ---- the second coverage definition: pileup.experimental ------------------ */

/* Per-region sums behind the 13 outputs of `experimental` (reference
 * metacov/pileup.py:150-173).  With L = end-start and the reference's names:
 *   cov   = cov_sum / L            covc = covw_sum / L
 *   den   = n_starts / L           denc = cor_sum / L        cf = cor_sum / n_starts
 *   cov2  = cov2_sum / L           wnf  = wnf_sum / L
 *   nz    = L - n_starts           allreads = secondary + nreads + improper
 * no_reflen counts the proper-pair reads whose `reference_length` is None
 * (the reference raises TypeError on the first one, pileup.py:134-137). */
typedef struct mcov_exp_stats {
  double  covw_sum;
  double  cor_sum;
  double  wnf_sum;
  int64_t cov_sum;
  int64_t cov2_sum;
  int32_t n_starts;
  int32_t nreads;
  int32_t secondary;
  int32_t improper;
  int32_t no_reflen;
  int32_t n_pairs;
} mcov_exp_stats;

/* Replaces the read loop of `experimental(bam, k_cor, k_len, fasta, ref, start,
 * end)` (reference metacov/pileup.py:90-146) for g regions of ONE contig set in
 * a coordinate-sorted file.  Host arrays (file order): pos, flag, cig_off[n+1],
 * cig as for mcov_push_reads; name_hash = mcov_bam_name_hash (the reference joins
 * mates through a dict keyed by query_name); kmer_code = mcov_bam_qas_kmer(k_len)
 * (-1 = the lookup raises KeyError); kcor[2][4^k_len] / kcor_has[2][4^k_len] =
 * the two dicts of load_kmerhist as tables (index: first base most significant,
 * A0 C1 G2 T3; kcor_has = key present); k_len <= 12, or kcor == NULL for "no
 * correction" (every lookup raises KeyError -> rcor = 1).  Region i covers
 * [r_start[i], r_end[i]) of the contig whose reads are the records
 * [r_lb[i], r_ub[i]) -- any superset of the records `bam.fetch` would return
 * (the kernel applies the exact overlap test).  out: host, g records. */
int  mcov_experimental_run(mcov_ctx* ctx, int64_t n, const int32_t* pos, const uint16_t* flag,
                           const uint32_t* cig_off, const uint32_t* cig, const uint64_t* name_hash,
                           const int32_t* kmer_code, int32_t k_len, const double* kcor, const uint8_t* kcor_has,
                           int32_t g, const int32_t* r_start, const int32_t* r_end,
                           const int64_t* r_lb, const int64_t* r_ub, mcov_exp_stats* out);

/* cor_revsum of reference metacov/pileup.py:78-83: out[i] = sum over j <
 * min(L-i, n_w) of w[j] * cor_rev[i+j] (the O(L*900) loop of np.inner calls). */
int  mcov_exp_revsum(mcov_ctx* ctx, int64_t L, const double* cor_rev, int32_t n_w, const double* w, double* out);

/* ---- host BAM decoding (replaces pysam.AlignmentFile, cli.py:56, 211) ---- */

typedef struct mcov_bam mcov_bam;

int  mcov_bam_open(mcov_bam** out, const char* path, char* err, int errlen);
void mcov_bam_close(mcov_bam* b);
int32_t mcov_bam_n_ref(const mcov_bam* b);
const char* mcov_bam_ref_name(const mcov_bam* b, int32_t tid);
int32_t mcov_bam_ref_len(const mcov_bam* b, int32_t tid);
const char* mcov_bam_header_text(const mcov_bam* b);
/* BAI metadata pseudo-bin sums (pysam `.mapped` / `.unmapped`, cli.py:73-75);
 * returns MCOV_ERR_IO if there is no index next to the BAM. */
int  mcov_bam_index_stats(const mcov_bam* b, int64_t* mapped, int64_t* unmapped);
/* Same from the path of the .bam file (looks for <path>.bai, then <path minus .bam>.bai). */
int  mcov_bai_stats(const char* bam_path, int64_t* mapped, int64_t* unmapped);
/* Decode the whole file (every record, like IteratorRowAll scan.pyx:204) into
 * SoA arrays owned by the handle; pointers stay valid until close. */
int  mcov_bam_load(mcov_bam* b, int n_threads);
int64_t mcov_bam_n_records(const mcov_bam* b);
int64_t mcov_bam_n_cigar(const mcov_bam* b);
const int32_t*  mcov_bam_tid(const mcov_bam* b);
const int32_t*  mcov_bam_pos(const mcov_bam* b);
const uint16_t* mcov_bam_flag(const mcov_bam* b);
const uint8_t*  mcov_bam_mapq(const mcov_bam* b);
const int32_t*  mcov_bam_lseq(const mcov_bam* b);
const int32_t*  mcov_bam_isize(const mcov_bam* b);
const uint32_t* mcov_bam_cig_off(const mcov_bam* b);
const uint32_t* mcov_bam_cig(const mcov_bam* b);
/* Packed SEQ (only the k-mer histogram needs it) and the per-read windows it is
 * cut into: out[n][(win_bases+1)/2], forward reads their first win_bases bases,
 * reverse reads their last win_bases (nt16, high nibble first, missing = 15). */
int  mcov_bam_load_seq(mcov_bam* b);
int  mcov_bam_seq_windows(const mcov_bam* b, int32_t win_bases, uint8_t* out);
/* FNV-1a 64 of every read name (`read.query_name`, pileup.py:101); valid after mcov_bam_load_seq. */
const uint64_t* mcov_bam_name_hash(const mcov_bam* b);
/* out[n]: 2-bit code of the first k_len bases of `read.query_alignment_sequence` (pileup.py:109,
 * 123; first base most significant, A0 C1 G2 T3), -1 when shorter or not ACGT.  k_len <= 15. */
int  mcov_bam_qas_kmer(const mcov_bam* b, int32_t k_len, int32_t* out);

/* ---- streaming host reader: a BAM read, inflated and parsed in batches ------
 * Replaces the record loop of reference metacov/scan.pyx:653-667 (`cnext()` over
 * pysam's IteratorRowAll) for the coverage path without ever holding the file:
 * mcov_bam_stream_next decodes the next `batch_reads` records (BGZF blocks inflated on
 * n_threads host threads, 0 = all) into PINNED SoA buffers owned by the stream (two
 * sets, so batch k can still be copied to the GPU while batch k+1 is decoded; a
 * batch's arrays stay valid until the second call after the one that returned them)
 * and puts in front of them the reads of the earlier batches that mcov_stream_push
 * asked to see again: pass the resend point it returned (resend_tid < 0 on the first
 * call).  Returns 1 with *out filled, 0 after the batch flagged `last`, or a negative
 * mcov_status (mcov_bam_stream_error has the text). */
typedef struct mcov_bam_stream mcov_bam_stream;
typedef struct mcov_bam_batch {
  int64_t n;              /* reads in the batch, carried ones included        */
  int64_t n_carry;        /* leading reads repeated from earlier batches       */
  int64_t n_cigar;        /* CIGAR ops of the batch                            */
  int32_t last;           /* 1: the file ends with this batch                  */
  int32_t reserved;
  const int32_t*  tid;
  const int32_t*  pos;
  const uint16_t* flag;
  const uint8_t*  mapq;
  const int32_t*  l_seq;
  const int32_t*  isize;
  const int32_t*  reflen; /* reference length of each read (sum of M D N = X)  */
  const uint32_t* cig_off;   /* n + 1 */
  const uint32_t* cig;
} mcov_bam_batch;
int  mcov_bam_stream_open(mcov_bam_stream** out, const char* path, int64_t batch_reads, int n_threads, char* err, int errlen);
void mcov_bam_stream_close(mcov_bam_stream* s);
int32_t mcov_bam_stream_n_ref(const mcov_bam_stream* s);
const char* mcov_bam_stream_ref_name(const mcov_bam_stream* s, int32_t tid);
int32_t mcov_bam_stream_ref_len(const mcov_bam_stream* s, int32_t tid);
const char* mcov_bam_stream_header_text(const mcov_bam_stream* s);
const char* mcov_bam_stream_error(const mcov_bam_stream* s);
int  mcov_bam_stream_next(mcov_bam_stream* s, int32_t resend_tid, int32_t resend_pos, mcov_bam_batch* out);
int64_t mcov_bam_stream_records(const mcov_bam_stream* s);   /* distinct records handed out so far */
/* Same, and the batch packed as a transport block in pinned memory owned by the stream (valid like the
 * batch's arrays).  *block is NULL when the batch does not qualify (long-read CIGARs, unsorted file):
 * push the columns of *out instead. */
int  mcov_bam_stream_next_block(mcov_bam_stream* s, int32_t resend_tid, int32_t resend_pos, int with_mapq,
                                const void** block, int64_t* bytes, mcov_bam_batch* out);

/* BAM writer (bench / test support): SoA columns -> BGZF-compressed BAM (+ the metadata-only .bai the
 * coverage path reads); names "r<i>", pseudo-random ACGT bases, no qualities.  level: zlib level. */
int  mcov_bam_write(const char* path, int32_t n_ref, const char* const* ref_name, const int32_t* ref_len, int64_t n,
                    const int32_t* tid, const int32_t* pos, const uint16_t* flag, const uint8_t* mapq,
                    const uint32_t* cig_off, const uint32_t* cig, const int32_t* isize, int level, int n_threads);

/* ---- synthetic workloads (bench / test support; include/mcov_synth.h) ---- */

struct mcov_synth_params;

/* ---- GPU-side BAM decode (SURVEY.md 8(f) row 3) ----------------------------
 * Replaces, for the coverage path, `pysam.AlignmentFile` + `IteratorRowAll`
 * (reference metacov/scan.pyx:204, 216; cli.py:56) without the host decode of
 * mcov_bam_open / mcov_bam_load: the COMPRESSED file image goes to the device,
 * every BGZF block is inflated by one GPU thread, the record chain is walked in
 * parallel (guessed segment starts, every link verified: exact) and the SoA
 * columns are written to device memory owned by the context -- valid until the
 * next mcov_bam_decode_gpu or mcov_destroy, and ready for
 * mcov_depth_sorted(..., MCOV_MEM_DEVICE).  file_bytes: the whole .bam file in
 * host memory (pinned memory makes the copy fast).  The inflated stream and
 * the SoA must fit the device.  `inflated` points at the inflated stream
 * (header_bytes = offset of the first alignment record: magic, header text and
 * the reference table lie before it). */
typedef struct mcov_bam_dev {
  int64_t n_records, n_cigar, inflated_bytes, header_bytes, n_segments;
  int32_t n_ref, reserved;
  const int32_t*  tid;
  const int32_t*  pos;
  const uint16_t* flag;
  const uint8_t*  mapq;
  const int32_t*  l_seq;
  const int32_t*  isize;
  const uint32_t* cig_off;   /* n_records + 1 */
  const uint32_t* cig;
  const uint8_t*  inflated;
} mcov_bam_dev;
int  mcov_bam_decode_gpu(mcov_ctx* ctx, const void* file_bytes, int64_t n_bytes, int verify_crc, mcov_bam_dev* out);
/* The same straight from the file (the image is mapped, not read into a buffer of the caller's). */
int  mcov_bam_decode_gpu_file(mcov_ctx* ctx, const char* path, int verify_crc, mcov_bam_dev* out);
/* SAM text decoded on the device into the same columns.  The header (the '@'
 * lines before the first record; references from @SQ SN:/LN:) is read on the
 * host; the whole image goes to the device in chunks of chunk_bytes (0: 64 MiB)
 * while the newlines of each copied chunk are counted, and the lines are parsed
 * there (SAM spec 1.4 with the BAM encoding of htslib's sam_parse1: POS-1,
 * RNAME '*' -> -1, an RNAME that is not an @SQ name is an error, CIGAR ops
 * len<<4|op, l_seq = length of SEQ or 0 for '*'; optional fields are skipped).
 * `inflated` points at the text and header_bytes is the header's length;
 * n_segments is 0.  A malformed line is MCOV_ERR_IO and mcov_last_error names
 * its 1-based line number and the field; more than 2^32-1 CIGAR ops in the file
 * is MCOV_ERR_RANGE.  The columns are valid until the next decode on the
 * context, like those of mcov_bam_decode_gpu.  Synchronises. */
int  mcov_sam_decode_gpu(mcov_ctx* ctx, const void* bytes, int64_t n_bytes, int64_t chunk_bytes, mcov_bam_dev* out);
int  mcov_sam_decode_gpu_file(mcov_ctx* ctx, const char* path, int64_t chunk_bytes, mcov_bam_dev* out);
/* SAM text that arrives in pieces (a pipe, stdin), decoded a chunk of whole
 * lines at a time into the same columns.  mcov_sam_chunk_begin takes the
 * header -- every '@' line in front of the first record and nothing else --,
 * validates it like mcov_sam_decode_gpu, uploads the @SQ table and starts the
 * line count; n_ref (optional) receives the number of @SQ lines.
 * mcov_sam_chunk_decode parses every complete line of bytes[0, n) (through
 * its last LF; everything when `last` is set, the final line may then lack its
 * LF) and sets *consumed to the bytes it parsed: the caller keeps the rest in
 * front of its next piece.  *consumed == 0 without `last` means the piece held
 * no complete line.  The columns of `out` describe this chunk only (indices
 * local to it, header_bytes 0) and stay valid until the next decode on the
 * context, as do mcov_bam_gpu_names_seq and mcov_bam_gpu_mapped, which serve
 * this chunk.  A malformed line is MCOV_ERR_IO naming its 1-based line number
 * in the whole stream (header lines and the lines of earlier chunks
 * included); a '@' line after the header is such an error.  Synchronises: the
 * caller may reuse `bytes` when the call returns. */
int  mcov_sam_chunk_begin(mcov_ctx* ctx, const void* header_bytes, int64_t n, int32_t* n_ref);
int  mcov_sam_chunk_decode(mcov_ctx* ctx, const void* bytes, int64_t n, int last, int64_t* consumed, mcov_bam_dev* out);
/* The longest line of the stream begun by mcov_sam_chunk_begin, over the chunks
 * decoded so far: its bytes with the LF (a last line without an LF: to the end
 * of the stream); counted on the device from each chunk's line index.  -1
 * without a chunked decode. */
int64_t mcov_sam_chunk_longest_line(const mcov_ctx* ctx);
/* pysam's `mapped` / `unmapped` of the file last decoded on this context (BAM or
 * SAM), counted on the device from its columns with the BAI metadata
 * definitions: mapped = records with tid >= 0 and without flag 0x4, unmapped =
 * every other record.  Synchronises. */
int  mcov_bam_gpu_mapped(mcov_ctx* ctx, int64_t* mapped, int64_t* unmapped);
/* Test hook: the SAM rules of mcov_sam_decode_gpu (the same field helpers,
 * csrc/k_sam.cuh) run line by line on the host, so that the CPU suite can
 * check them.  Not a product path: the decoders have no CPU fallback.  With
 * tid == NULL only the counts are filled (n_records, n_cigar, n_ref,
 * header_bytes); otherwise every non-NULL array must hold n_records entries
 * (cig_off n_records + 1, cig n_cigar, seq_win n_records x (win_bases+1)/2).
 * name_hash / kmer_code / seq_win are the outputs of mcov_bam_gpu_names_seq.
 * MCOV_ERR_IO on a malformed line: fail_line (1-based) and fail_field (0-10 =
 * QNAME..QUAL, 11 = fewer than 11 fields or an empty line, 12 = a header line
 * after a record) are set and err holds the message. */
typedef struct mcov_sam_host_cols {
  int64_t n_records, n_cigar, header_bytes, fail_line;
  int32_t n_ref, fail_field, k_len, win_bases;
  int32_t* tid; int32_t* pos; uint16_t* flag; uint8_t* mapq; int32_t* l_seq; int32_t* isize;
  uint32_t* cig_off; uint32_t* cig;
  uint64_t* name_hash; int32_t* kmer_code; uint8_t* seq_win;
} mcov_sam_host_cols;
int  mcov_sam_parse_host(const void* bytes, int64_t n_bytes, mcov_sam_host_cols* cols, char* err, int err_len);
/* Read names and SEQ of the file last decoded on this context (BAM or SAM), computed on the
 * device from the inflated stream or the SAM text (no host reader is opened).  Each output is
 * optional (NULL = not wanted) and lies in host or device memory per mem_kind:
 *   name_hash_out  u64[n]  FNV-1a 64 of `read.query_name`, the key of the
 *                  reference's mate dict (metacov/pileup.py:101-118)
 *                  == mcov_bam_name_hash;
 *   kmer_code_out  i32[n]  code of `query_alignment_sequence[0:k_len]`
 *                  (pileup.py:109-110, 123), -1 = no key  == mcov_bam_qas_kmer;
 *   seq_win_out    u8[n][(win_bases+1)/2]  the read's first (forward) / last
 *                  (reverse) win_bases bases as nt16 nibbles, what the k-mer
 *                  histogram reads (scan.pyx:240-259, 513-520)
 *                  == mcov_bam_seq_windows.
 * MCOV_ERR_STATE without a decoded file, MCOV_ERR_IO if a record's SEQ leaves
 * the record.  Synchronises. */
int  mcov_bam_gpu_names_seq(mcov_ctx* ctx, int32_t k_len, int32_t win_bases,
                            uint64_t* name_hash_out, int32_t* kmer_code_out, uint8_t* seq_win_out, int mem_kind);

/* A BAM of ANY size through the GPU decoder into the streamed depth pass: the file
 * is read chunk_bytes at a time (<= 0: 64 MiB) into pinned memory by a host thread
 * while the GPU inflates the previous chunk, establishes its record chain (a record
 * cut by the chunk border is completed with the next chunk), writes the columns and
 * pushes them, led by the reads the pass wants again, through mcov_stream_push from
 * device memory.  The host does nothing but read().  Replaces the `cnext()` loop of
 * reference metacov/scan.pyx:653-667 over a file that is never held.  Needs the
 * file's contig table (mcov_set_contigs; header e.g. from mcov_bam_stream_open);
 * on MCOV_OK the depth is ready (statistics, copies, exports).  A file that is not
 * coordinate sorted is reported by the first synchronising call after it
 * (MCOV_ERR_UNSORTED), like mcov_stream_push. */
typedef struct mcov_bam_gpu_stream_info {
  int64_t n_records, n_chunks, n_segments, inflated_bytes, file_bytes, max_carry;
} mcov_bam_gpu_stream_info;
int  mcov_bam_gpu_stream_depth(mcov_ctx* ctx, const char* path, int64_t chunk_bytes, int verify_crc,
                               mcov_bam_gpu_stream_info* info);
/* A / C / G / T counts at every reference position: pysam's
 * AlignmentFile.count_coverage over the whole file, on the device.
 * mcov_base_counts counts the records of the file last decoded on this
 * context (mcov_bam_decode_gpu*, mcov_sam_decode_gpu*: path NULL), or of the BAM
 * file at `path` read through the streamed decoder chunk_bytes at a time (<= 0:
 * 64 MiB; like mcov_bam_gpu_stream_depth, the context's contig table must be
 * the file's, and the columns of an earlier decode are gone afterwards).  The
 * context's contig table (mcov_set_contigs) places the counts.
 *   Records: those placed on a contig (0 <= tid < n_contigs, pos >= 0), minus
 *   those with a flag of 0x4 | 0x100 | 0x200 | 0x400 (MCOV_BC_ALL, pysam's
 *   read_callback="all"; MCOV_BC_NOFILTER skips none).  A record without SEQ
 *   counts nothing.  Every (query, reference) pair of an M, = or X op counts
 *   at its reference position when the base is A, C, G or T and, with
 *   quality_threshold != 0, the read has qualities (BAM: first QUAL byte not
 *   0xFF; SAM: QUAL not '*') and the base's quality is >= quality_threshold
 *   (a negative threshold only asks for qualities).  Pairs at or past the
 *   contig's end are dropped.  No MAPQ or orphan filter, no max_depth cap;
 *   the pileup filter of mcov_set_filter does not apply.
 *   Any read order: one warp per read (k_bc_any), global atomics.
 * The counts live apart from the depth store, which, with its statistics
 * caches, is left as it was.  MCOV_ERR_NOMEM, before anything is allocated,
 * when the 16 bytes a slot do not fit the free device memory (the message
 * holds both byte counts); MCOV_ERR_IO naming the first record (0-based, file
 * order) whose CIGAR consumes more query bases than its SEQ holds -- nothing
 * is read past SEQ or QUAL --, or whose SEQ / QUAL leave the BAM record;
 * MCOV_ERR_STATE without contigs or a decoded file.  After an error the
 * context is usable and holds no counts.  Synchronises. */
enum {
  MCOV_BC_ALL = 0,        /* skip unmapped, secondary, QC-fail and duplicate records */
  MCOV_BC_NOFILTER = 1    /* count every placed record                               */
};
int  mcov_base_counts(mcov_ctx* ctx, const char* path, int64_t chunk_bytes, int32_t quality_threshold, int mode);
/* The counts of the last mcov_base_counts at [start, end) of contig tid into
 * host_out[4 * (end - start)]: the A counts, then C, G and T, each end - start
 * long.  MCOV_ERR_STATE without counts for the current contig table,
 * MCOV_ERR_ARG for a region outside the contig.  Synchronises. */
int  mcov_copy_base_counts(mcov_ctx* ctx, int32_t tid, int32_t start, int32_t end, uint32_t* host_out);

/* Alleles from the counts of the last mcov_base_counts (csrc/alleles.cu; the
 * rules are restated in oracle/alleles.py).  At a position with counts n_A,
 * n_C, n_G, n_T and N their 64-bit sum:
 *   covered    N >= min_coverage;
 *   present    allele b: n_b >= min_count and (double)n_b >= min_freq * (double)N;
 *   consensus  the largest count, ties to the first of A C G T;
 *   pi_p       1 - ((fA*fA + fC*fC) + (fG*fG + fT*fT)), f_b = (double)n_b / N,
 *              in this order and without FMA contraction (bit-identical to numpy);
 *   kind       at a covered position: 1 SNV (two or more alleles present),
 *              2 SUB (reference base known, consensus differs), 4 POPSUB
 *              (reference base known, some allele present, the reference's not).
 * The reference base of a position is A, C, G or T from mcov_set_reference
 * (case-insensitive); anything else, or use_reference = 0, is unknown.
 * min_coverage >= 1, min_count >= 1, 0 <= min_freq <= 1, use_reference 0 / 1,
 * else MCOV_ERR_ARG.  MCOV_ERR_STATE without counts for the current contig
 * table, or with use_reference while some contig has had no mcov_set_reference
 * since the last mcov_set_contigs.  The depth store, its statistics caches and
 * the counts are never written; after an error the context is usable. */
typedef struct mcov_allele_params {
  uint32_t min_coverage, min_count;
  double   min_freq;
  int32_t  use_reference;
  int32_t  pad;
} mcov_allele_params;
/* One region: length = end - start (positions past the contig end have zero
 * counts), depth_sum = sum of N, pi_sum = sum of pi_p over covered positions
 * (summed in a fixed order: the same counts give the same bits), the others
 * count positions.  64 bytes. */
typedef struct mcov_allele_stats {
  int64_t length, covered, depth_sum;
  double  pi_sum;
  int64_t snv, ref_covered, sub, popsub;
} mcov_allele_stats;
/* One site (kind != 0): 0-based position, the counts, ref 'A' 'C' 'G' 'T' or
 * 'N' (unknown), consensus 'A' 'C' 'G' or 'T', kind bits.  32 bytes. */
typedef struct mcov_allele_site {
  int32_t  tid, pos;
  uint32_t cnt[4];
  uint8_t  ref, consensus, kind, pad[5];
} mcov_allele_site;
/* The reference of contig tid: n ASCII bytes, n the contig's length, kept on
 * the device (one byte a slot) until the next mcov_set_contigs.  MCOV_ERR_NOMEM,
 * before anything is allocated, when the store does not fit the free device
 * memory (the message holds both byte counts).  Synchronises. */
int  mcov_set_reference(mcov_ctx* ctx, int32_t tid, const char* ascii, int32_t n);
/* The records of g regions [start, end) of contig tid (0 <= start <= end; a
 * region may overlap others and reach past its contig) into host_out[g].
 * Synchronises. */
int  mcov_allele_stats_run(mcov_ctx* ctx, int64_t g, const int32_t* tid, const int32_t* start, const int32_t* end,
                           const mcov_allele_params* params, mcov_allele_stats* host_out);
/* Every site of every contig, in slot order (= by tid, then pos), into a list
 * kept on the device; their number in *n_sites_out.  Synchronises. */
int  mcov_allele_sites(mcov_ctx* ctx, const mcov_allele_params* params, int64_t* n_sites_out);
/* The sites [first, first + n) of the last mcov_allele_sites into host_out[n].
 * MCOV_ERR_STATE without a list for the current contig table, MCOV_ERR_ARG for
 * a range outside it.  Synchronises. */
int  mcov_allele_sites_read(mcov_ctx* ctx, int64_t first, int64_t n, mcov_allele_site* host_out);

/* Samples compared position by position (csrc/compare.cu; the rules are
 * restated in oracle/compare.py).  A sample keeps one signature byte a slot,
 * made from its counts with the allele rules above (no reference):
 *   0x80       covered;
 *   bits 4-5   the consensus (0-3 = A C G T);
 *   bits 0-3   the present mask (bit b: allele b present);
 * 0x00 where not covered, and in every padding and end slot.  For a pair
 * (a, b) at a position: compared = covered in both; the allele set of a sample
 * is its present mask OR its consensus' bit (never empty where covered);
 * con_snp = compared and the consensuses differ; pop_snp = compared and the
 * two allele sets are disjoint (a pop_snp is always a con_snp).  The pair calls
 * take sig[n_sig], device arrays of mcov_n_slots(ctx) signature bytes on ctx's
 * GPU (4-byte aligned) made under a contig table equal to ctx's, and
 * pairs[2 * n_pairs], indices into sig with a != b.  MCOV_ERR_ARG for fewer
 * than two signatures, no pair, a pair index out of range or a == b, a pointer
 * that is null or not device memory on ctx's GPU, or a bad region;
 * MCOV_ERR_STATE without a contig table.  The depth store, its caches, the
 * counts and the reference store are never written; after an error the
 * context is usable. */
/* One (pair, region): length = end - start, positions covered in a, in b, in
 * both (compared), con_snp and pop_snp positions.  48 bytes. */
typedef struct mcov_compare_stats {
  int64_t length, covered_a, covered_b, compared, con_snp, pop_snp;
} mcov_compare_stats;
/* One site of a pair (a con_snp position): the pair's index, the position, both
 * signature bytes, kind bits 1 con_snp (always set), 2 pop_snp.  16 bytes. */
typedef struct mcov_compare_site {
  int32_t pair, tid, pos;
  uint8_t sig_a, sig_b, kind, pad;
} mcov_compare_site;
/* The signature of every slot from the counts of the last mcov_base_counts into
 * dev_out[mcov_n_slots(ctx)] (device memory on ctx's GPU).
 * params->use_reference must be 0 (else MCOV_ERR_ARG).  MCOV_ERR_STATE without
 * counts for the current contig table.  Synchronises. */
int  mcov_allele_signature(mcov_ctx* ctx, const mcov_allele_params* params, uint8_t* dev_out);
/* The records of every pair over g regions [start, end) of contig tid
 * (0 <= start <= end; regions may overlap and reach past their contig, where
 * nothing is covered) into host_out[n_pairs * g], pair-major.  Synchronises. */
int  mcov_compare_run(mcov_ctx* ctx, int32_t n_sig, const uint8_t* const* sig, int32_t n_pairs, const int32_t* pairs,
                      int64_t g, const int32_t* tid, const int32_t* start, const int32_t* end, mcov_compare_stats* host_out);
/* Every site of every pair, in (pair, tid, pos) order, into a list kept on the
 * device; their number in *n_sites_out.  MCOV_ERR_NOMEM, with the byte count,
 * when the list does not fit.  Synchronises. */
int  mcov_compare_sites(mcov_ctx* ctx, int32_t n_sig, const uint8_t* const* sig, int32_t n_pairs, const int32_t* pairs,
                        int64_t* n_sites_out);
/* The sites [first, first + n) of the last mcov_compare_sites into
 * host_out[n].  MCOV_ERR_STATE without a list for the current contig table,
 * MCOV_ERR_ARG for a range outside it.  Synchronises. */
int  mcov_compare_sites_read(mcov_ctx* ctx, int64_t first, int64_t n, mcov_compare_site* host_out);

/* Linkage between nearby SNV sites from the reads and their mates
 * (csrc/linkage.cu; the rules are restated in oracle/linkage.py).
 *   sites   the SNV sites (kind bit 1) of the counts of the last
 *           mcov_base_counts under sites.min_coverage / min_freq / min_count,
 *           exactly those mcov_allele_sites lists with use_reference = 0.  At
 *           a site the major allele is the consensus and the minor allele the
 *           largest of the other three counts (ties to the first of A C G T).
 *   units   the records mcov_base_counts counts, grouped by the FNV-1a 64 of
 *           QNAME (~0 folded to ~0 - 1, the key of mcov_bam_gpu_names_seq):
 *           mates and supplementary pieces are one unit; equal keys are one
 *           unit, collisions included (two names collide with odds of about
 *           2^-64 a pair).  A record whose QNAME is '*' is a unit of its own.
 *   calls   a record gives a base at a site when the site's position is the
 *           reference position of one of its M / = / X pairs, the base is A,
 *           C, G or T and, with a non-zero quality_threshold, its quality is
 *           at least the threshold: the bases the counts counted, under the
 *           quality_threshold and mode the counts were made with.  A unit has
 *           call 0 (major) or 1 (minor) at a site when all its bases there are
 *           that allele; any disagreement, or a third allele, is no call.
 *   pairs   sites s < t of one contig with 0 < pos_t - pos_s <= max_distance;
 *           every unit with calls at both adds 1 to n[call_s][call_t].  A pair
 *           is listed when n_AB + n_Ab + n_aB + n_ab >= min_reads, in (tid,
 *           pos_a, pos_b) order (upper case: the major allele).
 * path NULL reads the records of the last device decode (BAM or SAM); a path
 * reads the BAM again through the streamed decoder (a second decode of the
 * file), with chunk_bytes as in mcov_bam_gpu_stream_depth.  The counts must be
 * those of the same records.  MCOV_ERR_ARG for bad parameters
 * (sites.use_reference must be 0); MCOV_ERR_STATE without counts for the
 * current contig table, or without a decoded file when path is NULL;
 * MCOV_ERR_NOMEM, before the
 * allocation, when a buffer does not fit the free device memory (the message
 * holds both byte counts); MCOV_ERR_IO as mcov_base_counts reports it.  The
 * depth store, its caches, the counts, the reference store and the allele and
 * compare site lists are never written; after an error the context is
 * usable.  Synchronises. */
typedef struct mcov_linkage_params {
  mcov_allele_params sites;      /* the SNV rules; sites.use_reference must be 0 */
  int32_t  max_distance;         /* 1 .. 100000 */
  uint32_t min_reads;            /* >= 1 */
} mcov_linkage_params;
/* One listed pair: the sites' 0-based positions, their alleles as 'A' 'C' 'G'
 * 'T' and the four haplotype counts.  32 bytes. */
typedef struct mcov_linkage_pair {
  int32_t  tid, pos_a, pos_b;
  uint8_t  major_a, minor_a, major_b, minor_b;
  uint32_t n_AB, n_Ab, n_aB, n_ab;
} mcov_linkage_pair;
/* SNV sites; (record, site) bases; units with at least one such base;
 * candidate pairs (site pairs within max_distance). */
typedef struct mcov_linkage_info { int64_t n_sites, n_observations, n_units, n_candidates; } mcov_linkage_info;
/* The pairs, into a list kept on the device; their number in *n_pairs_out,
 * the totals above in *info (may be NULL). */
int  mcov_linkage(mcov_ctx* ctx, const char* path, int64_t chunk_bytes, const mcov_linkage_params* params,
                  int64_t* n_pairs_out, mcov_linkage_info* info);
/* The pairs [first, first + n) of the last mcov_linkage into host_out[n].
 * MCOV_ERR_STATE without a list for the current contig table, MCOV_ERR_ARG for
 * a range outside it.  Synchronises. */
int  mcov_linkage_read(mcov_ctx* ctx, int64_t first, int64_t n, mcov_linkage_pair* host_out);

/* Genes profiled codon by codon from the counts of the last mcov_base_counts
 * and the reference (csrc/genes.cu; the rules are restated in oracle/genes.py).
 *   gene     (tid, start, end, strand +1 / -1, phase 0-2), 0-based half-open,
 *            0 <= start < end <= the contig's length.  Its codons are read
 *            from its 5' end after phase bases (from start on +, back from end
 *            on -): K = (end - start - phase) / 3 of them (0 if negative), a
 *            trailing 1-2 bases belong to none; on - the bases are
 *            complemented.  Codon index 0 is the 5'-most codon.
 *   called   a codon whose three positions are covered (the allele rules
 *            above) and whose three reference bases are known.  Everything
 *            below counts over called codons only.
 *   sites3   n3 + s3 = 9 a called codon: of its 3 positions x 3 other bases,
 *            the changes that alter the amino acid (n3) or not (s3) under the
 *            standard code, '*' counted as an amino acid (Nei-Gojobori in
 *            thirds).
 *   SNV      a position where two or more alleles are present; major = the
 *            consensus, minor = the largest of the other three counts (ties
 *            to the first of A C G T).  S when the codon with the major and
 *            the codon with the minor at this position (reference bases at
 *            the other two) translate alike, else N; M for every SNV position
 *            of a codon that holds two or more.
 *   SUB      a position whose consensus differs from the reference: the
 *            reference codon against the codon with the consensus at this
 *            position, S or N; M for a codon with two or more.
 * The gene call takes the allele parameters with use_reference = 1 (else
 * MCOV_ERR_ARG, as for bad parameters, a gene outside its contig, a strand
 * other than +1 / -1 or a phase outside 0-2).  MCOV_ERR_STATE without counts
 * for the current contig table or with a contig that has had no
 * mcov_set_reference.  The depth store, its caches, the counts, the reference
 * store and the allele, compare and linkage lists are never written; after an
 * error the context is usable. */
/* One gene: length = end - start, codons = K, codons_called, the expected
 * sites in thirds (n_sites3 + s_sites3 = 9 codons_called), SNV and SUB
 * positions by type.  96 bytes. */
typedef struct mcov_gene_stats {
  int64_t length, codons, codons_called, n_sites3, s_sites3;
  int64_t snv_n, snv_s, snv_m, sub_n, sub_s, sub_m, pad;
} mcov_gene_stats;
/* One (gene, position) with kind SNV or SUB in a called codon: the gene's
 * index, the contig and 0-based position, the codon index and the position in
 * it (0-2 from the 5' end), the reference codon as three letters in gene
 * orientation, the major (consensus) and minor allele in genomic orientation
 * as allele_sites gives them, the amino acids of the reference codon and of
 * the codon with the major / minor allele here, kind bits (1 SNV, 2 SUB) and
 * the SNV and SUB types 'N' 'S' 'M'.  minor, aa_minor and snv_type are 0 off
 * SNV positions, sub_type 0 off SUB positions.  32 bytes. */
typedef struct mcov_gene_site {
  int64_t  gene;
  int32_t  tid, pos, codon;
  uint8_t  codon_pos, ref_codon[3], major, minor, aa_ref, aa_major, aa_minor, kind, snv_type, sub_type;
} mcov_gene_site;
/* The records of g genes into host_out[g].  With n_sites_out, every site of
 * every gene, in (gene, pos) order (pos ascending on both strands; a position
 * in two genes is listed once for each), into a list kept on the device, and
 * their number in *n_sites_out; NULL skips the list.  MCOV_ERR_NOMEM, with the
 * byte count, when the list does not fit (test hook MCOV_GENE_FREE_BYTES).
 * Synchronises. */
int  mcov_gene_run(mcov_ctx* ctx, int64_t g, const int32_t* tid, const int32_t* start, const int32_t* end,
                   const int32_t* strand, const int32_t* phase, const mcov_allele_params* params,
                   mcov_gene_stats* host_out, int64_t* n_sites_out);
/* The sites [first, first + n) of the last mcov_gene_run with a list into
 * host_out[n].  MCOV_ERR_STATE without a list for the current contig table,
 * MCOV_ERR_ARG for a range outside it.  Synchronises. */
int  mcov_gene_sites_read(mcov_ctx* ctx, int64_t first, int64_t n, mcov_gene_site* host_out);

/* Test hooks: the device inflate / CRC-32 code (csrc/inflate.cuh) compiled for the host, so that the CPU
 * suite can check it against zlib.  mcov_inflate_host returns 0 or a positive decoder status. */
int  mcov_inflate_host(const uint8_t* src, uint32_t clen, uint8_t* dst, uint32_t ulen);
int  mcov_inflate_host_win(const uint8_t* src, uint32_t clen, uint8_t* dst, uint32_t ulen, uint32_t window);   /* with the circular output window the GPU keeps in shared memory */
uint32_t mcov_crc32_host(const uint8_t* p, uint32_t n);
uint32_t mcov_crc32_sliced_host(const uint8_t* p, uint32_t n, int nlanes);   /* the warp's lane-sliced CRC, folded on the host */

/* n_cigar of reads [i0, i0+n) -> out[n] (host or device memory per mem_kind;
 * device work is enqueued on `stream`, a cudaStream_t or NULL). */
int  mcov_synth_gen_ncigar(const struct mcov_synth_params* P, int64_t i0, int64_t n,
                       uint32_t* out, int mem_kind, void* stream);
/* Fill the SoA of reads [i0, i0+n).  read_start[n_contigs+1] / contig_len are
 * GLOBAL tables in the same memory kind as the outputs; tid_out = contig -
 * tid_base.  cig_off[n+1] are offsets into cig.  reflen_out may be NULL. */
int  mcov_synth_gen_reads(const struct mcov_synth_params* P, int64_t i0, int64_t n,
                     const int64_t* read_start, const int32_t* contig_len, int32_t n_contigs,
                     int32_t tid_base, const uint32_t* cig_off,
                     int32_t* tid, int32_t* pos, uint16_t* flag, uint8_t* mapq, int32_t* isize,
                     uint32_t* cig, int64_t* reflen_out, int mem_kind, void* stream);

/* Same with 64-bit CIGAR offsets (a batch of 2^32 or more ops). */
int  mcov_synth_gen_reads_wide(const struct mcov_synth_params* P, int64_t i0, int64_t n,
                     const int64_t* read_start, const int32_t* contig_len, int32_t n_contigs,
                     int32_t tid_base, const uint64_t* cig_off,
                     int32_t* tid, int32_t* pos, uint16_t* flag, uint8_t* mapq, int32_t* isize,
                     uint32_t* cig, int64_t* reflen_out, int mem_kind, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* METACOV_B200_H */
