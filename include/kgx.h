/*
 * kgx.h -- C ABI of the B200-native kangaroo jump engine (libkgx.so).
 *
 * This is the drop-in boundary for ONE path of JeanLucPons/Kangaroo: the GPU jump engine behind
 * `class GPUEngine` (reference GPU/GPUEngine.h:40-84, GPU/GPUEngine.cu).  The reference's interface is a C++
 * class taking host `Int` objects; the portable part of it is restated here as plain pointers and sizes so
 * that the C++ shim (kangaroo_b200/csrc/GPUEngine_b200.cu -> class GPUEngine, unchanged header), the
 * ctypes tests, bench.py and the NCCL rank driver all bind the same entry points.
 *
 * Conventions
 *   - field elements: 4 x uint64_t little-endian limbs (reference Int::bits64[0..3]);
 *   - distances: 2 x uint64_t, ALREADY biased by the wild offset for odd kIdx (the shim / Python host side
 *     adds and removes `wildOffset` exactly like GPUEngine.cu:407-411, 477, 526, 672);
 *   - kangaroo arrays are in kIdx order, n = groups * threads_per_group * KGX_GPU_GRP_SIZE entries
 *     (GPUEngine.cu:390-418); herd type = kIdx & 1;
 *   - every call returns 0 on success, a negative value on error with text in kgx_last_error();
 *     nothing throws, nothing falls back to the CPU: without a CUDA device kgx_create() fails.
 */
#ifndef KGX_H
#define KGX_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define KGX_NB_JUMP       32   /* Constants.h:29  */
#define KGX_GPU_GRP_SIZE  128  /* Constants.h:32  */
#define KGX_NB_RUN        64   /* Constants.h:35: jumps per kangaroo per launch */
#define KGX_ITEM_SIZE     56   /* GPUEngine.h:31: DP record {x[32], d[16], kIdx[8]} */

typedef struct kgx_engine kgx_engine;

/* DP record exactly as the reference kernel writes it (GPUMath.h:173-188, GPUEngine.cu:653-671). */
typedef struct {
  uint64_t x[4];
  uint64_t d[2];     /* biased 128-bit distance */
  uint64_t kidx;
} kgx_item;

/* --- static helpers (GPUEngine::GetGridSize / PrintCudaInfo, GPUEngine.cu:275-375) --- */
int  kgx_device_count(void);
/* Fills non-positive *x / *y with defaults: x = 2*SMs, y = 128 (GPUEngine.cu:301-303 on an unknown SM). */
int  kgx_grid_default(int dev, int* x, int* y);
/* "name|SMs|cc_major|cc_minor|totalMemMB" into buf */
int  kgx_device_info(int dev, char* buf, int buflen);

/* --- life cycle (GPUEngine ctor/dtor, GPUEngine.cu:144-263) --- */
kgx_engine* kgx_create(int dev, int groups, int threads_per_group, uint32_t max_found);
/* Same, with the jump kernel chosen by the caller instead of by herd size: KGX_KERNEL_STREAM = per-thread groups
 * streamed through HBM (the benchmarked kernel), KGX_KERNEL_RESIDENT = shared-memory tile kernel; stream_g = kangaroos
 * per thread of the stream kernel (even, 2..4096; 0 = adaptive).  Used by the parity tests to pin BOTH kernels to the
 * oracle and the reference fixtures on every grid. */
#define KGX_KERNEL_AUTO     0
#define KGX_KERNEL_STREAM   1
#define KGX_KERNEL_RESIDENT 2
#define KGX_KERNEL_TMEM     3   /* tile kernel with y and the prefix products in tensor memory (tcgen05.ld/st): 2048-kangaroo tiles */
kgx_engine* kgx_create_ex(int dev, int groups, int threads_per_group, uint32_t max_found, int kernel, int stream_g);
/* 1 = stream kernel, 2 = resident kernel, 3 = TMEM tile kernel (what kgx_create / kgx_create_ex resolved to) */
int         kgx_kernel_kind(kgx_engine* e);
void        kgx_destroy(kgx_engine* e);
const char* kgx_last_error(kgx_engine* e);      /* e may be NULL: error of the last failed kgx_create */
uint64_t    kgx_num_kangaroos(kgx_engine* e);   /* groups * threads_per_group * 128 */
uint64_t    kgx_memory_bytes(kgx_engine* e);    /* device bytes held (GPUEngine::GetMemory) */

/* --- USE_SYMMETRY engine mode (reference: compile-time switch Constants.h:25).  mode:
 *       0                    off
 *       KGX_SYM_LASTJUMP (1) the reference's DEVICE rule (GPUCompute.h:53-60, 91-94), which Kangaroo::Check replays on the CPU
 *                            (Check.cpp:534-556): jump = x mod 32, bumped when it repeats the previous jump of the kangaroo
 *       KGX_SYM_CLASS    (2) the rule of the reference's working symmetric path SolveKeyCPU (Kangaroo.cpp:381-384, 422-428):
 *                            jump = x mod 16 + 16 * symClass, symClass flipping at every class switch
 *     Both apply the equivalence-class switch after every jump (y > (p-1)/2 -> point negated, distance negated).  Distances
 *     crossing this ABI (upload, download, patch, create_herd, DP items) are then SIGNED 128-bit two's complement values and
 *     NO wild offset is applied (the reference's biased-unsigned device form cannot represent the sign changes: its
 *     ModNeg256Order writes 256 bits into a 128-bit slot, GPUMath.h:533-547).  The per-kangaroo rule state (lastJump /
 *     symClass) is reset by upload / patch / create_herd like GPUEngine.cu:413-416, 532-536.  Call before the herd is uploaded. --- */
#define KGX_SYM_LASTJUMP 1
#define KGX_SYM_CLASS    2
int kgx_set_symmetry(kgx_engine* e, int on);
int kgx_get_symmetry(kgx_engine* e);

/* --- GPUEngine::SetParams (GPUEngine.cu:559-590): jd 32x2, jpx/jpy 32x4 limbs --- */
int kgx_set_params(kgx_engine* e, uint64_t dp_mask, const uint64_t* jd, const uint64_t* jpx, const uint64_t* jpy);

/* --- GPUEngine::SetKangaroos / GetKangaroos / SetKangaroo (GPUEngine.cu:381-538) --- */
int kgx_upload(kgx_engine* e, const uint64_t* px, const uint64_t* py, const uint64_t* d);   /* n x 4, n x 4, n x 2 */
int kgx_download(kgx_engine* e, uint64_t* px, uint64_t* py, uint64_t* d);
int kgx_patch(kgx_engine* e, uint64_t kidx, const uint64_t px[4], const uint64_t py[4], const uint64_t d[2]);
/* Asynchronous GetKangaroos for checkpoints (SURVEY 8f/f3; Kangaroo.cpp:618-626, Backup.cpp:449-572): _begin snapshots the
 * herd in stream order (after the launch in flight) without blocking the caller or later launches; _read waits for that
 * snapshot only and copies it to the host arrays (kIdx order, distances still biased). */
int kgx_snapshot_begin(kgx_engine* e);
int kgx_snapshot_read(kgx_engine* e, uint64_t* px, uint64_t* py, uint64_t* d);

/* --- work-file walks (reference: Kangaroo::SaveWork with -ws, Backup.cpp:535-545; FetchWalks, Backup.cpp:211-231).
 *     One KGX_WALK_SIZE-byte record per kangaroo, record i = kIdx i (herd type = i & 1): {x[4], y[4], d[4]} as 64-bit
 *     little-endian limbs, d the UNBIASED distance mod n (wild: biased - wild_offset mod n; symmetric engines: the signed
 *     distance mod n, wild_offset ignored) -- what GetKangaroos returns.
 *   kgx_walks_begin  converts the herd into device staging in stream order (after the launch in flight) and returns
 *                    without blocking the caller or later launches;
 *   kgx_walks_read   waits for that conversion only and copies records [first, first + count) to `out` on a stream of
 *                    its own (pinned `out` makes it fast); may be called from another host thread than the launches;
 *   kgx_walks_end    ends the export (waits for the conversion if it is still running); the n x 96-byte staging
 *                    buffer is kept for the next export and freed by kgx_destroy;
 *   kgx_walks_load   writes `count` <= n records to kIdx [0, count) (distances re-biased and truncated to 128 bits like
 *                    SetKangaroos; padding slots follow; lastJump / symClass reset), leaving the other kangaroos as they
 *                    are.  verify != 0: recomputes d*G (tame) / key + d*G (wild; +-key on symmetric engines) for every
 *                    record, *n_bad = records that do not match, their first bad_cap indices (ascending) in bad_idx.
 *     Refused while a snapshot or a walk export is pending. --- */
#define KGX_WALK_SIZE 96
int kgx_walks_begin(kgx_engine* e, const uint64_t wild_offset[2]);
int kgx_walks_read(kgx_engine* e, void* out, uint64_t first, uint64_t count);
int kgx_walks_end(kgx_engine* e);
int kgx_walks_load(kgx_engine* e, const void* recs, uint64_t count, const uint64_t wild_offset[2],
                   const uint64_t keyx[4], const uint64_t keyy[4], int verify,
                   uint64_t* n_bad, uint64_t* bad_idx, uint32_t bad_cap);

/* --- herd creation on the device (SURVEY 8f/f2; replaces the CPU side of Kangaroo::CreateHerd, Kangaroo.cpp:670-738):
 *     kangaroo i starts at scalars[i]*G, plus `key` when (i + first_type) is odd (wild).  scalars: n x 4 limbs (mod the
 *     group order), d128: n x 2 limbs stored as the (biased) distances. --- */
int kgx_create_herd(kgx_engine* e, const uint64_t* scalars, const uint64_t* d128, const uint64_t keyx[4], const uint64_t keyy[4], int first_type);

/* --- GPUEngine::callKernel (GPUEngine.cu:540-557): zero the DP count, start NB_RUN jumps, asynchronous --- */
int kgx_launch_async(kgx_engine* e);
/* First half of GPUEngine::Launch (GPUEngine.cu:607-675): wait for the in-flight launch (sleeping unless
 * spin != 0), optionally start the NEXT launch before reading back (relaunch != 0; DP slabs are double
 * buffered so the copy overlaps the new kernel), then copy min(found, max_found, cap) records to `items`.
 * *n_items = records copied, *n_found = records the kernel wanted to write (may exceed max_found: lost). */
int kgx_collect(kgx_engine* e, kgx_item* items, uint32_t cap, uint32_t* n_items, uint32_t* n_found, int spin, int relaunch);
/* Blocks until every queued launch / copy finished. */
int kgx_sync(kgx_engine* e);

/* --- device-resident access for the multi-GPU DP gather and for bench.py (no host copies) --- */
/* Device pointer to the DP slab of the most recently COMPLETED launch: [u32 count][max_found x 56 B]. */
void*    kgx_dp_slab_device(kgx_engine* e);
uint32_t kgx_max_found(kgx_engine* e);
/* HashTable::Convert on the device (HashTable.cpp:75-100; SURVEY 8f/f1) for the most recently completed launch:
 * *out = device pointer to [u32 count][count x 40-byte DP {u32 kIdx; u32 h; u128 x; u128 tagged d}] (Kangaroo.h:94-101). */
int      kgx_convert_dps(kgx_engine* e, const uint64_t wild_offset[2], void** out);
/* Milliseconds the last completed launch spent on the device (CUDA events on the engine's stream). */
float    kgx_last_launch_ms(kgx_engine* e);
/* Jumps per launch override for tests (default KGX_NB_RUN). */
int      kgx_set_jumps_per_launch(kgx_engine* e, int n_run);
/* Number of kernels this engine has launched so far (jump + pack/unpack/patch), for bench.py's gpu_launches. */
uint64_t kgx_kernel_launches(kgx_engine* e);

/* Debug (KGX_PROF=1 in the environment at kgx_create): phase cycle counters summed over warp 0 of every CTA:
 * out = {serial section, modular inverse alone, parallel phase, tile-steps}; resets them. -1 when disabled. */
int      kgx_debug_prof(kgx_engine* e, uint64_t out[4]);

/* --- rank-0 distinguished-point table in device memory (SURVEY 8f row f1; kgx_dptable.cuh).  The decisions of the host
 *     table's kgi_add (include/kgx_ingest.h: HashTable::Add) on records that are already on the device, and exports in
 *     work-file order for kgi_fill_sorted.  Open addressing, linear probing, h-major home slots, 40 bytes per slot and at
 *     most KGX_DPT_LOAD entries per slot: about 57 bytes per entry of capacity.
 *   kgx_dpt_create        a table for `capacity` entries (at most kgx_dpt_max_capacity()) on device `dev`, collecting at
 *                         most max_events events per insert; NULL on failure, text in kgx_dpt_last_error(NULL)
 *   kgx_dpt_memory_bytes  device bytes such a table holds (export / load scratch included, insert scratch not: it grows
 *                         to 12 bytes per record of the largest batch)
 *   kgx_dpt_insert        stream-ordered on `stream` (a cudaStream_t; NULL = the legacy default stream): the 40-byte DP
 *                         records of `nranks` ranks, rank r's counts[r] records at recs + r * stride * 40 (one rank:
 *                         stride ignored, e.g. the records of kgx_convert_dps).  Records are decided in (rank, index)
 *                         order like consecutive kgi_add calls.  At most two inserts may await kgx_dpt_events.
 *   kgx_dpt_events        waits for the oldest pending insert and copies its events (KGX_DPT_EVENT_SIZE-byte kgi_event
 *                         records, any order) to ev[0..cap); *n_ev = events produced (the excess over cap is dropped, as
 *                         kgi_add), *entries = table entries after that insert.  0, -1 when a record had h >= 2^18
 *                         (skipped, like kgi_add), -2 when a probe ran off the table, -3 on a CUDA or usage error.
 *   kgx_dpt_count         entries after every insert queued so far (waits for them)
 *   kgx_dpt_export_begin  snapshot point: the export holds the inserts queued before this call (stream-ordered behind them on
 *                         `stream`); later inserts proceed and are not part of it
 *   kgx_dpt_export_read   from any host thread: entries of buckets [first_bucket, first_bucket + k), k <= max_buckets as
 *                         many as fit in entries_cap, sorted by (x[1], x[0]) inside each bucket, as 32-byte {x[2], d[2]}
 *                         entries; counts[0..k) = entries per bucket.  k = 0 once first_bucket reaches 2^18.
 *   kgx_dpt_export_end    ends the export
 *   kgx_dpt_load          bulk load of distinct entries in work-file order (h[n], entries32 = n x 32 bytes; resume);
 *                         synchronous, refused while inserts or an export are pending --- */
typedef struct kgx_dpt kgx_dpt;
#define KGX_DPT_EVENT_SIZE 48
#define KGX_DPT_LOAD       0.7
kgx_dpt*    kgx_dpt_create(int dev, uint64_t capacity, uint32_t max_events);
void        kgx_dpt_destroy(kgx_dpt* t);
const char* kgx_dpt_last_error(kgx_dpt* t);
uint64_t    kgx_dpt_memory_bytes(uint64_t capacity);
uint64_t    kgx_dpt_max_capacity(void);
uint64_t    kgx_dpt_capacity(kgx_dpt* t);
int         kgx_dpt_insert(kgx_dpt* t, const void* recs, uint32_t stride, const uint32_t* counts, uint32_t nranks, void* stream);
int         kgx_dpt_events(kgx_dpt* t, void* ev, uint32_t cap, uint32_t* n_ev, uint64_t* entries);
int         kgx_dpt_pending(kgx_dpt* t);
int         kgx_dpt_count(kgx_dpt* t, uint64_t* entries);
int         kgx_dpt_export_begin(kgx_dpt* t, void* stream);
int         kgx_dpt_export_read(kgx_dpt* t, uint32_t first_bucket, uint32_t max_buckets, void* entries, uint64_t entries_cap,
                                uint32_t* counts, uint32_t* n_buckets, uint64_t* n_entries);
int         kgx_dpt_export_end(kgx_dpt* t);
int         kgx_dpt_load(kgx_dpt* t, const uint32_t* h, const void* entries32, uint64_t n);

/* --- device-side unit-test / microbenchmark hooks (kgx_field.cuh, kgx_modinv.h) --- */
/* op: 0 = mul, 1 = sqr, 2 = sub, 3 = inv.  a, b, out: n x 4 limbs on the HOST. */
int kgx_test_field(int dev, int op, int n, const uint64_t* a, const uint64_t* b, uint64_t* out);
/* Raw device throughput probes: kind 0 = IMAD.WIDE.U32 issue rate (the multiplier roofline bench.py reports against),
 * 1 = ModMult chains, 2 = ModSqr chains, 3 = modular inverses.  *ms = device time, *ops = operations executed. */
int kgx_bench_raw(int dev, int kind, int iters, float* ms, double* ops);

#ifdef __cplusplus
}
#endif
#endif
