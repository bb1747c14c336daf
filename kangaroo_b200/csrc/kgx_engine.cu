// kgx_engine.cu -- host side of the B200 jump engine behind the C ABI of include/kgx.h.
//
// Replaces the host half of the reference's GPU/GPUEngine.cu (ctor/dtor :144-263, SetKangaroos/GetKangaroos/
// SetKangaroo :381-538, callKernel :540-557, SetParams :559-590, Launch :607-679) with a stream-ordered
// design: one non-blocking stream per engine, device-side pack/unpack kernels instead of per-block host
// transposes, double-buffered DP slabs so the readback of launch i overlaps launch i+1, CUDA-event timing of
// every launch.  No CPU fallback exists: every entry point fails when CUDA does.
#include <cuda_runtime.h>
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <unistd.h>
#include "../../include/kgx.h"
#include "kgx_kernel.cuh"
#include "kgx_herd.cuh"
#include "kgx_walks.cuh"
#include "kgx_dptable.cuh"

using namespace kgx;

static char g_create_err[256] = "";

struct kgx_engine {
  int dev = 0, groups = 0, tpg = 0, sms = 0;
  int T = 0, K = 0, cfg = 0, ctasPerSM = 0, smemBytes = 0;   // tile geometry (kgx_kernel.cuh Cfg<T,K>)
  u64 n = 0, nPadded = 0;
  u32 numTiles = 0, maxFound = 0;
  int nRun = KGX_NB_RUN;
  uint4* state = nullptr;
  uint4* pre = nullptr;      // streaming mode: prefix-product scratch
  bool streamMode = false;
  bool tmemMode = false;     // TMEM-backed tile kernel (jump_kernel_tmem<16>)
  int streamCtas = 2;
  bool symmetry = false;     // USE_SYMMETRY engine mode (kgx_set_symmetry): class switch + cycle rule, signed distances
  int symRule = 0;           // KGX_SYM_LASTJUMP / KGX_SYM_CLASS
  int pfDist = 2;            // KGX_STREAM_PF: L2 prefetch distance of the stream kernel in kangaroos (measured: 0 -> 14.04,
                             // 2 -> 14.44, 4 -> 14.40, 8 -> 14.24 GJump/s, profiles/r2c_sweep_prefetch.txt)
  uint8_t* aux = nullptr;    // symmetric mode: lastJump per slot
  bool warpInv = true;       // stream kernel: one warp-wide shuffle-butterfly inverse per pass (false: one per thread)
  u32* slab[2] = {nullptr, nullptr};   // DP slabs [count][maxFound*14]
  u32* slabPinned = nullptr;
  u32* dp40 = nullptr;       // [count][maxFound x 10 words]: converted records of the last completed launch
  u32* jtab = nullptr;
  u32* herdTab = nullptr;    // 256 x 16 words: 2^i * G (built on first kgx_create_herd)
  uint4 *stgX = nullptr, *stgY = nullptr, *stgD = nullptr;   // device staging (AoS, kIdx order)
  u64 dpMask = 0;
  bool haveParams = false, inflight = false;
  int cur = 0;                 // slab the in-flight (or last) launch writes
  int done = -1;               // slab of the most recently completed launch
  cudaStream_t stream = nullptr, copyStream = nullptr;
  cudaEvent_t evStart[2] = {nullptr, nullptr}, evStop[2] = {nullptr, nullptr};
  cudaEvent_t evSnap = nullptr;   // snapshot (checkpoint) staging complete
  bool snapPending = false;
  u64* stgW = nullptr;            // walk export staging: n x 96-byte work-file records (allocated by the first kgx_walks_begin)
  cudaStream_t walkStream = nullptr;   // D2H of exported walks: its own stream, so kgx_collect's copies never queue behind it
  cudaEvent_t evWalks = nullptr;  // walk export complete
  bool walksPending = false;
  float lastMs = 0.f;
  unsigned long long* prof = nullptr;   // KGX_PROF=1: phase cycle counters
  u64 launches = 0;
  size_t slabBytes = 0, stateBytes = 0;
  char err[256] = "";
};

#define CK(e, call)                                                                            \
  do {                                                                                         \
    cudaError_t _s = (call);                                                                   \
    if (_s != cudaSuccess) {                                                                   \
      snprintf((e)->err, sizeof((e)->err), "%s: %s", #call, cudaGetErrorString(_s));           \
      return -1;                                                                               \
    }                                                                                          \
  } while (0)

// Tile geometries compiled in.  The default was picked by the sweep recorded in profiles/ (KGX_CFG="T,K" overrides).
// kernSym: the symmetric-mode (USE_SYMMETRY) instantiation; only the default geometry carries one (others: NULL).
struct CfgEntry { int T, K, smem, ctas; void (*kern)(LaunchParams); void (*kernSym)(LaunchParams); };
#define KGX_CFG_ENTRY(T_, K_) { T_, K_, Cfg<T_, K_>::SMEM_BYTES, Cfg<T_, K_>::CTAS_PER_SM, jump_kernel<T_, K_, false>, nullptr }
#define KGX_CFG_ENTRY_SYM(T_, K_) { T_, K_, Cfg<T_, K_>::SMEM_BYTES, Cfg<T_, K_>::CTAS_PER_SM, jump_kernel<T_, K_, false>, jump_kernel<T_, K_, true> }
static const CfgEntry g_cfgs[] = {
  KGX_CFG_ENTRY_SYM(128, 7), KGX_CFG_ENTRY(128, 4), KGX_CFG_ENTRY(128, 5), KGX_CFG_ENTRY(64, 7), KGX_CFG_ENTRY(64, 5),
  KGX_CFG_ENTRY(64, 6), KGX_CFG_ENTRY(64, 4), KGX_CFG_ENTRY(96, 6), KGX_CFG_ENTRY(256, 3), KGX_CFG_ENTRY(32, 8), KGX_CFG_ENTRY(32, 12),
};
static const int g_ncfg = sizeof(g_cfgs) / sizeof(g_cfgs[0]);
#ifndef KGX_DEFAULT_CFG
#define KGX_DEFAULT_CFG 0
#endif
#ifndef KGX_DEFAULT_STREAM
#define KGX_DEFAULT_STREAM 1   // streaming kernel is the faster one on B200 (profiles/r1_sweep.txt); KGX_MODE=resident selects the tile kernel
#endif

extern "C" {

int kgx_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

int kgx_grid_default(int dev, int* x, int* y) {
  if (*x > 0 && *y > 0) return 0;
  int n = kgx_device_count();
  if (n == 0 || dev >= n) return -1;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) return -1;
  if (*x <= 0) *x = 2 * prop.multiProcessorCount;   // GPUEngine.cu:301
  if (*y <= 0) *y = 128;                            // GPUEngine.cu:303 (sm_100 is not in the reference's core table)
  return 0;
}

int kgx_device_info(int dev, char* buf, int buflen) {
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) return -1;
  snprintf(buf, buflen, "%s|%d|%d|%d|%.1f", prop.name, prop.multiProcessorCount, prop.major, prop.minor,
           (double)prop.totalGlobalMem / 1048576.0);
  return 0;
}

const char* kgx_last_error(kgx_engine* e) { return e ? e->err : g_create_err; }

void kgx_destroy(kgx_engine* e) {
  if (!e) return;
  cudaSetDevice(e->dev);
  if (e->stream) cudaStreamSynchronize(e->stream);
  cudaFree(e->dp40); cudaFree(e->herdTab); cudaFree(e->state); cudaFree(e->pre); cudaFree(e->slab[0]); cudaFree(e->slab[1]); cudaFree(e->jtab);
  cudaFree(e->stgX); cudaFree(e->stgY); cudaFree(e->stgD); cudaFree(e->aux);
  if (e->slabPinned) cudaFreeHost(e->slabPinned);
  for (int i = 0; i < 2; i++) { if (e->evStart[i]) cudaEventDestroy(e->evStart[i]); if (e->evStop[i]) cudaEventDestroy(e->evStop[i]); }
  if (e->evSnap) cudaEventDestroy(e->evSnap);
  cudaFree(e->stgW);
  if (e->evWalks) cudaEventDestroy(e->evWalks);
  if (e->walkStream) cudaStreamDestroy(e->walkStream);
  if (e->stream) cudaStreamDestroy(e->stream);
  if (e->copyStream) cudaStreamDestroy(e->copyStream);
  delete e;
}

kgx_engine* kgx_create(int dev, int groups, int threads_per_group, uint32_t max_found) {
  return kgx_create_ex(dev, groups, threads_per_group, max_found, KGX_KERNEL_AUTO, 0);
}

// kernel: KGX_KERNEL_AUTO / _STREAM / _RESIDENT; stream_g: kangaroos per thread of the stream kernel (0 = adaptive).
// The environment (KGX_MODE, KGX_STREAM_G, KGX_CFG) only fills in what the arguments leave on "auto".
kgx_engine* kgx_create_ex(int dev, int groups, int threads_per_group, uint32_t max_found, int kernel, int stream_g) {
  kgx_engine* e = new kgx_engine();
  auto fail = [&](const char* what, cudaError_t s) -> kgx_engine* {
    snprintf(g_create_err, sizeof g_create_err, "kgx_create: %s: %s", what, cudaGetErrorString(s));
    cudaGetLastError();   // do not leave a sticky error behind for the next engine of this process
    kgx_destroy(e);
    return nullptr;
  };
  if (groups <= 0 || threads_per_group <= 0 || max_found == 0) {
    snprintf(g_create_err, sizeof g_create_err, "kgx_create: bad arguments");
    delete e; return nullptr;
  }
  int cnt = 0;
  cudaError_t s = cudaGetDeviceCount(&cnt);
  if (s != cudaSuccess || cnt == 0) {
    snprintf(g_create_err, sizeof g_create_err, "kgx_create: no CUDA device (%s)", cudaGetErrorString(s));
    cudaGetLastError(); delete e; return nullptr;
  }
  if ((s = cudaSetDevice(dev)) != cudaSuccess) return fail("cudaSetDevice", s);
  cudaDeviceProp prop;
  if ((s = cudaGetDeviceProperties(&prop, dev)) != cudaSuccess) return fail("cudaGetDeviceProperties", s);
  e->dev = dev; e->groups = groups; e->tpg = threads_per_group; e->sms = prop.multiProcessorCount;
  e->n = (u64)groups * (u64)threads_per_group * KGX_GPU_GRP_SIZE;
  e->cfg = KGX_DEFAULT_CFG;
  if (const char* env = getenv("KGX_CFG")) {
    int t = 0, k = 0, found = -1;
    if (sscanf(env, "%d,%d", &t, &k) == 2)
      for (int i = 0; i < g_ncfg; i++) if (g_cfgs[i].T == t && g_cfgs[i].K == k) found = i;
    if (found < 0) { snprintf(g_create_err, sizeof g_create_err, "kgx_create: KGX_CFG=%s is not a compiled tile geometry", env); delete e; return nullptr; }
    e->cfg = found;
  }
  e->T = g_cfgs[e->cfg].T; e->K = g_cfgs[e->cfg].K; e->smemBytes = g_cfgs[e->cfg].smem; e->ctasPerSM = g_cfgs[e->cfg].ctas;
  {
    const char* mode = getenv("KGX_MODE");
    if (kernel == KGX_KERNEL_STREAM) mode = "stream";
    else if (kernel == KGX_KERNEL_RESIDENT) mode = "resident";
    else if (kernel == KGX_KERNEL_TMEM) mode = "tmem";
    else if (kernel != KGX_KERNEL_AUTO) { snprintf(g_create_err, sizeof g_create_err, "kgx_create_ex: bad kernel selector %d", kernel); delete e; return nullptr; }
    // default: the streaming kernel for herds of 400 k kangaroos and more (it wants many kangaroos per thread on every
    // SM to amortise the per-thread inverse), the shared-memory tile kernel below that (its inverse is shared by a whole
    // tile, so it keeps ~6.9 GJump/s down to ~270 k kangaroos) -- measured crossover, profiles/r1g_sweep.txt
    e->streamMode = mode ? (strcmp(mode, "stream") == 0) : (KGX_DEFAULT_STREAM != 0 && e->n >= 400000ull);
    if (mode && strcmp(mode, "stream") && strcmp(mode, "resident") && strcmp(mode, "tmem")) {
      snprintf(g_create_err, sizeof g_create_err, "kgx_create: KGX_MODE must be stream, resident or tmem"); delete e; return nullptr;
    }
    if (mode && !strcmp(mode, "tmem")) {
      e->tmemMode = true;
      e->T = CfgTm<16>::T; e->K = CfgTm<16>::K; e->smemBytes = CfgTm<16>::SMEM_BYTES; e->ctasPerSM = 2;
    }
    if (e->streamMode) {
      // kangaroos per thread: 128 (the reference's GPU_GRP_SIZE) when the herd fills two CTAs per SM with it; smaller
      // herds get a smaller group so that the grid still covers the chip (one wave of 2 CTAs/SM), at the price of more
      // inversions per jump.  KGX_STREAM_G overrides.
      int ctas = 2;
      if (const char* sc = getenv("KGX_STREAM_CTAS")) ctas = atoi(sc);
      if (ctas != 2 && ctas != 3) { snprintf(g_create_err, sizeof g_create_err, "kgx_create: KGX_STREAM_CTAS must be 2 or 3"); delete e; return nullptr; }
      bool invChosen = false;
      if (const char* si = getenv("KGX_STREAM_INV")) {
        invChosen = true;
        if (!strcmp(si, "thread")) e->warpInv = false;
        else if (strcmp(si, "warp")) { snprintf(g_create_err, sizeof g_create_err, "kgx_create: KGX_STREAM_INV must be warp or thread"); delete e; return nullptr; }
      }
      const u64 slots = (u64)ctas * prop.multiProcessorCount * 128;       // threads of one wave
      long long g = (long long)((e->n + slots - 1) / slots);               // round UP: never more tiles than one wave
      g = (g + 1) & ~1LL;
      if (g > 128) g = 128;
      if (g < 2) g = 2;
      if (stream_g > 0) g = stream_g;
      else if (const char* sg = getenv("KGX_STREAM_G")) g = atoi(sg);
      if (g < 2 || g > 4096 || (g & 1)) { snprintf(g_create_err, sizeof g_create_err, "kgx_create: stream group size (KGX_STREAM_G) must be an even number in [2, 4096]"); delete e; return nullptr; }
      // group inverse: the warp-wide shuffle butterfly (one uniform inverse per warp and pass) for long groups, one inverse per
      // thread for short ones, where the butterfly's 10 extra multiplications per lane weigh more than lane divergence inside
      // the variable-time inverse -- measured equal at G = 128 (14.16 vs 14.23 GJump/s), 3 % apart at G = 28 (profiles/r2b_sweep.txt)
      if (!invChosen) e->warpInv = g >= 64;
      if (const char* pf = getenv("KGX_STREAM_PF")) e->pfDist = atoi(pf);
      e->streamCtas = ctas;
      e->T = 128; e->K = (int)g; e->smemBytes = 0; e->ctasPerSM = ctas;
    }
  }
  const u64 TILE = (u64)e->T * e->K;
  e->numTiles = (u32)((e->n + TILE - 1) / TILE);
  e->nPadded = (u64)e->numTiles * TILE;
  e->maxFound = max_found;
  e->stateBytes = (size_t)e->nPadded * CHUNKS * 16;
  e->slabBytes = (size_t)max_found * KGX_ITEM_SIZE + 4;
  if ((s = cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking)) != cudaSuccess) return fail("cudaStreamCreate", s);
  if ((s = cudaStreamCreateWithFlags(&e->copyStream, cudaStreamNonBlocking)) != cudaSuccess) return fail("cudaStreamCreate", s);
  for (int i = 0; i < 2; i++) {
    if ((s = cudaEventCreate(&e->evStart[i])) != cudaSuccess) return fail("cudaEventCreate", s);
    if ((s = cudaEventCreateWithFlags(&e->evStop[i], cudaEventBlockingSync)) != cudaSuccess) return fail("cudaEventCreate", s);
  }
  if ((s = cudaMalloc(&e->state, e->stateBytes)) != cudaSuccess) return fail("cudaMalloc(state)", s);
  if (e->streamMode && (s = cudaMalloc(&e->pre, (size_t)e->nPadded * 32)) != cudaSuccess) return fail("cudaMalloc(pre)", s);
  for (int i = 0; i < 2; i++) {
    if ((s = cudaMalloc(&e->slab[i], e->slabBytes)) != cudaSuccess) return fail("cudaMalloc(slab)", s);
    if ((s = cudaMemsetAsync(e->slab[i], 0, 4, e->stream)) != cudaSuccess) return fail("cudaMemset(slab)", s);  // Check.cpp:526 collects before any launch
  }
  if ((s = cudaMalloc(&e->jtab, JT_WORDS * 4)) != cudaSuccess) return fail("cudaMalloc(jtab)", s);
  if (getenv("KGX_PROF")) {
    if ((s = cudaMalloc(&e->prof, 64)) != cudaSuccess) return fail("cudaMalloc(prof)", s);
    cudaMemset(e->prof, 0, 64);
  }
  if ((s = cudaHostAlloc(&e->slabPinned, e->slabBytes, cudaHostAllocDefault)) != cudaSuccess) return fail("cudaHostAlloc", s);
  if (e->tmemMode) {
    if ((s = cudaFuncSetAttribute(jump_kernel_tmem<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, e->smemBytes)) != cudaSuccess)
      return fail("cudaFuncSetAttribute(smem, tmem kernel)", s);
  } else if (!e->streamMode &&
      (s = cudaFuncSetAttribute(g_cfgs[e->cfg].kern, cudaFuncAttributeMaxDynamicSharedMemorySize, e->smemBytes)) != cudaSuccess)
    return fail("cudaFuncSetAttribute(smem)", s);
  if ((s = cudaStreamSynchronize(e->stream)) != cudaSuccess) return fail("sync", s);
  return e;
}

uint64_t kgx_num_kangaroos(kgx_engine* e) { return e->n; }
int kgx_kernel_kind(kgx_engine* e) { return e->streamMode ? KGX_KERNEL_STREAM : (e->tmemMode ? KGX_KERNEL_TMEM : KGX_KERNEL_RESIDENT); }
uint64_t kgx_memory_bytes(kgx_engine* e) { return e->stateBytes + (e->pre ? e->nPadded * 32 : 0) + 2 * e->slabBytes + JT_WORDS * 4; }
uint32_t kgx_max_found(kgx_engine* e) { return e->maxFound; }
float kgx_last_launch_ms(kgx_engine* e) { return e->lastMs; }
uint64_t kgx_kernel_launches(kgx_engine* e) { return e->launches; }
// debug: read and reset the phase counters (KGX_PROF=1): serial, modinv, parallel cycles, tile-steps
int kgx_debug_prof(kgx_engine* e, uint64_t out[4]) {
  if (!e->prof) return -1;
  cudaStreamSynchronize(e->stream);
  cudaMemcpy(out, e->prof, 32, cudaMemcpyDeviceToHost);
  cudaMemset(e->prof, 0, 64);
  return 0;
}
int kgx_set_jumps_per_launch(kgx_engine* e, int n_run) {
  if (n_run <= 0) { snprintf(e->err, sizeof e->err, "kgx_set_jumps_per_launch: n_run must be > 0"); return -1; }
  e->nRun = n_run; return 0;
}

// USE_SYMMETRY engine mode (SURVEY 8f/f4).  Must be chosen before the herd is uploaded: it allocates the lastJump bytes,
// switches the jump kernels to their symmetric instantiation and makes every distance crossing the ABI a SIGNED 128-bit
// two's complement value (no wild-offset bias).
int kgx_set_symmetry(kgx_engine* e, int on) {
  CK(e, cudaSetDevice(e->dev));
  if (e->inflight) { snprintf(e->err, sizeof e->err, "kgx_set_symmetry: a launch is in flight"); return -1; }
  if (on && e->tmemMode) { snprintf(e->err, sizeof e->err, "kgx_set_symmetry: the TMEM tile kernel has no symmetric instantiation"); return -1; }
  if (on && !e->streamMode && !g_cfgs[e->cfg].kernSym) {
    snprintf(e->err, sizeof e->err, "kgx_set_symmetry: tile geometry %d,%d has no symmetric instantiation", e->T, e->K); return -1;
  }
  if (on && e->streamMode && e->streamCtas != 2) {
    snprintf(e->err, sizeof e->err, "kgx_set_symmetry: the symmetric stream kernel is the 2-CTA variant only"); return -1;
  }
  if (on != 0 && on != KGX_SYM_LASTJUMP && on != KGX_SYM_CLASS) { snprintf(e->err, sizeof e->err, "kgx_set_symmetry: mode must be 0, 1 (lastJump rule) or 2 (symClass rule)"); return -1; }
  if (on && !e->aux) CK(e, cudaMalloc(&e->aux, e->nPadded));
  if (on) CK(e, cudaMemsetAsync(e->aux, on == KGX_SYM_CLASS ? 0 : 32, e->nPadded, e->stream));
  e->symRule = on;
  if (on && !e->streamMode)
    CK(e, cudaFuncSetAttribute(g_cfgs[e->cfg].kernSym, cudaFuncAttributeMaxDynamicSharedMemorySize, e->smemBytes));
  e->symmetry = on != 0;
  return 0;
}
int kgx_get_symmetry(kgx_engine* e) { return e->symmetry ? e->symRule : 0; }

// word w (0..7 jpx, 8..15 jpy, 16..19 jd) of jump j in the device table: uint4 jt[w / 4][j], component w % 4 (kgx_kernel.cuh)
static inline int jt_word(int w, int j) { return ((w >> 2) * 32 + j) * 4 + (w & 3); }

int kgx_set_params(kgx_engine* e, uint64_t dp_mask, const uint64_t* jd, const uint64_t* jpx, const uint64_t* jpy) {
  CK(e, cudaSetDevice(e->dev));
  u32 tab[JT_WORDS];
  for (int j = 0; j < 32; j++) {
    for (int w = 0; w < 8; w++) {
      tab[jt_word(w, j)] = (u32)(jpx[4 * j + w / 2] >> (32 * (w & 1)));
      tab[jt_word(8 + w, j)] = (u32)(jpy[4 * j + w / 2] >> (32 * (w & 1)));
    }
    for (int w = 0; w < 4; w++) tab[jt_word(16 + w, j)] = (u32)(jd[2 * j + w / 2] >> (32 * (w & 1)));
  }
  CK(e, cudaStreamSynchronize(e->stream));   // a running kernel may still read the old table
  CK(e, cudaMemcpy(e->jtab, tab, sizeof tab, cudaMemcpyHostToDevice));
  e->dpMask = dp_mask;
  e->haveParams = true;
  return 0;
}

static int ensure_staging(kgx_engine* e) {
  if (e->stgX) return 0;
  CK(e, cudaMalloc(&e->stgX, e->n * 32));
  CK(e, cudaMalloc(&e->stgY, e->n * 32));
  CK(e, cudaMalloc(&e->stgD, e->n * 16));
  return 0;
}
static void free_staging(kgx_engine* e) {
  cudaFree(e->stgX); cudaFree(e->stgY); cudaFree(e->stgD);
  e->stgX = e->stgY = e->stgD = nullptr;
}

int kgx_upload(kgx_engine* e, const uint64_t* px, const uint64_t* py, const uint64_t* d) {
  CK(e, cudaSetDevice(e->dev));
  if (e->snapPending) { snprintf(e->err, sizeof e->err, "kgx_upload: snapshot pending (read it first)"); return -1; }
  if (ensure_staging(e)) return -1;
  CK(e, cudaMemcpyAsync(e->stgX, px, e->n * 32, cudaMemcpyHostToDevice, e->stream));
  CK(e, cudaMemcpyAsync(e->stgY, py, e->n * 32, cudaMemcpyHostToDevice, e->stream));
  CK(e, cudaMemcpyAsync(e->stgD, d, e->n * 16, cudaMemcpyHostToDevice, e->stream));
  u32 blocks = (u32)((e->nPadded + 255) / 256);
  pack_kernel<<<blocks, 256, 0, e->stream>>>(e->state, e->stgX, e->stgY, e->stgD, e->n, e->nPadded, e->T, e->K, e->aux, e->symRule == KGX_SYM_CLASS ? 0 : 32);
  e->launches++;
  CK(e, cudaGetLastError());
  CK(e, cudaStreamSynchronize(e->stream));
  free_staging(e);
  return 0;
}

int kgx_download(kgx_engine* e, uint64_t* px, uint64_t* py, uint64_t* d) {
  CK(e, cudaSetDevice(e->dev));
  if (e->snapPending) { snprintf(e->err, sizeof e->err, "kgx_download: snapshot pending (read it first)"); return -1; }
  if (ensure_staging(e)) return -1;
  u32 blocks = (u32)((e->n + 255) / 256);
  unpack_kernel<<<blocks, 256, 0, e->stream>>>(e->state, e->stgX, e->stgY, e->stgD, e->n, e->T, e->K);   // stream order: after the in-flight launch
  e->launches++;
  CK(e, cudaGetLastError());
  CK(e, cudaMemcpyAsync(px, e->stgX, e->n * 32, cudaMemcpyDeviceToHost, e->stream));
  CK(e, cudaMemcpyAsync(py, e->stgY, e->n * 32, cudaMemcpyDeviceToHost, e->stream));
  CK(e, cudaMemcpyAsync(d, e->stgD, e->n * 16, cudaMemcpyDeviceToHost, e->stream));
  CK(e, cudaStreamSynchronize(e->stream));
  free_staging(e);
  return 0;
}

// ---- asynchronous checkpoint (SURVEY 8f/f3; reference: SolveKeyGPU parks on saveMutex while GetKangaroos copies the
// whole herd with blocking memcpys, Kangaroo.cpp:618-626).  kgx_snapshot_begin() enqueues, in stream order (i.e. after the
// launch in flight), a device-side copy of the herd into kIdx-ordered staging and returns at once; later launches run
// on; kgx_snapshot_read() waits for that copy only and moves it to the host on the copy stream.
int kgx_snapshot_begin(kgx_engine* e) {
  CK(e, cudaSetDevice(e->dev));
  if (e->snapPending) { snprintf(e->err, sizeof e->err, "kgx_snapshot_begin: previous snapshot not read"); return -1; }
  if (ensure_staging(e)) return -1;
  if (!e->evSnap) CK(e, cudaEventCreateWithFlags(&e->evSnap, cudaEventBlockingSync | cudaEventDisableTiming));
  u32 blocks = (u32)((e->n + 255) / 256);
  unpack_kernel<<<blocks, 256, 0, e->stream>>>(e->state, e->stgX, e->stgY, e->stgD, e->n, e->T, e->K);
  e->launches++;
  CK(e, cudaGetLastError());
  CK(e, cudaEventRecord(e->evSnap, e->stream));
  e->snapPending = true;
  return 0;
}

int kgx_snapshot_read(kgx_engine* e, uint64_t* px, uint64_t* py, uint64_t* d) {
  CK(e, cudaSetDevice(e->dev));
  if (!e->snapPending) { snprintf(e->err, sizeof e->err, "kgx_snapshot_read: no snapshot pending"); return -1; }
  CK(e, cudaStreamWaitEvent(e->copyStream, e->evSnap, 0));
  CK(e, cudaMemcpyAsync(px, e->stgX, e->n * 32, cudaMemcpyDeviceToHost, e->copyStream));
  CK(e, cudaMemcpyAsync(py, e->stgY, e->n * 32, cudaMemcpyDeviceToHost, e->copyStream));
  CK(e, cudaMemcpyAsync(d, e->stgD, e->n * 16, cudaMemcpyDeviceToHost, e->copyStream));
  CK(e, cudaStreamSynchronize(e->copyStream));
  e->snapPending = false;
  free_staging(e);
  return 0;
}

// ---- work-file walks (kgx_walks.cuh; reference: SaveWork -ws, Backup.cpp:535-545, FetchWalks :211-231) ----
// kgx_walks_begin converts the herd into 96-byte records in device staging, enqueued in stream order (after the launch
// in flight) like kgx_snapshot_begin, and returns at once.  kgx_walks_read copies a range of them out on the walk stream
// and waits for that copy only, so a writer thread can drain the export while the caller keeps launching.
int kgx_walks_begin(kgx_engine* e, const uint64_t wild_offset[2]) {
  CK(e, cudaSetDevice(e->dev));
  if (e->walksPending) { snprintf(e->err, sizeof e->err, "kgx_walks_begin: previous walk export not ended"); return -1; }
  if (e->snapPending) { snprintf(e->err, sizeof e->err, "kgx_walks_begin: snapshot pending (read it first)"); return -1; }
  if (!e->stgW) CK(e, cudaMalloc(&e->stgW, (size_t)e->n * KGX_WALK_SIZE));
  if (!e->walkStream) CK(e, cudaStreamCreateWithFlags(&e->walkStream, cudaStreamNonBlocking));
  if (!e->evWalks) CK(e, cudaEventCreateWithFlags(&e->evWalks, cudaEventBlockingSync | cudaEventDisableTiming));
  walks_export_kernel<<<(u32)((e->n + 255) / 256), 256, 0, e->stream>>>(e->state, e->stgW, e->n, e->T, e->K,
                                                                         wild_offset[0], wild_offset[1], e->symmetry ? 1 : 0);
  e->launches++;
  CK(e, cudaGetLastError());
  CK(e, cudaEventRecord(e->evWalks, e->stream));
  e->walksPending = true;
  return 0;
}

int kgx_walks_read(kgx_engine* e, void* out, uint64_t first, uint64_t count) {
  CK(e, cudaSetDevice(e->dev));
  if (!e->walksPending) { snprintf(e->err, sizeof e->err, "kgx_walks_read: no walk export pending"); return -1; }
  if (first > e->n || count > e->n - first) { snprintf(e->err, sizeof e->err, "kgx_walks_read: range past the herd"); return -1; }
  if (count == 0) return 0;
  CK(e, cudaStreamWaitEvent(e->walkStream, e->evWalks, 0));
  CK(e, cudaMemcpyAsync(out, e->stgW + first * WALK_WORDS, (size_t)count * KGX_WALK_SIZE, cudaMemcpyDeviceToHost, e->walkStream));
  CK(e, cudaStreamSynchronize(e->walkStream));
  return 0;
}

int kgx_walks_end(kgx_engine* e) {
  CK(e, cudaSetDevice(e->dev));
  if (!e->walksPending) return 0;
  CK(e, cudaEventSynchronize(e->evWalks));
  e->walksPending = false;   // stgW stays allocated for the next export (freed by kgx_destroy): no cudaMalloc / cudaFree,
                             // which can block or synchronise the device, on every checkpoint
  return 0;
}

int kgx_walks_load(kgx_engine* e, const void* recs, uint64_t count, const uint64_t wild_offset[2],
                   const uint64_t keyx[4], const uint64_t keyy[4], int verify,
                   uint64_t* n_bad, uint64_t* bad_idx, uint32_t bad_cap) {
  CK(e, cudaSetDevice(e->dev));
  if (e->walksPending || e->snapPending) { snprintf(e->err, sizeof e->err, "kgx_walks_load: snapshot or walk export pending"); return -1; }
  if (count > e->n) { snprintf(e->err, sizeof e->err, "kgx_walks_load: %llu records for a herd of %llu", (unsigned long long)count, (unsigned long long)e->n); return -1; }
  if (n_bad) *n_bad = 0;
  if (count == 0) return 0;
  if (verify && !e->herdTab) {
    CK(e, cudaMalloc(&e->herdTab, 256 * 16 * 4));
    herd_table_kernel<<<1, 32, 0, e->stream>>>(e->herdTab);
    e->launches++;
    CK(e, cudaGetLastError());
  }
  u64* dRecs = nullptr; u32* dKey = nullptr; uint8_t* dBad = nullptr;
  uint8_t* hBad = nullptr;
  uint64_t key[8];
  memcpy(key, keyx, 32); memcpy(key + 4, keyy, 32);
  auto body = [&]() -> int {      // CK returns from the lambda, so the scratch buffers are always released below
    CK(e, cudaMalloc(&dRecs, (size_t)count * KGX_WALK_SIZE));
    CK(e, cudaMemcpyAsync(dRecs, recs, (size_t)count * KGX_WALK_SIZE, cudaMemcpyHostToDevice, e->stream));
    walks_import_kernel<<<(u32)((e->nPadded + 255) / 256), 256, 0, e->stream>>>(e->state, dRecs, count, e->n, e->nPadded, e->T, e->K,
        wild_offset[0], wild_offset[1], e->symmetry ? 1 : 0, e->aux, e->symRule == KGX_SYM_CLASS ? 0 : 32);
    e->launches++;
    CK(e, cudaGetLastError());
    if (verify) {
      CK(e, cudaMalloc(&dKey, 64));
      CK(e, cudaMalloc(&dBad, count));
      CK(e, cudaMemcpyAsync(dKey, key, 64, cudaMemcpyHostToDevice, e->stream));
      walks_verify_kernel<<<(u32)((count + 127) / 128), 128, 0, e->stream>>>(e->herdTab, dRecs, count, dKey, e->symmetry ? 1 : 0, dBad);
      e->launches++;
      CK(e, cudaGetLastError());
      hBad = static_cast<uint8_t*>(malloc(count));
      if (!hBad) { snprintf(e->err, sizeof e->err, "kgx_walks_load: out of host memory"); return -1; }
      CK(e, cudaMemcpyAsync(hBad, dBad, count, cudaMemcpyDeviceToHost, e->stream));
    }
    CK(e, cudaStreamSynchronize(e->stream));
    if (verify) {
      uint64_t nb = 0;
      for (uint64_t i = 0; i < count; i++)
        if (hBad[i]) { if (bad_idx && nb < bad_cap) bad_idx[nb] = i; nb++; }
      if (n_bad) *n_bad = nb;
    }
    return 0;
  };
  const int rc = body();
  cudaFree(dRecs); cudaFree(dKey); cudaFree(dBad); free(hBad);
  return rc;
}

int kgx_patch(kgx_engine* e, uint64_t kidx, const uint64_t px[4], const uint64_t py[4], const uint64_t d[2]) {
  CK(e, cudaSetDevice(e->dev));
  if (kidx >= e->n) { snprintf(e->err, sizeof e->err, "kgx_patch: kidx out of range"); return -1; }
  PatchArgs a;
  memcpy(&a.c[0], px, 32); memcpy(&a.c[2], py, 32); memcpy(&a.c[4], d, 16);
  patch_kernel<<<1, 32, 0, e->stream>>>(e->state, kidx, a, e->T, e->K, e->aux, e->symRule == KGX_SYM_CLASS ? 0 : 32);   // stream order == the reference's blocking memcpy order (Kangaroo.cpp:607)
  e->launches++;
  CK(e, cudaGetLastError());
  // padding slots replicate kangaroo (s % n): keep them walking their stale copy -- harmless, their DPs are dropped.
  return 0;
}

// Kangaroo::CreateHerd on the device (Kangaroo.cpp:670-738): positions d*G (tame) / key + d*G (wild) for all n
// kangaroos straight into the engine state.  scalars: n x 4 limbs (d mod group order, exactly what the reference
// feeds ComputePublicKeys); d128: n x 2 limbs (the biased distances to store); key: x[4], y[4].
int kgx_create_herd(kgx_engine* e, const uint64_t* scalars, const uint64_t* d128, const uint64_t keyx[4], const uint64_t keyy[4], int first_type) {
  CK(e, cudaSetDevice(e->dev));
  if (e->snapPending) { snprintf(e->err, sizeof e->err, "kgx_create_herd: snapshot pending (read it first)"); return -1; }
  if (!e->herdTab) {
    CK(e, cudaMalloc(&e->herdTab, 256 * 16 * 4));
    herd_table_kernel<<<1, 32, 0, e->stream>>>(e->herdTab);
    e->launches++;
    CK(e, cudaGetLastError());
  }
  if (ensure_staging(e)) return -1;
  u32 *dScal = nullptr, *dKey = nullptr;
  uint64_t key[8];
  memcpy(key, keyx, 32); memcpy(key + 4, keyy, 32);
  auto body = [&]() -> int {      // CK returns from the lambda, so the scratch buffers are always released below
    CK(e, cudaMalloc(&dScal, e->n * 32));
    CK(e, cudaMalloc(&dKey, 64));
    CK(e, cudaMemcpyAsync(dScal, scalars, e->n * 32, cudaMemcpyHostToDevice, e->stream));
    CK(e, cudaMemcpyAsync(dKey, key, 64, cudaMemcpyHostToDevice, e->stream));
    CK(e, cudaMemcpyAsync(e->stgD, d128, e->n * 16, cudaMemcpyHostToDevice, e->stream));
    herd_kernel<<<(u32)((e->n + 127) / 128), 128, 0, e->stream>>>(e->herdTab, dScal, dKey, first_type, e->n,
                                                                 reinterpret_cast<u32*>(e->stgX), reinterpret_cast<u32*>(e->stgY),
                                                                 e->symmetry ? 1 : 0, reinterpret_cast<u32*>(e->stgD));
    e->launches++;
    CK(e, cudaGetLastError());
    u32 blocks = (u32)((e->nPadded + 255) / 256);
    pack_kernel<<<blocks, 256, 0, e->stream>>>(e->state, e->stgX, e->stgY, e->stgD, e->n, e->nPadded, e->T, e->K, e->aux, e->symRule == KGX_SYM_CLASS ? 0 : 32);
    e->launches++;
    CK(e, cudaGetLastError());
    CK(e, cudaStreamSynchronize(e->stream));
    return 0;
  };
  const int rc = body();
  cudaFree(dScal); cudaFree(dKey);
  free_staging(e);
  return rc;
}

int kgx_launch_async(kgx_engine* e) {
  CK(e, cudaSetDevice(e->dev));
  if (!e->haveParams) { snprintf(e->err, sizeof e->err, "kgx_launch_async: kgx_set_params not called"); return -1; }
  if (e->inflight) { snprintf(e->err, sizeof e->err, "kgx_launch_async: previous launch not collected"); return -1; }
  int sidx = e->cur ^ 1;
  LaunchParams p;
  p.state = e->state; p.jtab = e->jtab; p.out = e->slab[sidx]; p.dpMask = e->dpMask; p.nKangaroos = e->n;
  p.numTiles = e->numTiles; p.maxFound = e->maxFound; p.nRun = e->nRun; p.prof = e->prof; p.pre = e->pre; p.G = e->K; p.aux = e->aux; p.symRule = e->symRule; p.pfDist = e->pfDist;
  CK(e, cudaMemsetAsync(e->slab[sidx], 0, 4, e->stream));            // GPUEngine.cu:543
  CK(e, cudaEventRecord(e->evStart[sidx], e->stream));
  u32 grid = (u32)(e->ctasPerSM * e->sms);
  if (grid > e->numTiles) grid = e->numTiles;
  if (e->streamMode) {
    if (e->symmetry) stream_kernel<128, 2, true, true><<<grid, 128, 0, e->stream>>>(p);
    else if (e->streamCtas == 3) {
      if (e->warpInv) stream_kernel<128, 3, true, false><<<grid, 128, 0, e->stream>>>(p);
      else stream_kernel<128, 3, false, false><<<grid, 128, 0, e->stream>>>(p);
    } else {
      if (e->warpInv) stream_kernel<128, 2, true, false><<<grid, 128, 0, e->stream>>>(p);
      else stream_kernel<128, 2, false, false><<<grid, 128, 0, e->stream>>>(p);
    }
  }
  else if (e->tmemMode) jump_kernel_tmem<16><<<grid, 128, e->smemBytes, e->stream>>>(p);
  else if (e->symmetry) g_cfgs[e->cfg].kernSym<<<grid, e->T, e->smemBytes, e->stream>>>(p);
  else g_cfgs[e->cfg].kern<<<grid, e->T, e->smemBytes, e->stream>>>(p);
  e->launches++;
  CK(e, cudaGetLastError());
  CK(e, cudaEventRecord(e->evStop[sidx], e->stream));
  e->cur = sidx;
  e->inflight = true;
  return 0;
}

int kgx_collect(kgx_engine* e, kgx_item* items, uint32_t cap, uint32_t* n_items, uint32_t* n_found, int spin, int relaunch) {
  CK(e, cudaSetDevice(e->dev));
  *n_items = 0; *n_found = 0;
  int sidx = e->cur;
  if (e->inflight) {
    if (spin) {
      cudaError_t q;
      while ((q = cudaEventQuery(e->evStop[sidx])) == cudaErrorNotReady) { }
      CK(e, q);                                       // anything but success / not-ready is a failed launch
    } else {
      CK(e, cudaEventSynchronize(e->evStop[sidx]));   // blocking-sync event: the host thread sleeps (GPUEngine.cu:620-629)
    }
    CK(e, cudaGetLastError());
    CK(e, cudaEventElapsedTime(&e->lastMs, e->evStart[sidx], e->evStop[sidx]));
    e->inflight = false;
    e->done = sidx;
  }
  if (relaunch) { if (kgx_launch_async(e)) return -1; }   // second half of GPUEngine::Launch, issued BEFORE the readback
  // read back slab `sidx` (the new launch writes the other slab)
  // (on its own stream, so it does not queue behind the kernel just started)
  CK(e, cudaMemcpyAsync(e->slabPinned, e->slab[sidx], 4, cudaMemcpyDeviceToHost, e->copyStream));
  CK(e, cudaStreamSynchronize(e->copyStream));
  u32 found = e->slabPinned[0];
  *n_found = found;
  u32 nrec = found > e->maxFound ? e->maxFound : found;
  if (nrec > cap) nrec = cap;
  if (nrec) {
    CK(e, cudaMemcpyAsync(e->slabPinned + 1, e->slab[sidx] + 1, (size_t)nrec * KGX_ITEM_SIZE, cudaMemcpyDeviceToHost, e->copyStream));
    CK(e, cudaStreamSynchronize(e->copyStream));
    memcpy(items, e->slabPinned + 1, (size_t)nrec * KGX_ITEM_SIZE);
  }
  *n_items = nrec;
  return 0;
}

int kgx_sync(kgx_engine* e) {
  CK(e, cudaSetDevice(e->dev));
  CK(e, cudaStreamSynchronize(e->stream));
  if (e->inflight) {
    CK(e, cudaEventElapsedTime(&e->lastMs, e->evStart[e->cur], e->evStop[e->cur]));
    e->inflight = false; e->done = e->cur;
  }
  return 0;
}

// HashTable::Convert on the device for the most recently completed launch (SURVEY 8f/f1).  wild_offset: 2 limbs.
// Returns the device pointer of [u32 count][count x 40-byte DP records] through *out (valid until the next call).
int kgx_convert_dps(kgx_engine* e, const uint64_t wild_offset[2], void** out) {
  CK(e, cudaSetDevice(e->dev));
  if (!e->dp40) CK(e, cudaMalloc(&e->dp40, (size_t)e->maxFound * 40 + 4));
  const int sidx = e->done >= 0 ? e->done : e->cur;
  dp_convert_kernel<<<64, 256, 0, e->copyStream>>>(e->slab[sidx], e->dp40, e->maxFound, wild_offset[0], wild_offset[1], e->symmetry ? 1 : 0);
  e->launches++;
  CK(e, cudaGetLastError());
  CK(e, cudaStreamSynchronize(e->copyStream));
  *out = e->dp40;
  return 0;
}

void* kgx_dp_slab_device(kgx_engine* e) { return e->done >= 0 ? (void*)e->slab[e->done] : (void*)e->slab[e->cur]; }

// ---- test / microbench hooks ----
#define CKH(call) do { cudaError_t _s = (call); if (_s != cudaSuccess) { snprintf(g_create_err, sizeof g_create_err, "%s: %s", #call, cudaGetErrorString(_s)); return -1; } } while (0)

int kgx_test_field(int dev, int op, int n, const uint64_t* a, const uint64_t* b, uint64_t* out) {
  CKH(cudaSetDevice(dev));
  u32 *da, *db, *dout;
  CKH(cudaMalloc(&da, (size_t)n * 32)); CKH(cudaMalloc(&db, (size_t)n * 32)); CKH(cudaMalloc(&dout, (size_t)n * 32));
  CKH(cudaMemcpy(da, a, (size_t)n * 32, cudaMemcpyHostToDevice));
  CKH(cudaMemcpy(db, b, (size_t)n * 32, cudaMemcpyHostToDevice));
  test_field_kernel<<<(n + 127) / 128, 128>>>(op, n, da, db, dout);
  CKH(cudaGetLastError());
  CKH(cudaMemcpy(out, dout, (size_t)n * 32, cudaMemcpyDeviceToHost));
  cudaFree(da); cudaFree(db); cudaFree(dout);
  return 0;
}

int kgx_bench_raw(int dev, int kind, int iters, float* ms, double* ops) {
  CKH(cudaSetDevice(dev));
  cudaDeviceProp prop; CKH(cudaGetDeviceProperties(&prop, dev));
  u32* sink; CKH(cudaMalloc(&sink, 4));
  cudaEvent_t a, b; CKH(cudaEventCreate(&a)); CKH(cudaEventCreate(&b));
  const int blocks = prop.multiProcessorCount * 8, threads = 256;
  bench_raw_kernel<<<blocks, threads>>>(kind, iters / 8 + 1, sink);   // warm-up
  CKH(cudaDeviceSynchronize());
  CKH(cudaEventRecord(a));
  bench_raw_kernel<<<blocks, threads>>>(kind, iters, sink);
  CKH(cudaEventRecord(b));
  CKH(cudaEventSynchronize(b));
  CKH(cudaGetLastError());
  CKH(cudaEventElapsedTime(ms, a, b));
  double per_thread = kind == 0 ? 8.0 * iters : (kind == 3 ? 1.0 * iters : 2.0 * iters);
  *ops = per_thread * (double)blocks * threads;
  cudaFree(sink); cudaEventDestroy(a); cudaEventDestroy(b);
  return 0;
}

}  // extern "C"

// ---- device DP table (kgx_dptable.cuh; C ABI include/kgx.h kgx_dpt_*) ----
namespace {
constexpr double DPT_LOAD = 0.7;                      // entries per slot at capacity (KGX_DPT_LOAD)
constexpr uint64_t DPT_TAIL = 1 << 16;                // slots past the last bucket for the last buckets' probes
constexpr uint32_t DPT_MAX_S = 9000;                  // slots per bucket: keeps a bucket's export sort inside dpt::MAXB
constexpr uint64_t DPT_SCRATCH = 1 << 22;             // entries of one export / bulk-load chunk (128 MiB)
constexpr uint32_t DPT_CHUNK_BUCKETS = 4096;          // buckets counted per export read
constexpr int DPT_RING = 2;                           // inserts whose events have not been collected yet

uint32_t dpt_slots_per_bucket(uint64_t capacity) {
  const double s = std::ceil((double)capacity / DPT_LOAD / (double)dpt::HASH_SIZE);
  return s < 1 ? 1u : (s > 4e9 ? 0xFFFFFFFFu : (uint32_t)s);
}
uint64_t dpt_table_bytes(uint32_t S) { return ((uint64_t)dpt::HASH_SIZE * S + DPT_TAIL) * 40; }
char g_dpt_err[256] = "";
}  // namespace

struct kgx_dpt {
  int dev = 0;
  uint64_t capacity = 0;
  dpt::Table tab{};
  uint32_t epoch = 0, evCap = 0;
  cudaStream_t stream = nullptr, expStream = nullptr;
  // inserts: batch scratch (grown to the largest batch) and a ring of event buffers, device + pinned host
  uint32_t batchCap = 0;
  uint32_t* L = nullptr; uint32_t* head = nullptr; unsigned long long* res = nullptr;
  uint8_t* evDev[DPT_RING] = {nullptr, nullptr};
  uint8_t* evHost[DPT_RING] = {nullptr, nullptr};
  cudaEvent_t evDone[DPT_RING] = {nullptr, nullptr};
  int ringHead = 0, pending = 0;
  // export / bulk load
  ulonglong2* scratch = nullptr;
  uint32_t* dH = nullptr;                             // bulk load: buckets of a chunk
  uint32_t* dCounts = nullptr; unsigned long long* dOff = nullptr;
  uint32_t* hCounts = nullptr; unsigned long long* hOff = nullptr;
  dpt::EvHeader* dHdr = nullptr; dpt::EvHeader* hHdr = nullptr;
  cudaEvent_t evExp = nullptr;
  bool exporting = false;
  uint32_t expEpoch = 0;
  char err[256] = "";
};

extern "C" {

const char* kgx_dpt_last_error(kgx_dpt* t) { return t ? t->err : g_dpt_err; }

uint64_t kgx_dpt_memory_bytes(uint64_t capacity) {
  return dpt_table_bytes(dpt_slots_per_bucket(capacity)) + DPT_SCRATCH * 36 + 8;
}

uint64_t kgx_dpt_max_capacity(void) { return (uint64_t)(DPT_LOAD * DPT_MAX_S * dpt::HASH_SIZE); }

void kgx_dpt_destroy(kgx_dpt* t) {
  if (!t) return;
  cudaSetDevice(t->dev);
  if (t->stream) cudaStreamSynchronize(t->stream);
  if (t->expStream) cudaStreamSynchronize(t->expStream);
  for (int i = 0; i < DPT_RING; i++) {
    if (t->evDone[i]) { cudaEventSynchronize(t->evDone[i]); cudaEventDestroy(t->evDone[i]); }
    cudaFree(t->evDev[i]);
    if (t->evHost[i]) cudaFreeHost(t->evHost[i]);
  }
  cudaFree(t->tab.meta); cudaFree(t->tab.ent); cudaFree(t->tab.count);
  cudaFree(t->L); cudaFree(t->head); cudaFree(t->res);
  cudaFree(t->scratch); cudaFree(t->dH); cudaFree(t->dCounts); cudaFree(t->dOff); cudaFree(t->dHdr);
  if (t->hCounts) cudaFreeHost(t->hCounts);
  if (t->hOff) cudaFreeHost(t->hOff);
  if (t->hHdr) cudaFreeHost(t->hHdr);
  if (t->evExp) cudaEventDestroy(t->evExp);
  if (t->stream) cudaStreamDestroy(t->stream);
  if (t->expStream) cudaStreamDestroy(t->expStream);
  delete t;
}

kgx_dpt* kgx_dpt_create(int dev, uint64_t capacity, uint32_t max_events) {
  kgx_dpt* t = new kgx_dpt();
  auto fail = [&](const char* what, cudaError_t s) -> kgx_dpt* {
    snprintf(g_dpt_err, sizeof g_dpt_err, "kgx_dpt_create: %s: %s", what, cudaGetErrorString(s));
    cudaGetLastError();
    kgx_dpt_destroy(t);
    return nullptr;
  };
  if (capacity == 0 || capacity > kgx_dpt_max_capacity() || max_events == 0) {
    snprintf(g_dpt_err, sizeof g_dpt_err, "kgx_dpt_create: capacity must be in [1, %llu] and max_events > 0",
             (unsigned long long)kgx_dpt_max_capacity());
    delete t; return nullptr;
  }
  cudaError_t s;
  if ((s = cudaSetDevice(dev)) != cudaSuccess) return fail("cudaSetDevice", s);
  t->dev = dev; t->capacity = capacity; t->evCap = max_events;
  t->tab.S = dpt_slots_per_bucket(capacity);
  t->tab.nslots = (uint64_t)dpt::HASH_SIZE * t->tab.S + DPT_TAIL;
  if ((s = cudaStreamCreateWithFlags(&t->stream, cudaStreamNonBlocking)) != cudaSuccess) return fail("cudaStreamCreate", s);
  if ((s = cudaStreamCreateWithFlags(&t->expStream, cudaStreamNonBlocking)) != cudaSuccess) return fail("cudaStreamCreate", s);
  if ((s = cudaMalloc(&t->tab.meta, t->tab.nslots * 8)) != cudaSuccess) return fail("cudaMalloc(meta)", s);
  if ((s = cudaMalloc(&t->tab.ent, t->tab.nslots * 32)) != cudaSuccess) return fail("cudaMalloc(entries)", s);
  if ((s = cudaMalloc(&t->tab.count, 8)) != cudaSuccess) return fail("cudaMalloc(count)", s);
  if ((s = cudaMemsetAsync(t->tab.meta, 0, t->tab.nslots * 8, t->stream)) != cudaSuccess) return fail("cudaMemset(meta)", s);
  if ((s = cudaMemsetAsync(t->tab.count, 0, 8, t->stream)) != cudaSuccess) return fail("cudaMemset(count)", s);
  const size_t evBytes = sizeof(dpt::EvHeader) + (size_t)max_events * sizeof(dpt::Event);
  for (int i = 0; i < DPT_RING; i++) {
    if ((s = cudaMalloc(&t->evDev[i], evBytes)) != cudaSuccess) return fail("cudaMalloc(events)", s);
    if ((s = cudaHostAlloc(&t->evHost[i], evBytes, cudaHostAllocDefault)) != cudaSuccess) return fail("cudaHostAlloc(events)", s);
    if ((s = cudaEventCreateWithFlags(&t->evDone[i], cudaEventDisableTiming)) != cudaSuccess) return fail("cudaEventCreate", s);
  }
  if ((s = cudaMalloc(&t->scratch, DPT_SCRATCH * 32)) != cudaSuccess) return fail("cudaMalloc(scratch)", s);
  if ((s = cudaMalloc(&t->dH, DPT_SCRATCH * 4)) != cudaSuccess) return fail("cudaMalloc(scratch)", s);
  if ((s = cudaMalloc(&t->dCounts, DPT_CHUNK_BUCKETS * 4)) != cudaSuccess) return fail("cudaMalloc(counts)", s);
  if ((s = cudaMalloc(&t->dOff, DPT_CHUNK_BUCKETS * 8)) != cudaSuccess) return fail("cudaMalloc(offsets)", s);
  if ((s = cudaMalloc(&t->dHdr, sizeof(dpt::EvHeader))) != cudaSuccess) return fail("cudaMalloc(header)", s);
  if ((s = cudaHostAlloc(&t->hCounts, DPT_CHUNK_BUCKETS * 4, cudaHostAllocDefault)) != cudaSuccess) return fail("cudaHostAlloc", s);
  if ((s = cudaHostAlloc(&t->hOff, DPT_CHUNK_BUCKETS * 8, cudaHostAllocDefault)) != cudaSuccess) return fail("cudaHostAlloc", s);
  if ((s = cudaHostAlloc(&t->hHdr, sizeof(dpt::EvHeader), cudaHostAllocDefault)) != cudaSuccess) return fail("cudaHostAlloc", s);
  if ((s = cudaEventCreateWithFlags(&t->evExp, cudaEventDisableTiming)) != cudaSuccess) return fail("cudaEventCreate", s);
  if ((s = cudaFuncSetAttribute(dpt::export_sort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dpt::SORT_SMEM)) != cudaSuccess)
    return fail("cudaFuncSetAttribute(export_sort_kernel)", s);
  if ((s = cudaStreamSynchronize(t->stream)) != cudaSuccess) return fail("sync", s);
  return t;
}

uint64_t kgx_dpt_capacity(kgx_dpt* t) { return t->capacity; }

#define CKT(call)                                                                              \
  do {                                                                                         \
    cudaError_t _s = (call);                                                                   \
    if (_s != cudaSuccess) {                                                                   \
      snprintf(t->err, sizeof(t->err), "%s: %s", #call, cudaGetErrorString(_s));              \
      return -3;                                                                               \
    }                                                                                          \
  } while (0)

static int dpt_grow(kgx_dpt* t, uint32_t n) {
  if (n <= t->batchCap) return 0;
  for (int k = 0; k < t->pending; k++) CKT(cudaEventSynchronize(t->evDone[(t->ringHead + k) % DPT_RING]));   // still in use
  uint32_t cap = t->batchCap ? t->batchCap : (1u << 16);
  while (cap < n) cap *= 2;
  cudaFree(t->L); cudaFree(t->head); cudaFree(t->res);
  t->L = nullptr; t->head = nullptr; t->res = nullptr; t->batchCap = 0;
  CKT(cudaMalloc(&t->L, (size_t)cap * 2 * 4));
  CKT(cudaMalloc(&t->head, (size_t)cap * 4));
  CKT(cudaMalloc(&t->res, (size_t)cap * 8));
  t->batchCap = cap;
  return 0;
}

int kgx_dpt_insert(kgx_dpt* t, const void* recs, uint32_t stride, const uint32_t* counts, uint32_t nranks, void* stream) {
  CKT(cudaSetDevice(t->dev));
  if (nranks == 0 || nranks > (uint32_t)dpt::MAX_RANKS) { snprintf(t->err, sizeof t->err, "kgx_dpt_insert: 1..%d ranks", dpt::MAX_RANKS); return -3; }
  if (t->pending == DPT_RING) { snprintf(t->err, sizeof t->err, "kgx_dpt_insert: %d inserts pending, collect their events first", DPT_RING); return -3; }
  dpt::Batch b;
  b.base = static_cast<const uint32_t*>(recs); b.stride = stride; b.nranks = nranks;
  uint64_t n = 0;
  for (uint32_t r = 0; r < nranks; r++) {
    if (nranks > 1 && counts[r] > stride) { snprintf(t->err, sizeof t->err, "kgx_dpt_insert: rank %u: %u records, stride %u", r, counts[r], stride); return -3; }
    b.prefix[r] = (uint32_t)n; n += counts[r];
  }
  b.prefix[nranks] = (uint32_t)n;
  if (n >= (1u << 31)) { snprintf(t->err, sizeof t->err, "kgx_dpt_insert: batch too large"); return -3; }
  if (int rc = dpt_grow(t, (uint32_t)n)) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int slot = (t->ringHead + t->pending) % DPT_RING;
  dpt::EvHeader* hdr = reinterpret_cast<dpt::EvHeader*>(t->evDev[slot]);
  dpt::Event* ev = reinterpret_cast<dpt::Event*>(t->evDev[slot] + sizeof(dpt::EvHeader));
  const uint32_t epoch = ++t->epoch;
  CKT(cudaMemsetAsync(hdr, 0, sizeof *hdr, st));
  if (n) {
    uint32_t lsize = 1;
    while (lsize < 2 * n) lsize <<= 1;
    const uint32_t blocks = (uint32_t)((n + 255) / 256);
    CKT(cudaMemsetAsync(t->L, 0xFF, (size_t)lsize * 4, st));
    dpt::dedup_kernel<<<blocks, 256, 0, st>>>(b, (uint32_t)n, t->L, lsize - 1, hdr);
    dpt::head_kernel<<<blocks, 256, 0, st>>>(b, (uint32_t)n, t->L, lsize - 1, t->tab, epoch, t->head, t->res, hdr);
    dpt::event_kernel<<<blocks, 256, 0, st>>>(b, (uint32_t)n, t->tab, t->head, t->res, hdr, ev, t->evCap);
  }
  dpt::snapshot_count_kernel<<<1, 1, 0, st>>>(t->tab.count, hdr);
  CKT(cudaGetLastError());
  CKT(cudaMemcpyAsync(t->evHost[slot], t->evDev[slot], sizeof(dpt::EvHeader) + (size_t)t->evCap * sizeof(dpt::Event),
                      cudaMemcpyDeviceToHost, st));
  CKT(cudaEventRecord(t->evDone[slot], st));
  t->pending++;
  return 0;
}

int kgx_dpt_events(kgx_dpt* t, void* out, uint32_t cap, uint32_t* n_ev, uint64_t* entries) {
  CKT(cudaSetDevice(t->dev));
  *n_ev = 0;
  if (t->pending == 0) { snprintf(t->err, sizeof t->err, "kgx_dpt_events: no insert pending"); return -3; }
  const int slot = t->ringHead;
  CKT(cudaEventSynchronize(t->evDone[slot]));
  t->ringHead = (t->ringHead + 1) % DPT_RING;
  t->pending--;
  const dpt::EvHeader* hdr = reinterpret_cast<const dpt::EvHeader*>(t->evHost[slot]);
  const uint32_t k = std::min(std::min(hdr->count, cap), t->evCap);
  memcpy(out, t->evHost[slot] + sizeof(dpt::EvHeader), (size_t)k * sizeof(dpt::Event));
  *n_ev = hdr->count;
  if (entries) *entries = hdr->entries;
  if (hdr->flags & dpt::FLAG_OVERFLOW) { snprintf(t->err, sizeof t->err, "kgx_dpt_events: a probe ran past the table's last slot"); return -2; }
  return (hdr->flags & dpt::FLAG_BAD) ? -1 : 0;
}

int kgx_dpt_pending(kgx_dpt* t) { return t->pending; }

int kgx_dpt_count(kgx_dpt* t, uint64_t* entries) {
  CKT(cudaSetDevice(t->dev));
  for (int k = 0; k < t->pending; k++) CKT(cudaEventSynchronize(t->evDone[(t->ringHead + k) % DPT_RING]));
  CKT(cudaMemcpyAsync(&t->hHdr->entries, t->tab.count, 8, cudaMemcpyDeviceToHost, t->stream));
  CKT(cudaStreamSynchronize(t->stream));
  *entries = t->hHdr->entries;
  return 0;
}

int kgx_dpt_export_begin(kgx_dpt* t, void* stream) {
  CKT(cudaSetDevice(t->dev));
  if (t->exporting) { snprintf(t->err, sizeof t->err, "kgx_dpt_export_begin: previous export not ended"); return -3; }
  t->expEpoch = t->epoch;
  CKT(cudaEventRecord(t->evExp, static_cast<cudaStream_t>(stream)));
  t->exporting = true;
  return 0;
}

int kgx_dpt_export_read(kgx_dpt* t, uint32_t first_bucket, uint32_t max_buckets, void* entries, uint64_t entries_cap,
                        uint32_t* counts, uint32_t* n_buckets, uint64_t* n_entries) {
  CKT(cudaSetDevice(t->dev));
  *n_buckets = 0; *n_entries = 0;
  if (!t->exporting) { snprintf(t->err, sizeof t->err, "kgx_dpt_export_read: no export begun"); return -3; }
  if (first_bucket >= dpt::HASH_SIZE || max_buckets == 0) return 0;
  const uint32_t nb = std::min(std::min(max_buckets, dpt::HASH_SIZE - first_bucket), DPT_CHUNK_BUCKETS);
  CKT(cudaStreamWaitEvent(t->expStream, t->evExp, 0));
  dpt::export_count_kernel<<<nb, 256, 0, t->expStream>>>(t->tab, first_bucket, t->expEpoch, t->dCounts);
  CKT(cudaGetLastError());
  CKT(cudaMemcpyAsync(t->hCounts, t->dCounts, (size_t)nb * 4, cudaMemcpyDeviceToHost, t->expStream));
  CKT(cudaStreamSynchronize(t->expStream));
  const uint64_t lim = std::min<uint64_t>(entries_cap, DPT_SCRATCH);
  uint64_t total = 0;
  uint32_t k = 0;
  for (; k < nb; k++) {
    const uint32_t c = t->hCounts[k];
    if (c > (uint32_t)dpt::MAXB) {
      snprintf(t->err, sizeof t->err, "kgx_dpt_export_read: bucket %u holds %u entries, more than %d", first_bucket + k, c, dpt::MAXB);
      return -3;
    }
    if (total + c > lim) break;
    t->hOff[k] = total;
    total += c;
  }
  if (k == 0) { snprintf(t->err, sizeof t->err, "kgx_dpt_export_read: room for %llu entries, bucket %u holds %u",
                         (unsigned long long)entries_cap, first_bucket, t->hCounts[0]); return -3; }
  CKT(cudaMemcpyAsync(t->dOff, t->hOff, (size_t)k * 8, cudaMemcpyHostToDevice, t->expStream));
  dpt::export_sort_kernel<<<k, dpt::SORT_THREADS, dpt::SORT_SMEM, t->expStream>>>(t->tab, first_bucket, t->expEpoch, t->dOff, t->scratch);
  CKT(cudaGetLastError());
  if (total) CKT(cudaMemcpyAsync(entries, t->scratch, total * 32, cudaMemcpyDeviceToHost, t->expStream));
  CKT(cudaStreamSynchronize(t->expStream));
  memcpy(counts, t->hCounts, (size_t)k * 4);
  *n_buckets = k; *n_entries = total;
  return 0;
}

int kgx_dpt_export_end(kgx_dpt* t) {
  CKT(cudaSetDevice(t->dev));
  if (!t->exporting) return 0;
  CKT(cudaStreamSynchronize(t->expStream));
  t->exporting = false;
  return 0;
}

int kgx_dpt_load(kgx_dpt* t, const uint32_t* h, const void* entries32, uint64_t n) {
  CKT(cudaSetDevice(t->dev));
  if (t->pending || t->exporting) { snprintf(t->err, sizeof t->err, "kgx_dpt_load: inserts or an export pending"); return -3; }
  const uint32_t epoch = ++t->epoch;
  CKT(cudaMemsetAsync(t->dHdr, 0, sizeof(dpt::EvHeader), t->stream));
  const uint8_t* e = static_cast<const uint8_t*>(entries32);
  for (uint64_t o = 0; o < n; o += DPT_SCRATCH) {
    const uint64_t k = std::min<uint64_t>(DPT_SCRATCH, n - o);
    CKT(cudaMemcpyAsync(t->dH, h + o, k * 4, cudaMemcpyHostToDevice, t->stream));
    CKT(cudaMemcpyAsync(t->scratch, e + o * 32, k * 32, cudaMemcpyHostToDevice, t->stream));
    dpt::load_kernel<<<(uint32_t)((k + 255) / 256), 256, 0, t->stream>>>(t->dH, t->scratch, k, t->tab, epoch, t->dHdr);
    CKT(cudaGetLastError());
  }
  CKT(cudaMemcpyAsync(t->hHdr, t->dHdr, sizeof(dpt::EvHeader), cudaMemcpyDeviceToHost, t->stream));
  CKT(cudaStreamSynchronize(t->stream));
  if (t->hHdr->flags & dpt::FLAG_OVERFLOW) { snprintf(t->err, sizeof t->err, "kgx_dpt_load: a probe ran past the table's last slot"); return -2; }
  if (t->hHdr->flags & dpt::FLAG_BAD) { snprintf(t->err, sizeof t->err, "kgx_dpt_load: h >= 2^18"); return -1; }
  return 0;
}

}  // extern "C"
