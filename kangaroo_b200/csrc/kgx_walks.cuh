// kgx_walks.cuh -- herd <-> work-file walk records on the device (kgx_walks_* in include/kgx.h).
//
// A work file written with kangaroos (reference: Kangaroo::SaveWork with -ws, Backup.cpp:535-545; read back by FetchWalks,
// :211-231) ends with one 96-byte record per kangaroo: {x[4], y[4], d[4]} as 64-bit little-endian limbs, record i being
// kangaroo kIdx i (herd type = i & 1).  d is the UNBIASED distance mod n -- exactly what GPUEngine::GetKangaroos returns:
//   tame                 the stored 128-bit distance, zero-extended;
//   wild                 (biased - wildOffset) mod n, so a negative distance appears as n - |d|;
//   symmetric engines    the signed 128-bit distance taken mod n (no offset).
// Export turns the tile state (any of the three layouts, padding slots skipped) straight into records; import is the
// inverse (records -> biased 128-bit distances, truncated like the reference's SetKangaroos) written into the tile state
// with the padding replication of pack_kernel; verify recomputes d*G (+key) with herd_point and compares.
#pragma once
#include "kgx_kernel.cuh"
#include "kgx_herd.cuh"

namespace kgx {

constexpr int WALK_WORDS = 12;   // u64 limbs per 96-byte record

__device__ __constant__ u64 kOrderN[4] = {0xBFD25E8CD0364141ull, 0xBAAEDCE6AF48A03Bull, 0xFFFFFFFFFFFFFFFEull, 0xFFFFFFFFFFFFFFFFull};

// r = n - m for a 128-bit m (m != 0, so the result is in (0, n))
__device__ __forceinline__ void order_minus128(u64* r, u64 m0, u64 m1) {
  u64 b = 0;
  r[0] = kOrderN[0] - m0; b = kOrderN[0] < m0;
  const u64 t1 = kOrderN[1] - m1; const u64 b1 = (kOrderN[1] < m1) | (t1 < b); r[1] = t1 - b; b = b1;
  r[2] = kOrderN[2] - b;   // n[2], n[3] are far from 0: the borrow stops here
  r[3] = kOrderN[3];
}

__device__ __forceinline__ void slot_of(u64 s, int T, int K, u64* tile, int* g, int* t) {
  const int TILE = T * K;
  *tile = s / TILE; const int r = (int)(s % TILE); *g = r / T; *t = r % T;
}

// state (tile layout) -> out[n][12] records in kIdx order.  One thread per kangaroo.
__global__ void walks_export_kernel(const uint4* __restrict__ state, u64* __restrict__ out, u64 n, int T, int K,
                                    u64 wo0, u64 wo1, int signedMode) {
  const u64 s = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  u64 tile; int g, t;
  slot_of(s, T, K, &tile, &g, &t);
  const uint4* src = state + tile * (K * CHUNKS * T);
  u64* r = out + s * WALK_WORDS;
#pragma unroll
  for (int c = 0; c < 4; c++) {
    const uint4 v = src[(g * CHUNKS + c) * T + t];
    r[2 * c] = (u64)v.x | ((u64)v.y << 32);
    r[2 * c + 1] = (u64)v.z | ((u64)v.w << 32);
  }
  const uint4 dv = src[(g * CHUNKS + 4) * T + t];
  const u64 d0 = (u64)dv.x | ((u64)dv.y << 32), d1 = (u64)dv.z | ((u64)dv.w << 32);
  u64 D[4] = {d0, d1, 0, 0};
  if (signedMode) {
    if (d1 >> 63) {                                 // negative: n - |d|
      const u64 m0 = ~d0 + 1, m1 = ~d1 + (m0 == 0);
      order_minus128(D, m0, m1);
    }
  } else if (s & 1ull) {                            // wild: d - wildOffset mod n
    if (d1 > wo1 || (d1 == wo1 && d0 >= wo0)) {
      D[0] = d0 - wo0; D[1] = d1 - wo1 - (d0 < wo0);
    } else {
      const u64 m0 = wo0 - d0, m1 = wo1 - d1 - (wo0 < d0);
      order_minus128(D, m0, m1);
    }
  }
#pragma unroll
  for (int w = 0; w < 4; w++) r[8 + w] = D[w];
}

// recs[count][12] -> tile state for every slot s < nPadded whose source kangaroo (s, or s % n for padding) is < count;
// the other slots keep their state.  Rule state (lastJump / symClass) of the written slots is reset like pack_kernel.
__global__ void walks_import_kernel(uint4* __restrict__ state, const u64* __restrict__ recs, u64 count, u64 n, u64 nPadded,
                                    int T, int K, u64 wo0, u64 wo1, int signedMode, uint8_t* aux, int auxInit) {
  const u64 s = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= nPadded) return;
  const u64 src = s < n ? s : s % n;
  if (src >= count) return;
  const u64* r = recs + src * WALK_WORDS;
  u64 D[4] = {r[8], r[9], r[10], r[11]};
  u64 d0 = D[0], d1 = D[1];
  if (signedMode) {
    // d mod n -> signed 128-bit: values above n/2 are negative, stored as low 128 bits of d - n
    bool gtHalf = false;
    const u64 half[4] = {0xDFE92F46681B20A0ull, 0x5D576E7357A4501Dull, 0xFFFFFFFFFFFFFFFFull, 0x7FFFFFFFFFFFFFFFull};
    for (int w = 3; w >= 0; w--) if (D[w] != half[w]) { gtHalf = D[w] > half[w]; break; }
    if (gtHalf) { d0 = D[0] - kOrderN[0]; d1 = D[1] - kOrderN[1] - (D[0] < kOrderN[0]); }
  } else if (src & 1ull) {
    // (d + wildOffset) mod n, truncated to 128 bits (GPUEngine.cu:407-411)
    u64 t[4], c = 0;
    t[0] = D[0] + wo0; c = t[0] < wo0;
    t[1] = D[1] + wo1 + c; c = (t[1] < wo1) | (c & (t[1] == wo1));
    t[2] = D[2] + c; c = c & (t[2] == 0);
    t[3] = D[3] + c; c = c & (t[3] == 0);
    bool ge = c != 0;
    if (!ge) { ge = true; for (int w = 3; w >= 0; w--) if (t[w] != kOrderN[w]) { ge = t[w] > kOrderN[w]; break; } }
    if (ge) { const u64 b = t[0] < kOrderN[0]; t[0] -= kOrderN[0]; t[1] = t[1] - kOrderN[1] - b; }
    d0 = t[0]; d1 = t[1];
  }
  u64 tile; int g, t;
  slot_of(s, T, K, &tile, &g, &t);
  uint4* dst = state + tile * (K * CHUNKS * T);
#pragma unroll
  for (int c = 0; c < 4; c++)
    dst[(g * CHUNKS + c) * T + t] = make_uint4((u32)r[2 * c], (u32)(r[2 * c] >> 32), (u32)r[2 * c + 1], (u32)(r[2 * c + 1] >> 32));
  dst[(g * CHUNKS + 4) * T + t] = make_uint4((u32)d0, (u32)(d0 >> 32), (u32)d1, (u32)(d1 >> 32));
  if (aux) aux[tile * (u64)(T * K) + (u64)g * T + t] = (uint8_t)auxInit;
}

// bad[i] = 1 when record i is not d*G (tame, even i) / key + d*G (wild, odd i).  Symmetric engines negate point and
// distance together, so a wild walk sits at +-key + d*G: both signs are accepted there.  The point at infinity is
// stored as (0, 0) by herd creation and is accepted in that form.  key: 16 words (x, y).
__global__ void walks_verify_kernel(const u32* __restrict__ tab, const u64* __restrict__ recs, u64 count, const u32* __restrict__ key,
                                    int signedMode, uint8_t* __restrict__ bad) {
  const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const u64* r = recs + i * WALK_WORDS;
  u32 k[8], rx[8], ry[8];
#pragma unroll
  for (int w = 0; w < 4; w++) {
    rx[2 * w] = (u32)r[w]; rx[2 * w + 1] = (u32)(r[w] >> 32);
    ry[2 * w] = (u32)r[4 + w]; ry[2 * w + 1] = (u32)(r[4 + w] >> 32);
    k[2 * w] = (u32)r[8 + w]; k[2 * w + 1] = (u32)(r[8 + w] >> 32);
  }
  const bool wild = (i & 1ull) != 0;
  auto matches = [&](const u32* q) -> bool {
    u32 X[8], Y[8];
    if (!herd_point(tab, k, q, X, Y)) {
      u32 o = 0;
      for (int w = 0; w < 8; w++) o |= rx[w] | ry[w];
      return o == 0;
    }
    u32 diff = 0;
    for (int w = 0; w < 8; w++) diff |= (X[w] ^ rx[w]) | (Y[w] ^ ry[w]);
    return diff == 0;
  };
  bool ok = matches(wild ? key : nullptr);
  if (!ok && wild && signedMode) {
    u32 nk[16];
    for (int w = 0; w < 8; w++) nk[w] = key[w];
    fe_neg(nk + 8, key + 8);
    ok = matches(nk);
  }
  bad[i] = ok ? 0 : 1;
}

}  // namespace kgx
