// kgx_dptable.cuh -- rank-0 distinguished-point table in device memory (C ABI: include/kgx.h kgx_dpt_*; SURVEY.md 8f row f1,
// device half).  Same decisions as the host table (kgx_ingest.cpp, the reference's HashTable::Add), made where the gathered
// DP records already are.
//
// Layout.  Open addressing with linear probing over nslots = 2^18 * S + KGX_DPT_TAIL slots.  Slot s holds
//   meta[s] = (epoch << 32) | (h + 1)      (0 = empty; epoch = the insert call that stored it, 1, 2, ...)
//   ent[s]  = {x[2], d[2]}                 (the 32-byte work-file entry)
// 40 bytes per slot.  The home slot is h-major: h * S + floor(x[1].hi32 * S / 2^32), so bucket h's entries lie in
// [h * S, first stop slot at or after (h + 1) * S) -- what makes a bucket-range export a slot-range scan.  S is chosen so
// that the table holds `capacity` entries at a load of at most KGX_DPT_LOAD; probing never wraps (running off the tail is
// reported as an overflow, which a load of 0.7 makes practically impossible).
//
// Insert of one batch (records in batch order = rank, then index inside the rank):
//   dedup   each record claims (atomicCAS) or finds its key (h, x) in a batch-local index table; atomicMin keeps the lowest
//           record index there, so every key of the batch ends with its first record ("head")
//   head    every record learns its head; heads probe the table.  A slot of the current epoch was empty before this batch,
//           so it cannot hold the head's key and is passed over without reading its entry; an empty slot ends the search
//           (no deletions) and is claimed by CAS on meta, then x and d are written.  Keys of one batch are distinct
//           heads, so no two threads ever insert or wait for the same key.
//   event   each record compares with what the host table would have stored when it arrived: the table's entry when the
//           key was there before the batch, else its head's record (the head itself is ADD_OK).
// Exports filter on epoch <= L (the last insert before kgx_dpt_export_begin), so they are a snapshot of inserts 1..L and
// may run on their own stream while later inserts proceed: those only fill slots that were empty at L.
#pragma once
#include <cstdint>

namespace kgx {
namespace dpt {

constexpr uint32_t HASH_SIZE = 1u << 18;
constexpr uint64_t TYPE = 0x4000000000000000ULL;
constexpr uint32_t EMPTY32 = 0xFFFFFFFFu;
constexpr uint64_t RES_NEW = ~0ULL - 1, RES_FAIL = ~0ULL;
constexpr int MAXB = 8192;                    // entries of one bucket the export can sort in shared memory
constexpr int SORT_THREADS = 1024;
constexpr size_t SORT_SMEM = (size_t)MAXB * (8 + 8 + 4);
constexpr int MAX_RANKS = 64;
constexpr uint32_t FLAG_BAD = 1, FLAG_OVERFLOW = 2;

struct Event { uint32_t kind, rank, kidx, h; uint64_t d_old[2], d_new[2]; };   // kgi_event
static_assert(sizeof(Event) == 48, "kgi_event layout");
struct EvHeader { uint32_t count, flags; unsigned long long entries; };

struct Table {
  unsigned long long* meta;
  ulonglong2* ent;                            // 2 per slot: x, d
  uint64_t nslots;
  uint32_t S;
  unsigned long long* count;                  // entries stored
};

struct Batch {
  const uint32_t* base;                       // 40-byte records, 4-byte aligned (kgx_convert_dps output starts at +4)
  uint32_t stride;                            // records between two ranks' segments
  uint32_t nranks;
  uint32_t prefix[MAX_RANKS + 1];             // prefix[r] = records of ranks < r
};

struct Rec { uint32_t kidx, h, rank; uint64_t x0, x1, d0, d1; };

__device__ __forceinline__ uint64_t w64(const uint32_t* p) { return (uint64_t)p[0] | ((uint64_t)p[1] << 32); }

__device__ __forceinline__ Rec load_rec(const Batch& b, uint32_t i) {
  uint32_t r = 0;
  while (r + 1 < b.nranks && i >= b.prefix[r + 1]) r++;
  const uint32_t* p = b.base + ((uint64_t)r * b.stride + (i - b.prefix[r])) * 10;
  Rec o;
  o.kidx = p[0]; o.h = p[1]; o.rank = r;
  o.x0 = w64(p + 2); o.x1 = w64(p + 4); o.d0 = w64(p + 6); o.d1 = w64(p + 8);
  return o;
}

__device__ __forceinline__ uint64_t home(const Table& t, uint32_t h, uint64_t x1) {
  return (uint64_t)h * t.S + (((x1 >> 32) * t.S) >> 32);
}

__device__ __forceinline__ uint32_t mix(uint32_t h, uint64_t x0, uint64_t x1) {
  uint64_t v = x0 ^ (x1 * 0x9E3779B97F4A7C15ULL) ^ ((uint64_t)h << 40);
  v ^= v >> 31; v *= 0xBF58476D1CE4E5B9ULL; v ^= v >> 29;
  return (uint32_t)v;
}

__device__ __forceinline__ bool same_key(const Rec& a, const Rec& b) { return a.h == b.h && a.x0 == b.x0 && a.x1 == b.x1; }

// 1. every key of the batch -> its lowest record index in L (lmask + 1 entries, EMPTY32-filled)
__global__ void dedup_kernel(Batch b, uint32_t n, uint32_t* L, uint32_t lmask, EvHeader* hdr) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Rec r = load_rec(b, i);
  if (r.h >= HASH_SIZE) { atomicOr(&hdr->flags, FLAG_BAD); return; }
  for (uint32_t p = mix(r.h, r.x0, r.x1) & lmask;; p = (p + 1) & lmask) {
    const uint32_t v = atomicCAS(&L[p], EMPTY32, i);
    if (v == EMPTY32) return;
    if (same_key(load_rec(b, v), r)) { atomicMin(&L[p], i); return; }
  }
}

// 2. head of every record; heads look their key up in the table and insert it when absent
__global__ void head_kernel(Batch b, uint32_t n, const uint32_t* L, uint32_t lmask, Table t, uint32_t epoch,
                            uint32_t* head, unsigned long long* res, EvHeader* hdr) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Rec r = load_rec(b, i);
  if (r.h >= HASH_SIZE) { head[i] = EMPTY32; return; }
  uint32_t hd = EMPTY32;
  for (uint32_t p = mix(r.h, r.x0, r.x1) & lmask;; p = (p + 1) & lmask) {
    const uint32_t v = L[p];
    if (v == EMPTY32) break;                            // cannot happen: dedup_kernel entered every valid record's key
    if (same_key(load_rec(b, v), r)) { hd = v; break; }
  }
  head[i] = hd;
  if (hd != i) return;
  const unsigned long long mine = ((unsigned long long)epoch << 32) | (r.h + 1);
  for (uint64_t s = home(t, r.h, r.x1);; s++) {
    if (s >= t.nslots) { atomicOr(&hdr->flags, FLAG_OVERFLOW); res[i] = RES_FAIL; return; }
    unsigned long long m = *(volatile unsigned long long*)&t.meta[s];
    if (m == 0) {
      m = atomicCAS(&t.meta[s], 0ULL, mine);
      if (m == 0) {
        t.ent[2 * s] = make_ulonglong2(r.x0, r.x1);
        t.ent[2 * s + 1] = make_ulonglong2(r.d0, r.d1);
        atomicAdd(t.count, 1ULL);
        res[i] = RES_NEW;
        return;
      }
    }
    if ((uint32_t)(m >> 32) != epoch && (uint32_t)m == r.h + 1) {
      const ulonglong2 x = t.ent[2 * s];
      if (x.x == r.x0 && x.y == r.x1) { res[i] = s; return; }
    }
  }
}

// 3. HashTable::Add's verdict for every record, in the form kgi_add reports it
__global__ void event_kernel(Batch b, uint32_t n, Table t, const uint32_t* head, const unsigned long long* res,
                             EvHeader* hdr, Event* ev, uint32_t cap) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t hd = head[i];
  if (hd == EMPTY32) return;
  const unsigned long long rs = res[hd];
  if (rs == RES_FAIL || (rs == RES_NEW && hd == i)) return;
  const Rec r = load_rec(b, i);
  uint64_t s0, s1;
  if (rs == RES_NEW) { const Rec f = load_rec(b, hd); s0 = f.d0; s1 = f.d1; }
  else { const ulonglong2 d = t.ent[2 * rs + 1]; s0 = d.x; s1 = d.y; }
  Event e;
  e.rank = r.rank; e.kidx = r.kidx; e.h = r.h;
  e.d_new[0] = r.d0; e.d_new[1] = r.d1;
  if (s0 == r.d0 && s1 == r.d1) {                       // ADD_DUPLICATE
    e.kind = 1; e.d_old[0] = 0; e.d_old[1] = 0;
  } else {                                              // ADD_COLLISION: same herd -> reset, else tame/wild
    e.kind = ((s1 ^ r.d1) & TYPE) ? 2 : 1;
    e.d_old[0] = s0; e.d_old[1] = s1;
  }
  const uint32_t k = atomicAdd(&hdr->count, 1u);
  if (k < cap) ev[k] = e;
}

__global__ void snapshot_count_kernel(const unsigned long long* count, EvHeader* hdr) { hdr->entries = *count; }

// bulk load of unique entries (resume): claim the first empty slot from home
__global__ void load_kernel(const uint32_t* h, const ulonglong2* e, uint64_t n, Table t, uint32_t epoch, EvHeader* hdr) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t hh = h[i];
  if (hh >= HASH_SIZE) { atomicOr(&hdr->flags, FLAG_BAD); return; }
  const ulonglong2 x = e[2 * i], d = e[2 * i + 1];
  const unsigned long long mine = ((unsigned long long)epoch << 32) | (hh + 1);
  for (uint64_t s = home(t, hh, x.y);; s++) {
    if (s >= t.nslots) { atomicOr(&hdr->flags, FLAG_OVERFLOW); return; }
    if (*(volatile unsigned long long*)&t.meta[s] == 0 && atomicCAS(&t.meta[s], 0ULL, mine) == 0) {
      t.ent[2 * s] = x; t.ent[2 * s + 1] = d;
      atomicAdd(t.count, 1ULL);
      return;
    }
  }
}

// Calls f(slot) for every slot of bucket h stored by an insert <= L: the bucket's home range, then its spill up to the
// first slot that was empty at L.  All threads of the block must call it.
template <typename F>
__device__ void scan_bucket(const Table& t, uint32_t h, uint32_t L, F f) {
  __shared__ unsigned long long stopAt;
  const uint64_t b0 = (uint64_t)h * t.S, b1 = b0 + t.S;
  auto mine = [&](unsigned long long m) { return m != 0 && (uint32_t)(m >> 32) <= L && (uint32_t)m == h + 1; };
  for (uint64_t s = b0 + threadIdx.x; s < b1; s += blockDim.x)
    if (mine(t.meta[s])) f(s);
  for (uint64_t w = b1;; w += blockDim.x) {
    if (threadIdx.x == 0) stopAt = ~0ULL;
    __syncthreads();
    const uint64_t s = w + threadIdx.x;
    unsigned long long m = 0;
    if (s >= t.nslots) atomicMin(&stopAt, (unsigned long long)s);
    else {
      m = t.meta[s];
      if (m == 0 || (uint32_t)(m >> 32) > L) atomicMin(&stopAt, (unsigned long long)s);
    }
    __syncthreads();
    const unsigned long long stop = stopAt;
    if (s < stop && mine(m)) f(s);
    __syncthreads();
    if (stop != ~0ULL) return;
  }
}

// entries of buckets [h0, h0 + nb) stored by inserts <= L -> counts[]
__global__ void export_count_kernel(Table t, uint32_t h0, uint32_t L, uint32_t* counts) {
  __shared__ uint32_t c;
  if (threadIdx.x == 0) c = 0;
  __syncthreads();
  scan_bucket(t, h0 + blockIdx.x, L, [&](uint64_t) { atomicAdd(&c, 1u); });
  __syncthreads();
  if (threadIdx.x == 0) counts[blockIdx.x] = c;
}

// bucket h0 + blockIdx.x sorted by (x[1], x[0]) into out[off[blockIdx.x] ...]; buckets over MAXB entries were refused
// by the caller from export_count_kernel's counts
__global__ void __launch_bounds__(SORT_THREADS) export_sort_kernel(Table t, uint32_t h0, uint32_t L, const unsigned long long* off,
                                                                   ulonglong2* out) {
  extern __shared__ unsigned long long sm[];
  unsigned long long* khi = sm;
  unsigned long long* klo = sm + MAXB;
  uint32_t* idx = reinterpret_cast<uint32_t*>(sm + 2 * MAXB);
  __shared__ uint32_t c;
  if (threadIdx.x == 0) c = 0;
  __syncthreads();
  scan_bucket(t, h0 + blockIdx.x, L, [&](uint64_t s) {
    const uint32_t k = atomicAdd(&c, 1u);
    if (k < MAXB) { const ulonglong2 x = t.ent[2 * s]; khi[k] = x.y; klo[k] = x.x; idx[k] = (uint32_t)s; }
  });
  __syncthreads();
  const uint32_t n = c;
  if (n == 0 || n > MAXB) return;
  uint32_t P = 1;
  while (P < n) P <<= 1;
  for (uint32_t k = n + threadIdx.x; k < P; k += blockDim.x) { khi[k] = ~0ULL; klo[k] = ~0ULL; idx[k] = EMPTY32; }
  __syncthreads();
  for (uint32_t size = 2; size <= P; size <<= 1) {         // bitonic sort on (x[1], x[0], slot)
    for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
      for (uint32_t j = threadIdx.x; j < P / 2; j += blockDim.x) {
        const uint32_t a = 2 * j - (j & (stride - 1)), bb = a + stride;
        const bool up = (a & size) == 0;
        const bool gt = khi[a] != khi[bb] ? khi[a] > khi[bb] : (klo[a] != klo[bb] ? klo[a] > klo[bb] : idx[a] > idx[bb]);
        if (gt == up) {
          unsigned long long t0 = khi[a]; khi[a] = khi[bb]; khi[bb] = t0;
          t0 = klo[a]; klo[a] = klo[bb]; klo[bb] = t0;
          const uint32_t t1 = idx[a]; idx[a] = idx[bb]; idx[bb] = t1;
        }
      }
      __syncthreads();
    }
  }
  const unsigned long long o = off[blockIdx.x];
  for (uint32_t k = threadIdx.x; k < n; k += blockDim.x) {
    const uint64_t s = idx[k];
    out[2 * (o + k)] = t.ent[2 * s];
    out[2 * (o + k) + 1] = t.ent[2 * s + 1];
  }
}

}  // namespace dpt
}  // namespace kgx
