// kgx_ingest.cpp -- rank-0 distinguished-point table and its batched ingest (C ABI: include/kgx_ingest.h;
// SURVEY.md 8f row f1, host half).
//
// The table keeps the reference's semantics and on-disk layout (HashTable.{h,cpp}) so that work files stay interchangeable
// with the reference program: 2^18 buckets indexed by bits 128..145 of x, each an array of {x: 128 LSBs, d: tagged 128-bit
// distance} sorted by x; inserting an x that is already stored is ADD_DUPLICATE when d is equal too, else ADD_COLLISION.
// The bucket capacity the reference would have allocated (16 on first use, +4 when nearly full) is tracked because work
// files record it.  The code is this project's own; tests/test_ingest_cpu.py pins it to golden data written by the
// reference's HashTable.
//
// Reference path being replaced: Kangaroo::SolveKeyGPU's DP loop, Kangaroo.cpp:594-612 --
//   LOCK(ghMutex); for every DP: AddToTable(x, d, type) -> HashTable::Add -> [ADD_COLLISION] CollisionCheck -> CheckKey x4
// one thread, one mutex, one malloc per entry.  Here the records of all GPUs arrive as one 40-byte-record buffer per step
// (already converted on the device, kgx_convert_dps) and are inserted by a pool of workers sharded by bucket
// (h mod workers): an insert touches only its own bucket, so shards never share one and no lock is taken.
#include <algorithm>
#include <condition_variable>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <thread>
#include <vector>
#include "../../include/kgx_ingest.h"

#define HEADW_MAGIC 0xFA6A8001u      // Kangaroo.h:120

namespace {

const uint32_t HASH_SIZE = 1u << 18;                 // HashTable.h: HASH_SIZE_BIT 18
const uint64_t SIGN = 0x8000000000000000ULL, TYPE = 0x4000000000000000ULL, DIST_MASK = 0x3FFFFFFFFFFFFFFFULL;
enum { ADD_OK, ADD_DUPLICATE, ADD_COLLISION };

struct DP40 { uint32_t kidx, h; uint64_t x[2], d[2]; };   // Kangaroo.h:94-101
static_assert(sizeof(DP40) == 40, "DP record must be 40 bytes");

struct Entry { uint64_t x[2], d[2]; };                     // HashTable.h ENTRY: 32 bytes on disk
static_assert(sizeof(Entry) == 32, "table entry must be 32 bytes");

struct Bucket {
  std::vector<Entry> items;                                // sorted by (x[1], x[0])
  uint32_t cap = 0;                                        // the reference's maxItem, written to work files
};

struct Job {
  const DP40* recs = nullptr;
  uint32_t n = 0, rank = 0;
};

inline bool x_less(const Entry& e, const uint64_t x[2]) {
  return e.x[1] != x[1] ? e.x[1] < x[1] : e.x[0] < x[0];
}

// HashTable::Add semantics; on ADD_COLLISION *hit is the stored entry with the same x
int bucket_add(Bucket& b, const Entry& e, const Entry** hit) {
  if (b.cap == 0) b.cap = 16;
  if (b.items.empty()) { b.items.push_back(e); return ADD_OK; }
  if (b.items.size() >= b.cap - 1) b.cap += 4;
  auto it = std::lower_bound(b.items.begin(), b.items.end(), e.x, x_less);
  if (it != b.items.end() && it->x[0] == e.x[0] && it->x[1] == e.x[1]) {
    if (it->d[0] == e.d[0] && it->d[1] == e.d[1]) return ADD_DUPLICATE;   // same point twice or same-herd collision
    *hit = &*it;
    return ADD_COLLISION;
  }
  b.items.insert(it, e);
  return ADD_OK;
}

// --- secp256k1 for Kangaroo::CheckKey: 4 x 64-bit little-endian limbs ---------------------------------------
typedef unsigned __int128 u128;
struct U256 { uint64_t v[4]; };
const U256 FP = {{0xFFFFFFFEFFFFFC2FULL, ~0ULL, ~0ULL, ~0ULL}};
const U256 FN = {{0xBFD25E8CD0364141ULL, 0xBAAEDCE6AF48A03BULL, 0xFFFFFFFFFFFFFFFEULL, ~0ULL}};
const U256 GX = {{0x59F2815B16F81798ULL, 0x029BFCDB2DCE28D9ULL, 0x55A06295CE870B07ULL, 0x79BE667EF9DCBBACULL}};
const U256 GY = {{0x9C47D08FFB10D4B8ULL, 0xFD17B448A6855419ULL, 0x5DA4FBFC0E1108A8ULL, 0x483ADA7726A3C465ULL}};

bool is_zero(const U256& a) { return (a.v[0] | a.v[1] | a.v[2] | a.v[3]) == 0; }
bool eq(const U256& a, const U256& b) { return memcmp(a.v, b.v, sizeof a.v) == 0; }
bool geq(const U256& a, const U256& b) {
  for (int i = 3; i >= 0; i--)
    if (a.v[i] != b.v[i]) return a.v[i] > b.v[i];
  return true;
}
uint64_t add_c(U256& r, const U256& a, const U256& b) {
  u128 c = 0;
  for (int i = 0; i < 4; i++) { c += (u128)a.v[i] + b.v[i]; r.v[i] = (uint64_t)c; c >>= 64; }
  return (uint64_t)c;
}
uint64_t sub_b(U256& r, const U256& a, const U256& b) {
  uint64_t br = 0;
  for (int i = 0; i < 4; i++) {
    const u128 t = (u128)a.v[i] - b.v[i] - br;
    r.v[i] = (uint64_t)t;
    br = (uint64_t)(t >> 64) & 1;
  }
  return br;
}
// (a + b) mod m, (a - b) mod m for a, b < m
U256 add_mod(const U256& a, const U256& b, const U256& m) {
  U256 r, s;
  const uint64_t c = add_c(r, a, b);
  if (c || geq(r, m)) { sub_b(s, r, m); return s; }
  return r;
}
U256 sub_mod(const U256& a, const U256& b, const U256& m) {
  U256 r, s;
  if (sub_b(r, a, b)) { add_c(s, r, m); return s; }
  return r;
}
U256 neg_mod(const U256& a, const U256& m) { return is_zero(a) ? a : sub_mod(m, a, m); }

U256 fmul(const U256& a, const U256& b) {                  // mod p = 2^256 - 0x1000003D1
  uint64_t w[8] = {0};
  for (int i = 0; i < 4; i++) {
    u128 c = 0;
    for (int j = 0; j < 4; j++) { c += (u128)a.v[i] * b.v[j] + w[i + j]; w[i + j] = (uint64_t)c; c >>= 64; }
    w[i + 4] = (uint64_t)c;
  }
  const uint64_t K = 0x1000003D1ULL;
  U256 r;
  u128 c = 0;
  for (int i = 0; i < 4; i++) { c += (u128)w[i + 4] * K + w[i]; r.v[i] = (uint64_t)c; c >>= 64; }
  uint64_t top = (uint64_t)c;                               // < 2^34: fold once more
  while (top) {
    c = (u128)top * K;
    for (int i = 0; i < 4; i++) { c += r.v[i]; r.v[i] = (uint64_t)c; c >>= 64; }
    top = (uint64_t)c;
  }
  if (geq(r, FP)) { U256 s; sub_b(s, r, FP); r = s; }
  return r;
}
U256 finv(const U256& a) {                                 // a^(p-2)
  U256 e = FP, r = {{1, 0, 0, 0}}, base = a;
  e.v[0] -= 2;
  for (int i = 0; i < 256; i++) {
    if ((e.v[i / 64] >> (i % 64)) & 1) r = fmul(r, base);
    base = fmul(base, base);
  }
  return r;
}

struct Pt { U256 x, y; bool inf; };
Pt pt_add(const Pt& a, const Pt& b) {                      // affine
  if (a.inf) return b;
  if (b.inf) return a;
  U256 s;
  if (eq(a.x, b.x)) {
    if (is_zero(add_mod(a.y, b.y, FP))) return Pt{{{0}}, {{0}}, true};
    const U256 x2 = fmul(a.x, a.x);
    s = fmul(add_mod(add_mod(x2, x2, FP), x2, FP), finv(add_mod(a.y, a.y, FP)));
  } else {
    s = fmul(sub_mod(b.y, a.y, FP), finv(sub_mod(b.x, a.x, FP)));
  }
  Pt r;
  r.inf = false;
  r.x = sub_mod(sub_mod(fmul(s, s), a.x, FP), b.x, FP);
  r.y = sub_mod(fmul(s, sub_mod(a.x, r.x, FP)), a.y, FP);
  return r;
}
Pt mul_g(const U256& k) {
  Pt acc{{{0}}, {{0}}, true}, p{GX, GY, false};
  for (int i = 0; i < 256; i++) {
    if ((k.v[i / 64] >> (i % 64)) & 1) acc = pt_add(acc, p);
    p = pt_add(p, p);
  }
  return acc;
}

// HashTable::CalcDistAndType: b126 = herd, b127 = sign of the 126-bit distance -> distance mod n
U256 tagged_dist(const uint64_t d[2], uint32_t* type) {
  *type = (d[1] & TYPE) != 0;
  const U256 v = {{d[0], d[1] & DIST_MASK, 0, 0}};
  return (d[1] & SIGN) ? neg_mod(v, FN) : v;
}

}  // namespace

struct kgi_table {
  std::vector<Bucket> buckets = std::vector<Bucket>(HASH_SIZE);
  int nthreads = 1;
  std::vector<std::thread> workers;
  std::vector<std::vector<kgi_event>> evs;
  std::mutex mu;
  std::condition_variable cvStart, cvDone;
  uint64_t generation = 0;
  int pending = 0;
  bool quit = false, bad = false;
  Job job;
};

// Kangaroo::AddToTable(h, x, d) (Kangaroo.cpp:315-330) for one record, on the shard that owns bucket h
static void add_one(kgi_table* t, const DP40& r, uint32_t rank, std::vector<kgi_event>& out) {
  Entry e;
  memcpy(e.x, r.x, sizeof e.x);
  memcpy(e.d, r.d, sizeof e.d);
  const Entry* old = nullptr;
  const int st = bucket_add(t->buckets[r.h], e, &old);
  if (st == ADD_OK) return;
  kgi_event ev;
  memset(&ev, 0, sizeof ev);
  ev.rank = rank; ev.kidx = r.kidx; ev.h = r.h;
  ev.d_new[0] = r.d[0]; ev.d_new[1] = r.d[1];
  if (st == ADD_DUPLICATE) { ev.kind = KGI_EV_RESET; out.push_back(ev); return; }
  ev.d_old[0] = old->d[0]; ev.d_old[1] = old->d[1];
  ev.kind = ((old->d[1] ^ r.d[1]) & TYPE) ? KGI_EV_COLLISION : KGI_EV_RESET;   // same herd -> reset (Kangaroo.cpp:258-262)
  out.push_back(ev);
}

static void worker_main(kgi_table* t, int id) {
  uint64_t seen = 0;
  for (;;) {
    Job job;
    {
      std::unique_lock<std::mutex> lk(t->mu);
      t->cvStart.wait(lk, [&] { return t->quit || t->generation != seen; });
      if (t->quit) return;
      seen = t->generation;
      job = t->job;
    }
    std::vector<kgi_event>& out = t->evs[id];
    const uint32_t T = (uint32_t)t->nthreads;
    bool bad = false;
    for (uint32_t i = 0; i < job.n; i++) {
      const DP40& r = job.recs[i];
      if (r.h >= HASH_SIZE) { bad = true; continue; }
      if (r.h % T != (uint32_t)id) continue;
      add_one(t, r, job.rank, out);
    }
    {
      std::lock_guard<std::mutex> lk(t->mu);
      if (bad) t->bad = true;
      if (--t->pending == 0) t->cvDone.notify_all();
    }
  }
}

static void table_reset(kgi_table* t) {
  for (Bucket& b : t->buckets) { std::vector<Entry>().swap(b.items); b.cap = 0; }
}

extern "C" {

kgi_table* kgi_create(int threads) {
  kgi_table* t = new kgi_table();
  if (threads <= 0) {
    unsigned hc = std::thread::hardware_concurrency();
    threads = hc == 0 ? 1 : (hc > 8 ? 8 : (int)hc);
  }
  if (threads > 64) threads = 64;
  t->nthreads = threads;
  t->evs.resize(threads);
  for (int i = 0; i < threads; i++) t->workers.emplace_back(worker_main, t, i);
  return t;
}

void kgi_destroy(kgi_table* t) {
  if (!t) return;
  {
    std::lock_guard<std::mutex> lk(t->mu);
    t->quit = true;
  }
  t->cvStart.notify_all();
  for (auto& w : t->workers) w.join();
  delete t;
}

void kgi_reset(kgi_table* t) { table_reset(t); }

uint64_t kgi_count(kgi_table* t) {
  uint64_t n = 0;
  for (const Bucket& b : t->buckets) n += b.items.size();
  return n;
}

int kgi_threads(kgi_table* t) { return t->nthreads; }

int kgi_add(kgi_table* t, const void* dp40, uint32_t n, uint32_t rank, kgi_event* ev, uint32_t cap, uint32_t* n_ev) {
  *n_ev = 0;
  if (n == 0) return 0;
  {
    std::lock_guard<std::mutex> lk(t->mu);
    t->job.recs = static_cast<const DP40*>(dp40);
    t->job.n = n; t->job.rank = rank;
    t->pending = t->nthreads;
    t->bad = false;
    for (auto& v : t->evs) v.clear();
    t->generation++;
  }
  t->cvStart.notify_all();
  {
    std::unique_lock<std::mutex> lk(t->mu);
    t->cvDone.wait(lk, [&] { return t->pending == 0; });
  }
  uint32_t k = 0;
  for (auto& v : t->evs)
    for (auto& e : v) { if (k < cap) ev[k] = e; k++; }
  *n_ev = k;
  return t->bad ? -1 : 0;
}

int kgi_add_items(kgi_table* t, const void* items56, uint32_t n, uint32_t rank, const uint64_t wild_offset[2],
                  kgi_event* ev, uint32_t cap, uint32_t* n_ev) {
  // GPUEngine::Launch's un-biasing (GPUEngine.cu:653-675) + HashTable::Convert (HashTable.cpp:75-100).  Both the biased
  // distance and the offset are below 2^128, so d - offset (mod n) is either that 128-bit difference or n minus
  // (offset - d): Convert stores the magnitude with the sign bit, no 256-bit arithmetic needed.
  struct Item56 { uint64_t x[4], d[2], kidx; };
  const Item56* it = static_cast<const Item56*>(items56);
  std::vector<DP40> recs(n);
  const u128 wo = ((u128)wild_offset[1] << 64) | wild_offset[0];
  for (uint32_t i = 0; i < n; i++) {
    const uint64_t type = it[i].kidx & 1;
    u128 d = ((u128)it[i].d[1] << 64) | it[i].d[0];
    uint64_t sign = 0;
    if (type) {
      if (d >= wo) d -= wo;
      else { d = wo - d; sign = SIGN; }
    }
    DP40& r = recs[i];
    r.kidx = (uint32_t)it[i].kidx;
    r.h = (uint32_t)(it[i].x[2] & (HASH_SIZE - 1));
    r.x[0] = it[i].x[0]; r.x[1] = it[i].x[1];
    r.d[0] = (uint64_t)d;
    r.d[1] = ((uint64_t)(d >> 64) & DIST_MASK) | sign | (type << 62);
  }
  return kgi_add(t, recs.data(), n, rank, ev, cap, n_ev);
}

int kgi_resolve(kgi_table* t, const uint64_t d_old[2], const uint64_t d_new[2], const uint64_t keyx[4], const uint64_t keyy[4],
                const uint64_t range_start[4], uint64_t priv_out[4]) {
  (void)t;
  uint32_t ta, tb;
  const U256 da = tagged_dist(d_old, &ta), db = tagged_dist(d_new, &tb);
  if (ta == tb) return 0;                                        // Kangaroo.cpp:258-262
  const U256 Td = ta == 0 ? da : db, Wd = ta == 0 ? db : da;
  U256 kx, ky, start;
  memcpy(kx.v, keyx, 32); memcpy(ky.v, keyy, 32); memcpy(start.v, range_start, 32);
  const U256 kyNeg = neg_mod(ky, FP);
  for (int type = 0; type < 4; type++) {                          // Kangaroo::CheckKey, Kangaroo.cpp:218-253
    const U256 d1 = (type & 1) ? neg_mod(Td, FN) : Td;
    const U256 d2 = (type & 2) ? neg_mod(Wd, FN) : Wd;
    U256 pk = add_mod(d1, d2, FN);
    const Pt P = mul_g(pk);
    if (P.inf || !eq(P.x, kx)) continue;
    if (!eq(P.y, ky)) {                                           // -key: the symmetric hit
      if (!eq(P.y, kyNeg)) continue;
      pk = neg_mod(pk, FN);
    }
    pk = add_mod(pk, start, FN);
    memcpy(priv_out, pk.v, 32);
    return 1;
  }
  return 0;
}

int kgi_save_work(kgi_table* t, const char* path, uint32_t dp_bits, const uint64_t range_start[4], const uint64_t range_end[4],
                  const uint64_t keyx[4], const uint64_t keyy[4], uint64_t total_count, double total_time) {
  FILE* f = fopen(path, "wb");
  if (!f) return -1;
  // Kangaroo::SaveHeader (Backup.cpp:368-394), type HEADW, then HashTable::SaveTable (HashTable.cpp:375-396)
  const uint32_t head = HEADW_MAGIC, version = 0;
  bool ok = fwrite(&head, 4, 1, f) == 1 && fwrite(&version, 4, 1, f) == 1 && fwrite(&dp_bits, 4, 1, f) == 1;
  ok = ok && fwrite(range_start, 32, 1, f) == 1 && fwrite(range_end, 32, 1, f) == 1;
  ok = ok && fwrite(keyx, 32, 1, f) == 1 && fwrite(keyy, 32, 1, f) == 1;
  ok = ok && fwrite(&total_count, 8, 1, f) == 1 && fwrite(&total_time, 8, 1, f) == 1;
  for (uint32_t h = 0; ok && h < HASH_SIZE; h++) {
    const Bucket& b = t->buckets[h];
    const uint32_t nb = (uint32_t)b.items.size();
    ok = fwrite(&nb, 4, 1, f) == 1 && fwrite(&b.cap, 4, 1, f) == 1 && fwrite(b.items.data(), sizeof(Entry), nb, f) == nb;
  }
  const uint64_t totalWalk = 0;                                   // no kangaroos in this file (Backup.cpp:549-551)
  ok = ok && fwrite(&totalWalk, 8, 1, f) == 1;
  return (fclose(f) == 0 && ok) ? 0 : -1;
}

int kgi_load_work(kgi_table* t, const char* path, uint32_t* dp_bits, uint64_t* total_count, double* total_time) {
  FILE* f = fopen(path, "rb");
  if (!f) return -1;
  uint32_t head = 0, version = 0, dp = 0;
  uint64_t skip[16], cnt = 0; double tm = 0;
  bool ok = fread(&head, 4, 1, f) == 1 && fread(&version, 4, 1, f) == 1 && head == HEADW_MAGIC;
  ok = ok && fread(&dp, 4, 1, f) == 1 && fread(skip, 32, 4, f) == 4 && fread(&cnt, 8, 1, f) == 1 && fread(&tm, 8, 1, f) == 1;
  table_reset(t);
  for (uint32_t h = 0; ok && h < HASH_SIZE; h++) {
    Bucket& b = t->buckets[h];
    uint32_t nb = 0;
    ok = fread(&nb, 4, 1, f) == 1 && fread(&b.cap, 4, 1, f) == 1;
    if (ok) {
      b.items.resize(nb);
      ok = fread(b.items.data(), sizeof(Entry), nb, f) == nb;
    }
  }
  fclose(f);
  if (!ok) { table_reset(t); return -1; }
  if (dp_bits) *dp_bits = dp;
  if (total_count) *total_count = cnt;
  if (total_time) *total_time = tm;
  return 0;
}

}  // extern "C"
