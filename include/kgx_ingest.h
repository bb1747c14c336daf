/*
 * kgx_ingest.h -- C ABI of the rank-0 distinguished-point ingest (libkgx_ingest.so), SURVEY.md 8(f) row f1, host half.
 *
 * What it replaces: the body of the DP loop of Kangaroo::SolveKeyGPU (reference Kangaroo.cpp:594-612: under ghMutex,
 * per DP `AddToTable` -> HashTable::Add (HashTable.cpp:221-307) -> on ADD_COLLISION `CollisionCheck`), and the server-side
 * drain of Thread.cpp:165-234, for the in-box multi-GPU case where the DP records of ALL ranks arrive on rank 0 as one
 * buffer per step (NCCL gather, kangaroo_b200/dist.py).  The table keeps the semantics and the work-file layout of the
 * reference's `class HashTable`; records are inserted by a pool of worker threads sharded by bucket index (h mod threads)
 * -- buckets are independent, so no lock is needed -- instead of one thread under one mutex.
 *
 * Record format = the reference's wire/disk `DP` (Kangaroo.h:94-101), produced on the device by kgx_convert_dps():
 *   { uint32 kIdx; uint32 h; uint128 x (128 LSBs); uint128 d (b127 sign, b126 type, b125..0 |distance|) }   40 bytes.
 */
#ifndef KGX_INGEST_H
#define KGX_INGEST_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct kgi_table kgi_table;

#define KGI_EV_RESET     1   /* AddToTable returned false without ending the search (Kangaroo.cpp:600-609): duplicate point or
                                collision inside one herd -> the caller must re-create kangaroo (rank, kidx) */
#define KGI_EV_COLLISION 2   /* tame/wild collision: d_old / d_new are the two tagged 128-bit distances (HashTable.h:52-57) */

typedef struct {
  uint32_t kind;        /* KGI_EV_* */
  uint32_t rank;        /* rank tag passed to kgi_add for the NEW record */
  uint32_t kidx;        /* kIdx of the NEW record */
  uint32_t h;           /* bucket */
  uint64_t d_old[2];    /* stored entry (collision only) */
  uint64_t d_new[2];    /* new record */
} kgi_event;

/* threads <= 0: min(8, hardware concurrency).  NULL on failure. */
kgi_table* kgi_create(int threads);
void       kgi_destroy(kgi_table* t);
void       kgi_reset(kgi_table* t);                 /* HashTable::Reset */
uint64_t   kgi_count(kgi_table* t);                 /* HashTable::GetNbItem */
int        kgi_threads(kgi_table* t);

/* Insert n records (dp40: n x 40 bytes) tagged with `rank`.  One caller at a time per table (the workers are the parallelism).  Events (resets, collisions) are appended to ev[0..cap);
 * *n_ev = number of events produced (may exceed cap: the excess is dropped, resets are best-effort like the reference's).
 * Returns 0, or -1 on a malformed record (h >= 2^18). */
int kgi_add(kgi_table* t, const void* dp40, uint32_t n, uint32_t rank, kgi_event* ev, uint32_t cap, uint32_t* n_ev);

/* Same for the engine's raw 56-byte ITEMs (kgx_item: x[4], biased d[2], kidx): HashTable::Convert is applied on the host
 * exactly like Kangaroo::AddToTable(Int*,Int*,type) does (wild_offset = the engine's bias, 2 limbs, removed mod n). */
int kgi_add_items(kgi_table* t, const void* items56, uint32_t n, uint32_t rank, const uint64_t wild_offset[2],
                  kgi_event* ev, uint32_t cap, uint32_t* n_ev);

/* Kangaroo::CollisionCheck + CheckKey (Kangaroo.cpp:218-302): given the two tagged
 * distances of a KGI_EV_COLLISION, the search key (keyToSearch = P - start*G, 4+4 limbs) and range start (4 limbs), writes
 * the private key (4 limbs) and returns 1 when one of the four sign combinations matches +-key, else 0. */
int kgi_resolve(kgi_table* t, const uint64_t d_old[2], const uint64_t d_new[2], const uint64_t keyx[4], const uint64_t keyy[4],
                const uint64_t range_start[4], uint64_t priv_out[4]);

/* Work-file compatibility (SURVEY 8f/f3): write the table as a reference work file (Backup.cpp:368-394 header HEADW +
 * HashTable::SaveTable) that the reference's -winfo / -wcheck / -i / -wm read.  range_start/range_end/key: 4 limbs each. */
int kgi_save_work(kgi_table* t, const char* path, uint32_t dp_bits, const uint64_t range_start[4], const uint64_t range_end[4],
                  const uint64_t keyx[4], const uint64_t keyy[4], uint64_t total_count, double total_time);
/* Load the DP table of a reference work file (HEADW) into t; fills dp_bits / count / time when non-NULL.  0 on success. */
int kgi_load_work(kgi_table* t, const char* path, uint32_t* dp_bits, uint64_t* total_count, double* total_time);

#ifdef __cplusplus
}
#endif
#endif
