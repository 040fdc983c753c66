// placer.cu — read_placer scoring on the device cloud CSR (SURVEY.md §8f rank 2).
//
// Replaces, for scripts/read_placer.py:42-94 (ReadPlacer.add_reads) and scripts/cloud_contig.py:26-41,87-95
// (CloudContig.add_read, update_mapping_scores), the three data structures the greedy loop lives on:
//
//   cloud contig   clouds[pos][kmer] counters (cloud_contig.py:14, :33-35)  ->  open-addressing table keyed by
//                  (contig position << 32 | k-mer id); a k-mer id becomes "frequent" (freq_kmers, :36-38) when one
//                  of its positions reaches min_cloud_kmer_freq, and that (k-mer, position) pair is handed back
//                  exactly once (new_freq_kmers, :39)
//   kmers2pos      (read_placer.py:44-49)  ->  the inverted cloud CSR the recruitment path already builds
//                  (occ_ptr / occ: for every k-mer id the sorted units holding it) + unit -> (read, position in read)
//   scores         scores[r_id][contig position - position in read][position in read] += 1 (cloud_contig.py:90-94)
//                  -> a SET of (read, offset, position) triples and a table (read, offset) -> (distinct positions,
//                  total), which is all the selection rule reads: (len(score), sum(score.values())), read_placer.py:66-67
//
// The greedy loop itself (one read placed per iteration, read_placer.py:58-94) stays on the host: per iteration it
// launches update -> best, reads one small result back, picks the winner and launches add_read.
#include "cfk_common.cuh"

namespace {

using namespace cfk;

// The score tables of placer_update_kernel report a full table through counters[1], and the host repeats the call
// with 4x larger ones.  One thread walks every occurrence of its pair's k-mer serially, so a full table must not cost
// it a scan of the whole table per occurrence: probing there stops after PL_MAX_PROBES slots, which reports the table
// as full (a repeat with larger tables gives the same scores), and a thread stops once any thread reported it.
constexpr int64_t PL_MAX_PROBES = 1 << 12;

__device__ __forceinline__ int64_t pl_upsert(uint64_t* keys, int64_t cap, uint64_t key, int64_t max_probes) {
  int64_t slot = home_slot(mix64(key), cap);
  for (int64_t probes = 0; probes < max_probes; ++probes) {
    const uint64_t cur = ((volatile uint64_t*)keys)[slot];
    if (cur == key) return slot;
    if (cur == EMPTY) {
      const unsigned long long old = atomicCAS((unsigned long long*)(keys + slot), (unsigned long long)EMPTY,
                                               (unsigned long long)key);
      if (old == EMPTY || old == key) return slot;
    }
    if (++slot == cap) slot = 0;
  }
  return -1;
}

// CloudContig.add_read (cloud_contig.py:26-41) for one read: its units u0 .. u0 + n_units - 1 land on contig positions
// position .. ; thread per cloud entry.  counters[0] = pairs appended, counters[1] != 0: a table is full.
__global__ void placer_add_read_kernel(const int64_t* __restrict__ unit_ptr, const uint32_t* __restrict__ ids, int64_t u0,
                                       int32_t n_units, int64_t position, uint32_t min_freq, uint64_t* contig_keys,
                                       uint32_t* contig_cnt, int64_t cap, uint8_t* freq_flag, uint2* pairs, int64_t max_pairs,
                                       int64_t* counters) {
  const int64_t e0 = unit_ptr[u0], e1 = unit_ptr[u0 + n_units];
  const int64_t e = e0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= e1) return;
  int lo = 0, hi = n_units;  // unit_ptr[u0 + lo] <= e < unit_ptr[u0 + hi]
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (unit_ptr[u0 + mid] > e) hi = mid; else lo = mid;
  }
  const uint32_t id = ids[e];
  const uint64_t p = (uint64_t)(position + lo);
  const int64_t slot = pl_upsert(contig_keys, cap, (p << 32) | id, cap);
  if (slot < 0) {
    counters[1] = 1;
    return;
  }
  if (atomicAdd(contig_cnt + slot, 1u) + 1u == min_freq) {  // this (k-mer, position) just became frequent
    freq_flag[id] = 1;
    if (pairs == nullptr) return;  // prefix reads (read_placer.py:35-40): nobody looks at the returned list
    const int64_t at = (int64_t)atomicAdd((unsigned long long*)counters, 1ull);
    if (at < max_pairs) pairs[at] = make_uint2(id, (uint32_t)p);
    else counters[1] = 1;
  }
}

// The list add_reads starts from (read_placer.py:54-57): every position of every frequent k-mer -- frequent at SOME
// position, listed at ALL its positions (kmer_positions holds every position the k-mer was added at).
__global__ void placer_initial_pairs_kernel(const uint64_t* __restrict__ contig_keys, int64_t cap,
                                            const uint8_t* __restrict__ freq_flag, uint2* pairs, int64_t max_pairs,
                                            int64_t* counters) {
  for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < cap; s += (int64_t)gridDim.x * blockDim.x) {
    const uint64_t key = contig_keys[s];
    if (key == EMPTY) continue;
    const uint32_t id = (uint32_t)key;
    if (!freq_flag[id]) continue;
    const int64_t at = (int64_t)atomicAdd((unsigned long long*)counters, 1ull);
    if (at < max_pairs) pairs[at] = make_uint2(id, (uint32_t)(key >> 32));
    else counters[1] = 1;
  }
}

// update_mapping_scores (cloud_contig.py:87-95): for every (k-mer, contig position) of the list and every occurrence
// (read, position in read) of the k-mer among the reads being placed with contig position >= position in read.
// Thread per pair (n_pairs is read on the device: the host never waits for it).
__global__ void placer_update_kernel(const uint2* __restrict__ pairs, const int64_t* __restrict__ counters_pairs,
                                     int64_t max_pairs, const int64_t* __restrict__ occ_ptr, const uint32_t* __restrict__ occ,
                                     const int32_t* __restrict__ unit_read, const int64_t* __restrict__ read_first_unit,
                                     const uint8_t* __restrict__ read_sel, uint64_t* m1_keys, int64_t cap1,
                                     uint64_t* m2_keys, unsigned long long* m2_val, int64_t cap2, int64_t* counters) {
  const int64_t n_pairs = min(counters_pairs[0], max_pairs);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_pairs; i += (int64_t)gridDim.x * blockDim.x) {
    const uint2 pr = pairs[i];
    const int64_t cc_pos = pr.y;
    for (int64_t o = occ_ptr[pr.x]; o < occ_ptr[pr.x + 1]; ++o) {
      if (((volatile int64_t*)counters)[1]) return;  // a table is full: the host discards this call's scores
      const int64_t g = occ[o];
      const int64_t r = unit_read[g];
      if (!read_sel[r]) continue;
      const int64_t pos = g - read_first_unit[r];
      if (cc_pos < pos) continue;
      const uint64_t off = (uint64_t)(cc_pos - pos);  // < 2^32: contig positions are (checked in cfk_placer_add_read)
      // (read, offset) first: read < 2^24 (checked on the host), so the key is exact
      const int64_t s2 = pl_upsert(m2_keys, cap2, ((uint64_t)r << 32) | off, min(cap2, PL_MAX_PROBES));
      if (s2 < 0) {
        counters[1] = 1;
        continue;
      }
      // set of (read, offset, position), keyed by the (read, offset) slot, which never moves within a call:
      // slot < cap2 < 2^48, position < 2^16 (checked on the host), so the key is exact for any offset
      const uint64_t k1 = ((uint64_t)s2 << 16) | (uint64_t)pos;
      int64_t slot = home_slot(mix64(k1), cap1);
      bool fresh = false, placed = false;
      for (int64_t probes = 0, max_probes = min(cap1, PL_MAX_PROBES); probes < max_probes && !placed; ++probes) {
        const uint64_t cur = ((volatile uint64_t*)m1_keys)[slot];
        if (cur == k1) placed = true;
        else if (cur == EMPTY) {
          const unsigned long long old = atomicCAS((unsigned long long*)(m1_keys + slot), (unsigned long long)EMPTY,
                                                   (unsigned long long)k1);
          if (old == EMPTY) fresh = placed = true;
          else if (old == k1) placed = true;
        }
        if (!placed && ++slot == cap1) slot = 0;
      }
      if (!placed) {
        counters[1] = 1;
        continue;
      }
      atomicAdd(m2_val + s2, (fresh ? (1ull << 32) : 0ull) + 1ull);  // (distinct positions << 32) | total
    }
  }
}

// The selection of read_placer.py:61-79 over all (read, offset) scores: among the unused reads, the largest
// (distinct positions, total) that passes the three thresholds, then the largest offset, then the smallest read id
// (rank in sorted order).  One candidate per block goes to the host, which finishes the reduction.
struct PlBest {
  unsigned long long score;  // distinct positions << 32 | total; 0 = none
  uint32_t off;
  uint32_t rank;             // rank of the read id in sorted order: smaller wins
  uint32_t read;
  uint32_t pad;
};

__device__ __forceinline__ bool pl_better(const PlBest& a, const PlBest& b) {  // a beats b
  if (a.score != b.score) return a.score > b.score;
  if (a.off != b.off) return a.off > b.off;
  return a.rank < b.rank;
}

__global__ void __launch_bounds__(256) placer_best_kernel(const uint64_t* __restrict__ m2_keys,
                                                          const unsigned long long* __restrict__ m2_val, int64_t cap2,
                                                          const uint8_t* __restrict__ read_unused,
                                                          const uint32_t* __restrict__ read_rank, uint32_t min_unit,
                                                          uint32_t min_inters, uint32_t min_prop, PlBest* out) {
  __shared__ PlBest s_best[256];
  PlBest best{0ull, 0u, 0xFFFFFFFFu, 0u, 0u};
  for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < cap2; s += (int64_t)gridDim.x * blockDim.x) {
    const uint64_t key = m2_keys[s];
    if (key == EMPTY) continue;
    const uint32_t r = (uint32_t)(key >> 32);
    if (!read_unused[r]) continue;
    const unsigned long long v = m2_val[s];
    const uint64_t n_units = v >> 32, total = v & 0xFFFFFFFFull;
    if (n_units < min_unit || n_units * min_prop > total || total < min_inters) continue;
    const PlBest cand{v, (uint32_t)key, read_rank[r], r, 0u};
    if (pl_better(cand, best)) best = cand;
  }
  s_best[threadIdx.x] = best;
  __syncthreads();
  for (int h = 128; h >= 1; h >>= 1) {
    if ((int)threadIdx.x < h && pl_better(s_best[threadIdx.x + h], s_best[threadIdx.x])) s_best[threadIdx.x] = s_best[threadIdx.x + h];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[blockIdx.x] = s_best[0];
}

}  // namespace

extern "C" {

int cfk_placer_best_blocks(void) { return 296; }

int cfk_placer_add_read(const int64_t* unit_ptr, const uint32_t* ids, int64_t u0, int32_t n_units, int64_t n_entries_max,
                        int64_t position, uint32_t min_freq, uint64_t* contig_keys, uint32_t* contig_cnt, int64_t cap,
                        uint8_t* freq_flag, uint32_t* pairs, int64_t max_pairs, int64_t* counters, cfk_stream_t stream) {
  if (n_units < 0 || cap < 1 || max_pairs < 0 || position < 0 || n_entries_max < 0 || position + n_units >= (1ll << 32))
    return fail(CFK_ERR_INVALID, "cfk_placer_add_read: bad sizes");
  if (n_units == 0 || n_entries_max == 0) return CFK_OK;
  placer_add_read_kernel<<<(unsigned)blocks_for(n_entries_max, 256), 256, 0, (cudaStream_t)stream>>>(
      unit_ptr, ids, u0, n_units, position, min_freq, contig_keys, contig_cnt, cap, freq_flag, (uint2*)pairs, max_pairs, counters);
  CFK_CHECK_LAUNCH("placer_add_read_kernel", 1);
  return CFK_OK;
}

int cfk_placer_initial_pairs(const uint64_t* contig_keys, int64_t cap, const uint8_t* freq_flag, uint32_t* pairs,
                             int64_t max_pairs, int64_t* counters, cfk_stream_t stream) {
  if (cap < 1 || max_pairs < 0) return fail(CFK_ERR_INVALID, "cfk_placer_initial_pairs: bad sizes");
  const int64_t grid = blocks_for(cap, 256) < 148 * 8 ? blocks_for(cap, 256) : 148 * 8;
  placer_initial_pairs_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(contig_keys, cap, freq_flag, (uint2*)pairs,
                                                                            max_pairs, counters);
  CFK_CHECK_LAUNCH("placer_initial_pairs_kernel", 1);
  return CFK_OK;
}

int cfk_placer_update(const uint32_t* pairs, const int64_t* pair_counters, int64_t max_pairs, const int64_t* occ_ptr,
                      const uint32_t* occ, const int32_t* unit_read, const int64_t* read_first_unit, const uint8_t* read_sel,
                      uint64_t* m1_keys, int64_t cap1, uint64_t* m2_keys, uint64_t* m2_val, int64_t cap2, int64_t* counters,
                      cfk_stream_t stream) {
  if (cap1 < 1 || cap2 < 1 || cap2 >= (1ll << 48) || max_pairs < 0) return fail(CFK_ERR_INVALID, "cfk_placer_update: bad sizes");
  if (max_pairs == 0) return CFK_OK;
  const int64_t grid = blocks_for(max_pairs, 128) < 148 * 16 ? blocks_for(max_pairs, 128) : 148 * 16;
  placer_update_kernel<<<(unsigned)grid, 128, 0, (cudaStream_t)stream>>>((const uint2*)pairs, pair_counters, max_pairs, occ_ptr,
                                                                     occ, unit_read, read_first_unit, read_sel, m1_keys, cap1,
                                                                     m2_keys, (unsigned long long*)m2_val, cap2, counters);
  CFK_CHECK_LAUNCH("placer_update_kernel", 1);
  return CFK_OK;
}

int cfk_placer_best(const uint64_t* m2_keys, const uint64_t* m2_val, int64_t cap2, const uint8_t* read_unused,
                    const uint32_t* read_rank, uint32_t min_unit, uint32_t min_inters, uint32_t min_prop, uint64_t* out,
                    cfk_stream_t stream) {
  if (cap2 < 1) return fail(CFK_ERR_INVALID, "cfk_placer_best: bad sizes");
  static_assert(sizeof(PlBest) == 24, "three 64-bit words per block result");
  placer_best_kernel<<<296, 256, 0, (cudaStream_t)stream>>>(m2_keys, (const unsigned long long*)m2_val, cap2, read_unused,
                                                           read_rank, min_unit, min_inters, min_prop, (PlBest*)out);
  CFK_CHECK_LAUNCH("placer_best_kernel", 1);
  return CFK_OK;
}

}  // extern "C"
