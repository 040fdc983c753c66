// rr_filter.cu — the read recruitment pre-filter (SURVEY.md §8f rank 4, second half).
//
// Replaces the two edlibAlign calls of scripts/read_recruitment/rr.cpp:73-90: a read is kept when the unit, or its
// reverse complement, occurs somewhere in the read within `threshold` edits (edlib's HW mode: the whole unit against
// any infix of the read, EDLIB_TASK_DISTANCE with k = threshold; editDistance != -1 <=> best infix distance <= k).
//
// One thread per (read, strand): Myers' bit-vector algorithm in Hyyro's block form, the unit as the pattern cut into
// NW 64-bit words whose vertical deltas (Pv, Mv) stay in registers for the whole read; the match masks Peq[symbol][word]
// of both strands sit in shared memory.  Per text character the thread walks the NW blocks once, carrying the
// horizontal delta; the bottom-row score starts at |unit| (free start in the text: the top row is all zeros) and its
// running minimum is the infix distance.  Bits above |unit| in the last word never feed back into lower bits (carries
// only travel upwards), so the bottom row's delta is read at bit (|unit| - 1) mod 64 and no wildcard padding is needed.
// A strand stops as soon as its minimum is within the threshold (the caller only wants to know whether it is) unless
// exact distances are asked for.  Characters are compared as bytes, like edlib: a read symbol that the unit does not
// contain matches nothing.
#include "cfk_common.cuh"

namespace {

using namespace cfk;

constexpr int RR_THREADS = 128;
constexpr int RR_MAX_SYMBOLS = 8;  // distinct bytes of the unit (ACGT in practice) + slot 0 = "not in the unit"

// One unit of a launch: where its match masks and symbol table are, its length and threshold.
struct RrUnit {
  int64_t peq_off;            // first word of the unit's [2][RR_MAX_SYMBOLS][NW] block in RrArgs::peq
  int64_t keep_off;           // index * n_reads: the unit's row of out_keep
  int32_t index;              // the unit's row of sym_of [U][256]
  int32_t m;                  // unit length
  int32_t threshold;          // < 0: no limit (edlib's k = -1)
  int32_t pad;
};
constexpr int RR_UNITS_PER_LAUNCH = 64;  // blockIdx.y < this; a word class with more units takes several launches

struct RrArgs {
  const uint8_t* text;        // all reads, every read starts on a 16-byte boundary
  const int64_t* read_off;    // byte offset of read r
  const int64_t* read_len;
  const int32_t* order;       // items are dealt longest read first
  int64_t n_reads;
  const uint64_t* peq;        // per unit [2 strands][RR_MAX_SYMBOLS][NW], at RrUnit::peq_off
  const uint8_t* sym_of;      // per unit [256] byte -> symbol slot (0 = not in the unit)
  int32_t exact;              // != 0: never stop early, out_dist holds the exact infix distance
  int32_t* out_dist;          // [U][2 * n_reads] (read, strand), or NULL
  uint8_t* out_keep;          // [U][n_reads]
  RrUnit unit[RR_UNITS_PER_LAUNCH];  // blockIdx.y selects one (read from the parameter space: __grid_constant__)
};

template <int NW>
__global__ void __launch_bounds__(RR_THREADS) rr_filter_kernel(const __grid_constant__ RrArgs A) {
  __shared__ uint64_t s_peq[2 * RR_MAX_SYMBOLS * NW];
  __shared__ uint8_t s_sym[256];
  const RrUnit& U = A.unit[blockIdx.y];
  const uint64_t* g_peq = A.peq + U.peq_off;
  const uint8_t* g_sym = A.sym_of + 256 * (int64_t)U.index;
  for (int i = threadIdx.x; i < 2 * RR_MAX_SYMBOLS * NW; i += RR_THREADS) s_peq[i] = g_peq[i];
  for (int i = threadIdx.x; i < 256; i += RR_THREADS) s_sym[i] = g_sym[i];
  __syncthreads();
  const int32_t m = U.m;
  const int64_t item = (int64_t)blockIdx.x * RR_THREADS + threadIdx.x;
  if (item >= 2 * A.n_reads) return;
  const int64_t r = A.order[item >> 1];
  const int strand = (int)(item & 1);
  const uint64_t* peq = s_peq + strand * RR_MAX_SYMBOLS * NW;
  const int64_t n = A.read_len[r];
  const uint4* text = reinterpret_cast<const uint4*>(A.text + A.read_off[r]);
  const int last_bit = (m - 1) & 63;
  uint64_t Pv[NW], Mv[NW];
#pragma unroll
  for (int j = 0; j < NW; ++j) {
    Pv[j] = ~0ull;
    Mv[j] = 0ull;
  }
  int score = m, best = m;
  const int stop = A.exact ? -1 : U.threshold;  // best >= 0: a negative value never stops the scan
  for (int64_t t0 = 0; t0 < n; t0 += 16) {
    const uint4 chunk = __ldg(text + (t0 >> 4));
    const int cnt = (int)min((int64_t)16, n - t0);
#pragma unroll
    for (int wi = 0; wi < 4; ++wi) {
      uint32_t word = wi == 0 ? chunk.x : wi == 1 ? chunk.y : wi == 2 ? chunk.z : chunk.w;
#pragma unroll 1
      for (int c = 4 * wi; c < min(4 * wi + 4, cnt); ++c, word >>= 8) {
        const uint64_t* eqrow = peq + (int)s_sym[word & 0xFFu] * NW;
        int hin = 0;  // free start in the text: the top row is all zeros
#pragma unroll
        for (int j = 0; j < NW; ++j) {
          uint64_t Eq = eqrow[j];
          const uint64_t pv = Pv[j], mv = Mv[j];
          const uint64_t Xv = Eq | mv;
          if (hin < 0) Eq |= 1ull;
          const uint64_t Xh = (((Eq & pv) + pv) ^ pv) | Eq;
          uint64_t Ph = mv | ~(Xh | pv);
          uint64_t Mh = pv & Xh;
          const int bit = (j == NW - 1) ? last_bit : 63;
          const int hout = (int)((Ph >> bit) & 1ull) - (int)((Mh >> bit) & 1ull);
          Ph <<= 1;
          Mh <<= 1;
          if (hin < 0) Mh |= 1ull;
          else if (hin > 0) Ph |= 1ull;
          Pv[j] = Mh | ~(Xv | Ph);
          Mv[j] = Ph & Xv;
          hin = hout;
        }
        score += hin;  // the last block's delta at the unit's last row
        best = min(best, score);
      }
    }
    if (best <= stop) break;
  }
  const int64_t at = U.keep_off + r;
  if (A.out_dist != nullptr) A.out_dist[2 * at + strand] = best;
  if (U.threshold < 0 || best <= U.threshold) A.out_keep[at] = 1;
}

// A.unit[0 .. n_units) all have cfk_rr_words(m) == nw.
int rr_launch(int nw, const RrArgs& A, int n_units, cudaStream_t st) {
  const dim3 grid((unsigned)blocks_for(2 * A.n_reads, RR_THREADS), (unsigned)n_units);
  switch (nw) {
    case 4: rr_filter_kernel<4><<<grid, RR_THREADS, 0, st>>>(A); break;
    case 9: rr_filter_kernel<9><<<grid, RR_THREADS, 0, st>>>(A); break;
    case 17: rr_filter_kernel<17><<<grid, RR_THREADS, 0, st>>>(A); break;
    case 33: rr_filter_kernel<33><<<grid, RR_THREADS, 0, st>>>(A); break;
    default: rr_filter_kernel<52><<<grid, RR_THREADS, 0, st>>>(A); break;
  }
  CFK_CHECK_LAUNCH("rr_filter_kernel", 1);
  return CFK_OK;
}

// ---- units longer than 52 words: one warp per (segment, strand) ----------------------------------------------------
// The unit's nw = ceil(m / 64) words are split over the lanes, W consecutive words per lane, so Pv / Mv of a unit of up
// to 32 * W * 64 bases stay in registers.  The lanes form a wavefront: at step s lane L applies the block step of
// rr_filter_kernel to its W words for text character s - L, starting from the horizontal delta that lane L - 1 produced
// for that character at step s - 1 (lane 0 starts from 0: free start in the text).  That delta and the character's
// symbol slot travel up the lanes in one shuffle per step, so only lane 0 reads the text.  The bottom row is bit
// (m - 1) & 63 of word nw - 1, in lane (nw - 1) / W, which keeps score and best; a segment of n bases takes n + that lane
// steps.  Every 16 characters of the bottom lane the warp checks best against the stop rule of rr_filter_kernel, so
// out_dist without exact holds what rr_filter_kernel writes there.
// Match masks are lane-minor, [2 strands][RR_MAX_SYMBOLS][W][32 lanes]: word k of every lane is one 256-byte row of
// shared memory whatever symbol each lane holds, so a warp's load is free of bank conflicts.
constexpr int RRW_WARPS = 8;                 // warps per block; each takes one (segment, strand)
constexpr int RRW_THREADS = 32 * RRW_WARPS;
constexpr int RRW_MAX_BASES = 32 * 16 * 64;  // W = 16

template <int W>
__global__ void __launch_bounds__(RRW_THREADS) rr_filter_warp_kernel(const __grid_constant__ RrArgs A) {
  extern __shared__ uint64_t s_peq[];  // [2][RR_MAX_SYMBOLS][W][32]
  __shared__ uint8_t s_sym[256];
  const RrUnit& U = A.unit[blockIdx.y];
  const uint64_t* g_peq = A.peq + U.peq_off;
  const uint8_t* g_sym = A.sym_of + 256 * (int64_t)U.index;
  for (int i = threadIdx.x; i < 2 * RR_MAX_SYMBOLS * W * 32; i += RRW_THREADS) s_peq[i] = g_peq[i];
  for (int i = threadIdx.x; i < 256; i += RRW_THREADS) s_sym[i] = g_sym[i];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int64_t item = (int64_t)blockIdx.x * RRW_WARPS + (threadIdx.x >> 5);
  if (item >= 2 * A.n_reads) return;  // the whole warp
  const int64_t r = A.order[item >> 1];
  const int strand = (int)(item & 1);
  const uint64_t* peq = s_peq + strand * RR_MAX_SYMBOLS * W * 32 + lane;
  const int64_t n = A.read_len[r];
  const uint4* text = reinterpret_cast<const uint4*>(A.text + A.read_off[r]);
  const int32_t m = U.m;
  const int nw = (m + 63) >> 6;
  const int bottom_lane = (nw - 1) / W, bottom_k = (nw - 1) % W, last_bit = (m - 1) & 63;
  const bool bottom = lane == bottom_lane;
  uint64_t Pv[W], Mv[W];
#pragma unroll
  for (int k = 0; k < W; ++k) {
    Pv[k] = ~0ull;
    Mv[k] = 0ull;
  }
  int score = m, best = m;
  const int stop = A.exact ? -1 : U.threshold;
  uint4 chunk = make_uint4(0, 0, 0, 0);
  int from_below = 1;  // (horizontal delta + 1) | symbol slot << 2, from lane - 1 at the previous step
  const int64_t steps = n + bottom_lane;
  for (int64_t s = 0; s < steps; ++s) {
    const int64_t c = s - lane;  // this lane's text character
    int sym, hin;
    if (lane == 0) {
      if (c < n && (c & 15) == 0) chunk = __ldg(text + (c >> 4));
      const int q = (int)(c & 15);
      const uint32_t word = q < 4 ? chunk.x : q < 8 ? chunk.y : q < 12 ? chunk.z : chunk.w;
      sym = s_sym[(word >> (8 * (q & 3))) & 0xFFu];
      hin = 0;
    } else {
      sym = from_below >> 2;
      hin = (from_below & 3) - 1;
    }
    const bool active = c >= 0 && c < n;
    const uint64_t* eqrow = peq + sym * (W * 32);
    int delta = 0;
#pragma unroll
    for (int k = 0; k < W; ++k) {
      uint64_t Eq = eqrow[k * 32];
      const uint64_t pv = Pv[k], mv = Mv[k];
      const uint64_t Xv = Eq | mv;
      if (hin < 0) Eq |= 1ull;
      const uint64_t Xh = (((Eq & pv) + pv) ^ pv) | Eq;
      uint64_t Ph = mv | ~(Xh | pv);
      uint64_t Mh = pv & Xh;
      const int bit = (bottom && k == bottom_k) ? last_bit : 63;
      const int hout = (int)((Ph >> bit) & 1ull) - (int)((Mh >> bit) & 1ull);
      Ph <<= 1;
      Mh <<= 1;
      if (hin < 0) Mh |= 1ull;
      else if (hin > 0) Ph |= 1ull;
      if (active) {
        Pv[k] = Mh | ~(Xv | Ph);
        Mv[k] = Ph & Xv;
      }
      if (k == bottom_k) delta = hout;
      hin = hout;
    }
    if (bottom && active) {
      score += delta;
      best = min(best, score);
    }
    from_below = __shfl_up_sync(0xFFFFFFFFu, (hin + 1) | (sym << 2), 1);
    const int64_t done = s - bottom_lane + 1;  // characters the bottom lane has finished
    if (done > 0 && (done & 15) == 0 && __shfl_sync(0xFFFFFFFFu, best, bottom_lane) <= stop) break;
  }
  if (bottom) {
    const int64_t at = U.keep_off + r;
    if (A.out_dist != nullptr) A.out_dist[2 * at + strand] = best;
    if (U.threshold < 0 || best <= U.threshold) A.out_keep[at] = 1;
  }
}

// A.unit[0 .. n_units) all have cfk_rr_long_words(m) == w.
int rr_long_launch(int w, const RrArgs& A, int n_units, cudaStream_t st) {
  const dim3 grid((unsigned)blocks_for(2 * A.n_reads, RRW_WARPS), (unsigned)n_units);
  const int smem = 2 * RR_MAX_SYMBOLS * w * 32 * (int)sizeof(uint64_t);
  switch (w) {
    case 2: rr_filter_warp_kernel<2><<<grid, RRW_THREADS, smem, st>>>(A); break;
    case 4: rr_filter_warp_kernel<4><<<grid, RRW_THREADS, smem, st>>>(A); break;
    case 8: rr_filter_warp_kernel<8><<<grid, RRW_THREADS, smem, st>>>(A); break;
    default: {
      static unsigned long long smem_set = 0;  // 64 KB: above the default limit of 48 KB
      if (const cudaError_t e = ensure_dynamic_smem(rr_filter_warp_kernel<16>, smem, &smem_set))
        return fail(CFK_ERR_CUDA, "rr_filter_warp_kernel<16>: dynamic shared memory", e);
      rr_filter_warp_kernel<16><<<grid, RRW_THREADS, smem, st>>>(A);
      break;
    }
  }
  CFK_CHECK_LAUNCH("rr_filter_warp_kernel", 1);
  return CFK_OK;
}

// ---- streaming form (read_recruitment.recruit_file): raw file text in, output file text out ----------------------
// Both copy kernels are driven by the destination: one thread writes 16 consecutive output bytes with one 16-byte store
// and finds its source by a binary search over the sorted destination offsets, so 80-column FASTA lines and megabase
// single-line reads cost the same per byte.
constexpr int COPY_THREADS = 256;

// last i in [0, n) with key[i * stride] <= q (keys ascending, key[0] <= q)
__device__ __forceinline__ int64_t last_at_or_below(const int64_t* key, int64_t stride, int64_t n, int64_t q) {
  int64_t lo = 0, hi = n;
  while (hi - lo > 1) {
    const int64_t mid = (lo + hi) >> 1;
    if (key[mid * stride] <= q) lo = mid;
    else hi = mid;
  }
  return lo;
}

__device__ __forceinline__ uint4 pack16(const uint8_t* b) {
  uint32_t w[4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
    w[i] = (uint32_t)b[4 * i] | ((uint32_t)b[4 * i + 1] << 8) | ((uint32_t)b[4 * i + 2] << 16) | ((uint32_t)b[4 * i + 3] << 24);
  return make_uint4(w[0], w[1], w[2], w[3]);
}

// text[q] = the sequence byte that piece p places at q, 0 between records.  piece = [n][3] (source offset in raw,
// length, destination offset), destinations ascending and non-overlapping.
__global__ void __launch_bounds__(COPY_THREADS) rr_gather_kernel(const uint8_t* __restrict__ raw, const int64_t* __restrict__ piece,
                                                                 int64_t n_pieces, uint8_t* __restrict__ text, int64_t text_bytes) {
  const int64_t q0 = ((int64_t)blockIdx.x * COPY_THREADS + threadIdx.x) * 16;
  if (q0 >= text_bytes) return;
  uint8_t b[16];
  int64_t p = (n_pieces > 0 && piece[2] <= q0) ? last_at_or_below(piece + 2, 3, n_pieces, q0) : 0;
  int64_t src = 0, dst = INT64_MAX, end = INT64_MAX;
  if (p < n_pieces) src = piece[3 * p], end = (dst = piece[3 * p + 2]) + piece[3 * p + 1];
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    const int64_t q = q0 + k;
    while (q >= end && ++p < n_pieces) src = piece[3 * p], end = (dst = piece[3 * p + 2]) + piece[3 * p + 1];
    b[k] = (q >= dst && q < end) ? raw[src + (q - dst)] : 0;
  }
  reinterpret_cast<uint4*>(text)[q0 >> 4] = pack16(b);
}

// text[q] = base q - rec[r][3] of BAM record r (rec = [n][4] as cfk_bam_scan writes it, bam_seq = [n][2]: offset of the
// 4-bit SEQ in raw, reverse flag), 0 between records.  Every record starts on a 16-byte boundary, so the 16 bytes of a
// thread belong to one record's slot.
__global__ void __launch_bounds__(COPY_THREADS) rr_bam_gather_kernel(const uint8_t* __restrict__ raw,
                                                                     const int64_t* __restrict__ bam_seq,
                                                                     const int64_t* __restrict__ rec, int64_t n,
                                                                     uint8_t* __restrict__ text, int64_t text_bytes) {
  const int64_t q0 = ((int64_t)blockIdx.x * COPY_THREADS + threadIdx.x) * 16;
  if (q0 >= text_bytes) return;
  const int64_t r = last_at_or_below(rec + 3, 4, n, q0);
  const int64_t at = q0 - rec[4 * r + 3], len = rec[4 * r + 2], src = bam_seq[2 * r];
  const bool rev = bam_seq[2 * r + 1] != 0;
  const char* code = rev ? "=TGKCYSBAWRDMHVN" : "=ACMGRSVTWYHKDBN";  // complement = the 4 bits reversed
  uint8_t b[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    const int64_t i = at + k;
    uint8_t c = 0;
    if (i < len) {
      const int64_t j = rev ? len - 1 - i : i;
      const uint8_t v = raw[src + (j >> 1)];
      c = code[(j & 1) ? (v & 15) : (v >> 4)];
    }
    b[k] = c;
  }
  reinterpret_cast<uint4*>(text)[q0 >> 4] = pack16(b);
}

// sizes[r] = bytes of ">name\nsequence\n" when record r is kept, else 0.  A record is kept when any of its segments
// seg_keep[seg_ptr[r] .. seg_ptr[r + 1]) hit; seg_keep == NULL keeps every record.
__global__ void rr_keep_sizes_kernel(const uint8_t* __restrict__ seg_keep, const int64_t* __restrict__ seg_ptr,
                                     const int64_t* __restrict__ rec, int64_t n, int32_t* __restrict__ sizes) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  bool keep = seg_keep == nullptr;
  if (!keep)
    for (int64_t s = seg_ptr[r]; s < seg_ptr[r + 1] && !keep; ++s) keep = seg_keep[s] != 0;
  sizes[r] = keep ? (int32_t)(rec[4 * r + 1] + rec[4 * r + 2] + 3) : 0;
}

// out[out_off[r] ..] = ">" name "\n" sequence "\n" of record r (rec = [n][4]: name offset in raw, name length, sequence
// length, sequence offset in text); out_off = exclusive scan of the sizes, out_off[n] = total.
__global__ void __launch_bounds__(COPY_THREADS) rr_emit_kernel(const uint8_t* __restrict__ raw, const uint8_t* __restrict__ text,
                                                               const int64_t* __restrict__ rec, const int64_t* __restrict__ out_off,
                                                               int64_t n, int64_t max_bytes, uint8_t* __restrict__ out) {
  const int64_t total = min(out_off[n], max_bytes);
  const int64_t q0 = ((int64_t)blockIdx.x * COPY_THREADS + threadIdx.x) * 16;
  if (q0 >= total) return;
  int64_t r = last_at_or_below(out_off, 1, n + 1, q0);
  int64_t lo = out_off[r], hi = out_off[r + 1];
  uint8_t b[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    const int64_t q = q0 + k;
    if (q >= total) {
      b[k] = 0;
      continue;
    }
    while (q >= hi) lo = hi, hi = out_off[++r + 1];
    const int64_t at = q - lo, nl = rec[4 * r + 1];
    uint8_t c = '\n';
    if (at == 0) c = '>';
    else if (at <= nl) c = raw[rec[4 * r] + at - 1];
    else if (at > nl + 1 && q < hi - 1) c = text[rec[4 * r + 3] + at - nl - 2];
    b[k] = c;
  }
  if (q0 + 16 <= total) {
    reinterpret_cast<uint4*>(out)[q0 >> 4] = pack16(b);
  } else {
    for (int k = 0; q0 + k < total; ++k) out[q0 + k] = b[k];
  }
}

}  // namespace

extern "C" {

int cfk_rr_max_symbols(void) { return RR_MAX_SYMBOLS; }

/* words per strand of the peq table for a unit of m bases, or -1 if the unit is too long */
int cfk_rr_words(int32_t m) {
  if (m < 1) return -1;
  const int need = (m + 63) / 64;
  const int sizes[] = {4, 9, 17, 33, 52};
  for (int s : sizes)
    if (need <= s) return s;
  return -1;
}

int cfk_rr_filter(const uint8_t* text, const int64_t* read_off, const int64_t* read_len, const int32_t* order, int64_t n_reads,
                  const uint64_t* peq, const uint8_t* sym_of, int32_t m, int32_t threshold, int32_t exact, int32_t* out_dist,
                  uint8_t* out_keep, cfk_stream_t stream) {
  const int nw = cfk_rr_words(m);
  if (nw < 0) return fail(CFK_ERR_INVALID, "cfk_rr_filter: the unit must have 1..3328 bases");
  if (n_reads < 0 || n_reads >= (1ll << 30)) return fail(CFK_ERR_INVALID, "cfk_rr_filter: bad sizes");
  if (((uintptr_t)text & 15u) != 0) return fail(CFK_ERR_INVALID, "cfk_rr_filter: text must be 16-byte aligned");
  if (n_reads == 0) return CFK_OK;
  RrArgs A{text, read_off, read_len, order, n_reads, peq, sym_of, exact, out_dist, out_keep, {}};
  A.unit[0] = RrUnit{0, 0, 0, m, threshold, 0};
  return rr_launch(nw, A, 1, (cudaStream_t)stream);
}

int cfk_rr_filter_units(const uint8_t* text, const int64_t* seg_off, const int64_t* seg_len, const int32_t* order, int64_t n_seg,
                        int32_t n_units, const uint64_t* peq, const uint8_t* sym_of, const int32_t* unit_m,
                        const int32_t* unit_threshold, uint8_t* out_keep, cfk_stream_t stream) {
  if (n_seg < 0 || n_seg >= (1ll << 30) || n_units < 0 || (n_units > 0 && (unit_m == nullptr || unit_threshold == nullptr)))
    return fail(CFK_ERR_INVALID, "cfk_rr_filter_units: bad sizes");
  if (((uintptr_t)text & 15u) != 0) return fail(CFK_ERR_INVALID, "cfk_rr_filter_units: text must be 16-byte aligned");
  for (int32_t u = 0; u < n_units; ++u)
    if (cfk_rr_words(unit_m[u]) < 0) return fail(CFK_ERR_INVALID, "cfk_rr_filter_units: every unit must have 1..3328 bases");
  if (n_seg == 0 || n_units == 0) return CFK_OK;
  // one launch per word class present (several when a class has more than RR_UNITS_PER_LAUNCH units), all on `stream`
  const cudaStream_t st = (cudaStream_t)stream;
  for (int nw : {4, 9, 17, 33, 52}) {
    RrArgs A{text, seg_off, seg_len, order, n_seg, peq, sym_of, 0, nullptr, out_keep, {}};
    int n = 0;
    int64_t off = 0;
    for (int32_t u = 0; u < n_units; ++u) {
      const int w = cfk_rr_words(unit_m[u]);
      if (w == nw) {
        A.unit[n++] = RrUnit{off, u * n_seg, u, unit_m[u], unit_threshold[u], 0};
        if (n == RR_UNITS_PER_LAUNCH) {
          if (const int rc = rr_launch(nw, A, n, st)) return rc;
          n = 0;
        }
      }
      off += 2 * RR_MAX_SYMBOLS * w;
    }
    if (n > 0)
      if (const int rc = rr_launch(nw, A, n, st)) return rc;
  }
  return CFK_OK;
}

/* lanes' words of rr_filter_warp_kernel for a unit of m bases: the least W with ceil(ceil(m / 64) / W) <= 32 */
int cfk_rr_long_words(int32_t m) {
  if (m < 1 || m > RRW_MAX_BASES) return -1;
  const int need = (m + 63) / 64;
  for (int w : {2, 4, 8, 16})
    if (need <= 32 * w) return w;
  return -1;
}

int cfk_rr_filter_long(const uint8_t* text, const int64_t* seg_off, const int64_t* seg_len, const int32_t* order, int64_t n_seg,
                       int32_t n_units, const uint64_t* peq, const uint8_t* sym_of, const int32_t* unit_m,
                       const int32_t* unit_threshold, int32_t exact, int32_t* out_dist, uint8_t* out_keep,
                       cfk_stream_t stream) {
  if (n_seg < 0 || n_seg >= (1ll << 30) || n_units < 0 || (n_units > 0 && (unit_m == nullptr || unit_threshold == nullptr)))
    return fail(CFK_ERR_INVALID, "cfk_rr_filter_long: bad sizes");
  if (((uintptr_t)text & 15u) != 0) return fail(CFK_ERR_INVALID, "cfk_rr_filter_long: text must be 16-byte aligned");
  for (int32_t u = 0; u < n_units; ++u)
    if (cfk_rr_long_words(unit_m[u]) < 0)
      return fail(CFK_ERR_INVALID, "cfk_rr_filter_long: every unit must have 1..32768 bases");
  if (n_seg == 0 || n_units == 0) return CFK_OK;
  // one launch per lane-word class present (several when a class has more than RR_UNITS_PER_LAUNCH units)
  const cudaStream_t st = (cudaStream_t)stream;
  for (int w : {2, 4, 8, 16}) {
    RrArgs A{text, seg_off, seg_len, order, n_seg, peq, sym_of, exact, out_dist, out_keep, {}};
    int n = 0;
    int64_t off = 0;
    for (int32_t u = 0; u < n_units; ++u) {
      const int uw = cfk_rr_long_words(unit_m[u]);
      if (uw == w) {
        A.unit[n++] = RrUnit{off, u * n_seg, u, unit_m[u], unit_threshold[u], 0};
        if (n == RR_UNITS_PER_LAUNCH) {
          if (const int rc = rr_long_launch(w, A, n, st)) return rc;
          n = 0;
        }
      }
      off += 2 * RR_MAX_SYMBOLS * 32 * uw;
    }
    if (n > 0)
      if (const int rc = rr_long_launch(w, A, n, st)) return rc;
  }
  return CFK_OK;
}

int cfk_rr_gather(const uint8_t* raw, const int64_t* pieces, int64_t n_pieces, uint8_t* text, int64_t text_bytes,
                  cfk_stream_t stream) {
  if (n_pieces < 0 || text_bytes < 0 || (text_bytes & 15) != 0 || ((uintptr_t)text & 15u) != 0)
    return fail(CFK_ERR_INVALID, "cfk_rr_gather: bad sizes, or text not 16-byte aligned");
  if (text_bytes == 0) return CFK_OK;
  rr_gather_kernel<<<(unsigned)blocks_for(text_bytes / 16, COPY_THREADS), COPY_THREADS, 0, (cudaStream_t)stream>>>(
      raw, pieces, n_pieces, text, text_bytes);
  CFK_CHECK_LAUNCH("rr_gather_kernel", 1);
  return CFK_OK;
}

int cfk_rr_bam_gather(const uint8_t* raw, const int64_t* bam_seq, const int64_t* records, int64_t n_records, uint8_t* text,
                      int64_t text_bytes, cfk_stream_t stream) {
  if (n_records < 0 || text_bytes < 0 || (text_bytes & 15) != 0 || ((uintptr_t)text & 15u) != 0 ||
      (text_bytes > 0 && n_records == 0))
    return fail(CFK_ERR_INVALID, "cfk_rr_bam_gather: bad sizes, or text not 16-byte aligned");
  if (text_bytes == 0) return CFK_OK;
  rr_bam_gather_kernel<<<(unsigned)blocks_for(text_bytes / 16, COPY_THREADS), COPY_THREADS, 0, (cudaStream_t)stream>>>(
      raw, bam_seq, records, n_records, text, text_bytes);
  CFK_CHECK_LAUNCH("rr_bam_gather_kernel", 1);
  return CFK_OK;
}

int cfk_rr_keep_sizes(const uint8_t* seg_keep, const int64_t* seg_ptr, const int64_t* records, int64_t n_records,
                      int32_t* sizes, cfk_stream_t stream) {
  if (n_records < 0 || (seg_keep == nullptr) != (seg_ptr == nullptr))
    return fail(CFK_ERR_INVALID, "cfk_rr_keep_sizes: n_records < 0, or only one of seg_keep / seg_ptr given");
  if (n_records == 0) return CFK_OK;
  rr_keep_sizes_kernel<<<(unsigned)blocks_for(n_records, 256), 256, 0, (cudaStream_t)stream>>>(seg_keep, seg_ptr, records,
                                                                                                n_records, sizes);
  CFK_CHECK_LAUNCH("rr_keep_sizes_kernel", 1);
  return CFK_OK;
}

int cfk_rr_emit(const uint8_t* raw, const uint8_t* text, const int64_t* records, const int64_t* out_off, int64_t n_records,
                int64_t max_bytes, uint8_t* out, cfk_stream_t stream) {
  if (n_records < 0 || max_bytes < 0 || ((uintptr_t)out & 15u) != 0)
    return fail(CFK_ERR_INVALID, "cfk_rr_emit: bad sizes, or out not 16-byte aligned");
  if (n_records == 0 || max_bytes == 0) return CFK_OK;
  rr_emit_kernel<<<(unsigned)blocks_for((max_bytes + 15) / 16, COPY_THREADS), COPY_THREADS, 0, (cudaStream_t)stream>>>(
      raw, text, records, out_off, n_records, max_bytes, out);
  CFK_CHECK_LAUNCH("rr_emit_kernel", 1);
  return CFK_OK;
}

}  // extern "C"
