// bgzf.cu — DEFLATE (RFC 1951) decoder for the BGZF blocks of a compressed read file (SAM spec §4.1).
//
// A BGZF file is a series of independent gzip members of at most 64 KiB inflated each; the host finds them without
// inflating anything (cfk_bgzf_blocks, bam_scan.cpp) and this kernel inflates all the blocks of a chunk at once.
//
// One warp per block.  Lane 0 decodes the stream -- Huffman decoding is a serial walk over the bits -- into the block's
// output held whole in shared memory (ISIZE <= 65536), so back-references and the CRC pass read shared memory instead
// of making round trips to L2; then the whole warp copies the output out to global memory.  A 64 MiB chunk holds about
// a thousand blocks, so with three warps of 70 KiB shared memory per SM the grid covers every SM about twice.
//
// Bounds-checked by construction: every compressed byte read is checked against the block's payload length, every
// output write against ISIZE, and a back-reference may only reach into the block's own output (each member starts with
// an empty window).  A malformed stream therefore ends in a status, never in an access outside its block.
#include "cfk_common.cuh"

namespace {

using namespace cfk;

constexpr int BGZF_MAX_OUT = 65536;  // the largest ISIZE the host passes (cfk_bgzf_blocks)
constexpr int MAXBITS = 15;

__constant__ uint16_t c_lbase[29] = {3,  4,  5,  6,  7,  8,  9,  10, 11,  13,  15,  17,  19,  23, 27,
                                     31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
__constant__ uint8_t c_lext[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
__constant__ uint16_t c_dbase[30] = {1,   2,   3,   4,   5,   7,    9,    13,   17,   25,   33,   49,   65,    97,    129,
                                     193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
__constant__ uint8_t c_dext[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
__constant__ uint8_t c_clorder[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

// A canonical Huffman code as counts per length and symbols ordered by code (zlib's contrib/puff layout).
struct Huff {
  uint16_t count[MAXBITS + 1];
  uint16_t sym[288];
};

struct Shared {
  uint8_t out[BGZF_MAX_OUT];
  uint32_t crc[4][256];        // slice-by-4 tables of the gzip CRC-32
  Huff lit, dist;
  uint16_t offs[MAXBITS + 1];
  uint8_t lengths[320];
};

enum : int32_t { ST_OK = CFK_BGZF_OK, ST_BAD = CFK_BGZF_BAD_STREAM, ST_LEN = CFK_BGZF_BAD_LENGTH, ST_CRC = CFK_BGZF_BAD_CRC };

struct Bits {
  const uint8_t* in;
  int64_t pos, len;  // next byte of the payload to load, payload length
  uint64_t buf;
  int cnt;

  __device__ __forceinline__ void refill() {
    while (cnt <= 56 && pos < len) {
      buf |= (uint64_t)__ldg(in + pos++) << cnt;
      cnt += 8;
    }
  }
  // n <= 32 bits, least significant first; false when the payload ends first
  __device__ __forceinline__ bool get(int n, uint32_t& v) {
    if (cnt < n) {
      refill();
      if (cnt < n) return false;
    }
    v = (uint32_t)(buf & ((1ull << n) - 1));
    buf >>= n;
    cnt -= n;
    return true;
  }
};

// puff's construct(): 0 = complete code, > 0 = incomplete, < 0 = over-subscribed
__device__ int construct(Huff& h, uint16_t* offs, const uint8_t* length, int n) {
  for (int l = 0; l <= MAXBITS; ++l) h.count[l] = 0;
  for (int s = 0; s < n; ++s) h.count[length[s]]++;
  if (h.count[0] == n) return 0;  // no codes: "complete", decoding any symbol fails
  int left = 1;
  for (int l = 1; l <= MAXBITS; ++l) {
    left <<= 1;
    left -= h.count[l];
    if (left < 0) return left;
  }
  offs[1] = 0;
  for (int l = 1; l < MAXBITS; ++l) offs[l + 1] = offs[l] + h.count[l];
  for (int s = 0; s < n; ++s)
    if (length[s] != 0) h.sym[offs[length[s]]++] = (uint16_t)s;
  return left;
}

// the next symbol of code h, or -1 (payload ended, or a bit pattern without a code)
__device__ __forceinline__ int decode(const Huff& h, Bits& B) {
  if (B.cnt < MAXBITS) B.refill();
  int code = 0, first = 0, index = 0;
  const uint64_t bits = B.buf;
#pragma unroll
  for (int l = 1; l <= MAXBITS; ++l) {
    if (l > B.cnt) return -1;
    code |= (int)((bits >> (l - 1)) & 1u);
    const int count = h.count[l];
    if (code - count < first) {
      B.buf >>= l;
      B.cnt -= l;
      return h.sym[index + (code - first)];
    }
    index += count;
    first = (first + count) << 1;
    code <<= 1;
  }
  return -1;
}

// Huffman-coded data of one block, up to end-of-block.  Returns a status, ST_OK when end-of-block was reached.
__device__ int32_t codes(Shared& S, Bits& B, int& outcnt, int isize) {
  for (;;) {
    int sym = decode(S.lit, B);
    if (sym < 0) return ST_BAD;
    if (sym < 256) {
      if (outcnt >= isize) return ST_LEN;
      S.out[outcnt++] = (uint8_t)sym;
      continue;
    }
    if (sym == 256) return ST_OK;
    sym -= 257;
    if (sym >= 29) return ST_BAD;
    uint32_t e;
    if (!B.get(c_lext[sym], e)) return ST_BAD;
    const int len = c_lbase[sym] + (int)e;
    const int ds = decode(S.dist, B);
    if (ds < 0 || ds >= 30) return ST_BAD;
    if (!B.get(c_dext[ds], e)) return ST_BAD;
    const int dist = c_dbase[ds] + (int)e;
    if (dist > outcnt) return ST_BAD;  // before the start of the block's output
    if (len > isize - outcnt) return ST_LEN;
    uint8_t* o = S.out + outcnt;
    for (int i = 0; i < len; ++i) o[i] = o[i - dist];
    outcnt += len;
  }
}

__device__ int32_t stored(Shared& S, Bits& B, int& outcnt, int isize) {
  B.buf >>= B.cnt & 7;  // to a byte boundary, then hand the whole bytes still buffered back to the input
  B.cnt &= ~7;
  B.pos -= B.cnt >> 3;
  B.buf = 0;
  B.cnt = 0;
  if (B.len - B.pos < 4) return ST_BAD;
  const int len = B.in[B.pos] | (B.in[B.pos + 1] << 8);
  const int nlen = B.in[B.pos + 2] | (B.in[B.pos + 3] << 8);
  B.pos += 4;
  if (len != (~nlen & 0xffff)) return ST_BAD;
  if (len > B.len - B.pos) return ST_BAD;
  if (len > isize - outcnt) return ST_LEN;
  for (int i = 0; i < len; ++i) S.out[outcnt + i] = __ldg(B.in + B.pos + i);
  B.pos += len;
  outcnt += len;
  return ST_OK;
}

__device__ int32_t fixed_tables(Shared& S) {
  int s = 0;
  for (; s < 144; ++s) S.lengths[s] = 8;
  for (; s < 256; ++s) S.lengths[s] = 9;
  for (; s < 280; ++s) S.lengths[s] = 7;
  for (; s < 288; ++s) S.lengths[s] = 8;
  construct(S.lit, S.offs, S.lengths, 288);
  for (s = 0; s < 30; ++s) S.lengths[s] = 5;
  construct(S.dist, S.offs, S.lengths, 30);
  return ST_OK;
}

__device__ int32_t dynamic_tables(Shared& S, Bits& B) {
  uint32_t v;
  if (!B.get(14, v)) return ST_BAD;
  const int nlen = (int)(v & 31) + 257, ndist = (int)((v >> 5) & 31) + 1, ncode = (int)(v >> 10) + 4;
  if (nlen > 286 || ndist > 30) return ST_BAD;
  for (int i = 0; i < 19; ++i) {
    uint32_t l = 0;
    if (i < ncode && !B.get(3, l)) return ST_BAD;
    S.lengths[c_clorder[i]] = (uint8_t)l;
  }
  if (construct(S.lit, S.offs, S.lengths, 19) != 0) return ST_BAD;  // the code-length code must be complete
  int index = 0;
  while (index < nlen + ndist) {
    int sym = decode(S.lit, B);
    if (sym < 0) return ST_BAD;
    if (sym < 16) {
      S.lengths[index++] = (uint8_t)sym;
      continue;
    }
    uint8_t len = 0;
    uint32_t rep;
    if (sym == 16) {
      if (index == 0) return ST_BAD;
      len = S.lengths[index - 1];
      if (!B.get(2, rep)) return ST_BAD;
      rep += 3;
    } else if (sym == 17) {
      if (!B.get(3, rep)) return ST_BAD;
      rep += 3;
    } else {
      if (!B.get(7, rep)) return ST_BAD;
      rep += 11;
    }
    if (index + (int)rep > nlen + ndist) return ST_BAD;
    for (uint32_t k = 0; k < rep; ++k) S.lengths[index++] = len;
  }
  if (S.lengths[256] == 0) return ST_BAD;  // no end-of-block code
  if (construct(S.lit, S.offs, S.lengths, nlen) != 0) return ST_BAD;  // literal/length code: complete
  // distance code: complete, or the one incomplete form zlib writes -- a single code (of one bit); none at all is
  // accepted too and fails only if a distance is decoded (as in zlib and puff)
  const int err = construct(S.dist, S.offs, S.lengths + nlen, ndist);
  if (err < 0 || (err > 0 && ndist != S.dist.count[0] + S.dist.count[1])) return ST_BAD;
  return ST_OK;
}

// Inflates one payload into S.out; *outcnt = bytes written.  ST_OK only when the final block ends in the payload's
// last byte (a gzip reader takes the trailer from right after the DEFLATE stream) and exactly isize bytes came out.
__device__ int32_t inflate_block(Shared& S, const uint8_t* in, int64_t len, int isize, int& outcnt) {
  Bits B{in, 0, len, 0, 0};
  outcnt = 0;
  uint32_t last = 0, type = 0;
  do {
    if (!B.get(1, last) || !B.get(2, type)) return ST_BAD;
    int32_t st;
    if (type == 0) {
      st = stored(S, B, outcnt, isize);
    } else if (type == 1 || type == 2) {
      st = type == 1 ? fixed_tables(S) : dynamic_tables(S, B);
      if (st == ST_OK) st = codes(S, B, outcnt, isize);
    } else {
      st = ST_BAD;
    }
    if (st != ST_OK) return st;
  } while (!last);
  if (B.pos - (B.cnt >> 3) != len) return ST_BAD;  // bytes left between the DEFLATE stream and the trailer
  return outcnt == isize ? ST_OK : ST_LEN;
}

__device__ __forceinline__ uint32_t crc32_shared(const Shared& S, const uint8_t* p, int n) {
  uint32_t c = 0xffffffffu;
  int i = 0;
  for (; i + 4 <= n; i += 4) {  // p is 16-byte aligned
    c ^= *reinterpret_cast<const uint32_t*>(p + i);
    c = S.crc[3][c & 0xff] ^ S.crc[2][(c >> 8) & 0xff] ^ S.crc[1][(c >> 16) & 0xff] ^ S.crc[0][c >> 24];
  }
  for (; i < n; ++i) c = S.crc[0][(c ^ p[i]) & 0xff] ^ (c >> 8);
  return c ^ 0xffffffffu;
}

// rows [n][5]: payload offset in comp, payload length, ISIZE, CRC32, output offset
__global__ void __launch_bounds__(32) bgzf_inflate_kernel(const uint8_t* __restrict__ comp, const int64_t* __restrict__ rows,
                                                          int64_t n, uint8_t* __restrict__ out, int32_t* __restrict__ status) {
  extern __shared__ __align__(16) uint8_t smem[];
  Shared& S = *reinterpret_cast<Shared*>(smem);
  const int lane = threadIdx.x;
  for (int i = lane; i < 256; i += 32) {
    uint32_t c = (uint32_t)i;
    for (int k = 0; k < 8; ++k) c = (c & 1) ? 0xedb88320u ^ (c >> 1) : c >> 1;
    S.crc[0][i] = c;
  }
  __syncwarp();
  for (int i = lane; i < 256; i += 32) {
    uint32_t c = S.crc[0][i];
    for (int t = 1; t < 4; ++t) S.crc[t][i] = c = S.crc[0][c & 0xff] ^ (c >> 8);
  }
  __syncwarp();
  for (int64_t b = blockIdx.x; b < n; b += gridDim.x) {
    const int64_t* r = rows + 5 * b;
    const int64_t isize = r[2];
    int outcnt = 0;
    if (lane == 0) {
      int32_t st = ST_LEN;
      if (isize >= 0 && isize <= BGZF_MAX_OUT && r[1] >= 0) {
        st = inflate_block(S, comp + r[0], r[1], (int)isize, outcnt);
        if (st == ST_OK && crc32_shared(S, S.out, outcnt) != (uint32_t)r[3]) st = ST_CRC;
      }
      status[b] = st;
    }
    outcnt = __shfl_sync(FULL, outcnt, 0);
    __syncwarp();
    uint8_t* dst = out + r[4];
    for (int i = lane; i < outcnt; i += 32) dst[i] = S.out[i];
    __syncwarp();
  }
}

unsigned long long g_smem_set = 0;

}  // namespace

extern "C" int cfk_bgzf_inflate(const uint8_t* comp, const int64_t* blocks, int64_t n_blocks, uint8_t* out,
                                int32_t* status, cfk_stream_t stream) {
  if (n_blocks < 0 || (n_blocks > 0 && (comp == nullptr || blocks == nullptr || out == nullptr || status == nullptr)))
    return fail(CFK_ERR_INVALID, "cfk_bgzf_inflate: bad arguments");
  if (n_blocks == 0) return CFK_OK;
  const int smem = (int)sizeof(Shared);
  if (cudaError_t e = ensure_dynamic_smem(bgzf_inflate_kernel, smem, &g_smem_set))
    return fail(CFK_ERR_CUDA, "cfk_bgzf_inflate: shared memory attribute", e);
  const int64_t grid = n_blocks < (1 << 20) ? n_blocks : (1 << 20);
  bgzf_inflate_kernel<<<(unsigned)grid, 32, smem, (cudaStream_t)stream>>>(comp, blocks, n_blocks, out, status);
  CFK_CHECK_LAUNCH("bgzf_inflate_kernel", 1);
  return CFK_OK;
}
