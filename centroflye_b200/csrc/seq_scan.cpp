// seq_scan.cpp — FASTA / FASTQ record scanner of the streaming read recruitment filter (host code).
//
// One pass over a chunk of read-file text that finds what read_sequences() (centroflye_b200/read_recruitment.py:29-55,
// the restatement of rr.cpp's kseq_read loop) yields, without copying a byte: per record the name's place in the chunk
// and the sequence length, per stripped sequence line its place in the chunk and in the packed text the device filter
// reads.  Only line ends and line starts are touched (memchr); the byte copies happen on the device (rr_gather_kernel).
// The call keeps no state: the caller carries the bytes from `consumed` on into the next chunk.
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/cfk.h"

extern thread_local char cfk_g_err[512];  // cfk_last_error() (cfk.cu)

namespace {

// str.isspace() on ASCII: what str.split() and str.strip() without arguments remove
inline bool is_space(uint8_t c) { return c == ' ' || (c >= 9 && c <= 13) || (c >= 0x1c && c <= 0x1f); }

struct Line {
  int64_t b, e, next;  // content [b, e) without the line break; start of the following line
};

struct Scanner {
  const uint8_t* buf;
  int64_t len;
  bool eof;
  int64_t nl = -1, cr = -1;  // next '\n' / '\r' at or after the last position asked about (len: none)

  int64_t find(uint8_t c, int64_t& cache, int64_t pos) const {
    if (cache < pos) {
      const void* q = memchr(buf + pos, c, (size_t)(len - pos));
      cache = q ? (const uint8_t*)q - buf : len;
    }
    return cache;
  }

  // Universal newlines: "\n", "\r\n" and a lone "\r" end a line.  1: the line and where the next one starts are known;
  // 0: they are not (no line break yet, or a '\r' as the last byte, which may be the first half of "\r\n");
  // -1: no line starts at pos.  At the end of the input the last line needs no line break.
  int line(int64_t pos, Line& L) {
    if (pos >= len) return -1;
    const int64_t a = find('\n', nl, pos), b = find('\r', cr, pos);
    const int64_t e = a < b ? a : b;
    L.b = pos;
    L.e = e;
    if (e == len) {
      L.next = len;
      return eof ? 1 : 0;
    }
    if (buf[e] == '\n') {
      L.next = e + 1;
      return 1;
    }
    if (e + 1 < len) {
      L.next = e + 1 + (buf[e + 1] == '\n');
      return 1;
    }
    L.next = len;
    return eof ? 1 : 0;
  }
};

bool has_non_ascii(const uint8_t* p, int64_t n) {
  int64_t i = 0;
  for (; i + 8 <= n; i += 8) {
    uint64_t w;
    memcpy(&w, p + i, 8);
    if (w & 0x8080808080808080ull) return true;
  }
  for (; i < n; ++i)
    if (p[i] & 0x80) return true;
  return false;
}

}  // namespace

extern "C" int cfk_seq_scan(const uint8_t* buf_h, int64_t len, int32_t at_eof, int64_t* records_h, int64_t max_records,
                            int64_t* pieces_h, int64_t max_pieces, int64_t* out_h) {
  if (len < 0 || max_records < 0 || max_pieces < 0 || out_h == nullptr || (len > 0 && buf_h == nullptr) ||
      (max_records > 0 && records_h == nullptr) || (max_pieces > 0 && pieces_h == nullptr)) {
    snprintf(cfk_g_err, sizeof(cfk_g_err), "cfk_seq_scan: bad arguments");
    return CFK_ERR_INVALID;
  }
  for (int i = 0; i < 5; ++i) out_h[i] = 0;
  if (has_non_ascii(buf_h, len)) {
    out_h[4] = CFK_SCAN_NOT_ASCII;
    return CFK_OK;
  }
  Scanner S{buf_h, len, at_eof != 0};
  int64_t pos = 0, consumed = 0, n_rec = 0, n_piece = 0, text = 0, flags = 0;
  Line L;
  for (;;) {
    int s = S.line(pos, L);
    if (s <= 0) break;
    const uint8_t c0 = buf_h[pos];
    if (L.e == L.b || (c0 != '>' && c0 != '@')) {  // not a header: skipped
      pos = consumed = L.next;
      continue;
    }
    if (n_rec == max_records) {
      flags |= CFK_SCAN_FULL;
      break;
    }
    // name = (line[1:].split() or [""])[0]
    int64_t nb = L.b + 1;
    while (nb < L.e && is_space(buf_h[nb])) ++nb;
    int64_t ne = nb;
    while (ne < L.e && !is_space(buf_h[ne])) ++ne;
    const int64_t first_piece = n_piece;
    int64_t seq_len = 0;
    bool complete = false, full = false;
    pos = L.next;
    for (;;) {
      s = S.line(pos, L);
      if (s < 0) {  // no further line: the record ends with the input
        complete = S.eof;
        break;
      }
      const uint8_t c = buf_h[pos];
      if (c == '>' || c == '@') {  // the next record's header
        complete = true;
        break;
      }
      if (s == 0) break;
      pos = L.next;
      if (c == '+') {  // quality: whole lines while fewer characters than bases have been skipped
        int64_t left = seq_len;
        complete = true;
        while (left > 0) {
          s = S.line(pos, L);
          if (s < 0) {
            complete = S.eof;
            break;
          }
          if (s == 0) {
            complete = false;
            break;
          }
          left -= L.e - L.b;
          pos = L.next;
        }
        break;
      }
      int64_t b = L.b, e = L.e;  // a sequence line, strip()ped
      while (b < e && is_space(buf_h[b])) ++b;
      while (e > b && is_space(buf_h[e - 1])) --e;
      if (e > b) {
        if (n_piece == max_pieces) {
          full = true;
          break;
        }
        int64_t* p = pieces_h + 3 * n_piece++;
        p[0] = b;
        p[1] = e - b;
        p[2] = seq_len;
        seq_len += e - b;
      }
    }
    if (!complete) {
      if (full) flags |= CFK_SCAN_FULL;
      n_piece = first_piece;
      break;
    }
    for (int64_t i = first_piece; i < n_piece; ++i) pieces_h[3 * i + 2] += text;
    int64_t* r = records_h + 4 * n_rec++;
    r[0] = nb;
    r[1] = ne - nb;
    r[2] = seq_len;
    r[3] = text;
    text += (seq_len + 15) & ~(int64_t)15;
    consumed = pos;
  }
  out_h[0] = n_rec;
  out_h[1] = n_piece;
  out_h[2] = consumed;
  out_h[3] = text;
  out_h[4] = flags;
  return CFK_OK;
}
