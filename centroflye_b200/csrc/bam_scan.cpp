// bam_scan.cpp — host scanners of the compressed inputs of the streaming read recruitment filter.
//
// cfk_bgzf_blocks walks the gzip member headers of a BGZF file (SAM spec §4.1) and lists its blocks for the device
// inflater (bgzf.cu) without inflating anything.  cfk_bam_scan finds the records of a chunk of inflated BAM (SAM spec
// §4.2) in cfk_seq_scan's record layout, so the device gathers, filters and emits them as it does FASTA / FASTQ.
// Neither call keeps state: the caller carries the bytes from `consumed` on into the next buffer.
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/cfk.h"

extern thread_local char cfk_g_err[512];  // cfk_last_error() (cfk.cu)

namespace {

inline uint32_t u16(const uint8_t* p) { return p[0] | ((uint32_t)p[1] << 8); }
inline uint32_t u32(const uint8_t* p) { return p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }
inline int32_t i32(const uint8_t* p) { return (int32_t)u32(p); }

enum Member { MEMBER_OK, MEMBER_INCOMPLETE, MEMBER_NOT_BGZF };

// The gzip member (RFC 1952) at buf[p..len): a BGZF block has FEXTRA with a "BC" subfield of two bytes (BSIZE).
Member parse_member(const uint8_t* buf, int64_t len, int64_t p, int64_t* row) {
  const int64_t have = len - p;
  static const uint8_t magic[3] = {0x1f, 0x8b, 8};
  for (int i = 0; i < 3; ++i)
    if (i < have && buf[p + i] != magic[i]) return MEMBER_NOT_BGZF;
  if (have > 3 && ((buf[p + 3] & 0xe0) || !(buf[p + 3] & 4))) return MEMBER_NOT_BGZF;  // reserved bits, or no extra field
  if (have < 12) return MEMBER_INCOMPLETE;
  const uint8_t flg = buf[p + 3];
  const int64_t xlen = u16(buf + p + 10), x0 = p + 12, x1 = x0 + xlen;
  if (x1 > len) return MEMBER_INCOMPLETE;
  int64_t bsize = -1;
  for (int64_t q = x0; q + 4 <= x1;) {
    const int64_t slen = u16(buf + q + 2);
    if (q + 4 + slen > x1) return MEMBER_NOT_BGZF;
    if (buf[q] == 'B' && buf[q + 1] == 'C' && slen == 2) bsize = u16(buf + q + 4);
    q += 4 + slen;
  }
  if (bsize < 0) return MEMBER_NOT_BGZF;
  const int64_t end = p + bsize + 1;  // BSIZE is the member's size minus one
  if (end - 8 < x1) return MEMBER_NOT_BGZF;
  if (end > len) return MEMBER_INCOMPLETE;
  int64_t h = x1;
  for (int f = 8; f <= 16; f <<= 1)  // FNAME, FCOMMENT: zero-terminated strings
    if (flg & f) {
      const void* z = memchr(buf + h, 0, (size_t)(end - 8 - h > 0 ? end - 8 - h : 0));
      if (z == nullptr) return MEMBER_NOT_BGZF;
      h = (const uint8_t*)z - buf + 1;
    }
  if (flg & 2) h += 2;  // FHCRC
  if (h > end - 8) return MEMBER_NOT_BGZF;
  const uint32_t isize = u32(buf + end - 4);
  if (isize > 65536) return MEMBER_NOT_BGZF;
  row[0] = h;
  row[1] = end - 8 - h;
  row[2] = isize;
  row[3] = u32(buf + end - 8);
  return MEMBER_OK;
}

}  // namespace

extern "C" int cfk_bgzf_blocks(const uint8_t* buf_h, int64_t len, int64_t* blocks_h, int64_t max_blocks, int64_t* out_h) {
  if (len < 0 || max_blocks < 0 || out_h == nullptr || (len > 0 && buf_h == nullptr) ||
      (max_blocks > 0 && blocks_h == nullptr)) {
    snprintf(cfk_g_err, sizeof(cfk_g_err), "cfk_bgzf_blocks: bad arguments");
    return CFK_ERR_INVALID;
  }
  int64_t p = 0, n = 0, total = 0, flags = 0;
  for (;;) {
    while (p < len && buf_h[p] == 0) ++p;  // zero padding between and after members, as gzip readers skip it
    if (p == len || n == max_blocks) break;
    int64_t* row = blocks_h + 5 * n;
    const Member m = parse_member(buf_h, len, p, row);
    if (m != MEMBER_OK) {
      flags |= m == MEMBER_INCOMPLETE ? CFK_BGZF_INCOMPLETE : CFK_BGZF_NOT_BGZF;
      break;
    }
    row[4] = total;
    total += row[2];
    p = row[0] + row[1] + 8;  // the member's end
    ++n;
  }
  out_h[0] = n;
  out_h[1] = p;
  out_h[2] = total;
  out_h[3] = flags;
  return CFK_OK;
}

namespace {

int bam_error(int64_t index, int64_t offset, const char* what) {
  snprintf(cfk_g_err, sizeof(cfk_g_err), "cfk_bam_scan: BAM record %lld at offset %lld of the inflated stream: %s",
           (long long)index, (long long)offset, what);
  return CFK_ERR_INVALID;
}

// the header (magic, l_text, text, n_ref, references) at buf[0..len): its size, 0 if it is not complete, -1 if bad
int64_t bam_header(const uint8_t* buf, int64_t len) {
  if (len < 8) return 0;
  if (memcmp(buf, "BAM\1", 4) != 0) return -1;
  const int32_t l_text = i32(buf + 4);
  if (l_text < 0) return -1;
  int64_t p = 8 + (int64_t)l_text;
  if (p + 4 > len) return 0;
  const int32_t n_ref = i32(buf + p);
  if (n_ref < 0) return -1;
  p += 4;
  for (int32_t i = 0; i < n_ref; ++i) {
    if (p + 4 > len) return 0;
    const int32_t l_name = i32(buf + p);
    if (l_name < 0) return -1;
    p += 4 + (int64_t)l_name + 4;
    if (p > len) return 0;
  }
  return p;
}

}  // namespace

extern "C" int cfk_bam_scan(const uint8_t* buf_h, int64_t len, int32_t at_eof, int32_t header, int64_t first_index,
                            int64_t stream_offset, int64_t* records_h, int64_t max_records, int64_t* bam_seq_h,
                            int64_t* out_h) {
  if (len < 0 || max_records < 0 || out_h == nullptr || (len > 0 && buf_h == nullptr) ||
      (max_records > 0 && (records_h == nullptr || bam_seq_h == nullptr))) {
    snprintf(cfk_g_err, sizeof(cfk_g_err), "cfk_bam_scan: bad arguments");
    return CFK_ERR_INVALID;
  }
  for (int i = 0; i < 5; ++i) out_h[i] = 0;
  int64_t p = 0;
  if (header) {
    p = bam_header(buf_h, len);
    if (p < 0) {
      snprintf(cfk_g_err, sizeof(cfk_g_err), "cfk_bam_scan: the BAM header is malformed");
      return CFK_ERR_INVALID;
    }
    if (p == 0) {
      if (at_eof) {
        snprintf(cfk_g_err, sizeof(cfk_g_err), "cfk_bam_scan: the BAM file ends inside its header");
        return CFK_ERR_INVALID;
      }
      return CFK_OK;  // the caller grows the chunk
    }
  }
  int64_t n_rec = 0, n_aln = 0, text = 0, flags = 0;
  char msg[160];
  for (;;) {
    if (p == len) break;
    const int64_t index = first_index + n_aln, off = stream_offset + p;
    if (len - p < 4) {
      if (at_eof) return bam_error(index, off, "the file ends inside the record");
      break;
    }
    const int32_t block_size = i32(buf_h + p);
    if (block_size < 32) {
      snprintf(msg, sizeof(msg), "block_size %d is below the 32 fixed bytes", block_size);
      return bam_error(index, off, msg);
    }
    if (len - p - 4 < block_size) {
      if (at_eof) return bam_error(index, off, "the file ends inside the record");
      break;
    }
    const uint8_t* r = buf_h + p + 4;
    const int64_t l_read_name = r[8], n_cigar_op = u16(r + 12), flag = u16(r + 14), l_seq = i32(r + 16);
    if (l_read_name == 0) return bam_error(index, off, "l_read_name is 0");
    if (l_seq < 0) return bam_error(index, off, "l_seq is negative");
    const int64_t name = 32, cigar = name + l_read_name, seq = cigar + 4 * n_cigar_op, qual = seq + (l_seq + 1) / 2,
                  end = qual + l_seq;
    const char* past = cigar > block_size ? "read_name" : seq > block_size ? "cigar" : qual > block_size ? "seq"
                       : end > block_size ? "qual" : nullptr;
    if (past != nullptr) {
      snprintf(msg, sizeof(msg), "the %s field runs past block_size %d", past, block_size);
      return bam_error(index, off, msg);
    }
    if (r[cigar - 1] != 0) return bam_error(index, off, "read_name is not NUL-terminated");
    for (int64_t i = name; i < cigar - 1; ++i)
      if (r[i] < '!' || r[i] > '~') {
        snprintf(msg, sizeof(msg), "read_name byte 0x%02x is outside '!'..'~'", r[i]);
        return bam_error(index, off, msg);
      }
    if (!(flag & 0x900)) {  // secondary and supplementary alignments yield nothing
      if (n_rec == max_records) {
        flags |= CFK_SCAN_FULL;
        break;
      }
      int64_t* rec = records_h + 4 * n_rec;
      rec[0] = p + 4 + name;
      rec[1] = l_read_name - 1;
      rec[2] = l_seq;
      rec[3] = text;
      bam_seq_h[2 * n_rec] = p + 4 + seq;
      bam_seq_h[2 * n_rec + 1] = (flag & 0x10) != 0;
      ++n_rec;
      text += (l_seq + 15) & ~(int64_t)15;
    }
    ++n_aln;
    p += 4 + (int64_t)block_size;
  }
  out_h[0] = n_rec;
  out_h[1] = n_aln;
  out_h[2] = p;
  out_h[3] = text;
  out_h[4] = flags;
  return CFK_OK;
}
