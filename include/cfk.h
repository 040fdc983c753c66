/*
 * cfk.h — C ABI of the B200-native unique-k-mer recruitment path ("cfk" = centroFlye k-mers).
 *
 * The reference (seryrzu/centroFlye @ b2a4378) has no FFI: this stage is pure Python
 * (scripts/distance_based_kmer_recruitment.py, scripts/read_kmer_cloud.py).  These entry
 * points are what a binding for that path has to call; each one names the reference
 * function (file:line under /root/reference/scripts) whose work it replaces.  The Python
 * drop-in modules in centroflye_b200/ bind them with ctypes (INTEGRATION.md shows the stub).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in _h; the caller (PyTorch)
 *     owns all memory, the library allocates nothing and keeps no state between calls;
 *   - `stream` is a cudaStream_t passed as void*; calls only enqueue work on it;
 *   - return 0 on success, negative CFK_ERR_* otherwise; cfk_last_error() returns a
 *     thread-local message for the last failing call on this host thread;
 *   - a k-mer is a uint64 with its first base in the most significant used bits
 *     (A=0 C=1 G=2 T=3), 1 <= k <= 31; 0xFFFF_FFFF_FFFF_FFFF marks an empty slot;
 *   - reads are 2-bit packed, 16 bases per little-endian uint32 (base j at bits 2j..2j+1);
 *     base offsets index that packed space; every read starts on a 64-base boundary;
 *   - overflow of a caller-sized buffer is never silent: kernels keep counting in the
 *     `counters` words documented per call and the host wrapper grows and retries.
 */
#ifndef CFK_H
#define CFK_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CFK_OK 0
#define CFK_ERR_INVALID (-1)
#define CFK_ERR_CUDA (-2)

#define CFK_EMPTY_KEY 0xFFFFFFFFFFFFFFFFull
#define CFK_DOCFREQ_SET_SLOTS 49152 /* 32-bit slots of the per-read k-mer set in shared memory (192 KB) */
#ifndef CFK_DOCFREQ_PART_DISTINCT
#define CFK_DOCFREQ_PART_DISTINCT 2304 /* distinct k-mers one unit (group of hash partitions) of the two-phase stage A holds at a time */
#endif
#ifndef CFK_PAIR_WARPS
#define CFK_PAIR_WARPS 20         /* warps per block of the stage-C kernel (one block per SM) */
#endif
#ifndef CFK_PAIR_TABLE_BYTES
#define CFK_PAIR_TABLE_BYTES 11264 /* shared-memory counting table of one warp (multiple of 16) */
#endif

#ifndef CFK_SKETCH_BITS
#define CFK_SKETCH_BITS 13        /* log2 of the byte counters in one warp's stage-C sketch (10..13) */
#endif
#ifndef CFK_SKETCH_LOAD_DIV
#define CFK_SKETCH_LOAD_DIV 4     /* a sketch pass is planned for <= 2^CFK_SKETCH_BITS / this many cloud entries */
#endif
#define CFK_SKETCH_MIN_COV 3      /* cfk_pair_sketch serves min_cov in [3, 255]; cfk_pair_candidates serves any */
#define CFK_SKETCH_MAX_COV 255

typedef void* cfk_stream_t;

int cfk_abi_version(void);
const char* cfk_last_error(void);
/* static shared-memory / launch geometry, for DESIGN.md and bench.py's launch accounting */
int cfk_pair_table_bytes_per_warp(void);
int cfk_pair_warps_per_block(void);
/* number of kernels this library has enqueued since it was loaded (bench.py: gpu_launches) */
int64_t cfk_launch_count(void);

/* ---- stage A: document-frequency k-mer count --------------------------------------------
 * The table is open addressing over `cap` 16-byte slots { uint64 key ; uint32 n_reads ;
 * uint32 n_multi } stored as 2 x uint64 per slot (counts in the second word, n_reads low);
 * cfk_table_init writes (CFK_EMPTY_KEY, 0) into every slot.
 *
 * cfk_docfreq_count replaces get_kmer_freqs_from_ncrf_report,
 * distance_based_kmer_recruitment.py:39-63: for every read r and every DISTINCT k-mer of its
 * gap-free row n_reads[kmer] += 1, and n_multi[kmer] += 1 if the k-mer occurs in r more than
 * once (the closed form of the sequential update at :55-62, SURVEY.md §8a3).  The per-read
 * de-duplication (the reference's read_freq dict, :50-53) is done in shared memory by one
 * persistent thread block per read; `order` lists the read indices longest first (load
 * balance), n_blocks = number of SMs.  Calling again with more reads accumulates.
 * counters (zeroed by the caller): [0] != 0: table full (results invalid, grow and retry),
 * [1] != 0: internal set overflow (a bug), [2] read cursor.
 */
int cfk_table_init(uint64_t* table, int64_t cap, cfk_stream_t stream);
int cfk_docfreq_count(const uint32_t* packed, const int64_t* read_off, const int64_t* read_len, const int32_t* order,
                      int64_t n_reads, int k, uint64_t* table, int64_t cap, int64_t* counters, int32_t n_blocks,
                      cfk_stream_t stream);

/* Resident form of cfk_docfreq_count (the default path; same results, same table, same counters).
 * The work item is one (read, pass): a pass is a hash partition of the read's k-mer space small
 * enough for the per-read set, and the whole packed read is staged in shared memory beside the
 * set (224 KB: [read words | set]), so the per-read de-duplication of
 * distance_based_kmer_recruitment.py:50-53 never leaves the SM and the passes of a long read
 * run on different SMs.  cfk_docfreq_plan writes n_pass[i] = passes of read order[i]; the caller
 * turns it into item_ptr[n_reads + 1] with cfk_exclusive_scan and hands that to
 * cfk_docfreq_count_resident.  Reads of more than ~655 kb keep their words in global memory. */
int cfk_docfreq_plan(const int64_t* read_len, const int32_t* order, int64_t n_reads, int k, int32_t* n_pass,
                     cfk_stream_t stream);
int cfk_docfreq_count_resident(const uint32_t* packed, const int64_t* read_off, const int64_t* read_len,
                               const int32_t* order, const int64_t* item_ptr, int64_t n_reads, int k, uint64_t* table,
                               int64_t cap, int64_t* counters, int32_t n_blocks, cfk_stream_t stream);

/* Two-phase form of stage A (the default path of the engine; same counts as cfk_docfreq_count).
 * Replaces get_kmer_freqs_from_ncrf_report, distance_based_kmer_recruitment.py:39-63, and the band of
 * get_rare_kmers, :74-79, in two kernels and without a global hash table:
 *   cfk_docfreq_emit         per (read, pass) item the per-read de-duplication of :50-53 runs in shared memory (the
 *                            read arrives by one cp.async.bulk copy; probes are issued from warp-private queues so
 *                            that every probe runs on a full warp) and ONE 8-byte record per distinct k-mer of the read -- bits 0..2k-1 the
 *                            k-mer in the order the packed read holds it (base j of the k-mer at bits 2j..2j+1; phase 2
 *                            turns the distinct k-mers into keys), bit 63 set if the k-mer occurs in the read more
 *                            than once (:55-56) -- is appended
 *                            to hash partition p = floor(hash32(kmer) * n_parts / 2^32):
 *                            records[p * part_cap + i], i < cursors[p].
 *   cfk_docfreq_count_parts  one block per partition adds the records up in a shared-memory table (n_reads += 1,
 *                            n_multi += bit 63: :57-62 in closed form).  The partition's counts are final when its
 *                            block ends, so the filter of get_rare_kmers runs in the same kernel: k-mers with
 *                            n_multi <= max_nonuniq and lo <= n_reads <= hi go to rare_keys[] (+ rare_nreads[],
 *                            rare_nmulti[] when given), unordered, counters[4] = how many (may exceed max_rare:
 *                            nothing is written past it, the caller retries with more room).  dense != NULL: every
 *                            distinct k-mer is also written as a 16-byte table slot { key ; n_reads | n_multi << 32 }
 *                            without empty slots (a table for cfk_table_select / cfk_table_part_*), counters[5] =
 *                            how many (counted with or without dense).  `group` neighbouring partitions (= one
 *                            wider hash range) are counted as one unit when their distinct k-mers fit the block's
 *                            tables (CFK_DOCFREQ_PART_DISTINCT); a unit that does not fit is taken again partition by
 *                            partition (counters[6] counts those), so any group >= 1 gives the same results.
 *                            Records of one partition may come from n_src sources (the ranks of the
 *                            multi-GPU exchange): source s holds records[s * src_stride + p * part_cap + i],
 *                            i < cursors[s * n_parts + p]; or, with offsets != NULL, dense runs
 *                            records[offsets[s * n_parts + p] + i] (what the exchange delivers: cfk_records_pack
 *                            lays a rank's partitions back to back, out[offsets[p] + i], before the all-to-all).
 * cfk_docfreq_emit_plan writes n_pass[i] = passes of read order[i] (-> item_ptr by cfk_exclusive_scan).
 * cfk_docfreq_part_target() = k-mer occurrences to plan per partition (n_parts = ceil(occurrences / target)); a
 * partition may receive any number of records.  One with more distinct k-mers than a table holds
 * (CFK_DOCFREQ_PART_DISTINCT planned, CFK_DOCFREQ_PART_DISTINCT * 4 / 3 slots) is counted again by halves of its hash
 * range, then quarters, ... down to 64 sub-ranges; only a partition that does not fit even then sets counters[0].
 * A k-mer may be in at most 65536 reads (more sets counters[0] too).
 * cursors[] and counters[8] are zeroed by the caller.  counters[0] != 0: a partition buffer (emit) or a
 * partition's table / 16-bit extra-read counter (count) overflowed -- results invalid, the caller falls back to
 * cfk_docfreq_count_resident; [1] != 0 internal error; [2], [3] work tickets.  The shared-memory sets claim empty
 * slots with atomicCAS (a k-mer is in a set exactly once); everything else is plain loads and stores. */
int cfk_records_pack(const uint64_t* records, int64_t part_cap, const uint32_t* cursors, const int64_t* offsets,
                     int64_t n_parts, uint64_t* out, cfk_stream_t stream);
int cfk_docfreq_part_target(void);
int cfk_docfreq_part_distinct(void); /* CFK_DOCFREQ_PART_DISTINCT of the built library */
int cfk_docfreq_emit_plan(const int64_t* read_len, const int32_t* order, int64_t n_reads, int k, int32_t* n_pass,
                          cfk_stream_t stream);
int cfk_docfreq_emit(const uint32_t* packed, const int64_t* read_off, const int64_t* read_len, const int32_t* order,
                     const int64_t* item_ptr, int64_t n_reads, int k, uint64_t* records, int64_t part_cap,
                     int64_t n_parts, uint32_t* cursors, int64_t* counters, int32_t n_blocks, cfk_stream_t stream);
int cfk_docfreq_count_parts(const uint64_t* records, int64_t part_cap, const uint32_t* cursors, const int64_t* offsets,
                            int64_t n_parts, int32_t n_src, int64_t src_stride, int32_t group, int k, uint32_t lo, uint32_t hi,
                            uint32_t max_nonuniq, uint64_t* rare_keys, uint32_t* rare_nreads, uint32_t* rare_nmulti,
                            int64_t max_rare, uint64_t* dense, int64_t max_dense, int64_t* counters, int32_t n_blocks,
                            cfk_stream_t stream);

/* Total-occurrence count (SURVEY.md §8f rank 3): replaces get_kmer_counts_reads,
 * scripts/better_consensus_unit_reconstruction.py:127-135 -- every k-mer occurrence of every gap-free read row adds 1
 * (no per-read de-duplication).  Same table as cfk_docfreq_count; the count lands in the n_reads field, n_multi stays
 * 0.  The k-mer starts of the reads are cut into tiles of cfk_kmer_count_tile() positions: tile_read[t] = read of
 * tile t, tile_start[t] = its first k-mer start inside that read.  counters[0] != 0: table full. */
int cfk_kmer_count_tile(void);
int cfk_kmer_count_total(const uint32_t* packed, const int64_t* read_off, const int64_t* read_len, const int32_t* tile_read,
                         const int64_t* tile_start, int64_t n_tiles, int k, uint64_t* table, int64_t cap, int64_t* counters,
                         cfk_stream_t stream);

/* The same count with the two strands of a k-mer merged (SURVEY.md §8f rank 3, second half): what tandemQUAST gets from
 * `jellyfish count -m K -C` on the reads, scripts/ext/tandemQUAST/scripts/select_kmers.py:131-133 -- every k-mer
 * occurrence adds 1 to its CANONICAL form, the smaller of the k-mer and its reverse complement (A < C < G < T). */
int cfk_kmer_count_canonical(const uint32_t* packed, const int64_t* read_off, const int64_t* read_len, const int32_t* tile_read,
                             const int64_t* tile_start, int64_t n_tiles, int k, uint64_t* table, int64_t cap,
                             int64_t* counters, cfk_stream_t stream);

/* ---- repetitive k-mers of one sequence (SURVEY.md §8f rank 4) -----------------------------------
 * Replaces get_repetitive_kmers + get_convolution, scripts/unit_extractor.py:23-40.  `packed` = the sequence 2-bit packed
 * from base 0 (readable up to word n_bases / 16 + 2).  cfk_kmer_position_keys writes one key per k-mer start,
 * k-mer << pos_bits | position; after cfk_sort_u64 the occurrences of a k-mer are neighbours in position order (the
 * lists of :25-27) and cfk_adjacent_gaps gives gaps[i] = position(i) - position(i - 1) inside a k-mer's run, 0 at its
 * first occurrence (the differences of :36). */
int cfk_kmer_position_keys(const uint32_t* packed, int64_t n_bases, int k, int pos_bits, uint64_t* keys, cfk_stream_t stream);
int cfk_adjacent_gaps(const uint64_t* keys, int64_t n, int pos_bits, uint32_t* gaps, cfk_stream_t stream);

/* ---- read recruitment pre-filter (SURVEY.md §8f rank 4, second half) ---------------------------------
 * Replaces the two edlibAlign(unit / reverse complement, read, k = threshold, EDLIB_MODE_HW, EDLIB_TASK_DISTANCE) calls
 * of scripts/read_recruitment/rr.cpp:73-90: out_keep[r] = 1 when the best edit distance of the whole unit against any
 * infix of read r, on either strand, is <= threshold (threshold < 0: no limit, as edlib's k = -1).  Bit-parallel
 * (Myers / Hyyro) on 64-bit words, one thread per (read, strand).
 *   text      all reads as bytes, every read on a 16-byte boundary, 16 readable bytes behind the last one
 *   peq       [2 strands][cfk_rr_max_symbols()][cfk_rr_words(m)] match masks: bit i of word w of symbol s = the unit
 *             (strand 0) / its reverse complement (strand 1) has symbol s at base 64 w + i; symbol slot 0 = all zero
 *   sym_of    [256] byte -> symbol slot (0 for bytes the unit does not contain: they match nothing, as in edlib)
 *   out_dist  NULL, or [2 * n_reads]: the best distance seen per (read, strand) -- the exact infix distance when
 *             exact != 0, otherwise the first value <= threshold (the scan of a strand stops there)
 * out_keep is zeroed by the caller.  Units of up to 3328 bases. */
int cfk_rr_max_symbols(void);
int cfk_rr_words(int32_t m);
int cfk_rr_filter(const uint8_t* text, const int64_t* read_off, const int64_t* read_len, const int32_t* order, int64_t n_reads,
                  const uint64_t* peq, const uint8_t* sym_of, int32_t m, int32_t threshold, int32_t exact, int32_t* out_dist,
                  uint8_t* out_keep, cfk_stream_t stream);

/* cfk_rr_filter for U units at once over the same reads (read_recruitment.recruit_file_units): out_keep[u * n_seg + r]
 * = 1 iff unit u, or its reverse complement, occurs in read r within unit_threshold[u] edits (< 0: no limit).
 *   peq             each unit's [2][cfk_rr_max_symbols()][cfk_rr_words(unit_m[u])] block (cfk_rr_filter's layout), the
 *                   blocks of units 0 .. U-1 one after another
 *   sym_of          [U][256], one symbol table per unit
 *   unit_m, unit_threshold   HOST int32[U]; they are passed to the kernels by value
 *   out_keep        [U][n_seg], zeroed by the caller
 * Every unit_m is checked (1..3328) before anything is launched.  One launch per word class present (more for a
 * class of more than 64 units), all on `stream`.  The scan of a strand stops early as in cfk_rr_filter (no exact
 * distances). */
int cfk_rr_filter_units(const uint8_t* text, const int64_t* seg_off, const int64_t* seg_len, const int32_t* order, int64_t n_seg,
                        int32_t n_units, const uint64_t* peq, const uint8_t* sym_of, const int32_t* unit_m,
                        const int32_t* unit_threshold, uint8_t* out_keep, cfk_stream_t stream);

/* Units of 1..32768 bases (read_recruitment.recruit, and the streaming form with long_units, take this for units over
 * 3328 bases): one warp per (segment, strand), the unit's 64-bit words split over the 32 lanes, W consecutive words per lane;
 * cfk_rr_long_words(m) = the least W of {2, 4, 8, 16} with ceil(ceil(m / 64) / W) <= 32, or -1 outside 1..32768.
 *   peq             each unit's [2][cfk_rr_max_symbols()][W][32] block, lane-minor: entry [strand][s][k][L] is word
 *                   L * W + k of cfk_rr_filter's masks (zero past the unit), the blocks of units 0 .. U-1 one after
 *                   another
 *   sym_of          [U][256], one symbol table per unit
 *   unit_m, unit_threshold   HOST int32[U]
 *   out_dist        NULL, or [U][2 * n_seg]: as cfk_rr_filter's out_dist, per unit
 *   out_keep        [U][n_seg], zeroed by the caller
 * Every size and unit_m is checked before anything is launched.  One launch per W present (more for a W of more than
 * 64 units), all on `stream`.  exact != 0 never stops early, as in cfk_rr_filter; the distances and keep bits are
 * those of cfk_rr_filter for every unit both take. */
int cfk_rr_long_words(int32_t m);
int cfk_rr_filter_long(const uint8_t* text, const int64_t* seg_off, const int64_t* seg_len, const int32_t* order, int64_t n_seg,
                       int32_t n_units, const uint64_t* peq, const uint8_t* sym_of, const int32_t* unit_m,
                       const int32_t* unit_threshold, int32_t exact, int32_t* out_dist, uint8_t* out_keep,
                       cfk_stream_t stream);

/* ---- streaming read recruitment: read file text in, output file text out ---------------------------------------
 * cfk_seq_scan (HOST code) finds the records of one chunk of FASTA / FASTQ text exactly as read_sequences() yields them
 * (centroflye_b200/read_recruitment.py:29-55, the restatement of rr.cpp's kseq_read loop): "\n", "\r\n" and a lone "\r"
 * end a line; lines before a header ('>' or '@') are skipped; the name is the header after its first byte up to the
 * first whitespace (str.isspace on ASCII), after leading whitespace; sequence lines, each stripped of whitespace at
 * both ends, run until a line starting with '>', '@' or '+'; after '+' whole lines are skipped while fewer quality
 * characters than bases have been.  It writes
 *   records_h [n][4]   name offset in buf_h, name length, sequence length, sequence offset in the packed text (every
 *                      sequence on a 16-byte boundary, text_bytes in all), for every complete record;
 *   pieces_h  [n][3]   source offset in buf_h, length, destination offset in the packed text, per non-empty stripped
 *                      sequence line of those records, in order;
 *   out_h     [5]      n_records, n_pieces, consumed, text_bytes, flags.
 * `consumed` is where the first incomplete record (or unfinished line) begins: the caller carries buf_h[consumed:] into
 * the next chunk.  Without at_eof a record ending with the chunk is incomplete, and so is a '\r' as its last byte.  The
 * scan stops before a record that does not fit max_records / max_pieces (flag CFK_SCAN_FULL).  A byte >= 0x80 anywhere
 * in the chunk sets CFK_SCAN_NOT_ASCII and nothing else: str semantics differ from byte semantics there.
 *
 * The device part, on the chunk copied to the device as it is (raw):
 *   cfk_rr_gather      text[pieces[p][2] + i] = raw[pieces[p][0] + i]; 0 elsewhere; text 16-byte aligned, text_bytes a
 *                      multiple of 16 -> the text cfk_rr_filter reads;
 *   cfk_rr_keep_sizes  sizes[r] = bytes of ">name\nsequence\n" if any of the segments seg_keep[seg_ptr[r] ..
 *                      seg_ptr[r + 1]) of record r hit (seg_keep = cfk_rr_filter's out_keep over segments), else 0;
 *                      seg_keep = seg_ptr = NULL keeps every record -> out_off by cfk_exclusive_scan;
 *   cfk_rr_emit        out[out_off[r] ..] = ">name\nsequence\n" of every kept record, names from raw, sequences from
 *                      text; bytes at or beyond max_bytes are not written (launch size: max_bytes / 16 threads). */
#define CFK_SCAN_NOT_ASCII 1
#define CFK_SCAN_FULL 2
int cfk_seq_scan(const uint8_t* buf_h, int64_t len, int32_t at_eof, int64_t* records_h, int64_t max_records,
                 int64_t* pieces_h, int64_t max_pieces, int64_t* out_h);
int cfk_rr_gather(const uint8_t* raw, const int64_t* pieces, int64_t n_pieces, uint8_t* text, int64_t text_bytes,
                  cfk_stream_t stream);
int cfk_rr_keep_sizes(const uint8_t* seg_keep, const int64_t* seg_ptr, const int64_t* records, int64_t n_records,
                      int32_t* sizes, cfk_stream_t stream);
int cfk_rr_emit(const uint8_t* raw, const uint8_t* text, const int64_t* records, const int64_t* out_off, int64_t n_records,
                int64_t max_bytes, uint8_t* out, cfk_stream_t stream);

/* ---- compressed read files: BGZF blocks inflated on the device, unaligned BAM ----------------------------------
 * cfk_bgzf_blocks (HOST code) walks the gzip members (RFC 1952 headers: FLG, the XLEN subfields searched for "BC",
 * FNAME, FCOMMENT, FHCRC) of buf_h[0..len) and writes one row per complete BGZF block:
 *   blocks_h [n][5]    payload offset in buf_h, payload length (the raw DEFLATE data), ISIZE, CRC32, output offset
 *                      (the exclusive scan of ISIZE from 0);
 *   out_h    [4]       n_blocks, consumed, inflated bytes of the rows, flags.
 * Zero bytes between and after members are skipped.  The walk stops after max_blocks rows; before a member that ends
 * past len (CFK_BGZF_INCOMPLETE); and before one that is not BGZF -- no "BC" subfield, an ISIZE above 65536, a header
 * that does not fit BSIZE, or bytes that are no gzip member at all (CFK_BGZF_NOT_BGZF).  `consumed` is where it
 * stopped.
 *
 * cfk_bgzf_inflate inflates the rows (offsets into comp, on the device) into out[row[4] ..] and writes status[i]:
 * CFK_BGZF_OK, CFK_BGZF_BAD_STREAM (not a DEFLATE stream that ends with the payload, or a back-reference before the
 * block's start), CFK_BGZF_BAD_LENGTH (the stream yields more or fewer than ISIZE bytes) or CFK_BGZF_BAD_CRC.  All of
 * RFC 1951; every member starts with an empty window.  ISIZE must be at most 65536.
 *
 * cfk_bam_scan (HOST code) finds the records of one chunk of inflated BAM (SAM spec §4.2).  With `header` the chunk
 * starts at the stream's beginning and the header (magic, text, references) is skipped first; if it is not complete
 * nothing is consumed.  Secondary and supplementary alignments (flag & 0x900) are consumed and yield nothing.  It
 * writes, for every other complete record,
 *   records_h [n][4]   as cfk_seq_scan's: name offset in buf_h, name length, l_seq, 16-byte aligned text offset;
 *   bam_seq_h [n][2]   offset in buf_h of the 4-bit SEQ, 1 if the record is reverse-complemented (flag & 0x10);
 *   out_h     [5]      n_records, records consumed (every alignment), consumed, text_bytes, flags (CFK_SCAN_FULL).
 * Every record is validated (block_size, l_read_name, l_seq, fields within block_size, a NUL-terminated name of
 * '!'..'~'); an invalid record, or at_eof with a record or header cut off, fails naming the record's index
 * (first_index + records before it) and its offset in the inflated stream (stream_offset + offset in buf_h).
 *
 * cfk_rr_bam_gather writes the text cfk_rr_gather writes for FASTA / FASTQ: record r's SEQ decoded through
 * "=ACMGRSVTWYHKDBN" (reversed and complemented where flagged) at records[r][3], 0 elsewhere. */
#define CFK_BGZF_INCOMPLETE 1
#define CFK_BGZF_NOT_BGZF 2
#define CFK_BGZF_OK 0
#define CFK_BGZF_BAD_STREAM 1
#define CFK_BGZF_BAD_LENGTH 2
#define CFK_BGZF_BAD_CRC 3
int cfk_bgzf_blocks(const uint8_t* buf_h, int64_t len, int64_t* blocks_h, int64_t max_blocks, int64_t* out_h);
int cfk_bgzf_inflate(const uint8_t* comp, const int64_t* blocks, int64_t n_blocks, uint8_t* out, int32_t* status,
                     cfk_stream_t stream);
int cfk_bam_scan(const uint8_t* buf_h, int64_t len, int32_t at_eof, int32_t header, int64_t first_index,
                 int64_t stream_offset, int64_t* records_h, int64_t max_records, int64_t* bam_seq_h, int64_t* out_h);
int cfk_rr_bam_gather(const uint8_t* raw, const int64_t* bam_seq, const int64_t* records, int64_t n_records, uint8_t* text,
                      int64_t text_bytes, cfk_stream_t stream);

/* ---- read_placer scoring on the cloud CSR (SURVEY.md §8f rank 2) --------------------------------
 * Replaces the data structures of ReadPlacer.add_reads, scripts/read_placer.py:42-94, and of CloudContig.add_read /
 * update_mapping_scores, scripts/cloud_contig.py:26-41,87-95; the greedy loop (one read per iteration) stays on the
 * host (centroflye_b200/read_placer.py).  All tables are caller-allocated, keys initialised to CFK_EMPTY_KEY, values 0.
 *   cfk_placer_add_read       clouds[position + i][kmer] += 1 for the units u0 .. u0 + n_units - 1 of one read
 *                             (cloud_contig.py:30-35) in the table contig_keys/contig_cnt keyed position << 32 | id;
 *                             a (k-mer, position) whose counter reaches min_freq is appended to pairs[] as (id, position)
 *                             (new_freq_kmers, :36-39) and marks freq_flag[id].  n_entries_max >= the read's cloud entries.
 *   cfk_placer_initial_pairs  the list add_reads starts from (read_placer.py:54-57): every position of every k-mer
 *                             with freq_flag set.
 *   cfk_placer_update         update_mapping_scores (cloud_contig.py:87-95) for pairs[0 .. pair_counters[0]): every
 *                             occurrence (unit g of read r = unit_read[g], position g - read_first_unit[r]) of the k-mer
 *                             in a read with read_sel[r] and contig position >= position adds to the score of
 *                             (r, contig position - position): m1 = set of (r, offset, position), m2[(r, offset)] =
 *                             distinct positions << 32 | total -- (len(score), sum(score.values())) of :66-67.
 *   cfk_placer_best           the selection of read_placer.py:61-79: one candidate per block (cfk_placer_best_blocks()
 *                             blocks, 3 x uint64 each: score ; offset | rank << 32 ; read), 0 score = none.
 * counters[0] = pairs appended, counters[1] != 0: a table or pairs[] is full (the caller grows and repeats). */
int cfk_placer_best_blocks(void);
int cfk_placer_add_read(const int64_t* unit_ptr, const uint32_t* ids, int64_t u0, int32_t n_units, int64_t n_entries_max,
                        int64_t position, uint32_t min_freq, uint64_t* contig_keys, uint32_t* contig_cnt, int64_t cap,
                        uint8_t* freq_flag, uint32_t* pairs, int64_t max_pairs, int64_t* counters, cfk_stream_t stream);
int cfk_placer_initial_pairs(const uint64_t* contig_keys, int64_t cap, const uint8_t* freq_flag, uint32_t* pairs,
                             int64_t max_pairs, int64_t* counters, cfk_stream_t stream);
int cfk_placer_update(const uint32_t* pairs, const int64_t* pair_counters, int64_t max_pairs, const int64_t* occ_ptr,
                      const uint32_t* occ, const int32_t* unit_read, const int64_t* read_first_unit, const uint8_t* read_sel,
                      uint64_t* m1_keys, int64_t cap1, uint64_t* m2_keys, uint64_t* m2_val, int64_t cap2, int64_t* counters,
                      cfk_stream_t stream);
int cfk_placer_best(const uint64_t* m2_keys, const uint64_t* m2_val, int64_t cap2, const uint8_t* read_unused,
                    const uint32_t* read_rank, uint32_t min_unit, uint32_t min_inters, uint32_t min_prop, uint64_t* out,
                    cfk_stream_t stream);

/* Merge (key, n_reads, n_multi) records counted elsewhere (another GPU's shard) into a table:
 * the owner-side half of the multi-GPU all-to-all (SURVEY.md §8e).  counters[0] != 0: full. */
int cfk_table_merge(const uint64_t* keys, const uint32_t* nreads, const uint32_t* nmulti, int64_t n, uint64_t* table,
                    int64_t cap, int64_t* counters, cfk_stream_t stream);

/* ---- band filter -------------------------------------------------------------------------
 * Replaces the dict comprehension of get_rare_kmers, distance_based_kmer_recruitment.py:77-79,
 * and (lo = 0, hi = UINT32_MAX) the survivor rule of :58-62.  Stream-compacts every occupied
 * slot with n_multi <= max_nonuniq and lo <= n_reads <= hi into out_keys / out_nreads /
 * out_nmulti (any may be NULL).  If n_parts > 0 only keys with mix(key) % n_parts == part are
 * taken (hash partition for the multi-GPU exchange).  counters[0] (zeroed by the caller)
 * receives the number of matches even beyond max_out; nothing is written past max_out.
 */
int cfk_table_select(const uint64_t* table, int64_t cap, uint32_t lo, uint32_t hi, uint32_t max_nonuniq, int32_t n_parts,
                     int32_t part, uint64_t* out_keys, uint32_t* out_nreads, uint32_t* out_nmulti, int64_t max_out,
                     int64_t* counters, cfk_stream_t stream);

/* (n_reads, n_multi) of n given keys, 0 / 0 for keys the table does not hold: the per-rank half of the multi-GPU
 * "nominate, then sum" exchange (DESIGN.md section 5): only k-mers that reach ceil(lo / G) reads on SOME rank can reach
 * lo reads in total, so only those are looked up on every rank and summed. */
int cfk_table_lookup(const uint64_t* table, int64_t cap, const uint64_t* keys, int64_t n, uint32_t* out_nreads,
                     uint32_t* out_nmulti, cfk_stream_t stream);

/* Hash partition of a whole table for the multi-GPU exchange (SURVEY.md §8e): every occupied
 * slot goes to partition owner(key) = mix64(key ^ 0x9E3779B97F4A7C15) % n_parts (the rule
 * cfk_table_select applies), n_parts <= 64.  cfk_table_part_count adds the partition sizes to
 * counts[n_parts] (zeroed by the caller); cfk_table_part_scatter writes the records so that
 * partition p occupies [cursors[p], cursors[p] + count[p]) of the output arrays -- cursors
 * holds the exclusive prefix of the counts on entry and the end offsets on return.  This is the
 * send buffer layout of the NCCL all-to-all; the receiver feeds cfk_table_merge. */
int cfk_table_part_count(const uint64_t* table, int64_t cap, int32_t n_parts, int64_t* counts, cfk_stream_t stream);
int cfk_table_part_scatter(const uint64_t* table, int64_t cap, int32_t n_parts, int64_t* cursors, uint64_t* out_keys,
                           uint32_t* out_nreads, uint32_t* out_nmulti, cfk_stream_t stream);

/* In-place ascending sort of n uint64 keys (bitonic network, shared-memory tiles).  The rank
 * of a k-mer in the sorted rare set is its integer id everywhere downstream (the reference's
 * kmer_index, distance_based_kmer_recruitment.py:103, canonicalised). */
int cfk_sort_u64(uint64_t* keys, int64_t n, cfk_stream_t stream);
/* n_runs sorted runs of pairwise DISTINCT keys, back to back (run j = keys[run_ptr[j] .. run_ptr[j + 1]), run_ptr[n_runs] =
 * n on the device) -> out[0 .. n) sorted: the all-gathered, per-rank sorted rare keys of the multi-GPU path. */
int cfk_merge_sorted_runs(const uint64_t* keys, const int64_t* run_ptr, int32_t n_runs, int64_t n, uint64_t* out,
                          cfk_stream_t stream);

/* Static probe table over the sorted rare keys: key -> rank.  idx_keys pre-filled with
 * CFK_EMPTY_KEY; cap >= 2 n recommended. */
int cfk_index_build(const uint64_t* sorted_keys, int64_t n, uint64_t* idx_keys, uint32_t* idx_vals, int64_t cap,
                    int64_t* counters, cfk_stream_t stream);

/* ---- stage B: per-unit k-mer clouds ------------------------------------------------------
 * Replaces ReadKMerCloud.fromNCRF_record, read_kmer_cloud.py:18-31: for unit u (bases
 * [unit_off[u], unit_off[u] + unit_len[u]) of the packed stream) the SET of indexed k-mers
 * lying wholly inside it, as sorted unique ids written to tmp_ids[unit_kbase[u] ...] with
 * their number in unit_cnt[u].  unit_kbase = exclusive prefix of max(unit_len - k + 1, 0).
 */
int cfk_cloud_build(const uint32_t* packed, const int64_t* unit_off, const int32_t* unit_len,
                    const int64_t* unit_kbase, int64_t n_units, int k,
                    const uint64_t* idx_keys, const uint32_t* idx_vals, int64_t cap,
                    const uint32_t* filter, int32_t filter_bits,
                    uint32_t* tmp_ids, int32_t* unit_cnt, cfk_stream_t stream);
/* Optional pre-filter of cfk_cloud_build for an index that does not fit L2 (the rare set of several GPUs): a bitmap of
 * 2^filter_bits bits (zeroed by the caller), bit mix64(key) >> (64 - filter_bits) set for every key.  A clear bit
 * proves "not in the set"; a set bit sends the k-mer to the index as before, so results do not depend on it.
 * filter = NULL: every k-mer probes the index. */
int cfk_index_filter_build(const uint64_t* sorted_keys, int64_t n, int32_t filter_bits, uint32_t* filter, cfk_stream_t stream);
/* out[0] = 0, out[i + 1] = in[0] + ... + in[i]  (int32 -> int64); scratch holds
 * cfk_scan_scratch_elems(n) int64. */
int64_t cfk_scan_scratch_elems(int64_t n);
int cfk_exclusive_scan(const int32_t* in, int64_t* out, int64_t n, int64_t* scratch, cfk_stream_t stream);
/* Gather the per-unit id runs into CSR: ids[unit_ptr[u] + i] = tmp_ids[unit_kbase[u] + i]. */
int cfk_cloud_compact(const uint32_t* tmp_ids, const int64_t* unit_kbase, const int64_t* unit_ptr,
                      int64_t n_units, uint32_t* ids, cfk_stream_t stream);

/* ---- cloud multiplicity filter -----------------------------------------------------------
 * Replaces filter_reads_kmer_clouds, read_kmer_cloud.py:43-54.  mult[id] = number of
 * (read, unit) clouds of units [unit_lo, unit_hi) containing id (mult zeroed by the caller). */
int cfk_id_histogram(const int64_t* unit_ptr, const uint32_t* ids, int64_t unit_lo, int64_t unit_hi,
                     int32_t* mult, cfk_stream_t stream);
/* new_cnt[u] = number of ids of unit u with min_mult <= mult[id] <= max_mult. */
int cfk_cloud_filter_count(const int64_t* unit_ptr, const uint32_t* ids, int64_t n_units, const int32_t* mult,
                           int64_t min_mult, int64_t max_mult, int32_t* new_cnt, cfk_stream_t stream);
int cfk_cloud_filter_write(const int64_t* unit_ptr, const uint32_t* ids, int64_t n_units, const int32_t* mult,
                           int64_t min_mult, int64_t max_mult, const int64_t* new_ptr, uint32_t* new_ids,
                           cfk_stream_t stream);

/* ---- stage C/D: unit-distance k-mer pair graph -------------------------------------------
 * Occurrence lists (the inverted cloud CSR): occ[occ_ptr[a] ...] = sorted global unit indices
 * whose cloud contains id a.  occ_ptr = exclusive scan of the cfk_id_histogram output (int64[n_kmers + 1],
 * occ_ptr[n_kmers] < 2^32); cursor = uint32[n_kmers] of scratch (any contents). */
int cfk_occ_fill(const int64_t* unit_ptr, const uint32_t* ids, int64_t unit_lo, int64_t unit_hi,
                 const int64_t* occ_ptr, int64_t n_kmers, uint32_t* cursor, uint32_t* occ, cfk_stream_t stream);
int cfk_occ_sort(const int64_t* occ_ptr, uint32_t* occ, int64_t n_kmers, cfk_stream_t stream);
/* The same inversion for the ids of [id_lo, id_hi) only, over all n_units units (multi-GPU: rank r inverts its 1/G of the
 * id space of the all-gathered clouds, the lists are all-gathered in rank order = id order).  mult (zeroed by the
 * caller), occ_ptr (exclusive scan of mult, int64[id_hi - id_lo + 1]) and cursor (scratch) are indexed by id - id_lo;
 * the lists inside a unit must be sorted (they are: cfk_cloud_build).  cfk_occ_sort then sorts the slice's lists. */
int cfk_occ_slice_histogram(const int64_t* unit_ptr, const uint32_t* ids, int64_t n_units, int64_t id_lo, int64_t id_hi,
                            int32_t* mult, cfk_stream_t stream);
int cfk_occ_slice_fill(const int64_t* unit_ptr, const uint32_t* ids, int64_t n_units, int64_t id_lo, int64_t id_hi,
                       const int64_t* occ_ptr, uint32_t* cursor, uint32_t* occ, cfk_stream_t stream);
/* occ_last[i] = unit_last[occ[i]]: the last unit of the read of every occurrence, laid out like occ
 * itself, so that cfk_pair_sketch / cfk_pair_join stream it instead of chasing unit_last[g]. */
int cfk_occ_last(const uint32_t* occ, int64_t n, const uint32_t* unit_last, uint32_t* occ_last, cfk_stream_t stream);

/* usplit[7 u + j - 1] (j = 1..7) = position in ids[] of the first id of unit u that is
 * >= (n_kmers * j) >> 3: the per-unit octant split table cfk_pair_candidates uses to cut a unit
 * list by id range without searching (uint32[7 n_units]; n_entries < 2^32). */
int cfk_unit_splits(const int64_t* unit_ptr, const uint32_t* ids, int64_t n_units, int64_t n_entries, int64_t n_kmers,
                    uint32_t* usplit, cfk_stream_t stream);

/* Replaces the counting loop of get_kmer_dist_map, distance_based_kmer_recruitment.py:111-127,
 * fused with the candidate pass of filter_dist_tuples (:133-138).  The reference keeps one
 * counter per (d, a, b); here every source id a (a_begin, a_begin + a_stride, ... < a_end) is
 * handled by one warp that cuts the distances [max(min_d,1), max_d] into chunks [d0, d1]
 * (d1 - d0 <= 30), sums  sum_{d in chunk} cnt[d][a][b]  in a warp-private shared-memory table and
 * emits the pair candidate (a, b, d0, d1) as 4 x uint32 whenever that sum reaches min_cov -- a
 * necessary condition for cnt[d][a][b] >= min_cov at some d of the chunk.  Every (a, b, d)
 * belongs to exactly one emitted or rejected chunk, so cfk_pair_join sees each possible edge once.
 * unit_last[g] = index of the last unit of g's read; usplit = cfk_unit_splits output or NULL
 * (binary search instead); n_entries = unit_ptr[n_units] must be < 2^32.
 * counters (zeroed by the caller): [0] candidates found (also beyond max_cand; nothing is
 * written past max_cand), [1] dynamic work cursor, [2] pair increments (the reference's number
 * of `+= 1` executions at :126, in closed form), [3] table overflows that forced a smaller chunk.
 */
int cfk_pair_candidates(const int64_t* unit_ptr, const uint32_t* ids, const uint32_t* unit_last,
                        const int64_t* occ_ptr, const uint32_t* occ, const uint32_t* usplit, int64_t n_entries,
                        int64_t n_kmers, int64_t a_begin, int64_t a_end, int32_t a_stride,
                        int32_t min_d, int32_t max_d, uint32_t min_cov,
                        uint32_t* cand, int64_t max_cand, int64_t* counters, int32_t n_blocks, cfk_stream_t stream);

/* The same contract as cfk_pair_candidates (same reference lines, same counters, same
 * (a, b, d0, d1) output consumed by cfk_pair_join) for CFK_SKETCH_MIN_COV <= min_cov <=
 * CFK_SKETCH_MAX_COV, an order of magnitude cheaper: instead of exact per-(a, b) counters a warp
 * keeps 2^CFK_SKETCH_BITS saturating byte counters indexed by a hash of b -- an upper bound of
 * sum_d cnt[d][a][b] -- and only ids whose counter reaches min_cov enter a small exact set that
 * is emitted.  The emitted pairs are a SUPERSET of the pairs whose chunk total reaches min_cov;
 * cfk_pair_join computes the exact counts either way, so the edges are identical.
 * codes = cfk_sketch_codes output, a buffer of cfk_sketch_codes_elems(n_entries, n_units) uint16
 * (8-byte aligned) private to these two functions: per cloud entry the hash of its id (low
 * CFK_SKETCH_BITS bits) and, in bit 15, whether another id of the same unit with the same hash
 * precedes it, stored in 128-entry blocks per unit so that a lane fetches the four entries it
 * serves in a step with one 8-byte load (the tail of a unit's last block is padding).
 * (cfk_pair_sketch's occ_last: see below.) */
int cfk_sketch_bits(void);
int cfk_sketch_warps_per_block(void);
int64_t cfk_sketch_codes_elems(int64_t n_entries, int64_t n_units);
/* perm_ids (optional, uint32[cfk_sketch_codes_elems], 16-byte aligned, elems < 2^32): bank-aware placement.  The
 * entries of every 128-entry block are reordered so that the byte counters a row of 32 lanes touches lie in 32
 * different shared-memory banks wherever the block allows it (lane = bank, row = rank among the block's entries of
 * that bank; overflow fills the free slots of the last rows), and perm_ids receives the id behind every code slot.
 * NULL keeps the ids' own order.  Pass the same pointer (or NULL) to cfk_pair_sketch. */
int cfk_sketch_codes(const int64_t* unit_ptr, const uint32_t* ids, int64_t n_units, uint16_t* codes, uint32_t* perm_ids,
                     cfk_stream_t stream);
/* occ_last = cfk_occ_last output, or NULL (unit_last[g] is looked up instead).
 * Output layout: every warp fills its own chunks of 256 candidate slots (one atomic on the cursor per chunk instead
 * of one per pass); the unused tail of a chunk holds holes, a = 0xFFFFFFFF, which cfk_pair_join skips.  counters[0] is
 * therefore the number of SLOTS handed out (size cand for it, plus a chunk per warp when retrying), counters[4] the
 * number of candidates among them. */
int cfk_pair_sketch(const int64_t* unit_ptr, const uint32_t* ids, const uint16_t* codes, const uint32_t* perm_ids,
                    const uint32_t* unit_last,
                    const int64_t* occ_ptr, const uint32_t* occ, const uint32_t* occ_last, int64_t n_entries, int64_t n_kmers, int64_t a_begin,
                    int64_t a_end, int32_t a_stride, int32_t min_d, int32_t max_d, uint32_t min_cov,
                    uint32_t* cand, int64_t max_cand, int64_t* counters, int32_t n_blocks, cfk_stream_t stream);

/* Replaces both loops of filter_dist_tuples, distance_based_kmer_recruitment.py:131-149, for
 * the pair candidates: joins the occurrence lists of a and b to get the exact cnt[d][a][b] for
 * every d in [d0, d1] and all_occ = sum over d' in [max(min_d,1), max_d] of cnt[d'][a][b];
 * keeps (a, b, d, cnt) iff cnt >= min_cov and (double)cnt / (double)all_occ >= rel_threshold
 * (IEEE double division, the operation Python performs at :145), appends it to edges and flags
 * both endpoints in selected[] (uint8, zeroed by the caller).
 * counters (zeroed): [0] edges found (also beyond max_edges; nothing is written past
 * max_edges), [2] number of (a, b, d) with cnt >= min_cov (the reference's candidate dict).
 * occ_last = cfk_occ_last output, or NULL. */
int cfk_pair_join(const uint32_t* cand, int64_t n_cand, const int64_t* occ_ptr, const uint32_t* occ, const uint32_t* occ_last,
                  const uint32_t* unit_last, int32_t min_d, int32_t max_d, uint32_t min_cov, double rel_threshold,
                  uint32_t* edges, int64_t max_edges, uint8_t* selected, int64_t* counters, cfk_stream_t stream);

/* Indices of non-zero flags, ascending (the recruited k-mer ids).  counters[0] zeroed. */
int cfk_flag_indices(const uint8_t* flags, int64_t n, uint32_t* out, int64_t* counters, cfk_stream_t stream);

/* ---- native NCRF ingestion (host code; SURVEY.md §8f rank 1) --------------------------------
 * One pass from the report text to the flat host arrays the device consumes, replacing the
 * per-record Python of NCRF_Report.__init__ (scripts/ncrf_parser.py:61-118: 2-line records, '#'
 * and blank lines dropped, longest alignment per read id kept if r_al_len >= min_record_len,
 * '-' strand rows reverse-complemented with utils/bio.py:27-29), of the gap removal in
 * distance_based_kmer_recruitment.py:47 / read_kmer_cloud.py:25, and of the unit segmentation
 * get_motif_alignments(n) (scripts/ncrf_parser.py:28-59: non-overlapping leftmost matches of
 * motif * n in the gap-free upper-cased motif row, partial first / last unit kept when longer
 * than 0.2 * len(motif)).  All pointers are HOST pointers (numpy / pinned torch buffers).
 *
 * cfk_ncrf_open parses, selects and segments (n_threads <= 0: all cores) into an opaque context;
 * the size queries tell the caller how much to allocate; cfk_ncrf_export writes
 *   packed_h[n_words]        2-bit packed gap-free reads, every read on a 64-base boundary,
 *   read_off_h / read_len_h [n_records],  read_unit_ptr_h [n_records + 1],
 *   unit_off_h / unit_len_h / unit_read_h [n_units]   (may be NULL),
 *   ids_h [ids_bytes]        record ids in dict order, '\n' after each        (may be NULL),
 *   fields_h [8 * n_records] r_len, r_al_len, r_st, r_en, strand (+1 / -1), m_al_len, score,
 *                            alignment columns                               (may be NULL);
 * a symbol outside upper-case ACGT in a read row is an error (CFK_ERR_INVALID), as in the Python
 * host path.  cfk_ncrf_close frees the context.  Errors: cfk_ncrf_last_error(). */
typedef struct cfk_ncrf cfk_ncrf_t;
const char* cfk_ncrf_last_error(void);
int cfk_ncrf_open(const char* path, int64_t min_record_len, int32_t n_per_match, int32_t n_threads, cfk_ncrf_t** out);
int64_t cfk_ncrf_n_records(const cfk_ncrf_t* ctx);
int64_t cfk_ncrf_n_seen(const cfk_ncrf_t* ctx);
int64_t cfk_ncrf_n_words(const cfk_ncrf_t* ctx);
int64_t cfk_ncrf_n_bases(const cfk_ncrf_t* ctx);
int64_t cfk_ncrf_n_units(const cfk_ncrf_t* ctx);
int64_t cfk_ncrf_ids_bytes(const cfk_ncrf_t* ctx);
int cfk_ncrf_export(const cfk_ncrf_t* ctx, uint32_t* packed_h, int64_t* read_off_h, int64_t* read_len_h,
                    int64_t* read_unit_ptr_h, int64_t* unit_off_h, int32_t* unit_len_h, int32_t* unit_read_h,
                    char* ids_h, int64_t* fields_h);
void cfk_ncrf_close(cfk_ncrf_t* ctx);

/* ---- native result writer (host code; SURVEY.md §8 row a9) ------------------------------------
 * Writes the edge file of output_results, distance_based_kmer_recruitment.py:165-171: one line
 * "{dist} {kmer_i} {kmer_j} {cnt}\n" per edge, k-mers decoded from keys_sorted_h[id] (id = rank in the sorted rare
 * set), formatted by n_threads host threads (<= 0: all cores) and written in the given order; byte-identical to the
 * Python writer.  All pointers are HOST pointers; ids outside [0, n_keys) are an error. */
const char* cfk_writer_last_error(void);
int cfk_write_edges(const char* path, const uint64_t* keys_sorted_h, int64_t n_keys, int32_t k, const int64_t* dist_h,
                    const int64_t* i_h, const int64_t* j_h, const int64_t* freq_h, int64_t n_edges, int32_t n_threads);
/* The same file from the rows cfk_pair_join writes, copied to the host as they are: rows_h = uint32[n_edges][4] =
 * (i, j, dist, cnt).  Spares the caller four strided int64 column copies (80 ms for 8e6 edges). */
int cfk_write_edges_rows(const char* path, const uint64_t* keys_sorted_h, int64_t n_keys, int32_t k, const uint32_t* rows_h,
                         int64_t n_edges, int32_t n_threads);

#ifdef __cplusplus
}
#endif
#endif /* CFK_H */
