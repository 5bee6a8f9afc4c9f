/*
 * nmb200.h -- C ABI of libnmb200.so, the B200 (sm_100a) data plane for nanomotif's
 * motif-scoring hot path.
 *
 * The reference (MicrobialDarkMatter/nanomotif 1.1.2) is pure Python and has no FFI of its
 * own; the operator boundary is a set of Python callables (SURVEY.md section 8b).  Each entry
 * point below names the reference callable(s) whose arithmetic it replaces.  The Python mirror
 * of the reference API (nanomotif_b200/api.py) binds these with ctypes; INTEGRATION.md shows
 * the stub a nanomotif maintainer would add.
 *
 * Conventions
 *   - every function returns 0 on success or a negative nmb_status; it never throws and never
 *     aborts.  nmb_last_error() returns a thread-local message for the last failure.
 *   - all pointers are DEVICE pointers unless the parameter name ends in _h.
 *   - the caller owns every buffer; nothing is allocated behind the caller's back except the
 *     small per-call scratch documented at the function.
 *   - functions enqueue work on `stream` (a cudaStream_t passed as void*) and return without
 *     synchronising; they keep no global state, so N host threads/processes can drive N GPUs.
 *   - no torch / C++ types cross the boundary.
 *
 * Packed layout ("tile records", described in DESIGN.md section 3)
 *   The assembly lives in one global position space.  Contig c occupies positions
 *   [start_c, start_c + len_c), start_c a multiple of NMB_CHUNK_BP (512); consecutive contigs are
 *   separated by >= NMB_MIN_GAP_BP positions flagged non-ACGT.  The space is cut into tiles of
 *   NMB_TILE_BP (65536) positions.  Per tile t:
 *     seq record  : uint32 x[NMB_TILE_WORDS+8], y[NMB_TILE_WORDS+8], int32 chunk_info[128]
 *                   x = high code bit, y = low code bit (A=0 T=1 G=2 C=3, nanomotif/constants.py:1);
 *                   4 halo words of the neighbouring tiles are duplicated on each side (natural
 *                   order) so that one bulk copy (TMA) brings a self-contained tile into shared memory.
 *                   The 2048 body words of a plane are LANE-INTERLEAVED: word w of the tile (chunk
 *                   t = w/16, word j = w%16 of the chunk) is stored at slot NMB_WORD_SLOT(w) =
 *                   (j/4)*512 + t*4 + j%4, so that the 128 lanes of a CTA, each owning one chunk, read
 *                   consecutive 16-byte vectors (bank-conflict-free LDS.128, coalesced LDG.128).
 *                   chunk_info[q] = contig id (< 2^28) of 512-bp chunk q, -1 for an empty chunk; bit 30
 *                   set when the chunk or a neighbouring chunk holds a non-ACGT letter of a contig,
 *                   else bit 29 set when the chunk or its two halo words touch inter-contig padding
 *                   (bit 28: the chunk itself holds a non-ACGT letter).
 *     class record: uint32 plane[4][NMB_TILE_WORDS] per mod type, each plane lane-interleaved as above:
 *                   0 = methylated '+', 1 = unmethylated '+', 2 = methylated '-', 3 = unmethylated '-'
 *                   (fraction_mod >= high / <= low, nanomotif/find_motifs_bin.py:1308-1314).
 *   The non-ACGT plane is a flat uint32 array with 4 leading pad words.
 */
#ifndef NMB200_H
#define NMB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NMB_ABI_VERSION 10 /* 2: lane-interleaved tile records (NMB_WORD_SLOT), chunk_info flag bits 28-30; 3: table ingest; 4: nmb_pack_motifs; 5: per-bin sweep slots; 6: degenerate bipartite sweep; 7: sweep candidate pruning; 8: one sweep entry point per filter and histogram kind (slots and prune as arguments); 9: nmb_sweep_lookup, motif counts gathered from the finished sweep histograms; 10: sibling runs (nmb_compile_motifs_siblings, nmb_scan_count_siblings) replace the family finder */

#if defined(__GNUC__)
#define NMB_API __attribute__((visibility("default")))
#else
#define NMB_API
#endif

#define NMB_CHUNK_WORDS 16
#define NMB_CHUNK_BP 512
#define NMB_TILE_WORDS 2048
#define NMB_TILE_BP 65536
#define NMB_TILE_CHUNKS 128
#define NMB_HALO_WORDS 4
#define NMB_SEQ_PLANE_WORDS (NMB_TILE_WORDS + 2 * NMB_HALO_WORDS)           /* 2056 */
#define NMB_SEQ_REC_WORDS (2 * NMB_SEQ_PLANE_WORDS + NMB_TILE_CHUNKS)       /* 4240 */
#define NMB_CLS_REC_WORDS (4 * NMB_TILE_WORDS)                              /* 8192 */
/* slot of tile word w (0..2047) inside a lane-interleaved plane */
#define NMB_WORD_SLOT(w) ((((w) & 12) << 7) | (((w) >> 4) << 2) | ((w) & 3))
#define NMB_MIN_GAP_BP 64
#define NMB_MAX_MOTIF_LEN 62
#define NMB_MAX_WINDOW 61
#define NMB_MAX_MOTIFS_PER_ITEM 32

typedef enum nmb_status {
    NMB_OK = 0,
    NMB_ERR_INVALID = -1, /* bad argument */
    NMB_ERR_CUDA = -2,    /* CUDA runtime error, see nmb_last_error() */
    NMB_ERR_NO_DEVICE = -3,
    NMB_ERR_CAPACITY = -4 /* caller-provided output too small */
} nmb_status;

/* One motif, already stripped of flanking wildcards (nanomotif/motif.py:213-224).
 * allowed[j] is the set of bases accepted at motif position j: bit0=A bit1=T bit2=G bit3=C
 * (order of nanomotif/constants.py:21-28); 0xF is the regex wildcard '.', which is the only
 * thing a non-ACGT contig letter matches (regex-literal semantics, nanomotif/utils.py:61-66). */
typedef struct nmb_motif {
    uint8_t allowed[NMB_MAX_MOTIF_LEN];
    uint8_t len;     /* 1..NMB_MAX_MOTIF_LEN */
    uint8_t mod_pos; /* 0..len-1 */
} nmb_motif; /* 64 bytes */

/* Device view of a packed assembly (all device pointers). */
typedef struct nmb_assembly {
    const uint32_t *seq_records;   /* [n_tiles][NMB_SEQ_REC_WORDS] */
    const uint32_t *nonacgt;       /* [NMB_HALO_WORDS + n_tiles*NMB_TILE_WORDS + NMB_HALO_WORDS] */
    const int64_t *contig_start;   /* [n_contigs] global start position (multiple of 512) */
    const int64_t *contig_len;     /* [n_contigs] */
    int32_t n_contigs;
    int32_t n_tiles;
} nmb_assembly;

/* One homogeneous unit of scan work: motifs [motif_begin, motif_begin+motif_count) of one
 * mod type against tiles [tile_begin, tile_begin+tile_count), counting only contigs
 * [contig_begin, contig_end).  Output row of (motif m, group g) is
 *     out[(out_base + (m - motif_begin) * n_groups + g) * 4 + {0: n_mod '+', 1: n_nomod '+',
 *                                                           2: n_mod '-', 3: n_nomod '-'}]
 * group_mode 0: g = 0 (one posterior per motif: motif_model_bin, find_motifs_bin.py:1265-1283)
 *            1: g = contig - contig_begin (one row per contig: motif_model_contig / the table)
 *            2: g = contig_group[contig], negative = contig skipped. */
typedef struct nmb_job {
    int32_t motif_begin;
    int32_t motif_count;
    int32_t modtype;
    int32_t tile_begin;
    int32_t tile_count;
    int32_t contig_begin;
    int32_t contig_end;
    int32_t group_mode;
    int32_t n_groups;
    int32_t item_offset; /* exclusive prefix sum of tile_count*ceil(motif_count/motifs_per_item) */
    int64_t out_base;
} nmb_job; /* 48 bytes */

NMB_API int nmb_abi_version(void);
NMB_API const char *nmb_last_error(void);
/* Number of SMs of the current device (grid sizing), or negative status. */
NMB_API int nmb_device_sm_count(void);

/* ---- K1: loaders (replaces nanomotif/fasta.py:35-49 + nanomotif/seq.py:53-55 string storage,
 *      and the per-call polars splits of nanomotif/find_motifs_bin.py:1308-1314) ---- */

/* ASCII contigs (concatenated in `ascii`, contig c at byte offset ascii_off[c], length
 * contig_len[c], any case) -> tile records + non-ACGT plane.  Buffers must be sized as in
 * nmb_assembly; they are fully overwritten. */
NMB_API int nmb_pack_sequence(const uint8_t *ascii, const int64_t *ascii_off, const int64_t *contig_start,
                      const int64_t *contig_len, int32_t n_contigs, int32_t n_tiles,
                      uint32_t *seq_records, uint32_t *nonacgt, void *stream);

/* Pileup rows -> class records.  Row r belongs to contig contig_id[r] (negative = ignored),
 * 0-based forward-strand position pos[r], strand[r] (0 '+', 1 '-'), mod type index modtype[r]
 * (NULL = all rows are type 0), fraction_mod[r] (= column 11 / 100, nanomotif/dataload.py:85).
 * A row is methylated iff fraction >= high and unmethylated iff fraction <= low, compared in
 * float64 exactly like the reference.  class_records [n_modtypes][n_tiles][4][NMB_TILE_WORDS] is
 * zeroed first.  Rows must be unique per (contig, pos, strand, modtype) -- the reference's
 * np.isin(assume_unique=True) makes the same assumption (find_motifs_bin.py:1258-1261). */
NMB_API int nmb_build_class_planes(const int32_t *contig_id, const int64_t *pos, const uint8_t *strand,
                           const uint8_t *modtype, const double *fraction_mod, int64_t n_rows,
                           double low, double high, const nmb_assembly *assembly_h,
                           int32_t n_modtypes, uint32_t *class_records, void *stream);

/* nmb_build_class_planes without the clear: ORs the rows into existing records (several tables, e.g. one per
 * (bin, mod_type) as nanomotif partitions its pileup, find_motifs_bin.py:416).  *dup_count (device int64, may be
 * NULL; ADDED to) counts rows whose class bit was already set, i.e. rows that repeat a (contig, pos, strand,
 * modtype): the reference counts such rows twice (np.isin keeps duplicates), bit-planes cannot. */
NMB_API int nmb_add_class_planes(const int32_t *contig_id, const int64_t *pos, const uint8_t *strand,
                                 const uint8_t *modtype, const double *fraction_mod, int64_t n_rows, double low,
                                 double high, const nmb_assembly *assembly_h, int32_t n_modtypes,
                                 uint32_t *class_records, int64_t *dup_count, void *stream);

/* Same class records from COMPACT rows (7 bytes per row instead of 22 over PCIe): pos int32, flags =
 * strand | mod type index << 1, percent_x100 = modkit's two-decimal percentage as an exact integer key
 * (0..10000).  Rows are grouped by contig: rows of contig c are [contig_row_off[c], contig_row_off[c+1]).
 * A row is methylated iff key >= key_high and unmethylated iff key <= key_low, where the keys are the
 * integer images of the reference's float64 tests fl(fl(key/100)/100) >= high / <= low computed by the
 * caller over the 10001 grid values (nanomotif_b200.device.threshold_keys) -- bit-equivalent to
 * nmb_build_class_planes on pileups whose column 11 has two decimals.  A key above 10000 (nmb_bed_parse's
 * 0xFFFF: not on the grid, or not a number) puts the row in neither class. */
NMB_API int nmb_build_class_planes_compact(const int32_t *pos, const uint8_t *flags, const uint16_t *percent_x100,
                                   const int64_t *contig_row_off, int64_t n_rows, int32_t key_low,
                                   int32_t key_high, const nmb_assembly *assembly_h, int32_t n_modtypes,
                                   uint32_t *class_records, void *stream);

/* Block-wise variant for loaders that stream the pileup: nmb_clear_class_planes zeroes the records once,
 * nmb_add_class_planes_compact ORs one block of compact rows into them (same arguments and semantics as
 * nmb_build_class_planes_compact, which is clear + add).  Blocks may arrive in any order and on copies that
 * overlap earlier blocks' scans; a mod type's planes are complete once every block holding its rows is in. */
NMB_API int nmb_clear_class_planes(const nmb_assembly *assembly_h, int32_t n_modtypes, uint32_t *class_records,
                                   void *stream);
NMB_API int nmb_add_class_planes_compact(const int32_t *pos, const uint8_t *flags, const uint16_t *percent_x100,
                                         const int64_t *contig_row_off, int64_t n_rows, int32_t key_low,
                                         int32_t key_high, const nmb_assembly *assembly_h, int32_t n_modtypes,
                                         uint32_t *class_records, void *stream);

/* ---- K6: modkit bedMethyl text -> pileup columns on the device (replaces the CSV scan of
 *      nanomotif/dataload.py:72-100 and the row materialisation of epymetheus.query_pileup_records,
 *      dataload.py:109-120) ---- */

/* Ascending positions i with src[i] == value (e.g. '\n').  Two-call pattern like
 * nmb_compact_positions: capacity 0 only counts (*n_out, device int64); scratch holds
 * ceil(n_bytes/4096)+1 int64. */
NMB_API int nmb_index_bytes(const uint8_t *src, int64_t n_bytes, int32_t value, int64_t *scratch,
                            int64_t *out_index, int64_t capacity, int64_t *n_out, void *stream);

/* One row per text line (line r starts at newline_pos[r-1]+1, line 0 at 0; a final line without '\n'
 * counts; '\r' ends a line too).  Columns (1-based, tab separated, dataload.py:15-34): 1 contig name ->
 * contig_id through the table (hash = FNV-1a 64 of the name, ascending; ids; name bytes by rank), -1 when
 * unknown, -2 for an empty or malformed (< 18 fields) line; 2 -> position; 4 -> mod_type = index of the
 * code in modtype_keys (the code's bytes, first byte most significant, <= 8 bytes) or 255; 6 -> strand 0
 * '+', 1 '-', 2 other; 10 -> n_valid_cov; 11 -> fraction_mod = value/100 (dataload.py:85; value = the
 * correctly rounded double of the decimal text) and percent_x100 = the exact two-decimal key 0..10000 or
 * 0xFFFF when the text has more decimals or is out of range; 12 -> n_mod, 17 -> n_diff (outputs may be
 * NULL).  Fields that are not plain decimal numbers (NA, null, exponents) give -1 / NaN.  status[4]
 * (device int32) counts malformed lines, empty lines, non-numeric fields, rows of unknown contigs. */
NMB_API int nmb_bed_parse(const uint8_t *text, int64_t n_bytes, const int64_t *newline_pos, int64_t n_lines,
                          const uint64_t *contig_hash, const int32_t *contig_ids, const int64_t *contig_name_off,
                          const uint8_t *contig_names, int32_t n_contigs, const uint64_t *modtype_keys,
                          int32_t n_modtypes, int32_t *contig_id, int64_t *position, uint8_t *strand,
                          uint8_t *mod_type, int64_t *n_valid_cov, double *fraction_mod, uint16_t *percent_x100,
                          int64_t *n_mod, int64_t *n_diff, int32_t *status, void *stream);

/* String column of a host TABLE (the frames nanomotif hands to its workers, find_motifs_bin.py:399-427: contig,
 * strand and mod_type are polars Utf8 columns, i.e. Arrow utf8 / large_utf8 buffers) -> ids on the device.
 * Row r's string is data[offsets[r] .. offsets[r+1]) with 4- or 8-byte offsets (offset_bytes); it is looked up
 * in a name table laid out as for nmb_bed_parse (FNV-1a 64 hashes ascending, ids, name bytes by rank) and
 * out[r] = its id, or `missing`.  out is int32 (out_bytes 4) or uint8 (out_bytes 1). */
NMB_API int nmb_lookup_strings(const uint8_t *data, const void *offsets, int32_t offset_bytes, int64_t n_rows,
                               const uint64_t *name_hash, const int32_t *name_ids, const int64_t *name_off,
                               const uint8_t *names, int32_t n_names, int32_t missing, void *out, int32_t out_bytes,
                               void *stream);

/* ---- K7: BGZF inflate (bgzip-compressed pileups, docs/source/required_files.md:21; the reference reads them
 *      through epymetheus.query_pileup_records / bgzf_pileup, dataload.py:109-120) ----
 * Block b holds block_in_len[b] bytes of raw DEFLATE data at comp + block_in_off[b] (after its gzip header) and
 * inflates to exactly block_out_len[b] bytes (its ISIZE) at out + block_out_off[b]; block_crc32 (may be NULL)
 * is the CRC-32 of the inflated bytes.  One warp per block, blocks are independent.  status[b] = 0 or the
 * first error (1 block type, 2 stored header, 3 code lengths, 4 symbol, 5 distance, 6 output overflow,
 * 7 input overrun, 8 size mismatch, 9 CRC mismatch). */
NMB_API int nmb_bgzf_inflate(const uint8_t *comp, const int64_t *block_in_off, const int32_t *block_in_len,
                             const int64_t *block_out_off, const int32_t *block_out_len,
                             const uint32_t *block_crc32, int32_t n_blocks, uint8_t *out, int32_t *status,
                             void *stream);

/* FASTA text on the device (replaces the host parse of nanomotif/fasta.py:35-49 load_fasta_fastx): lines as in
 * nmb_bed_parse (newline index from nmb_index_bytes; n_lines = n_newlines + 1 when the text does not end with a
 * newline); blanks and '\r' at both ends of a line are stripped.  nmb_fasta_lines: kind[r] = 1 for a header line
 * ('>'), payload[r] = bytes nmb_fasta_copy will write for line r -- the sequence bytes of sequence lines
 * (want_headers = 0) or the header text after '>' (want_headers = 1).  nmb_fasta_copy writes each line's payload at
 * out + out_off[r] (out_off = exclusive scan of payload, nmb_exclusive_scan_i64).  Contig k = the sequence lines
 * between header k and header k + 1; case is kept (nmb_pack_sequence upper-cases). */
NMB_API int nmb_fasta_lines(const uint8_t *text, int64_t n_bytes, const int64_t *newline_pos, int64_t n_newlines,
                            int64_t n_lines, int32_t want_headers, uint8_t *kind, int64_t *payload, void *stream);
NMB_API int nmb_fasta_copy(const uint8_t *text, int64_t n_bytes, const int64_t *newline_pos, int64_t n_newlines,
                           int64_t n_lines, int32_t want_headers, const int64_t *out_off, uint8_t *out, void *stream);
/* In-place exclusive prefix sum of n int64 (one block); *total (device) = the sum. */
NMB_API int nmb_exclusive_scan_i64(int64_t *values, int64_t n, int64_t *total, void *stream);

/* dst[i] = src[index[i]] for elements of 1, 2, 4 or 8 bytes (row compaction after the filters). */
NMB_API int nmb_gather_rows(const void *src, int32_t elem_bytes, const int64_t *index, int64_t n, void *dst,
                            void *stream);

/* ---- pileup filters (replace the polars expressions of nanomotif/dataload.py:191-247); every
 *      function writes keep[r] in {0,1} in input row order ---- */

/* filter_pileup (dataload.py:191-200): keep rows with Nvalid_cov > min_coverage (strict). */
NMB_API int nmb_filter_coverage(const int64_t *n_valid_cov, int64_t n_rows, int64_t min_coverage, uint8_t *keep,
                        void *stream);

/* filter_pileup_minimummod_frequency (dataload.py:202-226): group_id[r] identifies the row's
 * (contig, mod_type) pair (dense ids 0..n_groups-1); a group is kept when more than
 * min_mods_pr_contig of its rows have fraction > methylation_threshold and that count divided by the
 * group's row count exceeds min_mod_frequency.  group_counts: scratch of 2*n_groups int64 (returned
 * holding [rows, rows above threshold] per group). */
NMB_API int nmb_filter_min_mod_frequency(const int32_t *group_id, const double *fraction_mod, int64_t n_rows,
                                 int32_t n_groups, double methylation_threshold, double min_mod_frequency,
                                 int64_t min_mods_pr_contig, int64_t *group_counts, uint8_t *keep,
                                 void *stream);

/* filter_pileup_adjacency_filter (dataload.py:228-247): a row is kept when its fraction is below the
 * threshold or equals the maximum fraction over the rows of the same (contig, strand) -- any mod
 * type -- whose position lies within +-adjacency_distance.  Rows must be sorted by (contig_id, pos);
 * *unsorted_flag (device int32) is set to 1 when they are not (the keep mask is then meaningless). */
NMB_API int nmb_filter_adjacency(const int32_t *contig_id, const int64_t *pos, const uint8_t *strand,
                         const double *fraction_mod, int64_t n_rows, double methylation_threshold,
                         int32_t adjacency_distance, uint8_t *keep, int32_t *unsorted_flag, void *stream);

/* ---- K2: scan + gather-join + segmented reduce (replaces utils.subseq_indices utils.py:44-67,
 *      methylated_motif_occourances find_motifs_bin.py:1234-1263, the count step of
 *      motif_model_contig :1285-1331 and the per-bin sum of motif_model_bin :1265-1283) ---- */

/* Compile motifs into per-strand scan programs (forward motif and its reverse complement,
 * nanomotif/motif.py:260-266).  programs: n_motifs * nmb_program_bytes() bytes. */
NMB_API int nmb_program_bytes(void);
NMB_API int nmb_compile_motifs(const nmb_motif *motifs, int32_t n_motifs, void *programs, void *stream);

/* Count methylated / unmethylated motif occurrences.  jobs: device array of n_jobs nmb_job with
 * item_offset filled for `motifs_per_item` (1..32); n_items = total items.  out (int64) is
 * ACCUMULATED into (zero it to get counts).  contig_group may be NULL unless a job uses
 * group_mode 2.  max_motif_len = longest motif in the batch (selects the halo width). */
NMB_API int nmb_scan_count(const nmb_assembly *assembly_h, const uint32_t *class_records,
                   const void *programs, const nmb_job *jobs, int32_t n_jobs, int32_t n_items,
                   int32_t motifs_per_item, int32_t max_motif_len, const int32_t *contig_group,
                   int64_t *out, int32_t grid_ctas /* 0 = auto */, void *stream);

/* nmb_scan_count with DYNAMIC item scheduling: the persistent CTAs draw work items from work_counter (two device
 * int32, {next item, finished CTAs}: zero before the FIRST launch; the kernel leaves them zero, so the same pair
 * serves every later launch on the stream) instead of a static round-robin.  Same counts; launches whose items differ
 * in cost (3 vs 4 motifs per job, dead chains) end without the static split's tail. */
NMB_API int nmb_scan_count_balanced(const nmb_assembly *assembly_h, const uint32_t *class_records, const void *programs,
                                    const nmb_job *jobs, int32_t n_jobs, int32_t n_items, int32_t motifs_per_item,
                                    int32_t max_motif_len, const int32_t *contig_group, int64_t *out, int32_t grid_ctas,
                                    int32_t *work_counter, void *stream);

/* nmb_compile_motifs that also groups the motifs into SIBLINGS: siblings (nmb_sibling_bytes(n_motifs) bytes of device
 * memory, overwritten) receives per motif its link to the previous motif -- same len and mod_pos, the same allowed set
 * at every position but at most one -- and the program of the motif with the position where it differs from the next
 * motif made a wildcard (the parent of a search expansion's children, find_motifs_bin.py:1116-1145).  Same launch. */
NMB_API int64_t nmb_sibling_bytes(int32_t n_motifs);
NMB_API int nmb_compile_motifs_siblings(const nmb_motif *motifs, int32_t n_motifs, void *programs, void *siblings,
                                        void *stream);

/* nmb_scan_count with SIBLING RUNS: inside every work item's block of motifs_per_item motifs, runs of consecutive
 * linked motifs that differ at one common position are scored as ONE parent chain plus a four-base split of the parent's
 * occurrences at that position (warps with a non-ACGT letter in reach score the members one by one).  Same counts as
 * nmb_scan_count, bit for bit.  programs / siblings: from nmb_compile_motifs_siblings over the same n_motifs records;
 * work_counter: as for nmb_scan_count_balanced, or NULL for the static item split. */
NMB_API int nmb_scan_count_siblings(const nmb_assembly *assembly_h, const uint32_t *class_records, const void *programs,
                                    const void *siblings, int32_t n_motifs, const nmb_job *jobs, int32_t n_jobs,
                                    int32_t n_items, int32_t motifs_per_item, int32_t max_motif_len,
                                    const int32_t *contig_group, int64_t *out, int32_t grid_ctas, int32_t *work_counter,
                                    void *stream);

/* ---- K3: occurrence positions (subseq_indices output and the save_motif_positions=True lists
 *      of motif_model_contig, find_motifs_bin.py:1322-1329) ---- */

/* Match bit-plane of ONE program strand over tiles [tile_begin, tile_begin+tile_count):
 * bit p of match_plane (flat, word index = global_pos/32, no pad, n_tiles*NMB_TILE_WORDS words) is
 * set iff the motif occurs with its mod_pos at global position p.  Compile the motif with
 * mod_pos = 0 to get start positions (utils.subseq_indices); strand 0 = forward program, 1 = its
 * reverse complement.  motif_len selects the halo width. */
NMB_API int nmb_match_plane(const nmb_assembly *assembly_h, const void *programs, int32_t motif_index,
                    int32_t strand, int32_t motif_len, int32_t tile_begin, int32_t tile_count,
                    uint32_t *match_plane, void *stream);

/* Literal non-ACGT letters in a motif string (regex-literal semantics of utils.subseq_indices, utils.py:61-66: an 'N'
 * in the motif matches the contig letter N and nothing else).  plane[p] &= (upper(ascii[p + shift]) == letter) for
 * the n_words words of a flat match plane over ONE contig of n letters starting at global position 0; positions whose
 * p + shift falls outside [0, n) are cleared.  The caller matches the motif with such positions as wildcards
 * (nmb_match_plane) and ANDs one letter plane per literal. */
NMB_API int nmb_letter_plane(const uint8_t *ascii, int64_t n, int32_t letter, int64_t shift, uint32_t *plane,
                             int64_t n_words, void *stream);

/* Ascending positions of the set bits of plane & (mask or all-ones) within the global position
 * range [pos_begin, pos_end).  Two passes on the same stream: tile_counts is scratch of
 * ceil((pos_end-pos_begin)/NMB_TILE_BP)+2 int64.  Positions are written relative to pos_begin.
 * *n_out (device int64) receives the total; at most capacity positions are written. */
NMB_API int nmb_compact_positions(const uint32_t *plane, const uint32_t *mask /* may be NULL */,
                          int64_t pos_begin, int64_t pos_end, int64_t *tile_counts,
                          int64_t *out_pos, int64_t capacity, int64_t *n_out, void *stream);

/* Gather-join in pileup order: flag[r] = bit (base + pos[r]) of plane (0 when out of
 * [0, limit)).  This is np.isin(positions, motif_index) of find_motifs_bin.py:1258-1261. */
NMB_API int nmb_test_positions(const uint32_t *plane, int64_t base, int64_t limit, const int64_t *pos,
                       int64_t n, uint8_t *flag, void *stream);

/* ---- K4: motif-growth step (replaces DNAsequence.sample_at_indices seq.py:170-189,
 *      EqualLengthDNASet.reverse_compliment :387-389, convert_to_DNAarray :474-478,
 *      DNAarray.filter_sequence_matches :499-524, DNAarray.pssm :526-537 and the KL/argmax part of
 *      MotifSearcher._motif_child_nodes_kl_dist_max find_motifs_bin.py:957-1000) ---- */

/* Windows of width 2*padding+1 <= NMB_MAX_WINDOW around global positions gpos[i] (strand[i] 1 =
 * reverse-complement the window).  Window i is stored as three uint64: x bits, y bits, N bits
 * (bit j = window column j).  The caller has already applied the reference's strict bound
 * padding < i < len - padding (seq.py:186). */
NMB_API int nmb_extract_windows(const nmb_assembly *assembly_h, const int64_t *gpos, const uint8_t *strand,
                        int64_t n, int32_t padding, uint64_t *windows /* [n][3] */, void *stream);

/* For each of n_motifs full-width masks (allowed[j] per window column, len = window width):
 * rows kept by filter_sequence_matches(keep_matches=True), i.e. one-hot(row) <= mask everywhere,
 * restricted to rows with alive[i] != 0 (alive may be NULL); hist[m][j][b] = column sums of the
 * kept one-hot rows, n_active[m] = kept rows.  n_counts_all = 1: a non-ACGT letter adds 1 to all
 * four bases (DNAarray.pssm, seq.py:41-48,537); 0: it adds nothing (EqualLengthDNASet.pssm exact-
 * letter counts, seq.py:413-421).  hist/n_active are overwritten.  keep[m*n + i] (may be NULL)
 * receives the per-row decision. */
NMB_API int nmb_window_hist(const uint64_t *windows, const uint8_t *alive, int64_t n, int32_t width,
                    const nmb_motif *masks, int32_t n_motifs, int32_t n_counts_all,
                    int32_t *hist /* [n_motifs][width][4] */, int64_t *n_active, uint8_t *keep,
                    void *stream);

/* Batched form for many searches at once: motif m examines rows [row_begin[m], row_end[m]) only
 * (max_rows = the largest range, sizes the grid).  keep_rows (may be NULL) is ONE array of n flags:
 * row i receives the decision of the motif whose range contains it, so the ranges of the motifs of
 * one call must be disjoint when keep_rows is given. */
NMB_API int nmb_window_hist_ranges(const uint64_t *windows, const uint8_t *alive, int64_t n, int32_t width,
                           const nmb_motif *masks, int32_t n_motifs, const int64_t *row_begin,
                           const int64_t *row_end, int64_t max_rows, int32_t n_counts_all, int32_t *hist,
                           int64_t *n_active, uint8_t *keep_rows, void *stream);

/* PSSM + KL(meth || background) per column in float64: pssm[m][b][j] = hist/n_active (4 x width,
 * rows A,T,G,C), kl[m][j] = sum_b p ln(p/q) after per-column renormalisation of both (scipy.stats.
 * entropy semantics: 0 ln 0 = 0, p>0 & q=0 -> inf).  bg_pssm is [4][width] float64. */
NMB_API int nmb_pssm_kl(const int32_t *hist, const int64_t *n_active, int32_t n_motifs, int32_t width,
                const double *bg_pssm, double *pssm, double *kl, void *stream);

/* ---- K5: contig x motif methylation-pattern table (replaces the external Rust operator
 *      epymetheus.methylation_pattern, call site nanomotif/main.py:167-178; spec in DESIGN.md) ----
 * Rows = the pileup rows of ONE mod type that pass the read-coverage filters, sorted by contig:
 * gpos (global position), strand (0 '+', 1 '-'), contig_id, n_mod, n_valid_cov.  plane_fwd /
 * plane_rev = match planes (nmb_match_plane, aligned at mod_pos) of the motif and of its reverse
 * complement.  A row is an observation when the bit of its strand's plane is set at gpos. */

/* stats[c] = {n_motif_obs, sum n_mod, sum n_valid_cov}; offsets[0..n_contigs] = exclusive prefix sum
 * of n_motif_obs (offsets[n_contigs] = total); cursor[c] = 0 (scratch for nmb_pattern_median). */
NMB_API int nmb_pattern_stats(const int64_t *gpos, const uint8_t *strand, const int32_t *contig_id,
                      const int32_t *n_mod, const int32_t *n_valid_cov, int64_t n_rows,
                      const uint32_t *plane_fwd, const uint32_t *plane_rev, int32_t n_contigs,
                      int64_t *stats, int64_t *offsets, int32_t *cursor, void *stream);

/* median[c] = median of n_mod / n_valid_cov over the observations of contig c (mean of the two
 * middle values for an even count, NaN without observations).  fractions: scratch of
 * offsets[n_contigs] doubles.  Must follow nmb_pattern_stats on the same stream. */
NMB_API int nmb_pattern_median(const int64_t *gpos, const uint8_t *strand, const int32_t *contig_id,
                       const int32_t *n_mod, const int32_t *n_valid_cov, int64_t n_rows,
                       const uint32_t *plane_fwd, const uint32_t *plane_rev, int32_t n_contigs,
                       const int64_t *offsets, int32_t *cursor, double *fractions, double *median,
                       void *stream);

/* ---- K5, tile-driven: many motifs per launch (pattern_scan.cu) ----
 * Join index of ONE mod type.  Rows (any order; (contig, position, strand) unique) take part when their
 * mod_type equals want_modtype (mod_type may be NULL), the contig / position is inside the assembly,
 * n_valid_cov >= min_valid_read_coverage and n_valid_cov / (n_valid_cov + n_diff) >=
 * min_valid_cov_to_diff_fraction (float64).  Outputs: valid_records [n_tiles][2][NMB_TILE_WORDS] (bit-planes
 * valid '+', valid '-', lane-interleaved), rank_dir [2][n_tiles*NMB_TILE_WORDS] (rows before each word, in
 * (strand, position) order), payload [n_rows][2] int32 = (n_mod, n_valid_cov) in that order, *n_valid_rows
 * (device int64).  scratch: ceil(2*n_tiles*NMB_TILE_WORDS/2048)+2 int64. */
NMB_API int nmb_pattern_index_build(const nmb_assembly *assembly_h, const int32_t *contig_id, const int64_t *pos,
                                    const uint8_t *strand, const uint8_t *mod_type, int32_t want_modtype,
                                    const int64_t *n_mod, const int64_t *n_valid_cov, const int64_t *n_diff,
                                    int64_t n_rows, int64_t min_valid_read_coverage,
                                    double min_valid_cov_to_diff_fraction, uint32_t *valid_records,
                                    uint32_t *rank_dir, int64_t *scratch, int32_t *payload, int64_t *n_valid_rows,
                                    void *stream);

/* One pass of n_motifs compiled motifs (nmb_compile_motifs) over the whole assembly.  phase 0 ADDS into
 * stats [n_motifs][n_contigs][3] = {n_motif_obs, sum n_mod, sum n_valid_cov}; phase 1 writes the
 * per-occurrence fractions n_mod / n_valid_cov of segment (motif, contig) at fractions[offsets[seg] + k],
 * k counted through cursor[seg] (nmb_segment_offsets sets both up from the phase-0 stats). */
NMB_API int nmb_pattern_scan(const nmb_assembly *assembly_h, const uint32_t *valid_records, const uint32_t *rank_dir,
                             const int32_t *payload, const void *programs, int32_t n_motifs, int32_t motifs_per_item,
                             int32_t max_motif_len, int32_t phase, int64_t *stats, const int64_t *offsets,
                             int32_t *cursor, double *fractions, int32_t grid_ctas, void *stream);

/* nmb_pattern_scan with dynamic item scheduling (work_counter as for nmb_scan_count_balanced). */
NMB_API int nmb_pattern_scan_balanced(const nmb_assembly *assembly_h, const uint32_t *valid_records,
                                      const uint32_t *rank_dir, const int32_t *payload, const void *programs,
                                      int32_t n_motifs, int32_t motifs_per_item, int32_t max_motif_len, int32_t phase,
                                      int64_t *stats, const int64_t *offsets, int32_t *cursor, double *fractions,
                                      int32_t grid_ctas, int32_t *work_counter, void *stream);

/* offsets[0..n_segments] = exclusive prefix sum of stats[i][0]; cursor[i] = 0. */
NMB_API int nmb_segment_offsets(const int64_t *stats, int64_t n_segments, int64_t *offsets, int32_t *cursor,
                                void *stream);

/* median[i] = exact median of fractions[offsets[i] .. offsets[i+1]) (mean of the two middle values for an
 * even count, NaN for an empty segment). */
NMB_API int nmb_segment_median(const double *fractions, const int64_t *offsets, int64_t n_segments, double *median,
                               void *stream);

/* ---- K9: binnary feature matrix from the K5 arrays on the device (replaces the polars pipeline of
 *      nanomotif/main.py:192-205 + binnary/data_processing.py:174-213,255-269: threshold filter, add_bin, per-bin
 *      weighted mean, within-bin imputation, pivot) ----
 * stats [n_motifs][n_contigs][3] and value [n_motifs][n_contigs] are nmb_pattern_scan / nmb_segment_median outputs
 * (value NULL = weighted mean, sum n_mod / sum n_valid_cov).  Binned contigs are given grouped by bin (CSR: bin_off
 * [n_bins + 1], bin_contigs ascending inside a bin).  nmb_bin_means: keep[m][c] = the cell passes n_motif_obs *
 * mean_read_cov >= threshold and its contig is binned; bin_mean / bin_has [n_motifs][n_bins] = sum(value * n_obs) /
 * sum(n_obs) over the kept cells of the bin (summed in ascending contig order, deterministic) and whether any cell
 * was kept; contig_has[c] = the contig has a kept cell.  nmb_bin_matrix: matrix[r][f] for contig rows[r] and motif
 * feats[f] = own value if kept, else the bin mean if the bin has one, else 0 (contig_bin[c] = bin of contig c). */
NMB_API int nmb_bin_means(const int64_t *stats, const double *value, int32_t n_motifs, int32_t n_contigs,
                          const int64_t *bin_off, const int32_t *bin_contigs, int32_t n_bins, double threshold, uint8_t *keep,
                          double *bin_mean, uint8_t *bin_has, uint8_t *contig_has, void *stream);
NMB_API int nmb_bin_matrix(const int64_t *stats, const double *value, const uint8_t *keep, const double *bin_mean,
                           const uint8_t *bin_has, const int32_t *contig_bin, int32_t n_contigs, int32_t n_bins,
                           const int32_t *rows, int64_t n_rows, const int32_t *feats, int32_t n_feat, double *matrix,
                           void *stream);

/* ---- K8: exhaustive candidate sweep (BASELINE.json configs[4]): counts of EVERY IUPAC motif of length 4..8
 *      at every modified position from one pass over the assembly (csrc/sweep.cu) ----
 * hist: nmb_sweep_hist_size() uint32 counters per slot (a slot is one histogram, e.g. one per bin; n_slots of them
 * stacked), zeroed by the caller; counters ADD, so several calls (contig ranges, GPUs after an all-reduce)
 * accumulate.  For k = 4..8 the block at sum_{j<k} j*2*5^j holds [o = 0..k-1][class: 0 methylated, 1
 * unmethylated][5^k windows]; a window's index is its letters as base-5 digits, first letter most significant, letter
 * states A=0 T=1 G=2 C=3 other=4.  Counted: every pileup row of the class planes (one mod type) under every window
 * that lies inside one counted contig; '-' rows count under the reverse complement of the window at the mirrored
 * offset.  contig_slot == NULL: one histogram (n_slots must be 1), the contigs of [contig_begin, contig_end) counted.
 * Otherwise contig_slot[c] (device int32, one entry per contig of the assembly) = the slot that the rows under the
 * windows of contig c count into, -1 (or any value outside [0, n_slots)) skips the contig, and the contig range is
 * ignored.  A window never leaves its contig, so contigs of different slots may share tiles. */
NMB_API int64_t nmb_sweep_hist_size(void);
NMB_API int nmb_sweep_hist(const nmb_assembly *assembly_h, const uint32_t *class_records_of_modtype, int32_t tile_begin,
                           int32_t tile_count, int32_t contig_begin, int32_t contig_end, const int32_t *contig_slot,
                           int32_t n_slots, uint32_t *hist, void *stream);
/* nmb_sweep_hist leaves the histograms RAW: only the k = 8 block is counted row by row (8 atomic adds per pileup row
 * instead of 30); the blocks of k < 8 hold just the windows at contig ends that have no one-letter extension inside
 * the contig.  nmb_sweep_finalize completes n_slots (1..65535) stacked histograms in place, hist[k] += marginal of
 * hist[k+1] over the trailing letter, k = 7 .. 4.  Call it ONCE, after every nmb_sweep_hist call (and after the
 * histograms of several GPUs have been summed: raw histograms add, finalized ones must not be finalized again). */
NMB_API int nmb_sweep_finalize(uint32_t *hist, int32_t n_slots, void *stream);

/* The bipartite half of the sweep: shapes X{a} N{g} Y{b}, a, b in {3, 4}, g in 4..8, concrete letters only.
 * hist: nmb_sweep_bipartite_size() uint32 counters per slot (zeroed by the caller, counters add); contig_begin,
 * contig_end, contig_slot and n_slots as for nmb_sweep_hist.  Shapes are stored g major, then (3,3) (3,4) (4,3)
 * (4,4); a shape's block is [o = 0..a+b-1 over the concrete letters][class][4^(a+b)] with window index
 * xL | yL << a | xR << 2a | yR << (2a + b), x / y = high / low code bit of each letter (A=0 T=1 G=2 C=3), letter i of
 * a part at bit i. */
NMB_API int64_t nmb_sweep_bipartite_size(void);
NMB_API int nmb_sweep_bipartite(const nmb_assembly *assembly_h, const uint32_t *class_records_of_modtype,
                                int32_t tile_begin, int32_t tile_count, int32_t contig_begin, int32_t contig_end,
                                const int32_t *contig_slot, int32_t n_slots, uint32_t *hist, void *stream);

/* Like nmb_sweep_hist, nmb_sweep_bipartite leaves RAW histograms: only the shapes (4, g, 4) are counted row by row
 * (40 atomic adds per pileup row instead of 140); (4,g,3), (3,g,4) and (3,g,3) hold just the windows whose extending
 * letter is not a concrete letter of the same contig.  nmb_sweep_bipartite_finalize completes n_slots (1..65535)
 * stacked histograms in place by summing the longer shapes over the dropped letter.  Call it ONCE after all passes /
 * after summing the GPUs' raw histograms. */
NMB_API int nmb_sweep_bipartite_finalize(uint32_t *hist, int32_t n_slots, void *stream);

/* dst[slot][hi][lo] = src[slot * src_slot_stride + (hi * 5 + digit) * axis_stride + lo] with lo < axis_stride, for
 * n_slots (1..65535) sources: fixes one base-5 axis (the modified position's own letter) and drops it.  n_out =
 * elements of dst per slot. */
NMB_API int nmb_sweep_slice(const uint32_t *src, int64_t src_slot_stride, int32_t n_slots, uint32_t *dst,
                            int64_t n_out, int64_t axis_stride, int32_t digit, void *stream);

/* dst[outer][15][inner] = sums of src[outer][5][inner] over the letters of each IUPAC code, in the order of
 * nanomotif/constants.py:2 (A T G C R Y S W K M B D H V N; N also takes the "other" state, like the regex
 * wildcard).  Applied to every axis in turn it turns window counts into the counts of every IUPAC motif. */
NMB_API int nmb_sweep_expand(const uint32_t *src, uint32_t *dst, int64_t outer, int64_t inner, void *stream);

/* Indices i of a finished table with n_mod[i] >= min_mod and posterior mean (5 + n_mod) / (10 + n_mod +
 * n_nomod) >= min_mean (Beta(5,5) prior, nanomotif/model.py:8-9), in no particular order; *n_out (device int64)
 * = number of hits, of which at most `capacity` are written. */
NMB_API int nmb_sweep_filter(const uint32_t *n_mod, const uint32_t *n_nomod, int64_t n, double min_mean,
                             int64_t min_mod, int64_t *out_index, int64_t capacity, int64_t *n_out, void *stream);

/* One candidate of the per-slot filters: table index (IUPAC) or counter index in the slot's bipartite histogram. */
typedef struct nmb_sweep_hit {
    int32_t slot;
    uint32_t index;
    uint32_t n_mod;
    uint32_t n_nomod;
} nmb_sweep_hit; /* 16 bytes */

/* The three per-slot candidate filters below record every motif with n_mod >= min_mod and posterior mean
 * (5 + n_mod) / (10 + n_mod + n_nomod) >= min_mean -- nmb_sweep_filter's test, bit for bit -- as nmb_sweep_hit
 * records.  *n_out (device int64) = number of hits, in no particular order, of which at most `capacity` are written.
 *
 * prune (0 or 1): 1 also drops the candidates that are a redundant specialisation or a mixture of a one-letter
 * neighbour in the same table; the records are then a subset of those with prune = 0.  For a candidate M and every
 * letter other than the modified one: a widening P puts there a letter of the lattice that covers M's letter (one
 * more base), a narrowing C one that M's letter covers; Q = P - M or M - C, n_mod and n_nomod separately, mean(Q) =
 * (5 + q_mod) / (10 + q_mod + q_nomod).  M is pruned when (a) some widening P passes the filter and mean(Q) >=
 * min_mean, or (b) some narrowing C passes and mean(Q) < min_mean.  Neighbours need not be candidates themselves (a
 * flanking N, the pseudo-letter *).  Lattices, as sets of letter states (see nmb_sweep_prune_lattice): contiguous
 * k-mers, the 15 IUPAC letters over A T G C other (N also takes "other"); bipartite ACGT halves, A T G C and * = ACGT;
 * bipartite IUPAC halves, the 14 letters other than N and * = ACGT. */

/* The LAST nmb_sweep_expand pass of a (k, mod_pos) table fused with the filter: n_mod / n_nomod are stacked
 * [n_slots][5][inner], inner = 15^(k-2) (every axis but the most significant one already expanded); the kernel
 * expands that axis in registers and records (slot, table index of the 15^(k-1) table, n_mod, n_nomod).  Motifs in
 * canonical form only: no N as the first or last letter (the modified position's own letter, at mod_pos 0 or k-1, is
 * the fixed base and never N).  The 15^(k-1) table is not written. */
NMB_API int nmb_sweep_expand_filter(const uint32_t *n_mod, const uint32_t *n_nomod, int64_t n_slots, int64_t inner,
                                    int32_t k, int32_t mod_pos, double min_mean, int64_t min_mod, int32_t prune,
                                    nmb_sweep_hit *out, int64_t capacity, int64_t *n_out, void *stream);
/* Candidates of n_slots FINISHED bipartite histograms stacked at nmb_sweep_bipartite_size(): the n_mod counters
 * (class 0) whose concrete letter at the counter's offset o is `canonical` (A=0 T=1 G=2 C=3) and that pass the
 * filter; index = the n_mod counter's position in its slot's histogram (n_nomod sits 4^(a+b) counters later). */
NMB_API int nmb_sweep_bipartite_filter(const uint32_t *hist, int32_t n_slots, int32_t canonical, double min_mean,
                                       int64_t min_mod, int32_t prune, nmb_sweep_hit *out, int64_t capacity,
                                       int64_t *n_out, void *stream);

/* ---- K8 degenerate bipartite motifs (ABI 6): X{a} N{g} Y{b} whose halves use the 14 IUPAC letters other than N
 *      (A T G C R Y S W K M B D H V, the order of nmb_sweep_expand without N), from the FINISHED bipartite
 *      histograms.  Exact: such a letter matches only ACGT contig letters, and the bipartite histograms skip every
 *      window with a non-ACGT letter in a half, so a motif's count is the sum of the ACGT counters of the concrete
 *      motifs it stands for.  N in a half is not covered (it would need a non-ACGT state in the histogram pass). ----
 * Slice: dst[slot][w] (4^(a+b-1) uint32 per slot) = the class-`cls` counters (0 methylated, 1 unmethylated) of shape
 * (a, g, b) with the modified base at motif position mod_pos (inside X or Y, gap counted) for the n_slots (1..65535)
 * finished histograms stacked at nmb_sweep_bipartite_size(); the letter at mod_pos is fixed to `canonical` (A=0 T=1
 * G=2 C=3) and w holds the other a + b - 1 letters as base-4 digits in that code, first motif letter most
 * significant. */
NMB_API int nmb_sweep_bip_iupac_slice(const uint32_t *hist, int32_t n_slots, int32_t a, int32_t g, int32_t b,
                                      int32_t mod_pos, int32_t cls, int32_t canonical, uint32_t *dst, void *stream);
/* dst[outer][14][inner] = sums of src[outer][4][inner] over the concrete letters of each of the 14 letters.  Applied
 * to the a + b - 1 axes of a slice, last axis first, it gives the table of all 14^(a+b-1) motifs, index = the letters
 * other than the modified one as base-14 digits, first letter most significant. */
NMB_API int nmb_sweep_bip_iupac_expand(const uint32_t *src, uint32_t *dst, int64_t outer, int64_t inner, void *stream);
/* The last nmb_sweep_bip_iupac_expand pass fused with the filter (see the candidate filters above): n_mod / n_nomod
 * stacked [n_slots][4][inner], inner = 14^(a+b-2) (every axis but the first expanded; a power of 14 below 2^32 / 14,
 * from which the number of axes follows); records (slot, table index, n_mod, n_nomod); the table is not written. */
NMB_API int nmb_sweep_bip_iupac_expand_filter(const uint32_t *n_mod, const uint32_t *n_nomod, int64_t n_slots,
                                              int64_t inner, double min_mean, int64_t min_mod, int32_t prune,
                                              nmb_sweep_hit *out, int64_t capacity, int64_t *n_out, void *stream);

/* Host query, no device work: the lattice the pruning filters use (0 contiguous, 1 bipartite ACGT, 2 bipartite
 * IUPAC), in table letter order with the widest letter (N or *) last.  states[i]: bit s set when letter i stands for
 * state s (A=0 T=1 G=2 C=3 other=4); widen[i] / narrow[i]: bit j set when letter j covers letter i / letter i covers
 * letter j.  Writes up to 15 entries per array and returns the number of letters. */
NMB_API int nmb_sweep_prune_lattice(int32_t lattice, uint32_t *states, uint32_t *widen, uint32_t *narrow);

/* ---- K8 lookup (ABI 9): the counts of any list of motifs in every slot, gathered from the FINISHED histograms ----
 * A motif's count is the sum of the histogram cells of the concrete motifs it stands for, with the modified letter
 * fixed.  One record per motif says which cells; the kernel knows no motif layout.  cells = product of n_states[p]
 * over p < n_pos; cell (d_0, .., d_{n_pos-1}) (mixed radix, the last position the least significant digit) has its
 * class-0 counter at base + sum_p offset[p][d_p] and its class-1 counter class_step counters later, both relative to
 * the slot's histogram.  Concrete letters and the modified letter are folded into base, so a concrete motif has
 * n_pos = 0 and one cell.  Contiguous k-mers (kind 0): base = sum_{j<k} j*2*5^j + mod_pos*2*5^k + the digits of the
 * concrete letters times 5^(k-1-i), class_step = 5^k, offset = state x 5^(k-1-i) for the states a letter stands for
 * (N: all five).  Bipartite (kind 1): base = the shape's block + o*2*4^(a+b) + the concrete letters' window bits,
 * class_step = 4^(a+b), offset = the window index bits of each state (x << xbit | y << ybit, see above). */
typedef struct nmb_sweep_query {
    int32_t kind;          /* 0: IUPAC histogram (hist), 1: bipartite histogram (bip) */
    int32_t n_pos;         /* degenerate positions, 0..7 */
    int64_t base;          /* class-0 counter of cell 0 */
    int32_t class_step;    /* class-1 counter - class-0 counter */
    uint8_t n_states[7];   /* states of degenerate position p: 1..5 (kind 0), 1..4 (kind 1) */
    uint8_t reserved;      /* 0 */
    int32_t offset[7][5];  /* counter offset of state d at degenerate position p, >= 0 */
} nmb_sweep_query; /* 168 bytes */

/* out[r][q][0..1] (device int64, row-major [n_rows][n_queries][2]) = the exact sums of the class-0 (methylated) and
 * class-1 (unmethylated) counters of query q in slot slots[r] (device int32; NULL: slot r); a negative slot gives a
 * row of zeros.  hist: finished IUPAC histograms stacked at nmb_sweep_hist_size(); bip: finished bipartite
 * histograms stacked at nmb_sweep_bipartite_size(), or NULL when no query has kind 1.  queries: device records.
 * Every existing table entry equals its sum mod 2^32.  A record the kernel cannot read safely (kind, n_pos or
 * n_states out of range, a negative offset, a counter past the end of its histogram, kind 1 with bip NULL) gives -1
 * in both entries.  n_rows 0..65535.  Deterministic (no atomics); one launch. */
NMB_API int nmb_sweep_lookup(const uint32_t *hist, const uint32_t *bip, const int32_t *slots, int32_t n_rows,
                             const nmb_sweep_query *queries, int64_t n_queries, int64_t *out, void *stream);

/* ---- host helper: CPython's random.sample(range(n), k) on a transplanted MT19937 state (the reference draws its
 *      background windows with random.sample, nanomotif/seq.py:202-225; its picks depend only on n, k and the
 *      generator's word stream).  state = the 624 key words + position of random.getstate(); out receives the k
 *      picks in draw order and the state advances exactly as CPython's would (set branch and pool branch of
 *      Lib/random.py).  Host pointers; no device work. ---- */
typedef struct nmb_mt19937 {
    uint32_t key[624];
    int32_t pos;
} nmb_mt19937;
NMB_API int nmb_mt_sample(nmb_mt19937 *state_h, int64_t n, int64_t k, int64_t *out_h);
/* count consecutive samples from the same stream; sample i is written at out_h + sum(k_h[0..i)). */
NMB_API int nmb_mt_sample_many(nmb_mt19937 *state_h, const int64_t *n_h, const int64_t *k_h, int64_t count,
                               int64_t *out_h);

/* ---- host helper: a batch of motif strings -> nmb_motif records, i.e. Motif.new_stripped_motif + Motif.split
 *      (nanomotif/motif.py:213-245) + the allowed-set bits above, for every motif of a scoring request at once (a
 *      lock-step search round packs the <= 4 children of every search).  text_h = the motif strings back to back
 *      (ASCII), motif i = [offset_h[i], offset_h[i+1]); mod_pos_h[i] = its mod_position (may be NULL when
 *      mod_pos_override >= 0, which replaces every mod position AFTER the strip); strip != 0 drops flanking '.' and
 *      re-bases the mod position (an all-wildcard motif is left as it is).  status_h[i] = 0 and out_h[i] filled, or
 *      1 (out_h[i] zeroed) for a motif this path refuses: a character other than A C G T . [ ], an unmatched or empty
 *      class, more than NMB_MAX_MOTIF_LEN positions, no constrained position, mod position outside the stripped
 *      motif.  Host pointers; no device work. ---- */
NMB_API int nmb_pack_motifs(const char *text_h, const int64_t *offset_h, const int32_t *mod_pos_h, int32_t n,
                            int32_t strip, int32_t mod_pos_override, nmb_motif *out_h, uint8_t *status_h);

/* ---- host -> device staging of PAGEABLE host buffers (the Arrow buffers of the frames nanomotif hands to its
 *      workers, find_motifs_bin.py:399-427).  n_threads host threads each own a CUDA stream and two pinned slots of
 *      slot_bytes (allocated by nmb_stager_create -- the one allocation this library makes -- and freed by
 *      nmb_stager_destroy); a copy is split into slot-sized chunks, memcpy()ed into the slots in parallel and sent by
 *      DMA, ordered after the work already on `stream`, with `stream` ordered after it.  nmb_stager_copy returns when
 *      the source has been READ (it may be freed), not when the DMA has finished.  src_host/dst_dev: host and device
 *      pointers.  Not re-entrant per stager: one copy at a time. ---- */
typedef struct nmb_stager nmb_stager;
NMB_API int nmb_stager_create(int64_t slot_bytes, int32_t n_threads, nmb_stager **out);
NMB_API int nmb_stager_copy(nmb_stager *stager, void *dst_dev, const void *src_host, int64_t bytes, void *stream);
/* Narrowing copy: dst_dev[i] = (int32) src_host[i] for n int64 values (pileup positions, Arrow large_utf8 offsets: half
 * the bytes over PCIe); *overflow_h (host) = 1 when a value did not fit in int32 -- the destination is then garbage
 * and the caller copies the column as it is. */
NMB_API int nmb_stager_copy_narrow(nmb_stager *stager, int32_t *dst_dev, const int64_t *src_host, int64_t n,
                                   int32_t *overflow_h, void *stream);
/* Same copy from MANY host pieces (the contig strings of a bin): piece p holds bytes [piece_off_h[p], piece_off_h[p+1])
 * of the destination, piece_off_h[0] = 0; srcs_h / piece_off_h are host arrays of n_src pointers / n_src + 1 offsets. */
NMB_API int nmb_stager_gather(nmb_stager *stager, void *dst_dev, const void *const *srcs_h, const int64_t *piece_off_h,
                              int64_t n_src, void *stream);
NMB_API int nmb_stager_destroy(nmb_stager *stager);

#ifdef __cplusplus
}
#endif
#endif /* NMB200_H */
