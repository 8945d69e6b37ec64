/* fmb200.h -- C-ABI of libfmb200.so: B200-native batched FM-index search.
 *
 * This is the drop-in boundary for the data-parallel hot path of SGSSGene/fmindex-collection (SURVEY.md §8b).
 * The reference is a header-only C++ template library without an FFI; the C++ shim in include/fmb200/ mirrors
 * its search entry points 1:1 and calls only the functions declared here.  Every entry point names the
 * reference interface it replaces (paths relative to /root/reference/src/fmindex-collection/).
 *
 * Conventions
 *   - plain C types; the caller owns every host buffer, the library owns all device memory;
 *   - every function returns 0 on success or a negative FMB_E* code; fmb_last_error() (thread local) has the text;
 *   - no CPU fallback: without a usable CUDA device every compute entry point fails with FMB_ENODEVICE;
 *   - symbols are uint8_t in [0, sigma); symbol 0 is the sequence delimiter (fmindex/BiFMIndex.h:26 FirstSymb=1) unless the
 *     index was created with FMB_INDEX_NO_DELIM;
 *   - rows / text positions are 64-bit in the interface; one index holds n < 2^32 - 64 rows, larger collections are searched as
 *     several indices over disjoint sets of sequences (fmb_search_and_locate_parts);
 *   - one fmb_index lives on one GPU.  Multi-GPU = one index replica per device (fmb_index_replicate), queries sharded by
 *     fmb_search_and_locate_multi or by the caller (one process per GPU: bench.py); there is no collective on the search path.
 */
#ifndef FMB200_H
#define FMB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FMB_OK          0
#define FMB_EINVAL     -1   /* bad argument                                              */
#define FMB_ENODEVICE  -2   /* no CUDA device / device index out of range                */
#define FMB_ECUDA      -3   /* a CUDA runtime call or kernel failed                      */
#define FMB_ENOMEM     -4   /* host or device allocation failed                          */
#define FMB_EUNSUPPORTED -5 /* valid request outside what this build implements          */
#define FMB_EOVERFLOW  -6   /* result/frontier capacity exceeded and growing was refused */

typedef struct fmb_index   fmb_index;    /* device image of a BiFMIndex / FMIndex                         */
typedef struct fmb_queries fmb_queries;  /* device-resident query batch                                   */
typedef struct fmb_results fmb_results;  /* device-resident result set: cursors (hits) or located rows    */

/* One reported cursor = the arguments of the reference delegate `(size_t qidx, cursor, size_t e)`
 * (search/SearchNg26.h:414-421); cursor = BiFMIndexCursor{lb, lbRev, len, steps} (fmindex/BiFMIndexCursor.h:22-37).
 * Unidirectional / exact searches report lb_rev = 0 (LeftBiFMIndexCursor has none, BiFMIndexCursor.h:203-256). */
typedef struct {
    uint64_t qidx, lb, lb_rev, len, steps, e;
} fmb_hit;

/* One located row = the arguments of fmc::Search's report callback `(qidx, seqId, pos + offset, e)`
 * (search/search.h:55-60) with (seqId, pos, offset) = index.locate(row) (fmindex/BiFMIndex.h:177-202). */
typedef struct {
    uint64_t qidx, seq, pos, e;
} fmb_loc;

/* compact form of fmb_loc for bulk transfers (valid because n < 2^32 in this build) */
typedef struct {
    uint32_t qidx, seq, pos, e;
} fmb_loc32;

typedef struct {
    uint64_t n;                /* rows = text length incl. delimiters                      */
    uint32_t sigma;
    uint32_t bidirectional;    /* 1 = BiFMIndex, 0 = FMIndex                               */
    uint64_t n_samples;        /* sampled suffix-array entries                             */
    uint64_t n_delims;         /* rows of the BWT holding symbol 0                         */
    uint64_t device_bytes;     /* HBM used by the index image                              */
    uint32_t occ_block_bytes;  /* bytes fetched by one rank lookup (32 for sigma<=5)       */
    uint32_t occ_block_rows;   /* BWT rows covered by one occ block                        */
    int32_t  device;
    uint32_t tables;           /* optional accelerating tables the image holds, FMB_TABLE_* bits  */
    uint32_t flags;            /* FMB_INDEX_* variant bits                                  */
    uint32_t text_tables;      /* text check tables of exact search, FMB_TEXT_* bits        */
} fmb_index_info;
#define FMB_TABLE_PAIR     1u   /* two-symbol pair table (128-byte lines)          */
#define FMB_TABLE_KMER     2u   /* k-mer interval table                            */
#define FMB_TABLE_JUMP     4u   /* LF^16 jump table, direction 0                   */
#define FMB_TABLE_JUMP_REV 8u   /* LF^16 jump table, direction 1                   */
#define FMB_TABLE_LOCBLOCK 16u  /* combined occ + marker records for locate        */
#define FMB_TABLE_LOCROW   32u  /* locate shortcut table, or the suffix array that replaces it (text-regular sampling, sigma <= 5) */
#define FMB_TABLE_BIKMER   64u  /* bidirectional k-mer table for scheme roots      */
#define FMB_TABLE_JUMP4    128u /* LF^4 jump tables (tails shorter than 16 symbols) */
#define FMB_TABLE_JUMP32   256u /* direction 0 holds merged LF^16 / LF^32 entries (32 symbols per lookup in exact search) */
#define FMB_TABLE_ANCHORS  512u /* anchor table of text extraction (built on the first extraction call)                  */
/* fmb_index_info.text_tables (sigma <= 5 with delimiter, needs the locate shortcut): once the interval of an exact search is one row,
 * the rest of the read is compared with the text at that row's position and the final row is read from the inverse suffix array */
#define FMB_TEXT_CHECK     1u   /* inverse suffix array (4 bytes per row) + 2-bit text + sequence starts                 */
#define FMB_TEXT_LOCATE    2u   /* text-regular sampling: locate takes the rows the text check found (no index access)   */

/* work counters of the last search/locate call on a result set (device-side counting, optional) */
typedef struct {
    uint64_t extensions;       /* cursor extensions executed                                */
    uint64_t occ_lookups;      /* occ blocks fetched (1 when both interval ends share a block, else 2) */
    uint64_t lf_steps;         /* LF steps walked by locate                                 */
    uint64_t frontier_peak;    /* largest breadth-first frontier (scheme search)            */
    double   kernel_ms;        /* device time of the call (CUDA events)                     */
    double   main_kernel_ms;   /* device time of the dominant kernel alone (search / LF walk) */
    uint64_t line_requests;    /* 128-byte-line requests issued by the two-symbol exact kernel (physical work) */
    uint64_t h2d_bytes;        /* fmb_search_and_locate*: bytes the call copied host -> device (symbols, offsets, ...)   */
    uint64_t d2h_bytes;        /* ... and device -> host (located rows)                                                 */
} fmb_stats;

const char* fmb_last_error(void);
int fmb_device_count(void);                       /* number of CUDA devices, 0 if none     */
const char* fmb_version(void);

/* ---- index ---------------------------------------------------------------------------------------------- */

/* Replaces the constructors BiFMIndex(bwt, bwtRev, SparseArray) (fmindex/BiFMIndex.h:40-51) and
 * FMIndex(bwt, SparseArray) (fmindex/FMIndex.h:28-32): takes the BWT bytes (and the BWT of the reversed text,
 * NULL for a unidirectional index) plus the sampled suffix array in the generic form "bit i of sample_bitmap
 * set <=> row i carries a sample; samples listed in row order" (suffixarray/SparseArray.h:44-70).
 * Builds the device occurrence tables (K1), C (utils.h:200-206) and the sample tables. */
int fmb_index_create(fmb_index** out, int device, uint32_t sigma, uint64_t n,
                     const uint8_t* bwt, const uint8_t* bwt_rev,
                     const uint64_t* sample_bitmap, const uint32_t* sample_seq, const uint32_t* sample_pos,
                     uint64_t n_samples);

/* The index variants of the reference (fmindex/BiFMIndex.h:17-28): BiFMIndex<...>::NoDelim -- FirstSymb = 0, symbol 0 is an ordinary
 * symbol of an omega-sorted (circular) text instead of the sequence delimiter -- and BiFMIndex<...>::ReuseRev -- no bwtRev: the one BWT
 * of text + reversed text serves both directions (fmindex/BiFMIndexCursor.h fetchRightBwt).  bwt_rev must be NULL with
 * FMB_INDEX_REUSE_REV.  Indices without delimiter use the generic occurrence-table layout whatever their alphabet size.  The GPU
 * builder (fmb_index_build) produces delimited indices only; these variants are created from the BWT of a reference index. */
#define FMB_INDEX_NO_DELIM   1u
#define FMB_INDEX_REUSE_REV  2u
int fmb_index_create_ex(fmb_index** out, int device, uint32_t sigma, uint64_t n,
                        const uint8_t* bwt, const uint8_t* bwt_rev,
                        const uint64_t* sample_bitmap, const uint32_t* sample_seq, const uint32_t* sample_pos,
                        uint64_t n_samples, uint32_t flags);

/* Replaces BiFMIndex(Sequences, samplingRate, threads) (fmindex/BiFMIndex.h:107-167) / FMIndex(Sequences, ...)
 * (fmindex/FMIndex.h:58-112): `text` is the concatenation s0 0 s1 0 ... built by createSequences
 * (utils.h:382-464).  Suffix sorting (libsais in the reference, utils.h:97-129), BWT (utils.h:145-163), the BWT
 * of the reversed text (BiFMIndex.h:82-91) and the text-space sampling `pos_in_sequence % rate == 0`
 * (BiFMIndex.h:121-135) all run on the GPU.  text may be a host pointer, or a device pointer on `device` when
 * text_on_device != 0. */
int fmb_index_build(fmb_index** out, int device, uint32_t sigma, const uint8_t* text, uint64_t n,
                    uint32_t sampling_rate, int bidirectional, int text_on_device);

/* On-disk form of an index, replacing saveIndex / loadIndex (fmindex/diskStorage.h:13-27; cereal archive of
 * (bwt, bwtRev, C, annotatedArray), fmindex/BiFMIndex.h:209-215).  The file holds the same content in a flat versioned
 * layout -- BWT bytes of both directions, sample marker bitmap, samples in row order, each section with a checksum
 * (layout in csrc/fmb_io.cu) -- and every device table is rebuilt on the GPU when it is loaded.  fmb_index_load
 * validates magic, version, section sizes and checksums BEFORE it touches the device and fails with FMB_EINVAL on any
 * mismatch. */
int fmb_index_save(const fmb_index* ix, const char* path);
int fmb_index_load(fmb_index** out, int device, const char* path);
/* the section checksum of the file format (64-bit FNV-style over little-endian 8-byte words, tail zero padded) */
uint64_t fmb_checksum64(const void* data, uint64_t bytes);

void fmb_index_destroy(fmb_index* ix);
int  fmb_index_get_info(const fmb_index* ix, fmb_index_info* info);
int  fmb_index_get_C(const fmb_index* ix, uint64_t* C /* sigma+1 */);           /* member C, BiFMIndex.h:34 */

/* Export the index content to host buffers (any pointer may be NULL): BWT bytes (n each), sample bitmap
 * ((n+63)/64 words), samples (n_samples each).  Lets a host-side reference index be constructed from exactly
 * the same data (BiFMIndex.h:40). */
int fmb_index_export(const fmb_index* ix, uint8_t* bwt, uint8_t* bwt_rev, uint64_t* sample_bitmap,
                     uint32_t* sample_seq, uint32_t* sample_pos);

/* Raw bytes of the one-symbol occurrence table of direction `dir` -- the blocks the kernels read (layout in csrc/fmb_device.cuh; 32 bytes
 * per 64 rows for sigma <= 5, *block_bytes per 64 rows otherwise).  out == NULL only reports the size.  fmb200::HostMirror<Sigma>
 * (fmb200/host_mirror.hpp), the host-side String_c over the same layout (string/concepts.h:26-87), produces identical bytes. */
int fmb_index_export_blocks(const fmb_index* ix, int dir, uint8_t* out, uint64_t capacity, uint64_t* bytes, uint32_t* block_bytes);

/* ---- String_c concept, batched (string/concepts.h:26-87).  dir 0 = bwt, 1 = bwtRev.  All pointers host. ---- */
int fmb_string_symbol(const fmb_index* ix, int dir, const uint64_t* idx, uint64_t count, uint8_t* out);
int fmb_string_rank(const fmb_index* ix, int dir, const uint64_t* idx, const uint8_t* symb, uint64_t count, uint64_t* out);
int fmb_string_prefix_rank(const fmb_index* ix, int dir, const uint64_t* idx, const uint8_t* symb, uint64_t count, uint64_t* out);
/* out_rs / out_prs: count x sigma, row-major; out_prs may be NULL (all_ranks vs all_ranks_and_prefix_ranks) */
int fmb_string_all_ranks(const fmb_index* ix, int dir, const uint64_t* idx, uint64_t count, uint64_t* out_rs, uint64_t* out_prs);

/* ---- cursor steps, batched (fmindex/BiFMIndexCursor.h:113-128 extendLeft/Right(symb); :58-82 all symbols) ---- */
/* cur/out: count x 4 words {lb, lbRev, len, steps}; symb[i] < sigma extends by one symbol */
int fmb_cursor_extend(const fmb_index* ix, int right, const uint64_t* cur, const uint8_t* symb, uint64_t count, uint64_t* out);
/* out: count x sigma x 4 words */
int fmb_cursor_extend_all(const fmb_index* ix, int right, const uint64_t* cur, uint64_t count, uint64_t* out);

/* ---- queries --------------------------------------------------------------------------------------------- */

/* `Sequences queries` of the reference (concepts.h:12-24), flattened: symbols of all queries back to back and
 * offsets[nq+1].  Host pointers (pinned memory is copied faster).  The batch is bound to the device of `ix`. */
int  fmb_queries_upload(fmb_queries** out, const fmb_index* ix, const uint8_t* symbols, const uint64_t* offsets, uint64_t nq);
/* Reverse-complement doubling (the example's loadQueries with reverse = true, example/utils.h:62-74; main.cpp:71): the device
 * batch holds 2 nq queries -- uploaded query i as query 2i and its reverse complement (reversed, every symbol c < sigma
 * replaced by complement[c]; DNA: {0,4,3,2,1}) as query 2i+1 -- but only the nq forward reads cross PCIe. */
int  fmb_queries_upload_revcomp(fmb_queries** out, const fmb_index* ix, const uint8_t* symbols, const uint64_t* offsets, uint64_t nq,
                                const uint8_t* complement /* sigma entries */);
/* The same batch from 2-bit packed host symbols (sigma <= 5): symbol i of the batch is the field [2i, 2i+2) of the little-endian word
 * stream `packed`, holding symbol - 1; positions whose symbol has no 2-bit code (the delimiter 0, anything >= sigma) are listed, in
 * ascending order, in exc_pos with their symbol in exc_sym (the packed field there is ignored).  `offsets` may be a slice of a larger
 * batch (offsets[0] != 0): positions are those of the whole batch.  A quarter of the bytes crosses PCIe; the reference has no such
 * entry point -- its FASTA reader (example/utils.h:27-105) produces byte sequences, fmb200/io.hpp can pack while parsing. */
int  fmb_queries_upload_packed(fmb_queries** out, const fmb_index* ix, const uint32_t* packed, const uint64_t* offsets, uint64_t nq,
                               const uint64_t* exc_pos, const uint8_t* exc_sym, uint64_t n_exc);
/* Host-side packer for that form: packs symbols[first, first + count) into their fields of `words` (which must hold
 * (first + count + 15) / 16 + 1 words; fields outside the range are left alone, so disjoint ranges whose borders are multiples of 16
 * can be packed by different threads) and lists the symbols without 2-bit code in exc_pos / exc_sym (ascending positions; at most
 * exc_capacity are written).  Returns the number of exceptions found. */
uint64_t fmb_pack_symbols(const uint8_t* symbols, uint64_t first, uint64_t count, uint32_t sigma, uint32_t* words,
                          uint64_t* exc_pos, uint8_t* exc_sym, uint64_t exc_capacity);
void fmb_queries_destroy(fmb_queries* q);
uint64_t fmb_queries_count(const fmb_queries* q);

/* ---- searches (results stay on the device until fetched) -------------------------------------------------- */

/* search_no_errors::search(index, queries, delegate) (search/SearchNoErrors.h:13-26 per query, :29-85 batched).
 * One hit per query with a non-empty interval; works on both index kinds. */
int fmb_search_exact(const fmb_index* ix, const fmb_queries* q, fmb_results** out);

/* search_ng26::search<Edit>(index, queries, scheme, partition, delegate) (search/SearchNg26.h:427-433).
 * Scheme = n_searches x n_parts arrays pi, l, u (search_scheme/Search.h:19-28, pi zero based as produced by
 * search_scheme/generator/*.h); partition = n_parts part lengths (search_scheme/expand.h:324-343).
 * Every query must have length sum(partition).  Reports every cursor the reference reports (as a multiset). */
int fmb_search_scheme(const fmb_index* ix, const fmb_queries* q, int edit,
                      uint32_t n_searches, uint32_t n_parts, const uint32_t* pi, const uint32_t* l, const uint32_t* u,
                      const uint32_t* partition, fmb_results** out);

/* The same call with the hit limit `n` of the reference (search/SearchNg26.h:408-433, search_n_impl; fmc::search_n,
 * search/search.h:37-45): per query the cursors are reported in the order the reference's depth-first search finds
 * them (searches of the scheme in order, SearchNg26.h:385-390) until n ROWS are reached; the cursor that crosses the
 * limit is clipped to the rows still missing (:414-417).  n = UINT64_MAX: no limit (= fmb_search_scheme); n = 0: no
 * result.  The device enumerates alignments in its own order and orders / cuts afterwards (hits come back sorted by qidx,
 * then discovery order).  Small limits (n <= 8) also bound the WORK: the kernel keeps the n smallest discovery-order keys found per
 * query (a cursor of len rows counts min(len, n) times) and drops every subtree that cannot beat the n-th, and it starts the searches
 * of the scheme one after the other; larger n bound the output only.  FMB_EUNSUPPORTED when errors x key width exceed the 56-bit ordering key (e.g. more than 4 errors on
 * 150-symbol DNA queries). */
int fmb_search_scheme_n(const fmb_index* ix, const fmb_queries* q, int edit,
                        uint32_t n_searches, uint32_t n_parts, const uint32_t* pi, const uint32_t* l, const uint32_t* u,
                        const uint32_t* partition, uint64_t n, fmb_results** out);

/* search_pseudo::search<Edit>(index, queries, expandedScheme, delegate) (search/SearchPseudo.h:171-186) on the PART form of the
 * expanded scheme (the host side folds the per-symbol pi / l / u back into parts, include/fmb200/search.hpp): edit != 0 is
 * search_distance (:100-165) -- edit distance WITHOUT the redundancy filter of search_ng26, i.e. insertions and deletions may
 * follow every kind of step and every alignment is reported, duplicates included; edit == 0 is search_hm (= fmb_search_scheme
 * with Hamming distance). */
int fmb_search_scheme_pseudo(const fmb_index* ix, const fmb_queries* q, int edit,
                             uint32_t n_searches, uint32_t n_parts, const uint32_t* pi, const uint32_t* l, const uint32_t* u,
                             const uint32_t* partition, fmb_results** out);

/* search_backtracking::search(index, queries, maxError, delegate) (search/Backtracking.h:85-88); Hamming,
 * works on unidirectional indices. */
int fmb_search_backtracking(const fmb_index* ix, const fmb_queries* q, uint32_t max_errors, fmb_results** out);

/* LocateLinear{index, cursor} over every row of every hit (locate.h:15-57) with index.locate(row)
 * (BiFMIndex.h:177-202, FMIndex.h:114-124); output rows carry pos + offset like search/search.h:55-60. */
int fmb_locate(const fmb_index* ix, const fmb_results* hits, fmb_results** out);

/* index.locate(idx) for `count` arbitrary SA rows in one launch (fmindex/BiFMIndex.h:177-202, FMIndex.h:114-124):
 * (seqId, pos) of the nearest sampled row on the LF path and the number of LF steps walked; the text position of
 * row i is pos[i] + steps[i].  All pointers host. */
int fmb_locate_rows(const fmb_index* ix, const uint64_t* rows, uint64_t count, uint32_t* seq, uint32_t* pos, uint64_t* steps);

/* index.single_locate_step(idx) = annotatedArray.value(idx) (fmindex/BiFMIndex.h:204-206, suffixarray/SparseArray.h:63-70):
 * has[i] = 1 and (seq[i], pos[i]) = the sample when row i is sampled, else has[i] = 0. */
int fmb_sample_value(const fmb_index* ix, const uint64_t* rows, uint64_t count, uint8_t* has, uint32_t* seq, uint32_t* pos);

/* ---- text extraction: reconstructText (utils.h:672) and substrings of it, on the GPU.  All pointers host. ----
 * The index holds no copy of the text; the text is read back from the BWT with backward LF walks.  The first call that needs it builds
 * the anchor table (FMB_TABLE_ANCHORS: every sampled row and every delimiter row with its text position, 8 bytes per anchor, counted
 * in device_bytes; FMB_ENOMEM when it does not fit the image budget in force at that call, the index stays usable).  A range (seq, begin, end) is the
 * symbols [begin, end) of sequence seq, delimiter excluded.  Every walk between two anchors takes LF^16 steps of direction 0 where the
 * index has that table, LF^4 steps for the rest and single LF steps on the occurrence blocks otherwise; stats->line_requests counts
 * jump-table lookups, stats->lf_steps single LF steps (stats may be NULL).  FMB_EUNSUPPORTED for FMB_INDEX_NO_DELIM indices, which
 * have no sequence boundaries.  Works on ReuseRev and unidirectional indices. */
int fmb_index_sequence_count(const fmb_index* ix, uint64_t* count);                       /* = number of delimiters, no launch */
int fmb_index_sequence_lengths(const fmb_index* ix, uint64_t* lengths /* count */);       /* symbols per sequence, no delimiter */
/* Range i is written to out + offsets[i] (offsets: count + 1 entries, offsets[count] = bytes written).  FMB_EINVAL, before any launch
 * once the table exists, for seq >= count, begin > end or end > length; and for capacity < the bytes needed, which offsets[count]
 * then reports. */
int fmb_extract(const fmb_index* ix, const uint64_t* seq, const uint64_t* begin, const uint64_t* end, uint64_t count,
                uint8_t* out, uint64_t capacity, uint64_t* offsets /* count + 1 */, fmb_stats* stats);
/* the whole text s0 0 s1 0 ... 0, n bytes: the input of fmb_index_build, so build -> reconstruct round-trips (capacity >= n) */
int fmb_index_reconstruct_text(const fmb_index* ix, uint8_t* out, uint64_t capacity);

/* ---- super-maximal exact matches (SMEMs): the seeds of reads that exact and k-error search cannot place -------------------------
 * A query symbol 0 (the delimiter) or >= sigma never matches.  The interval [i, j) (j > i) of a query Q of length m OCCURS when Q[i:j]
 * holds no non-matching symbol and is a substring of one sequence of the collection (never across a delimiter); its SA interval
 * (lb, len) of direction 0 is then what fmb_search_exact reports for the query Q[i:j].  [i, j) is an SMEM when it occurs, i == 0 or
 * [i-1, j) does not occur, and j == m or [i, j+1) does not occur: the occurring intervals that are maximal under containment.  Starts
 * and ends both increase strictly from one SMEM of a query to the next.  The reference library has no counterpart. */
typedef struct { uint64_t qidx, begin, end, lb, len; } fmb_smem;          /* SA interval of direction 0, as exact search reports it */
typedef struct { uint64_t qidx, begin, end, seq, pos; } fmb_smem_loc;     /* pos = text position of Q[begin] in sequence seq        */
/* Every SMEM of every query of the batch with end - begin >= min_len (min_len <= 1: all of them), ordered by qidx, then begin (result
 * kind 2).  stats: extensions / occ_lookups count the bidirectional steps as the one-symbol exact kernel counts its steps, line_requests
 * the lookups of the bidirectional k-mer table, and the locate shortcut, sample, sequence start and text word lookups of the text
 * path (FMB_TEXT_CHECK; results never depend on which tables the image holds).  FMB_EUNSUPPORTED, before any launch, for a
 * unidirectional index (no right step) and for FMB_INDEX_NO_DELIM indices (no sequence borders).  FMB_EOVERFLOW when the record list
 * cannot grow to what the batch needs or holds 2^32 records or more. */
int fmb_search_smems(const fmb_index* ix, const fmb_queries* q, uint32_t min_len, fmb_results** out);
/* Per SMEM of `smems` (kind 2) the first min(len, max_occ) rows lb, lb + 1, ... of its interval, located (result kind 3): every
 * occurrence when len <= max_occ, a deterministic cap on repeats otherwise (max_occ = UINT64_MAX: no cap).  Rows come grouped by SMEM
 * in record order, within an SMEM in row order.  FMB_EINVAL for another result kind, FMB_EOVERFLOW for 2^32 rows or more (as
 * fmb_locate), FMB_EUNSUPPORTED as fmb_search_smems. */
int fmb_locate_smems(const fmb_index* ix, const fmb_results* smems, uint64_t max_occ, fmb_results** out);
int fmb_results_fetch_smems(const fmb_results* r, fmb_smem* out, uint64_t capacity);              /* kind 2 only, else FMB_EINVAL */
int fmb_results_fetch_smem_locs(const fmb_results* r, fmb_smem_loc* out, uint64_t capacity);      /* kind 3 only, else FMB_EINVAL */

/* ---- results ----------------------------------------------------------------------------------------------- */
uint64_t fmb_results_count(const fmb_results* r);
/* 0 = hits (cursors), 1 = located rows, 2 = SMEMs (fmb_search_smems), 3 = located rows of SMEMs (fmb_locate_smems) */
int  fmb_results_kind(const fmb_results* r);
int  fmb_results_fetch_hits(const fmb_results* r, fmb_hit* out, uint64_t capacity);
int  fmb_results_fetch_locs(const fmb_results* r, fmb_loc* out, uint64_t capacity);
int  fmb_results_fetch_locs32(const fmb_results* r, fmb_loc32* out, uint64_t capacity);
int  fmb_results_get_stats(const fmb_results* r, fmb_stats* out);
void fmb_results_destroy(fmb_results* r);

/* ---- one-call end-to-end path: fmc::Search{index, queries, editDistance, errors}() (search/search.h:47-75)
 *      with an explicit scheme (n_searches = 0 selects exact search).  Host queries in, located rows out;
 *      uploads, kernels and downloads are pipelined over chunks of queries (persistent host threads and streams owned by the
 *      index).  `out` must hold `capacity` rows; *n_out receives the number of rows found (if it exceeds capacity the call fails
 *      with FMB_EOVERFLOW).  Rows come grouped by ascending ranges of qidx (chunk order). ---- */
int fmb_search_and_locate(const fmb_index* ix, const uint8_t* symbols, const uint64_t* offsets, uint64_t nq,
                          int edit, uint32_t n_searches, uint32_t n_parts, const uint32_t* pi, const uint32_t* l,
                          const uint32_t* u, const uint32_t* partition,
                          fmb_loc32* out, uint64_t capacity, uint64_t* n_out, fmb_stats* stats);

/* the same call on 2-bit packed host queries (see fmb_queries_upload_packed) */
int fmb_search_and_locate_packed(const fmb_index* ix, const uint32_t* packed, const uint64_t* offsets, uint64_t nq,
                                 const uint64_t* exc_pos, const uint8_t* exc_sym, uint64_t n_exc,
                                 int edit, uint32_t n_searches, uint32_t n_parts, const uint32_t* pi, const uint32_t* l,
                                 const uint32_t* u, const uint32_t* partition,
                                 fmb_loc32* out, uint64_t capacity, uint64_t* n_out, fmb_stats* stats);

/* ---- multi GPU (SURVEY.md section 8e): the index is replicated once per GPU, one call shards the queries, nothing is exchanged ----
 * fmb_index_replicate copies the finished device image of `src` to `device` (peer-to-peer over NVLink when the devices allow it, else
 * through the host) instead of building it again.  fmb_search_and_locate_multi splits the nq queries into contiguous shards of
 * ceil(nq / n_replicas) queries, shard g is searched by replicas[g] (all replicas at the same time, each with its own host threads and
 * streams); the rows of shard g are written to out + g * shard_capacity and counted in n_out[g]; qidx is the index in the whole batch.
 * FMB_EOVERFLOW when a shard found more rows than shard_capacity (n_out[g] then holds the capacity it needs). */
int fmb_index_replicate(const fmb_index* src, int device, fmb_index** out);
int fmb_search_and_locate_multi(const fmb_index* const* replicas, uint32_t n_replicas,
                                const uint8_t* symbols, const uint64_t* offsets, uint64_t nq,
                                int edit, uint32_t n_searches, uint32_t n_parts, const uint32_t* pi, const uint32_t* l,
                                const uint32_t* u, const uint32_t* partition,
                                fmb_loc32* out, uint64_t shard_capacity, uint64_t* n_out /* n_replicas */, fmb_stats* stats);

/* ---- collections beyond one index (n >= 2^32 - 64 rows; the reference switches to a 64-bit suffix array there, utils.h:243-247) ----
 * The device image keeps 32-bit rows, so a larger collection is split at sequence borders into parts, one fmb_index per part (on one
 * device when the images fit -- fmb_set_image_budget -- or on several).  fmb_search_and_locate_parts searches the WHOLE batch in every
 * part at the same time; the rows of part p are written to out + p * part_capacity, counted in n_out[p], and carry the sequence
 * numbers of the whole collection (seq + seq_base[p]).  An occurrence lies in exactly one sequence, hence in exactly one part: the
 * located rows of all parts together are those of one index over the whole collection (as a multiset; hit limits per query would
 * apply per part and are not offered here). */
int fmb_search_and_locate_parts(const fmb_index* const* parts, uint32_t n_index_parts, const uint64_t* seq_base,
                                const uint8_t* symbols, const uint64_t* offsets, uint64_t nq,
                                int edit, uint32_t n_searches, uint32_t n_parts, const uint32_t* pi, const uint32_t* l,
                                const uint32_t* u, const uint32_t* partition,
                                fmb_loc32* out, uint64_t part_capacity, uint64_t* n_out /* n_index_parts */, fmb_stats* stats);

/* Exact-search kernel selection.  FMB_EXACT_AUTO (default): two-symbol steps on the 128-byte pair table when the
 * index has one (sigma <= 5), else one-symbol steps (generic layout: four-symbol jumps once the interval is one row).
 * FMB_EXACT_ONE_SYMBOL: the one-symbol kernel, one symbol per step on every layout, which also fills
 * the algorithmic work counters fmb_stats.extensions / occ_lookups (SURVEY.md §8d) -- the two-symbol kernel reports
 * fmb_stats.line_requests instead.  FMB_EXACT_NO_TEXT: the two-symbol kernel without the text check of single-row intervals
 * (FMB_TEXT_CHECK): the LF^16 / LF^32 / LF^4 jumps walk the rest of the read.  Results are identical in every mode. */
#define FMB_EXACT_AUTO        0
#define FMB_EXACT_ONE_SYMBOL  1
#define FMB_EXACT_TWO_SYMBOL  2
#define FMB_EXACT_NO_TEXT     3
int  fmb_index_set_exact_mode(fmb_index* ix, int mode);

/* Locate kernel selection.  FMB_LOCATE_AUTO (default): the locate shortcut table when the index has one (per row the
 * sample its LF walk ends at and the walk's length, precomputed at build time: two fetches per row), else the LF walk.
 * FMB_LOCATE_WALK: always walk (the kernel SURVEY.md §8 a13 describes).  Results are identical. */
#define FMB_LOCATE_AUTO  0
#define FMB_LOCATE_WALK  1
int  fmb_index_set_locate_mode(fmb_index* ix, int mode);

/* ---- synthetic data + pinned host memory helpers (bench / tests) ------------------------------------------- */
/* T[i] = 1 + (splitmix64(seed + i) % (sigma-1)) for i < n-1, T[n-1] = 0; written to a device buffer owned by the
 * library (free with fmb_device_free).  The same generator is restated in fmb200/synth.py for the CPU side. */
int  fmb_synth_text_device(int device, uint32_t sigma, uint64_t n, uint64_t seed, uint8_t** d_text);
/* nq reads of `length` symbols copied from d_text at offsets splitmix64(i * 0x632BE59BD9B4E019 + seed) % (n - length)
 * (never covering the final delimiter); written back to back into a device buffer owned by the library. */
int  fmb_synth_reads_device(int device, const uint8_t* d_text, uint64_t n, uint64_t nq, uint32_t length, uint64_t seed, uint8_t** d_reads);
/* the same reads with e = hash % (max_errors+1) planted edits each (substitutions only when edit == 0, else a mix of
 * substitutions, insertions and deletions that keeps the length); 3 <= length <= 512 */
int  fmb_synth_reads_err_device(int device, const uint8_t* d_text, uint64_t n, uint64_t nq, uint32_t length, uint64_t seed,
                                uint32_t sigma, uint32_t max_errors, int edit, uint8_t** d_reads);
/* locate-heavy workload: the random text of fmb_synth_text_device with `copies` copies of a unit of unit_len symbols
 * (each copy with sub_per_mille/1000 substituted symbols) in disjoint slots; reads = windows of the unit */
int  fmb_synth_repeat_text_device(int device, uint32_t sigma, uint64_t n, uint64_t seed, uint32_t unit_len, uint32_t copies,
                                  uint32_t sub_per_mille, uint8_t** d_text);
int  fmb_synth_unit_reads_device(int device, uint32_t sigma, uint64_t nq, uint32_t length, uint64_t seed, uint32_t unit_len, uint8_t** d_reads);
/* Measurement aid (SURVEY.md section 8d: "the harness must additionally measure an empirical ceiling with an independent random gather
 * over a table of the index's size"): `requests` independent random reads over one of the index's own tables, each issued the way the
 * search kernels issue it -- FMB_GATHER_PAIR_LINE: one 128-byte pair line by 4 lanes x 32 B; FMB_GATHER_OCC_BLOCK: one 32-byte occ block
 * (sigma > 5: one block of the generic layout); FMB_GATHER_JUMP_ENTRY: one 8/16-byte jump-table entry.  Reports requests per second
 * (best of three launches, CUDA events), the table size and the bytes one request uses. */
#define FMB_GATHER_PAIR_LINE  0
#define FMB_GATHER_OCC_BLOCK  1
#define FMB_GATHER_JUMP_ENTRY 2
int  fmb_measure_gather(const fmb_index* ix, int table, uint64_t requests, double* requests_per_s, uint64_t* table_bytes, uint32_t* request_bytes);
/* HBM budget of the index images created AFTER this call (process wide; 0 = no limit, the default: every table the device can hold;
 * the environment variable FMB_IMAGE_GB sets the same).  Beyond the occurrence blocks every table of an image is optional -- results
 * never depend on them -- and trades memory for speed; with a budget they are admitted in the order of what they buy per byte: pair +
 * k-mer tables, locate blocks, LF^16 table of direction 0, of direction 1, bidirectional k-mer table, locate shortcut, merged LF^32
 * entries, LF^4 tables (3 Gbp DNA: 15 / 39 / 63 / 76 / 100 / 146 GB; measured throughputs in profiles/r02_image_budget_curve.json). */
int  fmb_set_image_budget(uint64_t bytes);
/* All work of `ix` is enqueued on `stream` (a cudaStream_t of the index's device, e.g. the caller's timing
 * stream) instead of the index's private stream.  NULL restores the private stream. */
int  fmb_index_set_stream(fmb_index* ix, void* stream);
/* number of kernels of this library launched by the calling process so far (bench.py's gpu_launches) */
uint64_t fmb_kernel_launch_count(void);
int  fmb_device_free(int device, void* p);
int  fmb_copy_to_host(int device, void* dst_host, const void* src_device, uint64_t bytes);
void* fmb_host_alloc_pinned(uint64_t bytes);
void  fmb_host_free_pinned(void* p);

#ifdef __cplusplus
}
#endif
#endif /* FMB200_H */
