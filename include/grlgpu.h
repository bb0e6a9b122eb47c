/*
 * grlgpu.h -- C ABI of the B200 (sm_100a) parse phase of grlBWT.
 *
 * The reference (ddiazdom/grlBWT) has no FFI: the path sits behind C++ templates. This header is the
 * boundary a maintainer binds instead of those templates; every entry point cites the reference
 * interface it replaces (paths relative to the reference tree). Conventions: plain pointers and
 * sizes, caller-owned buffers, int status (0 = ok, < 0 = grlgpu_status), no exceptions and no
 * exit() across the boundary, one context driven by one host thread, one context per GPU.
 * There is no CPU fallback: every call fails with GRLGPU_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef GRLGPU_H
#define GRLGPU_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct grlgpu_ctx grlgpu_ctx;

enum grlgpu_status {
    GRLGPU_OK = 0,
    GRLGPU_ERR_ARG = -1,        /* bad argument (null pointer, symbol width not in {1,2,4,8}, empty text) */
    GRLGPU_ERR_ILL_FORMED = -2, /* "Error: the file is ill formed" (external/cdt/lib/utils.cpp:177-180) */
    GRLGPU_ERR_CUDA = -3,       /* CUDA runtime error / no device */
    GRLGPU_ERR_NOMEM = -4,      /* device memory exhausted */
    GRLGPU_ERR_STATE = -5,      /* call out of order (no text, phase already finished, ...) */
    GRLGPU_ERR_LIMIT = -6       /* dictionary of one round exceeds 2^32 symbols or the table 2^31 slots; symbol 2^64 - 1, or
                                   alphabet + dictionary symbols + 8 above 2^64 */
};

/* flags of grlgpu_create */
#define GRLGPU_FLAG_SMALL_TABLE 1ull /* tests: start the phrase table tiny so the regrow path runs */
#define GRLGPU_FLAG_FORCE_SLOW_SCAN 2ull /* tests: always take the long-run (summary/resolve) LMS path */
#define GRLGPU_FLAG_FORCE_UNCACHED 8ull /* tests: dedup every phrase with the thread-per-phrase kernel (no cached tiles) */
#define GRLGPU_FLAG_SMALL_PILOT 16ull /* tests: one pilot tile, so small inputs exercise pilot + remainder */
#define GRLGPU_FLAG_FORCE_DOUBLING 32ull /* tests: refine suffix groups by prefix doubling even when key extension would do */
#define GRLGPU_FLAG_KEEP_DICT 4ull /* tests: keep the last round's dictionary for grlgpu_fetch_dictionary */
#define GRLGPU_FLAG_FORCE_WALK 64ull /* tests: grlgpu_invert walks every string, grlgpu_fm_locate walks every occurrence and grlgpu_fm_extract walks every request from its string's end, whatever the chain lengths */
#define GRLGPU_FLAG_FORCE_JUMP 128ull /* tests: grlgpu_invert runs pointer jumping, grlgpu_fm_locate answers from its table and grlgpu_fm_extract starts from the samples, whatever the chain lengths */

/* = str_collection (external/cdt/include/utils.h:20-28) as filled by collection_stats (utils.cpp:100-189) */
typedef struct {
    uint64_t n_syms;
    uint64_t n_strings;
    uint64_t longest_string;
    uint64_t min_sym;
    uint64_t max_sym;
    uint64_t max_sym_freq; /* byte alphabet: highest histogram count; wider alphabets: n_syms (utils.cpp:117) */
    uint64_t sep_sym;
} grlgpu_stats_t;

/* what one parse round reports (the "Stats:" block of par_round, lib/exact_algo/exact_par_phase.cpp:484-488,
 * plus the sizes the caller needs to fetch the level's artefacts) */
typedef struct {
    uint64_t round;          /* 1-based */
    uint64_t n_in;           /* cells of the round's input text */
    uint64_t n_strings;
    uint64_t parse_len;      /* p: phrase occurrences = cells of the output parse ("Parse size") */
    uint64_t n_phrases;      /* d: distinct phrases ("Parsing phrases") */
    uint64_t dict_syms;      /* sum of phrase lengths ("Number of symbols in the phrases") */
    uint64_t max_freq;       /* highest phrase frequency */
    uint64_t alphabet;       /* A: alphabet size of the input text (= tot_phrases of the previous round) */
    uint64_t tot_phrases;    /* ranks handed out = "Number of unsolved BWT blocks" */
    uint64_t n_pre_runs;     /* runs of the preliminary BWT of this level */
    uint64_t algorithmic_bytes; /* B_r = n*w + p*w' + dict_syms*w + 8*d (SURVEY.md 8d) */
    uint32_t cell_bytes_in;  /* w  */
    uint32_t cell_bytes_out; /* w' by sym_width(tot_phrases)+1 (exact_par_phase.cpp:456-465) */
    uint32_t sym_bytes;      /* element width (4 or 8) of rule_l / rule_r / pre_sym in grlgpu_fetch_level */
    uint32_t done;           /* 1 when parse_len == n_strings (exact_par_phase.cpp:496) */
    float device_ms;         /* CUDA-event time of the whole round on the context's stream */
    float text_pass_ms;      /* of which: boundary scan + compaction + dedup (text read) */
    float dict_ms;           /* of which: dictionary gather + suffix ordering + ranks + rules */
    float rewrite_ms;        /* of which: rewrite */
} grlgpu_round_t;

/* context on one device. replaces: construction of the parse strategy (exact_par_phase.cpp:265-283) */
int grlgpu_create(grlgpu_ctx** ctx, int device, uint64_t flags);
/* same, but every kernel and copy is issued on the caller's CUDA stream (a cudaStream_t), so the
 * caller can bracket calls with its own events (bench.py passes torch's current stream) */
int grlgpu_create_on_stream(grlgpu_ctx** ctx, int device, uint64_t flags, void* cuda_stream);
int grlgpu_destroy(grlgpu_ctx* ctx);

/* round-1 input, caller-owned HOST memory, copied to the device. replaces: i_file_stream over the
 * input file (external/cdt/include/file_streams.hpp:93-105) */
int grlgpu_set_text(grlgpu_ctx* ctx, const void* text, uint64_t n_syms, int sym_bytes);
/* same, text already resident in DEVICE memory (16-byte aligned); borrowed, not copied, never written */
int grlgpu_set_text_device(grlgpu_ctx* ctx, const void* dev_text, uint64_t n_syms, int sym_bytes);

/* Streaming ingest of the round-1 input (what i_file_stream's 8 MB windows do for the reference,
 * external/cdt/include/file_streams.hpp:93-105): begin allocates the device text and two pinned staging buffers of
 * stage_bytes (0: 16 MB); stage hands out the next free buffer (*cap bytes of it may be filled, e.g. by read() from the input
 * file); commit enqueues its copy to the device on the copy stream and returns at once, so the caller fills the other
 * buffer meanwhile; end waits for the last copy. The bytes must be committed in text order. */
int grlgpu_text_begin(grlgpu_ctx* ctx, uint64_t n_syms, int sym_bytes, uint64_t stage_bytes);
int grlgpu_text_stage(grlgpu_ctx* ctx, void** buf, uint64_t* cap);
int grlgpu_text_commit(grlgpu_ctx* ctx, uint64_t bytes);
int grlgpu_text_end(grlgpu_ctx* ctx);

/* replaces: collection_stats<sym_type>() (utils.cpp:100-189); validates sep == min && last == sep */
int grlgpu_stats(grlgpu_ctx* ctx, grlgpu_stats_t* out);

/* one parse round on the device. replaces: par_round<strategy>() (exact_par_phase.cpp:374-497):
 * get_phrases (parsing_strategies.h:244-275 / :618-642), dictionary + process_dictionary
 * (exact_par_phase.hpp:106-183, exact_par_phase.cpp:97-263), metasymbol assignment (:427-450),
 * parse_text (parsing_strategies.h:388-497 / :644-676). The new parse stays on the device. */
int grlgpu_round(grlgpu_ctx* ctx, grlgpu_round_t* out);

/* artefacts of the last round for the induction phase, copied to caller-owned host buffers.
 * replaces: files dict_lev_k (exact_par_phase.hpp:189-203) and pre_bwt_lev_k (exact_par_phase.cpp:150-155).
 *   rule_l, rule_r : tot_phrases elements of sym_bytes each (dict[2u], dict[2u+1] of produce_grammar,
 *                    numeric conventions of exact_par_phase.cpp:19-20: alphabet A+3, dummy A+3+tot+1)
 *   has_hocc       : tot_phrases bytes (phrases_has_hocc)
 *   pre_sym/len    : n_pre_runs runs, maximal; dummies A+1 (from BWT i+1) and A+2 (from hocc buffer)
 * any pointer may be NULL to skip that array. */
int grlgpu_fetch_level(grlgpu_ctx* ctx, void* rule_l, void* rule_r, uint8_t* has_hocc, void* pre_sym, uint64_t* pre_len);

/* same copies, issued on a second stream: the call returns at once and the NEXT round may run while they are in
 * flight (give pinned host buffers, or the driver stages and the overlap is lost). The level's device buffers
 * stay parked until grlgpu_fetch_wait, which must be called before the host buffers are read. After this call the
 * level can no longer be fetched again. */
int grlgpu_fetch_level_async(grlgpu_ctx* ctx, void* rule_l, void* rule_r, uint8_t* has_hocc, void* pre_sym, uint64_t* pre_len);
/* grlgpu_fetch_level with 32-bit run lengths (async != 0: as grlgpu_fetch_level_async, completed by grlgpu_fetch_wait).
 * The run lengths of a level sum to at most n_in + parse_len: GRLGPU_ERR_LIMIT when that is >= 2^32 (use the 64-bit call).
 * 4 bytes less per preliminary-BWT run over PCIe; replaces the same files as grlgpu_fetch_level. */
int grlgpu_fetch_level32(grlgpu_ctx* ctx, void* rule_l, void* rule_r, uint8_t* has_hocc, void* pre_sym, uint32_t* pre_len32, int async);
int grlgpu_fetch_wait(grlgpu_ctx* ctx);
/* Hand-over of the last level (grlgpu_round) or level slice (grlgpu_mg_round) to host-side fetch threads: the device arrays
 * are parked -- kept alive until grlgpu_fetch_wait -- and their DEVICE addresses returned; any host thread may copy them with
 * grlgpu_copy_to_host (blocking, on a stream of its own) while the context's thread runs the next round. len_bytes: width of
 * the run lengths handed out (4 only when n_in + parse_len < 2^32: GRLGPU_ERR_LIMIT otherwise). */
typedef struct {
    const void *rule_l, *rule_r, *has_hocc, *pre_sym, *pre_len;
    uint64_t tot, n_pre;       /* elements of rule_l / rule_r / has_hocc and of pre_sym / pre_len */
    uint32_t sym_bytes, len_bytes;
    int device;
} grlgpu_level_ptrs_t;
int grlgpu_level_park(grlgpu_ctx* ctx, int len_bytes, grlgpu_level_ptrs_t* out);
int grlgpu_copy_to_host(int device, void* dst, const void* dev_src, uint64_t bytes);
/* ---- induction phase on the device (grlbwt_b200/csrc/induce.cuh) -----------------------------------------------------
 * replaces, for collections of fewer than 2^32 symbols whose levels have 32-bit symbols, the host's level-by-level induction
 * (exact_algo::ind_phase<b>, lib/exact_algo/exact_ind_phase.cpp:111-386,:603-697): the levels never leave the device.
 *   grlgpu_keep_level     after a round, instead of fetching the level: keep its artefacts on the device
 *   grlgpu_level_adopt    multi-GPU: an empty kept level of the given sizes on THIS context; the ranks copy their slices into the
 *                         returned device arrays with grlgpu_copy_dev (rules at rank_base, runs at pre_first; pre_len is 64-bit)
 *   grlgpu_induce         the whole induction, deepest level first; final_parse: host buffer of n_strings cells in string
 *                         order, or NULL to use the context's own final parse. The kept levels are consumed.
 *                         GRLGPU_ERR_LIMIT / GRLGPU_ERR_NOMEM: the caller falls back to the host induction after
 *                         grlgpu_fetch_kept_level (the kept levels survive a failure).
 *   grlgpu_fetch_bwt      the level-0 BWT as maximal runs: n_runs 32-bit symbols and 32-bit lengths */
int grlgpu_keep_level(grlgpu_ctx* ctx);
int grlgpu_level_adopt(grlgpu_ctx* ctx, uint64_t alphabet, uint64_t tot, uint64_t n_pre, grlgpu_level_ptrs_t* out);
int grlgpu_copy_dev(int dst_device, void* dst, int src_device, const void* src, uint64_t bytes);
int grlgpu_kept_levels(const grlgpu_ctx* ctx);
int grlgpu_device_of(const grlgpu_ctx* ctx);  /* CUDA device of the context */
int grlgpu_fetch_kept_level(grlgpu_ctx* ctx, int level, uint64_t* alphabet, uint64_t* tot, uint64_t* n_pre, void* rule_l, void* rule_r, uint8_t* has_hocc,
                            void* pre_sym, uint64_t* pre_len);
int grlgpu_drop_kept(grlgpu_ctx* ctx);
int grlgpu_induce(grlgpu_ctx* ctx, const void* final_parse, uint64_t n_strings, int cell_bytes, uint64_t n_syms_total, uint64_t* n_runs);
int grlgpu_fetch_bwt(grlgpu_ctx* ctx, uint32_t* syms, uint32_t* lens);
/* the level-0 BWT as the image of the reference's .rl_bwt file (main.cpp:146-152 -> bwt_buff_writer): [sb u64][fb u64] then n_runs
 * records of sb symbol bytes + fb length bytes, little endian, packed on the device (16 + n_runs * (sb + fb) bytes travel instead of
 * 8 bytes per run). *n_bytes = size of the image; GRLGPU_ERR_ARG if cap_bytes is smaller (nothing is copied). */
int grlgpu_fetch_bwt_packed(grlgpu_ctx* ctx, int sb, int fb, void* out, uint64_t cap_bytes, uint64_t* n_bytes);
/* the same arrays as DEVICE addresses (valid until grlgpu_drop_kept / the next grlgpu_induce), for parallel grlgpu_copy_to_host */
int grlgpu_bwt_ptrs(grlgpu_ctx* ctx, const uint32_t** d_syms, const uint32_t** d_lens, uint64_t* n_runs);

/* inversion of a BCR BWT: the .rl_bwt image back to the collection (replaces scripts/reverse_bwt.cpp:5-54)
 * image: [sb u64][fb u64] + records of sb symbol bytes and fb length bytes, little endian (what grlgpu_fetch_bwt_packed and the CLI
 * write). The separator is the smallest symbol, N = its count; out receives the first min(n_seqs, N) strings, each followed by the
 * separator, as cells of cell_bytes little-endian bytes: byte for byte what `reverse_bwt image out [n_seqs] -a cell_bytes` writes.
 * GRLGPU_ERR_ARG: sb or fb outside 1..8, a partial record, no record, cell_bytes not in {1,2,4,8}, or cap_bytes smaller than
 * n_out * cell_bytes (info->n_out is then set). GRLGPU_ERR_LIMIT: n >= 0xfffffff0 or a symbol / length >= 2^32 (the host tool
 * reverse_bwt is the general path). GRLGPU_ERR_ILL_FORMED: the run list is not a BWT (its LF has a cycle without separator).
 * Needs no text in the context and leaves its text, levels and BWT untouched. The path (walk per string or pointer jumping) is
 * chosen from the chain lengths the call observes (GRLGPU_FLAG_FORCE_WALK / _JUMP force one, for tests). */
typedef struct {
    uint64_t n, n_strings, n_runs;   /* BWT length, separators, records of the image */
    uint64_t n_out;                  /* cells written (or needed, when cap_bytes is too small) */
    uint32_t path;                   /* 0 walk per string, 1 pointer jumping */
    uint32_t jump_rounds;
    float device_ms, lf_ms, invert_ms; /* CUDA events on the context's stream: whole call / table / inversion */
} grlgpu_invert_t;
int grlgpu_invert(grlgpu_ctx* ctx, const void* image, uint64_t image_bytes, int cell_bytes,
                  uint64_t n_seqs /* UINT64_MAX: all */, void* out, uint64_t cap_bytes, grlgpu_invert_t* info);

/* search of a BCR BWT: the .rl_bwt image loaded as a run-length FM-index on the device (grlbwt_b200/csrc/fm.cuh). The reference has
 * no such interface (its scripts/fm_index.h only serves reverse_bwt); the host tool fm_query is the general path and the same answers.
 * Conventions of grlgpu_invert: the separator is the smallest symbol of a non-empty record, N = its count, S_0 .. S_{N-1} the strings
 * in the order reverse_bwt writes them (input order). An occurrence of a pattern P (m >= 1 cells) is a pair (k, p) with
 * S_k[p .. p + m) = P; overlapping occurrences all count; a pattern containing the separator or a symbol absent from the BWT has none.
 *   grlgpu_fm_load    builds the index from an image (checks and GRLGPU_ERR_LIMIT exactly as grlgpu_invert) and keeps it in the
 *                     context: at most one index, so a load first drops the index already loaded (a failed load leaves none). Its
 *                     memory comes from the context's pool; the context's text, levels and BWT are left untouched.
 *   grlgpu_fm_count   backward search of n_pat patterns: pattern q is cells [pat_off[q], pat_off[q + 1]) of pat, cells of pat_bytes
 *                     little-endian bytes. sp_ep[2q], sp_ep[2q + 1] = the rows [sp, ep) whose suffix starts with the pattern, its
 *                     count ep - sp; a pattern without occurrence gets sp = ep = 0.
 *   grlgpu_fm_locate  every occurrence: occ_off[q] .. occ_off[q + 1] (n_pat + 1 entries) are pattern q's, listed in row order
 *                     sp, sp + 1, ..: str_id = k, str_pos = p. Each occurrence walks LF and psi from its row, at most
 *                     B = max(4096, n / 2048) steps; a longer walk makes the call, and every later call on the index, answer from
 *                     a table of (k, p) for every row, built once by pointer jumping (GRLGPU_FLAG_FORCE_WALK / _JUMP force one path).
 *   grlgpu_fm_drop    frees the index (grlgpu_destroy does too).
 * GRLGPU_ERR_ARG: pat_bytes not in {1,2,4,8}, pat_off[0] != 0, an empty pattern (offsets not increasing), cap_occ < n_occ (info->n_occ
 * is then set to the number needed). GRLGPU_ERR_STATE: count or locate without a loaded index. GRLGPU_ERR_ILL_FORMED: the run list is
 * not a BWT (its LF has a cycle without separator) and a locate met it. n_pat = 0 is accepted and writes nothing. */
typedef struct {
    uint64_t n, n_strings, n_runs;  /* BWT length, separators, records of the image */
    uint64_t sigma;                 /* distinct symbols of the records */
    uint64_t sep;                   /* the separator */
    float load_ms;                  /* CUDA events on the context's stream: image upload and every table of the index */
} grlgpu_fm_t;
typedef struct {
    uint64_t n_pat, n_pat_syms;     /* patterns and their cells */
    uint64_t n_occ;                 /* locate: occurrences (written, or needed when cap_occ is too small) */
    uint32_t path;                  /* locate: 0 walk per occurrence, 1 the table */
    uint32_t jump_rounds;           /* locate: pointer-jumping rounds when this call built the table, else 0 */
    float device_ms, search_ms, locate_ms; /* CUDA events on the context's stream: whole call (copies included) / backward search / locate */
} grlgpu_fm_query_t;
int grlgpu_fm_load(grlgpu_ctx* ctx, const void* image, uint64_t image_bytes, grlgpu_fm_t* info);
int grlgpu_fm_count(grlgpu_ctx* ctx, const void* pat, const uint64_t* pat_off /* n_pat + 1 cell offsets */, uint64_t n_pat, int pat_bytes,
                    uint64_t* sp_ep /* 2 * n_pat */, grlgpu_fm_query_t* info);
int grlgpu_fm_locate(grlgpu_ctx* ctx, const void* pat, const uint64_t* pat_off, uint64_t n_pat, int pat_bytes, uint64_t* occ_off /* n_pat + 1 */,
                     uint32_t* str_id, uint32_t* str_pos, uint64_t cap_occ, grlgpu_fm_query_t* info);
int grlgpu_fm_drop(grlgpu_ctx* ctx);

/* search with mismatches on the loaded index (the host tool fm_query -k is the general path and the same answers). An occurrence
 * of P with d mismatches is a pair (k, p) such that the window S_k[p .. p + m) lies inside string k and differs from P in exactly
 * d <= max_mismatches positions (Hamming distance). A pattern cell that is the separator or a symbol absent from the BWT never
 * matches; substitutions use the symbols of the BWT other than the separator. A hit is one distinct string Q with
 * Hamming(P, Q) <= max_mismatches that occurs: its rows [sp, ep) and its d. Hits of one pattern are disjoint and listed by
 * ascending sp, so its occurrences are listed in row order. max_mismatches = 0 gives the answers of grlgpu_fm_count / _locate
 * (without the empty intervals).
 *   grlgpu_fm_approx_count   pattern q's hits are hit_off[q] .. hit_off[q + 1] (n_pat + 1 entries): sp_ep[2h], sp_ep[2h + 1] and
 *                            hit_mm[h] = d. One thread per pattern runs a depth-first backward search over at most
 *                            max_mismatches + 1 frames, pruning every empty interval.
 *   grlgpu_fm_approx_locate  every occurrence of every hit: occ_off[q] .. occ_off[q + 1] are pattern q's, str_id = k, str_pos = p,
 *                            occ_mm = d, in row order; the locate paths, flags and table of grlgpu_fm_locate.
 * GRLGPU_ERR_ARG: the pattern checks of grlgpu_fm_count, max_mismatches > 3, a null array, or cap_hits < n_hits / cap_occ < n_occ
 * (info->n_hits / n_occ then hold the number needed; nothing is written). GRLGPU_ERR_STATE: no index loaded. GRLGPU_ERR_LIMIT:
 * n_pat >= 2^32 or 2^32 hits or more. GRLGPU_ERR_ILL_FORMED: locate only, as grlgpu_fm_locate. n_pat = 0 is accepted. */
typedef struct {
    uint64_t n_pat, n_pat_syms;     /* patterns and their cells */
    uint64_t n_hits;                /* hits (written, or needed when cap_hits is too small) */
    uint64_t n_occ;                 /* sum of ep - sp over the hits (locate: written, or needed when cap_occ is too small) */
    uint64_t n_lf;                  /* LF_c evaluations of the search */
    uint32_t path, jump_rounds;     /* locate, as grlgpu_fm_query_t */
    float device_ms, search_ms, locate_ms; /* CUDA events on the context's stream: whole call (copies included) / search / locate */
} grlgpu_fm_approx_t;
int grlgpu_fm_approx_count(grlgpu_ctx* ctx, const void* pat, const uint64_t* pat_off, uint64_t n_pat, int pat_bytes, uint32_t max_mismatches,
                           uint64_t* hit_off /* n_pat + 1 */, uint64_t* sp_ep /* 2 * cap_hits */, uint8_t* hit_mm, uint64_t cap_hits, grlgpu_fm_approx_t* info);
int grlgpu_fm_approx_locate(grlgpu_ctx* ctx, const void* pat, const uint64_t* pat_off, uint64_t n_pat, int pat_bytes, uint32_t max_mismatches,
                            uint64_t* occ_off /* n_pat + 1 */, uint32_t* str_id, uint32_t* str_pos, uint8_t* occ_mm, uint64_t cap_occ, grlgpu_fm_approx_t* info);

/* extract from the loaded index (the host tool fm_extract is the general path and writes the same cells):
 *   grlgpu_fm_extract  substrings of the indexed strings: request q = (str_id[q], from[q], len[q]) yields S_k[from .. e) with
 *                      k = str_id[q], e = min(from + len, L_k) (computed in 64 bits, so len = UINT32_MAX means "to the end");
 *                      from >= e yields nothing. Cells of cell_bytes little-endian bytes, each the symbol's low bytes (as
 *                      reverse_bwt's put_cell), no separators. out_off (n_req + 1 entries) receives the cell offsets:
 *                      request q is cells [out_off[q], out_off[q + 1]) of out.
 *                      Each request walks LF back from row k, the end of string k: a count pass of at most B = max(4096, n / 2048)
 *                      steps gives L_k, a write pass walks again. A string longer than B makes the call, and every later call on the
 *                      index, start from sampled rows instead: every 64th position of every string, taken from the locate table of
 *                      grlgpu_fm_locate (built by pointer jumping when no call built it before, and then shared by both calls).
 *                      GRLGPU_FLAG_FORCE_WALK / _JUMP force one path. A walk from row k always ends (the LF cycle of k holds the
 *                      separator row LF^-1(k)), so only the sampled path can meet a run list that is not a BWT.
 * GRLGPU_ERR_ARG: cell_bytes not in {1,2,4,8}, a null array with n_req > 0, some str_id >= N, or cap_cells < n_cells
 * (info->n_cells then holds the number needed, and device_ms / extract_ms the time spent, nothing is written). GRLGPU_ERR_STATE: no index loaded. GRLGPU_ERR_LIMIT: n_req >= 2^32.
 * GRLGPU_ERR_ILL_FORMED: the call needed the locate table and the run list is not a BWT. n_req = 0 is accepted. */
typedef struct {
    uint64_t n_req, n_cells;     /* requests; cells written (or needed, when cap_cells is too small) */
    uint32_t path;               /* 0 walk per request, 1 from the samples */
    uint32_t jump_rounds;        /* pointer-jumping rounds when this call built the locate table, else 0 */
    float device_ms, extract_ms; /* CUDA events on the context's stream: whole call (copies included) / the extraction */
} grlgpu_fm_extract_t;
int grlgpu_fm_extract(grlgpu_ctx* ctx, const uint32_t* str_id, const uint32_t* from, const uint32_t* len, uint64_t n_req,
                      int cell_bytes, uint64_t* out_off /* n_req + 1 */, void* out, uint64_t cap_cells, grlgpu_fm_extract_t* info);

/* LCP array of the loaded index (the host tool fm_lcp is the general path and writes the same values). Row j's suffix is
 * S_k[p .. L_k) followed by $_k, where (k, p) is the row's locate entry; rows j < N are the $_k rows. lcp[0] = 0 and, for j >= 1,
 * lcp[j] = the number of leading cells shared by the suffixes of rows j - 1 and j, where a separator never matches (itself
 * included): rows j < N have 0, no value crosses a string's end, and the values do not depend on how separators are tie-broken.
 *   grlgpu_fm_lcp  writes n values in row order. SA and the text come from a walk per string (the count pass of grlgpu_fm_extract,
 *                  bound B = max(4096, n / 2048)) or from the locate table of grlgpu_fm_locate: the table answers when it exists, when a
 *                  string is longer than B (built here by pointer jumping, then kept for every later call) or under
 *                  GRLGPU_FLAG_FORCE_JUMP; GRLGPU_FLAG_FORCE_WALK walks with bound n. Only the rows that start a BWT run or hold the
 *                  separator (irreducible) compare text; every other row follows from its LF successor.
 * GRLGPU_ERR_ARG: a null lcp with n > 0, or cap < n (info->n then holds n, nothing is written). GRLGPU_ERR_STATE: no index loaded.
 * GRLGPU_ERR_ILL_FORMED: the run list is not a BWT (its LF has a cycle without separator), through either path. */
typedef struct {
    uint64_t n;                 /* rows: entries written (or needed, when cap is too small) */
    uint64_t n_irreducible;     /* rows whose LCP was found by comparing cells */
    uint64_t sum_irreducible;   /* sum of those rows' LCP values */
    uint32_t path, jump_rounds; /* 0 walk per string, 1 the locate table; rounds when this call built the table, else 0 */
    float device_ms, sa_ms, lcp_ms; /* CUDA events: whole call incl. the copy out / SA + text / irreducible rows, scan and gather */
} grlgpu_fm_lcp_t;
int grlgpu_fm_lcp(grlgpu_ctx* ctx, uint32_t* lcp /* n */, uint64_t cap, grlgpu_fm_lcp_t* info);

/* digest of the last round's level artefacts, computed on the device before they are fetched: four sums mod 2^64
 * {rules weighted by rank, hocc marks weighted by rank, sum of the preliminary-BWT run lengths, runs weighted by symbol}.
 * The sums of the per-rank slices of a multi-GPU level add up to the single-GPU value, so bench.py can check that 1, 2,
 * 4 and 8 ranks produced the same dict_lev_k / pre_bwt_lev_k (exact_par_phase.hpp:189-203, exact_par_phase.cpp:150-155). */
int grlgpu_level_checksum(grlgpu_ctx* ctx, uint64_t* out4);

/* current parse (output of the last round): parse_len cells of cell_bytes_out bytes, cells = rank<<1|rep.
 * replaces: file tmp_input (exact_par_phase.cpp:307-308); after the last round this is the final parse
 * consumed by parse2bwt (exact_ind_phase.cpp:603-672) */
int grlgpu_fetch_parse(grlgpu_ctx* ctx, void* dst);
/* start offset of every string in the current parse, n_strings+1 entries (parsing_info::str_ptrs) */
int grlgpu_fetch_str_ptrs(grlgpu_ctx* ctx, uint64_t* dst);
/* dictionary of the last round in insertion-independent form, for tests: phrases listed in the A.2
 * order; syms: dict_syms u64 values, lens/freqs/metas: n_phrases entries (NULL to skip) */
int grlgpu_fetch_dictionary(grlgpu_ctx* ctx, uint64_t* syms, uint64_t* lens, uint64_t* freqs, uint64_t* metas);

/* Device memory that destroyed contexts left mapped for the next context of this process (mapping tens of GB costs more than a parse
 * phase; GRLGPU_POOL_CACHE=0 disables the cache) goes back to the driver; returns the bytes released. An allocation that would
 * otherwise fail does this by itself. */
uint64_t grlgpu_trim(void);

const char* grlgpu_strerror(int status);
const char* grlgpu_last_error(const grlgpu_ctx* ctx);   /* ctx == NULL: the calling thread's last error of a call without a context */

/* ---- multi-GPU rounds (SURVEY.md 8e) ----------------------------------------------------------------------
 * One context per GPU = one rank, each holding a shard of WHOLE strings (the reference's own split,
 * include/parsing_strategies.h:208-214, so no phrase crosses a shard). The library owns the whole round, exchanges
 * included; the global dictionary is never replicated: phrases are partitioned by owner (content hash), their suffix
 * entries by first-key range, the grammar rules by rank range (grlbwt_b200/csrc/mg2.cuh). All ranks make the same
 * calls in the same order:
 *     grlgpu_set_text[_device] (its shard)  ->  grlgpu_mg_stats  ->  grlgpu_mg_round until done
 *     after every round: grlgpu_mg_slice_info + grlgpu_mg_fetch_slice (this rank's part of the level)
 *     after the last: grlgpu_fetch_parse (one cell per local string; rank order = string order)
 * replaces: mt_parse_strat_t's thread fan-out + serial join_thread_phrases (parsing_strategies.h:244-386) and shards
 * suffix_induction / produce_pre_bwt / produce_grammar (exact_LMS_induction.h:94-158, exact_par_phase.cpp:14-242).
 *
 * Exchange backends (grlgpu_comm): NCCL -- one rank per process (bench.py under torchrun: rank 0 makes the id, the
 * launcher broadcasts its 128 bytes) or per host thread (the grlbwt CLI with --gpus N); "ipc" -- one rank per process
 * on ONE box: every rank stages what it sends in a device window that its peers map through CUDA IPC and pull from
 * with copy-engine DMA over NVLink, the rendezvous lives in a POSIX shared-memory segment named `session` ("/name",
 * the same string on every rank, e.g. broadcast by the launcher; rank 0 creates and unlinks it); "local" -- ranks are host
 * threads of one process that pull from each other's send buffers with peer copies (NVLink P2P between GPUs, plain
 * device copies when several ranks share one GPU: how the N > 1 path is tested on a 1-GPU box). NCCL is resolved
 * with dlopen at the first use; the library loads without it. */
typedef struct grlgpu_comm grlgpu_comm;
typedef struct grlgpu_local_group grlgpu_local_group;
int grlgpu_nccl_unique_id(void* id128);
int grlgpu_comm_create_nccl(grlgpu_comm** comm, const void* id128, int rank, int world, int device);
int grlgpu_comm_create_ipc(grlgpu_comm** comm, const char* session, int rank, int world, int device);
int grlgpu_local_group_create(grlgpu_local_group** group, int world);
int grlgpu_local_group_abort(grlgpu_local_group* group);   /* a rank failed: wake the ranks waiting for it (they return GRLGPU_ERR_STATE) */
int grlgpu_local_group_destroy(grlgpu_local_group* group);
int grlgpu_comm_create_local(grlgpu_comm** comm, grlgpu_local_group* group, int rank, int device);
int grlgpu_comm_destroy(grlgpu_comm* comm);
/* bytes this rank sent in bulk exchanges so far, bulk / small collectives issued, backend description */
int grlgpu_comm_info(const grlgpu_comm* comm, uint64_t* bytes_sent, uint64_t* n_bulk, uint64_t* n_small, char* kind, int kind_cap);
/* host wall time (ms) this rank has spent inside bulk exchanges (from "my data is ready" to "everything has arrived", so it
 * includes waiting for slower peers) and inside the small gathers */
int grlgpu_comm_times(const grlgpu_comm* comm, double* ms_bulk, double* ms_small);
/* in-process ranks on different GPUs: let the listed devices read this context's memory pool directly (NVLink P2P) */
int grlgpu_set_peers(grlgpu_ctx* ctx, const int* devices, int n_devices);
int grlgpu_can_peer(int device_a, int device_b);   /* 1 if the two devices can address each other's memory (NVLink / PCIe P2P) */

/* byte alphabets: the 256-bin symbol histogram behind grlgpu_stats */
int grlgpu_histogram(grlgpu_ctx* ctx, uint64_t* hist256);
/* collection_stats (utils.cpp:100-189) over ALL shards; fixes the global alphabet and string count in the context.
 * Fails with GRLGPU_ERR_ILL_FORMED on every rank if any shard is ill formed. */
int grlgpu_mg_stats(grlgpu_ctx* ctx, grlgpu_comm* comm, grlgpu_stats_t* global_out);
/* one parse round over all ranks (= grlgpu_round; the scalars of `out` describe the GLOBAL round, algorithmic_bytes and
 * the times this rank's share). */
int grlgpu_mg_round(grlgpu_ctx* ctx, grlgpu_comm* comm, grlgpu_round_t* out);

/* this rank's part of the level produced by the last grlgpu_mg_round: rules / hocc marks of the ranks
 * [rank_base, rank_base + tot_local) and the preliminary-BWT runs [pre_first, pre_first + n_pre_local) of the level
 * (runs that continue across two ranks' ranges are already merged into the earlier rank's last run) */
typedef struct {
    uint64_t rank_base, tot_local;
    uint64_t pre_first, n_pre_local;
    uint64_t exchange_bytes;   /* bulk bytes this rank sent to its peers during the round */
    uint64_t n_in_local, parse_len_local; /* cells of this rank's shard before / after the round (grlgpu_fetch_parse copies parse_len_local cells) */
    uint32_t sym_bytes;        /* element width (4 or 8) of rule_l / rule_r / pre_sym */
    uint32_t reserved;
} grlgpu_slice_t;
int grlgpu_mg_slice_info(grlgpu_ctx* ctx, grlgpu_slice_t* out);
/* copies the slice into caller-owned HOST buffers (NULL skips an array); pre_len elements are len_bytes (4 or 8) wide.
 * async != 0: copies run on the copy stream while the next round computes; complete them with grlgpu_fetch_wait. */
int grlgpu_mg_fetch_slice(grlgpu_ctx* ctx, void* rule_l, void* rule_r, uint8_t* has_hocc, void* pre_sym, void* pre_len, int len_bytes, int async);
/* grlgpu_level_checksum of the slice: the four sums of all ranks add up (mod 2^64) to the single-GPU level's */
int grlgpu_mg_slice_checksum(grlgpu_ctx* ctx, uint64_t* out4);

/* launch accounting: number of kernel launches issued by this context so far, and (after
 * grlgpu_profile_enable(ctx, 1)) per-kernel CUDA-event durations measured live on the launch stream.
 * grlgpu_profile_entry returns 1 past the last entry; model_bytes = expected DRAM bytes of the launches. */
int grlgpu_profile_enable(grlgpu_ctx* ctx, int on);
int grlgpu_profile_reset(grlgpu_ctx* ctx);
uint64_t grlgpu_launch_count(const grlgpu_ctx* ctx);
int grlgpu_profile_entry(grlgpu_ctx* ctx, int index, char* name, int name_cap, uint64_t* launches, double* total_ms, uint64_t* model_bytes);

/* self-test hooks for the device primitives the path is built from (host buffers in / out) */
int grlgpu_selftest_scan(const uint32_t* in, uint64_t n, uint64_t* out_exclusive, uint64_t* total);
int grlgpu_selftest_sort(uint64_t* keys, uint32_t* vals, uint64_t n, int n_bits);
/* exclusive scan with input and output of one type (elem_bytes 4: uint32_t, wrapping mod 2^32; 8: uint64_t). The device arrays start
 * elem_offset elements into their allocation (an odd offset makes them not 16-byte aligned); in_place != 0 scans the input array over itself */
int grlgpu_selftest_scan_same(const void* in, uint64_t n, int elem_bytes, uint64_t elem_offset, int in_place, void* out_exclusive, void* total);
/* (uint32_t key, uint32_t value) pairs: partition_shift < 0 sorts on the low n_bits (radix_sort_pairs_u32, whole 8-bit digits), else one
 * stable partition pass on the digit at partition_shift (radix_partition_u32) */
int grlgpu_selftest_sort32(uint32_t* keys, uint32_t* vals, uint64_t n, int n_bits, int partition_shift);
int grlgpu_selftest_compact(const uint32_t* bits, const uint32_t* prev_bits, uint64_t n_bits, uint64_t* out, uint64_t* count);
/* the shared-memory rendezvous of the "ipc" backend WITHOUT its device windows (runs on a box without a GPU): `rounds` barriers and small
 * all-gathers of varying size between `world` processes that all pass the same `session`; GRLGPU_OK when every byte arrived intact */
int grlgpu_selftest_ipc_rendezvous(const char* session, int rank, int world, int rounds);

#ifdef __cplusplus
}
#endif
#endif /* GRLGPU_H */
