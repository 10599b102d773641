/*
 * rnascan_b200 -- C ABI of the B200 (sm_100a) motif-scoring library, librnascan_b200.so.
 *
 * This is the drop-in boundary for rnascan's sliding-window scoring path.  The reference
 * has exactly one native entry point on that path,
 *
 *     rnascan.BioAddons.motifs._pwm.calculate(sequence, matrix) -> float32[n-m+1]
 *         /root/reference/rnascan/BioAddons/motifs/_pwm.c:79-121 (arithmetic :8-70)
 *
 * called once per window by Biopython's search() from rnascan.py:263; everything else
 * on the path is Python (matrix.py:25-43 one-hot structure scoring, rnascan.py:293-315
 * averaged-profile scoring, rnascan.py:440-465 background counting).  The entry points
 * below replace those loops; each cites what it replaces.  INTEGRATION.md shows the
 * ctypes binding a maintainer of the reference would add.
 *
 * Conventions
 *  - plain C types only; `d_*` pointers are CUDA device addresses, others are host;
 *  - every function returns 0 (RS_OK) or an RS_ERR_* code; rs_last_error() gives text;
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); all work
 *    is enqueued on it, nothing synchronises, nothing allocates: the caller supplies the
 *    workspace (rs_scan_workspace_bytes) and reads counters after syncing the stream
 *    (ONE exception, stated at its declaration: the tensor-core path of rs_scan_batched waits
 *    for its candidate and hit counts, which size the exact pass and the ordering);
 *  - no process-global mutable state: the three knobs (rs_set_reserved_sms, rs_set_batched_path,
 *    rs_prof_begin/_end) and rs_last_error are per calling THREAD, so concurrent callers do
 *    not see each other's settings; everything else is re-entrant like the reference's
 *    _pwm.calculate (_pwm.c has no state, SURVEY.md 8b);
 *  - there is NO CPU fallback: without a CUDA device every device entry point fails.
 *
 * Symbol stream ("codes"), 1 byte per symbol, records concatenated with ONE separator:
 *    bits 0-2 letter index, bit 3 "not counted in the background", 0xFF separator.
 *    RNA   : A=0 C=1 G=2 U/T=3 (either case), anything else 0x0C (window -> NaN)
 *    struct: B=0 E=1 H=2 L=3 M=4 R=5 T=6 ; lower case = index|8 (scored, not counted:
 *            rnascan.py:196-197 + :450-453 count case-sensitively) ; anything else 0x0F
 *    alpha : any other alphabet of 1..31 distinct ASCII letters, none of them lower case a-z
 *            (rs_host_encode_alpha): bits 0-4 index of the UPPER-CASED byte in the caller's
 *            letters, bit 5 set for a lower-case byte (scored, not counted), anything else
 *            0x1F.  0xFF & 31 = 31 >= A, so a separator invalidates a window without a test.
 *    A window that contains a separator is not a window of any record; hit scans never
 *    report it, dense outputs hold NaN there.
 *  Device arrays read by the scan kernels must be allocated with rs_padded_count(n)
 *  elements (codes) / rows (profiles); the padding is never interpreted.
 *
 * Structure channel order everywhere in this ABI is B,E,H,L,M,R,T (the profile file
 * order, pfmutil.py:62-69); PSSM tables are row-major [W][channels].
 */
#ifndef RNASCAN_B200_H
#define RNASCAN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RS_OK            0
#define RS_ERR_INVALID   1   /* bad argument (the reference raises ValueError)          */
#define RS_ERR_CUDA      2   /* CUDA runtime error, including "no device"               */
#define RS_ERR_WORKSPACE 3   /* workspace too small                                     */

#define RS_SEP        0xFF
#define RS_RNA_OTHER  0x0C
#define RS_SS_OTHER   0x0F
#define RS_ALPHA_OTHER 0x1F  /* alphabet layout: byte that is no letter of the alphabet      */
#define RS_ALPHA_LOWER 0x20  /* alphabet layout: lower-case letter (scored, not counted)     */
#define RS_MAX_W      64     /* widest motif the scan kernels accept                    */

#define RS_F32 0
#define RS_F64 1

#define RS_MODE_STRUCT 0     /* hit iff struct score > m                                */
#define RS_MODE_AND    1     /* hit iff seq score > m AND struct score > m (combine(),  */
                             /* rnascan.py:416-434 is an inner join of two thresholded  */
                             /* result sets, SURVEY.md H9)                              */

/* ---- library ---------------------------------------------------------------------- */
int         rs_version(void);
const char *rs_last_error(void);                       /* thread-local                  */
int         rs_device_info(int *sm_count, int *cc_major, int *cc_minor);
int64_t     rs_padded_count(int64_t n);                /* elements/rows to allocate     */
int64_t     rs_scan_workspace_bytes(int64_t n, int64_t hit_capacity);

/* SMs the persistent scan kernels launched BY THE CALLING THREAD leave unoccupied (default 0).  Set it to 1 while a collective runs
 * beside a scan (the all-reduce of the background counts in sharded runs): a persistent kernel that fills
 * every SM's shared memory would otherwise make the collective's kernel wait for the scan to end.      */
int rs_set_reserved_sms(int n);

/* ---- measurement hook (bench.py; no reference counterpart) --------------------------
 * Between rs_prof_begin and rs_prof_end every scan entry point called by the same thread records a CUDA event pair
 * tightly around its main kernel on the caller's stream (at most max_records pairs);
 * rs_prof_end waits for them and returns the per-launch durations in milliseconds.     */
int rs_prof_begin(int max_records);
int rs_prof_end(float *ms_out, int capacity, int *n_records);

/* ---- FASTA text -> symbol stream (replaces fileinput + Bio.SeqIO.parse, rnascan.py:170-174, and
 * Seq.transcribe()/upper(), rnascan.py:186-193, for file inputs) -------------------------------
 * Two passes over an ASCII buffer: rs_host_fasta_index sizes the outputs, rs_host_fasta_fill writes
 * the pre-processed letters (text), their codes, per-record offsets/lengths and the header lines.
 * kind 0 = RNA target alphabet (T->U, upper-cased), 1 = structure contexts (unchanged).      */
int rs_host_fasta_index(const uint8_t *buf, int64_t n, int64_t *n_records, int64_t *n_symbols,
                        int64_t *title_bytes);
int rs_host_fasta_fill(const uint8_t *buf, int64_t n, int kind, uint8_t *text, uint8_t *codes,
                       int64_t *rec_off, int64_t *rec_len, char *titles, int64_t *title_off);

/* ---- averaged-profile text -> float64 rows (replaces the per-file pd.read_table + del struct['PO'] of
 * rnascan.py:296-297 for plain pfmutil.format_pfm files: header PO + B,E,H,L,M,R,T in any order, one
 * tab-separated row per position).  Numbers are converted with pandas' own default algorithm
 * (precise_xstrtod of its C tokenizer: NOT correctly rounded), restated in profile_ingest.cpp, so the
 * rows -- and every score computed from them -- are bit-identical to what the reference reads.
 * rs_host_profiles_open reads and indexes all files on `threads` host threads: rows_per_file[i] = number
 * of rows, or -1 when file i is outside the plain format (the caller parses it with pandas);
 * rs_host_profiles_fill writes file i's rows, channels in B,E,H,L,M,R,T order, at out + 7*row_offsets[i]
 * and sets status[i] = RS_OK, or RS_ERR_INVALID when a field turns out not to be a plain number (again:
 * pandas).  rs_host_profiles_close frees the batch.  rs_host_parse_doubles exposes the converter alone
 * ('\n'-separated tokens; ok[k] = 0 where it declines).                                               */
int rs_host_profiles_open(const char *const *paths, int64_t n_files, int threads, void **handle,
                          int64_t *rows_per_file);
int rs_host_profiles_fill(void *handle, int threads, double *out, const int64_t *row_offsets, int *status);
int rs_host_profiles_close(void *handle);
int rs_host_parse_doubles(const char *text, int64_t n_bytes, double *out, int64_t capacity, int64_t *n_out,
                          uint8_t *ok);

/* ---- host-side encoding (CPU threads; replaces str.upper()/transcribe() + the char
 *      switch of _pwm.c:41-63 and the dict lookup of matrix.py:36-41) ---------------- */
int rs_host_encode_rna(const uint8_t *text, int64_t n, uint8_t *codes);
int rs_host_encode_struct(const uint8_t *text, int64_t n, uint8_t *codes);
/* The alphabet layout for `letters` (n_letters of them, 1..31; RS_ERR_INVALID with a message when a
 * letter is repeated, lower case a-z or not ASCII).  Replaces str.upper() + the dict lookup of
 * matrix.py:36-41 for alphabets other than GAUC and BEHLMRT.                                   */
int rs_host_encode_alpha(const uint8_t *text, int64_t n, const uint8_t *letters, int n_letters,
                         uint8_t *codes);

/* log2(p / b) tables in the arithmetic of Python's math.log(p / b, 2) as Biopython's log_odds
 * uses it (called at rnascan.py:248): prob, out [W][A] row-major, bg [A] normalised.        */
int rs_host_log_odds(const double *prob, const double *bg, int W, int A, double *out);

/* ---- dot-bracket -> structural contexts (replaces scripts/parse_secondary_structure.cpp:65-221,
 * the C++ tool run_folding pipes RNAfold centroids through; O(L) instead of O(L^2)) ------------
 * Structure r is text[offsets[r] .. +lengths[r]) over the alphabet ( ) . ; its annotation over
 * B,E,H,L,M,R,T is written to `out` at the same offsets.  status[r] (may be NULL) = RS_OK or
 * RS_ERR_INVALID (unbalanced parentheses / foreign characters -- the reference has undefined
 * behaviour there).  Host function, multi-threaded over structures.                          */
int rs_host_annotate_structures(const char *text, const int64_t *offsets, const int64_t *lengths,
                                int64_t n_structs, char *out, int *status);

/* ---- hits.tab text from hit arrays (replaces the per-record DataFrames + pd.concat + pd.merge +
 * DataFrame.to_csv of rnascan.py:284-286,401-413,416-434,555-567; same bytes) -------------------
 * Strings come as (blob, offsets[n+1]) pairs indexed by rec[r]; Start = start0[r] + 1,
 * End = start0[r] + width; fragments are text[text_pos[r] .. +width) (NULL prints ".").
 * score kinds: 0 float32 (already rounded) as numpy float32 text; 1 the same widened to a Python
 * float; 2 float64 with Python's round(x, 3) applied here; 3 float64 unrounded (averaged profiles);
 * 4 int32 thousandths of round(x, 3) as rs_scores_dense_struct_milli delivers them (single-modality only).
 * rs_host_format_hits: score_kind | 0x100 prints Start and End as float64 text ("12.0"), which is what
 * pandas makes of a profile directory in which some file had no hit.
 * Returns RS_OK and *written; RS_ERR_WORKSPACE when `capacity` is too small (*written = need);
 * RS_ERR_INVALID when a value is outside the covered text formats (caller falls back).        */
int rs_host_format_hits(int64_t n_rows, int64_t match_id_first, const int64_t *rec, const char *id_blob,
                        const int64_t *id_off, const char *desc_blob, const int64_t *desc_off,
                        const char *motif_id, const int64_t *start0, int64_t width, const uint8_t *text,
                        const int64_t *text_pos, int score_kind, const void *scores, char *out,
                        int64_t capacity, int64_t *written);
int rs_host_format_hits_combined(int64_t n_rows, int64_t match_id_first, const int64_t *rec,
                                 const char *id_blob, const int64_t *id_off, const char *desc_blob,
                                 const int64_t *desc_off, const char *sdesc_blob, const int64_t *sdesc_off,
                                 const char *motif_seq, const char *motif_struct, const int64_t *start0,
                                 int64_t width, const uint8_t *seq_text, const uint8_t *struct_text,
                                 const int64_t *text_pos, int seq_kind, const float *seq_scores,
                                 int struct_kind, const double *struct_scores, char *out, int64_t capacity,
                                 int64_t *written);

/* ---- background counts (replaces the Seq.count loop of rnascan.py:450-453) ---------
 * d_counts8[k] += number of symbols with index k and bit 3 clear (k = 0..7); exact
 * integers.  The caller zeroes d_counts8 first (so shards can accumulate).            */
int rs_hist(const uint8_t *d_codes, int64_t n, uint64_t *d_counts8, void *stream);
/* Same for NUCLEOTIDE streams only (codes 0-3, RS_RNA_OTHER, RS_SEP as rs_host_encode_rna
 * writes them): two index bit-planes instead of three, half the arithmetic; bins 4..7 stay 0.  */
int rs_hist_rna(const uint8_t *d_codes, int64_t n, uint64_t *d_counts8, void *stream);
/* Same for ALPHABET-layout streams (rs_host_encode_alpha): d_counts32[k] += symbols with index k and
 * bit 5 clear (k = 0..31; bin 31 counts the non-letters 0x1F, bins >= A stay 0 otherwise).      */
int rs_hist_alpha(const uint8_t *d_codes, int64_t n, uint64_t *d_counts32, void *stream);

/* ---- dense scores: the calculate() semantics, every window, NaN in band ------------
 * seq    : _pwm.c:34-68   out[i] = (float)(sum_j table[j][code]) double accumulation
 * struct : matrix.py:25-43 out[i] = sum_j table[j][code] in double
 * profile: rnascan.py:302-307 out[i] = sum_j nan_to_num(dot(profile[i+j,:], table[j,:]))
 * n_out = n - W + 1 values are written (nothing if n < W).                            */
int rs_scores_dense_seq(const uint8_t *d_codes, int64_t n, const double *table_Wx4, int W,
                        float *d_out, void *stream);
int rs_scores_dense_struct(const uint8_t *d_codes, int64_t n, const double *table_Wx7, int W,
                           double *d_out, void *stream);
/* Structure scores as rnascan PRINTS them: Python's round(score, 3) (rnascan.py:273) of the float64 score, as an
 * int32 number of thousandths -- 4 B per position instead of 8 for every-position output (-m -inf), the text
 * "k/1000" is exactly what repr(round(score, 3)) gives.  Special values: RS_MILLI_NAN (no score: the window
 * holds an invalid symbol or a separator), RS_MILLI_NINF (score -inf), RS_MILLI_NEG0 (rounds to -0.0),
 * RS_MILLI_RANGE (|score| >= 2e6 or +inf: use rs_scores_dense_struct).  W <= 16.                          */
#define RS_MILLI_NAN   (-2147483647 - 1)
#define RS_MILLI_NINF  (-2147483647)
#define RS_MILLI_NEG0  (-2147483646)
#define RS_MILLI_RANGE (-2147483645)
int rs_scores_dense_struct_milli(const uint8_t *d_codes, int64_t n, const double *table_Wx7, int W,
                                 int32_t *d_out, void *stream);
int rs_scores_dense_profile(const void *d_profile, int profile_dtype, int64_t n_rows,
                            const uint8_t *d_codes /* may be NULL: no separators */,
                            const double *table_Wx7, int W, double *d_out, void *stream);
/* alpha  : matrix.py:25-43 for any alphabet of A = 1..31 letters (rs_host_encode_alpha codes),
 *          table [W][A] in the caller's letter order; out[i] = sum_j table[j][code] in double.
 *          A <= 7 runs the structure kernels, 8..31 kernels with a 32-column table row.   */
int rs_scores_dense_alpha(const uint8_t *d_codes, int64_t n, const double *table_WxA, int W, int A,
                          double *d_out, void *stream);

/* ---- profile statistics, once per uploaded profile ---------------------------------
 * d_stats[0] = max over rows of sum_c |p[r][c]| ; d_stats[1] = number of non-finite
 * entries ; d_stats[2] = number of negative entries.  Feeds the guard band of
 * rs_scan_fused: pass profile_absrow_max = NaN there unless [1] == [2] == 0.          */
int rs_profile_stats(const void *d_profile, int profile_dtype, int64_t n_rows,
                     double *d_stats3, void *stream);

/* ---- thresholded scans: Biopython<=1.77 search(threshold, both=False) as driven by
 *      rnascan.py:263 -- strict `>`, NaN/-inf windows never reported -----------------
 * Hits come back sorted by position in the symbol stream.  d_counters[0] = number of
 * hits found (may exceed hit_capacity: then only the first hit_capacity are stored and
 * the caller re-runs with a larger buffer), d_counters[1] = windows re-scored exactly
 * (guard band + hits; diagnostic).
 *
 * rs_scan_seq           : float32 scores, bit-identical to _pwm.c for every hit.
 * rs_scan_struct_onehot : float64 scores as matrix.py:25-43.
 * rs_scan_pair_onehot   : both streams, hit iff both > m (two-FASTA RNASS mode).
 * rs_scan_fused         : sequence PSSM + averaged 7-channel profile in one pass.
 *                         The profile correlation runs in fp32 as a conservative filter;
 *                         every window within the guard band of the threshold is
 *                         re-scored in fp64 exactly as rnascan.py:302-307, so hit sets
 *                         and reported scores do not depend on the fp32 arithmetic.
 *                         d_hit_seq may be NULL in RS_MODE_STRUCT.                     */
int rs_scan_seq(const uint8_t *d_codes, int64_t n, const double *table_Wx4, int W,
                double threshold, int64_t hit_capacity, int64_t *d_hit_pos,
                float *d_hit_score, uint64_t *d_counters2, void *d_work, int64_t work_bytes,
                void *stream);
int rs_scan_struct_onehot(const uint8_t *d_codes, int64_t n, const double *table_Wx7, int W,
                          double threshold, int64_t hit_capacity, int64_t *d_hit_pos,
                          double *d_hit_score, uint64_t *d_counters2, void *d_work,
                          int64_t work_bytes, void *stream);
/* rs_scan_alpha         : rs_scan_struct_onehot for an alphabet-layout stream of A = 1..31 letters,
 *                         table [W][A] (as rs_scores_dense_alpha; replaces search() over
 *                         matrix.py:25-43, rnascan.py:263, for alphabets other than BEHLMRT).    */
int rs_scan_alpha(const uint8_t *d_codes, int64_t n, const double *table_WxA, int W, int A,
                  double threshold, int64_t hit_capacity, int64_t *d_hit_pos, double *d_hit_score,
                  uint64_t *d_counters2, void *d_work, int64_t work_bytes, void *stream);
int rs_scan_pair_onehot(const uint8_t *d_seq_codes, const uint8_t *d_struct_codes, int64_t n,
                        const double *seq_table_Wx4, const double *struct_table_Wx7, int W,
                        double threshold, int64_t hit_capacity, int64_t *d_hit_pos,
                        float *d_hit_seq, double *d_hit_struct, uint64_t *d_counters2,
                        void *d_work, int64_t work_bytes, void *stream);
int rs_scan_fused(const uint8_t *d_codes, const void *d_profile, int profile_dtype, int64_t n,
                  const double *seq_table_Wx4 /* NULL in RS_MODE_STRUCT */,
                  const double *struct_table_Wx7, int W, double threshold,
                  double profile_absrow_max, int mode, int64_t hit_capacity,
                  int64_t *d_hit_pos, float *d_hit_seq, double *d_hit_struct,
                  uint64_t *d_counters2, void *d_work, int64_t work_bytes, void *stream);

/* ---- one-hot threshold scans without waiting for the host's log-odds ---------------------
 * The exact log-odds need the host's libm (Python's math.log(p / b, 2), called by Biopython's
 * log_odds at rnascan.py:248) and the background counts (rnascan.py:445-457), i.e. a device ->
 * host -> device round trip between rs_hist and the scan.  These three calls take it off the
 * critical path; results are identical to rs_scan_seq / rs_scan_struct_onehot.
 *
 * rs_provisional_table : from DEVICE-resident counts (rs_hist output, all-reduced by the caller
 *     if sharded) and the motif's probabilities prob[W][alphabet] (device column order: A,C,G,U
 *     or B,E,H,L,M,R,T), writes d_table_margin[0 .. W*alphabet) = log2(p / b) with the device's
 *     log2 (within a few ulps of the host table) and d_table_margin[W*alphabet] = a bound on
 *     |exact - provisional| of any window score.
 *     A stand-alone utility (W <= 16): the scan below derives the same table itself.
 * rs_scan_onehot_begin : decision pass with the provisional table of (d_counts8, prob); a window
 *     is a CANDIDATE when its provisional score + margin + extra_margin exceeds the threshold (a
 *     superset of the exact hits; extra_margin >= 0 is extra slack, 0 in production).  W <= 16.
 * rs_scan_onehot_finish: with the exact host table: candidates come back in position order with
 *     their exact scores (float32 for alphabet 4, float64 for 7).  A candidate that is not a hit
 *     under the exact table has d_hit_pos = -1 (drop it); d_counters2[0] = entries written,
 *     d_counters2[1] = how many of them are -1 (0 unless a score lies within the margin of the
 *     threshold).  Same d_work / hit_capacity / stream as rs_scan_onehot_begin.
 * rs_scan_onehot_begin_notify : rs_scan_onehot_begin that also TELLS THE HOST the counts, without a
 *     copy, an event or a stream synchronisation: the first kernel it launches stores
 *     h_notify8[c] = (tag << 48) | d_counts8[c]  for c = 0..7 into page-locked host memory the device
 *     can address (cudaHostAlloc; the pointer is used as is, unified addressing).  tag = 1..65535, a
 *     new value per call; counts are below 2^48.  The host spins until all eight words show the tag
 *     (the stores are not ordered among themselves), builds its exact table while the scan runs and
 *     has rs_scan_onehot_finish queued before the scan ends.  d_clear8 (or NULL): eight device
 *     counters zeroed by the same kernel, e.g. the NEXT call's histogram target (must differ from
 *     d_counts8).  h_notify8 NULL: no notification (= rs_scan_onehot_begin).                        */
int rs_provisional_table(const uint64_t *d_counts8, const double *prob, int W, int alphabet,
                         double *d_table_margin /* W*alphabet + 1 doubles */, void *stream);
int rs_scan_onehot_begin(int alphabet, const uint8_t *d_codes, int64_t n,
                         const uint64_t *d_counts8, const double *prob, int W, double threshold,
                         double extra_margin, int64_t hit_capacity, void *d_work,
                         int64_t work_bytes, void *stream);
int rs_scan_onehot_begin_notify(int alphabet, const uint8_t *d_codes, int64_t n,
                                const uint64_t *d_counts8, const double *prob, int W,
                                double threshold, double extra_margin, int64_t hit_capacity,
                                void *d_work, int64_t work_bytes, uint64_t *h_notify8,
                                uint32_t tag, uint64_t *d_clear8, void *stream);
int rs_scan_onehot_finish(int alphabet, const uint8_t *d_codes, int64_t n, const double *table,
                          int W, double threshold, int64_t hit_capacity, int64_t *d_hit_pos,
                          void *d_hit_score, uint64_t *d_counters2, void *d_work,
                          int64_t work_bytes, void *stream);

/* ---- sequence half of the combined decision, applied to an ordered candidate list -------
 * combine() (rnascan.py:416-434) joins two result sets thresholded with the same -m, so a
 * combined hit = structure score > m AND sequence score > m.  Only the sequence side depends
 * on the data's background (rnascan.py:507-511; the averaged-profile mode cannot compute a
 * structure background, rnascan.py:533-540).  A caller can therefore run the structure-only
 * candidate scan (rs_scan_fused, RS_MODE_STRUCT) while rs_hist, the all-reduce of the counts
 * and the host log-odds are still in flight on another stream, and then call this:
 * the first min(*d_n_candidates, hit_capacity) entries of d_hit_pos (ascending) / d_hit_struct
 * (may be NULL) are the candidates; windows whose sequence score (_pwm.c:34-68 arithmetic,
 * float32) also exceeds `threshold` are kept IN PLACE, in order, with their scores in d_hit_seq;
 * d_counters2[0] = survivors.  d_n_candidates (device) must not alias d_counters2.  Results are
 * identical to rs_scan_fused in RS_MODE_AND with the same tables.                          */
int rs_refine_hits_seq(const uint8_t *d_codes, int64_t n, const double *seq_table_Wx4, int W,
                       double threshold, const uint64_t *d_n_candidates, int64_t hit_capacity,
                       int64_t *d_hit_pos, float *d_hit_seq, double *d_hit_struct,
                       uint64_t *d_counters2, void *d_work, int64_t work_bytes, void *stream);

/* The same decision split in two calls around the arrival of the background, cheaper than
 * rs_scan_fused(RS_MODE_STRUCT) + rs_refine_hits_seq because the candidates are never ordered on
 * their own: rs_scan_fused_candidates runs the structure-only scan and leaves its hits staged per
 * tile inside d_work (d_cand_counters2[0] = candidates found; above hit_capacity => re-run larger;
 * *staged_tiles, written on the host before returning, must be passed on);
 * rs_scan_fused_resolve applies the sequence PSSM to the staged candidates while ordering them.
 * Same d_work / hit_capacity / stream for both; d_counters2[0] = hits.  Results are identical to
 * rs_scan_fused(RS_MODE_AND).                                                               */
int rs_scan_fused_candidates(const uint8_t *d_codes, const void *d_profile, int profile_dtype,
                             int64_t n, const double *struct_table_Wx7, int W, double threshold,
                             double profile_absrow_max, int64_t hit_capacity,
                             uint64_t *d_cand_counters2, void *d_work, int64_t work_bytes,
                             int64_t *staged_tiles, void *stream);
/* rs_scan_fused_candidates that also takes the sequence's background counts in the same pass (the symbols are staged
 * for the scan anyway): d_counts8[0..3] += letters A,C,G,U (not zeroed here).  For streams so long that the
 * histogram's second read of the symbols costs more than waiting for the counts until the scan has finished;
 * needs the fp32 filter path (float32 rows, W <= 24, finite / -inf tables, finite threshold), n >= W.          */
int rs_scan_fused_candidates_counting(const uint8_t *d_codes, const void *d_profile, int profile_dtype,
                                      int64_t n, const double *struct_table_Wx7, int W, double threshold,
                                      double profile_absrow_max, int64_t hit_capacity,
                                      uint64_t *d_cand_counters2, uint64_t *d_counts8, void *d_work,
                                      int64_t work_bytes, int64_t *staged_tiles, void *stream);
int rs_scan_fused_resolve(const uint8_t *d_codes, int64_t n, const double *seq_table_Wx4, int W,
                          double threshold, int64_t staged_tiles, int64_t hit_capacity,
                          int64_t *d_hit_pos, float *d_hit_seq, double *d_hit_struct,
                          uint64_t *d_counters2, void *d_work, int64_t work_bytes, void *stream);

/* ---- filter + gather + resolve: averaged-profile scans whose EXACT rows stay in host memory ------
 * The reference scores the float64 rows pd.read_table gives it (rnascan.py:296-297, :302-307).  At
 * 56 B/row those rows are the whole end-to-end cost of a scan (PCIe), and the hit decision only needs
 * them for the few windows near the threshold.  So the device gets a FILTER FORM of the rows,
 *     RS_ROWS_F32         float32[n][7]  -- the rows themselves are float32 (exact rows == filter rows)
 *     RS_ROWS_F32_SHADOW  float32[n][7]  -- round-to-nearest shadow of float64 rows (guard band widened)
 *     RS_ROWS_Q8          uint8[n][8]    -- {q_B..q_T, symbol code}; p ~ q * q8_scale / 255, 0 <= p <= q8_scale
 *                                           (rs_host_quantize_q8); d_codes is ignored (may be NULL)
 *     RS_ROWS_Q4          uint32[n]      -- nibble c = floor(p_c * 15 / q8_scale) for the seven channels, top nibble
 *                                           = symbol code & 15 (rs_host_quantize_q4); 4 B per position; the
 *                                           guard band is wider (q8_scale / 15 * sum of the POSITIVE table
 *                                           entries), so it suits high thresholds on a slow link; d_codes ignored
 * rs_filter_profile returns, in position order, every window whose exact score COULD exceed the
 * threshold (and, when seq_table is given, whose sequence score does: _pwm.c:34-68 arithmetic) as
 * d_cand_pos[k] = pos_base + window start; d_counters2[0] = candidates found (above cand_capacity the
 * excess is dropped: re-run larger), [1] = windows that passed the fp32 filter.  d_cand_sym (RS_ROWS_Q4 only, may be
 * NULL) receives each candidate's W symbols, 2 bits each (symbol j in bits 2j, 2j+1; bit 63: one of them is not
 * A,C,G,U; W <= 24): rs_refine_candidates_packed then applies a sequence table that only became known later
 * (computed background) ON THE DEVICE -- survivors in order, d_counters2[0] = their number -- before anything is
 * gathered.  With RS_ROWS_Q8 / RS_ROWS_Q4 and
 * d_counts8 != NULL the letters A,C,G,U (codes 0..3) of rows [0, count_rows) are ADDED to
 * d_counts8[0..3] in the same pass (the background counts of rnascan.py:450-453; not zeroed here).
 * The host then gathers each candidate's W rows and W symbols (rs_host_gather_windows) and
 * rs_resolve_candidates decides and scores them exactly as rs_scan_fused does (same arithmetic, same
 * strict `>`; seq_table NULL = RS_MODE_STRUCT, else RS_MODE_AND): hits in order, d_counters2[0] = hits.
 * Results are identical to rs_scan_fused on the exact rows.  W <= 24; the tables must be finite or
 * -inf and the threshold finite (else RS_ERR_INVALID: use rs_scan_fused).                          */
#define RS_ROWS_F32        0
#define RS_ROWS_F32_SHADOW 1
#define RS_ROWS_Q8         2
#define RS_ROWS_Q4         3
int64_t rs_filter_workspace_bytes(int64_t n, int64_t cand_capacity);
int rs_filter_profile(const uint8_t *d_codes, const void *d_rows, int row_format, double q8_scale, int64_t n,
                      const double *seq_table_Wx4 /* NULL: no sequence check in this pass */,
                      const double *struct_table_Wx7, int W, double threshold, double absrow_max,
                      int64_t pos_base, int64_t count_rows, uint64_t *d_counts8 /* may be NULL */,
                      int64_t cand_capacity, int64_t *d_cand_pos, uint64_t *d_cand_sym /* may be NULL */,
                      uint64_t *d_counters2, void *d_work, int64_t work_bytes, void *stream);
int64_t rs_refine_packed_workspace_bytes(int64_t n_cand);
int rs_refine_candidates_packed(const int64_t *d_cand_pos, const uint64_t *d_cand_sym, int64_t n_cand,
                                const double *seq_table_Wx4, int W, double threshold, int64_t *d_out_pos,
                                uint64_t *d_counters2, void *d_work, int64_t work_bytes, void *stream);
int64_t rs_resolve_workspace_bytes(int64_t n_cand);
int rs_resolve_candidates(const int64_t *d_cand_pos, int64_t n_cand,
                          const void *d_win_rows /* [n_cand][W][7] */, int rows_dtype /* RS_F32 | RS_F64 */,
                          const uint8_t *d_win_codes /* [n_cand][W] */, const double *seq_table_Wx4,
                          const double *struct_table_Wx7, int W, double threshold, int64_t *d_hit_pos,
                          float *d_hit_seq, double *d_hit_struct, uint64_t *d_counters2, void *d_work,
                          int64_t work_bytes, void *stream);
/* Host helpers of the same protocol (host threads, no CUDA):
 * rs_host_rows_stats      out4 = {max_r sum_c |p|, #non-finite, #negative, max |p|} over float rows;
 * rs_host_rows_to_f32     float64 -> float32, round to nearest (the RS_ROWS_F32_SHADOW form);
 * rs_host_quantize_q8     the RS_ROWS_Q8 form: q = rint(p * 255 / scale), byte 7 = codes[r] (0 if NULL);
 *                         *n_out_of_range = entries outside [0, scale] or non-finite (then the form must
 *                         not be used);
 * rs_host_quantize_q4     the RS_ROWS_Q4 form: nibble c = floor(p_c * 15 / scale) (never above p), top nibble =
 *                         codes[r] & 15; *n_out_of_range as above;
 * rs_host_gather_windows  rows [pos[k], pos[k] + W) and their symbols (codes[(pos + j) * code_stride], so
 *                         byte 7 of 8-byte quantised rows serves with stride 8; code_stride = -4: `codes` points at
 *                         4-byte quantised rows, the symbols are their top nibbles; NULL = none) for every candidate;
 * rs_host_copy            memcpy on several threads (memory-mapped pack / pageable rows -> pinned staging).  */
int rs_host_rows_stats(const void *rows, int rows_dtype, int64_t n_rows, int threads, double *out4);
int rs_host_rows_to_f32(const double *rows, int64_t n_values, float *out, int threads);
int rs_host_copy(void *dst, const void *src, int64_t n_bytes, int threads);
int rs_host_quantize_q8(const void *rows, int rows_dtype, int64_t n_rows, const uint8_t *codes, double scale,
                        uint8_t *out_rows8, int threads, int64_t *n_out_of_range);
int rs_host_quantize_q4(const void *rows, int rows_dtype, int64_t n_rows, const uint8_t *codes, double scale,
                        uint32_t *out_rows4, int threads, int64_t *n_out_of_range);
int rs_host_gather_windows(const void *rows, int rows_dtype, int64_t n_rows, const uint8_t *codes,
                           int64_t code_stride, const int64_t *pos, int64_t n_cand, int W, void *out_rows,
                           uint8_t *out_codes, int threads);

/* ---- batched many-PFM scan (BASELINE config 5: 256 RNAcompete-style motif pairs) -------
 * The reference scans one PFM (pair) per process run; a motif collection means running
 * rnascan.py:490-576 once per motif.  Here all motifs are scanned over the SAME resident
 * streams in one call.  Motif m has width widths[m] <= table_stride_rows and tables
 * seq_tables[m][table_stride_rows][4] (NULL in RS_MODE_STRUCT) and
 * struct_tables[m][table_stride_rows][7] (rows >= widths[m] are ignored).
 * Hits come back grouped by motif (ascending), sorted by position inside a motif:
 * d_hit_motif[k], d_hit_pos[k], d_hit_seq[k], d_hit_struct[k].  After syncing the stream,
 * d_bases[m] .. d_bases[m+1] is motif m's slice, d_bases[n_motifs] the total (if it exceeds
 * hit_capacity the excess was dropped: re-run with a larger buffer); d_motif_counters2[2m]
 * = hits of motif m, [2m+1] = windows re-scored exactly for motif m.
 * Semantics per motif are exactly rs_scan_fused's.                                        */
int64_t rs_scan_batched_workspace_bytes(int64_t n, int n_motifs, int table_stride_rows,
                                        int64_t hit_capacity);
/* Per calling thread: 0 = choose (tensor cores from 32 motifs on, fp32 profiles, W <= 12), 1 = per-motif
 * CUDA-core loop, 2 = tensor cores or RS_ERR_INVALID.  Both paths return identical results.  The tensor-core
 * path synchronises the stream twice (the candidate count sizes the exact pass, the hit count the ordering):
 * the one entry point of this ABI that waits for the device.                                  */
int rs_set_batched_path(int path);
int rs_last_batched_path(void);          /* 1 or 2: the path the last rs_scan_batched call took */
int rs_scan_batched(const uint8_t *d_codes, const void *d_profile, int profile_dtype, int64_t n,
                    int n_motifs, const int *widths, const double *seq_tables,
                    const double *struct_tables, int table_stride_rows, double threshold,
                    double profile_absrow_max, int mode, int64_t hit_capacity, int32_t *d_hit_motif,
                    int64_t *d_hit_pos, float *d_hit_seq, double *d_hit_struct,
                    uint64_t *d_motif_counters2 /* [2*n_motifs] */, uint64_t *d_bases /* [n_motifs+1] */,
                    void *d_work, int64_t work_bytes, void *stream);

/* The same for float64 rows (what rnascan parses from structure.<id>.txt, rnascan.py:296-297) resident on the
 * device together with their float32 shadow (rs_host_rows_to_f32): the tensor-core filter reads the shadow
 * (guard band widened by its rounding), candidates are re-scored from the float64 rows.  Results are
 * identical to rs_scan_batched(d_exact_f64, RS_F64, ...).                                            */
int rs_scan_batched_shadow(const uint8_t *d_codes, const float *d_shadow_f32, const double *d_exact_f64,
                           int64_t n, int n_motifs, const int *widths, const double *seq_tables,
                           const double *struct_tables, int table_stride_rows, double threshold,
                           double profile_absrow_max, int mode, int64_t hit_capacity, int32_t *d_hit_motif,
                           int64_t *d_hit_pos, float *d_hit_seq, double *d_hit_struct,
                           uint64_t *d_motif_counters2, uint64_t *d_bases, void *d_work, int64_t work_bytes,
                           void *stream);

/* ---- many one-hot PSSMs over ONE symbol stream (a motif collection over a FASTA input) -----------
 * The reference scans one PFM per process run (rnascan.py:490-576); here M motifs are scanned over the
 * same resident stream in one call.  alphabet 4: RNA-layout codes, scores as rs_scan_seq (float32, into
 * d_hit_f32); alphabet 7: structure-layout codes, scores as rs_scan_struct_onehot (float64, d_hit_f64).
 * Motif m has width widths[m] (1..16, <= table_stride_rows <= 16) and table tables[m][table_stride_rows]
 * [alphabet] (rows >= widths[m] are ignored); the threshold must be finite.  n < 2^32.
 * Hits come back grouped by motif (ascending), sorted by position inside a motif: d_hit_motif[k],
 * d_hit_pos[k], score[k].  After syncing the stream, d_bases[m] .. d_bases[m+1] is motif m's slice and
 * d_bases[n_motifs] the total (if it exceeds hit_capacity nothing beyond the capacity was stored: re-run
 * with a larger buffer).  Per motif the hits and scores are exactly rs_scan_seq's / rs_scan_struct_onehot's.
 * Motifs are processed in groups of 256 (one k-mer decision table of 2 MB / 1 MB each).                  */
int64_t rs_scan_onehot_many_workspace_bytes(int alphabet, int64_t n, int n_motifs, int table_stride_rows);
int rs_scan_onehot_many(int alphabet, const uint8_t *d_codes, int64_t n, int n_motifs, const int *widths,
                        const double *tables, int table_stride_rows, double threshold, int64_t hit_capacity,
                        int32_t *d_hit_motif, int64_t *d_hit_pos, float *d_hit_f32, double *d_hit_f64,
                        uint64_t *d_bases, void *d_work, int64_t work_bytes, void *stream);
/* ---- many (sequence, structure) motif pairs over two aligned symbol streams ---------------------------
 * Replaces, for a collection of M pairs in the combined two-FASTA mode, the per-pair search() of both inputs
 * (rnascan.py:263, run once per motif on each input) and the combine() inner join (rnascan.py:416-434).
 * d_seq_codes (RNA layout) and d_struct_codes (structure layout) are n symbols each, separators at the same
 * places.  Pair m has one width widths[m] (1..16, <= table_stride_rows <= 16) for its sequence table
 * seq_tables[m][table_stride_rows][4] (ACGU) and its structure table struct_tables[m][table_stride_rows][7]
 * (BEHLMRT).  A window is a hit when its float32 sequence score > threshold AND its float64 structure
 * score > threshold; both scores are stored (d_hit_seq, d_hit_struct).  Everything else is
 * rs_scan_onehot_many's contract: finite threshold, n < 2^32, 16-byte aligned code pointers, hits grouped by
 * pair and in position order inside a pair, d_bases[M+1], re-run on overflow.  Per pair, positions and both
 * scores are exactly rs_scan_pair_onehot's with that pair's two tables.                                   */
int64_t rs_scan_pair_onehot_many_workspace_bytes(int64_t n, int n_motifs, int table_stride_rows);
int rs_scan_pair_onehot_many(const uint8_t *d_seq_codes, const uint8_t *d_struct_codes, int64_t n,
                             int n_motifs, const int *widths,
                             const double *seq_tables,    /* [M][stride][4], ACGU   */
                             const double *struct_tables, /* [M][stride][7], BEHLMRT */
                             int table_stride_rows, double threshold, int64_t hit_capacity,
                             int32_t *d_hit_motif, int64_t *d_hit_pos, float *d_hit_seq,
                             double *d_hit_struct, uint64_t *d_bases, void *d_work, int64_t work_bytes,
                             void *stream);

#ifdef __cplusplus
}
#endif
#endif /* RNASCAN_B200_H */
