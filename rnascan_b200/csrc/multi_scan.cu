// Many one-hot PSSMs over ONE symbol stream in one call (rs_scan_onehot_many): a motif collection scanned
// over a FASTA input, the RNA layout (A = 4, float32 scores as _pwm.c:34-68) or the structure layout
// (A = 7, float64 scores as matrix.py:25-43).  Per motif the result is exactly rs_scan_seq /
// rs_scan_struct_onehot's: same hits, same scores, position order.
// Pair mode (rs_scan_pair_onehot_many): M (sequence, structure) motif pairs over an RNA stream and a structure
// stream of the same layout; a hit needs both scores above the threshold, as rs_scan_pair_onehot per pair.
// Both streams get their own k-mer table and the two rows are ANDed before the transpose.
//
// Per group of up to 256 motifs:
//  1. kmer_mask_build_kernel (batched_tc.cu) tabulates, for every k-mer a window can start with (RNA: 8-mers of
//     2-bit codes, 65 536 rows; structure: 5-mers of 3-bit codes, 32 768 rows), which motifs can pass: the
//     decision itself for W <= k, a rigorous upper bound for wider motifs.  One row = ceil(M/32) words
//     (2 MB / 1 MB for 256 motifs: resident in L2).
//  2. multi_count: every warp owns a contiguous range of positions; 32 positions at a time it reads their
//     table words (restricted to the motifs no wider than the distance to the first invalid symbol or
//     separator), transposes the 32 x 32 bit block with shuffles so that lane l holds a 32-position bitmap of
//     one motif, re-scores the candidates of motifs wider than k exactly, and counts hits per (range, motif).
//  3. multi_offsets / multi_bases turn the counts into each (range, motif)'s first output slot.
//  4. multi_write repeats the traversal and writes every hit with its exact score to its slot.
// No atomics and no sort: the output is grouped by motif and in position order by construction.
#include "common.cuh"

#define MS_THREADS    256
#define MS_WARPS      (MS_THREADS / 32)
#define MS_GROUP      256                  // motifs per pass (8 table words per k-mer row)
#define MS_WORDS      (MS_GROUP / 32)
#define MS_WMAX       RS_KMER_WMAX         // widest motif
#define MS_MAX_RANGES 32768                // warp ranges per pass (bounds the count array: 32 MB per group)
#define MS_MIN_RANGE  1024                 // positions per warp range at least

static int64_t ms_rows(int A) { return A == 4 ? 65536 : 32768; }

static int64_t ms_range_len(int64_t n)
{
    int64_t len = rs_roundup((n + MS_MAX_RANGES - 1) / MS_MAX_RANGES, 32);
    return len < MS_MIN_RANGE ? MS_MIN_RANGE : len;
}
static int64_t ms_n_ranges(int64_t n) { return n > 0 ? (n + ms_range_len(n) - 1) / ms_range_len(n) : 0; }

struct MsLayout {
    int64_t off_tab, off_tab2, off_w, off_mask, off_mask2, off_cnt, off_tot, total;
};
// pair: A = 4 plus the structure stream's tables and k-mer table (regions of size 0 otherwise)
static MsLayout ms_layout(int A, bool pair, int64_t n, int n_motifs, int stride_rows)
{
    MsLayout l;
    int64_t off = 0;
    l.off_tab = off;   off += rs_roundup((int64_t)n_motifs * stride_rows * A * 8, 256);
    l.off_tab2 = off;  off += pair ? rs_roundup((int64_t)n_motifs * stride_rows * 7 * 8, 256) : 0;
    l.off_w = off;     off += rs_roundup((int64_t)n_motifs * 4, 256);
    l.off_mask = off;  off += ms_rows(A) * MS_WORDS * 4;
    l.off_mask2 = off; off += pair ? ms_rows(7) * MS_WORDS * 4 : 0;
    l.off_cnt = off;  off += rs_roundup(ms_n_ranges(n) * MS_GROUP * 4, 256);
    l.off_tot = off;  off += MS_GROUP * 8;
    l.total = off;
    return l;
}

struct MsParams {
    const uint8_t *codes;
    int64_t n, range_len, n_ranges;
    const uint32_t *mask;                // [rows][words]: bit (31 - k) of word c = motif 32 c + k of the group
    int words;
    const double *tables;                // the group's tables [gM][stride][A]
    const uint8_t *codes2;               // pair mode: the structure stream, its k-mer table and tables [gM][stride][7]
    const uint32_t *mask2;
    const double *tables2;
    const int *widths;                   // [gM]
    int stride, gM, motif0;
    double threshold;
    uint32_t *counts;                    // [n_ranges][MS_GROUP]: hits, then the exclusive offset inside the motif
    const unsigned long long *bases;     // d_bases (write pass)
    int64_t cap;
    int32_t *hit_motif;
    int64_t *hit_pos;
    float *hit_f32;
    double *hit_f64;
};

// lane r bit c -> lane c bit r (each step swaps one bit of the row index with the same bit of the column index)
__device__ __forceinline__ uint32_t ms_transpose32(uint32_t x, int lane)
{
    const uint32_t masks[5] = {0x0000FFFFu, 0x00FF00FFu, 0x0F0F0F0Fu, 0x33333333u, 0x55555555u};
#pragma unroll
    for (int s = 0; s < 5; s++) {
        const int j = 16 >> s;
        const uint32_t m = masks[s];
        const uint32_t y = __shfl_xor_sync(0xffffffffu, x, j);
        x = (lane & j) ? ((x & ~m) | ((y & ~m) >> j)) : ((x & m) | ((y & m) << j));
    }
    return x;
}

// The reference's decision for one window: sequential float64 adds (rs_exact_onehot_window); A = 4 casts to
// float32 once and compares widened (SURVEY.md N1), A = 7 compares the float64 sum.  NaN / -inf never pass.
template <int A>
__device__ __forceinline__ bool ms_exact(const uint8_t *codes, const double *tab, int W, double thr, double &score)
{
    double s;
    const bool ok = rs_exact_onehot_window<A, A>(codes, tab, W, s);
    if (A == 4) s = (double)(float)s;
    score = s;
    return ok && s > thr;
}

// The k-mer starting at pos (RNA: 8 symbols of 2 bits, structure: 5 of 3 bits) and f = the valid symbols from
// pos on (<= 16, up to the first invalid symbol, separator or the stream end).  pos < n.
template <int A>
__device__ __forceinline__ void ms_kmer(const uint8_t *codes, int64_t pos, int64_t n, uint32_t &kmer, int &f)
{
    const uint32_t *cw = reinterpret_cast<const uint32_t *>(codes + (pos & ~(int64_t)3));
    const unsigned sh = (unsigned)(pos & 3) * 8u;
    uint32_t raw[5], x[4];
#pragma unroll
    for (int i = 0; i < 5; i++) raw[i] = __ldg(cw + i);
#pragma unroll
    for (int i = 0; i < 4; i++) x[i] = __funnelshift_r(raw[i], raw[i + 1], sh);
    f = 16;
#pragma unroll
    for (int i = 3; i >= 0; i--) {                      // RNA: bits 2, 3 (other, separator); structure: index 7
        const uint32_t bad = A == 4 ? (x[i] & 0x0C0C0C0Cu) : (x[i] & (x[i] >> 1) & (x[i] >> 2) & 0x01010101u);
        if (bad) f = 4 * i + ((__ffs(bad) - 1) >> 3);
    }
    if (n - pos < f) f = (int)(n - pos);
    if (A == 4)                                         // symbol j in bits 2j, 2j+1
        kmer = (((x[0] & 0x03030303u) * 0x01041040u) >> 24) | ((((x[1] & 0x03030303u) * 0x01041040u) >> 24) << 8);
    else                                                // symbol j in bits 3j .. 3j+2
        kmer = (x[0] & 7u) | ((x[0] >> 5) & 0x38u) | ((x[0] >> 10) & 0x1C0u) | ((x[0] >> 15) & 0xE00u) |
               ((x[1] & 7u) << 12);
}

// PAIR (A = 4 only): p.codes is the RNA stream, p.codes2 the structure stream; a window is a hit when both
// motifs of the pair pass.  The table bits decide alone up to width KD, where both tables are exact.
template <int A, bool PAIR, bool WRITE>
__global__ void __launch_bounds__(MS_THREADS, 4) multi_scan_kernel(const MsParams p)
{
    static_assert(!PAIR || A == 4, "pair mode: RNA stream + structure stream");
    constexpr int K = A == 4 ? 8 : 5;
    constexpr int KD = PAIR ? 5 : K;
    __shared__ uint32_t s_cnt[MS_WARPS][MS_GROUP];          // count pass: hits; write pass: next slot in the motif
    __shared__ unsigned long long s_base[WRITE ? MS_GROUP : 1];
    __shared__ uint32_t s_wmask[MS_WMAX + 1][MS_WORDS];     // [f]: motifs no wider than f
    __shared__ int s_w[MS_GROUP];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int m = tid; m < MS_GROUP; m += MS_THREADS) {
        s_w[m] = m < p.gM ? p.widths[m] : 0;
        if (WRITE) s_base[m] = m < p.gM ? p.bases[p.motif0 + m] : 0ull;
    }
    __syncthreads();
    for (int e = tid; e < (MS_WMAX + 1) * MS_WORDS; e += MS_THREADS) {
        const int f = e / MS_WORDS, c = e % MS_WORDS;
        uint32_t bits = 0;
        for (int k = 0; k < 32; k++) {
            const int W = s_w[32 * c + k];
            if (W && W <= f) bits |= 1u << (31 - k);
        }
        s_wmask[f][c] = bits;
    }
    const int64_t range = (int64_t)blockIdx.x * MS_WARPS + warp;
    const bool live = range < p.n_ranges;
    for (int m = lane; m < MS_GROUP; m += 32)
        s_cnt[warp][m] = (WRITE && live) ? p.counts[range * MS_GROUP + m] : 0u;
    __syncthreads();
    if (!live) return;

    const int64_t r0 = range * p.range_len;
    const int64_t r1 = min(r0 + p.range_len, p.n);
    for (int64_t p0 = r0; p0 < r1; p0 += 32) {
        const int64_t pos = p0 + lane;
        uint32_t kmer = 0, kmer2 = 0;
        int f = 0;                                          // valid symbols from pos on, in both streams (<= 16)
        if (pos < r1) {
            ms_kmer<A>(p.codes, pos, p.n, kmer, f);
            if (PAIR) {
                int f2;
                ms_kmer<7>(p.codes2, pos, p.n, kmer2, f2);
                f = min(f, f2);
            }
        }
        for (int c = 0; c < p.words; c++) {
            uint32_t v = f ? (__ldg(p.mask + (size_t)kmer * p.words + c) & s_wmask[f][c]) : 0u;
            if (PAIR && v) v &= __ldg(p.mask2 + (size_t)kmer2 * p.words + c);
            if (!__any_sync(0xffffffffu, v)) continue;
            v = ms_transpose32(v, lane);                    // bit i: position p0 + i, motif 32 c + 31 - lane
            if (!v) continue;
            const int m = 32 * c + 31 - lane;
            const int W = s_w[m];
            const double *tab = p.tables + (size_t)m * p.stride * A;
            if (!WRITE && W <= KD) {                        // the table bits are the decision
                s_cnt[warp][m] += __popc(v);
                continue;
            }
            uint32_t slot = s_cnt[warp][m];
            for (uint32_t b = v; b; b &= b - 1) {
                const int64_t q = p0 + (__ffs(b) - 1);
                double s = 0.0, s2 = 0.0;                   // the write pass needs every score
                bool hit = true;
                if (WRITE || W > K) hit = ms_exact<A>(p.codes + q, tab, W, p.threshold, s) || W <= K;
                if (PAIR && (WRITE || W > 5))
                    hit = (ms_exact<7>(p.codes2 + q, p.tables2 + (size_t)m * p.stride * 7, W, p.threshold, s2) ||
                           W <= 5) && hit;
                if (!hit) continue;
                if (WRITE) {
                    const unsigned long long dst = s_base[m] + slot;
                    if ((int64_t)dst < p.cap) {
                        p.hit_motif[dst] = p.motif0 + m;
                        p.hit_pos[dst] = q;
                        if (A == 4) p.hit_f32[dst] = (float)s;
                        else        p.hit_f64[dst] = s;
                        if (PAIR)   p.hit_f64[dst] = s2;
                    }
                }
                slot++;
            }
            s_cnt[warp][m] = slot;
        }
    }
    if (!WRITE) {
        __syncwarp();
        for (int m = lane; m < MS_GROUP; m += 32) p.counts[range * MS_GROUP + m] = s_cnt[warp][m];
    }
}

// counts[r][m] -> exclusive prefix over r (per motif), tot[m] = motif m's hits.  Block b: motifs 32 b .. 32 b + 31,
// lane = motif, the 32 warps take contiguous slices of the ranges.
__global__ void __launch_bounds__(1024) multi_offsets_kernel(uint32_t *counts, int64_t n_ranges,
                                                             unsigned long long *tot)
{
    __shared__ unsigned long long s_part[32][33];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int m = blockIdx.x * 32 + lane;
    const int64_t per = (n_ranges + 31) / 32;
    const int64_t a = min((int64_t)warp * per, n_ranges), b = min(a + per, n_ranges);
    unsigned long long sum = 0;
    for (int64_t r = a; r < b; r++) sum += counts[r * MS_GROUP + m];
    s_part[warp][lane] = sum;
    __syncthreads();
    unsigned long long run = 0;
    for (int w = 0; w < warp; w++) run += s_part[w][lane];
    if (warp == 31) tot[m] = run + sum;
    for (int64_t r = a; r < b; r++) {
        const uint32_t v = counts[r * MS_GROUP + m];
        counts[r * MS_GROUP + m] = (uint32_t)run;
        run += v;
    }
}

// bases[motif0 + i] = bases[motif0] + hits of the group's motifs before i; bases[motif0 + gM] = the running total
__global__ void __launch_bounds__(MS_GROUP) multi_bases_kernel(unsigned long long *bases, const unsigned long long *tot,
                                                               int motif0, int gM)
{
    __shared__ unsigned long long s[MS_GROUP];
    const int i = threadIdx.x;
    const unsigned long long carry = bases[motif0];
    const unsigned long long v = i < gM ? tot[i] : 0ull;
    s[i] = v;
    __syncthreads();
    for (int d = 1; d < MS_GROUP; d <<= 1) {
        const unsigned long long t = i >= d ? s[i - d] : 0ull;
        __syncthreads();
        s[i] += t;
        __syncthreads();
    }
    if (i < gM) bases[motif0 + i] = carry + s[i] - v;
    if (i == MS_GROUP - 1) bases[motif0 + gM] = carry + s[i];
}

static bool ms_shape_ok(int A, int64_t n, int n_motifs, int stride_rows)
{
    if (A != 4 && A != 7) { rs_set_error("alphabet %d: 4 (RNA layout) or 7 (structure layout)", A); return false; }
    if (n < 0 || n >= ((int64_t)1 << 32)) { rs_set_error("stream length %lld outside [0, 2^32)", (long long)n); return false; }
    if (n_motifs < 1) { rs_set_error("no motifs"); return false; }
    if (stride_rows < 1 || stride_rows > MS_WMAX) {
        rs_set_error("table stride %d outside [1, %d]", stride_rows, MS_WMAX);
        return false;
    }
    return true;
}

extern "C" int64_t rs_scan_onehot_many_workspace_bytes(int alphabet, int64_t n, int n_motifs, int table_stride_rows)
{
    if (!ms_shape_ok(alphabet, n, n_motifs, table_stride_rows)) return -1;
    return ms_layout(alphabet, false, n, n_motifs, table_stride_rows).total;
}

extern "C" int64_t rs_scan_pair_onehot_many_workspace_bytes(int64_t n, int n_motifs, int table_stride_rows)
{
    if (!ms_shape_ok(4, n, n_motifs, table_stride_rows)) return -1;
    return ms_layout(4, true, n, n_motifs, table_stride_rows).total;
}

template <bool WRITE>
static void ms_launch(int A, bool pair, unsigned grid, cudaStream_t st, const MsParams &p)
{
    if (pair)        multi_scan_kernel<4, true, WRITE><<<grid, MS_THREADS, 0, st>>>(p);
    else if (A == 4) multi_scan_kernel<4, false, WRITE><<<grid, MS_THREADS, 0, st>>>(p);
    else             multi_scan_kernel<7, false, WRITE><<<grid, MS_THREADS, 0, st>>>(p);
}

// Both entry points.  pair: A = 4, codes2 / tables2 the structure stream and tables, scores into d_hit_f32
// (sequence) and d_hit_f64 (structure).
static int ms_scan(int A, bool pair, const uint8_t *d_codes, const uint8_t *d_codes2, int64_t n, int n_motifs,
                   const int *widths, const double *tables, const double *tables2, int table_stride_rows,
                   double threshold, int64_t hit_capacity, int32_t *d_hit_motif, int64_t *d_hit_pos,
                   float *d_hit_f32, double *d_hit_f64, uint64_t *d_bases, void *d_work, int64_t work_bytes,
                   cudaStream_t st)
{
    if (!ms_shape_ok(A, n, n_motifs, table_stride_rows)) return RS_ERR_INVALID;
    if (!widths || !tables || (pair && !tables2) || !d_bases) {
        rs_set_error("null widths, tables or bases"); return RS_ERR_INVALID;
    }
    for (int m = 0; m < n_motifs; m++)
        if (widths[m] < 1 || widths[m] > table_stride_rows) {
            rs_set_error("motif %d: width %d outside [1, %d] (widths above %d are not supported)", m, widths[m],
                         table_stride_rows, MS_WMAX);
            return RS_ERR_INVALID;
        }
    if (!isfinite(threshold)) { rs_set_error("threshold must be finite"); return RS_ERR_INVALID; }
    if (n > 0 && (!d_codes || ((uintptr_t)d_codes & 15) || (pair && (!d_codes2 || ((uintptr_t)d_codes2 & 15))))) {
        rs_set_error("codes pointer must be non-null and 16-byte aligned"); return RS_ERR_INVALID;
    }
    const bool f32 = A == 4, f64 = A == 7 || pair;
    if (hit_capacity < 0 ||
        (hit_capacity > 0 && (!d_hit_motif || !d_hit_pos || (f32 && !d_hit_f32) || (f64 && !d_hit_f64)))) {
        rs_set_error("bad hit buffers"); return RS_ERR_INVALID;
    }
    const MsLayout l = ms_layout(A, pair, n, n_motifs, table_stride_rows);
    if (!d_work || work_bytes < l.total) {
        rs_set_error("workspace too small: need %lld bytes", (long long)l.total); return RS_ERR_WORKSPACE;
    }
    RS_CUDA(cudaMemsetAsync(d_bases, 0, sizeof(uint64_t) * ((size_t)n_motifs + 1), st));
    if (n == 0) return RS_OK;
    uint8_t *wk = (uint8_t *)d_work;
    double *d_tab = (double *)(wk + l.off_tab);
    double *d_tab2 = (double *)(wk + l.off_tab2);
    int *d_w = (int *)(wk + l.off_w);
    uint32_t *d_mask = (uint32_t *)(wk + l.off_mask);
    uint32_t *d_mask2 = (uint32_t *)(wk + l.off_mask2);
    uint32_t *d_cnt = (uint32_t *)(wk + l.off_cnt);
    unsigned long long *d_tot = (unsigned long long *)(wk + l.off_tot);
    // (pageable sources: cudaMemcpyAsync returns once they are staged)
    RS_CUDA(cudaMemcpyAsync(d_tab, tables, (size_t)n_motifs * table_stride_rows * A * 8, cudaMemcpyHostToDevice, st));
    if (pair)
        RS_CUDA(cudaMemcpyAsync(d_tab2, tables2, (size_t)n_motifs * table_stride_rows * 7 * 8, cudaMemcpyHostToDevice,
                                st));
    RS_CUDA(cudaMemcpyAsync(d_w, widths, (size_t)n_motifs * 4, cudaMemcpyHostToDevice, st));

    MsParams p = {};
    p.codes = d_codes; p.n = n; p.range_len = ms_range_len(n); p.n_ranges = ms_n_ranges(n);
    p.mask = d_mask; p.stride = table_stride_rows; p.threshold = threshold; p.counts = d_cnt;
    p.codes2 = pair ? d_codes2 : nullptr; p.mask2 = pair ? d_mask2 : nullptr;
    p.bases = (const unsigned long long *)d_bases; p.cap = hit_capacity;
    p.hit_motif = d_hit_motif; p.hit_pos = d_hit_pos; p.hit_f32 = d_hit_f32; p.hit_f64 = d_hit_f64;
    const unsigned grid = (unsigned)((p.n_ranges + MS_WARPS - 1) / MS_WARPS);
    rs_prof_start(st);
    for (int g0 = 0; g0 < n_motifs; g0 += MS_GROUP) {
        const int gM = n_motifs - g0 < MS_GROUP ? n_motifs - g0 : MS_GROUP;
        p.words = (gM + 31) / 32; p.gM = gM; p.motif0 = g0;
        p.tables = d_tab + (size_t)g0 * table_stride_rows * A; p.widths = d_w + g0;
        int rc = rs_kmer_mask_build(A, d_mask, p.words, p.tables, p.widths, gM, table_stride_rows, threshold, st);
        if (rc) return rc;
        if (pair) {
            p.tables2 = d_tab2 + (size_t)g0 * table_stride_rows * 7;
            rc = rs_kmer_mask_build(7, d_mask2, p.words, p.tables2, p.widths, gM, table_stride_rows, threshold, st);
            if (rc) return rc;
        }
        ms_launch<false>(A, pair, grid, st, p);
        RS_CUDA(cudaGetLastError());
        multi_offsets_kernel<<<(unsigned)p.words, 1024, 0, st>>>(d_cnt, p.n_ranges, d_tot);
        multi_bases_kernel<<<1, MS_GROUP, 0, st>>>((unsigned long long *)d_bases, d_tot, g0, gM);
        RS_CUDA(cudaGetLastError());
        ms_launch<true>(A, pair, grid, st, p);
        RS_CUDA(cudaGetLastError());
    }
    rs_prof_stop(st);
    return RS_OK;
}

extern "C" int rs_scan_onehot_many(int alphabet, const uint8_t *d_codes, int64_t n, int n_motifs, const int *widths,
                                   const double *tables, int table_stride_rows, double threshold, int64_t hit_capacity,
                                   int32_t *d_hit_motif, int64_t *d_hit_pos, float *d_hit_f32, double *d_hit_f64,
                                   uint64_t *d_bases, void *d_work, int64_t work_bytes, void *stream)
{
    return ms_scan(alphabet, false, d_codes, nullptr, n, n_motifs, widths, tables, nullptr, table_stride_rows,
                   threshold, hit_capacity, d_hit_motif, d_hit_pos, d_hit_f32, d_hit_f64, d_bases, d_work, work_bytes,
                   (cudaStream_t)stream);
}

extern "C" int rs_scan_pair_onehot_many(const uint8_t *d_seq_codes, const uint8_t *d_struct_codes, int64_t n,
                                        int n_motifs, const int *widths, const double *seq_tables,
                                        const double *struct_tables, int table_stride_rows, double threshold,
                                        int64_t hit_capacity, int32_t *d_hit_motif, int64_t *d_hit_pos,
                                        float *d_hit_seq, double *d_hit_struct, uint64_t *d_bases, void *d_work,
                                        int64_t work_bytes, void *stream)
{
    return ms_scan(4, true, d_seq_codes, d_struct_codes, n, n_motifs, widths, seq_tables, struct_tables,
                   table_stride_rows, threshold, hit_capacity, d_hit_motif, d_hit_pos, d_hit_seq, d_hit_struct,
                   d_bases, d_work, work_bytes, (cudaStream_t)stream);
}
