// One-hot PSSM scans over symbol codes: sequence (A=4, float32 scores), structure
// context (A=7, float64 scores) and any other alphabet of up to 31 letters (float64
// scores), dense or thresholded, single stream or a pair of streams (two-FASTA RNASS mode).
//
// Replaces   _pwm.c:34-68 (driven per window by Biopython search(), rnascan.py:263)
//            BioAddons/motifs/matrix.py:25-43 (_py_calculate)
//
// Arithmetic: sequential double adds of table[j][code] in j order, then one cast to float
// for the sequence alphabet -- the reference's exact operation order, so results are
// bit-identical.  Persistent CTAs stream tiles of symbol codes into a shared-memory ring
// with 1-D bulk async copies; the W x 8 double table is staged in shared memory; lanes of
// a warp take consecutive windows (conflict-free byte gathers, coalesced dense stores).
// Hits are found with a first pass that only keeps a bit per window, ordered with warp
// ballot/popc + a block prefix sum + ONE atomic per tile, and re-scored when written.
#include "common.cuh"

#define OH_THREADS 256
#define OH_PER     16
#define OH_TILE    (OH_THREADS * OH_PER)     // 4096 windows per tile
#define OH_STAGES  3
#define OH_TS      8                         // table row stride in doubles (RNA and structure layouts)
#define OH_TS_ALPHA 32                       // table row stride of the alphabet layout (8..31 letters)

// TS = 32 carries no PAIR table: 64 x 32 doubles are already 16 KB of the 32 764 B of kernel parameters.
template <int TS>
struct OneHotParamsT {
    const uint8_t *codes_a;      // sequence codes (A=4), structure codes (A=7) or alphabet codes
    const uint8_t *codes_b;      // PAIR: structure codes
    void          *dense_out;    // float* (A=4) or double* (otherwise)
    int64_t        n, padded, n_tiles;
    double         threshold;
    int            W;
    int            n_letters;    // TS = 32: letters of the alphabet (valid indices 0 .. n_letters-1)
    HitStage       st;
    double         ta[RS_MAX_W * TS];        // table for stream a, row stride TS
    double         tb[TS == OH_TS ? RS_MAX_W * OH_TS : 1];   // table for stream b (PAIR)
};
typedef OneHotParamsT<OH_TS> OneHotParams;

__host__ __device__ constexpr uint32_t oh_ru16(uint32_t x) { return (x + 15u) & ~15u; }

// DENSE: every window, else hits.  A: alphabet of stream a (0: the alphabet layout, prm.n_letters letters).
// PAIR: second stream (A_b = 7), hits only.  TS: table row stride of stream a (OH_TS or OH_TS_ALPHA).
template <int A, bool PAIR, bool DENSE, int TS = OH_TS>
__global__ void __launch_bounds__(OH_THREADS) onehot_kernel(const __grid_constant__ OneHotParamsT<TS> prm)
{
    constexpr uint32_t CODE_BYTES = oh_ru16(OH_TILE + RS_MAX_W - 1);
    constexpr uint32_t STAGE_BYTES = CODE_BYTES * (PAIR ? 2 : 1);
    __shared__ __align__(128) uint8_t s_stage[OH_STAGES * STAGE_BYTES];
    __shared__ __align__(16) double s_ta[RS_MAX_W * TS];
    __shared__ __align__(16) double s_tb[PAIR ? RS_MAX_W * OH_TS : 1];
    __shared__ uint64_t bars[OH_STAGES];
    __shared__ unsigned s_cnt[OH_THREADS / 32][OH_PER];
    __shared__ unsigned long long s_base;

    const int W = prm.W;
    const int n_letters = A ? A : prm.n_letters;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int k = tid; k < W * TS; k += OH_THREADS) {
        s_ta[k] = prm.ta[k];
        if (PAIR) s_tb[k] = prm.tb[k];
    }
    if (tid == 0) {
        for (int s = 0; s < OH_STAGES; s++) mbar_init(&bars[s], 1);
        fence_mbar_init();
    }
    __syncthreads();

    const int64_t stride = gridDim.x, first = blockIdx.x;
    const int64_t my_tiles = first < prm.n_tiles ? (prm.n_tiles - first + stride - 1) / stride : 0;
    const uint32_t need = oh_ru16(OH_TILE + W - 1);

    auto issue = [&](int64_t it) {
        const int s = (int)(it % OH_STAGES);
        const int64_t t0 = (first + it * stride) * OH_TILE;
        const uint32_t bytes = (uint32_t)min((int64_t)need, prm.padded - t0);
        uint8_t *dst = s_stage + (size_t)s * STAGE_BYTES;
        mbar_expect_tx(&bars[s], bytes * (PAIR ? 2 : 1));
        bulk_g2s(dst, prm.codes_a + t0, bytes, &bars[s]);
        if (PAIR) bulk_g2s(dst + CODE_BYTES, prm.codes_b + t0, bytes, &bars[s]);
    };
    if (tid == 0)
        for (int64_t it = 0; it < OH_STAGES - 1 && it < my_tiles; it++) issue(it);

    // score of window w of the staged tile; returns hit decision, fills scores
    auto score = [&](const uint8_t *ca, const uint8_t *cb, int w, int64_t gpos, float &fa, double &da,
                     double &db) -> bool {
        if (gpos + W > prm.n) return false;
        double sa;
        bool ok = rs_exact_onehot_window<A, TS>(ca + w, s_ta, W, sa, n_letters);
        if (A == 4) { fa = (float)sa; da = (double)fa; }      // _pwm.c:65 ; compare widened (note N1)
        else        { fa = 0.f; da = sa; }
        if (!ok || !(da > prm.threshold)) return false;
        if (PAIR) {
            double sb;
            if (!rs_exact_onehot_window<7, OH_TS>(cb + w, s_tb, W, sb)) return false;
            db = sb;
            return sb > prm.threshold;
        }
        return true;
    };

    for (int64_t it = 0; it < my_tiles; it++) {
        const int s = (int)(it % OH_STAGES);
        if (tid == 0 && it + OH_STAGES - 1 < my_tiles) issue(it + OH_STAGES - 1);
        mbar_wait(&bars[s], (uint32_t)((it / OH_STAGES) & 1));
        const int64_t tile = first + it * stride;
        const int64_t t0 = tile * OH_TILE;
        const uint8_t *ca = s_stage + (size_t)s * STAGE_BYTES;
        const uint8_t *cb = PAIR ? ca + CODE_BYTES : nullptr;

        if (DENSE) {
#pragma unroll 4
            for (int k = 0; k < OH_PER; k++) {
                const int w = warp * (32 * OH_PER) + k * 32 + lane;
                const int64_t gpos = t0 + w;
                if (gpos + W <= prm.n) {
                    double sa;
                    bool ok = rs_exact_onehot_window<A, TS>(ca + w, s_ta, W, sa, n_letters);
                    if (A == 4) reinterpret_cast<float *>(prm.dense_out)[gpos] = ok ? (float)sa : nanf("");
                    else        reinterpret_cast<double *>(prm.dense_out)[gpos] = ok ? sa : nan("");
                }
            }
            __syncthreads();
            continue;
        }

        unsigned hitmask = 0;
#pragma unroll 4
        for (int k = 0; k < OH_PER; k++) {
            const int w = warp * (32 * OH_PER) + k * 32 + lane;
            float fa; double da, db;
            if (score(ca, cb, w, t0 + w, fa, da, db)) hitmask |= 1u << k;
        }
        const int any = __syncthreads_or(hitmask != 0);
        if (any) {
            for (int k = 0; k < OH_PER; k++) {
                unsigned b = __ballot_sync(0xffffffffu, (hitmask >> k) & 1u);
                if (lane == 0) s_cnt[warp][k] = __popc(b);
            }
            __syncthreads();
            unsigned before = 0, total = 0;
            for (int ww = 0; ww < OH_THREADS / 32; ww++)
#pragma unroll
                for (int k = 0; k < OH_PER; k++) {
                    unsigned v = s_cnt[ww][k];
                    if (ww < warp) before += v;
                    total += v;
                }
            if (tid == 0) {
                unsigned long long base = atomicAdd(prm.st.counters, (unsigned long long)total);
                s_base = base;
                prm.st.tile_seg[tile] = make_ulonglong2(base, (unsigned long long)total);
            }
            __syncthreads();
            unsigned long long kk = s_base + before;
            for (int k = 0; k < OH_PER; k++) {
                unsigned b = __ballot_sync(0xffffffffu, (hitmask >> k) & 1u);
                if ((hitmask >> k) & 1u) {
                    unsigned long long dst = kk + __popc(b & ((1u << lane) - 1u));
                    if ((int64_t)dst < prm.st.capacity) {
                        const int w = warp * (32 * OH_PER) + k * 32 + lane;
                        float fa; double da, db = 0.0;
                        score(ca, cb, w, t0 + w, fa, da, db);
                        prm.st.pos[dst] = t0 + w;
                        if (A == 4) prm.st.seq[dst] = fa;
                        else        prm.st.str[dst] = da;
                        if (PAIR)   prm.st.str[dst] = db;
                    }
                }
                kk += __popc(b);
            }
            __syncthreads();
        } else if (tid == 0) {
            prm.st.tile_seg[tile] = make_ulonglong2(0ull, 0ull);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Dense scores for W <= 16 with the motif width known at compile time (the generic kernel above
// spends ~20 instructions per symbol on loop control and 64-bit addressing).  Lanes take
// consecutive windows (coalesced stores); a window's bytes are fetched as aligned words (four
// lanes share a word: broadcast, no bank conflict) and aligned with funnel shifts; each symbol
// costs shift + mask (giving the byte offset of its table entry directly), one LDS.64 and one
// fp64 add -- still the reference's sequential j-order sum (_pwm.c:36-60, matrix.py:34-38).
#define DW_THREADS 256
#define DW_PER     16
#define DW_TILE    (DW_THREADS * DW_PER)
#define DW_STAGES  3
#define DW_STAGE_BYTES (DW_TILE + 32)

// Python's round(x, 3) of a float as an integer number of thousandths (rnascan.py:273 rounds every reported
// structure score): the correctly rounded decimal, ties to even only when x * 1000 is EXACTLY half way.
// x * 1000 = p + e exactly (e from one FMA); rint(p) is already right unless p sits exactly on a half, where
// the sign of e decides.  Sentinels: RS_MILLI_NAN (no score: invalid symbol / separator), RS_MILLI_NINF
// (-inf: a zero-probability letter), RS_MILLI_NEG0 (rounds to -0.0, which prints as "-0.0"),
// RS_MILLI_RANGE (|x| >= 2e6 or +inf: the caller takes the float64 path).
__device__ __noinline__ int32_t rs_round3_milli_exact(double x)
{
    if (x != x) return RS_MILLI_NAN;
    if (x == -INFINITY) return RS_MILLI_NINF;
    if (!(fabs(x) < 2.0e6)) return RS_MILLI_RANGE;
    const double p = __dmul_rn(x, 1000.0);
    const double e = __fma_rn(x, 1000.0, -p);
    double r = rint(p);
    const double d = __dsub_rn(p, r);
    if (d == 0.5 && e > 0.0) r += 1.0;
    else if (d == -0.5 && e < 0.0) r -= 1.0;
    if (r == 0.0 && (x < 0.0 || (x == 0.0 && signbit(x)))) return RS_MILLI_NEG0;
    return (int32_t)r;
}
// The common case is decided in float32: pf = float(x) * 1000 is within |pf| * 2^-22 of x * 1000; unless its
// fractional part lies that close to a half, the nearest integer of pf is the nearest integer of x * 1000 and no
// tie is in sight.  Everything else (near-ties: ~1 % of windows, |x| >= 4194, NaN, infinities) takes the exact
// path above.  (Measured at W = 7, 125 M windows: float64 output 0.279 ms; this 0.365 ms; the exact path for
// every window 0.390 ms; a conversion built from integer operations on the double's bits 0.418 ms.)
__device__ __forceinline__ int32_t rs_round3_milli(double x)
{
    const float pf = (float)x * 1000.f;
    const float apf = fabsf(pf);
    if (apf < 4194304.f) {                                       // (false for NaN / inf)
        const float r = rintf(pf);
        const float g = fabsf(pf - r);                           // exact
        if (0.5f - g > apf * 2.3841858e-7f + 1e-30f) {           // safely away from a half
            const int k = (int)r;
            if (k == 0 && (__double2hiint(x) < 0)) return RS_MILLI_NEG0;
            return k;
        }
    }
    return rs_round3_milli_exact(x);
}

// OUT: 0 = the calculate() types (float32 for A = 4, float64 for A = 7), 1 = int32 thousandths (A = 7).
// (Tried and dropped: a 7^4-entry table of the exact prefix ((t0 + t1) + t2) + t3, one LDS.64 instead of four --
// its random 8-byte reads collide on the banks about as often as they save wavefronts: 0.285 vs 0.282 ms at W = 7.)
// What bounds it (round 2): the load/store unit.  Per 32 windows the kernel needs W LDS.64 of table entries (2
// wavefronts each: 256 bytes into the registers at 128 B per clock), ~3 wavefronts of window symbols and 2 line
// accesses for the store: 19 LSU cycles at W = 7, i.e. 0.263 ms for 125 M windows at 1.9 GHz; measured 0.284-0.289.
// Eight consecutive windows per thread (each symbol's table offset and validity formed once, 37 instead of 58
// instructions per window, 16-byte stores) was built and measured: bit-identical, but 0.346 ms -- a lane's 64
// contiguous output bytes make every store instruction touch 16 lines instead of 2, and the table lookups, which
// are the bulk of the LSU time, are not reduced by it.
// TS = OH_TS_ALPHA (A = 0): the alphabet layout, index = code & 31, valid below prm.n_letters.
template <int A, int W, int OUT, int TS = OH_TS>
__global__ void __launch_bounds__(DW_THREADS) dense_w_kernel(const __grid_constant__ OneHotParamsT<TS> prm)
{
    constexpr int NW = (W + 3) / 4;                       // words holding one window's symbols
    constexpr uint32_t OFF_MASK = (TS - 1) << 3;          // byte offset of the entry within its table row
    __shared__ __align__(128) uint8_t s_stage[DW_STAGES * DW_STAGE_BYTES];
    __shared__ __align__(16) double s_ta[W * TS];
    __shared__ uint64_t bars[DW_STAGES];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t letters4 = (uint32_t)prm.n_letters * 0x01010101u;
    for (int k = tid; k < W * TS; k += DW_THREADS) s_ta[k] = prm.ta[k];
    if (tid == 0) {
        for (int s = 0; s < DW_STAGES; s++) mbar_init(&bars[s], 1);
        fence_mbar_init();
    }
    __syncthreads();
    const int64_t stride = gridDim.x, first = blockIdx.x;
    const int64_t my_tiles = first < prm.n_tiles ? (prm.n_tiles - first + stride - 1) / stride : 0;
    auto issue = [&](int64_t it) {
        const int s = (int)(it % DW_STAGES);
        const int64_t t0 = (first + it * stride) * DW_TILE;
        const uint32_t bytes = (uint32_t)min((int64_t)DW_STAGE_BYTES, prm.padded - t0);
        mbar_expect_tx(&bars[s], bytes);
        bulk_g2s(s_stage + (size_t)s * DW_STAGE_BYTES, prm.codes_a + t0, bytes, &bars[s]);
    };
    if (tid == 0)
        for (int64_t it = 0; it < DW_STAGES - 1 && it < my_tiles; it++) issue(it);
    const uint32_t tab = smem_u32(s_ta);

    for (int64_t it = 0; it < my_tiles; it++) {
        const int s = (int)(it % DW_STAGES);
        if (tid == 0 && it + DW_STAGES - 1 < my_tiles) issue(it + DW_STAGES - 1);
        mbar_wait(&bars[s], (uint32_t)((it / DW_STAGES) & 1));
        const int64_t t0 = (first + it * stride) * DW_TILE;
        const uint32_t *words = reinterpret_cast<const uint32_t *>(s_stage + (size_t)s * DW_STAGE_BYTES);
#pragma unroll 4
        for (int k = 0; k < DW_PER; k++) {
            const int w = warp * (32 * DW_PER) + k * 32 + lane;
            const uint32_t *q = words + (w >> 2);
            const unsigned sh = (unsigned)(w & 3) * 8u;
            uint32_t x[NW];
            uint32_t prev = q[0];
#pragma unroll
            for (int i = 0; i < NW; i++) {
                const uint32_t nxt = q[i + 1];
                x[i] = __funnelshift_r(prev, nxt, sh);
                prev = nxt;
            }
            // validity: A = 4 -> any of bits 2,3 set; A = 7 -> (code & 7) == 7; TS = 32 -> (code & 31) >= n_letters
            uint32_t bad = 0;
#pragma unroll
            for (int i = 0; i < NW; i++) {
                const uint32_t m = (i == NW - 1 && (W & 3)) ? (0xFFFFFFFFu >> (32 - 8 * (W & 3))) : 0xFFFFFFFFu;
                if (TS == OH_TS_ALPHA) bad |= __vcmpgeu4(x[i] & 0x1F1F1F1Fu, letters4) & m;
                else if (A == 4)       bad |= x[i] & (0x0C0C0C0Cu & m);
                else                   bad |= x[i] & (x[i] >> 1) & (x[i] >> 2) & (0x01010101u & m);
            }
            double sum = 0.0;
#pragma unroll
            for (int j = 0; j < W; j++) {
                const int sb = 8 * (j & 3);
                const uint32_t off = sb >= 3 ? ((x[j >> 2] >> (sb - 3)) & OFF_MASK) : ((x[j >> 2] << 3) & OFF_MASK);
                double t;
                asm("ld.shared.f64 %0, [%1];" : "=d"(t) : "r"(tab + (uint32_t)(j * TS * 8) + off));
                sum = __dadd_rn(sum, t);
            }
            const int64_t gpos = t0 + w;
            if (gpos + W <= prm.n) {
                if (OUT == 1)    reinterpret_cast<int32_t *>(prm.dense_out)[gpos] = bad ? RS_MILLI_NAN : rs_round3_milli(sum);
                else if (A == 4) reinterpret_cast<float *>(prm.dense_out)[gpos] = bad ? nanf("") : (float)sum;
                else             reinterpret_cast<double *>(prm.dense_out)[gpos] = bad ? nan("") : sum;
            }
        }
        __syncthreads();
    }
}

template <int A, int W, int OUT, int TS>
static int launch_dense_w(OneHotParamsT<TS> &prm, cudaStream_t stream)
{
    prm.n_tiles = (prm.n + DW_TILE - 1) / DW_TILE;
    int64_t grid = (int64_t)rs_sm_count() * 6;
    if (grid > prm.n_tiles) grid = prm.n_tiles;
    rs_prof_start(stream);
    dense_w_kernel<A, W, OUT, TS><<<(unsigned)grid, DW_THREADS, 0, stream>>>(prm);
    rs_prof_stop(stream);
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

template <int A, int OUT, int TS>
static int dispatch_dense_w(int W, OneHotParamsT<TS> &prm, cudaStream_t stream)
{
    switch (W) {
#define DW_CASE(w) case w: return launch_dense_w<A, w, OUT, TS>(prm, stream);
        DW_CASE(1) DW_CASE(2) DW_CASE(3) DW_CASE(4) DW_CASE(5) DW_CASE(6) DW_CASE(7) DW_CASE(8)
        DW_CASE(9) DW_CASE(10) DW_CASE(11) DW_CASE(12) DW_CASE(13) DW_CASE(14) DW_CASE(15) DW_CASE(16)
#undef DW_CASE
    default: return -1;
    }
}

// ------------------------------------------------------------------------------------------------
template <int TS = OH_TS>
static void fill_table(double *dst, const double *src, int W, int A)
{
    for (int j = 0; j < W; j++)
        for (int c = 0; c < TS; c++) dst[j * TS + c] = c < A ? src[j * A + c] : 0.0;
}

static int check_args(const uint8_t *codes, int64_t n, const double *table, int W)
{
    if (!codes || !table) { rs_set_error("null codes or table"); return RS_ERR_INVALID; }
    if ((uintptr_t)codes & 15) { rs_set_error("codes pointer must be 16-byte aligned"); return RS_ERR_INVALID; }
    if (W < 1 || W > RS_MAX_W) { rs_set_error("motif width %d outside [1, %d]", W, RS_MAX_W); return RS_ERR_INVALID; }
    if (n < 0) { rs_set_error("negative length"); return RS_ERR_INVALID; }
    return RS_OK;
}

template <int A, bool PAIR, bool DENSE, int TS = OH_TS>
static int launch(const OneHotParamsT<TS> &prm, cudaStream_t stream)
{
    int per_sm = 2048 / OH_THREADS;
    if (TS != OH_TS) {                  // the wider table leaves room for fewer CTAs: one resident wave, no tail
        static int occ[RS_MAX_DEVICES] = {};
        const int dev = rs_current_device();
        if (!occ[dev]) {
            int v = 0;
            RS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, onehot_kernel<A, PAIR, DENSE, TS>, OH_THREADS, 0));
            occ[dev] = v > 0 ? v : 1;
        }
        per_sm = occ[dev];
    }
    int64_t grid = (int64_t)rs_sm_count() * per_sm;
    if (grid > prm.n_tiles) grid = prm.n_tiles;
    rs_prof_start(stream);
    onehot_kernel<A, PAIR, DENSE, TS><<<(unsigned)grid, OH_THREADS, 0, stream>>>(prm);
    rs_prof_stop(stream);
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

template <int A, int TS = OH_TS>
static int dense_impl(const uint8_t *d_codes, int64_t n, const double *table, int W, void *d_out, void *stream,
                      int n_letters = A)
{
    int rc = check_args(d_codes, n, table, W);
    if (rc) return rc;
    if (n < W) return RS_OK;
    if (!d_out) { rs_set_error("null output"); return RS_ERR_INVALID; }
    OneHotParamsT<TS> prm = {};
    prm.codes_a = d_codes; prm.dense_out = d_out; prm.n = n; prm.padded = rs_padded_count(n);
    prm.n_tiles = (n + OH_TILE - 1) / OH_TILE; prm.W = W; prm.n_letters = n_letters;
    fill_table<TS>(prm.ta, table, W, n_letters);
    if (W <= 16) return dispatch_dense_w<A, 0, TS>(W, prm, (cudaStream_t)stream);
    return launch<A, false, true, TS>(prm, (cudaStream_t)stream);
}

// Every window's structure score as Python's round(score, 3) in thousandths (what rnascan prints, rnascan.py:273):
// 4 bytes per position instead of 8.  W <= 16.
extern "C" int rs_scores_dense_struct_milli(const uint8_t *d_codes, int64_t n, const double *table, int W,
                                            int32_t *d_out, void *stream)
{
    int rc = check_args(d_codes, n, table, W);
    if (rc) return rc;
    if (W > 16) { rs_set_error("rs_scores_dense_struct_milli: W <= 16 (use rs_scores_dense_struct)"); return RS_ERR_INVALID; }
    if (n < W) return RS_OK;
    if (!d_out) { rs_set_error("null output"); return RS_ERR_INVALID; }
    OneHotParams prm = {};
    prm.codes_a = d_codes; prm.dense_out = d_out; prm.n = n; prm.padded = rs_padded_count(n);
    prm.W = W;
    fill_table(prm.ta, table, W, 7);
    return dispatch_dense_w<7, 1, OH_TS>(W, prm, (cudaStream_t)stream);
}

extern "C" int rs_scores_dense_seq(const uint8_t *d_codes, int64_t n, const double *table, int W, float *d_out,
                                   void *stream)
{
    return dense_impl<4>(d_codes, n, table, W, d_out, stream);
}
extern "C" int rs_scores_dense_struct(const uint8_t *d_codes, int64_t n, const double *table, int W,
                                      double *d_out, void *stream)
{
    return dense_impl<7>(d_codes, n, table, W, d_out, stream);
}

// TS = OH_TS_ALPHA: the alphabet layout with n_letters letters (A = 0), generic kernel for every width.
template <int A, bool PAIR, int TS = OH_TS>
static int scan_impl(const uint8_t *ca, const uint8_t *cb, int64_t n, const double *ta, const double *tb, int W,
                     double threshold, int64_t cap, int64_t *d_hit_pos, float *d_hit_seq, double *d_hit_str,
                     uint64_t *d_counters2, void *d_work, int64_t work_bytes, void *stream, int n_letters = A)
{
    cudaStream_t st = (cudaStream_t)stream;
    int rc = check_args(ca, n, ta, W);
    if (rc) return rc;
    if (PAIR && (rc = check_args(cb, n, tb, W))) return rc;
    if (!d_counters2 || cap < 0 || (cap > 0 && !d_hit_pos)) { rs_set_error("bad hit buffers"); return RS_ERR_INVALID; }
    if (cap > 0 && ((A == 4 && !d_hit_seq) || ((A != 4 || PAIR) && !d_hit_str))) {
        rs_set_error("missing score buffer"); return RS_ERR_INVALID;
    }
    if (threshold != threshold) { rs_set_error("threshold is NaN"); return RS_ERR_INVALID; }
    // W <= 16 goes through kmer_finish_kernel, which writes both counters itself (one memset node fewer)
    const bool masks = TS == OH_TS && W <= 16;
    if (n < W || !masks) RS_CUDA(cudaMemsetAsync(d_counters2, 0, 2 * sizeof(uint64_t), st));
    if (n < W) return RS_OK;
    WorkLayout wl = rs_work_layout(n, cap);
    if (!d_work || work_bytes < wl.total) { rs_set_error("workspace too small: need %lld bytes", (long long)wl.total); return RS_ERR_WORKSPACE; }
    if (masks && A == 4 && !PAIR && W <= 8)   // exact k-mer decision table: one lookup decides 9-W positions
        return rs_scan_seq_kmer(ca, n, ta, W, threshold, cap, d_hit_pos, d_hit_seq, d_counters2, d_work, st);
    if (masks && PAIR)
        return rs_scan_pair_masks(ca, cb, n, ta, tb, W, threshold, cap, d_hit_pos, d_hit_seq, d_hit_str, d_counters2,
                                  d_work, st);
    if (masks)                                // compile-time width, ballot hit masks, segment scan + expansion
        return rs_scan_onehot_masks(A, ca, n, ta, W, threshold, cap, d_hit_pos, d_hit_seq, d_hit_str, d_counters2,
                                    d_work, st);
    OneHotParamsT<TS> prm = {};
    prm.codes_a = ca; prm.codes_b = cb; prm.n = n; prm.padded = rs_padded_count(n);
    prm.n_tiles = (n + OH_TILE - 1) / OH_TILE; prm.W = W; prm.threshold = threshold; prm.n_letters = n_letters;
    uint8_t *wk = (uint8_t *)d_work;
    prm.st.pos = (int64_t *)(wk + wl.off_pos);
    prm.st.seq = d_hit_seq ? (float *)(wk + wl.off_seq) : nullptr;
    prm.st.str = d_hit_str ? (double *)(wk + wl.off_str) : nullptr;
    prm.st.tile_seg = (ulonglong2 *)(wk + wl.off_seg);
    prm.st.counters = (unsigned long long *)d_counters2;
    prm.st.capacity = cap;
    fill_table<TS>(prm.ta, ta, W, n_letters);
    if (PAIR) fill_table(prm.tb, tb, W, 7);
    rc = launch<A, PAIR, false, TS>(prm, st);
    if (rc) return rc;
    OrderDest od = {d_hit_pos, d_hit_seq, d_hit_str, nullptr, nullptr, 0};
    return rs_order_hits(prm.st, prm.n_tiles, od, wk + wl.off_scan, st);
}

extern "C" int rs_scan_seq(const uint8_t *d_codes, int64_t n, const double *table, int W, double threshold,
                           int64_t cap, int64_t *d_hit_pos, float *d_hit_score, uint64_t *d_counters2,
                           void *d_work, int64_t work_bytes, void *stream)
{
    return scan_impl<4, false>(d_codes, nullptr, n, table, nullptr, W, threshold, cap, d_hit_pos, d_hit_score,
                               nullptr, d_counters2, d_work, work_bytes, stream);
}
extern "C" int rs_scan_struct_onehot(const uint8_t *d_codes, int64_t n, const double *table, int W,
                                     double threshold, int64_t cap, int64_t *d_hit_pos, double *d_hit_score,
                                     uint64_t *d_counters2, void *d_work, int64_t work_bytes, void *stream)
{
    return scan_impl<7, false>(d_codes, nullptr, n, table, nullptr, W, threshold, cap, d_hit_pos, nullptr,
                               d_hit_score, d_counters2, d_work, work_bytes, stream);
}
extern "C" int rs_scan_pair_onehot(const uint8_t *d_seq_codes, const uint8_t *d_struct_codes, int64_t n,
                                   const double *seq_table, const double *struct_table, int W, double threshold,
                                   int64_t cap, int64_t *d_hit_pos, float *d_hit_seq, double *d_hit_struct,
                                   uint64_t *d_counters2, void *d_work, int64_t work_bytes, void *stream)
{
    return scan_impl<4, true>(d_seq_codes, d_struct_codes, n, seq_table, struct_table, W, threshold, cap,
                              d_hit_pos, d_hit_seq, d_hit_struct, d_counters2, d_work, work_bytes, stream);
}

// ---- any alphabet of 1..31 letters (the "alphabet" layout of rs_host_encode_alpha) ---------------------------------
// Replaces the dict lookup of _py_calculate (matrix.py:25-43) for alphabets other than BEHLMRT, and the window loop of
// pwm_scan_fwd (pfmutil.py:205-221).  Up to 7 letters run the structure instantiations: through code & 7 the layout's
// codes read as the letter's index, or as 7 for 0x1F and RS_SEP, and the table is zero-padded to 7 columns.
// 8..31 letters run the TS = 32 instantiations (index = code & 31; 0x1F and RS_SEP give 31 >= A).
static int alpha_table7(const double *table, int W, int A, double *t7)
{
    if (A < 1 || A > 31) { rs_set_error("alphabet of %d letters: 1..31 are supported", A); return RS_ERR_INVALID; }
    if (!table) { rs_set_error("null codes or table"); return RS_ERR_INVALID; }
    if (W < 1 || W > RS_MAX_W) { rs_set_error("motif width %d outside [1, %d]", W, RS_MAX_W); return RS_ERR_INVALID; }
    if (A <= 7)
        for (int j = 0; j < W; j++)
            for (int c = 0; c < 7; c++) t7[j * 7 + c] = c < A ? table[j * A + c] : 0.0;
    return RS_OK;
}

extern "C" int rs_scores_dense_alpha(const uint8_t *d_codes, int64_t n, const double *table, int W, int A,
                                     double *d_out, void *stream)
{
    double t7[RS_MAX_W * 7];
    int rc = alpha_table7(table, W, A, t7);
    if (rc) return rc;
    if (A <= 7) return dense_impl<7>(d_codes, n, t7, W, d_out, stream);
    return dense_impl<0, OH_TS_ALPHA>(d_codes, n, table, W, d_out, stream, A);
}

extern "C" int rs_scan_alpha(const uint8_t *d_codes, int64_t n, const double *table, int W, int A, double threshold,
                             int64_t cap, int64_t *d_hit_pos, double *d_hit_score, uint64_t *d_counters2,
                             void *d_work, int64_t work_bytes, void *stream)
{
    double t7[RS_MAX_W * 7];
    int rc = alpha_table7(table, W, A, t7);
    if (rc) return rc;
    if (A <= 7)
        return scan_impl<7, false>(d_codes, nullptr, n, t7, nullptr, W, threshold, cap, d_hit_pos, nullptr,
                                   d_hit_score, d_counters2, d_work, work_bytes, stream);
    return scan_impl<0, false, OH_TS_ALPHA>(d_codes, nullptr, n, table, nullptr, W, threshold, cap, d_hit_pos, nullptr,
                                            d_hit_score, d_counters2, d_work, work_bytes, stream, A);
}
