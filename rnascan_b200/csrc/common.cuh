// Shared device/host helpers for the rnascan_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include <float.h>
#include "../../include/rnascan_b200.h"

#define RS_CHANNELS 7            // B,E,H,L,M,R,T
#define RS_PAD      256          // rs_padded_count(n) = roundup(n, RS_PAD) + RS_PAD

// --------------------------------------------------------------------------- errors
void rs_set_error(const char *fmt, ...);
int  rs_cuda_fail(cudaError_t e, const char *what);
#define RS_CUDA(call)                                                     \
    do {                                                                  \
        cudaError_t e__ = (call);                                         \
        if (e__ != cudaSuccess) return rs_cuda_fail(e__, #call);          \
    } while (0)

static inline int64_t rs_roundup(int64_t x, int64_t m) { return (x + m - 1) / m * m; }
int rs_sm_count();               // SMs of the current device (cached)
int rs_grid_sms();               // SMs the persistent scan kernels may fill (rs_set_reserved_sms)
#define RS_MAX_DEVICES 64
int rs_current_device();         // cudaGetDevice clamped to [0, RS_MAX_DEVICES)
void rs_prof_start(cudaStream_t s);   // profiling hook (capi.cu): event pair around the main kernel
void rs_prof_stop(cudaStream_t s);

// --------------------------------------------------------------------------- PTX: mbarrier + 1-D bulk async copy (TMA engine, UBLKCP)
__device__ __forceinline__ uint32_t smem_u32(const void *p)
{
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// global -> shared bulk copy; dst, src 16-byte aligned, bytes a multiple of 16.
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
        ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// Look-back waits (order.cu, kmer_scan.cu) are bounded by WALL time, not by a spin count: a predecessor CTA always
// runs already (tickets are taken in launch order), so the wait is normally microseconds; under time-slicing, MPS,
// a debugger or a sanitizer it can legitimately be long, so only a full minute without progress is treated as a
// lost predecessor (trap: the launch fails instead of hanging the stream for ever).
__device__ __forceinline__ bool rs_spin_expired(unsigned long long &t_start)
{
    unsigned long long now;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
    if (t_start == 0ull) { t_start = now; return false; }
    return now - t_start > 60000000000ull;
}

// --------------------------------------------------------------------------- exact scoring primitives (shared by all kernels)
// numpy.nan_to_num on a double: NaN -> 0, +-inf -> +-DBL_MAX   (rnascan.py:306)
__device__ __forceinline__ double rs_nan_to_num(double d)
{
    if (d != d) return 0.0;
    if (isinf(d)) return d > 0 ? DBL_MAX : -DBL_MAX;
    return d;
}

// One window of the averaged-profile score, exactly rnascan.py:302-307:
//   sum_j nan_to_num( np.dot(profile row i+j, pssm row j) ).
// Both operands of that np.dot are strided pandas row views, so it runs OpenBLAS ddot's
// non-unit-stride loop; for 7 channels its compiled arithmetic is (oracle/pwm_oracle.c
// documents how this was established and pinned against the reference's own outputs):
//   m3 = x2*y2; m4 = x3*y3; t1 = fma(x0,y0,m3); t2 = fma(x1,y1,m4);
//   t1 = fma(x4,y4,t1); t1 = fma(x5,y5,t1); t1 = fma(x6,y6,t1); dot = t1 + t2
__device__ __forceinline__ double rs_ddot7(double x0, double x1, double x2, double x3, double x4, double x5,
                                           double x6, const double *y)
{
    const double m3 = __dmul_rn(x2, y[2]), m4 = __dmul_rn(x3, y[3]);
    double t1 = __fma_rn(x0, y[0], m3);
    const double t2 = __fma_rn(x1, y[1], m4);
    t1 = __fma_rn(x4, y[4], t1);
    t1 = __fma_rn(x5, y[5], t1);
    t1 = __fma_rn(x6, y[6], t1);
    return __dadd_rn(t1, t2);
}

template <typename PT>
__device__ __forceinline__ double rs_exact_profile_window(const PT *rows /* first row of window */,
                                                          const double *tab /* [W][7] */, int W)
{
    double score = 0.0;
    for (int j = 0; j < W; j++) {
        const PT *r = rows + j * RS_CHANNELS;
        const double d = rs_ddot7((double)r[0], (double)r[1], (double)r[2], (double)r[3], (double)r[4],
                                  (double)r[5], (double)r[6], tab + j * RS_CHANNELS);
        score = __dadd_rn(score, rs_nan_to_num(d));
    }
    return score;
}

// One window of a one-hot PSSM score: sequential double adds in j order (_pwm.c:36-60,
// matrix.py:34-38).  A = number of valid letters (4 or 7), table row stride TS doubles.
// The letter index is code & 7 for TS <= 8 (RNA and structure layouts) and code & 31 for TS = 32
// (alphabet layout, whose letter count is only known at run time: pass it as n_letters).
// Returns false when the window holds an invalid symbol (score is NaN in the reference).
template <int A, int TS>
__device__ __forceinline__ bool rs_exact_onehot_window(const uint8_t *codes, const double *tab, int W,
                                                       double &score, int n_letters = A)
{
    constexpr int MASK = TS > 8 ? TS - 1 : 7;
    double s = 0.0;
    bool ok = true;
    for (int j = 0; j < W; j++) {
        int idx = codes[j] & MASK;
        if (idx >= n_letters) { ok = false; break; }
        s = __dadd_rn(s, tab[j * TS + idx]);
    }
    score = s;
    return ok;
}

// true when symbols [0, W) hold no separator
__device__ __forceinline__ bool rs_no_separator(const uint8_t *codes, int W)
{
    for (int j = 0; j < W; j++)
        if (codes[j] == RS_SEP) return false;
    return true;
}

// --------------------------------------------------------------------------- hit staging
// Scan kernels append the hits of one tile, in position order, to a staging area at an
// atomically claimed offset and record (offset,count) per tile; order.cu then copies the
// segments out in tile order, so the final list is sorted by position.
struct HitStage {
    int64_t  *pos;        // staging arrays, capacity entries each
    float    *seq;
    double   *str;
    ulonglong2 *tile_seg; // per tile: (staging offset, count)   [n_tiles]
    unsigned long long *counters;   // [0] hits, [1] exact re-scores
    int64_t   capacity;
};

struct WorkLayout {
    int64_t off_pos, off_seq, off_str, off_seg, off_scan, off_lut, total;
};
WorkLayout rs_work_layout(int64_t n, int64_t capacity);
// Batched scans append every motif's ordered hits behind the previous motif's: `out_base`
// (device, may be NULL = 0) is added to the destination index, `out_motif` (may be NULL)
// receives `motif_id` for every hit written.
struct OrderDest {
    int64_t *pos; float *seq; double *str;
    const unsigned long long *out_base;
    int32_t *out_motif;
    int32_t  motif_id;
};
int64_t rs_order_tmp_bytes(int64_t max_tiles);    // scratch rs_order_hits needs for up to max_tiles tiles
int rs_order_hits(const HitStage &st, int64_t n_tiles, const OrderDest &dst, void *d_scan_tmp,
                  cudaStream_t stream);

// Append this tile's hits (bit i of `mask` = window i of this thread, consecutive windows
// per thread) to the staging area in position order.  All threads of the CTA call it.
template <int THREADS, typename RECOMPUTE>
__device__ __forceinline__ void emit_tile_hits(const HitStage &st, int64_t tile, unsigned mask, int nbits,
                                               RECOMPUTE recompute)
{
    __shared__ unsigned s_warp[THREADS / 32];
    __shared__ unsigned long long s_base;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned cnt = __popc(mask);
    unsigned incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        unsigned v = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += v;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    unsigned before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < THREADS / 32; w++) {
        unsigned v = s_warp[w];
        if (w < warp) before += v;
        total += v;
    }
    if (threadIdx.x == 0) {
        unsigned long long base = atomicAdd(st.counters, (unsigned long long)total);   // one atomic per tile
        s_base = base;
        st.tile_seg[tile] = make_ulonglong2(base, (unsigned long long)total);
    }
    __syncthreads();
    unsigned long long k = s_base + before + (incl - cnt);
    for (int i = 0; i < nbits; i++) {
        if (mask & (1u << i)) {
            if ((int64_t)k < st.capacity) recompute(i, (int64_t)k);
            k++;
        }
    }
}

// Same, with the sequence half of the combined decision applied to the staged (structure-only)
// candidates first; *d_total_out = survivors.
int rs_order_hits_seq_refined(const HitStage &st, int64_t n_tiles, const OrderDest &dst, void *d_scan_tmp,
                              cudaStream_t stream, const uint8_t *d_codes, int64_t n, const double *seq_table, int W,
                              double threshold, unsigned long long *d_total_out);

#define RS_MIN_TILE 512          // no scan kernel orders segments shorter than this (sizes the segment table)
int64_t rs_batched_tc_work_bytes(int64_t n, int n_motifs, int stride_rows, int64_t hit_capacity);
int rs_scan_batched_tc(const uint8_t *d_codes, const void *d_profile, int64_t n, int n_motifs, const int *widths,
                       const double *seq_tables, const double *struct_tables, int stride_rows, double threshold,
                       double profile_absrow_max, int mode, int64_t hit_capacity, int32_t *d_hit_motif,
                       int64_t *d_hit_pos, float *d_hit_seq, double *d_hit_struct, uint64_t *d_motif_counters2,
                       uint64_t *d_bases, void *d_work, int64_t work_bytes, cudaStream_t st,
                       const double *d_exact64 = nullptr);
int rs_scan_onehot_masks(int A, const uint8_t *d_codes, int64_t n, const double *table, int W, double threshold,
                         int64_t cap, int64_t *d_hit_pos, float *d_hit_seq, double *d_hit_str,
                         uint64_t *d_counters2, void *d_work, cudaStream_t st);
int rs_scan_pair_masks(const uint8_t *d_seq_codes, const uint8_t *d_struct_codes, int64_t n, const double *seq_table,
                       const double *struct_table, int W, double threshold, int64_t cap, int64_t *d_hit_pos,
                       float *d_hit_seq, double *d_hit_str, uint64_t *d_counters2, void *d_work, cudaStream_t st);
int64_t rs_kmer_work_bytes(int64_t n);   // workspace of the W <= 8 sequence scan (kmer_scan.cu)
#define RS_KMER_WMAX 16          // widest motif the k-mer decision masks take
// k-mer decision masks of one-hot motifs (batched_tc.cu): mask[kmer][word], bit (31 - k) of word c = motif 32 c + k
// may pass; alphabet 4: 8-mers (65536 rows), 7: 5-mers (32768 rows); device tables [n_motifs][stride_rows][alphabet].
int rs_kmer_mask_build(int alphabet, uint32_t *d_mask, int mask_words, const double *d_tables, const int *d_widths,
                       int n_motifs, int stride_rows, double threshold, cudaStream_t st);

int rs_scan_seq_kmer(const uint8_t *d_codes, int64_t n, const double *table, int W, double threshold, int64_t cap,
                     int64_t *d_hit_pos, float *d_hit_score, uint64_t *d_counters2, void *d_work, cudaStream_t st);
