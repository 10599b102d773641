// Averaged-structure (7-channel profile) scans, fused with the sequence PSSM.
//
// Replaces the pandas double loop of /root/reference/rnascan/rnascan.py:293-315
// (scan_averaged_structure) and, in RS_MODE_AND, the sequence scan + inner join of
// rnascan.py:258-275,416-434 for the combined mode.
//
// Two kernels:
//   fused_filter_kernel<W>   float32 profiles, W <= RS_FAST_W.  Persistent CTAs stream
//       tiles of (TILE+W-1) profile rows (28 B each) + symbol codes into a 3-stage shared
//       memory ring with 1-D bulk async copies (TMA engine) completing on mbarriers.  Each
//       thread correlates 9 consecutive windows from registers: every profile row is
//       loaded from shared memory once per thread and reused by up to W windows; the W x 7
//       table sits in the constant bank (kernel parameters), so the inner loop is pure
//       FFMA with a constant operand.  The fp32 result is only a FILTER: windows whose
//       fp32 score is within the guard band of the threshold are re-scored in fp64 in the
//       reference's exact operation order, and only those decide/emit hits.
//   profile_exact_kernel<PT> any profile dtype, any W <= RS_MAX_W, dense output or hits,
//       non-finite PSSM entries: everything in fp64 in the reference's order.
#include "common.cuh"

#include "profile_params.cuh"

// Exact evaluation of window `i` (tile-relative) from the staged tile; returns whether it
// is a hit and its scores.  Shared by the filter kernel's rare path and the exact kernel.
template <typename PT>
__device__ __forceinline__ bool exact_window(const ProfileParams &prm, const PT *prof, const uint8_t *codes,
                                             int i, int64_t gpos, float &seq_out, double &str_out)
{
    const int W = prm.W;
    if (gpos + W > prm.n) return false;
    double s = rs_exact_profile_window<PT>(prof + (size_t)i * RS_CHANNELS, prm.sd, W);
    str_out = s;
    if (!(s > prm.threshold)) return false;
    if (prm.mode == RS_MODE_AND) {
        double q;
        if (!rs_exact_onehot_window<4, 4>(codes + i, prm.qd, W, q)) return false;
        float qf = (float)q;                     // _pwm.c:65
        seq_out = qf;
        return (double)qf > prm.threshold;       // SURVEY.md note N1
    }
    seq_out = 0.f;
    return codes == nullptr || rs_no_separator(codes + i, W);
}

// Candidate test of the DEFERRED scans (rs_filter_profile): the exact rows are not on the device, so a
// window that passed the fp32 filter is kept unless the symbols alone rule it out -- it runs over the
// end of the stream, holds a separator, or (when the sequence table is already known) its sequence
// score fails.  rs_resolve_candidates decides from the exact rows.
__device__ __forceinline__ bool deferred_window(const ProfileParams &prm, const uint8_t *codes, int i, int64_t gpos)
{
    const int W = prm.W;
    if (gpos + W > prm.n) return false;
    if (prm.mode == RS_MODE_AND) {
        double q;
        if (!rs_exact_onehot_window<4, 4>(codes + i, prm.qd, W, q)) return false;
        return (double)(float)q > prm.threshold;
    }
    return rs_no_separator(codes + i, W);
}

// ------------------------------------------------------------------------------------------------
template <int W>
__global__ void __launch_bounds__(FT_THREADS, 2) fused_filter_kernel(const __grid_constant__ ProfileParams prm)
{
    constexpr int ROWS = FT_TILE + W - 1;
    constexpr uint32_t PROF_BYTES = ru16(ROWS * RS_CHANNELS * 4);
    constexpr uint32_t CODE_BYTES = ru16(ROWS);
    constexpr uint32_t STAGE_BYTES = PROF_BYTES + CODE_BYTES;
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem);
    uint8_t *stages = smem + 128;

    const int tid = threadIdx.x;
    if (tid == 0) {
        for (int s = 0; s < FT_STAGES; s++) mbar_init(&bars[s], 1);
        fence_mbar_init();
    }
    __syncthreads();

    const int64_t stride = gridDim.x;
    const int64_t first = blockIdx.x;
    const int64_t my_tiles = first < prm.n_tiles ? (prm.n_tiles - first + stride - 1) / stride : 0;
    const int64_t prof_end = prm.padded * (RS_CHANNELS * 4);

    auto issue = [&](int64_t it) {
        const int s = (int)(it % FT_STAGES);
        const int64_t t0 = (first + it * stride) * FT_TILE;
        uint8_t *dst = stages + (size_t)s * STAGE_BYTES;
        const int64_t pstart = t0 * (RS_CHANNELS * 4);
        const uint32_t pbytes = (uint32_t)min((int64_t)PROF_BYTES, prof_end - pstart);
        const uint32_t cbytes = (uint32_t)min((int64_t)CODE_BYTES, prm.padded - t0);
        mbar_expect_tx(&bars[s], pbytes + cbytes);
        bulk_g2s(dst, reinterpret_cast<const uint8_t *>(prm.profile) + pstart, pbytes, &bars[s]);
        bulk_g2s(dst + PROF_BYTES, prm.codes + t0, cbytes, &bars[s]);
    };

    if (tid == 0)
        for (int64_t it = 0; it < FT_STAGES - 1 && it < my_tiles; it++) issue(it);

    unsigned cnt[4] = {0u, 0u, 0u, 0u};

    for (int64_t it = 0; it < my_tiles; it++) {
        const int s = (int)(it % FT_STAGES);
        if (tid == 0 && it + FT_STAGES - 1 < my_tiles) issue(it + FT_STAGES - 1);
        mbar_wait(&bars[s], (uint32_t)((it / FT_STAGES) & 1));

        const int64_t tile = first + it * stride;
        const int64_t t0 = tile * FT_TILE;
        const float *prof = reinterpret_cast<const float *>(stages + (size_t)s * STAGE_BYTES);
        const uint8_t *codes = stages + (size_t)s * STAGE_BYTES + PROF_BYTES;
        const float *rows = prof + tid * (FT_P * RS_CHANNELS);

        // ---- dense fp32 filter: 9 windows x W rows x 7 channels, rows reused from registers
        float acc[FT_P];
#pragma unroll
        for (int i = 0; i < FT_P; i++) acc[i] = 0.f;
#pragma unroll
        for (int r = 0; r < FT_P + W - 1; r++) {
            float x[RS_CHANNELS];
#pragma unroll
            for (int c = 0; c < RS_CHANNELS; c++) x[c] = rows[r * RS_CHANNELS + c];
#pragma unroll
            for (int j = 0; j < W; j++) {
                const int i = r - j;
                if (i >= 0 && i < FT_P) {
#pragma unroll
                    for (int c = 0; c < RS_CHANNELS; c++)
                        acc[i] = fmaf(x[c], prm.sf[j * RS_CHANNELS + c], acc[i]);
                }
            }
        }

        // ---- background counts of the rows this thread owns (rs_scan_fused_candidates_counting): the symbols are
        //      staged anyway, so the separate histogram pass -- a second read of 1 of the 30 B per position -- goes away
        if (prm.count_on) {
            unsigned packed = 0;                                   // four byte counters, <= 9 each
#pragma unroll
            for (int r = 0; r < FT_P; r++) {
                const unsigned code = codes[tid * FT_P + r];
                const bool counted = code < 4u && t0 + tid * FT_P + r < prm.count_rows;
                packed += counted ? (1u << (8u * code)) : 0u;
            }
            cnt[0] += packed & 0xffu; cnt[1] += (packed >> 8) & 0xffu;
            cnt[2] += (packed >> 16) & 0xffu; cnt[3] += packed >> 24;
        }

        // ---- guard band: anything not provably below the threshold is re-scored exactly, the whole CTA sharing
        //      the tile's candidates (resolve_tile_candidates)
        unsigned candmask = 0;
#pragma unroll
        for (int i = 0; i < FT_P; i++)
            if (!(acc[i] <= prm.filt_thr)) candmask |= 1u << i;

        const int any = __syncthreads_or(candmask != 0);
        if (any) {
            resolve_tile_candidates<FT_THREADS, FT_P>(
                prm.st, tile, candmask,
                [&](int w) {
                    float sq; double st;
                    return prm.defer ? deferred_window(prm, codes, w, t0 + w)
                                     : exact_window<float>(prm, prof, codes, w, t0 + w, sq, st);
                },
                [&](int w, int64_t k) {
                    prm.st.pos[k] = prm.pos_base + t0 + w;
                    if (prm.defer) return;
                    float sq; double st;
                    exact_window<float>(prm, prof, codes, w, t0 + w, sq, st);
                    prm.st.str[k] = st;
                    if (prm.st.seq) prm.st.seq[k] = sq;
                });
        } else if (tid == 0) {
            prm.st.tile_seg[tile] = make_ulonglong2(0ull, 0ull);
        }
    }

    if (prm.count_on) {
#pragma unroll
        for (int k = 0; k < 4; k++) {
            unsigned v = cnt[k];
            for (int d = 16; d; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
            if ((tid & 31) == 0 && v) atomicAdd(prm.counts8 + k, (unsigned long long)v);
        }
    }
}

// ------------------------------------------------------------------------------------------------
template <typename PT>
__global__ void __launch_bounds__(EX_THREADS) profile_exact_kernel(const __grid_constant__ ProfileParams prm)
{
    const int W = prm.W;
    const int rows_max = EX_TILE + RS_MAX_W - 1;
    const uint32_t PROF_BYTES = ru16(rows_max * RS_CHANNELS * (uint32_t)sizeof(PT));
    const uint32_t CODE_BYTES = ru16(rows_max);
    const uint32_t STAGE_BYTES = PROF_BYTES + CODE_BYTES;
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem);
    uint8_t *stages = smem + 128;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        for (int s = 0; s < EX_STAGES; s++) mbar_init(&bars[s], 1);
        fence_mbar_init();
    }
    __syncthreads();

    const int64_t stride = gridDim.x, first = blockIdx.x;
    const int64_t my_tiles = first < prm.n_tiles ? (prm.n_tiles - first + stride - 1) / stride : 0;
    const int64_t prof_end = prm.padded * (int64_t)(RS_CHANNELS * sizeof(PT));
    const uint32_t need_prof = ru16((EX_TILE + W - 1) * RS_CHANNELS * (uint32_t)sizeof(PT));
    const uint32_t need_code = ru16(EX_TILE + W - 1);

    auto issue = [&](int64_t it) {
        const int s = (int)(it % EX_STAGES);
        const int64_t t0 = (first + it * stride) * EX_TILE;
        uint8_t *dst = stages + (size_t)s * STAGE_BYTES;
        const int64_t pstart = t0 * (int64_t)(RS_CHANNELS * sizeof(PT));
        const uint32_t pbytes = (uint32_t)min((int64_t)need_prof, prof_end - pstart);
        const uint32_t cbytes = prm.codes ? (uint32_t)min((int64_t)need_code, prm.padded - t0) : 0u;
        mbar_expect_tx(&bars[s], pbytes + cbytes);
        bulk_g2s(dst, reinterpret_cast<const uint8_t *>(prm.profile) + pstart, pbytes, &bars[s]);
        if (cbytes) bulk_g2s(dst + PROF_BYTES, prm.codes + t0, cbytes, &bars[s]);
    };
    if (tid == 0)
        for (int64_t it = 0; it < EX_STAGES - 1 && it < my_tiles; it++) issue(it);

    constexpr int PER = EX_TILE / EX_THREADS;       // 8 windows per thread, lane-contiguous
    for (int64_t it = 0; it < my_tiles; it++) {
        const int s = (int)(it % EX_STAGES);
        if (tid == 0 && it + EX_STAGES - 1 < my_tiles) issue(it + EX_STAGES - 1);
        mbar_wait(&bars[s], (uint32_t)((it / EX_STAGES) & 1));

        const int64_t tile = first + it * stride;
        const int64_t t0 = tile * EX_TILE;
        const PT *prof = reinterpret_cast<const PT *>(stages + (size_t)s * STAGE_BYTES);
        const uint8_t *codes = prm.codes ? stages + (size_t)s * STAGE_BYTES + PROF_BYTES : nullptr;

        unsigned hitmask = 0;
        for (int k = 0; k < PER; k++) {
            const int w = warp * (32 * PER) + k * 32 + lane;
            const int64_t gpos = t0 + w;
            if (prm.dense) {
                if (gpos + W <= prm.n) {
                    double sc = rs_exact_profile_window<PT>(prof + (size_t)w * RS_CHANNELS, prm.sd, W);
                    if (codes && !rs_no_separator(codes + w, W)) sc = nan("");
                    prm.dense_out[gpos] = sc;
                }
            } else {
                float sq; double st;
                if (exact_window<PT>(prm, prof, codes, w, gpos, sq, st)) hitmask |= 1u << k;
            }
        }
        if (prm.dense) {
            __syncthreads();
            continue;
        }
        const int any = __syncthreads_or(hitmask != 0);
        if (any) {
            // lane-contiguous mapping: order inside a warp is (k, lane); emit k by k
            __shared__ unsigned s_cnt[EX_THREADS / 32][PER];
            __shared__ unsigned long long s_base2;
            for (int k = 0; k < PER; k++) {
                unsigned b = __ballot_sync(0xffffffffu, (hitmask >> k) & 1u);
                if (lane == 0) s_cnt[warp][k] = __popc(b);
            }
            __syncthreads();
            unsigned before = 0, total = 0;
            for (int ww = 0; ww < EX_THREADS / 32; ww++)
                for (int k = 0; k < PER; k++) {
                    unsigned v = s_cnt[ww][k];
                    if (ww < warp) before += v;
                    total += v;
                }
            if (tid == 0) {
                unsigned long long base = atomicAdd(prm.st.counters, (unsigned long long)total);
                s_base2 = base;
                prm.st.tile_seg[tile] = make_ulonglong2(base, (unsigned long long)total);
            }
            __syncthreads();
            unsigned long long kk = s_base2 + before;
            for (int k = 0; k < PER; k++) {
                unsigned b = __ballot_sync(0xffffffffu, (hitmask >> k) & 1u);
                if ((hitmask >> k) & 1u) {
                    unsigned long long dst = kk + __popc(b & ((1u << lane) - 1u));
                    if ((int64_t)dst < prm.st.capacity) {
                        const int w = warp * (32 * PER) + k * 32 + lane;
                        float sq; double st;
                        exact_window<PT>(prm, prof, codes, w, t0 + w, sq, st);
                        prm.st.pos[dst] = t0 + w;
                        prm.st.str[dst] = st;
                        if (prm.st.seq) prm.st.seq[dst] = sq;
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
// profile statistics: [0] max_r sum_c |p[r][c]|, [1] non-finite entries, [2] negative entries
template <typename PT>
__global__ void profile_stats_kernel(const PT *p, int64_t n_rows, double *stats)
{
    double mx = 0.0;
    unsigned long long bad = 0, neg = 0;
    for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < n_rows;
         r += (int64_t)gridDim.x * blockDim.x) {
        double s = 0.0;
#pragma unroll
        for (int c = 0; c < RS_CHANNELS; c++) {
            double v = (double)p[r * RS_CHANNELS + c];
            if (!isfinite(v)) bad++;
            else { s += fabs(v); if (v < 0) neg++; }
        }
        mx = fmax(mx, s);
    }
    for (int d = 16; d; d >>= 1) {
        mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, d));
        bad += __shfl_xor_sync(0xffffffffu, bad, d);
        neg += __shfl_xor_sync(0xffffffffu, neg, d);
    }
    if ((threadIdx.x & 31) == 0) {
        // non-negative doubles order like their bit patterns
        atomicMax(reinterpret_cast<unsigned long long *>(stats), (unsigned long long)__double_as_longlong(mx));
        if (bad) atomicAdd(reinterpret_cast<unsigned long long *>(stats + 1), bad);
        if (neg) atomicAdd(reinterpret_cast<unsigned long long *>(stats + 2), neg);
    }
}
__global__ void stats_finish_kernel(double *stats)
{
    stats[1] = (double)(*reinterpret_cast<unsigned long long *>(stats + 1));
    stats[2] = (double)(*reinterpret_cast<unsigned long long *>(stats + 2));
}

// ------------------------------------------------------------------------------------------------
// host side
// Filter table + lowered threshold of the fp32 filter kernels.  Returns false when the filter cannot be
// used (non-finite threshold / row bound, +inf or NaN table entries): the exact kernel then runs.
//   rows of the table that hold -inf (zero-probability letters with pseudocount 0) are replaced by a
//   non-negative upper bound (nan_to_num makes such a row contribute 0 or -DBL_MAX, never more than
//   max(0, finite part));
//   value_scale: the device multiplies stored values by this to get p (1 for float rows, scale/255 for
//   quantised rows) -- folded into the table; quant_step: largest |p - stored * value_scale| per entry
//   (0 for float rows; the float32 shadow of float64 rows is covered by `shadow`).
static bool build_filter(ProfileParams &prm, const double *struct_table, int W, double threshold,
                         double profile_absrow_max, double value_scale, double quant_step, bool shadow,
                         bool one_sided = false)
{
    if (!(isfinite(threshold) && isfinite(profile_absrow_max) && profile_absrow_max >= 0 && profile_absrow_max < 1e30))
        return false;
    double S = 0.0, Sf = 0.0, A = 0.0, Apos = 0.0;
    for (int j = 0; j < W; j++) {
        bool row_nonfinite = false;
        double rowmax = 0.0, rowmax_f = 0.0;
        for (int c = 0; c < RS_CHANNELS; c++) {
            double v = struct_table[j * RS_CHANNELS + c];
            if (v != v || v == INFINITY) return false;           // NaN / +inf: exact kernel only
            if (v == -INFINITY) row_nonfinite = true;
        }
        for (int c = 0; c < RS_CHANNELS; c++) {
            double v = struct_table[j * RS_CHANNELS + c];
            double f = row_nonfinite ? ((isfinite(v) && v > 0) ? v : 0.0) : v;
            const float sf = f32_round_up(f * value_scale);
            prm.sf[j * RS_CHANNELS + c] = sf;
            if (!isfinite((double)sf)) return false;
            rowmax = fmax(rowmax, fabs(f));
            rowmax_f = fmax(rowmax_f, fabs((double)sf));
            A += fabs(f);
            if (f > 0) Apos += f;
        }
        S += rowmax;
        Sf += rowmax_f;
    }
    // |fp32 result - real value of sum(stored * sf)| <= gamma * sum|stored * sf| <= gamma * (R / value_scale + 4) * Sf
    // (a row of stored values sums to at most R / value_scale + 3.5 after rounding), and sf >= table * value_scale
    // entry wise for stored values >= 0; negative p are covered by the generous constant.
    const double R = fmax(profile_absrow_max, 1.0);
    double tol = ldexp(1.0, -23) * (double)(RS_CHANNELS * W + 8) * Sf * (R / value_scale + (quant_step > 0 ? 4.0 : 0.0));
    if (quant_step > 0 && !one_sided) tol += quant_step * A * (1.0 + 1e-9);      // |p - p~| <= quant_step per entry
    // floored values: 0 <= p - p~ < quant_step, so only positive table entries can be under-counted (the tiny
    // two-sided term covers the floating-point evaluation of the floor itself)
    if (quant_step > 0 && one_sided) tol += quant_step * Apos * (1.0 + 1e-9) + quant_step * A * 1e-9;
    if (shadow) tol += ldexp(1.0, -24) * R * S * 1.001 + ldexp(1.0, -149) * A;   // float32 rounding of float64 rows
    prm.filt_thr = f32_round_down(threshold - tol);
    return isfinite((double)prm.filt_thr);
}

template <int W>
static int launch_filter(const ProfileParams &prm, cudaStream_t stream)
{
    constexpr int ROWS = FT_TILE + W - 1;
    constexpr uint32_t STAGE_BYTES = ru16(ROWS * RS_CHANNELS * 4) + ru16(ROWS);
    const size_t smem = 128 + (size_t)FT_STAGES * STAGE_BYTES;
    static bool configured[RS_MAX_DEVICES] = {};          // the attribute is per device
    const int dev = rs_current_device();
    if (!configured[dev]) {
        RS_CUDA(cudaFuncSetAttribute(fused_filter_kernel<W>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured[dev] = true;
    }
    int64_t grid = (int64_t)rs_grid_sms() * 2;
    if (grid > prm.n_tiles) grid = prm.n_tiles;
    rs_prof_start(stream);
    fused_filter_kernel<W><<<(unsigned)grid, FT_THREADS, smem, stream>>>(prm);
    rs_prof_stop(stream);
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

template <int W>
struct FilterDispatch {
    static int run(int w, const ProfileParams &prm, cudaStream_t stream)
    {
        if (w == W) return launch_filter<W>(prm, stream);
        return FilterDispatch<W - 1>::run(w, prm, stream);
    }
};
template <>
struct FilterDispatch<0> {
    static int run(int, const ProfileParams &, cudaStream_t)
    {
        rs_set_error("internal: no filter kernel for this W");
        return RS_ERR_INVALID;
    }
};

template <typename PT>
static int launch_exact(const ProfileParams &prm, cudaStream_t stream)
{
    const int rows_max = EX_TILE + RS_MAX_W - 1;
    const size_t stage = ru16(rows_max * RS_CHANNELS * (uint32_t)sizeof(PT)) + ru16(rows_max);
    const size_t smem = 128 + (size_t)EX_STAGES * stage;
    static bool configured[RS_MAX_DEVICES] = {};          // the attribute is per device
    const int dev = rs_current_device();
    if (!configured[dev]) {
        RS_CUDA(cudaFuncSetAttribute(profile_exact_kernel<PT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured[dev] = true;
    }
    int64_t grid = (int64_t)rs_grid_sms() * (sizeof(PT) == 4 ? 3 : 1);
    if (grid > prm.n_tiles) grid = prm.n_tiles;
    rs_prof_start(stream);
    profile_exact_kernel<PT><<<(unsigned)grid, EX_THREADS, smem, stream>>>(prm);
    rs_prof_stop(stream);
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

static int check_common(const void *d_profile, int dtype, int64_t n, const double *struct_table, int W)
{
    if (!d_profile || !struct_table) { rs_set_error("null profile or table"); return RS_ERR_INVALID; }
    if (dtype != RS_F32 && dtype != RS_F64) { rs_set_error("profile_dtype must be RS_F32 or RS_F64"); return RS_ERR_INVALID; }
    if (W < 1 || W > RS_MAX_W) { rs_set_error("motif width %d outside [1, %d]", W, RS_MAX_W); return RS_ERR_INVALID; }
    if (n < 0) { rs_set_error("negative length"); return RS_ERR_INVALID; }
    if ((uintptr_t)d_profile & 15) { rs_set_error("profile pointer must be 16-byte aligned"); return RS_ERR_INVALID; }
    return RS_OK;
}

extern "C" int rs_profile_stats(const void *d_profile, int profile_dtype, int64_t n_rows, double *d_stats3,
                                void *stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    if (!d_profile || !d_stats3 || n_rows < 0) { rs_set_error("rs_profile_stats: bad argument"); return RS_ERR_INVALID; }
    RS_CUDA(cudaMemsetAsync(d_stats3, 0, 3 * sizeof(double), st));
    if (n_rows > 0) {
        int grid = rs_sm_count() * 8;
        if (profile_dtype == RS_F32)
            profile_stats_kernel<float><<<grid, 256, 0, st>>>((const float *)d_profile, n_rows, d_stats3);
        else if (profile_dtype == RS_F64)
            profile_stats_kernel<double><<<grid, 256, 0, st>>>((const double *)d_profile, n_rows, d_stats3);
        else { rs_set_error("bad profile_dtype"); return RS_ERR_INVALID; }
        RS_CUDA(cudaGetLastError());
    }
    stats_finish_kernel<<<1, 1, 0, st>>>(d_stats3);
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

extern "C" int rs_scores_dense_profile(const void *d_profile, int profile_dtype, int64_t n_rows,
                                       const uint8_t *d_codes, const double *table, int W, double *d_out,
                                       void *stream)
{
    int rc = check_common(d_profile, profile_dtype, n_rows, table, W);
    if (rc) return rc;
    if (n_rows < W) return RS_OK;
    if (!d_out) { rs_set_error("null output"); return RS_ERR_INVALID; }
    if (d_codes && ((uintptr_t)d_codes & 15)) { rs_set_error("codes pointer must be 16-byte aligned"); return RS_ERR_INVALID; }
    ProfileParams prm = {};
    prm.codes = d_codes; prm.profile = d_profile; prm.dense_out = d_out;
    prm.n = n_rows; prm.padded = rs_padded_count(n_rows);
    prm.n_tiles = (n_rows + EX_TILE - 1) / EX_TILE;
    prm.W = W; prm.dense = 1; prm.mode = RS_MODE_STRUCT; prm.threshold = 0;
    for (int k = 0; k < W * RS_CHANNELS; k++) prm.sd[k] = table[k];
    return profile_dtype == RS_F32 ? launch_exact<float>(prm, (cudaStream_t)stream)
                                   : launch_exact<double>(prm, (cudaStream_t)stream);
}

static int scan_fused_impl(const uint8_t *d_codes, const void *d_profile, int profile_dtype, int64_t n,
                           const double *seq_table, const double *struct_table, int W, double threshold,
                           double profile_absrow_max, int mode, int64_t hit_capacity, int64_t *d_hit_pos,
                           float *d_hit_seq, double *d_hit_struct, uint64_t *d_counters2, void *d_work,
                           int64_t work_bytes, void *stream, const unsigned long long *d_out_base,
                           int32_t *d_hit_motif, int32_t motif_id, int64_t *staged_tiles_out = nullptr,
                           uint64_t *d_counts8 = nullptr)
{
    cudaStream_t st = (cudaStream_t)stream;
    int rc = check_common(d_profile, profile_dtype, n, struct_table, W);
    if (rc) return rc;
    if (!d_codes || ((uintptr_t)d_codes & 15)) { rs_set_error("codes pointer null or not 16-byte aligned"); return RS_ERR_INVALID; }
    if (mode != RS_MODE_STRUCT && mode != RS_MODE_AND) { rs_set_error("bad mode"); return RS_ERR_INVALID; }
    if (mode == RS_MODE_AND && (!seq_table || !d_hit_seq)) { rs_set_error("RS_MODE_AND needs a sequence table and d_hit_seq"); return RS_ERR_INVALID; }
    if (!d_counters2 || hit_capacity < 0 ||
        (hit_capacity > 0 && !staged_tiles_out && (!d_hit_pos || !d_hit_struct))) {
        rs_set_error("bad hit buffers"); return RS_ERR_INVALID;
    }
    if (threshold != threshold) { rs_set_error("threshold is NaN"); return RS_ERR_INVALID; }
    RS_CUDA(cudaMemsetAsync(d_counters2, 0, 2 * sizeof(uint64_t), st));
    if (staged_tiles_out) *staged_tiles_out = 0;
    if (n < W) return RS_OK;
    WorkLayout wl = rs_work_layout(n, hit_capacity);
    if (!d_work || work_bytes < wl.total) { rs_set_error("workspace too small: need %lld bytes", (long long)wl.total); return RS_ERR_WORKSPACE; }

    // Combined mode: a window's profile rows only matter where its sequence score passes too (combine() is an AND,
    // rnascan.py:416-434) -- a fraction of a per cent of the windows at typical thresholds -- so the sequence scan
    // runs first and the rows of its hits alone are read (DESIGN.md 3.1).  Batched and staged callers keep the
    // structure-first kernels.
    if (mode == RS_MODE_AND && W <= RS_KMER_WMAX && !staged_tiles_out && !d_counts8 && !d_out_base && !d_hit_motif)
        return rs_scan_fused_seqfirst(d_codes, d_profile, profile_dtype, n, seq_table, struct_table, W, threshold,
                                      hit_capacity, d_hit_pos, d_hit_seq, d_hit_struct, nullptr, d_counters2, d_work,
                                      st);

    ProfileParams prm = {};
    prm.codes = d_codes; prm.profile = d_profile; prm.n = n; prm.padded = rs_padded_count(n);
    prm.threshold = threshold; prm.mode = mode; prm.W = W; prm.dense = 0;
    uint8_t *wk = (uint8_t *)d_work;
    prm.st.pos = (int64_t *)(wk + wl.off_pos);
    prm.st.seq = d_hit_seq ? (float *)(wk + wl.off_seq) : nullptr;
    prm.st.str = (double *)(wk + wl.off_str);
    prm.st.tile_seg = (ulonglong2 *)(wk + wl.off_seg);
    prm.st.counters = (unsigned long long *)d_counters2;
    prm.st.capacity = hit_capacity;

    bool fast = profile_dtype == RS_F32 && W <= RS_FAST_W &&
                build_filter(prm, struct_table, W, threshold, profile_absrow_max, 1.0, 0.0, false);
    for (int k = 0; k < W * RS_CHANNELS; k++) prm.sd[k] = struct_table[k];
    if (seq_table) for (int k = 0; k < W * 4; k++) prm.qd[k] = seq_table[k];

    int64_t n_tiles;
    if (d_counts8 && !fast) {
        rs_set_error("in-kernel background counts need the fp32 filter path (float32 profile, W <= %d, finite tables)", RS_FAST_W);
        return RS_ERR_INVALID;
    }
    if (fast) {
        n_tiles = (n + FT_TILE - 1) / FT_TILE;
        prm.n_tiles = n_tiles;
        prm.count_on = d_counts8 ? 1 : 0; prm.counts8 = (unsigned long long *)d_counts8; prm.count_rows = n;
        rc = FilterDispatch<RS_FAST_W>::run(W, prm, st);
    } else {
        n_tiles = (n + EX_TILE - 1) / EX_TILE;
        prm.n_tiles = n_tiles;
        rc = profile_dtype == RS_F32 ? launch_exact<float>(prm, st) : launch_exact<double>(prm, st);
    }
    if (rc) return rc;
    if (staged_tiles_out) {            // rs_scan_fused_candidates: leave the hits staged per tile
        *staged_tiles_out = n_tiles;
        return RS_OK;
    }
    OrderDest od = {d_hit_pos, d_hit_seq, d_hit_struct, d_out_base, d_hit_motif, motif_id};
    return rs_order_hits(prm.st, n_tiles, od, wk + wl.off_scan, st);
}

// ---- the combined scan in two halves, so that the half that needs the data's background can wait for it
extern "C" int rs_scan_fused_candidates(const uint8_t *d_codes, const void *d_profile, int profile_dtype, int64_t n,
                                        const double *struct_table, int W, double threshold,
                                        double profile_absrow_max, int64_t hit_capacity, uint64_t *d_cand_counters2,
                                        void *d_work, int64_t work_bytes, int64_t *staged_tiles, void *stream)
{
    if (!staged_tiles) { rs_set_error("rs_scan_fused_candidates: null staged_tiles"); return RS_ERR_INVALID; }
    return scan_fused_impl(d_codes, d_profile, profile_dtype, n, nullptr, struct_table, W, threshold,
                           profile_absrow_max, RS_MODE_STRUCT, hit_capacity, nullptr, nullptr, nullptr,
                           d_cand_counters2, d_work, work_bytes, stream, nullptr, nullptr, 0, staged_tiles);
}

// The same, taking the sequence's background counts in the same pass: d_counts8[0..3] += letters A,C,G,U of the
// stream (not zeroed here).  Needs the fp32 filter path (else RS_ERR_INVALID: use rs_hist_rna beside the scan).
extern "C" int rs_scan_fused_candidates_counting(const uint8_t *d_codes, const void *d_profile, int profile_dtype,
                                                 int64_t n, const double *struct_table, int W, double threshold,
                                                 double profile_absrow_max, int64_t hit_capacity,
                                                 uint64_t *d_cand_counters2, uint64_t *d_counts8, void *d_work,
                                                 int64_t work_bytes, int64_t *staged_tiles, void *stream)
{
    if (!staged_tiles || !d_counts8) { rs_set_error("rs_scan_fused_candidates_counting: null argument"); return RS_ERR_INVALID; }
    if (n < W) { rs_set_error("rs_scan_fused_candidates_counting: stream shorter than the motif (count with rs_hist_rna)"); return RS_ERR_INVALID; }
    return scan_fused_impl(d_codes, d_profile, profile_dtype, n, nullptr, struct_table, W, threshold,
                           profile_absrow_max, RS_MODE_STRUCT, hit_capacity, nullptr, nullptr, nullptr,
                           d_cand_counters2, d_work, work_bytes, stream, nullptr, nullptr, 0, staged_tiles, d_counts8);
}

extern "C" int rs_scan_fused_resolve(const uint8_t *d_codes, int64_t n, const double *seq_table, int W,
                                     double threshold, int64_t staged_tiles, int64_t hit_capacity,
                                     int64_t *d_hit_pos, float *d_hit_seq, double *d_hit_struct,
                                     uint64_t *d_counters2, void *d_work, int64_t work_bytes, void *stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    if (!d_codes || !seq_table || !d_counters2 || n < 0 || staged_tiles < 0) {
        rs_set_error("rs_scan_fused_resolve: bad argument"); return RS_ERR_INVALID;
    }
    if (W < 1 || W > RS_MAX_W) { rs_set_error("motif width %d outside [1, %d]", W, RS_MAX_W); return RS_ERR_INVALID; }
    if (threshold != threshold) { rs_set_error("threshold is NaN"); return RS_ERR_INVALID; }
    if (hit_capacity < 0 || (hit_capacity > 0 && (!d_hit_pos || !d_hit_seq || !d_hit_struct))) {
        rs_set_error("bad hit buffers"); return RS_ERR_INVALID;
    }
    WorkLayout wl = rs_work_layout(n, hit_capacity);
    if (!d_work || work_bytes < wl.total) { rs_set_error("workspace too small: need %lld bytes", (long long)wl.total); return RS_ERR_WORKSPACE; }
    if (staged_tiles > n / RS_MIN_TILE + 16) { rs_set_error("staged_tiles does not belong to this stream length"); return RS_ERR_INVALID; }
    RS_CUDA(cudaMemsetAsync(d_counters2, 0, 2 * sizeof(uint64_t), st));
    uint8_t *wk = (uint8_t *)d_work;
    HitStage hs = {};
    hs.pos = (int64_t *)(wk + wl.off_pos);
    hs.seq = (float *)(wk + wl.off_seq);
    hs.str = (double *)(wk + wl.off_str);
    hs.tile_seg = (ulonglong2 *)(wk + wl.off_seg);
    hs.counters = (unsigned long long *)d_counters2;
    hs.capacity = hit_capacity;
    OrderDest od = {d_hit_pos, d_hit_seq, d_hit_struct, nullptr, nullptr, 0};
    return rs_order_hits_seq_refined(hs, staged_tiles, od, wk + wl.off_scan, st, d_codes, n, seq_table, W, threshold,
                                     (unsigned long long *)d_counters2);
}

extern "C" int rs_scan_fused(const uint8_t *d_codes, const void *d_profile, int profile_dtype, int64_t n,
                             const double *seq_table, const double *struct_table, int W, double threshold,
                             double profile_absrow_max, int mode, int64_t hit_capacity, int64_t *d_hit_pos,
                             float *d_hit_seq, double *d_hit_struct, uint64_t *d_counters2, void *d_work,
                             int64_t work_bytes, void *stream)
{
    return scan_fused_impl(d_codes, d_profile, profile_dtype, n, seq_table, struct_table, W, threshold,
                           profile_absrow_max, mode, hit_capacity, d_hit_pos, d_hit_seq, d_hit_struct, d_counters2,
                           d_work, work_bytes, stream, nullptr, nullptr, 0);
}

extern "C" int rs_scan_fused_seqfirst_counted(const uint8_t *d_codes, const void *d_profile, int profile_dtype,
                                              int64_t n, const double *seq_table, const double *struct_table, int W,
                                              double threshold, int64_t hit_capacity, int64_t *d_hit_pos,
                                              float *d_hit_seq, double *d_hit_struct, uint64_t *d_cand_counters2,
                                              uint64_t *d_counters2, void *d_work, int64_t work_bytes, void *stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    int rc = check_common(d_profile, profile_dtype, n, struct_table, W);
    if (rc) return rc;
    if (!d_codes || ((uintptr_t)d_codes & 15)) { rs_set_error("codes pointer null or not 16-byte aligned"); return RS_ERR_INVALID; }
    if (W > RS_KMER_WMAX) { rs_set_error("the sequence-first scan covers motif widths 1..%d (got %d)", RS_KMER_WMAX, W); return RS_ERR_INVALID; }
    if (!seq_table || !d_cand_counters2 || !d_counters2 || hit_capacity < 0 ||
        (hit_capacity > 0 && (!d_hit_pos || !d_hit_seq || !d_hit_struct))) {
        rs_set_error("rs_scan_fused_seqfirst_counted: bad argument"); return RS_ERR_INVALID;
    }
    if ((const void *)d_cand_counters2 == (const void *)d_counters2) { rs_set_error("d_cand_counters2 and d_counters2 must differ"); return RS_ERR_INVALID; }
    if (threshold != threshold) { rs_set_error("threshold is NaN"); return RS_ERR_INVALID; }
    if (n < W) {
        RS_CUDA(cudaMemsetAsync(d_counters2, 0, 2 * sizeof(uint64_t), st));
        RS_CUDA(cudaMemsetAsync(d_cand_counters2, 0, 2 * sizeof(uint64_t), st));
        return RS_OK;
    }
    WorkLayout wl = rs_work_layout(n, hit_capacity);
    if (!d_work || work_bytes < wl.total) { rs_set_error("workspace too small: need %lld bytes", (long long)wl.total); return RS_ERR_WORKSPACE; }
    return rs_scan_fused_seqfirst(d_codes, d_profile, profile_dtype, n, seq_table, struct_table, W, threshold,
                                  hit_capacity, d_hit_pos, d_hit_seq, d_hit_struct, d_cand_counters2, d_counters2,
                                  d_work, st);
}

// ---- filter + gather + resolve: candidate positions only; the exact rows live on the host (resolve.cu)
extern "C" int64_t rs_filter_workspace_bytes(int64_t n, int64_t cand_capacity)
{
    return rs_filter_layout(n, cand_capacity).total;
}

extern "C" int rs_filter_profile(const uint8_t *d_codes, const void *d_rows, int row_format, double q8_scale,
                                 int64_t n, const double *seq_table, const double *struct_table, int W,
                                 double threshold, double absrow_max, int64_t pos_base, int64_t count_rows,
                                 uint64_t *d_counts8, int64_t cand_capacity, int64_t *d_cand_pos,
                                 uint64_t *d_cand_sym, uint64_t *d_counters2, void *d_work, int64_t work_bytes,
                                 void *stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    if (row_format != RS_ROWS_F32 && row_format != RS_ROWS_F32_SHADOW && row_format != RS_ROWS_Q8 &&
        row_format != RS_ROWS_Q4) {
        rs_set_error("row_format must be RS_ROWS_F32, RS_ROWS_F32_SHADOW, RS_ROWS_Q8 or RS_ROWS_Q4"); return RS_ERR_INVALID;
    }
    const bool q4 = row_format == RS_ROWS_Q4;
    const bool q8 = row_format == RS_ROWS_Q8 || q4;          // "quantised": the rows carry the symbols
    if (d_cand_sym && !q4) { rs_set_error("candidate symbols come with RS_ROWS_Q4 only"); return RS_ERR_INVALID; }
    if (!d_rows || ((uintptr_t)d_rows & 15) || !struct_table) { rs_set_error("rows pointer null or not 16-byte aligned, or null table"); return RS_ERR_INVALID; }
    if (!q8 && (!d_codes || ((uintptr_t)d_codes & 15))) { rs_set_error("codes pointer null or not 16-byte aligned"); return RS_ERR_INVALID; }
    if (W < 1 || W > RS_FAST_W) { rs_set_error("filter scans need 1 <= W <= %d", RS_FAST_W); return RS_ERR_INVALID; }
    if (n < 0 || cand_capacity < 0 || !d_counters2 || (cand_capacity > 0 && !d_cand_pos)) { rs_set_error("bad candidate buffers"); return RS_ERR_INVALID; }
    if (threshold != threshold) { rs_set_error("threshold is NaN"); return RS_ERR_INVALID; }
    if (d_counts8 && !q8) { rs_set_error("background counts are taken in the quantised scan only (use rs_hist_rna)"); return RS_ERR_INVALID; }
    if (q8 && !(q8_scale > 0.0 && isfinite(q8_scale))) { rs_set_error("q8_scale must be positive and finite"); return RS_ERR_INVALID; }
    RS_CUDA(cudaMemsetAsync(d_counters2, 0, 2 * sizeof(uint64_t), st));
    if (n == 0 || (n < W && !d_counts8)) return RS_OK;
    const FilterWork wl = rs_filter_layout(n, cand_capacity);
    if (!d_work || work_bytes < wl.total) { rs_set_error("workspace too small: need %lld bytes", (long long)wl.total); return RS_ERR_WORKSPACE; }

    ProfileParams prm = {};
    prm.codes = d_codes; prm.profile = d_rows; prm.n = n; prm.padded = rs_padded_count(n);
    prm.threshold = threshold; prm.mode = seq_table ? RS_MODE_AND : RS_MODE_STRUCT; prm.W = W;
    prm.defer = 1; prm.pos_base = pos_base;
    prm.count_on = d_counts8 ? 1 : 0; prm.counts8 = (unsigned long long *)d_counts8;
    prm.count_rows = d_counts8 ? (count_rows < n ? count_rows : n) : 0;
    uint8_t *wk = (uint8_t *)d_work;
    prm.st.pos = (int64_t *)(wk + wl.off_pos);
    prm.st.str = d_cand_sym ? (double *)(wk + wl.off_sym) : nullptr;
    prm.st.tile_seg = (ulonglong2 *)(wk + wl.off_seg);
    prm.st.counters = (unsigned long long *)d_counters2;
    prm.st.capacity = cand_capacity;
    const double vs = q4 ? q8_scale / 15.0 : (q8 ? q8_scale / 255.0 : 1.0);
    if (!build_filter(prm, struct_table, W, threshold, absrow_max, vs, q4 ? vs : (q8 ? 0.5 * vs : 0.0),
                      row_format == RS_ROWS_F32_SHADOW, q4)) {
        rs_set_error("the fp32 filter does not apply (non-finite threshold, table or row bound): use the exact scan");
        return RS_ERR_INVALID;
    }
    if (seq_table) for (int k = 0; k < W * 4; k++) prm.qd[k] = seq_table[k];
    prm.n_tiles = (n + FT_TILE - 1) / FT_TILE;
    int rc = q4 ? rs_filter_q4_launch(prm, W, st)
                : (q8 ? rs_filter_q8_launch(prm, W, st) : FilterDispatch<RS_FAST_W>::run(W, prm, st));
    if (rc) return rc;
    OrderDest od = {d_cand_pos, nullptr, (double *)d_cand_sym, nullptr, nullptr, 0};
    return rs_order_hits(prm.st, prm.n_tiles, od, wk + wl.off_scan, st);
}

// ------------------------------------------------------------------------------------------------
// Batched many-PFM scan, CUDA-core path: one fused scan per motif over the same resident
// streams; every motif's ordered hits are appended behind the previous motif's.
static thread_local int g_batched_path = 0;       // 0 auto, 1 CUDA-core loop, 2 tensor cores (error if not applicable)
static thread_local int g_batched_last = 0;       // path this thread's last rs_scan_batched call took (1 or 2)
extern "C" int rs_last_batched_path(void) { return g_batched_last; }
extern "C" int rs_set_batched_path(int path)
{
    if (path < 0 || path > 2) { rs_set_error("rs_set_batched_path: 0, 1 or 2"); return RS_ERR_INVALID; }
    g_batched_path = path;
    return RS_OK;
}
extern "C" int64_t rs_scan_batched_workspace_bytes(int64_t n, int n_motifs, int table_stride_rows,
                                                   int64_t hit_capacity)
{
    const int64_t a = rs_work_layout(n, hit_capacity).total;
    const int64_t b = rs_batched_tc_work_bytes(n, n_motifs, table_stride_rows, hit_capacity);
    return a > b ? a : b;
}

__global__ void batched_base_kernel(unsigned long long *bases, const unsigned long long *counters2, int m)
{
    bases[m + 1] = bases[m] + counters2[2 * m];
}

static int scan_batched_impl(const uint8_t *d_codes, const void *d_profile, int profile_dtype, int64_t n,
                               int n_motifs, const int *widths, const double *seq_tables,
                               const double *struct_tables, int table_stride_rows, double threshold,
                               double profile_absrow_max, int mode, int64_t hit_capacity, int32_t *d_hit_motif,
                               int64_t *d_hit_pos, float *d_hit_seq, double *d_hit_struct,
                               uint64_t *d_motif_counters2, uint64_t *d_bases, void *d_work, int64_t work_bytes,
                               void *stream, const double *d_exact64)
{
    cudaStream_t st = (cudaStream_t)stream;
    if (n_motifs < 1 || !widths || !struct_tables || !d_motif_counters2 || !d_bases) {
        rs_set_error("rs_scan_batched: bad argument"); return RS_ERR_INVALID;
    }
    if (table_stride_rows < 1 || table_stride_rows > RS_MAX_W) { rs_set_error("bad table_stride_rows"); return RS_ERR_INVALID; }
    if (mode == RS_MODE_AND && !seq_tables) { rs_set_error("RS_MODE_AND needs sequence tables"); return RS_ERR_INVALID; }
    if (hit_capacity > 0 && !d_hit_motif) { rs_set_error("null d_hit_motif"); return RS_ERR_INVALID; }
    for (int m = 0; m < n_motifs; m++)
        if (widths[m] < 1 || widths[m] > table_stride_rows) { rs_set_error("motif %d: width outside [1, stride]", m); return RS_ERR_INVALID; }
    // Tensor-core path (batched_tc.cu): worth it from a few dozen motifs on; needs fp32 profiles
    // and W <= 12.  It answers -1 when it does not apply, then the per-motif loop below runs.
    if (g_batched_path != 1 && profile_dtype == RS_F32 && (n_motifs >= 32 || g_batched_path == 2) && n >= 1) {
        if (!d_codes || !d_profile || ((uintptr_t)d_codes & 15) || ((uintptr_t)d_profile & 15)) {
            rs_set_error("codes/profile pointer null or not 16-byte aligned"); return RS_ERR_INVALID;
        }
        int rc = rs_scan_batched_tc(d_codes, d_profile, n, n_motifs, widths, seq_tables, struct_tables,
                                    table_stride_rows, threshold, profile_absrow_max, mode, hit_capacity,
                                    d_hit_motif, d_hit_pos, d_hit_seq, d_hit_struct, d_motif_counters2, d_bases,
                                    d_work, work_bytes, st, d_exact64);
        if (rc >= 0) { g_batched_last = 2; return rc; }
        if (g_batched_path == 2) return RS_ERR_INVALID;      // rs_last_error() says why it does not apply
    }
    g_batched_last = 1;
    RS_CUDA(cudaMemsetAsync(d_bases, 0, sizeof(uint64_t) * (size_t)(n_motifs + 1), st));
    RS_CUDA(cudaMemsetAsync(d_motif_counters2, 0, sizeof(uint64_t) * 2 * (size_t)n_motifs, st));
    for (int m = 0; m < n_motifs; m++) {
        const double *ts = seq_tables ? seq_tables + (size_t)m * table_stride_rows * 4 : nullptr;
        const double *tq = struct_tables + (size_t)m * table_stride_rows * RS_CHANNELS;
        int rc = scan_fused_impl(d_codes, d_exact64 ? (const void *)d_exact64 : d_profile,
                                 d_exact64 ? RS_F64 : profile_dtype, n, ts, tq, widths[m], threshold,
                                 profile_absrow_max, mode, hit_capacity, d_hit_pos, d_hit_seq, d_hit_struct,
                                 d_motif_counters2 + 2 * m, d_work, work_bytes, stream,
                                 (const unsigned long long *)d_bases + m, d_hit_motif, m);
        if (rc) return rc;
        batched_base_kernel<<<1, 1, 0, st>>>((unsigned long long *)d_bases,
                                             (const unsigned long long *)d_motif_counters2, m);
        RS_CUDA(cudaGetLastError());
    }
    return RS_OK;
}

extern "C" int rs_scan_batched(const uint8_t *d_codes, const void *d_profile, int profile_dtype, int64_t n,
                               int n_motifs, const int *widths, const double *seq_tables,
                               const double *struct_tables, int table_stride_rows, double threshold,
                               double profile_absrow_max, int mode, int64_t hit_capacity, int32_t *d_hit_motif,
                               int64_t *d_hit_pos, float *d_hit_seq, double *d_hit_struct,
                               uint64_t *d_motif_counters2, uint64_t *d_bases, void *d_work, int64_t work_bytes,
                               void *stream)
{
    return scan_batched_impl(d_codes, d_profile, profile_dtype, n, n_motifs, widths, seq_tables, struct_tables,
                             table_stride_rows, threshold, profile_absrow_max, mode, hit_capacity, d_hit_motif,
                             d_hit_pos, d_hit_seq, d_hit_struct, d_motif_counters2, d_bases, d_work, work_bytes, stream,
                             nullptr);
}

// float64 rows (what the CLI parses) with their float32 shadow: the tensor-core filter reads the shadow, every
// candidate is re-scored from the float64 rows -- results identical to rs_scan_batched on the float64 rows.
extern "C" int rs_scan_batched_shadow(const uint8_t *d_codes, const float *d_shadow_f32, const double *d_exact_f64,
                                      int64_t n, int n_motifs, const int *widths, const double *seq_tables,
                                      const double *struct_tables, int table_stride_rows, double threshold,
                                      double profile_absrow_max, int mode, int64_t hit_capacity,
                                      int32_t *d_hit_motif, int64_t *d_hit_pos, float *d_hit_seq,
                                      double *d_hit_struct, uint64_t *d_motif_counters2, uint64_t *d_bases,
                                      void *d_work, int64_t work_bytes, void *stream)
{
    if (!d_shadow_f32 || !d_exact_f64 || ((uintptr_t)d_exact_f64 & 15)) {
        rs_set_error("rs_scan_batched_shadow: null or misaligned rows"); return RS_ERR_INVALID;
    }
    return scan_batched_impl(d_codes, d_shadow_f32, RS_F32, n, n_motifs, widths, seq_tables, struct_tables,
                             table_stride_rows, threshold, profile_absrow_max, mode, hit_capacity, d_hit_motif,
                             d_hit_pos, d_hit_seq, d_hit_struct, d_motif_counters2, d_bases, d_work, work_bytes, stream,
                             d_exact_f64);
}
