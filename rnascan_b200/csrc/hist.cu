// Background letter counts over the symbol stream (exact integers).
//
// Replaces the per-letter Seq.count() passes of /root/reference/rnascan/rnascan.py:450-453.
// A symbol is counted in bin (code & 7) iff bit 3 of its code is clear (separators 0xFF,
// ambiguous bases 0x0C/0x0F and lower-case structure letters are not counted -- SURVEY.md H11).
//
// HBM-bound at 1 B/symbol: each thread streams 16-byte vectors.  Per 32-bit word the validity plane
// v (bit 0 of every counted byte) and the masked index planes b0, 2*b1, 4*b2 (each left at its own bit
// position: w & (v << s), no shift of the data) are formed with a handful of logic operations, and ALL
// the summing is done by dp4a -- dot products with 0x01010101 for the plane sums, dot products of two
// planes for the pair sums (the byte-wise multiply is free there) -- into 32-bit accumulators.  That
// moves the additions off the ALU pipe, which round 1's packed byte counters kept 60 % busy (ncu), and
// removes the periodic flushing of those counters.  Bin counts follow by inclusion-exclusion over the
// subset sums (v, b0, b1, b2, b0b1, b0b2, b1b2, b0b1b2) once per thread, then warp shuffles -> shared
// memory -> ONE global atomic per bin per CTA.
#include "common.cuh"

#define HI_THREADS 256
#define HI_UNROLL 4               // independent 16-byte loads in flight per thread (2 and 8 measured: no better;
                                  // so were 8 CTAs per SM at 32 registers and fewer, fatter CTAs)

// PLANES = 3: any stream (letter index in bits 0-2).  PLANES = 2: nucleotide streams, whose
// counted symbols are 0..3 (bit 2 never set with bit 3 clear): half the arithmetic.
// acc[T]: subset sum T (bit s of T set <=> plane s in the product) SCALED by scale(T) = prod 2^s.
template <int PLANES>
__device__ __forceinline__ void hist_word(unsigned w, unsigned (&acc)[1 << PLANES])
{
    const unsigned ONES = 0x01010101u;
    const unsigned v = ~(w >> 3) & ONES;                  // counted: bit 3 clear
    const unsigned b0 = w & v;
    const unsigned b1 = w & (v * 2u);                     // bit 1 of every counted byte, value 2
    acc[0] = __dp4a(v, ONES, acc[0]);
    acc[1] = __dp4a(b0, ONES, acc[1]);
    acc[2] = __dp4a(b1, ONES, acc[2]);                    // 2 * S1
    acc[3] = __dp4a(b0, b1, acc[3]);                      // 2 * S01
    if (PLANES == 3) {
        const unsigned b2 = w & (v * 4u);                 // value 4
        const unsigned b01 = b0 & (b1 >> 1);
        acc[4] = __dp4a(b2, ONES, acc[4]);                // 4 * S2
        acc[5] = __dp4a(b0, b2, acc[5]);                  // 4 * S02
        acc[6] = __dp4a(b1, b2, acc[6]);                  // 8 * S12
        acc[7] = __dp4a(b01, b2, acc[7]);                 // 4 * S012
    }
}

template <int PLANES, int UNROLL = HI_UNROLL>
__global__ void __launch_bounds__(HI_THREADS) hist_kernel(const uint8_t *__restrict__ codes, int64_t n,
                                                          unsigned long long *__restrict__ counts)
{
    constexpr int NS = 1 << PLANES;              // subset sums: index bit s set <=> plane s in the product
    unsigned long long tot[NS];
#pragma unroll
    for (int k = 0; k < NS; k++) tot[k] = 0;

    const int64_t nvec = n / 16;
    const uint4 *v = reinterpret_cast<const uint4 *>(codes);
    const int64_t gstride = (int64_t)gridDim.x * blockDim.x;
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;

    while (i < nvec) {
        // 32-bit accumulators: a word adds at most 4 * 16 to one of them; flushed every 2^20 vectors
        unsigned acc[NS];
#pragma unroll
        for (int k = 0; k < NS; k++) acc[k] = 0;
        for (int rep = 0; rep < (1 << 20) / UNROLL && i < nvec; rep++) {
            uint4 q[UNROLL];
#pragma unroll
            for (int u = 0; u < UNROLL; u++) {
                const int64_t j = i + u * gstride;
                q[u] = j < nvec ? __ldg(v + j) : make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
            }
            i += UNROLL * gstride;
#pragma unroll
            for (int u = 0; u < UNROLL; u++) {
                hist_word<PLANES>(q[u].x, acc);
                hist_word<PLANES>(q[u].y, acc);
                hist_word<PLANES>(q[u].z, acc);
                hist_word<PLANES>(q[u].w, acc);
            }
        }
#pragma unroll
        for (int k = 0; k < NS; k++) tot[k] += acc[k];
    }
    // undo the scaling of the plane sums (see hist_word)
    tot[2] >>= 1; tot[3] >>= 1;
    if (PLANES == 3) { tot[4] >>= 2; tot[5] >>= 2; tot[6] >>= 3; tot[7] >>= 2; }
    // tail symbols (n % 16) by the first threads of block 0
    if (blockIdx.x == 0 && threadIdx.x < (n & 15)) {
        const unsigned c = codes[nvec * 16 + threadIdx.x];
        if (!(c & 8)) {
            const unsigned b[3] = {c & 1, (c >> 1) & 1, (c >> 2) & 1};
#pragma unroll
            for (int T = 0; T < NS; T++) {
                unsigned p = 1;
#pragma unroll
                for (int s = 0; s < PLANES; s++)
                    if (T & (1 << s)) p &= b[s];
                tot[T] += p;
            }
        }
    }
    // inclusion-exclusion: count of index k = sum over supersets T of bits(k) of (-1)^{|T|-|k|} S[T]
    long long cnt[NS];
#pragma unroll
    for (int k = 0; k < NS; k++) {
        long long c = 0;
#pragma unroll
        for (int T = 0; T < NS; T++)
            if ((T & k) == k) c += (__popc(T ^ k) & 1) ? -(long long)tot[T] : (long long)tot[T];
        cnt[k] = c;
    }
    __shared__ unsigned long long s_bins[8];
    if (threadIdx.x < 8) s_bins[threadIdx.x] = 0;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < NS; k++) {
        long long c = cnt[k];
        for (int d = 16; d; d >>= 1) c += __shfl_xor_sync(0xffffffffu, c, d);
        if ((threadIdx.x & 31) == 0 && c) atomicAdd(&s_bins[k], (unsigned long long)c);
    }
    __syncthreads();
    if (threadIdx.x < NS && s_bins[threadIdx.x]) atomicAdd(&counts[threadIdx.x], s_bins[threadIdx.x]);
}

template <int PLANES>
static int hist_launch(const uint8_t *d_codes, int64_t n, uint64_t *d_counts8, void *stream)
{
    if (!d_codes || !d_counts8 || n < 0) { rs_set_error("rs_hist: bad argument"); return RS_ERR_INVALID; }
    if ((uintptr_t)d_codes & 15) { rs_set_error("codes pointer must be 16-byte aligned"); return RS_ERR_INVALID; }
    if (n == 0) return RS_OK;
    int64_t blocks = (n / 64 + HI_THREADS - 1) / HI_THREADS;
    // exactly one resident wave: the kernel is a grid-stride loop, a partial second wave is pure tail
    static int per_sm[RS_MAX_DEVICES] = {};
    const int dev = rs_current_device();
    if (!per_sm[dev]) {
        int v = 0;
        RS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, hist_kernel<PLANES, HI_UNROLL>, HI_THREADS, 0));
        per_sm[dev] = v > 0 ? v : 4;
    }
    int64_t cap = (int64_t)rs_sm_count() * per_sm[dev];
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    hist_kernel<PLANES><<<(unsigned)blocks, HI_THREADS, 0, (cudaStream_t)stream>>>(d_codes, n,
                                                                                 (unsigned long long *)d_counts8);
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

extern "C" int rs_hist_rna(const uint8_t *d_codes, int64_t n, uint64_t *d_counts8, void *stream)
{
    return hist_launch<2>(d_codes, n, d_counts8, stream);
}

extern "C" int rs_hist(const uint8_t *d_codes, int64_t n, uint64_t *d_counts8, void *stream)
{
    return hist_launch<3>(d_codes, n, d_counts8, stream);
}

// ---- alphabet layout (rs_host_encode_alpha): 32 bins, bin = code & 31, counted iff bit 5 is clear ----------------
// Replaces the same Seq.count() loop (rnascan.py:450-453) for alphabets of up to 31 letters.  Lower-case letters
// (bit 5) and separators (0xFF) are not counted; bin 31 collects the layout's "other" symbol 0x1F, which is no letter.
// Each lane owns one column of its warp's 32 x 32 counter block in shared memory (no bank conflicts, no contention):
// the increments are fire-and-forget shared atomics, so consecutive symbols of one lane do not wait for each other.
// A lane counts at most n / (threads of the grid) symbols: 32-bit counters hold any stream that fits on a device.
__global__ void __launch_bounds__(HI_THREADS) hist32_kernel(const uint8_t *__restrict__ codes, int64_t n,
                                                            unsigned long long *__restrict__ counts)
{
    __shared__ unsigned s_cnt[HI_THREADS / 32][32][32];       // [warp][bin][lane]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned (*mine)[32] = s_cnt[warp];
#pragma unroll
    for (int b = 0; b < 32; b++) mine[b][lane] = 0;
    auto count_word = [&](unsigned w) {
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const unsigned c = (w >> (8 * k)) & 0xFFu;
            if (!(c & 0x20u)) atomicAdd(&mine[c & 31u][lane], 1u);
        }
    };
    const int64_t nvec = n / 16;
    const uint4 *v = reinterpret_cast<const uint4 *>(codes);
    const int64_t gstride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nvec; i += HI_UNROLL * gstride) {
        uint4 q[HI_UNROLL];
#pragma unroll
        for (int u = 0; u < HI_UNROLL; u++) {
            const int64_t j = i + u * gstride;
            q[u] = j < nvec ? __ldg(v + j) : make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
        }
#pragma unroll
        for (int u = 0; u < HI_UNROLL; u++) {
            count_word(q[u].x); count_word(q[u].y); count_word(q[u].z); count_word(q[u].w);
        }
    }
    if (blockIdx.x == 0 && threadIdx.x < (n & 15)) {           // tail symbols (n % 16)
        const unsigned c = codes[nvec * 16 + threadIdx.x];
        if (!(c & 0x20u)) atomicAdd(&mine[c & 31u][lane], 1u);
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        unsigned long long sum = 0;
        for (int w = 0; w < HI_THREADS / 32; w++)
            for (int l = 0; l < 32; l++) sum += s_cnt[w][threadIdx.x][(l + threadIdx.x) & 31];
        if (sum) atomicAdd(&counts[threadIdx.x], sum);
    }
}

extern "C" int rs_hist_alpha(const uint8_t *d_codes, int64_t n, uint64_t *d_counts32, void *stream)
{
    if (!d_codes || !d_counts32 || n < 0) { rs_set_error("rs_hist_alpha: bad argument"); return RS_ERR_INVALID; }
    if ((uintptr_t)d_codes & 15) { rs_set_error("codes pointer must be 16-byte aligned"); return RS_ERR_INVALID; }
    if (n == 0) return RS_OK;
    int64_t blocks = (n / 64 + HI_THREADS - 1) / HI_THREADS;
    static int per_sm[RS_MAX_DEVICES] = {};                   // one resident wave, as hist_launch
    const int dev = rs_current_device();
    if (!per_sm[dev]) {
        int v = 0;
        RS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, hist32_kernel, HI_THREADS, 0));
        per_sm[dev] = v > 0 ? v : 4;
    }
    const int64_t cap = (int64_t)rs_sm_count() * per_sm[dev];
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    hist32_kernel<<<(unsigned)blocks, HI_THREADS, 0, (cudaStream_t)stream>>>(d_codes, n,
                                                                           (unsigned long long *)d_counts32);
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}
