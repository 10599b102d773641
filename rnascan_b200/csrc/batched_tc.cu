// Batched many-PFM scan on the 5th-generation tensor cores (tcgen05 + TMEM) -- BASELINE config 5.
//
// For M motifs the averaged-profile score is a dense contraction
//     score[i, m] = sum_{j < 12} sum_{c < 8} P[i + j][c] * S_m[j][c]           (rows j >= W_m are zero)
// i.e. a (positions x 96) * (96 x M) GEMM whose A operand is the im2col of the profile stream.
// The reference evaluates it one window, one motif, one row at a time (rnascan.py:302-307).
//
// Implicit im2col without any data expansion: profile rows are staged in shared memory as
// 8 bf16 = 16 bytes each (7 channels + a constant 1.0 that carries the per-motif threshold as a
// bias), so 8 consecutive rows ARE one canonical no-swizzle K-major core matrix (8 x 16 B).  The
// A-tile of tcgen05.mma for window rows j, j+1 is then just the staged rows at byte offset 16*j with
// stride-byte-offset 128 (8 positions down) and leading-byte-offset 16 (one row over): the twelve
// shifted views of the same 2.2 KB overlap in shared memory, the tensor core only sees addresses.
//
// The GEMM is a FILTER, never the answer: S is rounded UP to bf16, profile values to nearest, the
// threshold is lowered by a rigorous bound on the bf16/accumulation error, and every (position,
// motif) whose accumulator is > 0 becomes a candidate that batched_rescore_kernel re-scores in
// fp64 in the reference's exact operation order (together with the sequence PSSM).  Hits are
// sorted by (motif, position) and their scores recomputed exactly, so results are bit-identical
// to rs_scan_fused run once per motif.
//
// Warp roles (512 threads, 1 CTA/SM, persistent over 128-position tiles):
//   warp 0      TMA producer: bulk async copies of fp32 profile rows into a 4-stage ring
//   warp 1      MMA issuer: one lane issues 6 x tcgen05.mma (M128 N256 K16, bf16 -> fp32 in TMEM)
//   warp 2      TMEM allocator (512 columns = two 128x256 fp32 accumulators)
//   warps 4-7, 12-15  epilogue: two warps per TMEM lane quadrant, 128 motif columns each:
//               tcgen05.ld, sign-bit mask of the 32 accumulators per load (one funnel shift each),
//               candidates staged per warp in shared memory, flushed with one atomic per ~1000
//   warps 8-11  converters: fp32 rows -> bf16 x 8 rows (the A operand), fence.proxy.async; in RS_MODE_AND also
//               the SEQUENCE MASK of every position of the tile (one thread per position): the 8-mer the window
//               starts with indexes a 65536 x 256-bit table (kmer_mask_build_kernel: which motifs' sequence score can
//               pass), restricted to the motifs no wider than the distance to the first invalid symbol; 32 B per
//               position into an 8-stage shared-memory ring that the epilogue ANDs into its sign masks, so only
//               (position, motif) pairs that can be combined hits are ever staged
#include <cuda_bf16.h>
#include <string.h>
#include <vector>
#include "common.cuh"

#define TC_N        256                 // motifs per GEMM (UMMA N)
#define TC_WMAX     12                  // widest motif on this path
#define TC_M        128                 // positions per tile (UMMA M)
#define TC_ROWS     (TC_M + TC_WMAX - 1)             // 139 staged rows
#define TC_STAGES   4
#define TC_RAW_BYTES  3904              // ceil16(139 * 28)
#define TC_A_BYTES    2304              // ceil128(139 * 16)
#define TC_B_BYTES    (TC_WMAX * TC_N * 16)          // 49152
#define TC_THREADS  512
#define TC_CBUF     1024                // staged candidate keys per epilogue warp (>= 32 lanes x 32 motifs)
#define TC_MASK_STAGES 8                // sequence masks of 8 tiles in flight: the converters run at most 4 tiles ahead
                                        // of the MMAs, the MMAs 2 ahead of the epilogue, so a stage is long read when
                                        // it is written again

struct TcParams {
    const float   *profile;             // fp32 [padded][7]
    const uint16_t *bmat;               // bf16 bits [12][256][8] (K-major core-matrix order)
    int64_t        n, padded, n_tiles;
    int            motif_base;          // first motif of this group of 256
    unsigned long long *cand;           // candidate keys: motif << 40 | position
    unsigned long long *cand_count;
    int64_t        cand_capacity;
    // RS_MODE_AND: the sequence condition as a bit per (8-mer, motif), applied before a candidate is staged
    const uint8_t  *codes;              // symbol stream (NULL: structure-only scan, no mask)
    const uint32_t *seqmask;            // [65536][mask_words]: bit (31 - k) of word c = motif 32 c + k may pass
    int            mask_words;          // words per 8-mer over ALL motif groups
    uint32_t       wmask[TC_WMAX + 1][TC_N / 32];   // [f]: motifs of this group whose width is <= f
};

// ------------------------------------------------------------------------------------------------ PTX
__device__ __forceinline__ void tc_mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t *bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tc_mma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// 32 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t (&r)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        "tcgen05.wait::ld.sync.aligned;\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
// the same load without the wait, and the wait as a separate step that "touches" the destination
// registers (so no use of them can be scheduled before it): lets the next chunk's load fly while the
// current chunk is being processed
__device__ __forceinline__ void tc_ld32_issue(uint32_t taddr, uint32_t (&r)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tc_ld_wait(uint32_t (&r)[32])
{
    asm volatile("tcgen05.wait::ld.sync.aligned;\n"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                   "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
                   "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]),
                   "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
                 :
                 : "memory");
}
__device__ __forceinline__ float tc_max3(float a, float b, float c)
{
    float d;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
}

// no-swizzle K-major shared-memory matrix descriptor (units of 16 bytes), sm_100 version bit set
__device__ __forceinline__ uint64_t tc_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes)
{
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;                 // descriptor version for Blackwell
    return d;                               // layout_type (bits 61-63) = 0: SWIZZLE_NONE
}

// kind::f16 instruction descriptor: D fp32, A/B bf16, both K-major, N = 256, M = 128
#define TC_IDESC ((1u << 4) | (1u << 7) | (1u << 10) | ((TC_N >> 3) << 17) | ((TC_M >> 4) << 24))

// Diagnostic (compile with -DRS_TC_TIMELINE, read with tools/tc_timeline.py): clock64 stamps of the stage hand-offs of
// CTA 0's first 96 tiles.  [tile][0] MMA warp: operands ready, [1] accumulator stage free, [2] MMAs issued,
// [3] epilogue warp 4: accumulator full, [4] its chunks done, [5] converter warp 8: raw rows landed, [6] rows converted.
#ifdef RS_TC_TIMELINE
#define TC_TL_TILES 96
__device__ long long g_tc_timeline[TC_TL_TILES * 8];
#define TC_STAMP(it, k) do { if (blockIdx.x == 0 && (it) < TC_TL_TILES) g_tc_timeline[(it) * 8 + (k)] = clock64(); } while (0)
extern "C" int rs_debug_tc_timeline(long long *out)
{
    return cudaMemcpyFromSymbol(out, g_tc_timeline, sizeof(long long) * TC_TL_TILES * 8) == cudaSuccess ? 0 : 2;
}
#else
#define TC_STAMP(it, k) do { } while (0)
#endif

// ------------------------------------------------------------------------------------------------ kernel
__global__ void __launch_bounds__(TC_THREADS, 1) batched_tc_kernel(const __grid_constant__ TcParams prm)
{
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t *s_b = smem;                                           // 48 KB, B operand, resident
    uint8_t *s_a = s_b + TC_B_BYTES;                               // STAGES x bf16 rows
    uint8_t *s_raw = s_a + TC_STAGES * TC_A_BYTES;                 // STAGES x fp32 rows
    uint64_t *bars = reinterpret_cast<uint64_t *>(s_raw + TC_STAGES * TC_RAW_BYTES);
    uint64_t *raw_full = bars, *raw_empty = bars + TC_STAGES, *a_full = bars + 2 * TC_STAGES,
             *a_empty = bars + 3 * TC_STAGES, *acc_full = bars + 4 * TC_STAGES, *acc_empty = acc_full + 2,
             *b_full = acc_empty + 2, *mask_full = b_full + 1;
    uint32_t *s_tmem = reinterpret_cast<uint32_t *>(mask_full + TC_MASK_STAGES);
    unsigned long long *s_cand = reinterpret_cast<unsigned long long *>(smem + 96 * 1024);   // 4 x TC_CBUF keys
    uint4 *s_mask = reinterpret_cast<uint4 *>(smem + 160 * 1024);   // [TC_MASK_STAGES][2 halves][128 positions] x uint4

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        for (int s = 0; s < TC_STAGES; s++) {
            mbar_init(&raw_full[s], 1);
            mbar_init(&raw_empty[s], 4);        // one arrive per converter warp
            mbar_init(&a_full[s], 4);
            mbar_init(&a_empty[s], 1);          // tcgen05.commit
        }
        for (int t = 0; t < 2; t++) { mbar_init(&acc_full[t], 1); mbar_init(&acc_empty[t], 8); }
        mbar_init(b_full, 1);
        for (int k = 0; k < TC_MASK_STAGES; k++) mbar_init(&mask_full[k], 4);
        fence_mbar_init();
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)),
                     "r"(512u)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *s_tmem;

    const int64_t stride = gridDim.x, first = blockIdx.x;
    const int64_t my_tiles = first < prm.n_tiles ? (prm.n_tiles - first + stride - 1) / stride : 0;
    const int64_t prof_end = prm.padded * 28;

    if (warp == 0) {
        // ================= TMA producer
        if (lane == 0) {
            mbar_expect_tx(b_full, TC_B_BYTES);
            bulk_g2s(s_b, prm.bmat, TC_B_BYTES, b_full);
            for (int64_t it = 0; it < my_tiles; it++) {
                const int s = (int)(it % TC_STAGES);
                if (it >= TC_STAGES) mbar_wait(&raw_empty[s], (uint32_t)(((it / TC_STAGES) - 1) & 1));
                const int64_t pstart = (first + it * stride) * TC_M * 28;
                const uint32_t bytes = (uint32_t)min((int64_t)TC_RAW_BYTES, prof_end - pstart);
                mbar_expect_tx(&raw_full[s], bytes);
                bulk_g2s(s_raw + s * TC_RAW_BYTES, reinterpret_cast<const uint8_t *>(prm.profile) + pstart, bytes,
                         &raw_full[s]);
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer
        if (lane == 0) {
            mbar_wait(b_full, 0);
            const uint32_t b_addr = smem_u32(s_b);
            for (int64_t it = 0; it < my_tiles; it++) {
                const int s = (int)(it % TC_STAGES), t = (int)(it & 1);
                mbar_wait(&a_full[s], (uint32_t)((it / TC_STAGES) & 1));
                TC_STAMP(it, 0);
                if (it >= 2) mbar_wait(&acc_empty[t], (uint32_t)(((it >> 1) - 1) & 1));
                TC_STAMP(it, 1);
                tc_fence_after();
                const uint32_t a_addr = smem_u32(s_a + s * TC_A_BYTES);
                const uint32_t d_tmem = tmem_base + (uint32_t)t * TC_N;
#pragma unroll
                for (int k = 0; k < TC_WMAX / 2; k++) {
                    // A: rows shifted by 2k; SBO = 8 rows down (128 B), LBO = next window row (16 B)
                    const uint64_t da = tc_smem_desc(a_addr + 32u * k, 16u, 128u);
                    // B: [j][n][8]: SBO = 8 motifs down (128 B), LBO = next window row (256 * 16 B)
                    const uint64_t db = tc_smem_desc(b_addr + (uint32_t)(2 * k) * (TC_N * 16), TC_N * 16, 128u);
                    tc_mma_bf16(d_tmem, da, db, TC_IDESC, k > 0 ? 1u : 0u);
                }
                tc_commit(&a_empty[s]);          // A stage reusable once these MMAs have read it
                tc_commit(&acc_full[t]);         // accumulator complete
                TC_STAMP(it, 2);
            }
        }
    } else if ((warp >= 4 && warp < 8) || warp >= 12) {
        // ================= epilogue: lanes 32*(warp-4) .. +31 of the accumulator
        // Candidates (accumulator > 0) are staged per warp in shared memory and flushed to the
        // global list with ONE atomic per ~200 entries: a single global counter cannot take one
        // atomic per candidate (structure-only candidates are ~0.1 per position at m = 6).
        // Two warps per TMEM lane quadrant (warp % 4), each reading half of the 256 motif columns:
        // while one waits for its tcgen05.ld the other does the sign-mask arithmetic.
        const int q = warp & 3;
        const int half = warp >= 12 ? 1 : 0;
        unsigned long long *cbuf = s_cand + (half * 4 + q) * TC_CBUF;
        unsigned cnt = 0;                         // warp-uniform number of staged candidates
        auto flush = [&]() {
            unsigned long long base = 0;
            if (lane == 0) base = atomicAdd(prm.cand_count, (unsigned long long)cnt);
            base = __shfl_sync(0xffffffffu, base, 0);
            for (unsigned e = lane; e < cnt; e += 32)
                if ((int64_t)(base + e) < prm.cand_capacity) prm.cand[base + e] = cbuf[e];
            __syncwarp();
            cnt = 0;
        };
        // RS_MODE_AND: the converter warps leave every position's sequence mask (8 words = 256 motifs) in shared memory
        const bool use_mask = prm.codes != nullptr;
        for (int64_t it = 0; it < my_tiles; it++) {
            const int t = (int)(it & 1);
            uint4 mk = make_uint4(~0u, ~0u, ~0u, ~0u);
            if (use_mask) {
                const int ms = (int)(it % TC_MASK_STAGES);
                mbar_wait(&mask_full[ms], (uint32_t)((it / TC_MASK_STAGES) & 1));
                mk = s_mask[(ms * 2 + half) * TC_M + q * 32 + lane];      // lanes read consecutive 16-byte words
            }
            const uint32_t smask[TC_N / 64] = {mk.x, mk.y, mk.z, mk.w};
            mbar_wait(&acc_full[t], (uint32_t)((it >> 1) & 1));
            if (warp == 4 && lane == 0) TC_STAMP(it, 3);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)t * TC_N;
            const int64_t pos = (first + it * stride) * TC_M + q * 32 + lane;
            const bool in_range = pos < prm.n;
            // four chunks of 32 motif columns per warp and tile; the load of chunk i+1 is in flight while
            // chunk i is processed (two register buffers)
            constexpr int NCH = TC_N / 64;
            const int c_first = half * NCH;
            uint32_t va[32], vb[32];
            auto process = [&](uint32_t (&v)[32], int c, uint32_t seq_ok) {
                // sign bits of the 32 accumulators, one funnel shift each: candidate <=> sign clear
                // (accumulator >= +0; unused motif columns carry a -1 bias so they never qualify)
                uint32_t n0 = 0, n1 = 0, n2 = 0, n3 = 0;           // four independent chains of 8
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    n0 = __funnelshift_l(v[k], n0, 1);
                    n1 = __funnelshift_l(v[8 + k], n1, 1);
                    n2 = __funnelshift_l(v[16 + k], n2, 1);
                    n3 = __funnelshift_l(v[24 + k], n3, 1);
                }
                const uint32_t neg = (n0 << 24) | (n1 << 16) | (n2 << 8) | n3;        // bit (31-k) = sign of v[k]
                uint32_t cand = in_range ? (~neg & seq_ok) : 0u;
                if (__any_sync(0xffffffffu, cand != 0)) {                  // warp-uniform, ~40 % of chunks at m = 6
                    const unsigned mine = __popc(cand);
                    unsigned incl = mine;
#pragma unroll
                    for (int d = 1; d < 32; d <<= 1) {
                        const unsigned u = __shfl_up_sync(0xffffffffu, incl, d);
                        if (lane >= d) incl += u;
                    }
                    const unsigned total = __shfl_sync(0xffffffffu, incl, 31);
                    if (cnt + total > TC_CBUF) flush();                      // total <= 1024 = TC_CBUF
                    unsigned slot = cnt + incl - mine;
                    while (cand) {
                        const int b = 31 - __clz(cand);                      // highest bit first = lowest k first
                        cand &= ~(1u << b);
                        cbuf[slot++] = ((unsigned long long)(prm.motif_base + c * 32 + (31 - b)) << 40) |
                                       (unsigned long long)pos;
                    }
                    cnt += total;
                    __syncwarp();
                }
            };
            tc_ld32_issue(taddr + 32u * c_first, va);
#pragma unroll
            for (int i = 0; i < NCH; i++) {
                if ((i & 1) == 0) {
                    tc_ld_wait(va);
                    if (i + 1 < NCH) tc_ld32_issue(taddr + 32u * (c_first + i + 1), vb);
                    process(va, c_first + i, smask[i]);
                } else {
                    tc_ld_wait(vb);
                    if (i + 1 < NCH) tc_ld32_issue(taddr + 32u * (c_first + i + 1), va);
                    process(vb, c_first + i, smask[i]);
                }
            }
            tc_fence_before();
            __syncwarp();
            if (warp == 4 && lane == 0) TC_STAMP(it, 4);
            if (lane == 0) tc_mbar_arrive(&acc_empty[t]);
        }
        if (cnt) flush();
    } else if (warp >= 8 && warp < 12) {
        // ================= converters: fp32 x 7 -> bf16 x 8 (channel 7 := 1.0, the bias input)
        const int ct = tid - 256;                 // 0..127
        // RS_MODE_AND: sequence mask of position (tile, ct) = seqmask[8-mer its window starts with], restricted to
        // the motifs no wider than the distance to the first invalid symbol (prm.wmask).  The symbols are fetched one
        // tile ahead, the mask row is requested before the conversion work and stored after it.
        const bool use_mask = prm.codes != nullptr;
        auto load_codes = [&](int64_t it) {
            const int64_t pos = (first + it * stride) * TC_M + ct;
            uint4 w = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);       // beyond the end: separators
            if (pos < prm.n) {
                const uint32_t *cw = reinterpret_cast<const uint32_t *>(prm.codes + (pos & ~(int64_t)3));
                w = make_uint4(__ldg(cw), __ldg(cw + 1), __ldg(cw + 2), __ldg(cw + 3));
            }
            return w;
        };
        uint4 cw_next = make_uint4(0u, 0u, 0u, 0u);
        if (use_mask && my_tiles > 0) cw_next = load_codes(0);
        for (int64_t it = 0; it < my_tiles; it++) {
            const int s = (int)(it % TC_STAGES);
            uint4 m_lo = make_uint4(0u, 0u, 0u, 0u), m_hi = m_lo;
            int f = 0;
            if (use_mask) {
                const uint4 cw = cw_next;
                const unsigned sh = (unsigned)(((first + it * stride) * TC_M + ct) & 3) * 8u;
                const uint32_t w0 = __funnelshift_r(cw.x, cw.y, sh), w1 = __funnelshift_r(cw.y, cw.z, sh),
                               w2 = __funnelshift_r(cw.z, cw.w, sh);
                // 8-mer index: symbol k in bits 2k, 2k+1 (the multiply gathers four 2-bit fields into the top byte)
                const uint32_t kmer = (((w0 & 0x03030303u) * 0x01041040u) >> 24) |
                                      ((((w1 & 0x03030303u) * 0x01041040u) >> 24) << 8);
                // first symbol that is not A,C,G,U (bits 2,3 set: other, separator): a motif wider than that is out
                const uint32_t i0 = w0 & 0x0C0C0C0Cu, i1 = w1 & 0x0C0C0C0Cu, i2 = w2 & 0x0C0C0C0Cu;
                f = i0 ? (__ffs(i0) - 1) >> 3 : (i1 ? 4 + ((__ffs(i1) - 1) >> 3) : (i2 ? 8 + ((__ffs(i2) - 1) >> 3) : 12));
                const uint4 *row = reinterpret_cast<const uint4 *>(prm.seqmask + (size_t)kmer * prm.mask_words +
                                                                   (prm.motif_base >> 5));
                m_lo = __ldg(row); m_hi = __ldg(row + 1);
                if (it + 1 < my_tiles) cw_next = load_codes(it + 1);
            }
            mbar_wait(&raw_full[s], (uint32_t)((it / TC_STAGES) & 1));
            if (it >= TC_STAGES) mbar_wait(&a_empty[s], (uint32_t)(((it / TC_STAGES) - 1) & 1));
            if (warp == 8 && lane == 0) TC_STAMP(it, 5);
            const float *raw = reinterpret_cast<const float *>(s_raw + s * TC_RAW_BYTES);
            uint4 *arow = reinterpret_cast<uint4 *>(s_a + s * TC_A_BYTES);
            for (int r = ct; r < TC_ROWS; r += 128) {
                const float *p = raw + r * 7;
                __nv_bfloat162 h0 = __floats2bfloat162_rn(p[0], p[1]);
                __nv_bfloat162 h1 = __floats2bfloat162_rn(p[2], p[3]);
                __nv_bfloat162 h2 = __floats2bfloat162_rn(p[4], p[5]);
                __nv_bfloat162 h3 = __floats2bfloat162_rn(p[6], 1.0f);
                uint4 o;
                o.x = *reinterpret_cast<uint32_t *>(&h0);
                o.y = *reinterpret_cast<uint32_t *>(&h1);
                o.z = *reinterpret_cast<uint32_t *>(&h2);
                o.w = *reinterpret_cast<uint32_t *>(&h3);
                arow[r] = o;
            }
            if (use_mask) {
                const int ms = (int)(it % TC_MASK_STAGES);
                const uint32_t *wm = prm.wmask[f];
                s_mask[(ms * 2) * TC_M + ct] = make_uint4(m_lo.x & wm[0], m_lo.y & wm[1], m_lo.z & wm[2], m_lo.w & wm[3]);
                s_mask[(ms * 2 + 1) * TC_M + ct] = make_uint4(m_hi.x & wm[4], m_hi.y & wm[5], m_hi.z & wm[6], m_hi.w & wm[7]);
            }
            fence_proxy_async();                  // generic-proxy writes -> visible to the tensor core
            __syncwarp();
            if (warp == 8 && lane == 0) TC_STAMP(it, 6);
            if (lane == 0) {
                if (use_mask) tc_mbar_arrive(&mask_full[it % TC_MASK_STAGES]);
                tc_mbar_arrive(&a_full[s]); tc_mbar_arrive(&raw_empty[s]);
            }
        }
    }

    // ================= teardown
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// ------------------------------------------------------------------------------------------------ k-mer decision masks
// mask[kmer][word]: for the K symbols a window starts with, which motifs' one-hot score can exceed the threshold.
// A = 4: 8-mers of 2-bit codes (symbol j in bits 2j, 2j+1); A = 7: 5-mers of 3-bit codes (bits 3j .. 3j+2; index 7,
// an invalid symbol, passes nothing -- the callers mask motifs wider than the distance to it anyway).
// W <= K: the decision itself -- the reference's arithmetic (float64 adds in j order; A = 4 casts to float32 once
// and compares widened, _pwm.c:36-65 and SURVEY.md N1; A = 7 compares the float64 sum, matrix.py:34-38).
// W > K: the prefix sum, then the largest entry of every remaining row added in the same order.  Rounded addition
// is monotone, so that is >= the exact score of every window with this prefix: a superset, the exact pass decides
// (NaN: no bound, the window is a candidate).  Bit (31 - k) of word c stands for motif 32 c + k, the order in
// which the tensor-core epilogue's sign masks come out.
template <int A, int K>
__global__ void __launch_bounds__(256) kmer_mask_build_kernel(uint32_t *mask, int mask_words, const double *tables,
                                                              const int *widths, int n_motifs, int stride_rows,
                                                              double threshold)
{
    constexpr int BITS = A == 4 ? 2 : 3;
    constexpr int REST = RS_KMER_WMAX - K;
    // block (word, slab): the 32 motifs of one mask word, 1024 consecutive k-mers; their tables sit in shared memory
    __shared__ double s_tab[32 * K * A];          // first K rows of each motif
    __shared__ double s_rest[32][REST];           // W > K: the largest entry of each row beyond the K-th
    __shared__ int s_w[32];
    const int word = blockIdx.x, slab = blockIdx.y;
    for (int k = threadIdx.x; k < 32 * K * A; k += blockDim.x) {
        const int m = word * 32 + k / (K * A), e = k % (K * A);                // e = row * A + letter
        s_tab[k] = (m < n_motifs && e / A < stride_rows) ? tables[(size_t)m * stride_rows * A + e] : 0.0;
    }
    if (threadIdx.x < 32) {
        const int m = word * 32 + threadIdx.x;
        int W = 0;
        if (m < n_motifs) {
            W = widths[m];
            const double *tab = tables + (size_t)m * stride_rows * A;
            for (int j = K; j < W; j++) {
                double mx = tab[j * A];
                for (int c = 1; c < A; c++) mx = fmax(mx, tab[j * A + c]);
                s_rest[threadIdx.x][j - K] = mx;
            }
        }
        s_w[threadIdx.x] = W;
    }
    __syncthreads();
    for (int q = threadIdx.x; q < 1024; q += blockDim.x) {
        const uint32_t kmer = (uint32_t)slab * 1024u + (uint32_t)q;
        uint32_t bits = 0;
        for (int k = 0; k < 32; k++) {
            const int W = s_w[k];
            if (W == 0) break;
            const double *tab = s_tab + k * K * A;
            const int wp = W < K ? W : K;
            double sum = 0.0;
            bool valid = true;
            for (int j = 0; j < wp; j++) {
                const uint32_t d = (kmer >> (BITS * j)) & ((1u << BITS) - 1u);
                if (d >= (uint32_t)A) { valid = false; break; }
                sum = __dadd_rn(sum, tab[j * A + d]);
            }
            if (!valid) continue;
            for (int j = K; j < W; j++) sum = __dadd_rn(sum, s_rest[k][j - K]);
            const double cmp = A == 4 ? (double)(float)sum : sum;
            if (cmp > threshold || (W > K && sum != sum)) bits |= 1u << (31 - k);
        }
        mask[(size_t)kmer * mask_words + word] = bits;
    }
}

// Builds mask[rows][mask_words] for n_motifs device-resident tables [n_motifs][stride_rows][alphabet] (W <= 16).
int rs_kmer_mask_build(int alphabet, uint32_t *d_mask, int mask_words, const double *d_tables, const int *d_widths,
                       int n_motifs, int stride_rows, double threshold, cudaStream_t st)
{
    if (alphabet == 4)
        kmer_mask_build_kernel<4, 8><<<dim3((unsigned)mask_words, 64), 256, 0, st>>>(d_mask, mask_words, d_tables,
                                                                                     d_widths, n_motifs, stride_rows,
                                                                                     threshold);
    else
        kmer_mask_build_kernel<7, 5><<<dim3((unsigned)mask_words, 32), 256, 0, st>>>(d_mask, mask_words, d_tables,
                                                                                     d_widths, n_motifs, stride_rows,
                                                                                     threshold);
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

// ------------------------------------------------------------------------------------------------ exact re-score
struct RescoreParams {
    const uint8_t *codes;
    const float   *profile;
    const double  *exact64;             // float64 rows the float32 `profile` is a shadow of (or NULL): exact scores
    const double  *seq_tables;          // [M][stride][4] or NULL
    const double  *struct_tables;       // [M][stride][7]
    const int     *widths;              // [M]
    int            stride_rows, mode;
    int64_t        n;
    double         threshold;
    const unsigned long long *cand;
    const unsigned long long *cand_count;
    int64_t        cand_capacity;
    unsigned long long *hitkeys;        // out: keys of true hits (unordered)
    unsigned long long *hit_count;
    unsigned long long *motif_counters2;// [2M]: hits, re-scored
    int64_t        hit_capacity;
};

__device__ __forceinline__ bool tc_exact(const RescoreParams &prm, int m, int64_t pos, float &seq_out, double &str_out)
{
    const int W = prm.widths[m];
    if (pos + W > prm.n) return false;
    seq_out = 0.f;
    if (prm.mode == RS_MODE_AND) {
        // the sequence condition first: W byte gathers, and it rejects ~99.7 % of the structure candidates
        double qd;
        if (!rs_exact_onehot_window<4, 4>(prm.codes + pos, prm.seq_tables + (size_t)m * prm.stride_rows * 4, W, qd))
            return false;
        const float qf = (float)qd;                                  // _pwm.c:65
        seq_out = qf;
        if (!((double)qf > prm.threshold)) return false;             // SURVEY.md note N1
    } else if (!rs_no_separator(prm.codes + pos, W)) {
        return false;
    }
    const double *tab = prm.struct_tables + (size_t)m * prm.stride_rows * RS_CHANNELS;
    const double s = prm.exact64 ? rs_exact_profile_window<double>(prm.exact64 + pos * RS_CHANNELS, tab, W)
                                 : rs_exact_profile_window<float>(prm.profile + pos * RS_CHANNELS, tab, W);
    str_out = s;
    return s > prm.threshold;
}

// SMEM: the sequence tables of all motifs ([M][stride][4] doubles, 96 KB for 256 x 12) and the per-motif
// counters live in shared memory: the sequence condition -- which turns down ~99.7 % of the structure
// candidates -- then costs one global round trip (the window's symbols, five aligned words fetched
// together) instead of W dependent L2 accesses, and the counters are flushed once per CTA.
template <bool SMEM>
__global__ void __launch_bounds__(256) batched_rescore_kernel(const RescoreParams prm, int n_motifs)
{
    extern __shared__ __align__(16) uint8_t rs_smem[];
    double *s_seq = reinterpret_cast<double *>(rs_smem);
    const int seq_doubles = SMEM ? n_motifs * prm.stride_rows * 4 : 0;
    unsigned *s_cnt = reinterpret_cast<unsigned *>(rs_smem + (size_t)seq_doubles * 8);      // [2M]: hits, re-scored
    if (SMEM) {
        for (int k = threadIdx.x; k < seq_doubles; k += blockDim.x) s_seq[k] = prm.seq_tables[k];
        for (int k = threadIdx.x; k < 2 * n_motifs; k += blockDim.x) s_cnt[k] = 0u;
        __syncthreads();
    }
    unsigned long long total = *prm.cand_count;
    if ((int64_t)total > prm.cand_capacity) total = (unsigned long long)prm.cand_capacity;
    for (unsigned long long k = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; k < total;
         k += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned long long key = prm.cand[k];
        const int m = (int)(key >> 40);
        const int64_t pos = (int64_t)(key & ((1ull << 40) - 1));
        float sq; double st;
        bool hit;
        if (SMEM) {
            atomicAdd(&s_cnt[2 * m + 1], 1u);
            const int W = prm.widths[m];
            hit = pos + W <= prm.n;
            if (hit) {
                // the window's symbols: W <= 12 bytes from five aligned words (stream padding covers the over-read)
                const uint32_t *q = reinterpret_cast<const uint32_t *>(prm.codes + (pos & ~(int64_t)3));
                const unsigned sh = (unsigned)(pos & 3) * 8u;
                uint32_t w[5];
#pragma unroll
                for (int i = 0; i < 5; i++) w[i] = q[i];
                const double *tab = s_seq + (size_t)m * prm.stride_rows * 4;
                double qd = 0.0;
                bool ok = true;
#pragma unroll
                for (int j = 0; j < TC_WMAX; j++) {
                    if (j < W) {
                        const uint32_t c = (__funnelshift_r(w[j >> 2], w[(j >> 2) + 1], sh) >> (8 * (j & 3))) & 0xFFu;
                        ok = ok && (c & 7u) < 4u;
                        qd = __dadd_rn(qd, tab[j * 4 + (c & 3u)]);
                    }
                }
                const float qf = (float)qd;                                  // _pwm.c:65
                sq = qf;
                hit = ok && (double)qf > prm.threshold;                      // SURVEY.md note N1
                if (hit) {
                    const double *tq = prm.struct_tables + (size_t)m * prm.stride_rows * RS_CHANNELS;
                    st = prm.exact64 ? rs_exact_profile_window<double>(prm.exact64 + pos * RS_CHANNELS, tq, W)
                                     : rs_exact_profile_window<float>(prm.profile + pos * RS_CHANNELS, tq, W);
                    hit = st > prm.threshold;
                }
            }
            if (hit) atomicAdd(&s_cnt[2 * m], 1u);
        } else {
            atomicAdd(&prm.motif_counters2[2 * m + 1], 1ull);
            hit = tc_exact(prm, m, pos, sq, st);
            if (hit) atomicAdd(&prm.motif_counters2[2 * m], 1ull);
        }
        if (hit) {
            const unsigned long long slot = atomicAdd(prm.hit_count, 1ull);
            if ((int64_t)slot < prm.hit_capacity) prm.hitkeys[slot] = key;
        }
    }
    if (SMEM) {
        __syncthreads();
        for (int k = threadIdx.x; k < 2 * n_motifs; k += blockDim.x)
            if (s_cnt[k]) atomicAdd(&prm.motif_counters2[k], (unsigned long long)s_cnt[k]);
    }
}

// Ordering the hits by (motif, position).  The per-motif hit counts are known (bases[]), so the keys are
// first dropped into their motif's slice in arrival order (one atomic cursor per motif) and then ranked
// INSIDE the slice: keys are unique, the final index of a key is the number of smaller keys of its motif.
// Slices hold ~100 keys, so this is two small launches instead of a ~100-step bitonic network, which
// remains for very large hit lists.
#define SLICE_SORT_MAX 262144
__global__ void tc_bucket_kernel(const unsigned long long *__restrict__ keys, int64_t n_keys,
                                 const unsigned long long *__restrict__ bases, unsigned long long *cursor,
                                 unsigned long long *__restrict__ bucketed)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n_keys) return;
    const unsigned long long key = keys[i];
    const int m = (int)(key >> 40);
    bucketed[bases[m] + atomicAdd(&cursor[m], 1ull)] = key;
}
__global__ void tc_slice_rank_kernel(const unsigned long long *__restrict__ bucketed, int64_t n_keys,
                                     const unsigned long long *__restrict__ bases, unsigned long long *__restrict__ sorted)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n_keys) return;
    const unsigned long long key = bucketed[i];
    const int m = (int)(key >> 40);
    const unsigned long long lo = bases[m], hi = bases[m + 1];
    unsigned long long rank = 0;
    for (unsigned long long k = lo; k < hi; k++) rank += bucketed[k] < key;
    sorted[lo + rank] = key;
}

// bitonic sort of 64-bit keys (padded to a power of two with ~0)
__global__ void tc_pad_keys_kernel(unsigned long long *keys, const unsigned long long *count, int64_t cap, int64_t np2)
{
    unsigned long long n = *count;
    if ((int64_t)n > cap) n = (unsigned long long)cap;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < np2; i += (int64_t)gridDim.x * blockDim.x)
        if ((unsigned long long)i >= n) keys[i] = ~0ull;
}
__global__ void tc_bitonic_step_kernel(unsigned long long *keys, int64_t np2, int64_t j, int64_t k)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < np2; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t l = i ^ j;
        if (l > i) {
            const unsigned long long a = keys[i], b = keys[l];
            const bool up = (i & k) == 0;
            if ((a > b) == up) { keys[i] = b; keys[l] = a; }
        }
    }
}

// sorted keys -> final hit arrays with exact scores, motif slices
__global__ void batched_finalize_kernel(const RescoreParams prm, const unsigned long long *keys,
                                        int32_t *out_motif, int64_t *out_pos, float *out_seq, double *out_str)
{
    unsigned long long total = *prm.hit_count;
    if ((int64_t)total > prm.hit_capacity) total = (unsigned long long)prm.hit_capacity;
    for (unsigned long long k = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; k < total;
         k += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned long long key = keys[k];
        const int m = (int)(key >> 40);
        const int64_t pos = (int64_t)(key & ((1ull << 40) - 1));
        float sq = 0.f; double st = 0.0;
        tc_exact(prm, m, pos, sq, st);
        out_motif[k] = m;
        out_pos[k] = pos;
        if (out_seq) out_seq[k] = sq;
        out_str[k] = st;
    }
}
__global__ void __launch_bounds__(256) batched_bases_kernel(unsigned long long *bases, const unsigned long long *counters2,
                                                            int n_motifs)
{
    __shared__ unsigned long long s_scan[256];
    __shared__ unsigned long long s_carry;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (int m0 = 0; m0 < n_motifs; m0 += 256) {
        const int m = m0 + threadIdx.x;
        const unsigned long long v = m < n_motifs ? counters2[2 * m] : 0ull;
        s_scan[threadIdx.x] = v;
        __syncthreads();
        for (int d = 1; d < 256; d <<= 1) {
            const unsigned long long t = threadIdx.x >= d ? s_scan[threadIdx.x - d] : 0ull;
            __syncthreads();
            s_scan[threadIdx.x] += t;
            __syncthreads();
        }
        if (m < n_motifs) bases[m] = s_carry + s_scan[threadIdx.x] - v;
        __syncthreads();
        if (threadIdx.x == 255) s_carry += s_scan[255];
        __syncthreads();
    }
    if (threadIdx.x == 0) bases[n_motifs] = s_carry;
}

// ------------------------------------------------------------------------------------------------ host
static uint16_t bf16_round_up(double v)          // smallest bf16 >= v
{
    float f = (float)v;
    if ((double)f < v) f = nextafterf(f, INFINITY);               // f >= v
    uint32_t u;
    memcpy(&u, &f, 4);
    uint32_t hi = u & 0xFFFF0000u;                                // truncation = towards zero
    if (hi != u && f > 0) hi += 0x10000u;                         // positive: truncation went down, step up
    return (uint16_t)(hi >> 16);                                  // negative: towards zero is already >= f
}

// Candidates are (position, motif) pairs whose STRUCTURE score may pass; the sequence condition
// of the combined mode is only applied by the exact pass, so allow many more candidates than hits.
static int64_t tc_cand_capacity(int64_t n, int64_t hit_capacity) { return hit_capacity * 8 + (1 << 20) + n / 4; }

int64_t rs_batched_tc_work_bytes(int64_t n, int n_motifs, int stride_rows, int64_t hit_capacity)
{
    int64_t cand_cap = tc_cand_capacity(n, hit_capacity);
    int64_t np2 = 1;
    while (np2 < hit_capacity) np2 <<= 1;
    const int groups = (n_motifs + TC_N - 1) / TC_N;
    return 256 + (int64_t)groups * TC_B_BYTES + cand_cap * 8 + np2 * 8 + 1024 +
           rs_roundup((int64_t)n_motifs * stride_rows * 11 * 8, 256) + rs_roundup((int64_t)n_motifs * 4, 256) +
           (int64_t)65536 * groups * (TC_N / 32) * 4;           // sequence mask: 2 MB per group of 256 motifs
}

static int g_tc_seqmask = 1;          // experiment switch (tools/c5_perf.py): sequence mask in the epilogue on / off
extern "C" int rs_debug_set_tc_seqmask(int on) { g_tc_seqmask = on; return RS_OK; }

// Returns RS_OK, or -1 when this path does not apply (caller falls back to the CUDA-core loop).
int rs_scan_batched_tc(const uint8_t *d_codes, const void *d_profile, int64_t n, int n_motifs, const int *widths,
                       const double *seq_tables, const double *struct_tables, int stride_rows, double threshold,
                       double profile_absrow_max, int mode, int64_t hit_capacity, int32_t *d_hit_motif,
                       int64_t *d_hit_pos, float *d_hit_seq, double *d_hit_struct, uint64_t *d_motif_counters2,
                       uint64_t *d_bases, void *d_work, int64_t work_bytes, cudaStream_t st, const double *d_exact64)
{
    if (stride_rows > TC_WMAX || !isfinite(threshold) || !(profile_absrow_max >= 0) || !isfinite(profile_absrow_max)) {
        rs_set_error("tensor-core path: needs W <= %d, a finite threshold and a finite non-negative profile", TC_WMAX);
        return -1;
    }
    if (work_bytes < rs_batched_tc_work_bytes(n, n_motifs, stride_rows, hit_capacity)) {
        rs_set_error("tensor-core path: workspace %lld < %lld bytes (rs_scan_batched_workspace_bytes)",
                     (long long)work_bytes, (long long)rs_batched_tc_work_bytes(n, n_motifs, stride_rows, hit_capacity));
        return -1;
    }
    const int groups = (n_motifs + TC_N - 1) / TC_N;
    const double R = fmax(profile_absrow_max, 1.0);

    // ---- B operand + bias per motif (host), conservative roundings
    std::vector<uint16_t> bmat((size_t)groups * TC_WMAX * TC_N * 8, 0);
    for (int g = 0; g < groups; g++)                     // unused motif columns: accumulator = -1, never a candidate
        for (int col = 0; col < TC_N; col++)
            bmat[(size_t)g * TC_WMAX * TC_N * 8 + ((size_t)0 * TC_N + col) * 8 + 7] = 0xBF80;   // bf16(-1.0)
    for (int m = 0; m < n_motifs; m++) {
        const int g = m / TC_N, col = m % TC_N, W = widths[m];
        uint16_t *B = bmat.data() + (size_t)g * TC_WMAX * TC_N * 8;
        double S = 0.0;
        for (int j = 0; j < W; j++) {
            bool has_ninf = false;
            for (int c = 0; c < RS_CHANNELS; c++) {
                const double v = struct_tables[((size_t)m * stride_rows + j) * RS_CHANNELS + c];
                if (v != v || v == INFINITY) { rs_set_error("tensor-core path: +inf/NaN table entry"); return -1; }
                if (v == -INFINITY) has_ninf = true;
            }
            double rowmax = 0.0;
            for (int c = 0; c < RS_CHANNELS; c++) {
                const double v = struct_tables[((size_t)m * stride_rows + j) * RS_CHANNELS + c];
                // a row holding -inf contributes <= max(0, finite positive part) after nan_to_num
                const double f = has_ninf ? ((isfinite(v) && v > 0) ? v : 0.0) : v;
                const uint16_t h = bf16_round_up(f);
                B[((size_t)j * TC_N + col) * 8 + c] = h;
                uint32_t u = (uint32_t)h << 16;
                float hf;
                memcpy(&hf, &u, 4);
                rowmax = fmax(rowmax, fabs((double)hf));
            }
            S += rowmax;
        }
        // bf16 keeps 8 significant bits, so round-to-nearest (__floats2bfloat162_rn in the converter warps) is off
        // by up to half an ulp = 2^-8 relative: |sum (bf16(p) - p) * S~| <= 2^-8 * R * S   (p >= 0, S~ >= S
        // entrywise so p*S~ >= p*S); + fp32 accumulation of 96 products, generous: 2^-16 * R * S
        // (+ 2^-24 when the float32 rows are themselves a rounded shadow of float64 rows)
        const double eps = (ldexp(1.0, -8) + ldexp(1.0, -16) + (d_exact64 ? ldexp(1.0, -24) : 0.0)) * R * S * 1.01;
        const double thr_eff = threshold - eps;
        if (!isfinite(thr_eff) || fabs(thr_eff) > 1e30) { rs_set_error("tensor-core path: threshold out of range"); return -1; }
        B[((size_t)0 * TC_N + col) * 8 + 7] = bf16_round_up(-thr_eff);     // bias on the constant-1 channel
    }

    // ---- carve the workspace
    uint8_t *wk = (uint8_t *)d_work;
    int64_t off = 0;
    unsigned long long *cand_count = (unsigned long long *)(wk + off);
    unsigned long long *hit_count = cand_count + 1;                  off += 256;
    uint16_t *d_bmat = (uint16_t *)(wk + off);                       off += (int64_t)groups * TC_B_BYTES;
    const int64_t cand_cap = tc_cand_capacity(n, hit_capacity);
    unsigned long long *cand = (unsigned long long *)(wk + off);     off += cand_cap * 8;
    int64_t np2 = 1;
    while (np2 < hit_capacity) np2 <<= 1;
    unsigned long long *hitkeys = (unsigned long long *)(wk + off);  off += np2 * 8 + 1024;
    double *d_tq = (double *)(wk + off);                             off += (int64_t)n_motifs * stride_rows * 7 * 8;
    double *d_ts = (double *)(wk + off);                             off += (int64_t)n_motifs * stride_rows * 4 * 8;
    off = rs_roundup(off, 256);
    int *d_w = (int *)(wk + off);                                    off += rs_roundup((int64_t)n_motifs * 4, 256);
    uint32_t *d_seqmask = (uint32_t *)(wk + off);
    const int mask_words = groups * (TC_N / 32);

    RS_CUDA(cudaMemsetAsync(cand_count, 0, 16, st));
    RS_CUDA(cudaMemsetAsync(d_motif_counters2, 0, sizeof(uint64_t) * 2 * (size_t)n_motifs, st));
    RS_CUDA(cudaMemcpyAsync(d_bmat, bmat.data(), bmat.size() * 2, cudaMemcpyHostToDevice, st));
    RS_CUDA(cudaMemcpyAsync(d_tq, struct_tables, (size_t)n_motifs * stride_rows * 7 * 8, cudaMemcpyHostToDevice, st));
    if (seq_tables)
        RS_CUDA(cudaMemcpyAsync(d_ts, seq_tables, (size_t)n_motifs * stride_rows * 4 * 8, cudaMemcpyHostToDevice, st));
    RS_CUDA(cudaMemcpyAsync(d_w, widths, (size_t)n_motifs * 4, cudaMemcpyHostToDevice, st));
    // (pageable sources: cudaMemcpyAsync returns once they are staged, so `bmat` may go out of scope)

    // ---- tensor-core filter, one launch per group of 256 motifs
    // 160 KB of dynamic shared memory: more than half an SM's, so exactly one CTA (which owns all
    // 512 TMEM columns) is resident per SM
    const size_t smem = 160 * 1024 + TC_MASK_STAGES * TC_M * 32;      // + the sequence masks of 8 tiles
    static_assert(TC_B_BYTES + TC_STAGES * (TC_A_BYTES + TC_RAW_BYTES) + (21 + TC_MASK_STAGES) * 8 + 16 <= 96 * 1024, "smem layout");
    static_assert(96 * 1024 + 8 * TC_CBUF * 8 <= 160 * 1024, "smem layout");
    static bool configured[RS_MAX_DEVICES] = {};          // the attribute is per device
    const int dev = rs_current_device();
    if (!configured[dev]) {
        RS_CUDA(cudaFuncSetAttribute(batched_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured[dev] = true;
    }
    const bool use_mask = mode == RS_MODE_AND && seq_tables != nullptr && g_tc_seqmask;
    if (use_mask) {
        int rc = rs_kmer_mask_build(4, d_seqmask, mask_words, d_ts, d_w, n_motifs, stride_rows, threshold, st);
        if (rc) return rc;
    }
    TcParams tp = {};
    tp.codes = use_mask ? d_codes : nullptr; tp.seqmask = d_seqmask; tp.mask_words = mask_words;
    tp.profile = (const float *)d_profile; tp.n = n; tp.padded = rs_padded_count(n);
    tp.n_tiles = (n + TC_M - 1) / TC_M;
    tp.cand = cand; tp.cand_count = cand_count; tp.cand_capacity = cand_cap;
    int64_t grid = rs_sm_count();
    if (grid > tp.n_tiles) grid = tp.n_tiles;
    for (int g = 0; g < groups; g++) {
        tp.bmat = d_bmat + (size_t)g * TC_WMAX * TC_N * 8;
        tp.motif_base = g * TC_N;
        memset(tp.wmask, 0, sizeof(tp.wmask));
        for (int k = 0; k < TC_N && g * TC_N + k < n_motifs; k++)
            for (int f = widths[g * TC_N + k]; f <= TC_WMAX; f++) tp.wmask[f][k >> 5] |= 1u << (31 - (k & 31));
        rs_prof_start(st);
        batched_tc_kernel<<<(unsigned)grid, TC_THREADS, smem, st>>>(tp);
        rs_prof_stop(st);
        RS_CUDA(cudaGetLastError());
    }
    unsigned long long h_cand = 0;
    RS_CUDA(cudaMemcpyAsync(&h_cand, cand_count, 8, cudaMemcpyDeviceToHost, st));
    RS_CUDA(cudaStreamSynchronize(st));
    if ((int64_t)h_cand > cand_cap) {            // too many candidates for the workspace: use the CUDA-core loop
        rs_set_error("tensor-core path: %llu candidates exceed the workspace (%lld)", h_cand, (long long)cand_cap);
        return -1;
    }

    // ---- exact re-score, sort, finalize
    RescoreParams rp = {};
    rp.codes = d_codes; rp.profile = (const float *)d_profile; rp.exact64 = d_exact64; rp.seq_tables = seq_tables ? d_ts : nullptr;
    rp.struct_tables = d_tq; rp.widths = d_w; rp.stride_rows = stride_rows; rp.mode = mode; rp.n = n;
    rp.threshold = threshold; rp.cand = cand; rp.cand_count = cand_count; rp.cand_capacity = cand_cap;
    rp.hitkeys = hitkeys; rp.hit_count = hit_count; rp.motif_counters2 = (unsigned long long *)d_motif_counters2;
    rp.hit_capacity = hit_capacity;
    if (h_cand > 0) {
        const size_t tab_smem = (size_t)n_motifs * stride_rows * 4 * 8 + (size_t)n_motifs * 2 * 4;
        if (mode == RS_MODE_AND && tab_smem <= 100 * 1024) {
            static bool rs_configured[RS_MAX_DEVICES] = {};
            if (!rs_configured[dev]) {
                RS_CUDA(cudaFuncSetAttribute(batched_rescore_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             100 * 1024));
                rs_configured[dev] = true;
            }
            int blocks = (int)fmin((double)((h_cand + 255) / 256), (double)rs_sm_count() * 2);
            batched_rescore_kernel<true><<<blocks, 256, tab_smem, st>>>(rp, n_motifs);
        } else {
            int blocks = (int)fmin((double)((h_cand + 255) / 256), (double)rs_sm_count() * 8);
            batched_rescore_kernel<false><<<blocks, 256, 0, st>>>(rp, n_motifs);
        }
        RS_CUDA(cudaGetLastError());
    }
    batched_bases_kernel<<<1, 256, 0, st>>>((unsigned long long *)d_bases, (const unsigned long long *)d_motif_counters2,
                                          n_motifs);
    RS_CUDA(cudaGetLastError());
    unsigned long long h_hits = 0;
    RS_CUDA(cudaMemcpyAsync(&h_hits, hit_count, 8, cudaMemcpyDeviceToHost, st));
    RS_CUDA(cudaStreamSynchronize(st));
    if (h_hits == 0 || hit_capacity == 0) return RS_OK;
    const int64_t stored = (int64_t)h_hits < hit_capacity ? (int64_t)h_hits : hit_capacity;
    if ((int64_t)h_hits <= hit_capacity && stored <= SLICE_SORT_MAX && stored + n_motifs + 1 <= cand_cap) {
        // the candidate list is no longer needed: it holds the bucketed keys and the per-motif cursors
        unsigned long long *bucketed = cand, *cursor = cand + stored;
        RS_CUDA(cudaMemsetAsync(cursor, 0, (size_t)n_motifs * 8, st));
        const int blocks = (int)((stored + 255) / 256);
        tc_bucket_kernel<<<blocks, 256, 0, st>>>(hitkeys, stored, (const unsigned long long *)d_bases, cursor, bucketed);
        tc_slice_rank_kernel<<<blocks, 256, 0, st>>>(bucketed, stored, (const unsigned long long *)d_bases, hitkeys);
        RS_CUDA(cudaGetLastError());
        batched_finalize_kernel<<<blocks, 256, 0, st>>>(rp, hitkeys, d_hit_motif, d_hit_pos, d_hit_seq, d_hit_struct);
        RS_CUDA(cudaGetLastError());
        return RS_OK;
    }
    int64_t nsort = 1;
    while (nsort < stored) nsort <<= 1;
    const int sort_blocks = (int)fmin((double)((nsort + 255) / 256), (double)rs_sm_count() * 8);
    tc_pad_keys_kernel<<<sort_blocks, 256, 0, st>>>(hitkeys, hit_count, hit_capacity, nsort);
    for (int64_t k = 2; k <= nsort; k <<= 1)
        for (int64_t j = k >> 1; j > 0; j >>= 1)
            tc_bitonic_step_kernel<<<sort_blocks, 256, 0, st>>>(hitkeys, nsort, j, k);
    RS_CUDA(cudaGetLastError());
    batched_finalize_kernel<<<sort_blocks, 256, 0, st>>>(rp, hitkeys, d_hit_motif, d_hit_pos, d_hit_seq, d_hit_struct);
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}
