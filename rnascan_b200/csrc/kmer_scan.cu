// Sequence-PSSM threshold scan for W <= 8 through an EXACT k-mer decision table.
//
// Replaces, like onehot_scan.cu, _pwm.c:34-68 driven per window by Biopython search()
// (rnascan.py:263) -- but the per-window work is one table lookup instead of W dependent
// fp64 adds.  The nucleotide alphabet has 4 letters, so a window is a 2W-bit number: for
// W <= 8 every possible window fits a 16-bit index and the hit decision
//        (double)(float)(sum_j table[j][code_j])  >  threshold           (_pwm.c:36-65, N1)
// can be tabulated for all 65 536 8-mers up front, IN THE REFERENCE'S OWN ARITHMETIC
// (kmer_lut_kernel: sequential fp64 adds in j order, one cast to float).  The table is
// therefore not a filter with a guard band but the exact decision; scores are recomputed
// only for the windows that are reported.  An 8-mer holds Q = 9 - W consecutive windows,
// so one byte lookup decides Q positions at once.
//
// Per thread: 28 consecutive positions (7-word stride => conflict-free LDS.32), 9 words of
// symbol bytes are squeezed to 2 bits/symbol with one AND + one IMAD per word
// ((w & 0x03030303) * 0x01041040 gathers the four 2-bit fields into the top byte) and
// merged with PRMT; each lookup index is a funnel shift of that 72-bit string.  Invalid
// symbols (N, separators, padding) are ignored on the fast path -- they can only create
// false candidates, never lose a hit -- and candidates of threads whose bytes hold any
// invalid symbol are re-checked.
//
// The hot kernel is a pure stream: a producer warp feeds a 3-stage shared-memory ring with
// bulk async copies (full/empty mbarriers, no CTA-wide barrier), 8 consumer warps turn
// symbols into one 28-bit hit mask per thread (one coalesced 4-byte store) plus one count
// per warp segment (896 positions; mask words of segments without a hit are not even written).  No
// atomics, no divergent emission.  Ordering is ONE more launch (kmer_finish_kernel): a prefix sum over
// the segment counts, then the non-empty segments are expanded (popc/shuffle prefix inside the
// segment) with positions and exact scores written straight to their final, position-sorted place.
#include "common.cuh"
#include "provisional.cuh"
#include <type_traits>

#define KM_CONSUMERS   512                         // consumer threads (16 warps share one table; 2 CTAs per SM)
#define KM_THREADS     (KM_CONSUMERS + 32)         // + one producer warp
#define KM_P           28                          // positions per thread
#define KM_TILE        (KM_CONSUMERS * KM_P)       // 14336 = 28 * 512
#define KM_STAGES      3
#define KM_STAGE_BYTES (KM_TILE + 16)              // +8 symbols of halo, rounded to 16
#define KM_LUT_BYTES   65536
#define KM_WARPS       (KM_CONSUMERS / 32)
#define KM_SEG         (32 * KM_P)                 // 896 positions per warp segment
#define FIN_THREADS    1024                        // segments per CTA of the finish kernel (one per thread)
#define FIN_STAGE_BYTES 6048                       // profile finish: per-warp stage, 29 float windows of W <= 7

struct KmerWork {                 // carved out of the caller's workspace
    uint8_t  *lut;                // [65536]
    uint32_t *mask;               // [n_tiles * 256] hit mask per consumer thread
    uint32_t *segcnt;             // [n_segs] hits per warp segment
    unsigned long long *ticket;   // [2]  ticket, pad -- zeroed together with agg before every scan
    unsigned long long *agg;      // [n_ctas] finish kernel: 0 = not ready, else CTA aggregate + 1
};

struct KmerParams {
    const uint8_t *codes;
    int64_t        n, padded, n_tiles;
    KmerWork       wk;
};

struct KmerTable { double t[8 * 4]; };

__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// zero the finish kernel's ticket + aggregates from a kernel that runs before it anyway (saves a memset node)
__device__ __forceinline__ void zero_words(unsigned long long *w, int n_words)
{
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n_words; k += gridDim.x * blockDim.x) w[k] = 0ull;
}

// bit r of lut[idx] = window of W symbols starting at symbol r of the 8-mer `idx` is a hit
__global__ void kmer_lut_kernel(uint8_t *__restrict__ lut, const KmerTable tab, int W, double threshold,
                                unsigned long long *zero, int n_zero)
{
    zero_words(zero, n_zero);
    const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int Q = 9 - W;
    unsigned bits = 0;
    for (int r = 0; r < Q; r++) {
        double s = 0.0;
        for (int j = 0; j < W; j++) s = __dadd_rn(s, tab.t[j * 4 + ((idx >> (2 * (r + j))) & 3u)]);
        const float f = (float)s;                                  // _pwm.c:65
        if ((double)f > threshold) bits |= 1u << r;                // SURVEY.md note N1
    }
    lut[idx] = (uint8_t)bits;
}

// Same from a PROVISIONAL table (provisional.cuh) that every CTA derives from the device-resident counts.
// float casts are monotone, so every window the exact table would report has
// (float)(s + margin) > threshold here: the bits are a superset.
// Host notification (rs_scan_onehot_begin_notify): the counts go straight into page-locked host memory -- no copy
// engine, no event, no stream synchronisation between the histogram and the host's exact table.  Every word carries
// the call's 16-bit tag above the 48-bit count, so the eight stores need no ordering among themselves (no system-wide
// fence on the device): the host waits until all eight words show the tag.  clear8: another 8-counter array zeroed
// here (the NEXT step's histogram target).
struct CountsNotify {
    unsigned long long *host8;      // NULL: no notification
    unsigned long long tag;         // 1 .. 65535
    unsigned long long *clear8;     // or NULL
};

__device__ __forceinline__ void counts_notify(const unsigned long long *__restrict__ counts8, const CountsNotify &nt)
{
    if (threadIdx.x < 8) {
        if (nt.clear8) nt.clear8[threadIdx.x] = 0ull;
        if (nt.host8)
            *(volatile unsigned long long *)(nt.host8 + threadIdx.x) =
                (nt.tag << 48) | (counts8[threadIdx.x] & 0xFFFFFFFFFFFFull);
    }
}

__global__ void counts_notify_kernel(const unsigned long long *__restrict__ counts8, const CountsNotify nt)
{
    counts_notify(counts8, nt);
}

__global__ void kmer_lut_dev_kernel(uint8_t *__restrict__ lut, const unsigned long long *__restrict__ counts8,
                                    const __grid_constant__ ProvProb prob, double threshold, double extra_margin,
                                    const CountsNotify nt, unsigned long long *zero, int n_zero)
{
    __shared__ double tab[RS_PROV_MAX_W * 4];
    if (blockIdx.x == 0) counts_notify(counts8, nt);
    zero_words(zero, n_zero);
    const int W = prob.W;
    const double margin = rs_prov_table_cta<4>(counts8, prob, tab) + extra_margin;
    const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int Q = 9 - W;
    unsigned bits = 0;
    for (int r = 0; r < Q; r++) {
        double s = 0.0;
        for (int j = 0; j < W; j++) s = __dadd_rn(s, tab[j * 4 + ((idx >> (2 * (r + j))) & 3u)]);
        const float f = (float)__dadd_ru(s, margin);
        if ((double)f > threshold) bits |= 1u << r;
    }
    lut[idx] = (uint8_t)bits;
}

template <int W>
__global__ void __launch_bounds__(KM_THREADS, 2) kmer_scan_kernel(const __grid_constant__ KmerParams prm)
{
    constexpr int Q = 9 - W;
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t *full = reinterpret_cast<uint64_t *>(smem);          // [STAGES] tile landed
    uint64_t *empty = full + KM_STAGES;                           // [STAGES] tile consumed by all warps
    uint64_t *lutbar = empty + KM_STAGES;
    uint8_t *s_lut = smem + 128;
    uint8_t *stages = s_lut + KM_LUT_BYTES;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        for (int s = 0; s < KM_STAGES; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], KM_WARPS); }
        mbar_init(lutbar, 1);
        fence_mbar_init();
    }
    __syncthreads();

    const int64_t stride = gridDim.x, first = blockIdx.x;
    const int64_t my_tiles = first < prm.n_tiles ? (prm.n_tiles - first + stride - 1) / stride : 0;

    if (warp == KM_WARPS) {
        // ---------------- producer warp: one lane drives the TMA engine
        if (lane == 0) {
            mbar_expect_tx(lutbar, KM_LUT_BYTES);
            bulk_g2s(s_lut, prm.wk.lut, KM_LUT_BYTES, lutbar);
            for (int64_t it = 0; it < my_tiles; it++) {
                const int s = (int)(it % KM_STAGES);
                if (it >= KM_STAGES) mbar_wait(&empty[s], (uint32_t)(((it / KM_STAGES) - 1) & 1));
                const int64_t t0 = (first + it * stride) * KM_TILE;
                const uint32_t bytes = (uint32_t)min((int64_t)KM_STAGE_BYTES, prm.padded - t0);
                mbar_expect_tx(&full[s], bytes);
                bulk_g2s(stages + (size_t)s * KM_STAGE_BYTES, prm.codes + t0, bytes, &full[s]);
            }
        }
        return;
    }

    // -------------------- consumer warps
    mbar_wait(lutbar, 0);
    for (int64_t it = 0; it < my_tiles; it++) {
        const int s = (int)(it % KM_STAGES);
        mbar_wait(&full[s], (uint32_t)((it / KM_STAGES) & 1));

        const int64_t tile = first + it * stride;
        const uint8_t *sym = stages + (size_t)s * KM_STAGE_BYTES + tid * KM_P;
        const uint32_t *wp = reinterpret_cast<const uint32_t *>(sym);
        const int64_t g0 = tile * KM_TILE + (int64_t)tid * KM_P;

        // ---- 36 symbol bytes -> 72 bits, 2 per symbol, symbol k at bits 2k
        uint32_t x[9], inv = 0;
#pragma unroll
        for (int k = 0; k < 9; k++) {
            const uint32_t w = wp[k];
            inv |= w & 0x0C0C0C0Cu;                                // any symbol that is not A/C/G/U
            x[k] = (w & 0x03030303u) * 0x01041040u;                // four 2-bit fields -> top byte
        }
        const uint32_t r0 = __byte_perm(__byte_perm(x[0], x[1], 0x0073), __byte_perm(x[2], x[3], 0x0073), 0x5410);
        const uint32_t r1 = __byte_perm(__byte_perm(x[4], x[5], 0x0073), __byte_perm(x[6], x[7], 0x0073), 0x5410);
        const uint32_t r2 = x[8] >> 24;

        // ---- one decision byte per Q positions
        uint32_t hit = 0;
#pragma unroll
        for (int p = 0; p < KM_P; p += Q) {
            const int sh = 2 * p;
            uint32_t idx;
            if (sh + 16 <= 32)      idx = (r0 >> sh) & 0xFFFFu;
            else if (sh < 32)       idx = __funnelshift_r(r0, r1, sh) & 0xFFFFu;
            else if (sh + 16 <= 64) idx = (r1 >> (sh - 32)) & 0xFFFFu;
            else                    idx = __funnelshift_r(r1, r2, sh - 32) & 0xFFFFu;
            hit |= (uint32_t)s_lut[idx] << p;
        }
        hit &= (1u << KM_P) - 1u;

        // ---- candidates next to an invalid symbol or the end of the stream: check the bytes
        if (hit != 0 && (inv != 0 || g0 + KM_P + W > prm.n)) {
            uint32_t keep = 0;
            for (uint32_t h = hit; h; h &= h - 1) {
                const int p = __ffs(h) - 1;
                bool ok = g0 + p + W <= prm.n;
                for (int j = 0; j < W; j++) ok = ok && sym[p + j] < 4;
                if (ok) keep |= 1u << p;
            }
            hit = keep;
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[s]);                     // this warp is done with the stage

        const unsigned total = __reduce_add_sync(0xffffffffu, (unsigned)__popc(hit));
        if (total) prm.wk.mask[tile * KM_CONSUMERS + tid] = hit;       // only non-empty segments are expanded
        if (lane == 0) prm.wk.segcnt[tile * KM_WARPS + warp] = total;
    }
}

// ---- finish: prefix sum over the segment counts + expansion, ONE launch -----------------------
// One thread per segment takes part in the exclusive prefix sum (CTAs chained by ticket + look-back over
// the aggregates of the CTAs before them, as in order.cu); then the hits of the non-empty segments are
// expanded (per-warp queue, see below) with positions and EXACT scores written straight to their
// final, position-sorted place.
struct ExpandParams {
    const uint8_t *codes;
    KmerWork wk;
    int64_t n_segs, capacity;
    int n_ctas;
    unsigned long long *counters;
    OrderDest od;
    int W;
    int ppm;                  // positions per mask word: 28 (k-mer scan) or 32 (ballot masks)
    int verify;               // the masks are CANDIDATES (provisional table): re-decide with the exact score;
    double threshold;         //   a candidate that is not a hit gets position -1 and counts in counters[1]
    double ta[16 * 8];        // exact table, row stride A_STRIDE
    const uint8_t *codes_b;   // pair mode: structure stream scored with tb (row stride 8) into od.str
    double tb[16 * 8];
    // profile mode (kmer_finish_kernel<4, PT>): every candidate gets its W profile rows scored with sd (row stride 7),
    // and its exact sequence score is recomputed where the structure score passes; od receives every candidate at its
    // candidate index, position -1 unless both scores pass, and counters[1] counts the structure scores computed.
    // compact_hits_kernel then keeps the hits.
    const void *profile;
    double sd[16 * RS_CHANNELS];
    unsigned long long *zero;  // compact_hits_kernel's ticket + aggregates, zeroed here
    int n_zero;
};

__device__ __forceinline__ unsigned long long fin_block_scan(unsigned long long v, unsigned long long &total)
{
    __shared__ unsigned long long s_w[FIN_THREADS / 32];
    __shared__ unsigned long long s_total;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        unsigned long long t = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += t;
    }
    __syncthreads();                          // protect s_w / s_total across repeated calls
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        unsigned long long x = lane < FIN_THREADS / 32 ? s_w[lane] : 0ull, xi = x;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            unsigned long long t = __shfl_up_sync(0xffffffffu, xi, d);
            if (lane >= d) xi += t;
        }
        if (lane < FIN_THREADS / 32) s_w[lane] = xi - x;
        if (lane == 31) s_total = xi;
    }
    __syncthreads();
    total = s_total;
    return s_w[warp] + incl - v;
}

__device__ __forceinline__ void add_warp_count(unsigned long long *counter, unsigned v)
{
    v = __reduce_add_sync(0xffffffffu, v);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(counter, (unsigned long long)v);
}

// exact score of the (W <= 16)-symbol window at stream position `pos`: its bytes come from five aligned
// words fetched together (ONE memory round trip per hit instead of W dependent ones; the padding of the
// stream covers the over-read), then sequential fp64 adds in j order.
template <int A, int TS>
__device__ __forceinline__ double fin_window_score(const uint8_t *codes, int64_t pos, int W, const double *tab)
{
    const uint32_t *q = reinterpret_cast<const uint32_t *>(codes + (pos & ~(int64_t)3));
    const unsigned sh = (unsigned)(pos & 3) * 8u;
    uint32_t w[5];
#pragma unroll
    for (int i = 0; i < 5; i++) w[i] = q[i];
    double s = 0.0;
#pragma unroll
    for (int j = 0; j < 16; j++) {
        if (j < W) {
            const uint32_t x = __funnelshift_r(w[j >> 2], w[(j >> 2) + 1], sh);
            s = __dadd_rn(s, tab[j * TS + ((x >> (8 * (j & 3))) & (A == 4 ? 3u : 7u))]);
        }
    }
    return s;
}

// 16-byte global -> shared copy that bypasses the registers (LDGSTS); cp_async_wait_all waits for all of this
// thread's copies (the other lanes' copies are visible after a __syncwarp that follows their wait)
__device__ __forceinline__ void cp_async16(void *dst, const void *src)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all()
{
    asm volatile("cp.async.wait_all;" ::: "memory");
}

// A = 4: float32 sequence scores (row stride 4); A = 7: float64 structure scores (row stride 8).
// PT = float or double: combined mode over the profile rows (see ExpandParams::profile).
template <int A, typename PT = void>
__global__ void __launch_bounds__(FIN_THREADS) kmer_finish_kernel(const __grid_constant__ ExpandParams prm)
{
    constexpr int TS = A == 4 ? 4 : 8;
    constexpr bool PROFILE = !std::is_void<PT>::value;
    if (PROFILE) zero_words(prm.zero, prm.n_zero);
    __shared__ unsigned s_vb;
    if (threadIdx.x == 0) s_vb = (unsigned)atomicAdd(prm.wk.ticket, 1ull);
    __syncthreads();
    const unsigned vb = s_vb;
    const int64_t seg = (int64_t)vb * FIN_THREADS + threadIdx.x;
    const uint32_t segcnt = seg < prm.n_segs ? prm.wk.segcnt[seg] : 0u;
    unsigned long long total;
    const unsigned long long excl = fin_block_scan(segcnt, total);
    if (threadIdx.x == 0) {
        // counters[1] (candidates the exact table rejects) is zeroed HERE, by the first CTA, before its aggregate is
        // published: every other CTA reads that aggregate in its look-back before it scores anything
        if (vb == 0) prm.counters[1] = 0ull;
        __threadfence();
        ((volatile unsigned long long *)prm.wk.agg)[vb] = total + 1ull;
    }
    unsigned long long part = 0;
    for (unsigned p = threadIdx.x; p < vb; p += FIN_THREADS) {
        unsigned long long v;
        unsigned spins = 0;
        unsigned long long t_start = 0ull;
        while ((v = ((volatile unsigned long long *)prm.wk.agg)[p]) == 0ull) {
            __nanosleep(20);
            if ((++spins & 0xFFFFu) == 0u && rs_spin_expired(t_start)) __trap();   // a minute without the predecessor's aggregate
        }
        part += v - 1ull;
    }
    __threadfence();
    unsigned long long before;
    fin_block_scan(part, before);
    if (vb == (unsigned)(prm.n_ctas - 1) && threadIdx.x == 0) {
        prm.counters[0] = before + total;
        *prm.wk.ticket = 0ull;
    }
    if (prm.capacity <= 0) return;
    // Expansion.  A lane owns one segment: its 32 mask words (128 contiguous bytes) are fetched with eight
    // independent 16-byte loads.  Hits are sparse across (lane, word), so instead of scoring them where
    // they are found (a few active lanes per pass) every lane pushes its hits into a per-warp queue and the
    // warp scores queue entries 32 at a time with all lanes busy.  A queue entry is 32 bits: output index and
    // position, both relative to the warp's first (a warp's 32 segments cover < 2^15 positions and its
    // output slots are contiguous).
    constexpr unsigned QCAP = 256;
    __shared__ uint32_t q[FIN_THREADS / 32][QCAP];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned long long my_k = before + excl + (prm.od.out_base ? *prm.od.out_base : 0ull);
    const unsigned long long warp_k = __shfl_sync(0xffffffffu, my_k, 0);
    const int64_t warp_pos = (seg - lane) * 32 * (int64_t)prm.ppm;
    uint4 m[8];
    if (segcnt) {
        const uint4 *mv = reinterpret_cast<const uint4 *>(prm.wk.mask + seg * 32);
#pragma unroll
        for (int i = 0; i < 8; i++) m[i] = mv[i];
    } else {
#pragma unroll
        for (int i = 0; i < 8; i++) m[i] = make_uint4(0u, 0u, 0u, 0u);
    }
    auto score_entry = [&](uint32_t e) {
        const unsigned long long kk = warp_k + (e >> 16);
        const int64_t pos = warp_pos + (e & 0xFFFFu);
        if ((int64_t)kk < prm.capacity) {
            const double sc = fin_window_score<A, TS>(prm.codes, pos, prm.W, prm.ta);
            bool is_hit = true;
            if (prm.verify) {
                is_hit = (A == 4 ? (double)(float)sc : sc) > prm.threshold;     // _pwm.c:65 / note N1
                if (!is_hit) atomicAdd(prm.counters + 1, 1ull);
            }
            prm.od.pos[kk] = is_hit ? pos : -1;
            if (A == 4) prm.od.seq[kk] = (float)sc;                        // _pwm.c:65
            else        prm.od.str[kk] = sc;                               // matrix.py:34-42
            if (A == 4 && prm.codes_b)                                     // pair mode: structure score of the same window
                prm.od.str[kk] = fin_window_score<7, 8>(prm.codes_b, pos, prm.W, prm.tb);
            if (prm.od.out_motif) prm.od.out_motif[kk] = prm.od.motif_id;
        }
    };
    // Profile mode: the windows of queue entries first .. first + n - 1 (slot index & qm), in rounds of R.  A window's
    // W rows are 28 W (float) or 56 W (double) contiguous bytes; the lanes copy the 16-byte pieces of every window's
    // aligned hull into the warp's stage (all copies of a round in flight together, neighbouring windows served by the
    // same lines), then each lane scores one window from shared memory with the exact arithmetic.  Only a window whose
    // structure score passes has its symbols re-read for the sequence score.  The masks come from the exact sequence
    // table, so every in-capacity candidate is a structure score computed (counters[1]).
    using RowT = std::conditional_t<PROFILE, PT, float>;
    constexpr unsigned ROWB = RS_CHANNELS * sizeof(RowT);
    const unsigned WB = (unsigned)prm.W * ROWB;
    const unsigned NP = (WB + (16 - (unsigned)sizeof(RowT)) + 15) / 16;      // pieces of the widest hull
    const unsigned R = min(32u, (unsigned)FIN_STAGE_BYTES / (NP * 16));
    extern __shared__ __align__(16) uint8_t fin_stage[];
    unsigned n_struct = 0;
    auto score_profile = [&](unsigned first, unsigned n, unsigned qm) {
        uint8_t *stage = fin_stage + warp * FIN_STAGE_BYTES;
        const uint8_t *rows = reinterpret_cast<const uint8_t *>(prm.profile);
        for (unsigned r0 = 0; r0 < n; r0 += R) {
            const unsigned nr = min(R, n - r0);
            for (unsigned p = lane; p < nr * NP; p += 32) {
                const unsigned i = p / NP, k = p - i * NP;
                const uint32_t e = q[warp][(first + r0 + i) & qm];
                const int64_t b = (warp_pos + (e & 0xFFFFu)) * ROWB;
                const int64_t a = (b & ~(int64_t)15) + 16 * k;
                if ((int64_t)(warp_k + (e >> 16)) < prm.capacity && a < b + WB)
                    cp_async16(stage + (i * NP + k) * 16, rows + a);
            }
            cp_async_wait_all();
            __syncwarp();
            if ((unsigned)lane < nr) {
                const uint32_t e = q[warp][(first + r0 + lane) & qm];
                const unsigned long long kk = warp_k + (e >> 16);
                const int64_t pos = warp_pos + (e & 0xFFFFu);
                if ((int64_t)kk < prm.capacity) {
                    n_struct++;
                    const RowT *win = reinterpret_cast<const RowT *>(stage + lane * NP * 16 + ((pos * ROWB) & 15));
                    const double sc = rs_exact_profile_window<RowT>(win, prm.sd, prm.W);
                    bool is_hit = sc > prm.threshold;                                // rnascan.py:308, 416-434
                    if (is_hit) {
                        const double sq = fin_window_score<4, 4>(prm.codes, pos, prm.W, prm.ta);
                        is_hit = (double)(float)sq > prm.threshold;                  // _pwm.c:65 / note N1
                        if (is_hit) {
                            prm.od.seq[kk] = (float)sq;
                            prm.od.str[kk] = sc;
                        }
                    }
                    prm.od.pos[kk] = is_hit ? pos : -1;
                }
            }
            __syncwarp();
        }
    };
    // queue slots by a warp prefix over the lanes' hit counts (== segcnt): no per-slot coordination
    unsigned incl = segcnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned v = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += v;
    }
    const unsigned warp_total = __shfl_sync(0xffffffffu, incl, 31);
    if (warp_total == 0) return;
    const unsigned koff0 = (unsigned)(my_k - warp_k);       // == incl - segcnt
    if (warp_total <= QCAP) {
        // the usual case: every lane writes its own hits (position order), then full-lane scoring rounds
        unsigned e = incl - segcnt, koff = koff0;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const uint32_t w4[4] = {m[i].x, m[i].y, m[i].z, m[i].w};
#pragma unroll
            for (int t = 0; t < 4; t++) {
                const unsigned poff = (unsigned)((lane * 32 + i * 4 + t) * prm.ppm);
                for (uint32_t h = w4[t]; h; h &= h - 1)
                    q[warp][e++] = (koff++ << 16) | (poff + (unsigned)(__ffs(h) - 1));
            }
        }
        __syncwarp();
        if constexpr (PROFILE) {
            score_profile(0, warp_total, QCAP - 1);
            add_warp_count(prm.counters + 1, n_struct);
        } else {
            for (unsigned r = lane; r < warp_total; r += 32) score_entry(q[warp][r]);
        }
        return;
    }
    // dense segments: word by word through a 64-entry ring of the same queue
    unsigned head = 0, count = 0, koff = koff0;            // head, count: warp-uniform ring state
    auto drain = [&](unsigned n_take) {
        __syncwarp();
        if constexpr (PROFILE) score_profile(head, n_take, 63u);
        else if ((unsigned)lane < n_take) score_entry(q[warp][(head + lane) & 63u]);
        __syncwarp();
        head = (head + n_take) & 63u;
        count -= n_take;
    };
    if constexpr (PROFILE) {
        // the words in a run-time loop: one copy of the round code here instead of one per word (32 copies of a
        // profile round do not fit the instruction cache); the groups after the second are fetched again, one
        // group ahead, so that only two stay in registers
        const uint4 *mv = reinterpret_cast<const uint4 *>(prm.wk.mask + seg * 32);
        uint4 cur = m[0], nxt = m[1];
#pragma unroll 1
        for (int w = 0; w < 32; w++) {
            uint32_t h = (w & 2) ? ((w & 1) ? cur.w : cur.z) : ((w & 1) ? cur.y : cur.x);
            if ((w & 3) == 3) {
                cur = nxt;
                if (w < 24) nxt = segcnt ? mv[(w >> 2) + 2] : make_uint4(0u, 0u, 0u, 0u);
            }
            const unsigned poff = (unsigned)((lane * 32 + w) * prm.ppm);
            for (;;) {
                const unsigned has = __ballot_sync(0xffffffffu, h != 0);
                if (!has) break;
                while (count >= R) drain(R);                      // whole rounds
                if (h) {
                    const unsigned e = (head + count + __popc(has & ((1u << lane) - 1u))) & 63u;
                    q[warp][e] = (koff++ << 16) | (poff + (unsigned)(__ffs(h) - 1));
                    h &= h - 1;
                }
                count += __popc(has);
            }
        }
    } else {
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const uint32_t w4[4] = {m[i].x, m[i].y, m[i].z, m[i].w};
#pragma unroll
            for (int t = 0; t < 4; t++) {
                uint32_t h = w4[t];
                const unsigned poff = (unsigned)((lane * 32 + i * 4 + t) * prm.ppm);
                for (;;) {
                    const unsigned has = __ballot_sync(0xffffffffu, h != 0);
                    if (!has) break;
                    if (count > 32u) drain(32u);
                    if (h) {
                        const unsigned e = (head + count + __popc(has & ((1u << lane) - 1u))) & 63u;
                        q[warp][e] = (koff++ << 16) | (poff + (unsigned)(__ffs(h) - 1));
                        h &= h - 1;
                    }
                    count += __popc(has);
                }
            }
        }
    }
    while (count) drain(count < 32u ? count : 32u);
    if (PROFILE) add_warp_count(prm.counters + 1, n_struct);
}

// ---- one-hot threshold scan, W <= 16, any alphabet: exact scores, hit bits by warp ballot ----------
// Structure contexts (A = 7) and sequence motifs wider than the k-mer table (A = 4, 8 < W <= 16).
// Same scoring loop as dense_w_kernel (onehot_scan.cu): lanes take consecutive windows, symbols are
// fetched as aligned words + funnel shifts, one LDS.64 + one fp64 add per symbol in j order -- the
// reference's arithmetic, so the ballot bit IS the decision (score > m, strict).  Instead of a dense
// 4-8 B/position output each warp keeps 32 ballot words (1024 positions = one segment) and stores them
// with one coalesced 128-byte write; ordering and exact output scores are the segment scan + expansion
// shared with the k-mer scan.
#define MS_THREADS 256
#define MS_PER     32
#define MS_TILE    (MS_THREADS * MS_PER)           // 8192 positions; 1024 per warp
#define MS_STAGES  3
#define MS_STAGE_BYTES (MS_TILE + 32)

struct MaskScanParams {
    const uint8_t *codes;
    const uint8_t *codes_b;   // PAIR: structure stream
    int64_t n, padded, n_tiles;
    double threshold;
    KmerWork wk;
    const unsigned long long *d_counts8;   // candidates mode: provisional table from these counts (else NULL)
    double extra_margin;
    ProvProb prob;
    double ta[16 * 8];
    double tb[16 * 8];        // PAIR: structure table
};

// exact one-hot score of the window starting at byte w of a staged tile; `bad` != 0 <=> invalid symbol
template <int A, int W>
__device__ __forceinline__ double ms_score(const uint32_t *words, int w, uint32_t tab, uint32_t &bad)
{
    constexpr int NW = (W + 3) / 4;
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
    bad = 0;
#pragma unroll
    for (int i = 0; i < NW; i++) {
        const uint32_t m = (i == NW - 1 && (W & 3)) ? (0xFFFFFFFFu >> (32 - 8 * (W & 3))) : 0xFFFFFFFFu;
        if (A == 4) bad |= x[i] & (0x0C0C0C0Cu & m);
        else        bad |= x[i] & (x[i] >> 1) & (x[i] >> 2) & (0x01010101u & m);
    }
    double sum = 0.0;
#pragma unroll
    for (int j = 0; j < W; j++) {
        const int sb = 8 * (j & 3);
        const uint32_t off = sb >= 3 ? ((x[j >> 2] >> (sb - 3)) & 0x38u) : ((x[j >> 2] << 3) & 0x38u);
        double t;
        asm("ld.shared.f64 %0, [%1];" : "=d"(t) : "r"(tab + (uint32_t)(j * 64) + off));
        sum = __dadd_rn(sum, t);
    }
    return sum;
}

template <int A, int W, bool PAIR>
__global__ void __launch_bounds__(MS_THREADS) mask_scan_kernel(const __grid_constant__ MaskScanParams prm)
{
    constexpr int TS = 8;
    constexpr int NSTREAM = PAIR ? 2 : 1;
    constexpr int STAGES = PAIR ? 2 : MS_STAGES;          // static shared memory stays under 48 KB
    __shared__ __align__(128) uint8_t s_stage[STAGES * NSTREAM * MS_STAGE_BYTES];
    __shared__ __align__(16) double s_ta[W * TS];
    __shared__ __align__(16) double s_tb[PAIR ? W * TS : 1];
    __shared__ uint64_t bars[STAGES];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // candidates mode: provisional score + margin (rounded up) is compared, a superset of the exact hits
    double margin = 0.0;
    const bool provisional = !PAIR && prm.d_counts8 != nullptr;
    if (provisional) {
        margin = rs_prov_table_cta<TS>(prm.d_counts8, prm.prob, s_ta) + prm.extra_margin;
    } else {
        for (int k = tid; k < W * TS; k += MS_THREADS) {
            s_ta[k] = prm.ta[k];
            if (PAIR) s_tb[k] = prm.tb[k];
        }
    }
    if (tid == 0) {
        for (int s = 0; s < STAGES; s++) mbar_init(&bars[s], 1);
        fence_mbar_init();
    }
    __syncthreads();
    const int64_t stride = gridDim.x, first = blockIdx.x;
    const int64_t my_tiles = first < prm.n_tiles ? (prm.n_tiles - first + stride - 1) / stride : 0;
    auto issue = [&](int64_t it) {
        const int s = (int)(it % STAGES);
        const int64_t t0 = (first + it * stride) * MS_TILE;
        const uint32_t bytes = (uint32_t)min((int64_t)MS_STAGE_BYTES, prm.padded - t0);
        uint8_t *dst = s_stage + (size_t)s * NSTREAM * MS_STAGE_BYTES;
        mbar_expect_tx(&bars[s], bytes * NSTREAM);
        bulk_g2s(dst, prm.codes + t0, bytes, &bars[s]);
        if (PAIR) bulk_g2s(dst + MS_STAGE_BYTES, prm.codes_b + t0, bytes, &bars[s]);
    };
    if (tid == 0)
        for (int64_t it = 0; it < STAGES - 1 && it < my_tiles; it++) issue(it);
    const uint32_t tab = smem_u32(s_ta), tab_b = smem_u32(s_tb);

    for (int64_t it = 0; it < my_tiles; it++) {
        const int s = (int)(it % STAGES);
        if (tid == 0 && it + STAGES - 1 < my_tiles) issue(it + STAGES - 1);
        mbar_wait(&bars[s], (uint32_t)((it / STAGES) & 1));
        const int64_t tile = first + it * stride;
        const int64_t t0 = tile * MS_TILE;
        const uint32_t *words = reinterpret_cast<const uint32_t *>(s_stage + (size_t)s * NSTREAM * MS_STAGE_BYTES);
        const uint32_t *words_b = words + MS_STAGE_BYTES / 4;
        uint32_t mine = 0, total = 0;
#pragma unroll 4
        for (int k = 0; k < MS_PER; k++) {
            const int w = warp * (32 * MS_PER) + k * 32 + lane;
            uint32_t bad;
            double sum = ms_score<A, W>(words, w, tab, bad);
            if (provisional) sum = __dadd_ru(sum, margin);
            const double cmp = A == 4 ? (double)(float)sum : sum;          // _pwm.c:65 / note N1
            bool hit = !bad && cmp > prm.threshold && t0 + w + W <= prm.n;
            if (PAIR && hit) {                                             // both scores must pass (rnascan.py:416-434)
                uint32_t bad_b;
                const double sb = ms_score<7, W>(words_b, w, tab_b, bad_b);
                hit = !bad_b && sb > prm.threshold;
            }
            const uint32_t b = __ballot_sync(0xffffffffu, hit);
            if (lane == k) mine = b;
            total += __popc(b);
        }
        const int64_t seg = tile * (MS_THREADS / 32) + warp;
        if (total) prm.wk.mask[seg * 32 + lane] = mine;                    // one coalesced 128-byte store
        if (lane == 0) prm.wk.segcnt[seg] = total;
        __syncthreads();
    }
}

template <int A, int W>
static int launch_mask_scan(const MaskScanParams &prm, cudaStream_t stream)
{
    int64_t grid = (int64_t)rs_grid_sms() * (prm.codes_b ? 4 : 6);
    if (grid > prm.n_tiles) grid = prm.n_tiles;
    rs_prof_start(stream);
    if (A == 4 && prm.codes_b) mask_scan_kernel<4, W, true><<<(unsigned)grid, MS_THREADS, 0, stream>>>(prm);
    else mask_scan_kernel<A, W, false><<<(unsigned)grid, MS_THREADS, 0, stream>>>(prm);
    rs_prof_stop(stream);
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

template <int A>
static int dispatch_mask_scan(int W, const MaskScanParams &prm, cudaStream_t stream)
{
    switch (W) {
#define MS_CASE(w) case w: return launch_mask_scan<A, w>(prm, stream);
        MS_CASE(1) MS_CASE(2) MS_CASE(3) MS_CASE(4) MS_CASE(5) MS_CASE(6) MS_CASE(7) MS_CASE(8)
        MS_CASE(9) MS_CASE(10) MS_CASE(11) MS_CASE(12) MS_CASE(13) MS_CASE(14) MS_CASE(15) MS_CASE(16)
#undef MS_CASE
    default: rs_set_error("internal: mask scan needs W <= 16"); return RS_ERR_INVALID;
    }
}

static void carve_work(uint8_t *wk, int64_t n_masks, int64_t n_segs, int n_ctas, KmerWork &out)
{
    int64_t off = 0;
    out.lut = wk + off;                               off += KM_LUT_BYTES;
    out.mask = (uint32_t *)(wk + off);                off += rs_roundup(n_masks * 4, 256);
    out.segcnt = (uint32_t *)(wk + off);              off += rs_roundup(n_segs * 4, 256);
    out.ticket = (unsigned long long *)(wk + off);    off += 16;
    out.agg = (unsigned long long *)(wk + off);
    (void)n_ctas;
}
static int fin_ctas(int64_t n_segs) { return (int)((n_segs + FIN_THREADS - 1) / FIN_THREADS); }
static cudaError_t fin_arm(const KmerWork &wk, int n_ctas, cudaStream_t st)
{
    return cudaMemsetAsync(wk.ticket, 0, 16 + (size_t)n_ctas * 8, st);
}

template <int A>
static int finish_mask_scan(const uint8_t *d_codes, const KmerWork &wk, int64_t n_segs, int n_ctas, int ppm,
                            const double *table, int W, int64_t cap, int64_t *d_hit_pos, float *d_hit_seq,
                            double *d_hit_str, uint64_t *d_counters2, cudaStream_t st,
                            const uint8_t *d_codes_b = nullptr, const double *table_b = nullptr,
                            bool verify = false, double threshold = 0.0)
{
    ExpandParams ep = {};
    ep.codes = d_codes; ep.wk = wk; ep.n_segs = n_segs; ep.capacity = cap; ep.W = W; ep.ppm = ppm;
    ep.n_ctas = n_ctas; ep.counters = (unsigned long long *)d_counters2;
    ep.verify = verify ? 1 : 0; ep.threshold = threshold;
    ep.od = OrderDest{d_hit_pos, d_hit_seq, d_hit_str, nullptr, nullptr, 0};
    constexpr int TS = A == 4 ? 4 : 8;
    for (int j = 0; j < W; j++)
        for (int c = 0; c < A; c++) ep.ta[j * TS + c] = table[j * A + c];
    ep.codes_b = d_codes_b;
    if (table_b)
        for (int j = 0; j < W; j++)
            for (int c = 0; c < 7; c++) ep.tb[j * 8 + c] = table_b[j * 7 + c];
    kmer_finish_kernel<A><<<(unsigned)n_ctas, FIN_THREADS, 0, st>>>(ep);
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

struct OneHotGeom {
    bool kmer;
    int64_t n_tiles, n_segs, n_masks;
    int n_ctas, ppm;
};
static OneHotGeom onehot_geom(int A, int W, int64_t n)
{
    OneHotGeom g;
    g.kmer = A == 4 && W <= 8;
    if (g.kmer) {
        g.n_tiles = (n + KM_TILE - 1) / KM_TILE;
        g.n_segs = g.n_tiles * KM_WARPS;
        g.n_masks = g.n_tiles * KM_CONSUMERS;
        g.ppm = KM_P;
    } else {
        g.n_tiles = (n + MS_TILE - 1) / MS_TILE;
        g.n_segs = g.n_tiles * (MS_THREADS / 32);
        g.n_masks = g.n_segs * 32;
        g.ppm = 32;
    }
    g.n_ctas = fin_ctas(g.n_segs);
    return g;
}

// ---- combined mode, sequence first: compaction of the candidates' verdicts ----------------------------------
// kmer_finish_kernel<4, PT> leaves every candidate at its candidate index (position order) in the staging arrays,
// position -1 unless both scores passed.  One thread per CP_PER consecutive candidates takes part in an exclusive
// prefix sum of the survivors (CTAs chained by ticket + look-back, as in the finish kernel) and copies them out.
#define CP_THREADS 1024
#define CP_PER     8
#define CP_SPAN    (CP_THREADS * CP_PER)

struct CompactParams {
    const int64_t *pos;                    // staged verdicts, capacity entries
    const float *seq;
    const double *str;
    const unsigned long long *cand;        // [0] candidates (may exceed capacity), [1] structure scores computed
    int64_t capacity;
    unsigned long long *ticket, *agg;      // zeroed by the finish kernel
    int n_ctas;
    int64_t *out_pos;
    float *out_seq;
    double *out_str;
    unsigned long long *counters;          // [0] hits, [1] structure scores computed
};

__global__ void __launch_bounds__(CP_THREADS) compact_hits_kernel(const __grid_constant__ CompactParams prm)
{
    __shared__ unsigned s_vb;
    if (threadIdx.x == 0) s_vb = (unsigned)atomicAdd(prm.ticket, 1ull);
    __syncthreads();
    const unsigned vb = s_vb;
    const unsigned long long n_cand = prm.cand[0];
    const int64_t lim = (int64_t)n_cand < prm.capacity ? (int64_t)n_cand : prm.capacity;
    const int64_t k0 = ((int64_t)vb * CP_THREADS + threadIdx.x) * CP_PER;
    unsigned keep = 0;
#pragma unroll
    for (int i = 0; i < CP_PER; i++)
        if (k0 + i < lim && prm.pos[k0 + i] >= 0) keep |= 1u << i;
    unsigned long long total;
    const unsigned long long excl = fin_block_scan((unsigned long long)__popc(keep), total);
    if (threadIdx.x == 0) {
        __threadfence();
        ((volatile unsigned long long *)prm.agg)[vb] = total + 1ull;
    }
    unsigned long long part = 0;
    for (unsigned p = threadIdx.x; p < vb; p += CP_THREADS) {
        unsigned long long v;
        unsigned spins = 0;
        unsigned long long t_start = 0ull;
        while ((v = ((volatile unsigned long long *)prm.agg)[p]) == 0ull) {
            __nanosleep(20);
            if ((++spins & 0xFFFFu) == 0u && rs_spin_expired(t_start)) __trap();   // a minute without the predecessor's aggregate
        }
        part += v - 1ull;
    }
    __threadfence();
    unsigned long long before;
    fin_block_scan(part, before);
    if (vb == (unsigned)(prm.n_ctas - 1) && threadIdx.x == 0) {
        // candidates beyond the staging room were never scored: report their count, an upper bound of the hits,
        // so that the caller regrows the buffers
        prm.counters[0] = (int64_t)n_cand > prm.capacity ? n_cand : before + total;
        prm.counters[1] = prm.cand[1];
        *prm.ticket = 0ull;
    }
    unsigned long long dst = before + excl;
    for (uint32_t h = keep; h; h &= h - 1, dst++) {
        const int64_t k = k0 + __ffs(h) - 1;
        if ((int64_t)dst < prm.capacity) {
            prm.out_pos[dst] = prm.pos[k];
            prm.out_seq[dst] = prm.seq[k];
            prm.out_str[dst] = prm.str[k];
        }
    }
}

// Finish of the sequence-first combined scan: the masks in the workspace hold the sequence candidates (exact or
// provisional table); staging = the workspace's hit staging arrays, compaction state in its segment table.
template <typename PT>
static int finish_profile(const uint8_t *d_codes, const void *d_profile, int64_t n, const double *seq_table,
                          const double *struct_table, int W, double threshold, int64_t cap, int64_t *d_hit_pos,
                          float *d_hit_seq, double *d_hit_str, uint64_t *d_cand2, uint64_t *d_counters2,
                          uint8_t *d_work, cudaStream_t st)
{
    const WorkLayout wl = rs_work_layout(n, cap);
    const OneHotGeom g = onehot_geom(4, W, n);
    ExpandParams ep = {};
    carve_work(d_work + wl.off_lut, g.n_masks, g.n_segs, g.n_ctas, ep.wk);
    ep.codes = d_codes; ep.n_segs = g.n_segs; ep.capacity = cap; ep.W = W; ep.ppm = g.ppm; ep.n_ctas = g.n_ctas;
    ep.counters = (unsigned long long *)d_cand2; ep.threshold = threshold; ep.verify = 1;
    int64_t *s_pos = (int64_t *)(d_work + wl.off_pos);
    float *s_seq = (float *)(d_work + wl.off_seq);
    double *s_str = (double *)(d_work + wl.off_str);
    ep.od = OrderDest{s_pos, s_seq, s_str, nullptr, nullptr, 0};
    for (int k = 0; k < W * 4; k++) ep.ta[k] = seq_table[k];
    ep.profile = d_profile;
    for (int k = 0; k < W * RS_CHANNELS; k++) ep.sd[k] = struct_table[k];
    const int64_t span = cap < n ? cap : n;                   // never more candidates than windows
    const int cp_ctas = (int)(span / CP_SPAN + 1);
    unsigned long long *cp_state = (unsigned long long *)(d_work + wl.off_seg);   // ticket, pad, agg[cp_ctas]
    ep.zero = cp_state; ep.n_zero = 2 + cp_ctas;
    constexpr size_t smem = (size_t)(FIN_THREADS / 32) * FIN_STAGE_BYTES;     // the warps' window stages
    static bool configured[RS_MAX_DEVICES] = {};          // the attribute is per device
    const int dev = rs_current_device();
    if (!configured[dev]) {
        RS_CUDA(cudaFuncSetAttribute(kmer_finish_kernel<4, PT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured[dev] = true;
    }
    kmer_finish_kernel<4, PT><<<(unsigned)g.n_ctas, FIN_THREADS, smem, st>>>(ep);
    RS_CUDA(cudaGetLastError());
    CompactParams cp = {};
    cp.pos = s_pos; cp.seq = s_seq; cp.str = s_str; cp.cand = (const unsigned long long *)d_cand2;
    cp.capacity = cap; cp.ticket = cp_state; cp.agg = cp_state + 2; cp.n_ctas = cp_ctas;
    cp.out_pos = d_hit_pos; cp.out_seq = d_hit_seq; cp.out_str = d_hit_str;
    cp.counters = (unsigned long long *)d_counters2;
    compact_hits_kernel<<<(unsigned)cp_ctas, CP_THREADS, 0, st>>>(cp);
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

template <int W>
static int launch_kmer(const KmerParams &prm, cudaStream_t stream)
{
    const size_t smem = 128 + KM_LUT_BYTES + (size_t)KM_STAGES * KM_STAGE_BYTES;
    static bool configured[RS_MAX_DEVICES] = {};          // the attribute is per device
    const int dev = rs_current_device();
    if (!configured[dev]) {
        RS_CUDA(cudaFuncSetAttribute(kmer_scan_kernel<W>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured[dev] = true;
    }
    int64_t grid = (int64_t)rs_grid_sms() * 2;
    if (grid > prm.n_tiles) grid = prm.n_tiles;
    rs_prof_start(stream);
    kmer_scan_kernel<W><<<(unsigned)grid, KM_THREADS, smem, stream>>>(prm);
    rs_prof_stop(stream);
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

int64_t rs_kmer_work_bytes(int64_t n)
{
    const int64_t n_tiles = (n > 0 ? n : 0) / KM_TILE + 1;
    const int64_t n_segs = n_tiles * KM_WARPS;
    const int64_t n_ctas = n_segs / FIN_THREADS + 2;
    return KM_LUT_BYTES + rs_roundup(n_tiles * KM_CONSUMERS * 4, 256) + rs_roundup(n_segs * 4, 256) +
           rs_roundup(16 + n_ctas * 8, 256) + 256;
}

// ---- single-stream one-hot threshold scans, W <= 16, in two halves -------------------------------------
// begin : decision masks + segment counts into the workspace (k-mer table scan for A = 4, W <= 8, ballot
//         mask scan otherwise), from the exact host table or from a device-resident provisional table;
// finish: segment prefix + expansion with the exact host table (verify = the masks were only candidates).

template <int A>
static int onehot_begin(const uint8_t *d_codes, int64_t n, const double *table, const uint64_t *d_counts8,
                        const double *prob, double extra_margin, int W, double threshold, uint8_t *wk_lut,
                        cudaStream_t st, CountsNotify nt = CountsNotify())
{
    const OneHotGeom g = onehot_geom(A, W, n);
    KmerWork wk;
    carve_work(wk_lut, g.n_masks, g.n_segs, g.n_ctas, wk);
    if (!g.kmer) RS_CUDA(fin_arm(wk, g.n_ctas, st));     // k-mer path: the table kernel zeroes ticket + aggregates
    ProvProb pp = {};
    if (d_counts8) {
        pp.W = W; pp.A = A;
        for (int k = 0; k < W * A; k++) pp.p[k] = prob[k];
    }
    if (g.kmer) {
        KmerParams prm = {};
        prm.codes = d_codes; prm.n = n; prm.padded = rs_padded_count(n); prm.n_tiles = g.n_tiles; prm.wk = wk;
        if (d_counts8) {
            kmer_lut_dev_kernel<<<KM_LUT_BYTES / 256, 256, 0, st>>>(wk.lut, (const unsigned long long *)d_counts8, pp,
                                                                    threshold, extra_margin, nt, wk.ticket,
                                                                    2 + g.n_ctas);
        } else {
            KmerTable kt = {};
            for (int k = 0; k < W * 4; k++) kt.t[k] = table[k];
            kmer_lut_kernel<<<KM_LUT_BYTES / 256, 256, 0, st>>>(wk.lut, kt, W, threshold, wk.ticket, 2 + g.n_ctas);
        }
        RS_CUDA(cudaGetLastError());
        switch (W) {
        case 1: return launch_kmer<1>(prm, st);
        case 2: return launch_kmer<2>(prm, st);
        case 3: return launch_kmer<3>(prm, st);
        case 4: return launch_kmer<4>(prm, st);
        case 5: return launch_kmer<5>(prm, st);
        case 6: return launch_kmer<6>(prm, st);
        case 7: return launch_kmer<7>(prm, st);
        case 8: return launch_kmer<8>(prm, st);
        default: rs_set_error("internal: k-mer scan needs W <= 8"); return RS_ERR_INVALID;
        }
    }
    if (d_counts8 && (nt.host8 || nt.clear8)) {
        counts_notify_kernel<<<1, 32, 0, st>>>((const unsigned long long *)d_counts8, nt);
        RS_CUDA(cudaGetLastError());
    }
    MaskScanParams prm = {};
    prm.codes = d_codes; prm.n = n; prm.padded = rs_padded_count(n); prm.threshold = threshold;
    prm.n_tiles = g.n_tiles; prm.wk = wk; prm.extra_margin = extra_margin;
    prm.d_counts8 = (const unsigned long long *)d_counts8; prm.prob = pp;
    if (table)
        for (int j = 0; j < W; j++)
            for (int c = 0; c < 8; c++) prm.ta[j * 8 + c] = c < A ? table[j * A + c] : 0.0;
    return dispatch_mask_scan<A>(W, prm, st);
}

template <int A>
static int onehot_finish(const uint8_t *d_codes, int64_t n, const double *table, int W, double threshold, bool verify,
                         int64_t cap, int64_t *d_hit_pos, float *d_hit_seq, double *d_hit_str, uint64_t *d_counters2,
                         uint8_t *wk_lut, cudaStream_t st)
{
    const OneHotGeom g = onehot_geom(A, W, n);
    KmerWork wk;
    carve_work(wk_lut, g.n_masks, g.n_segs, g.n_ctas, wk);
    return finish_mask_scan<A>(d_codes, wk, g.n_segs, g.n_ctas, g.ppm, table, W, cap, d_hit_pos, d_hit_seq, d_hit_str,
                               d_counters2, st, nullptr, nullptr, verify, threshold);
}

// Called by rs_scan_seq / rs_scan_struct_onehot (onehot_scan.cu) for W <= 16.
int rs_scan_onehot_masks(int A, const uint8_t *d_codes, int64_t n, const double *table, int W, double threshold,
                         int64_t cap, int64_t *d_hit_pos, float *d_hit_seq, double *d_hit_str,
                         uint64_t *d_counters2, void *d_work, cudaStream_t st)
{
    uint8_t *wk = (uint8_t *)d_work + rs_work_layout(n, cap).off_lut;
    int rc = A == 4 ? onehot_begin<4>(d_codes, n, table, nullptr, nullptr, 0.0, W, threshold, wk, st)
                    : onehot_begin<7>(d_codes, n, table, nullptr, nullptr, 0.0, W, threshold, wk, st);
    if (rc) return rc;
    return A == 4 ? onehot_finish<4>(d_codes, n, table, W, threshold, false, cap, d_hit_pos, d_hit_seq, nullptr,
                                     d_counters2, wk, st)
                  : onehot_finish<7>(d_codes, n, table, W, threshold, false, cap, d_hit_pos, nullptr, d_hit_str,
                                     d_counters2, wk, st);
}
int rs_scan_seq_kmer(const uint8_t *d_codes, int64_t n, const double *table, int W, double threshold, int64_t cap,
                     int64_t *d_hit_pos, float *d_hit_score, uint64_t *d_counters2, void *d_work, cudaStream_t st)
{
    return rs_scan_onehot_masks(4, d_codes, n, table, W, threshold, cap, d_hit_pos, d_hit_score, nullptr, d_counters2,
                                d_work, st);
}

// Combined mode (RS_MODE_AND) of rs_scan_fused for W <= 16, sequence first: the k-mer / mask scan with the exact
// sequence table, then only the windows that pass it have their profile rows read and scored.  Same hits, scores and
// order as the structure-first kernels (same exact arithmetic).  d_cand2 (device, or NULL = inside the workspace):
// [0] sequence candidates, [1] structure scores computed; d_counters2[0] = hits (the candidate count instead when
// the candidates outgrew hit_capacity: regrow), [1] = structure scores computed.
int rs_scan_fused_seqfirst(const uint8_t *d_codes, const void *d_profile, int profile_dtype, int64_t n,
                           const double *seq_table, const double *struct_table, int W, double threshold, int64_t cap,
                           int64_t *d_hit_pos, float *d_hit_seq, double *d_hit_str, uint64_t *d_cand2,
                           uint64_t *d_counters2, void *d_work, cudaStream_t st)
{
    const WorkLayout wl = rs_work_layout(n, cap);
    uint8_t *wk = (uint8_t *)d_work;
    int rc = onehot_begin<4>(d_codes, n, seq_table, nullptr, nullptr, 0.0, W, threshold, wk + wl.off_lut, st);
    if (rc) return rc;
    if (!d_cand2) d_cand2 = (uint64_t *)(wk + wl.off_scan);      // unused by this path otherwise
    return profile_dtype == RS_F64
        ? finish_profile<double>(d_codes, d_profile, n, seq_table, struct_table, W, threshold, cap, d_hit_pos,
                                 d_hit_seq, d_hit_str, d_cand2, d_counters2, wk, st)
        : finish_profile<float>(d_codes, d_profile, n, seq_table, struct_table, W, threshold, cap, d_hit_pos,
                                d_hit_seq, d_hit_str, d_cand2, d_counters2, wk, st);
}

static int begin_finish_args(int alphabet, const uint8_t *d_codes, int64_t n, int W, double threshold)
{
    if (alphabet != 4 && alphabet != 7) { rs_set_error("alphabet must be 4 (A,C,G,U) or 7 (B,E,H,L,M,R,T)"); return RS_ERR_INVALID; }
    if (!d_codes || ((uintptr_t)d_codes & 15)) { rs_set_error("codes pointer null or not 16-byte aligned"); return RS_ERR_INVALID; }
    if (W < 1 || W > 16) { rs_set_error("the two-call scan covers motif widths 1..16 (got %d): use the one-call scan", W); return RS_ERR_INVALID; }
    if (n < 0) { rs_set_error("negative length"); return RS_ERR_INVALID; }
    if (threshold != threshold) { rs_set_error("threshold is NaN"); return RS_ERR_INVALID; }
    return RS_OK;
}

extern "C" int rs_scan_onehot_begin_notify(int alphabet, const uint8_t *d_codes, int64_t n, const uint64_t *d_counts8,
                                           const double *prob, int W, double threshold, double extra_margin,
                                           int64_t hit_capacity, void *d_work, int64_t work_bytes,
                                           uint64_t *h_notify8, uint32_t tag, uint64_t *d_clear8, void *stream)
{
    int rc = begin_finish_args(alphabet, d_codes, n, W, threshold);
    if (rc) return rc;
    if (!d_counts8 || !prob) { rs_set_error("null counts or probabilities"); return RS_ERR_INVALID; }
    if (!(extra_margin >= 0)) { rs_set_error("extra_margin must be >= 0"); return RS_ERR_INVALID; }
    if (d_clear8 == d_counts8) { rs_set_error("d_clear8 must not be the counts being read"); return RS_ERR_INVALID; }
    if (h_notify8 && (tag < 1 || tag > 65535)) { rs_set_error("notification tag must be 1..65535"); return RS_ERR_INVALID; }
    CountsNotify nt;
    nt.host8 = (unsigned long long *)h_notify8; nt.tag = tag; nt.clear8 = (unsigned long long *)d_clear8;
    cudaStream_t st = (cudaStream_t)stream;
    if (n < W) {                                        // nothing to scan: the host is still told the counts
        if (nt.host8 || nt.clear8) {
            counts_notify_kernel<<<1, 32, 0, st>>>((const unsigned long long *)d_counts8, nt);
            RS_CUDA(cudaGetLastError());
        }
        return RS_OK;
    }
    WorkLayout wl = rs_work_layout(n, hit_capacity);
    if (!d_work || work_bytes < wl.total) { rs_set_error("workspace too small: need %lld bytes", (long long)wl.total); return RS_ERR_WORKSPACE; }
    uint8_t *wk = (uint8_t *)d_work + wl.off_lut;
    return alphabet == 4 ? onehot_begin<4>(d_codes, n, nullptr, d_counts8, prob, extra_margin, W, threshold, wk, st, nt)
                         : onehot_begin<7>(d_codes, n, nullptr, d_counts8, prob, extra_margin, W, threshold, wk, st, nt);
}

extern "C" int rs_scan_onehot_begin(int alphabet, const uint8_t *d_codes, int64_t n, const uint64_t *d_counts8,
                                    const double *prob, int W, double threshold, double extra_margin,
                                    int64_t hit_capacity, void *d_work, int64_t work_bytes, void *stream)
{
    return rs_scan_onehot_begin_notify(alphabet, d_codes, n, d_counts8, prob, W, threshold, extra_margin, hit_capacity,
                                       d_work, work_bytes, nullptr, 0, nullptr, stream);
}

extern "C" int rs_scan_onehot_finish(int alphabet, const uint8_t *d_codes, int64_t n, const double *table, int W,
                                     double threshold, int64_t hit_capacity, int64_t *d_hit_pos, void *d_hit_score,
                                     uint64_t *d_counters2, void *d_work, int64_t work_bytes, void *stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    int rc = begin_finish_args(alphabet, d_codes, n, W, threshold);
    if (rc) return rc;
    if (!table || !d_counters2 || hit_capacity < 0 || (hit_capacity > 0 && (!d_hit_pos || !d_hit_score))) {
        rs_set_error("rs_scan_onehot_finish: bad argument"); return RS_ERR_INVALID;
    }
    if (n < W) {                                        // else: the finish kernel writes both counters itself
        RS_CUDA(cudaMemsetAsync(d_counters2, 0, 2 * sizeof(uint64_t), st));
        return RS_OK;
    }
    WorkLayout wl = rs_work_layout(n, hit_capacity);
    if (!d_work || work_bytes < wl.total) { rs_set_error("workspace too small: need %lld bytes", (long long)wl.total); return RS_ERR_WORKSPACE; }
    uint8_t *wk = (uint8_t *)d_work + wl.off_lut;
    return alphabet == 4 ? onehot_finish<4>(d_codes, n, table, W, threshold, true, hit_capacity, d_hit_pos,
                                            (float *)d_hit_score, nullptr, d_counters2, wk, st)
                         : onehot_finish<7>(d_codes, n, table, W, threshold, true, hit_capacity, d_hit_pos, nullptr,
                                            (double *)d_hit_score, d_counters2, wk, st);
}

// Two-stream AND scan (two-FASTA RNASS mode), W <= 16.
int rs_scan_pair_masks(const uint8_t *d_seq_codes, const uint8_t *d_struct_codes, int64_t n, const double *seq_table,
                       const double *struct_table, int W, double threshold, int64_t cap, int64_t *d_hit_pos,
                       float *d_hit_seq, double *d_hit_str, uint64_t *d_counters2, void *d_work, cudaStream_t st)
{
    WorkLayout wl = rs_work_layout(n, cap);
    MaskScanParams prm = {};
    prm.codes = d_seq_codes; prm.codes_b = d_struct_codes; prm.n = n; prm.padded = rs_padded_count(n);
    prm.threshold = threshold;
    prm.n_tiles = (n + MS_TILE - 1) / MS_TILE;
    const int64_t n_segs = prm.n_tiles * (MS_THREADS / 32);
    const int n_blocks = fin_ctas(n_segs);
    carve_work((uint8_t *)d_work + wl.off_lut, n_segs * 32, n_segs, n_blocks, prm.wk);
    RS_CUDA(fin_arm(prm.wk, n_blocks, st));
    for (int j = 0; j < W; j++)
        for (int c = 0; c < 8; c++) {
            prm.ta[j * 8 + c] = c < 4 ? seq_table[j * 4 + c] : 0.0;
            prm.tb[j * 8 + c] = c < 7 ? struct_table[j * 7 + c] : 0.0;
        }
    int rc = dispatch_mask_scan<4>(W, prm, st);
    if (rc) return rc;
    return finish_mask_scan<4>(d_seq_codes, prm.wk, n_segs, n_blocks, 32, seq_table, W, cap, d_hit_pos, d_hit_seq,
                               d_hit_str, d_counters2, st, d_struct_codes, struct_table);
}
