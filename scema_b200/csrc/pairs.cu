// K2 + K3 — all-pairs L2 distance between resampled histories, thresholded, compacted (sm_100a).
//
// Replaces the double loop of compare_histories_with_all_ranks (reference
// headers/strain2spline.h:603-611, and the MPI ring :571-599) that calls compare_L2_norm
// (:469-484) and choose_most_similar_history (:265-274, strict `diff < threshold`).
//
// Design (DESIGN.md "K2"):
//  * k_filter<..>: GEMM-form filter. For a 128x128 tile of the pair matrix it evaluates
//        acc = a.b - (|a|^2 + |b|^2)/2  ( = -d^2/2 )
//    as an FP64 dense contraction — DMMA (mma.sync m8n8k4 f64, the only FP64 tensor shape sm_100a
//    has in SASS) or, for comparison, CUDA-core DFMA register tiles — over operand tiles staged
//    into shared memory by the TMA engine (cp.async.bulk + mbarrier, double buffered), and
//    rejects every pair that PROVABLY fails the threshold: -2*acc > T_tile, where T_tile is
//    thr^2 widened by a rigorous rounding-error band that scales with the row norms.
//    Everything else (true edges plus a guard band around the threshold) is a survivor.
//  * Survivors go through a warp-aggregated atomic append into a candidate queue (K3 pattern).
//  * k_exact_queue recomputes every survivor by direct differences in the reference's exact
//    operation order (sequential k, separate multiply and add, IEEE sqrt) and appends the edges
//    (key = a<<shift|b, diff) with warp-aggregated atomics. Every emitted distance therefore
//    carries the reference's bits and the edge SET is identical to the reference's.
//  * k_exact_all is the filter-free anchor (SCEMA_PAIRS_EXACT) and the fallback when survivors
//    are too dense for a queue.
//  * The edge list is put in canonical (a,b) order with a radix sort on the packed key.
#include "common.cuh"
#include <cub/device/device_radix_sort.cuh>
#include <cmath>
#include <algorithm>
#include <functional>

namespace scema {

// ------------------------------------------------------------------------------------------------
// small PTX helpers (mbarrier + 1-D bulk tensor-memory-accelerator copies)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    while (!mbar_try_wait(bar, parity)) {}
}
// global -> shared bulk copy executed by the TMA engine (SASS: UBLKCP), completion on an mbarrier
__device__ __forceinline__ void tma_bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void dmma_m8n8k4(double &c0, double &c1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// K3: warp-aggregated append. All 32 lanes must call. Returns nothing; drops (but still counts)
// entries beyond cap so the host can detect overflow and retry with a larger buffer.
__device__ __forceinline__ void warp_append_edge(bool keep, uint64_t key, double val, unsigned long long *counter,
                                                 uint64_t cap, uint64_t *keys, double *vals)
{
    unsigned m = __ballot_sync(0xffffffffu, keep);
    if (m == 0) return;
    int lane = threadIdx.x & 31;
    int leader = __ffs(m) - 1;
    unsigned long long base = 0;
    if (lane == leader) base = atomicAdd(counter, (unsigned long long)__popc(m));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (keep) {
        uint64_t pos = base + __popc(m & ((1u << lane) - 1));
        if (pos < cap) { keys[pos] = key; vals[pos] = val; }
    }
}
__device__ __forceinline__ void warp_append_cand(bool keep, uint64_t packed, unsigned long long *counter, uint64_t cap,
                                                 uint64_t *queue)
{
    unsigned m = __ballot_sync(0xffffffffu, keep);
    if (m == 0) return;
    int lane = threadIdx.x & 31;
    int leader = __ffs(m) - 1;
    unsigned long long base = 0;
    if (lane == leader) base = atomicAdd(counter, (unsigned long long)__popc(m));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (keep) {
        uint64_t pos = base + __popc(m & ((1u << lane) - 1));
        if (pos < cap) queue[pos] = packed;
    }
}

// ------------------------------------------------------------------------------------------------
// prep: S[n][K] -> F[chunk][n_pad][ks] (zero padded), HN[n_pad] = -|row|^2/2, BM[block] = max |row|^2
// one warp per row
// ------------------------------------------------------------------------------------------------
// The last chunk may be narrower (kt columns, row stride kst) than the others (kc, ks).
__global__ void __launch_bounds__(256) k_prep(const double *__restrict__ S, uint64_t n, uint32_t K, uint64_t n_pad,
                                              uint32_t kc, uint32_t ks, uint32_t kt, uint32_t kst, uint32_t n_chunks,
                                              double *__restrict__ F, double *__restrict__ HN,
                                              unsigned long long *__restrict__ BM)
{
    const uint64_t row = (uint64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= n_pad) return;
    double nrm = 0.0;
    for (uint32_t c = 0; c < n_chunks; c++) {
        const bool tail = c == n_chunks - 1;
        const uint32_t w = tail ? kt : kc, st = tail ? kst : ks;
        double *dst = F + (uint64_t)c * n_pad * ks + row * st;
        for (uint32_t q = lane; q < st; q += 32) {
            uint32_t k = c * kc + q;
            double v = 0.0;
            if (q < w && k < K && row < n) v = S[row * K + k];
            dst[q] = v;
            nrm = fma(v, v, nrm);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) nrm += __shfl_xor_sync(0xffffffffu, nrm, o);
    if (lane == 0) {
        HN[row] = row < n ? -0.5 * nrm : -INFINITY;
        if (row < n) atomicMax(BM + row / TILE, (unsigned long long)__double_as_longlong(nrm));
    }
}

// ------------------------------------------------------------------------------------------------
// filter kernel
// ------------------------------------------------------------------------------------------------
struct FilterArgs {
    const double *F;           // [n_chunks][n_pad][KS]
    const double *HN;          // [n_pad]
    const double *BM;          // [n_blocks]
    const uint64_t *panel_start;  // [n_panels+1] prefix of strip groups
    unsigned long long *work_counter;
    unsigned long long *cand_count;
    uint64_t *cand;
    uint64_t cand_cap;
    uint64_t n, n_pad;
    uint32_t n_blocks, n_panels, n_chunks, strip_len;
    uint64_t n_groups_local;  // strip groups of this launch owned by this shard ...
    uint64_t lg_first;        // ... starting at this shard-local group index (group = local * n_shards + shard)
    uint32_t shard, n_shards;
    double T0, cband;
};

template <int KC, int KS, bool MULTI>
struct FilterSmem {
    static constexpr int A_BUFS = MULTI ? 2 : 1;
    static constexpr size_t tile_doubles = (size_t)TILE * KS;
    static constexpr size_t bytes = (A_BUFS + 2) * tile_doubles * 8 + (TILE + 2 * TILE) * 8 + 64;
};

template <int KC, int KS, bool MULTI, bool DMMA>
__global__ void __launch_bounds__(256, 1) k_filter(const FilterArgs a)
{
    using SM = FilterSmem<KC, KS, MULTI>;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double *As = reinterpret_cast<double *>(smem_raw);
    double *Bs = As + SM::A_BUFS * SM::tile_doubles;
    double *hA = Bs + 2 * SM::tile_doubles;
    double *hB = hA + TILE;
    uint64_t *bars = reinterpret_cast<uint64_t *>(hB + 2 * TILE);
    __shared__ unsigned long long s_item;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr uint32_t TILE_BYTES = (uint32_t)(SM::tile_doubles * 8);
    constexpr uint32_t HN_BYTES = TILE * 8;

    if (tid == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    uint32_t uses0 = 0, uses1 = 0;

    // thread -> accumulator mapping
    // DMMA: 8 warps as 2 (rows) x 4 (cols); warp tile 64 x 32 = 8 x 4 m8n8 fragments.
    //       fragment element e of (mi,ni): row = mi*8 + (lane>>2), col = ni*8 + 2*(lane&3) + e
    // FMA : 16 x 16 threads, each 8 x 8 pairs: row = ty + 16*mi, col = tx + 16*ni
    const int g = lane >> 2, t4 = lane & 3;
    const int wm = warp >> 2, wn = warp & 3;
    const int ty = tid >> 4, tx = tid & 15;

    while (true) {
        __syncthreads();  // s_item and all smem buffers are free again
        if (tid == 0) s_item = atomicAdd(a.work_counter, 1ull);
        __syncthreads();
        const uint64_t item = s_item;
        if (item >= a.n_groups_local * PANEL_ROWBLOCKS) break;
        const uint64_t grp = (a.lg_first + item / PANEL_ROWBLOCKS) * a.n_shards + a.shard;
        const uint32_t r = (uint32_t)(item % PANEL_ROWBLOCKS);
        // binary search: panel with panel_start[p] <= grp < panel_start[p+1]
        uint32_t lo = 0, hi = a.n_panels;
        while (hi - lo > 1) {
            uint32_t mid = (lo + hi) >> 1;
            if (a.panel_start[mid] <= grp) lo = mid; else hi = mid;
        }
        const uint32_t panel = lo;
        const uint32_t strip = (uint32_t)(grp - a.panel_start[panel]);
        const uint32_t I = panel * PANEL_ROWBLOCKS + r;
        if (I >= a.n_blocks) continue;
        uint32_t J0 = panel * PANEL_ROWBLOCKS + strip * a.strip_len;
        uint32_t J1 = J0 + a.strip_len;
        if (J1 > a.n_blocks) J1 = a.n_blocks;
        if (J0 < I) J0 = I;
        if (J0 >= J1) continue;
        const uint32_t n_tiles = J1 - J0;
        const uint32_t n_steps = n_tiles * a.n_chunks;
        const double bmI = a.BM[I];

        auto issue = [&](uint32_t q) {
            const uint32_t st = q & 1;
            const uint32_t jt = q / a.n_chunks, c = q - jt * a.n_chunks;
            const uint32_t J = J0 + jt;
            uint32_t bytes = TILE_BYTES;
            if (c == 0) bytes += HN_BYTES;
            if (MULTI) bytes += TILE_BYTES;
            if (q == 0) bytes += HN_BYTES + (MULTI ? 0u : TILE_BYTES);
            mbar_expect_tx(&bars[st], bytes);
            tma_bulk_g2s(Bs + st * SM::tile_doubles, a.F + ((uint64_t)c * a.n_pad + (uint64_t)J * TILE) * KS, TILE_BYTES,
                         &bars[st]);
            if (c == 0) tma_bulk_g2s(hB + st * TILE, a.HN + (uint64_t)J * TILE, HN_BYTES, &bars[st]);
            if (MULTI)
                tma_bulk_g2s(As + st * SM::tile_doubles, a.F + ((uint64_t)c * a.n_pad + (uint64_t)I * TILE) * KS,
                             TILE_BYTES, &bars[st]);
            if (q == 0) {
                tma_bulk_g2s(hA, a.HN + (uint64_t)I * TILE, HN_BYTES, &bars[st]);
                if (!MULTI) tma_bulk_g2s(As, a.F + (uint64_t)I * TILE * KS, TILE_BYTES, &bars[st]);
            }
        };

        if (tid == 0) issue(0);

        double acc[8][4][2];  // DMMA: [mi][ni][e]; FMA: [mi][ni*2+e] viewed as 8x8

        for (uint32_t q = 0; q < n_steps; q++) {
            const uint32_t st = q & 1;
            const uint32_t jt = q / a.n_chunks, c = q - jt * a.n_chunks;
            if (q + 1 < n_steps && tid == 0) issue(q + 1);
            if (st == 0) { mbar_wait(&bars[0], uses0 & 1); uses0++; }
            else         { mbar_wait(&bars[1], uses1 & 1); uses1++; }

            const double *Ab = MULTI ? As + st * SM::tile_doubles : As;
            const double *Bb = Bs + st * SM::tile_doubles;

            if (c == 0) {
                // acc starts at -(|a|^2+|b|^2)/2 so that after the contraction acc = -d^2/2
                const double *hb = hB + st * TILE;
                if (DMMA) {
#pragma unroll
                    for (int mi = 0; mi < 8; mi++) {
                        const double ha = hA[wm * 64 + mi * 8 + g];
#pragma unroll
                        for (int ni = 0; ni < 4; ni++) {
                            acc[mi][ni][0] = ha + hb[wn * 32 + ni * 8 + 2 * t4];
                            acc[mi][ni][1] = ha + hb[wn * 32 + ni * 8 + 2 * t4 + 1];
                        }
                    }
                } else {
#pragma unroll
                    for (int mi = 0; mi < 8; mi++) {
                        const double ha = hA[ty + 16 * mi];
#pragma unroll
                        for (int ni = 0; ni < 8; ni++) acc[mi][ni >> 1][ni & 1] = ha + hb[tx + 16 * ni];
                    }
                }
            }

            if (DMMA) {
                const double *ap = Ab + (wm * 64 + g) * KS + t4;
                const double *bp = Bb + (wn * 32 + g) * KS + t4;
#pragma unroll
                for (int ks = 0; ks < KC / 4; ks++) {
                    double af[8], bf[4];
#pragma unroll
                    for (int mi = 0; mi < 8; mi++) af[mi] = ap[mi * 8 * KS + ks * 4];
#pragma unroll
                    for (int ni = 0; ni < 4; ni++) bf[ni] = bp[ni * 8 * KS + ks * 4];
#pragma unroll
                    for (int mi = 0; mi < 8; mi++)
#pragma unroll
                        for (int ni = 0; ni < 4; ni++) dmma_m8n8k4(acc[mi][ni][0], acc[mi][ni][1], af[mi], bf[ni]);
                }
            } else {
                const double *ap = Ab + ty * KS;
                const double *bp = Bb + tx * KS;
#pragma unroll 4
                for (int k = 0; k < KC; k++) {
                    double af[8], bf[8];
#pragma unroll
                    for (int mi = 0; mi < 8; mi++) af[mi] = ap[mi * 16 * KS + k];
#pragma unroll
                    for (int ni = 0; ni < 8; ni++) bf[ni] = bp[ni * 16 * KS + k];
#pragma unroll
                    for (int mi = 0; mi < 8; mi++)
#pragma unroll
                        for (int ni = 0; ni < 8; ni++)
                            acc[mi][ni >> 1][ni & 1] = fma(af[mi], bf[ni], acc[mi][ni >> 1][ni & 1]);
                }
            }

            if (c == a.n_chunks - 1) {
                // ---- epilogue: provable rejection, survivors to the queue
                const uint32_t J = J0 + jt;
                const double T = (a.T0 + a.cband * (bmI + a.BM[J])) * (1.0 + 1e-15);
                const double negHalfT = -0.5 * T;
                bool any = false;
#pragma unroll
                for (int mi = 0; mi < 8; mi++)
#pragma unroll
                    for (int ni = 0; ni < 4; ni++) {
                        any |= !(acc[mi][ni][0] < negHalfT);
                        any |= !(acc[mi][ni][1] < negHalfT);
                    }
                if (__any_sync(0xffffffffu, any)) {
                    const uint64_t rbase = (uint64_t)I * TILE, cbase = (uint64_t)J * TILE;
#pragma unroll
                    for (int mi = 0; mi < 8; mi++)
#pragma unroll
                        for (int ni = 0; ni < 4; ni++)
#pragma unroll
                            for (int e = 0; e < 2; e++) {
                                uint64_t row, col;
                                if (DMMA) {
                                    row = rbase + wm * 64 + mi * 8 + g;
                                    col = cbase + wn * 32 + ni * 8 + 2 * t4 + e;
                                } else {
                                    row = rbase + ty + 16 * mi;
                                    col = cbase + tx + 16 * (ni * 2 + e);
                                }
                                const bool keep = !(acc[mi][ni][e] < negHalfT) && row < col && col < a.n;
                                warp_append_cand(keep, (row << 32) | col, a.cand_count, a.cand_cap, a.cand);
                            }
                }
            }
            __syncthreads();  // stage st may be refilled by the issue of the next iteration
        }
    }
}

// ------------------------------------------------------------------------------------------------
// filter kernel, warp-specialised (K2 v2, DMMA only)
//
// Same tiles, same arithmetic and same rejection rule as k_filter<.., DMMA=true>, different
// choreography: warp 8 is a producer (one lane: work queue, threshold per tile, TMA bulk copies),
// warps 0-7 are consumers. Stages are handed over with full/empty mbarriers instead of CTA-wide
// barriers, so a warp that finishes a tile starts the next one without waiting for the slowest warp
// and the two warps of a scheduler partition drift apart: one warp's epilogue and accumulator
// set-up overlap the other's DMMAs. The epilogue compares in the integer pipe (DMMA and every other
// FP64 instruction share one pipe — tools/fp64_peak.cu: DMMA + DFMA never exceeds 36.8 TFLOP/s): for
// a negative bound the test acc < bound is implied by hi32(acc) > hi32(bound) as unsigned integers,
// and pairs that only differ in the low word (2^-20 relative) simply stay survivors.
// ------------------------------------------------------------------------------------------------
struct StageMeta {
    uint32_t I, J, flags, lo_bound, span, pad0, pad1, pad2;
};
constexpr uint32_t META_FIRST = 1u, META_LAST = 2u, META_DONE = 4u;  // LAST also means: this is the (narrower) tail chunk

// KC = columns of a chunk, KT = columns of the last chunk (KT <= KC; KT == KC when there is one chunk)
template <int KC, bool MULTI>
struct WsSmem {
    static constexpr size_t tile_bytes = (size_t)TILE * KC * 8;
    static constexpr size_t stage_bytes = (MULTI ? 2 : 1) * tile_bytes + 2 * TILE * 8;  // [A] B hA hB
    static constexpr size_t fixed_bytes = (MULTI ? 0 : tile_bytes) + 1024;
    static constexpr size_t budget = 227 * 1024;
    static constexpr int raw_stages = (int)((budget - fixed_bytes) / stage_bytes);
    static constexpr int NST = raw_stages >= 4 ? 4 : (raw_stages >= 2 ? 2 : 1);  // power of two
    static constexpr size_t bytes = fixed_bytes + NST * stage_bytes;
};

__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// Register budget: 12 warps = 2 consumer warpgroups + 1 producer warpgroup (only its first warp
// works). Every scheduler partition hosts 2 consumer warps and 1 producer-group warp and owns 16384
// registers, so the kernel is compiled for 168 registers/thread and re-balanced at run time with
// setmaxnreg: producer group down to 40, consumers up to 232 (32*(2*232+40) = 16128).
// 64 x 32 warp tile += A[64 x KK] . B[32 x KK]^T out of shared memory (row stride KK, KK % 8 == 4)
template <int KK>
__device__ __forceinline__ void mma_warp_tile(double (&acc)[8][4][2], const double *__restrict__ ap, const double *__restrict__ bp)
{
#pragma unroll
    for (int ks = 0; ks < KK / 4; ks++) {
        double af[8], bf[4];
#pragma unroll
        for (int mi = 0; mi < 8; mi++) af[mi] = ap[mi * 8 * KK + ks * 4];
#pragma unroll
        for (int ni = 0; ni < 4; ni++) bf[ni] = bp[ni * 8 * KK + ks * 4];
#pragma unroll
        for (int mi = 0; mi < 8; mi++)
#pragma unroll
            for (int ni = 0; ni < 4; ni++) dmma_m8n8k4(acc[mi][ni][0], acc[mi][ni][1], af[mi], bf[ni]);
    }
}

template <int KC, int KT, bool MULTI>
__global__ void __launch_bounds__(384, 1) k_filter_ws(const FilterArgs a)
{
    using SM = WsSmem<KC, MULTI>;
    constexpr int NST = SM::NST;
    static_assert(NST >= 2, "need at least two stages");
    static_assert(KT <= KC && (MULTI || KT == KC), "tail chunk");
    constexpr int KS = KC;
    constexpr uint32_t TILE_BYTES = (uint32_t)SM::tile_bytes;
    constexpr uint32_t TAIL_BYTES = (uint32_t)((size_t)TILE * KT * 8);
    constexpr uint32_t HN_BYTES = TILE * 8;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    // layout: [resident A (non-MULTI)] | stage 0 | stage 1 | ... | meta[NST] | full[NST] | empty[NST]
    double *As = reinterpret_cast<double *>(smem_raw);
    unsigned char *stage0 = smem_raw + (MULTI ? 0 : SM::tile_bytes);
    StageMeta *metas = reinterpret_cast<StageMeta *>(stage0 + NST * SM::stage_bytes);
    uint64_t *full = reinterpret_cast<uint64_t *>(metas + NST);
    uint64_t *empty = full + NST;
    auto stageA = [&](int st) { return reinterpret_cast<double *>(stage0 + st * SM::stage_bytes); };
    auto stageB = [&](int st) { return reinterpret_cast<double *>(stage0 + st * SM::stage_bytes + (MULTI ? SM::tile_bytes : 0)); };
    auto stageHA = [&](int st) { return stageB(st) + (size_t)TILE * KS; };
    auto stageHB = [&](int st) { return stageHA(st) + TILE; };

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        for (int s = 0; s < NST; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], 8); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (warp >= 8) {
        // ------------------------------------------------------------------ producer (one lane)
        asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
        if (warp != 8 || lane != 0) return;
        uint32_t t = 0, ephase = (1u << NST) - 1u;  // a fresh barrier passes a parity-1 wait
        const uint64_t total = a.n_groups_local * PANEL_ROWBLOCKS;
        while (true) {
            const uint64_t item = atomicAdd(a.work_counter, 1ull);
            if (item >= total) break;
            const uint64_t grp = (a.lg_first + item / PANEL_ROWBLOCKS) * a.n_shards + a.shard;
            const uint32_t r = (uint32_t)(item % PANEL_ROWBLOCKS);
            uint32_t lo = 0, hi = a.n_panels;
            while (hi - lo > 1) {
                uint32_t mid = (lo + hi) >> 1;
                if (a.panel_start[mid] <= grp) lo = mid; else hi = mid;
            }
            const uint32_t panel = lo;
            const uint32_t strip = (uint32_t)(grp - a.panel_start[panel]);
            const uint32_t I = panel * PANEL_ROWBLOCKS + r;
            if (I >= a.n_blocks) continue;
            uint32_t J0 = panel * PANEL_ROWBLOCKS + strip * a.strip_len;
            uint32_t J1 = J0 + a.strip_len;
            if (J1 > a.n_blocks) J1 = a.n_blocks;
            if (J0 < I) J0 = I;
            if (J0 >= J1) continue;
            const double bmI = a.BM[I];
            for (uint32_t J = J0; J < J1; J++) {
                // rejection bound of the tile, as an unsigned range test on the high word
                const double T = (a.T0 + a.cband * (bmI + a.BM[J])) * (1.0 + 1e-15);
                const double negHalfT = -0.5 * T;
                uint32_t lo_bound = 0, span = 0;
                {
                    const uint32_t h = (uint32_t)__double2hiint(negHalfT);
                    if (negHalfT <= 0.0 && h >= 0x80000000u && h < 0xFFF00000u) {  // negative (or -0), finite
                        lo_bound = h + 1u;
                        span = 0xFFF00000u - lo_bound;
                    }
                }
                for (uint32_t c = 0; c < a.n_chunks; c++, t++) {
                    const int st = (int)(t & (NST - 1));
                    mbar_wait(&empty[st], (ephase >> st) & 1u);
                    ephase ^= 1u << st;
                    const bool new_A = !MULTI && J == J0 && c == 0;
                    if (new_A)  // every earlier tile must have released the resident A tile
                        for (int o = 0; o < NST; o++)
                            if (o != st) mbar_wait(&empty[o], (ephase >> o) & 1u);  // peek, phase not consumed
                    StageMeta m;
                    m.I = I; m.J = J;
                    m.flags = (c == 0 ? META_FIRST : 0u) | (c == a.n_chunks - 1 ? META_LAST : 0u);
                    m.lo_bound = lo_bound; m.span = span; m.pad0 = m.pad1 = m.pad2 = 0;
                    metas[st] = m;
                    const bool tail = MULTI && c == a.n_chunks - 1;  // narrower last chunk: row stride KT
                    const uint32_t tb = tail ? TAIL_BYTES : TILE_BYTES;
                    const uint32_t kst = tail ? KT : KS;
                    const double *Fc = a.F + (uint64_t)c * a.n_pad * KS;
                    uint32_t bytes = tb + (c == 0 ? 2 * HN_BYTES : 0u);
                    if (MULTI || new_A) bytes += tb;
                    mbar_expect_tx(&full[st], bytes);
                    tma_bulk_g2s(stageB(st), Fc + (uint64_t)J * TILE * kst, tb, &full[st]);
                    if (c == 0) {
                        tma_bulk_g2s(stageHA(st), a.HN + (uint64_t)I * TILE, HN_BYTES, &full[st]);
                        tma_bulk_g2s(stageHB(st), a.HN + (uint64_t)J * TILE, HN_BYTES, &full[st]);
                    }
                    if (MULTI)
                        tma_bulk_g2s(stageA(st), Fc + (uint64_t)I * TILE * kst, tb, &full[st]);
                    else if (new_A)
                        tma_bulk_g2s(As, a.F + (uint64_t)I * TILE * KS, TILE_BYTES, &full[st]);
                }
            }
        }
        const int st = (int)(t & (NST - 1));
        mbar_wait(&empty[st], (ephase >> st) & 1u);
        StageMeta m = {};
        m.flags = META_DONE;
        metas[st] = m;
        mbar_arrive(&full[st]);
        return;
    }

    // ---------------------------------------------------------------------- consumers (8 warps)
    asm volatile("setmaxnreg.inc.sync.aligned.u32 232;");
    // 2 (rows) x 4 (cols) warps; warp tile 64 x 32 = 8 x 4 m8n8 fragments;
    // fragment element e of (mi,ni): row = mi*8 + (lane>>2), col = ni*8 + 2*(lane&3) + e
    const int g = lane >> 2, t4 = lane & 3;
    const int wm = warp >> 2, wn = warp & 3;
    double acc[8][4][2];
    uint32_t t = 0, fphase = 0;
    while (true) {
        const int st = (int)(t & (NST - 1));
        mbar_wait(&full[st], (fphase >> st) & 1u);
        fphase ^= 1u << st;
        t++;
        const StageMeta m = metas[st];
        if (m.flags & META_DONE) break;
        const double *Ab = MULTI ? stageA(st) : As;
        const double *Bb = stageB(st);
        if (m.flags & META_FIRST) {
            // acc starts at -(|a|^2+|b|^2)/2 so that after the contraction acc = -d^2/2
            const double *ha = stageHA(st), *hb = stageHB(st);
#pragma unroll
            for (int mi = 0; mi < 8; mi++) {
                const double hav = ha[wm * 64 + mi * 8 + g];
#pragma unroll
                for (int ni = 0; ni < 4; ni++) {
                    acc[mi][ni][0] = hav + hb[wn * 32 + ni * 8 + 2 * t4];
                    acc[mi][ni][1] = hav + hb[wn * 32 + ni * 8 + 2 * t4 + 1];
                }
            }
        }
        if (KT != KC && (m.flags & META_LAST))
            mma_warp_tile<KT>(acc, Ab + (wm * 64 + g) * KT + t4, Bb + (wn * 32 + g) * KT + t4);
        else
            mma_warp_tile<KC>(acc, Ab + (wm * 64 + g) * KC + t4, Bb + (wn * 32 + g) * KC + t4);
        // this warp is done with the stage's shared memory (and, at the last tile of an item, with A)
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[st]);

        if (m.flags & META_LAST) {
            // ---- epilogue: provable rejection (integer range test), survivors to the queue
            bool any = false;
#pragma unroll
            for (int mi = 0; mi < 8; mi++)
#pragma unroll
                for (int ni = 0; ni < 4; ni++) {
                    any |= ((uint32_t)__double2hiint(acc[mi][ni][0]) - m.lo_bound) >= m.span;
                    any |= ((uint32_t)__double2hiint(acc[mi][ni][1]) - m.lo_bound) >= m.span;
                }
            if (__any_sync(0xffffffffu, any)) {
                const uint64_t rbase = (uint64_t)m.I * TILE, cbase = (uint64_t)m.J * TILE;
#pragma unroll
                for (int mi = 0; mi < 8; mi++)
#pragma unroll
                    for (int ni = 0; ni < 4; ni++)
#pragma unroll
                        for (int e = 0; e < 2; e++) {
                            const uint64_t row = rbase + wm * 64 + mi * 8 + g;
                            const uint64_t col = cbase + wn * 32 + ni * 8 + 2 * t4 + e;
                            const bool keep = (((uint32_t)__double2hiint(acc[mi][ni][e]) - m.lo_bound) >= m.span) &&
                                              row < col && col < a.n;
                            warp_append_cand(keep, (row << 32) | col, a.cand_count, a.cand_cap, a.cand);
                        }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// exact recompute of the survivors + K3 compaction of the edges
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_exact_queue(const double *__restrict__ S, uint32_t K, const uint64_t *__restrict__ cand,
                                                     const unsigned long long *__restrict__ cand_count, uint64_t cand_cap,
                                                     double thr, uint32_t key_shift, unsigned long long *edge_count,
                                                     uint64_t edge_cap, uint64_t *__restrict__ keys, double *__restrict__ vals)
{
    uint64_t n_c = *cand_count;
    if (n_c > cand_cap) n_c = cand_cap;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const uint64_t rounds = (n_c + stride - 1) / stride;
    for (uint64_t rd = 0; rd < rounds; rd++) {
        const uint64_t idx = rd * stride + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
        bool keep = false;
        uint64_t key = 0;
        double d = 0.0;
        if (idx < n_c) {
            const uint64_t pk = cand[idx];
            const uint64_t i = pk >> 32, j = pk & 0xffffffffull;
            d = exact_l2(S + i * K, S + j * K, K);
            keep = d < thr;  // strict, strain2spline.h:272
            key = (i << key_shift) | j;
        }
        warp_append_edge(keep, key, d, edge_count, edge_cap, keys, vals);
    }
}

// Filter-free all-pairs kernel: 64x64 pair tiles, 4x4 pairs per thread, K streamed through shared
// memory in chunks while the per-pair sums keep the reference's sequential-k order.
constexpr int XT = 64, XKC = 32;
__global__ void __launch_bounds__(256) k_exact_all(const double *__restrict__ S, uint64_t n, uint32_t K, double thr,
                                                   uint32_t key_shift, uint32_t shard, uint32_t n_shards, uint32_t I_first,
                                                   unsigned long long *edge_count, uint64_t edge_cap,
                                                   uint64_t *__restrict__ keys, double *__restrict__ vals)
{
    const uint32_t I = I_first + blockIdx.y, J = blockIdx.x;
    if (J < I) return;
    if (((uint64_t)I + J) % n_shards != shard) return;
    __shared__ double As[XT][XKC + 1], Bs[XT][XKC + 1];
    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
    double sum[4][4];
#pragma unroll
    for (int p = 0; p < 4; p++)
#pragma unroll
        for (int q = 0; q < 4; q++) sum[p][q] = 0.0;
    const uint64_t r0 = (uint64_t)I * XT, c0 = (uint64_t)J * XT;
    for (uint32_t k0 = 0; k0 < K; k0 += XKC) {
        const uint32_t kn = K - k0 < (uint32_t)XKC ? K - k0 : (uint32_t)XKC;
        __syncthreads();
        for (int e = tid; e < XT * XKC; e += 256) {
            const int rr = e / XKC, kk = e - rr * XKC;
            double va = 0.0, vb = 0.0;
            if ((uint32_t)kk < kn) {
                if (r0 + rr < n) va = S[(r0 + rr) * K + k0 + kk];
                if (c0 + rr < n) vb = S[(c0 + rr) * K + k0 + kk];
            }
            As[rr][kk] = va;
            Bs[rr][kk] = vb;
        }
        __syncthreads();
        for (uint32_t kk = 0; kk < kn; kk++) {
            double av[4], bv[4];
#pragma unroll
            for (int p = 0; p < 4; p++) av[p] = As[ty + 16 * p][kk];
#pragma unroll
            for (int q = 0; q < 4; q++) bv[q] = Bs[tx + 16 * q][kk];
#pragma unroll
            for (int p = 0; p < 4; p++)
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    const double diff = __dsub_rn(av[p], bv[q]);
                    sum[p][q] = __dadd_rn(sum[p][q], __dmul_rn(diff, diff));
                }
        }
    }
#pragma unroll
    for (int p = 0; p < 4; p++)
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const uint64_t row = r0 + ty + 16 * p, col = c0 + tx + 16 * q;
            const double d = __dsqrt_rn(sum[p][q]);
            const bool keep = row < col && col < n && d < thr;
            warp_append_edge(keep, (row << key_shift) | col, d, edge_count, edge_cap, keys, vals);
        }
}

// Legacy nearest neighbour of every history (choose_most_similar_history, strain2spline.h:277-289: the smallest
// distance to ANY other history, ties to the lowest ID, NaN distances ignored) without the O(N^2) lists: the tiles of
// k_exact_all, PASS 1 keeps the smallest distance per row (non-negative doubles order as unsigned integers),
// PASS 2 the lowest ID among the histories at exactly that distance.
template <int PASS>
__global__ void __launch_bounds__(256) k_nearest(const double *__restrict__ S, uint64_t n, uint32_t K, const uint32_t *__restrict__ ids,
                                                 uint32_t I_first, unsigned long long *__restrict__ minbits,
                                                 unsigned int *__restrict__ minid)
{
    const uint32_t I = I_first + blockIdx.y, J = blockIdx.x;
    if (J < I) return;
    __shared__ double As[XT][XKC + 1], Bs[XT][XKC + 1];
    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
    double sum[4][4];
#pragma unroll
    for (int p = 0; p < 4; p++)
#pragma unroll
        for (int q = 0; q < 4; q++) sum[p][q] = 0.0;
    const uint64_t r0 = (uint64_t)I * XT, c0 = (uint64_t)J * XT;
    for (uint32_t k0 = 0; k0 < K; k0 += XKC) {
        const uint32_t kn = K - k0 < (uint32_t)XKC ? K - k0 : (uint32_t)XKC;
        __syncthreads();
        for (int e = tid; e < XT * XKC; e += 256) {
            const int rr = e / XKC, kk = e - rr * XKC;
            double va = 0.0, vb = 0.0;
            if ((uint32_t)kk < kn) {
                if (r0 + rr < n) va = S[(r0 + rr) * K + k0 + kk];
                if (c0 + rr < n) vb = S[(c0 + rr) * K + k0 + kk];
            }
            As[rr][kk] = va;
            Bs[rr][kk] = vb;
        }
        __syncthreads();
        for (uint32_t kk = 0; kk < kn; kk++) {
            double av[4], bv[4];
#pragma unroll
            for (int p = 0; p < 4; p++) av[p] = As[ty + 16 * p][kk];
#pragma unroll
            for (int q = 0; q < 4; q++) bv[q] = Bs[tx + 16 * q][kk];
#pragma unroll
            for (int p = 0; p < 4; p++)
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    const double diff = __dsub_rn(av[p], bv[q]);
                    sum[p][q] = __dadd_rn(sum[p][q], __dmul_rn(diff, diff));
                }
        }
    }
#pragma unroll
    for (int p = 0; p < 4; p++)
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const uint64_t row = r0 + ty + 16 * p, col = c0 + tx + 16 * q;
            const double d = __dsqrt_rn(sum[p][q]);
            if (!(row < col && col < n) || d != d) continue;
            const unsigned long long bits = (unsigned long long)__double_as_longlong(d);
            if (PASS == 1) {
                atomicMin(minbits + row, bits);
                atomicMin(minbits + col, bits);
            } else {
                if (bits == minbits[row]) atomicMin(minid + row, ids[col]);
                if (bits == minbits[col]) atomicMin(minid + col, ids[row]);
            }
        }
}

int nearest_run(scema_ctx *ctx, uint32_t *nearest_id_host, double *nearest_diff_host)
{
    if (!ctx->have_spline) return fail(ctx, SCEMA_ERR_STATE, "Spline is not up to date.");
    const uint64_t n = ctx->n;
    if (n == 0) return SCEMA_OK;
    { const int rcw = wait_rows(ctx); if (rcw) return rcw; }
    DevBuf d_ids, d_bits, d_minid;
    std::vector<unsigned long long> bits(n, 0x7ff0000000000000ull);  // +inf: also what the reference starts from (:256)
    int rc = SCEMA_OK;
    auto run = [&]() -> int {
        SCEMA_CUDA(ctx, d_ids.reserve(n * sizeof(uint32_t)));
        SCEMA_CUDA(ctx, d_bits.reserve(n * sizeof(unsigned long long)));
        SCEMA_CUDA(ctx, d_minid.reserve(n * sizeof(unsigned int)));
        SCEMA_CUDA(ctx, cudaMemcpyAsync(d_ids.p, ids_of(ctx).data(), n * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
        SCEMA_CUDA(ctx, cudaMemcpyAsync(d_bits.p, bits.data(), n * sizeof(unsigned long long), cudaMemcpyHostToDevice, ctx->stream));
        SCEMA_CUDA(ctx, cudaMemsetAsync(d_minid.p, 0xff, n * sizeof(unsigned int), ctx->stream));
        const uint32_t nbx = (uint32_t)((n + XT - 1) / XT);
        for (int pass = 1; pass <= 2; pass++)
            for (uint32_t i0 = 0; i0 < nbx; i0 += 65535u) {
                const dim3 grid(nbx, std::min<uint32_t>(65535u, nbx - i0));
                if (pass == 1)
                    k_nearest<1><<<grid, 256, 0, ctx->stream>>>(ctx->d_spline, n, ctx->K, d_ids.as<uint32_t>(), i0,
                                                               d_bits.as<unsigned long long>(), d_minid.as<unsigned int>());
                else
                    k_nearest<2><<<grid, 256, 0, ctx->stream>>>(ctx->d_spline, n, ctx->K, d_ids.as<uint32_t>(), i0,
                                                               d_bits.as<unsigned long long>(), d_minid.as<unsigned int>());
                ctx->launches++;
            }
        SCEMA_CUDA(ctx, cudaGetLastError());
        if (nearest_diff_host)
            SCEMA_CUDA(ctx, cudaMemcpyAsync(nearest_diff_host, d_bits.p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        if (nearest_id_host)
            SCEMA_CUDA(ctx, cudaMemcpyAsync(nearest_id_host, d_minid.p, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        SCEMA_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        return SCEMA_OK;
    };
    rc = run();
    d_ids.release(); d_bits.release(); d_minid.release();
    return rc;
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
// Warp-specialised DMMA kernel: n-1 chunks of kc columns and a last one of kt <= kc, all from the
// bank-conflict-free widths (== 4 mod 8); least padding first, then fewest chunks.
static void choose_chunks_tail(uint32_t K, uint32_t *kc, uint32_t *kt, uint32_t *n_chunks)
{
    static const uint32_t widths[] = {12, 20, 28, 36, 44, 52, 60};
    for (uint32_t w : widths)
        if (K <= w) { *kc = w; *kt = w; *n_chunks = 1; return; }
    static const uint32_t mains[] = {36, 44, 52};
    uint64_t best_cost = ~0ull;
    for (uint32_t m : mains) {
        const uint32_t nn = (K + m - 1) / m;            // chunks when all but the last are m wide
        const uint32_t rest = K - (nn - 1) * m;         // 1 .. m columns left for the tail
        uint32_t t = m;
        for (uint32_t w : widths)
            if (w >= rest && w <= m) { t = w; break; }
        const uint64_t padded = (uint64_t)(nn - 1) * m + t;
        const uint64_t cost = padded * 64 + nn;          // padding dominates, chunk count breaks ties
        if (cost < best_cost) { best_cost = cost; *kc = m; *kt = t; *n_chunks = nn; }
    }
}

static void choose_chunks(uint32_t K, uint32_t *kc, uint32_t *n_chunks)
{
    static const uint32_t single[] = {12, 20, 28, 36, 44, 52, 60};
    for (uint32_t s : single)
        if (K <= s) { *kc = s; *n_chunks = 1; return; }
    static const uint32_t multi[] = {44, 52};
    uint32_t best_kc = 52, best_n = (K + 51) / 52;
    uint64_t best_pad = (uint64_t)best_kc * best_n;
    for (uint32_t m : multi) {
        uint32_t nn = (K + m - 1) / m;
        if ((uint64_t)m * nn < best_pad) { best_pad = (uint64_t)m * nn; best_kc = m; best_n = nn; }
    }
    *kc = best_kc; *n_chunks = best_n;
}

template <int KC, bool MULTI, bool DMMA>
static int launch_filter_t(scema_ctx *ctx, const FilterArgs &fa)
{
    constexpr int KS = DMMA ? KC : KC + 1;
    auto kern = k_filter<KC, KS, MULTI, DMMA>;
    const size_t smem = FilterSmem<KC, KS, MULTI>::bytes;
    if (smem > ctx->smem_optin) return fail(ctx, SCEMA_ERR_CUDA, "filter kernel shared memory exceeds device limit");
    SCEMA_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    uint64_t items = fa.n_groups_local * PANEL_ROWBLOCKS;
    unsigned grid = (unsigned)std::min<uint64_t>((uint64_t)ctx->sm_count, std::max<uint64_t>(items, 1));
    kern<<<grid, 256, smem, ctx->stream>>>(fa);
    ctx->launches++;
    SCEMA_CUDA(ctx, cudaGetLastError());
    return SCEMA_OK;
}

template <int KC, int KT, bool MULTI>
static int launch_filter_ws_t(scema_ctx *ctx, const FilterArgs &fa)
{
    auto kern = k_filter_ws<KC, KT, MULTI>;
    const size_t smem = WsSmem<KC, MULTI>::bytes;
    if (smem > ctx->smem_optin) return fail(ctx, SCEMA_ERR_CUDA, "filter kernel shared memory exceeds device limit");
    SCEMA_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    uint64_t items = fa.n_groups_local * PANEL_ROWBLOCKS;
    unsigned grid = (unsigned)std::min<uint64_t>((uint64_t)ctx->sm_count, std::max<uint64_t>(items, 1));
    kern<<<grid, 384, smem, ctx->stream>>>(fa);
    ctx->launches++;
    SCEMA_CUDA(ctx, cudaGetLastError());
    return SCEMA_OK;
}

template <int KC>
static int launch_filter_ws_tail(scema_ctx *ctx, const FilterArgs &fa, uint32_t kt)
{
    switch (kt) {
    case 12: if (12 <= KC) return launch_filter_ws_t<KC, (12 <= KC ? 12 : KC), true>(ctx, fa); break;
    case 20: if (20 <= KC) return launch_filter_ws_t<KC, (20 <= KC ? 20 : KC), true>(ctx, fa); break;
    case 28: if (28 <= KC) return launch_filter_ws_t<KC, (28 <= KC ? 28 : KC), true>(ctx, fa); break;
    case 36: if (36 <= KC) return launch_filter_ws_t<KC, (36 <= KC ? 36 : KC), true>(ctx, fa); break;
    case 44: if (44 <= KC) return launch_filter_ws_t<KC, (44 <= KC ? 44 : KC), true>(ctx, fa); break;
    case 52: if (52 <= KC) return launch_filter_ws_t<KC, (52 <= KC ? 52 : KC), true>(ctx, fa); break;
    }
    return fail(ctx, SCEMA_ERR_INVALID, "no filter kernel instantiation for this tail chunk size");
}

static int launch_filter_ws(scema_ctx *ctx, const FilterArgs &fa, uint32_t kc, uint32_t kt, bool multi)
{
    if (!multi) {
        switch (kc) {
        case 12: return launch_filter_ws_t<12, 12, false>(ctx, fa);
        case 20: return launch_filter_ws_t<20, 20, false>(ctx, fa);
        case 28: return launch_filter_ws_t<28, 28, false>(ctx, fa);
        case 36: return launch_filter_ws_t<36, 36, false>(ctx, fa);
        case 44: return launch_filter_ws_t<44, 44, false>(ctx, fa);
        case 52: return launch_filter_ws_t<52, 52, false>(ctx, fa);
        case 60: return launch_filter_ws_t<60, 60, false>(ctx, fa);
        }
    } else {
        switch (kc) {
        case 36: return launch_filter_ws_tail<36>(ctx, fa, kt);
        case 44: return launch_filter_ws_tail<44>(ctx, fa, kt);
        case 52: return launch_filter_ws_tail<52>(ctx, fa, kt);
        }
    }
    return fail(ctx, SCEMA_ERR_INVALID, "no filter kernel instantiation for this chunk size");
}

template <bool DMMA>
static int launch_filter(scema_ctx *ctx, const FilterArgs &fa, uint32_t kc, bool multi)
{
    if (!multi) {
        switch (kc) {
        case 12: return launch_filter_t<12, false, DMMA>(ctx, fa);
        case 20: return launch_filter_t<20, false, DMMA>(ctx, fa);
        case 28: return launch_filter_t<28, false, DMMA>(ctx, fa);
        case 36: return launch_filter_t<36, false, DMMA>(ctx, fa);
        case 44: return launch_filter_t<44, false, DMMA>(ctx, fa);
        case 52: return launch_filter_t<52, false, DMMA>(ctx, fa);
        case 60: return launch_filter_t<60, false, DMMA>(ctx, fa);
        }
    } else {
        switch (kc) {
        case 44: return launch_filter_t<44, true, DMMA>(ctx, fa);
        case 52: return launch_filter_t<52, true, DMMA>(ctx, fa);
        }
    }
    return fail(ctx, SCEMA_ERR_INVALID, "no filter kernel instantiation for this chunk size");
}

static uint32_t bits_for(uint64_t n)
{
    uint32_t b = 1;
    while (b < 32 && (1ull << b) < n) b++;
    return b;
}

// A sharded prepare lets the filter start before the FP64 rows of the other GPUs have arrived (tc_shard_commit):
// everything that reads the rows themselves waits for that event first.
int wait_rows(scema_ctx *ctx)
{
    if (ctx->rows_ready_event) {
        SCEMA_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, (cudaEvent_t)ctx->rows_ready_event, 0));
        ctx->rows_ready_event = nullptr;
    }
    return SCEMA_OK;
}

static int prepare_filter(scema_ctx *ctx, int variant)
{
    FilterLayout &fl = ctx->fl;
    if (ctx->filter_for_spline_version == ctx->spline_version && ctx->filter_variant == variant && fl.n == ctx->n &&
        fl.K == ctx->K)
        return SCEMA_OK;
    fl.K = ctx->K;
    fl.n = ctx->n;
    { const int rcw = wait_rows(ctx); if (rcw) return rcw; }
    static const char *k2_env = getenv("SCEMA_K2");
    const bool ws = variant == SCEMA_PAIRS_DMMA && !(k2_env && strcmp(k2_env, "v1") == 0);
    if (ws) choose_chunks_tail(fl.K, &fl.kc, &fl.kt, &fl.n_chunks);
    else { choose_chunks(fl.K, &fl.kc, &fl.n_chunks); fl.kt = fl.kc; }
    fl.n_blocks = (fl.n + TILE - 1) / TILE;
    fl.n_pad = fl.n_blocks * TILE;
    const uint32_t ks = variant == SCEMA_PAIRS_DMMA ? fl.kc : fl.kc + 1;
    const uint32_t kst = variant == SCEMA_PAIRS_DMMA ? fl.kt : fl.kt + 1;
    SCEMA_CUDA(ctx, ctx->d_filter.reserve((size_t)fl.n_chunks * fl.n_pad * ks * sizeof(double)));
    SCEMA_CUDA(ctx, ctx->d_halfnorm.reserve(fl.n_pad * sizeof(double)));
    SCEMA_CUDA(ctx, ctx->d_blockmax.reserve(fl.n_blocks * sizeof(double)));
    SCEMA_CUDA(ctx, cudaMemsetAsync(ctx->d_blockmax.p, 0, fl.n_blocks * sizeof(double), ctx->stream));
    k_prep<<<(unsigned)((fl.n_pad + 7) / 8), 256, 0, ctx->stream>>>(ctx->d_spline, fl.n, fl.K, fl.n_pad, fl.kc, ks, fl.kt, kst,
                                                                     fl.n_chunks, ctx->d_filter.as<double>(),
                                                                     ctx->d_halfnorm.as<double>(),
                                                                     ctx->d_blockmax.as<unsigned long long>());
    ctx->launches++;
    SCEMA_CUDA(ctx, cudaGetLastError());
    ctx->filter_for_spline_version = ctx->spline_version;
    ctx->filter_variant = variant;
    return SCEMA_OK;
}

static int ensure_edge_buffers(scema_ctx *ctx, uint64_t cap)
{
    if (cap <= ctx->edge_cap) return SCEMA_OK;
    for (int b = 0; b < 2; b++) {
        SCEMA_CUDA(ctx, ctx->d_edge_key[b].reserve(cap * sizeof(uint64_t)));
        SCEMA_CUDA(ctx, ctx->d_edge_val[b].reserve(cap * sizeof(double)));
    }
    ctx->edge_cap = cap;
    return SCEMA_OK;
}

static int sort_edges(scema_ctx *ctx);

// Schedule of one compare: panels of PANEL_ROWBLOCKS row blocks, column strips of strip_len tiles.
struct Schedule {
    uint64_t nb = 0, tiles = 0, groups = 0;
    uint32_t strip_len = 0, n_panels = 0;
    std::vector<uint64_t> ps;  // [n_panels+1] prefix of strip groups per panel
};

static void make_schedule(const scema_ctx *ctx, uint64_t n, Schedule &sc)
{
    sc.nb = (n + TILE - 1) / TILE;
    sc.tiles = sc.nb * (sc.nb + 1) / 2;
    sc.strip_len = (uint32_t)std::min<uint64_t>(64, std::max<uint64_t>(4, sc.tiles / ((uint64_t)ctx->sm_count * 8)));
    sc.n_panels = (uint32_t)((sc.nb + PANEL_ROWBLOCKS - 1) / PANEL_ROWBLOCKS);
    sc.ps.assign(sc.n_panels + 1, 0);
    for (uint32_t p = 0; p < sc.n_panels; p++) {
        uint64_t cols = sc.nb - (uint64_t)p * PANEL_ROWBLOCKS;
        sc.ps[p + 1] = sc.ps[p] + (cols + sc.strip_len - 1) / sc.strip_len;
    }
    sc.groups = sc.ps[sc.n_panels];
}

// shard-local index of the first group >= g owned by `shard`
static uint64_t local_index(uint64_t g, uint32_t shard, uint32_t n_shards)
{
    return g > shard ? (g - shard + n_shards - 1) / n_shards : 0;
}

// Evaluate the pairs of panels [p0, p1) that belong to this shard: filter + exact recompute (or the
// filter-free kernel), retried with larger buffers on overflow, then the canonical (a,b) sort.
// Leaves the edges in d_edge_key/val[ctx->edge_cur], their number in ctx->n_edges. *variant may be
// switched to SCEMA_PAIRS_EXACT when the survivors are too dense for a queue.
// `overlap` (optional) is host work to do while the GPU runs the first pass: it is called once, after
// the kernels are queued and before the host blocks on the counter read-back.
static int compare_panels(scema_ctx *ctx, double thr, int *variant, uint32_t shard, uint32_t n_shards, const Schedule &sc,
                          uint32_t p0, uint32_t p1, const std::function<int()> &overlap = nullptr)
{
    const uint64_t n = ctx->n;
    const uint32_t K = ctx->K;
    unsigned long long *d_cnt = ctx->d_counters.as<unsigned long long>();
    size_t free_b = 0, total_b = 0;
    uint64_t passes = 0;
    int rc;
    ctx->n_edges = 0;
    ctx->edge_cur = 0;
    // pairs this call evaluates: the rows of panels [p0, p1) against everything to their right, this shard's share
    double pairs_call = 0.0;
    {
        const double panel_rows = (double)PANEL_ROWBLOCKS * TILE;
        const double r0 = std::min<double>((double)n, p0 * panel_rows), r1 = std::min<double>((double)n, p1 * panel_rows);
        pairs_call = ((r1 - r0) * (double)n - 0.5 * (r1 * r1 - r0 * r0)) / (double)n_shards;
    }
    while (true) {
        passes++;
        if (passes > 8) return fail(ctx, SCEMA_ERR_NOMEM, "compare: buffers kept overflowing");
        SCEMA_CUDA(ctx, cudaMemsetAsync(d_cnt, 0, 8 * sizeof(uint64_t), ctx->stream));
        if (*variant == SCEMA_PAIRS_EXACT) {
            rc = wait_rows(ctx);
            if (rc) return rc;
            const uint32_t nbx = (uint32_t)((n + XT - 1) / XT);
            const uint32_t per_panel = PANEL_ROWBLOCKS * (TILE / XT);
            const uint32_t i_first = (uint32_t)std::min<uint64_t>((uint64_t)p0 * per_panel, nbx);
            const uint32_t i_end = (uint32_t)std::min<uint64_t>((uint64_t)p1 * per_panel, nbx);
            t_begin(ctx, SCEMA_T_FILTER);
            // gridDim.y stops at 65535: row slabs of that many 64-row blocks, so any n < 2^32 works
            for (uint32_t i0 = i_first; i0 < i_end; i0 += 65535u) {
                k_exact_all<<<dim3(nbx, std::min<uint32_t>(65535u, i_end - i0)), 256, 0, ctx->stream>>>(
                    ctx->d_spline, n, K, thr, ctx->key_shift, shard, n_shards, i0, d_cnt + 1, ctx->edge_cap,
                    ctx->d_edge_key[0].as<uint64_t>(), ctx->d_edge_val[0].as<double>());
                ctx->launches++;
            }
            t_end(ctx, SCEMA_T_FILTER);
            SCEMA_CUDA(ctx, cudaGetLastError());
        } else if (*variant == SCEMA_PAIRS_TC) {
            SCEMA_CUDA(ctx, ctx->d_cand.reserve(ctx->cand_cap * sizeof(uint64_t)));
            t_begin(ctx, SCEMA_T_FILTER);
            // one panel = PANEL_ROWBLOCKS * TILE = 2048 rows = 8 row tiles of 256
            rc = tc_launch(ctx, p0 * (PANEL_ROWBLOCKS * TILE / 256), p1 * (PANEL_ROWBLOCKS * TILE / 256), 0, 0xffffffffu, shard, n_shards,
                           d_cnt + 0, nullptr, 0);
            if (rc) return rc;
            t_end(ctx, SCEMA_T_FILTER);
            rc = wait_rows(ctx);  // sharded prepare: the filter ran on the gathered fp16 images; the rows themselves are needed from here on
            if (rc) return rc;
            t_begin(ctx, SCEMA_T_EXACT);
            k_exact_queue<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(ctx->d_spline, K, ctx->d_cand.as<uint64_t>(), d_cnt + 0,
                                                                      ctx->cand_cap, thr, ctx->key_shift, d_cnt + 1,
                                                                      ctx->edge_cap, ctx->d_edge_key[0].as<uint64_t>(),
                                                                      ctx->d_edge_val[0].as<double>());
            ctx->launches++;
            t_end(ctx, SCEMA_T_EXACT);
            SCEMA_CUDA(ctx, cudaGetLastError());
        } else {
            const FilterLayout &fl = ctx->fl;
            SCEMA_CUDA(ctx, ctx->d_cand.reserve(ctx->cand_cap * sizeof(uint64_t)));
            FilterArgs fa;
            fa.F = ctx->d_filter.as<double>();
            fa.HN = ctx->d_halfnorm.as<double>();
            fa.BM = ctx->d_blockmax.as<double>();
            fa.panel_start = ctx->d_panel_start.as<uint64_t>();
            fa.work_counter = d_cnt + 3;
            fa.cand_count = d_cnt + 0;
            fa.cand = ctx->d_cand.as<uint64_t>();
            fa.cand_cap = ctx->cand_cap;
            fa.n = n;
            fa.n_pad = fl.n_pad;
            fa.n_blocks = (uint32_t)sc.nb;
            fa.n_panels = sc.n_panels;
            fa.n_chunks = fl.n_chunks;
            fa.strip_len = sc.strip_len;
            fa.lg_first = local_index(sc.ps[p0], shard, n_shards);
            fa.n_groups_local = local_index(sc.ps[p1], shard, n_shards) - fa.lg_first;
            fa.shard = shard;
            fa.n_shards = n_shards;
            const double eps = 1.1102230246251565e-16;  // 2^-53
            fa.T0 = thr * thr * (1.0 + (2.0 * K + 16.0) * eps) * (1.0 + 4.0 * eps);
            fa.cband = (4.0 * K + 64.0) * eps;

            t_begin(ctx, SCEMA_T_FILTER);
            // SCEMA_K2=v1 selects the barrier-synchronised DMMA kernel (kept for A/B measurements)
            static const char *k2_env = getenv("SCEMA_K2");
            const bool ws = !(k2_env && strcmp(k2_env, "v1") == 0);
            rc = *variant == SCEMA_PAIRS_DMMA ? (ws ? launch_filter_ws(ctx, fa, fl.kc, fl.kt, fl.n_chunks > 1)
                                                    : launch_filter<true>(ctx, fa, fl.kc, fl.n_chunks > 1))
                                              : launch_filter<false>(ctx, fa, fl.kc, fl.n_chunks > 1);
            if (rc) return rc;
            t_end(ctx, SCEMA_T_FILTER);

            t_begin(ctx, SCEMA_T_EXACT);
            k_exact_queue<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(ctx->d_spline, K, ctx->d_cand.as<uint64_t>(), d_cnt + 0,
                                                                      ctx->cand_cap, thr, ctx->key_shift, d_cnt + 1,
                                                                      ctx->edge_cap, ctx->d_edge_key[0].as<uint64_t>(),
                                                                      ctx->d_edge_val[0].as<double>());
            ctx->launches++;
            t_end(ctx, SCEMA_T_EXACT);
            SCEMA_CUDA(ctx, cudaGetLastError());
        }
        SCEMA_CUDA(ctx, cudaMemcpyAsync(ctx->h_counters, d_cnt, 8 * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
        if (overlap && passes == 1) {
            rc = overlap();
            if (rc) return rc;
        }
        SCEMA_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        const uint64_t n_cand = ctx->h_counters[0], n_edge = ctx->h_counters[1];
        if (*variant != SCEMA_PAIRS_EXACT && n_cand > ctx->cand_cap) {
            // The survivors did not fit (the up-front estimate of compare_begin was too low, or the filter was pinned).
            // Cheapest way on, by the same cost model: repeat with a larger queue, with both fp16 slices, with the FP64
            // DMMA filter, or without a filter. Filters split the pair matrix between shards differently, so a sharded
            // compare never changes filter on its own (every shard would have to): it reports SCEMA_ERR_DENSE instead.
            SCEMA_CUDA(ctx, cudaMemGetInfo(&free_b, &total_b));
            const uint64_t want = n_cand + n_cand / 4;
            const bool can_grow = want * sizeof(uint64_t) <= (free_b + ctx->d_cand.bytes) / 2;
            const double kf = 60.0 / (double)std::max<uint32_t>(K, 1);
            const double Pc = pairs_call, requeue = (double)n_cand / (RATE_QUEUE * kf);
            if (*variant == SCEMA_PAIRS_TC) {
                const uint32_t nc = tc_chunks_for(K);
                if (ctx->tc_mode == 1 && ctx->tc_slices == 1 && nc == 1) {
                    if (can_grow && requeue <= Pc * (1.0 / RATE_TC2 - 1.0 / RATE_TC1)) { ctx->cand_cap = want; continue; }
                    rc = tc_prepare(ctx, thr, 2, ctx->tc_band_wanted, 0, nullptr, nullptr);  // same tiles, same shards
                    if (rc) return rc;
                    continue;
                }
                if (can_grow && (requeue <= Pc / (RATE_DMMA * kf) || ctx->tc_mode == 0)) { ctx->cand_cap = want; continue; }
                if (n_shards > 1) {
                    if (can_grow) { ctx->cand_cap = want; continue; }
                    return fail(ctx, SCEMA_ERR_DENSE, "compare: survivors too dense for this shard's queue; repeat on every shard with SCEMA_PAIRS_DMMA");
                }
                *variant = SCEMA_PAIRS_DMMA;  // guard band 2^-40 of the norms instead of 2^-9 / 2^-13
                rc = prepare_filter(ctx, SCEMA_PAIRS_DMMA);
                if (rc) return rc;
                SCEMA_CUDA(ctx, ctx->d_panel_start.reserve(sc.ps.size() * sizeof(uint64_t)));
                SCEMA_CUDA(ctx, cudaMemcpyAsync(ctx->d_panel_start.p, sc.ps.data(), sc.ps.size() * sizeof(uint64_t),
                                                cudaMemcpyHostToDevice, ctx->stream));
                SCEMA_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
                continue;
            }
            if (can_grow) { ctx->cand_cap = want; continue; }
            if (n_shards > 1)
                return fail(ctx, SCEMA_ERR_DENSE, "compare: survivors too dense for this shard's queue; repeat on every shard with SCEMA_PAIRS_EXACT");
            *variant = SCEMA_PAIRS_EXACT;  // survivors too dense for a queue: filter-free kernel
            continue;
        }
        if (n_edge > ctx->edge_cap) {
            rc = ensure_edge_buffers(ctx, n_edge + n_edge / 8);
            if (rc) return rc;
            continue;
        }
        ctx->counters[1] += n_cand;
        ctx->counters[3] += passes;
        if (*variant == SCEMA_PAIRS_TC) {
            ctx->counters[5] = ctx->tc_slices;
            if (ctx->tc_band) {  // tiles the band schedule actually walked (k_tc_band_plan)
                unsigned long long misc[4];
                SCEMA_CUDA(ctx, cudaMemcpy(misc, ctx->d_tc_misc.p, sizeof(misc), cudaMemcpyDeviceToHost));
                ctx->counters[7] = misc[3];
            }
        }
        ctx->n_edges = n_edge;
        break;
    }
    return sort_edges(ctx);
}

// canonical order: ascending (a,b) == ascending packed key
static int sort_edges(scema_ctx *ctx)
{
    if (ctx->n_edges > 1) {
        t_begin(ctx, SCEMA_T_SORT);
        cub::DoubleBuffer<uint64_t> dk(ctx->d_edge_key[0].as<uint64_t>(), ctx->d_edge_key[1].as<uint64_t>());
        cub::DoubleBuffer<double> dv(ctx->d_edge_val[0].as<double>(), ctx->d_edge_val[1].as<double>());
        size_t tmp = 0;
        const int end_bit = (int)std::min<uint32_t>(64, 2 * ctx->key_shift);
        SCEMA_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, tmp, dk, dv, (int64_t)ctx->n_edges, 0, end_bit, ctx->stream));
        SCEMA_CUDA(ctx, ctx->d_sort_tmp.reserve(tmp));
        SCEMA_CUDA(ctx, cub::DeviceRadixSort::SortPairs(ctx->d_sort_tmp.p, tmp, dk, dv, (int64_t)ctx->n_edges, 0, end_bit,
                                                        ctx->stream));
        ctx->launches += 2 * ((end_bit + 7) / 8) + 1;
        ctx->edge_cur = dk.selector;
        t_end(ctx, SCEMA_T_SORT);
        SCEMA_CUDA(ctx, cudaGetLastError());
    }
    return SCEMA_OK;
}

// Install an edge list computed elsewhere (the union of the shards' lists, multi.cu) as this context's result: copied
// into the context's own buffers (grown as needed), put in canonical (a, b) order, served by scema_get_edges and friends.
int edges_adopt(scema_ctx *ctx, const uint64_t *d_keys, const double *d_vals, uint64_t total)
{
    int rc = ensure_edge_buffers(ctx, std::max<uint64_t>(total, 1));
    if (rc) return rc;
    if (total) {
        SCEMA_CUDA(ctx, cudaMemcpyAsync(ctx->d_edge_key[0].p, d_keys, total * sizeof(uint64_t), cudaMemcpyDeviceToDevice, ctx->stream));
        SCEMA_CUDA(ctx, cudaMemcpyAsync(ctx->d_edge_val[0].p, d_vals, total * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    }
    ctx->n_edges = total;
    ctx->edge_cur = 0;
    ctx->have_edges = true;
    ctx->counters[2] = total;
    return sort_edges(ctx);
}

// Common front end: argument checks, buffers, filter copy and schedule. Returns 1 when there is
// nothing to compare (result: no edges). plan_pairs: the pairs the filter choice is made for (0: this shard's share of
// the whole triangle).
static int compare_begin(scema_ctx *ctx, double thr, int &variant, uint32_t shard, uint32_t n_shards, Schedule &sc, uint64_t plan_pairs = 0)
{
    if (!ctx->have_spline) return fail(ctx, SCEMA_ERR_STATE, "Spline is not up to date.");
    if (n_shards == 0 || shard >= n_shards) return fail(ctx, SCEMA_ERR_INVALID, "compare: bad shard");
    if (variant < 0 || variant > 3) return fail(ctx, SCEMA_ERR_INVALID, "compare: bad variant");
    // the tcgen05 filter takes rows of up to 10 chunks of 64 columns (K <= 636); wider rows take the DMMA filter
    if (variant == SCEMA_PAIRS_TC && (ctx->have_spline && !tc_supported(ctx))) variant = SCEMA_PAIRS_DMMA;
    if (ctx->n >= (1ull << 32)) return fail(ctx, SCEMA_ERR_INVALID, "compare: more than 2^32-1 histories");
    for (int i = 0; i < 8; i++) ctx->counters[i] = 0;
    for (int w = SCEMA_T_PREP; w <= SCEMA_T_SORT; w++) { ctx->ev_used[w] = false; ctx->acc_ms[w] = 0.f; }
    ctx->n_edges = 0;
    ctx->have_edges = true;
    ctx->edge_cur = 0;
    ctx->key_shift = bits_for(ctx->n);
    const uint64_t n = ctx->n;
    // diff >= 0 or NaN, so nothing passes a non-positive or NaN threshold
    if (n < 2 || !(thr > 0.0)) return -1;

    SCEMA_CUDA(ctx, ctx->d_counters.reserve(8 * sizeof(uint64_t)));
    if (!ctx->h_counters) SCEMA_CUDA(ctx, cudaMallocHost(&ctx->h_counters, 8 * sizeof(uint64_t)));
    int rc = ensure_edge_buffers(ctx, std::max<uint64_t>(1ull << 20, 16 * n));
    if (rc) return rc;
    make_schedule(ctx, n, sc);
    ctx->counters[4] = sc.tiles;
    const uint64_t queue_floor = std::max<uint64_t>(1ull << 20, 32 * n);  // grows with the batch: a context that started small must not mistake a full queue for a wide guard band
    if (variant != SCEMA_PAIRS_EXACT) t_begin(ctx, SCEMA_T_PREP);
    if (variant == SCEMA_PAIRS_TC) {
        // How many fp16 slices, or another filter altogether? Pinned by SCEMA_TC_SLICES=1|2 (3: the projected 16-column
        // filter), otherwise decided from a sample of the pairs (tc_prepare / tc_choose; the same rows and threshold keep
        // their earlier decision): survivors of every option estimated in FP64 BEFORE the first launch, so the common
        // case is one pass.
        static const char *sl_env = getenv("SCEMA_TC_SLICES");
        const int pin = sl_env ? atoi(sl_env) : 0;
        uint32_t slices = (pin >= 1 && pin <= 3) ? (uint32_t)pin : 0u;
        if (slices == 2 && !tc_two_slices_possible(ctx)) slices = 1;  // K > 60: hi slices only
        if (slices == 3 && !tc_proj_possible(ctx->K)) slices = 1;
        ctx->tc_mode = slices ? 0u : 1u;                              // 1: automatic (compare_panels may change it on overflow)
        // SCEMA_NORM_BAND=1 (one-shot compares only): rows in norm order, tiles beyond the threshold's reach skipped
        const char *band_env = getenv("SCEMA_NORM_BAND");
        const bool want_band = ctx->tc_band_allowed && band_env && atoi(band_env) == 1;
        int choice = 1;
        uint64_t est = 0;
        rc = tc_prepare(ctx, thr, slices, want_band, plan_pairs ? plan_pairs : n * (n - 1) / 2 / n_shards, &choice, &est);
        if (rc) return rc;
        if (choice == 0) variant = SCEMA_PAIRS_DMMA;
        else if (choice < 0) variant = SCEMA_PAIRS_EXACT;
        else ctx->cand_cap = std::max<uint64_t>(ctx->cand_cap, std::max<uint64_t>(queue_floor, est + est / 4));
    }
    if (variant == SCEMA_PAIRS_DMMA || variant == SCEMA_PAIRS_FMA) {
        rc = prepare_filter(ctx, variant);
        if (rc) return rc;
        SCEMA_CUDA(ctx, ctx->d_panel_start.reserve(sc.ps.size() * sizeof(uint64_t)));
        SCEMA_CUDA(ctx, cudaMemcpyAsync(ctx->d_panel_start.p, sc.ps.data(), sc.ps.size() * sizeof(uint64_t),
                                        cudaMemcpyHostToDevice, ctx->stream));
        SCEMA_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // sc.ps may not outlive the copy otherwise
        ctx->cand_cap = std::max<uint64_t>(ctx->cand_cap, queue_floor);
    }
    if (ctx->ev_used[SCEMA_T_PREP]) t_end(ctx, SCEMA_T_PREP);
    return SCEMA_OK;
}

// pairs (a, b), a < b, with a in the row panels [0, p1) of n rows
static uint64_t prefix_pairs(uint64_t n, uint32_t p1)
{
    const uint64_t r1 = std::min<uint64_t>(n, (uint64_t)p1 * PANEL_ROWBLOCKS * TILE);
    return r1 * n - r1 * (r1 + 1) / 2;
}

// The rounds of scema_knn and the scema_query_* calls (knn.cu): every pair (a, b), a < b, with a in the row panels
// [0, p1) (p1 = 0: all of them), one GPU, no audit. plan_prefix: the filter is chosen for the pairs of those panels (a
// small query in front of a large matrix must not be planned as the whole triangle: that overestimates its survivors by
// up to (n + m) / 2m); otherwise for the whole triangle, as scema_knn does. The edges are left as after compare_run,
// counters[0] = the pairs of the panels; *variant becomes the filter that ran.
int compare_prefix_run(scema_ctx *ctx, double thr, int *variant, uint32_t p1, bool plan_prefix)
{
    Schedule sc;
    int rc = compare_begin(ctx, thr, *variant, 0, 1, sc, plan_prefix && p1 ? prefix_pairs(ctx->n, p1) : 0);
    if (rc < 0) return SCEMA_OK;
    if (rc) return rc;
    const uint32_t p_end = p1 ? std::min<uint32_t>(p1, sc.n_panels) : sc.n_panels;
    rc = compare_panels(ctx, thr, variant, 0, 1, sc, 0, p_end);
    if (rc) return rc;
    ctx->counters[0] = prefix_pairs(ctx->n, p_end);
    ctx->counters[2] = ctx->n_edges;
    return SCEMA_OK;
}

// Run-time audit (SCEMA_AUDIT=<samples>, off by default): the filters reject pairs on the strength of an error budget
// that — for the tcgen05 filter — rests on one measured hardware property (fp32 accumulation of a kind::f16 step,
// DESIGN.md "K2-TC"). The audit recomputes `samples` pairs exactly (half uniformly random, half between histories whose
// indices are close, where similar histories concentrate) and requires every one that the reference calls an edge to BE
// in the emitted list (binary search in the sorted keys). A miss fails the compare loudly.
__global__ void __launch_bounds__(256) k_audit(const double *__restrict__ S, uint64_t n, uint32_t K, double thr, uint32_t key_shift,
                                               const uint64_t *__restrict__ keys, uint64_t n_edges, uint64_t samples, uint64_t seed,
                                               unsigned long long *__restrict__ out)
{
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= samples) return;
    auto mix = [](uint64_t z) {
        z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
        z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
        return z ^ (z >> 31);
    };
    uint64_t i = mix(seed + 2 * t) % n, j;
    if (t & 1) j = (i + 1 + mix(seed + 2 * t + 1) % 32) % n;   // a near index
    else j = mix(seed + 2 * t + 1) % n;
    if (i == j) return;
    if (i > j) { const uint64_t x = i; i = j; j = x; }
    const double d = exact_l2(S + i * K, S + j * K, K);
    if (!(d < thr)) return;
    atomicAdd(out + 0, 1ull);  // sampled pairs that are edges
    const uint64_t key = (i << key_shift) | j;
    uint64_t lo = 0, hi = n_edges;
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if (keys[mid] < key) lo = mid + 1; else hi = mid;
    }
    if (!(lo < n_edges && keys[lo] == key)) atomicAdd(out + 1, 1ull);
}

static int audit_run(scema_ctx *ctx, double thr)
{
    const char *e = getenv("SCEMA_AUDIT");
    const uint64_t samples = e ? (uint64_t)atoll(e) : 0;
    if (!samples || ctx->n < 2) return SCEMA_OK;
    unsigned long long *d_cnt = ctx->d_counters.as<unsigned long long>();
    SCEMA_CUDA(ctx, cudaMemsetAsync(d_cnt + 4, 0, 2 * sizeof(uint64_t), ctx->stream));
    if (const char *f = getenv("SCEMA_AUDIT_THR_FACTOR")) thr *= atof(f);  // test hook: audit against a larger threshold than the compare used
    k_audit<<<(unsigned)((samples + 255) / 256), 256, 0, ctx->stream>>>(ctx->d_spline, ctx->n, ctx->K, thr, ctx->key_shift,
                                                                         ctx->d_edge_key[ctx->edge_cur].as<uint64_t>(), ctx->n_edges, samples,
                                                                         0x5ca1ab1eull + ctx->spline_version, d_cnt + 4);
    ctx->launches++;
    SCEMA_CUDA(ctx, cudaGetLastError());
    SCEMA_CUDA(ctx, cudaMemcpyAsync(ctx->h_counters, d_cnt, 8 * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    SCEMA_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->audit_edges = ctx->h_counters[4];
    ctx->audit_missing = ctx->h_counters[5];
    if (ctx->audit_missing)
        return fail(ctx, SCEMA_ERR_STATE, "audit: " + std::to_string(ctx->audit_missing) + " of " + std::to_string(ctx->audit_edges) +
                                              " sampled reference edges are missing from the emitted list (filter unsound on this device?)");
    return SCEMA_OK;
}

int compare_run(scema_ctx *ctx, double thr, int variant, uint32_t shard, uint32_t n_shards)
{
    Schedule sc;
    ctx->tc_band_allowed = true;   // the whole pair matrix in one launch: the norm-band schedule applies
    int rc = compare_begin(ctx, thr, variant, shard, n_shards, sc);
    ctx->tc_band_allowed = false;
    if (rc < 0) return SCEMA_OK;
    if (rc) return rc;
    rc = compare_panels(ctx, thr, &variant, shard, n_shards, sc, 0, sc.n_panels);
    if (rc) return rc;
    ctx->counters[2] = ctx->n_edges;
    if (n_shards == 1) ctx->counters[0] = ctx->n * (ctx->n - 1) / 2;
    if (n_shards == 1 && variant != SCEMA_PAIRS_EXACT) return audit_run(ctx, thr);  // a shard's list only holds its own tiles
    return SCEMA_OK;
}

// ------------------------------------------------------------------------------------------------
// scema_cluster from host buffers, pipelined (SCEMA_PAIRS_TC, K <= 60)
//
// The raw steps of a large batch take longer to cross PCIe than the whole clustering takes on the GPU
// (config 4: 1.7 GB, ~65 ms, against ~65 ms of kernels), so the batch is cut into ranges of histories.
// Range c is copied on a second stream; as soon as it has landed it is resampled (K1 plan per range),
// its fp16 operand copies are built, and the tcgen05 filter evaluates the COLUMN panel of the pair
// matrix that pairs range c with itself and every earlier range — all of which is on the device by
// then — while range c+1 is still on the bus. The survivors of all panels share one queue; the exact
// recompute and the sort run once at the end. The operand scale has to be one power of two for all rows
// but the rows are not all there when the first panel starts: it is frozen after range 0 with six
// binades of headroom (rows that still outgrow it lose their fp16 image and survive against everybody,
// k_tc_prep), which changes which pairs survive, never the edge list.
// ------------------------------------------------------------------------------------------------
bool pipeline_wanted(uint64_t n)
{
    const char *e = getenv("SCEMA_PIPELINE");         // 0 disables
    if (e && atoi(e) == 0) return false;
    const char *m = getenv("SCEMA_PIPELINE_MIN_N");    // smallest batch that is pipelined (tests lower it)
    const uint64_t min_n = m ? (uint64_t)atoll(m) : 65536;
    return n >= min_n && n >= 4096;
}

// Ranges of the pipeline: up to 16, whole panels (2048 rows, hence whole 256-row tiles) each.
void pipeline_bounds(uint64_t n, std::vector<uint64_t> &bounds)
{
    const uint64_t panel_rows = (uint64_t)PANEL_ROWBLOCKS * TILE;
    const uint64_t n_ranges = std::min<uint64_t>(16, std::max<uint64_t>(2, n / 65536));
    const uint64_t per = ((n + n_ranges - 1) / n_ranges + panel_rows - 1) / panel_rows * panel_rows;
    bounds.assign(1, 0);
    while (bounds.back() < n) bounds.push_back(std::min<uint64_t>(n, bounds.back() + per));
}

static int pipeline_queue_copy(scema_ctx *ctx, const double *steps_host, const uint64_t *offsets, uint64_t r)
{
    const uint64_t s0 = offsets[ctx->pipe_bounds[r]], s1 = offsets[ctx->pipe_bounds[r + 1]];
    if (s1 > s0)
        SCEMA_CUDA(ctx, cudaMemcpyAsync(ctx->steps_own.as<double>() + s0 * 6, steps_host + s0 * 6, (s1 - s0) * 6 * sizeof(double),
                                        cudaMemcpyHostToDevice, ctx->copy_stream));
    SCEMA_CUDA(ctx, cudaEventRecord(ctx->copy_events[r], ctx->copy_stream));
    return SCEMA_OK;
}

// First act of the pipeline, before anything else touches the batch: the first four ranges start travelling at once
// (~17 ms of copies at config 4); the host-side work that follows — validation of the offsets, factor tables, K1 plan,
// a few ms with small host->device copies of its own, which queue behind what is already on the copy engine — runs
// meanwhile, and only then are the remaining ranges queued. The offsets are scanned once here (monotone, no history
// beyond the length limit) because they size the device buffer; set_histories reports what is wrong with a bad array.
int pipeline_begin(scema_ctx *ctx, const double *steps_host, const uint64_t *offsets, uint64_t n)
{
    pipeline_bounds(n, ctx->pipe_bounds);
    const uint64_t n_ranges = ctx->pipe_bounds.size() - 1;
    ctx->pipe_early = 0;
    if (!ctx->copy_stream) SCEMA_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    while (ctx->copy_events.size() < n_ranges) {
        cudaEvent_t e;
        SCEMA_CUDA(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        ctx->copy_events.push_back(e);
    }
    const uint64_t early = std::min<uint64_t>(4, n_ranges);
    // the offsets size the device buffer below: a bad array must come back as SCEMA_ERR_INVALID from set_histories
    // (which repeats this scan), not as an out-of-memory error from here (~0.3 ms for 10^6 histories)
    for (uint64_t i = 0; i < n; i++)
        if (offsets[i + 1] < offsets[i] || offsets[i + 1] - offsets[i] > 0x7fffffffull / 64) return SCEMA_OK;
    // the previous batch's kernels may still read the buffer the copies are about to overwrite
    SCEMA_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    SCEMA_CUDA(ctx, ctx->steps_own.reserve(std::max<uint64_t>(offsets[n], 1) * 6 * sizeof(double)));
    for (uint64_t r = 0; r < early; r++) {
        const int rc = pipeline_queue_copy(ctx, steps_host, offsets, r);
        if (rc) return rc;
        ctx->pipe_early = r + 1;
    }
    return SCEMA_OK;
}

static int cluster_pipelined_impl(scema_ctx *ctx, const double *steps_host, uint32_t P, double thr, bool *done)
{
    *done = false;
    const uint64_t n = ctx->hn;
    const std::vector<uint64_t> &bounds = ctx->pipe_bounds;
    const uint64_t n_ranges = bounds.size() - 1;
    const uint64_t early = ctx->pipe_early;
    int rc;
    rc = resample_prepare(ctx, P, bounds);
    if (rc) return rc;
    for (int i = 0; i < 8; i++) ctx->counters[i] = 0;
    for (int w = SCEMA_T_RESAMPLE; w <= SCEMA_T_SORT; w++) { ctx->ev_used[w] = false; ctx->acc_ms[w] = 0.f; }
    ctx->n_edges = 0;
    ctx->edge_cur = 0;
    ctx->key_shift = bits_for(n);
    SCEMA_CUDA(ctx, ctx->d_counters.reserve(8 * sizeof(uint64_t)));
    if (!ctx->h_counters) SCEMA_CUDA(ctx, cudaMallocHost(&ctx->h_counters, 8 * sizeof(uint64_t)));
    rc = ensure_edge_buffers(ctx, std::max<uint64_t>(1ull << 20, 16 * n));
    if (rc) return rc;
    ctx->cand_cap = std::max<uint64_t>(ctx->cand_cap, std::max<uint64_t>(1ull << 20, 32 * n));  // grows with the batch: a context that started small must not mistake a full queue for a wide guard band
    SCEMA_CUDA(ctx, ctx->d_cand.reserve(ctx->cand_cap * sizeof(uint64_t)));
    rc = tc_prepare_begin(ctx, thr, 1);
    if (rc) return rc;
    unsigned long long *d_cnt = ctx->d_counters.as<unsigned long long>();
    SCEMA_CUDA(ctx, cudaMemsetAsync(d_cnt, 0, 8 * sizeof(uint64_t), ctx->stream));
    SCEMA_CUDA(ctx, cudaStreamSynchronize(ctx->stream));

    // ---- queue the remaining copies, then the per-range work
    for (uint64_t r = early; r < n_ranges; r++)
        if ((rc = pipeline_queue_copy(ctx, steps_host, ctx->h_offsets.data(), r))) return rc;
    const uint64_t n_pad = (n + 255) / 256 * 256;
    t_begin(ctx, SCEMA_T_FILTER);  // in this mode "filter" spans the whole overlapped region (K1, operand prep and filter of every range)
    for (uint64_t r = 0; r < n_ranges; r++) {
        SCEMA_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->copy_events[r], 0));
        rc = resample_launch_range(ctx, P, r);
        if (rc) return rc;
        const uint64_t r0 = bounds[r], r1 = bounds[r + 1];
        const uint64_t r1p = r + 1 == n_ranges ? n_pad : r1;  // the last range also writes the padding rows
        rc = r == 0 ? tc_centre_rows(ctx, r0, r1) : SCEMA_OK;  // centre and scale come from the first range
        if (!rc) rc = tc_stats_rows(ctx, r0, r1, r == 0);
        if (!rc && r == 0) rc = tc_fix_scale(ctx, 6);
        if (!rc && r == 0) {
            // is the one-slice filter (64 columns or projected) the right one for this data? (sample of the first range; the
            // host waits for range 0 here, the later copies keep travelling) If not, the ordinary path decides with all rows
            // in hand. The basis, like centre and scale, comes from the first range: later rows outside its span land in
            // the residual coordinate, which costs survivors, never edges.
            bool proj_ok = tc_proj_possible(ctx->K);
            if (proj_ok) rc = tc_basis_range(ctx, r0, r1, &proj_ok);
            uint64_t counts[6];
            if (!rc) rc = tc_plan_rows(ctx, r1, counts, proj_ok);
            int choice = 1, centred = 1;
            uint64_t est = 0;
            if (!rc) {
                tc_choose(n * (n - 1) / 2, ctx->K, counts, tc_plan_sample_size(), (uint64_t)ctx->mem_budget, true, proj_ok, &choice, &centred,
                          &est);
                if (!(choice == 3 || (choice == 1 && centred)) || est + est / 4 > ctx->cand_cap) { t_end(ctx, SCEMA_T_FILTER); return SCEMA_OK; }
                ctx->tc_proj = choice == 3;
            }
        }
        if (!rc) rc = tc_prep_rows(ctx, r0, r1p);
        if (!rc) rc = tc_launch(ctx, 0, (uint32_t)(r1p / 256), (uint32_t)(r0 / 256), (uint32_t)(r1p / 256), 0, 1, d_cnt + 0, nullptr, 0);
        if (rc) return rc;
    }
    t_end(ctx, SCEMA_T_FILTER);

    // ---- survivors -> edges (repeated only if the edge buffers were too small)
    for (int pass = 0; pass < 4; pass++) {
        SCEMA_CUDA(ctx, cudaMemsetAsync(d_cnt + 1, 0, sizeof(uint64_t), ctx->stream));
        t_begin(ctx, SCEMA_T_EXACT);
        k_exact_queue<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(ctx->d_spline, ctx->K, ctx->d_cand.as<uint64_t>(), d_cnt + 0, ctx->cand_cap,
                                                                  thr, ctx->key_shift, d_cnt + 1, ctx->edge_cap,
                                                                  ctx->d_edge_key[0].as<uint64_t>(), ctx->d_edge_val[0].as<double>());
        ctx->launches++;
        t_end(ctx, SCEMA_T_EXACT);
        SCEMA_CUDA(ctx, cudaGetLastError());
        SCEMA_CUDA(ctx, cudaMemcpyAsync(ctx->h_counters, d_cnt, 8 * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
        SCEMA_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        const uint64_t n_cand = ctx->h_counters[0], n_edge = ctx->h_counters[1];
        if (n_cand > ctx->cand_cap) return SCEMA_OK;  // too many survivors for the one-slice band: the ordinary path sorts it out
        if (n_edge > ctx->edge_cap) {
            rc = ensure_edge_buffers(ctx, n_edge + n_edge / 8);
            if (rc) return rc;
            continue;
        }
        ctx->counters[1] = n_cand;
        ctx->counters[3] = (uint64_t)pass + 1;
        ctx->counters[5] = 1;
        ctx->counters[6] = n_ranges;
        ctx->n_edges = n_edge;
        rc = sort_edges(ctx);
        if (rc) return rc;
        ctx->counters[0] = n * (n - 1) / 2;
        ctx->counters[2] = ctx->n_edges;
        ctx->have_edges = true;
        *done = true;
        return SCEMA_OK;
    }
    return SCEMA_OK;
}

int cluster_pipelined(scema_ctx *ctx, const double *steps_host, uint32_t P, double thr, bool *done)
{
    const int rc = cluster_pipelined_impl(ctx, steps_host, P, thr, done);
    // on failure copies of the caller's buffer may still be in flight; the buffer is the caller's again on return
    if (rc && ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
    if (!rc && !*done && ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
    return rc;
}

// Streaming compare: the panels are evaluated in chunks of panels_per_chunk; each chunk's sorted
// edges are copied to pinned host memory and handed to `sink` while the GPU already works on the
// next chunk. Rows (index a) of consecutive chunks are disjoint and increasing, so the concatenation
// of the chunks is the same (a,b)-sorted list scema_compare produces — without ever holding more
// than one chunk of edges on the device.
int compare_stream_run(scema_ctx *ctx, double thr, int variant, uint32_t shard, uint32_t n_shards, uint32_t panels_per_chunk,
                       scema_edge_sink sink, void *user, uint64_t *n_total)
{
    Schedule sc;
    if (n_total) *n_total = 0;
    int rc = compare_begin(ctx, thr, variant, shard, n_shards, sc);
    if (rc < 0) { ctx->have_edges = false; return SCEMA_OK; }
    if (rc) return rc;
    if (panels_per_chunk == 0) panels_per_chunk = 64;
    struct Staged { uint64_t m = 0; bool pending = false; };
    Staged st[2];
    std::vector<uint32_t> ha, hb;
    const uint64_t mask = (1ull << ctx->key_shift) - 1;
    uint64_t total = 0;
    auto deliver = [&](int slot) -> int {
        if (!st[slot].pending) return SCEMA_OK;
        st[slot].pending = false;
        SCEMA_CUDA(ctx, cudaEventSynchronize(ctx->stage_ev[slot]));
        const uint64_t m = st[slot].m;
        const uint64_t *keys = ctx->h_stage_key[slot];
        ha.resize(m); hb.resize(m);
        for (uint64_t e = 0; e < m; e++) { ha[e] = (uint32_t)(keys[e] >> ctx->key_shift); hb[e] = (uint32_t)(keys[e] & mask); }
        total += m;
        if (m && sink && sink(user, ha.data(), hb.data(), ctx->h_stage_val[slot], m) != 0)
            return fail(ctx, SCEMA_ERR_STATE, "compare_stream: sink asked to stop");
        return SCEMA_OK;
    };
    uint32_t chunk = 0;
    for (uint32_t p0 = 0; p0 < sc.n_panels; p0 += panels_per_chunk, chunk++) {
        const uint32_t p1 = std::min<uint32_t>(sc.n_panels, p0 + panels_per_chunk);
        const int slot = (int)(chunk & 1);
        // the previous chunk's edges are unpacked and consumed on the host while this one computes:
        // compare_panels blocks the host only at its counter read-back, after its kernels are queued
        rc = compare_panels(ctx, thr, &variant, shard, n_shards, sc, p0, p1, [&]() { return deliver(slot ^ 1); });
        if (rc) return rc;
        const uint64_t m = ctx->n_edges;
        if (m > ctx->stage_cap[slot]) {
            if (ctx->h_stage_key[slot]) { cudaFreeHost(ctx->h_stage_key[slot]); cudaFreeHost(ctx->h_stage_val[slot]); }
            ctx->h_stage_key[slot] = nullptr; ctx->h_stage_val[slot] = nullptr; ctx->stage_cap[slot] = 0;
            const uint64_t cap = m + m / 4 + 1024;
            SCEMA_CUDA(ctx, cudaMallocHost(&ctx->h_stage_key[slot], cap * sizeof(uint64_t)));
            SCEMA_CUDA(ctx, cudaMallocHost(&ctx->h_stage_val[slot], cap * sizeof(double)));
            ctx->stage_cap[slot] = cap;
        }
        if (m) {
            SCEMA_CUDA(ctx, cudaMemcpyAsync(ctx->h_stage_key[slot], ctx->d_edge_key[ctx->edge_cur].p, m * sizeof(uint64_t),
                                            cudaMemcpyDeviceToHost, ctx->stream));
            SCEMA_CUDA(ctx, cudaMemcpyAsync(ctx->h_stage_val[slot], ctx->d_edge_val[ctx->edge_cur].p, m * sizeof(double),
                                            cudaMemcpyDeviceToHost, ctx->stream));
        }
        SCEMA_CUDA(ctx, cudaEventRecord(ctx->stage_ev[slot], ctx->stream));
        st[slot].m = m;
        st[slot].pending = true;
        // fold this chunk's phase timings in before the events are re-recorded by the next chunk
        if (p1 < sc.n_panels) {
            SCEMA_CUDA(ctx, cudaEventSynchronize(ctx->stage_ev[slot]));
            for (int w = SCEMA_T_FILTER; w <= SCEMA_T_SORT; w++)
                if (ctx->ev_used[w]) {
                    float t = 0.f;
                    if (cudaEventElapsedTime(&t, ctx->ev[2 * w], ctx->ev[2 * w + 1]) == cudaSuccess) ctx->acc_ms[w] += t;
                    else cudaGetLastError();
                    ctx->ev_used[w] = false;
                }
        }
    }
    for (int k = 0; k < 2; k++) {
        rc = deliver((int)((chunk + k) & 1));  // older of the two first
        if (rc) return rc;
    }
    ctx->counters[2] = total;
    if (n_shards == 1) ctx->counters[0] = ctx->n * (ctx->n - 1) / 2;
    ctx->have_edges = false;  // the edges went to the sink; nothing is retained on the device
    ctx->n_edges = 0;
    if (n_total) *n_total = total;
    return SCEMA_OK;
}

// ------------------------------------------------------------------------------------------------
// FP64 issue-rate probes (roofline denominators; MEASURED_PEAKS.json has no FP64 figure)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_peak_dfma(double *out, double a, double b, int iters)
{
    double acc[16];
#pragma unroll
    for (int i = 0; i < 16; i++) acc[i] = threadIdx.x * 1e-9 + i;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int i = 0; i < 16; i++) acc[i] = fma(acc[i], a, b);
    }
    double s = 0;
#pragma unroll
    for (int i = 0; i < 16; i++) s += acc[i];
    if (s == 123.456) out[0] = s;
}
__global__ void __launch_bounds__(256) k_peak_dmma(double *out, double av, double bv, int iters)
{
    constexpr int NACC = 8;  // independent accumulator fragments per warp
    double c[NACC][2];
#pragma unroll
    for (int i = 0; i < NACC; i++) c[i][0] = c[i][1] = 0.0;
    const double a = av + threadIdx.x * 1e-12, b = bv;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int i = 0; i < NACC; i++) dmma_m8n8k4(c[i][0], c[i][1], a, b);
    }
    double s = 0;
#pragma unroll
    for (int i = 0; i < NACC; i++) s += c[i][0] + c[i][1];
    if (s == 123.456) out[0] = s;
}

int fp64_peak_run(scema_ctx *ctx, double out[2])
{
    SCEMA_CUDA(ctx, ctx->d_counters.reserve(8 * sizeof(uint64_t)));
    double *d = ctx->d_counters.as<double>();
    const int iters = 8192, blocks = ctx->sm_count * 8;
    cudaEvent_t e0, e1;
    SCEMA_CUDA(ctx, cudaEventCreate(&e0));
    SCEMA_CUDA(ctx, cudaEventCreate(&e1));
    for (int which = 0; which < 2; which++) {
        float best = 1e30f;
        for (int rep = 0; rep < 7; rep++) {
            SCEMA_CUDA(ctx, cudaEventRecord(e0, ctx->stream));
            if (which == 0) k_peak_dfma<<<blocks, 256, 0, ctx->stream>>>(d, 1.0000001, 1e-9, iters);
            else k_peak_dmma<<<blocks, 256, 0, ctx->stream>>>(d, 1.0, 1e-9, iters);
            ctx->launches++;
            SCEMA_CUDA(ctx, cudaEventRecord(e1, ctx->stream));
            SCEMA_CUDA(ctx, cudaEventSynchronize(e1));
            float ms;
            SCEMA_CUDA(ctx, cudaEventElapsedTime(&ms, e0, e1));
            if (rep >= 2 && ms < best) best = ms;
        }
        const double threads = (double)blocks * 256;
        const double flops = which == 0 ? threads * iters * 16 * 2.0 : threads / 32 * iters * 8 * (8 * 8 * 4 * 2.0);
        out[which] = flops / (best * 1e-3) / 1e12;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return SCEMA_OK;
}

}  // namespace scema
