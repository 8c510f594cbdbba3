// K2, tensor-core filter on tcgen05 (SCEMA_PAIRS_TC) — the all-pairs distance of
// compare_histories_with_all_ranks / compare_L2_norm (reference headers/strain2spline.h:546-614,
// :469-484) filtered on the 5th-generation tensor cores, survivors recomputed exactly.
//
// sm_100a has no FP64 kind on tcgen05, so the FP64 contraction a.b of the GEMM form
//        d^2 = |a|^2 + |b|^2 - 2 a.b
// is evaluated on split operands: every scaled FP64 element is cut into two fp16 slices
// a = a_hi + a_lo + r (|r| <= 2^-22 |a|), and one accumulator collects
//        a_hi.b_hi + a_lo.b_hi + a_hi.b_lo            (kind::f16, fp32 accumulate in TMEM)
// The four spare columns of every 64-wide slice carry the row terms, so the tensor core itself
// produces   acc = a.b - h_i - h_j   with h_i = (|a_i|^2 (1 - c) - T'(1/2 + 2c) - e0) / 2, c = 2^-13, and
// the pair is PROVABLY rejected by the reference iff acc < 0 — the epilogue only looks at sign bits
// (one LOP3 per two pairs). Everything else (true edges + a guard band that covers the slicing
// residual and the fp32 accumulation of the tensor core, DESIGN.md "K2-TC") is a survivor and goes
// through the same exact FP64 recompute (k_exact_queue) as the DMMA path: the edge list and the
// distance bits are identical to the reference's.
//
// Kernel: warp-specialised, persistent, one CTA per SM, one 128 x 256 tile per CTA (CG = 1, the default) or
// CG = 2: the two SMs of a TPC on one 256 x 256 tile (tcgen05.mma.cta_group::2: each CTA holds 128 rows of A
// and 128 of the 256 B rows, so B traffic from L2 and the shared-memory reads per SM are halved). Operand blocks are stored in
// global memory exactly as the 128-byte-swizzled K-major image tcgen05 wants in shared memory, so one
// block = one contiguous 1-D bulk copy of the TMA engine (no tensor map).
#include "common.cuh"
#include "tc_sched.h"
#include <cuda_fp16.h>
#include <cub/device/device_radix_sort.cuh>
#include <type_traits>
#include <algorithm>
#include <cmath>
#include <vector>

namespace scema {
namespace tc {

constexpr uint32_t ROWS = 128;                     // rows per operand block
constexpr uint32_t SLICE_BYTES = ROWS * 128;       // 128 rows x 64 fp16, SW128 K-major
constexpr uint32_t BLOCK_BYTES = 2 * SLICE_BYTES;  // hi | lo
constexpr uint32_t COLT = 256;                     // B rows (= pair-matrix columns) per tile
constexpr uint32_t KMAX = 60;                      // data columns per slice (4 more carry the row terms)
// Projected (narrow) operands: PROJ_R coordinates of the centred row in an orthonormal basis of the sample's leading
// principal directions, the norm of the residual, 4 fold columns = 16 fp16 = 32 bytes per row, K-major SWIZZLE_32B
constexpr uint32_t PROJ_R = 11;
constexpr uint32_t NROW_BYTES = 32;
constexpr uint32_t NBLOCK_BYTES = ROWS * NROW_BYTES;  // 4 KB per 128-row block

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
// Wait for a barrier phase. The whole loop is one PTX block (no compiler-visible divergence, hence no BSSY/BSYNC and
// no reconvergence code around it: the single-thread roles execute three of these per tile and their instruction
// count IS the critical path). Bounded: after WAIT_SPINS failed polls (each poll itself blocks for a hardware time
// slice; seconds in total) the thread traps, so a protocol bug ends the kernel instead of hanging the GPU.
constexpr uint32_t WAIT_SPINS = 1u << 26;
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int /*tag*/)
{
    asm volatile(
        "{\n"
        ".reg .pred P1, P2;\n"
        ".reg .u32 n;\n"
        "mov.u32 n, 0;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "add.u32 n, n, 1;\n"
        "setp.lt.u32 P2, n, %2;\n"
        "@P2 bra LAB_WAIT;\n"
        "trap;\n"
        "DONE:\n"
        "}\n" ::"r"(bar),
        "r"(parity), "r"(WAIT_SPINS)
        : "memory");
}
// arrive on the barrier at the same shared-memory offset in CTA `cta` of the cluster
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar, uint32_t cta)
{
    asm volatile(
        "{\n"
        ".reg .b32 ra;\n"
        "mapa.shared::cluster.u32 ra, %0, %1;\n"
        "mbarrier.arrive.shared::cluster.b64 _, [ra];\n"
        "}\n" ::"r"(bar),
        "r"(cta)
        : "memory");
}
__device__ __forceinline__ void mbar_arrive_local(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
// One lane of a converged warp. The single-thread roles (TMA producer, MMA issuer) run their loops with the WHOLE warp
// converged and only the issuing instructions under this predicate: addresses, descriptors and barrier phases are then
// warp-uniform for the compiler and live in uniform registers. (Round 1 ran these loops inside `if (lane == 0)`: in
// divergent code every UTCHMMA / UBLKCP / UTCBAR is wrapped in an ELECT + R2UR.BROADCAST + BRA.U.ANY loop, and the
// issuer needed ~1000 cycles of instruction latency per tile for 512 cycles of tensor work — ncu source page,
// profiles/r02_k2_issue_loop.txt.)
__device__ __forceinline__ bool elect_one()
{
    uint32_t pred;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "elect.sync _|p, 0xffffffff;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ uint32_t and3(uint32_t a, uint32_t b, uint32_t c)
{
    uint32_t d;
    asm("lop3.b32 %0, %1, %2, %3, 0x80;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ void fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ uint32_t cluster_rank()
{
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all()
{
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

template <int CG>
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate)
{
    if (CG == 1)
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "setp.ne.b32 p, %4, 0;\n"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
            "}\n" ::"r"(d_tmem),
            "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
            : "memory");
    else
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "setp.ne.b32 p, %4, 0;\n"
            "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
            "}\n" ::"r"(d_tmem),
            "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
            : "memory");
}
// arrive on `bar` (same offset in every CTA of the group) once all MMAs issued so far have completed
template <int CG>
__device__ __forceinline__ void umma_commit(uint32_t bar)
{
    if (CG == 1)
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
    else
        asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
                     "h"((uint16_t)3)
                     : "memory");
}
template <int CG>
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t cols)
{
    if (CG == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    } else {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
}
template <int CG>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols)
{
    if (CG == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// 32 lanes x 64 consecutive fp32 columns: thread t of the warp gets row (lane base + t)
__device__ __forceinline__ void tmem_ld64(uint32_t taddr, uint32_t (&v)[64])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x64.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, "
        "%32, %33, %34, %35, %36, %37, %38, %39, %40, %41, %42, %43, %44, %45, %46, %47, "
        "%48, %49, %50, %51, %52, %53, %54, %55, %56, %57, %58, %59, %60, %61, %62, %63}, [%64];\n"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31]), "=r"(v[32]),
          "=r"(v[33]), "=r"(v[34]), "=r"(v[35]), "=r"(v[36]), "=r"(v[37]), "=r"(v[38]), "=r"(v[39]), "=r"(v[40]),
          "=r"(v[41]), "=r"(v[42]), "=r"(v[43]), "=r"(v[44]), "=r"(v[45]), "=r"(v[46]), "=r"(v[47]), "=r"(v[48]),
          "=r"(v[49]), "=r"(v[50]), "=r"(v[51]), "=r"(v[52]), "=r"(v[53]), "=r"(v[54]), "=r"(v[55]), "=r"(v[56]),
          "=r"(v[57]), "=r"(v[58]), "=r"(v[59]), "=r"(v[60]), "=r"(v[61]), "=r"(v[62]), "=r"(v[63])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 64-bit shared-memory matrix descriptor, K-major, 128-byte swizzle: 8-row groups 1024 bytes apart
// (SBO), descriptor version 1 (sm_100), layout type 2 = SWIZZLE_128B. Address and offsets in 16-byte units.
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr)
{
    const uint32_t hi = (1024u >> 4) | (1u << 14) | (2u << 29);
    return ((uint64_t)hi << 32) | (uint64_t)((smem_addr >> 4) & 0x3FFFu);
}
// The same for the narrow operands: rows of 32 bytes (K = 16 fp16, exactly one MMA step), 8-row groups 256 bytes apart,
// layout type 6 = SWIZZLE_32B (16-byte chunk c of row r stored at chunk c ^ ((r >> 2) & 1)).
__device__ __forceinline__ uint64_t make_desc32(uint32_t smem_addr)
{
    const uint32_t hi = (256u >> 4) | (1u << 14) | (6u << 29);
    return ((uint64_t)hi << 32) | (uint64_t)((smem_addr >> 4) & 0x3FFFu);
}

struct Args {
    const unsigned char *HA, *HB;  // [n_pad/128][hi|lo][128 rows][128 bytes, 16-byte chunks XOR-swizzled by row & 7]
    unsigned long long *cand_count;
    uint64_t *cand;
    uint64_t cand_cap;
    uint64_t n;
    uint32_t NT;       // column tiles (256 rows each)
    uint32_t I0, I1;   // row range of this launch, in 256-row tiles
    uint32_t C0, C1;   // column range of this launch, in 256-row tiles (all pairs: 0 .. NT)
    uint32_t strip_len;
    uint32_t shard, n_shards;
    uint32_t slices;   // 2: a_hi.b_hi + a_lo.b_hi + a_hi.b_lo; 1: a_hi.b_hi only (coarser guard band, a third of the MMAs)
    uint32_t nc;       // 64-column chunks per row (K <= 60: 1); a 128-row block holds nc x [hi | lo]
    uint32_t compact;  // 1: hi-only operand copies (a 128-row block holds nc x hi, 16 KB each): the layout a sharded
                       // compare all-gathers between the GPUs (one slice only)
    // shared-memory plan (tc_launch): A buffers of a_bytes each, then a ring of 2^lg_nst B stages
    uint32_t a_bytes, n_abuf, lg_nst, stage_bytes, data_bytes;
    // norm-band mode (rows sorted by norm): band schedule + map from sorted position to row index
    const uint32_t *band_item_start, *band_jend, *perm;
    uint32_t band_row_tiles;
    float *dbg;        // debug: every accumulator of every tile, dbg[row * dbg_ld + col]
    uint64_t dbg_ld;
};

template <int CG>
__device__ __forceinline__ void sched_init(Sched<CG> &sc, const Args &, const SchedArgs &sa, uint32_t unit, uint32_t n_units)
{
    sc.init(sa, unit, n_units);
}
template <int CG>
__device__ __forceinline__ void sched_init(BandSched<CG> &sc, const Args &a, const SchedArgs &sa, uint32_t unit, uint32_t n_units)
{
    sc.init(a.band_item_start, a.band_jend, a.band_row_tiles, sa.strip_len, sa.shard, sa.n_shards, unit, n_units);
}

template <int CG>
struct Smem {
    static constexpr uint32_t B_ROWS = COLT / CG;                 // B rows held by one CTA
    static constexpr uint32_t B_SLICE = B_ROWS * 128;             // bytes of one slice of a B stage (one chunk)
    static constexpr uint32_t B_STAGE = 2 * B_SLICE;
    static constexpr uint32_t DATA_MAX = 224 * 1024;              // operand tiles: A buffers, then the B ring
    static constexpr uint32_t MAXST = 16;
    static constexpr uint32_t n_bars = 3 * MAXST + 6;             // full, pfull, empty | a_empty[2] tfull[2] tempty[2]
    static constexpr uint32_t tail = n_bars * 8 + 16 + 1024;      // barriers, TMEM address, slack to align the base to 1024
};

// WIDE = false: rows of one chunk (K <= 60) with a compile-time shared-memory plan (A double-buffered at a 32 KB
// stride, B ring behind it); WIDE = true: several chunks per row, plan from tc_launch.
// BAND = true: rows are sorted by norm and only the band of tiles the triangle inequality cannot rule out is walked.
// NARROW = true: projected 16-column operands (k_tc_prep_proj), 4 KB per 128-row block, one MMA step per tile.
template <int CG, bool DBG, bool WIDE, bool BAND, bool NARROW = false>
__global__ void __launch_bounds__(384, 1) k_filter_tc(const Args a)
{
    using SchedT = typename std::conditional<BAND, BandSched<CG>, Sched<CG>>::type;
    using SM = Smem<CG>;
    constexpr uint32_t MAXST = SM::MAXST;
    extern __shared__ unsigned char smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    const uint32_t k_nc = WIDE ? a.nc : 1u;                               // chunks per row
    const uint32_t k_nabuf = WIDE ? a.n_abuf : 2u;                        // A buffers
    const uint32_t k_abytes = WIDE ? a.a_bytes : NARROW ? NBLOCK_BYTES : BLOCK_BYTES;  // bytes per A buffer
    const uint32_t sA = base, sB = base + k_nabuf * k_abytes, sBar = base + a.data_bytes;
    auto bar_full = [&](uint32_t i) { return sBar + 8 * i; };
    auto bar_pfull = [&](uint32_t i) { return sBar + 8 * (MAXST + i); };
    auto bar_empty = [&](uint32_t i) { return sBar + 8 * (2 * MAXST + i); };
    auto bar_aempty = [&](uint32_t i) { return sBar + 8 * (3 * MAXST + i); };
    auto bar_tfull = [&](uint32_t i) { return sBar + 8 * (3 * MAXST + 2 + i); };
    auto bar_tempty = [&](uint32_t i) { return sBar + 8 * (3 * MAXST + 4 + i); };
    // B ring: one stage = one 64-column chunk of a column tile (its hi rows alone with one slice, which gives
    // twice the stages in the same memory); A: all chunks of the row tile, double-buffered over items when it fits
    const uint32_t lg_nst = a.lg_nst, nst_mask = (1u << lg_nst) - 1u, stage_bytes = a.stage_bytes;
    // bytes of one chunk of an A tile in shared memory, of one slice of a 128-row block, of one chunk of a 128-row
    // block in global memory
    const uint32_t a_chunk = NARROW ? NBLOCK_BYTES : a.slices == 1 ? SLICE_BYTES : BLOCK_BYTES;
    const uint32_t b_slice = NARROW ? NBLOCK_BYTES : SLICE_BYTES;
    const uint32_t g_chunk = NARROW ? NBLOCK_BYTES : a.compact ? SLICE_BYTES : BLOCK_BYTES;
    const uint64_t gblk = (uint64_t)k_nc * g_chunk;                      // bytes of a 128-row block in global memory
    const uint32_t off_tmem = a.data_bytes + SM::n_bars * 8;
    volatile uint32_t *tmem_slot = reinterpret_cast<volatile uint32_t *>(smem_raw + (base - raw) + off_tmem);

    const uint32_t tid = threadIdx.x, lane = tid & 31;
    const uint32_t warp = __shfl_sync(0xffffffffu, tid >> 5, 0);  // warp-uniform for the compiler
    const uint32_t rank = CG == 2 ? cluster_rank() : 0u;
    const SchedArgs sa = {a.NT, a.I0, a.I1, a.C0, a.C1, a.strip_len, a.shard, a.n_shards};
    const uint32_t unit = blockIdx.x / CG, n_units = gridDim.x / CG;

    if (tid == 0) {
        for (uint32_t i = 0; i < MAXST; i++) { mbar_init(bar_full(i), 1); mbar_init(bar_pfull(i), 1); mbar_init(bar_empty(i), 1); }
        for (uint32_t i = 0; i < 2; i++) { mbar_init(bar_aempty(i), 1); mbar_init(bar_tfull(i), 1); mbar_init(bar_tempty(i), 8 * CG); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) tmem_alloc<CG>(base + off_tmem, 512);
    fence_before();
    if (CG == 2) cluster_sync_all(); else __syncthreads();
    fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ------------------------------------------------------------------ producer: TMA bulk copies
        // (whole warp converged; one elected lane arms the barrier and issues the copies)
        SchedT sc;
        sched_init(sc, a, sa, unit, n_units);
        uint32_t I, J0, J1, t = 0, item = 0;
        const uint32_t nc = k_nc, n_abuf = k_nabuf, a_bytes = k_abytes, slices = NARROW ? 1u : a.slices;
        const unsigned char *const HA = a.HA, *const HB = a.HB;
        while (sc.next(I, J0, J1)) {
            const uint32_t ab = n_abuf == 2 ? (item & 1u) : 0u;
            mbar_wait(bar_aempty(ab), ((n_abuf == 2 ? (item >> 1) : item) & 1u) ^ 1u, 1);
            for (uint32_t J = J0; J < J1; J++)
                for (uint32_t c = 0; c < nc; c++, t++) {
                    const uint32_t st = t & nst_mask;
                    mbar_wait(bar_empty(st), ((t >> lg_nst) & 1u) ^ 1u, 2);
                    const bool first = J == J0 && c == 0;  // the item's A tile (all chunks) rides on its first stage
                    const uint32_t dst = sB + st * stage_bytes;
                    if (elect_one()) {
                        mbar_expect_tx(bar_full(st), (COLT / CG / ROWS) * a_chunk + (first ? nc * a_chunk : 0u));
                        if (first)
                            for (uint32_t ca = 0; ca < nc; ca++)
                                bulk_g2s(sA + ab * a_bytes + ca * a_chunk, HA + (uint64_t)(I * CG + rank) * gblk + (uint64_t)ca * g_chunk,
                                         a_chunk, bar_full(st));
                        if (CG == 2) {
                            bulk_g2s(dst, HB + (uint64_t)(J * 2 + rank) * gblk + (uint64_t)c * g_chunk, a_chunk, bar_full(st));
                        } else {
                            // 256 B rows of one CTA: the hi slices of both 128-row blocks, then both lo slices
                            const unsigned char *b0 = HB + (uint64_t)(J * 2) * gblk + (uint64_t)c * g_chunk;
                            bulk_g2s(dst, b0, b_slice, bar_full(st));
                            bulk_g2s(dst + b_slice, b0 + gblk, b_slice, bar_full(st));
                            if (slices != 1) {
                                bulk_g2s(dst + 2 * SLICE_BYTES, b0 + SLICE_BYTES, SLICE_BYTES, bar_full(st));
                                bulk_g2s(dst + 3 * SLICE_BYTES, b0 + gblk + SLICE_BYTES, SLICE_BYTES, bar_full(st));
                            }
                        }
                    }
                    __syncwarp();
                }
            item++;
        }
    } else if (warp == 1) {
        if (rank == 0) {
            // -------------------------------------------------------------- MMA issuer (leader CTA)
            // whole warp converged, the MMAs and their commits issued by one elected lane (always the same one)
            // instruction descriptor: D fp32, A/B fp16, both K-major, N = 256, M = 128 * CG
            const uint32_t idesc = (1u << 4) | ((COLT >> 3) << 17) | (((128u * CG) >> 4) << 24);
            SchedT sc;
            sched_init(sc, a, sa, unit, n_units);
            uint32_t I, J0, J1, t = 0, item = 0, tile = 0;
            const uint32_t n_terms = a.slices == 1 ? 1u : 3u, nc = k_nc, n_abuf = k_nabuf, a_bytes = k_abytes;
            while (sc.next(I, J0, J1)) {
                const uint32_t ab = n_abuf == 2 ? (item & 1u) : 0u;
                const uint32_t a_tile = sA + ab * a_bytes;
                for (uint32_t J = J0; J < J1; J++, tile++) {
                    const uint32_t as = tile & 1u;
                    const uint32_t d_tmem = tmem_base + as * COLT;
                    for (uint32_t c = 0; c < nc; c++, t++) {
                        // operands first (they were prefetched: the barrier is normally complete already), the
                        // accumulator stage last, so that nothing but the MMA issue follows the epilogue's release
                        const uint32_t st = t & nst_mask, ph = (t >> lg_nst) & 1u;
                        mbar_wait(bar_full(st), ph, 4);
                        if (CG == 2) mbar_wait(bar_pfull(st), ph, 5);
                        const uint64_t adesc = NARROW ? make_desc32(a_tile) : make_desc(a_tile + c * a_chunk);
                        const uint64_t bdesc = NARROW ? make_desc32(sB + st * stage_bytes) : make_desc(sB + st * stage_bytes);
                        if (c == 0) mbar_wait(bar_tempty(as), ((tile >> 1) & 1u) ^ 1u, 3);
                        fence_after();
                        if (elect_one()) {
                            // a_hi.b_hi (one slice), then a_lo.b_hi and a_hi.b_lo (two slices); narrow: the whole row is
                            // one K = 16 step
                            if (NARROW) {
                                umma_f16<CG>(d_tmem, adesc, bdesc, idesc, 0u);
                            } else {
#pragma unroll
                                for (uint32_t kk = 0; kk < 4; kk++)
                                    umma_f16<CG>(d_tmem, adesc + 2 * kk, bdesc + 2 * kk, idesc, (c | kk) != 0 ? 1u : 0u);
                            }
                            if (!NARROW && n_terms != 1) {
#pragma unroll
                                for (uint32_t kk = 0; kk < 4; kk++)
                                    umma_f16<CG>(d_tmem, adesc + (SLICE_BYTES >> 4) + 2 * kk, bdesc + 2 * kk, idesc, 1u);
#pragma unroll
                                for (uint32_t kk = 0; kk < 4; kk++)
                                    umma_f16<CG>(d_tmem, adesc + 2 * kk, bdesc + (SM::B_SLICE >> 4) + 2 * kk, idesc, 1u);
                            }
                            umma_commit<CG>(bar_empty(st));
                            if (c == nc - 1) {
                                umma_commit<CG>(bar_tfull(as));
                                if (J == J1 - 1) umma_commit<CG>(bar_aempty(ab));
                            }
                        }
                        __syncwarp();
                    }
                }
                item++;
            }
        } else if (CG == 2) {
            // ---------------------------- peer CTA: tell the leader when this CTA's half of a stage landed
            SchedT sc;
            sched_init(sc, a, sa, unit, n_units);
            uint32_t I, J0, J1, t = 0;
            const uint32_t nc_fw = k_nc;
            while (sc.next(I, J0, J1))
                for (uint32_t q = (J1 - J0) * nc_fw; q > 0; q--, t++) {
                    const uint32_t st = t & nst_mask;
                    mbar_wait(bar_full(st), (t >> lg_nst) & 1u, 6);
                    if (elect_one()) mbar_arrive_cluster(bar_pfull(st), 0);
                    __syncwarp();
                }
        }
    } else if (warp >= 4) {
        // ---------------------------------------------------------------------- epilogue (8 warps)
        // warp -> (TMEM lane quarter it may read, column half of the tile)
        const uint32_t q = warp & 3u, half = (warp - 4u) >> 2;
        SchedT sc;
        sched_init(sc, a, sa, unit, n_units);
        uint32_t I, J0, J1, tile = 0;
        while (sc.next(I, J0, J1)) {
            const uint64_t row = (uint64_t)(I * CG + rank) * ROWS + q * 32 + lane;
            for (uint32_t J = J0; J < J1; J++, tile++) {
                const uint32_t as = tile & 1u;
                mbar_wait(bar_tfull(as), (tile >> 1) & 1u, 7);
                fence_after();
                uint32_t v0[64], v1[64];
                const uint32_t taddr = tmem_base + ((q * 32u) << 16) + as * COLT + half * 128u;
                tmem_ld64(taddr, v0);
                tmem_ld64(taddr + 64u, v1);
                tmem_ld_wait();
                // the accumulator stage is free again as soon as the values sit in registers
                fence_before();
                __syncwarp();
                if (lane == 0) {
                    if (CG == 2) mbar_arrive_cluster(bar_tempty(as), 0);
                    else mbar_arrive_local(bar_tempty(as));
                }
                // acc < 0 for every pair <=> the AND of the bit patterns keeps the sign bit
                // Eight independent chains of three-input ANDs, spelled in PTX: left to the compiler, the 128 values are
                // re-associated into ONE chain of 64 dependent LOP3s (~5 cycles each = 310 of the warp's ~710 cycles per
                // tile, profiles/r02_ncu_filter_tc_roles.txt)
                uint32_t an[8];
#pragma unroll
                for (int c = 0; c < 8; c++) an[c] = v0[c] & v1[c];
#pragma unroll
                for (int c = 8; c < 64; c++) an[c & 7] = and3(an[c & 7], v0[c], v1[c]);
                const uint32_t all_neg = and3(and3(an[0], an[1], an[2]), and3(an[3], an[4], an[5]), an[6] & an[7]);
                const uint64_t col0 = (uint64_t)J * COLT + half * 128u;
                if (DBG && a.dbg) {
#pragma unroll
                    for (int c = 0; c < 64; c++) {
                        a.dbg[row * a.dbg_ld + col0 + c] = __uint_as_float(v0[c]);
                        a.dbg[row * a.dbg_ld + col0 + 64 + c] = __uint_as_float(v1[c]);
                    }
                }
                if (__any_sync(0xffffffffu, (all_neg >> 31) == 0u)) {
                    // survivors of this warp's 32 x 128 accumulators: one bit mask per lane, one atomic per warp
                    // (a queue counter hit once per column serialises in L2 when many tiles carry survivors)
                    uint32_t km[4] = {0u, 0u, 0u, 0u};
#pragma unroll
                    for (int c = 0; c < 128; c++) {
                        const uint64_t col = col0 + c;
                        const uint32_t bitsv = c < 64 ? v0[c & 63] : v1[c & 63];
                        const bool keep = (bitsv >> 31) == 0u && row < col && col < a.n;
                        km[c >> 5] |= (keep ? 1u : 0u) << (c & 31);
                    }
                    const uint32_t mine = __popc(km[0]) + __popc(km[1]) + __popc(km[2]) + __popc(km[3]);
                    uint32_t incl = mine;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const uint32_t up = __shfl_up_sync(0xffffffffu, incl, o);
                        if ((int)lane >= o) incl += up;
                    }
                    const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
                    if (total) {
                        unsigned long long base = 0;
                        if (lane == 31) base = atomicAdd(a.cand_count, (unsigned long long)total);
                        unsigned long long pos = __shfl_sync(0xffffffffu, base, 31) + (incl - mine);
#pragma unroll
                        for (int w = 0; w < 4; w++) {
                            uint32_t m = km[w];
                            while (m) {
                                const uint32_t b = __ffs(m) - 1;
                                m &= m - 1;
                                if (pos < a.cand_cap) {
                                    uint64_t ri = row, ci = col0 + 32u * w + b;
                                    if (BAND) {  // sorted positions -> row indices, smaller one first
                                        const uint32_t pr = a.perm[ri], pc = a.perm[ci];
                                        ri = pr < pc ? pr : pc;
                                        ci = pr < pc ? pc : pr;
                                    }
                                    a.cand[pos] = (ri << 32) | ci;
                                }
                                pos++;
                            }
                        }
                    }
                }
            }
        }
    }

    // teardown: nobody may leave (or free TMEM) while its partner CTA can still signal it
    fence_before();
    if (CG == 2) cluster_sync_all(); else __syncthreads();
    fence_after();
    if (warp == 2) tmem_dealloc<CG>(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------
// operand preparation
// ------------------------------------------------------------------------------------------------
// pass 1: row norms (FP64) and the largest finite magnitude of the rows [r0, r1)
// ---- centre of the filter copies. d(a, b) = d(a - m, b - m) for ANY vector m, and the guard band of the filter scales
// with |a - m|^2 + |b - m|^2: on production-shaped data (every quadrature point on nearly the same stretch path,
// FE_problem.h:1091-1103; rows differ by ~1 % of their norm) the band of the un-centred rows keeps every pair, that of
// the centred rows only real neighbours. m = column MEDIANS over a fixed sample of <= 4096 rows (non-finite entries
// skipped): a mean is dragged away from the bulk by one row at 1e200 or by a minority cloud far from everybody else,
// a median is not; and it is deterministic, so every rank of a sharded compare derives the same m from the same rows.
// One block per column, bitonic sort in shared memory. The exact recompute never sees m: k_exact_queue reads the
// original rows.
constexpr uint32_t CENTRE_SAMPLE = 4096;
__global__ void __launch_bounds__(256) k_tc_centre_median(const double *__restrict__ S, uint64_t r0, uint64_t r1, uint32_t K,
                                                          double *__restrict__ centre)
{
    __shared__ double v[CENTRE_SAMPLE];
    __shared__ unsigned int s_cnt;
    const uint32_t k = blockIdx.x;
    const uint64_t n = r1 - r0;
    const uint64_t ns = n < CENTRE_SAMPLE ? n : CENTRE_SAMPLE;
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    unsigned int mine = 0;
    for (uint32_t j = threadIdx.x; j < CENTRE_SAMPLE; j += blockDim.x) {
        double x = INFINITY;  // padding and non-finite entries sort to the end
        if (j < ns) {
            const double y = S[(r0 + j * (n / ns)) * K + k];
            if (isfinite(y)) { x = y; mine++; }
        }
        v[j] = x;
    }
    atomicAdd(&s_cnt, mine);
    __syncthreads();
    for (uint32_t size = 2; size <= CENTRE_SAMPLE; size <<= 1)
        for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
            for (uint32_t t = threadIdx.x; t < CENTRE_SAMPLE / 2; t += blockDim.x) {
                const uint32_t lo = 2 * t - (t & (stride - 1)), hi = lo + stride;
                const bool up = (lo & size) == 0;
                const double a = v[lo], b = v[hi];
                if ((a > b) == up) { v[lo] = b; v[hi] = a; }
            }
            __syncthreads();
        }
    if (threadIdx.x == 0) centre[k] = s_cnt ? v[(s_cnt - 1) / 2] : 0.0;
}

__global__ void __launch_bounds__(256) k_tc_rowstats(const double *__restrict__ S, const double *__restrict__ centre, uint64_t r0,
                                                     uint64_t r1, uint32_t K, double *__restrict__ NRM,
                                                     unsigned long long *__restrict__ gmax)
{
    __shared__ double s_max[8];
    const uint64_t row = r0 + (uint64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double nrm = 0.0, m = 0.0;
    if (row < r1)
        for (uint32_t k = lane; k < K; k += 32) {
            const double v = __dsub_rn(S[row * K + k], centre[k]);
            nrm = fma(v, v, nrm);
            m = fmax(m, fabs(v));
        }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        nrm += __shfl_xor_sync(0xffffffffu, nrm, o);
        m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    }
    if (lane == 0) {
        if (row < r1) NRM[row] = nrm;
        s_max[warp] = (row < r1 && isfinite(nrm)) ? m : 0.0;  // rows with a non-finite norm take no part in the scale
        if (gmax && row < r1 && !isfinite(nrm)) atomicAdd(gmax + 4, 1ull);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double bm = 0.0;
#pragma unroll
        for (int w = 0; w < 8; w++) bm = fmax(bm, s_max[w]);
        if (gmax && bm > 0.0) atomicMax(gmax, (unsigned long long)__double_as_longlong(bm));  // non-negative doubles order as integers
    }
}

constexpr uint32_t HIST_BINS = 2112;   // exponent of a squared norm + 1075 (0: zero norm)
constexpr uint32_t PLAN_WORD = 8 + HIST_BINS;  // five counters of the survivor-density sample behind the histogram
constexpr uint32_t MISC_WORDS = 8 + HIST_BINS + 8;
constexpr uint32_t MAX_OUTLIERS = 16;  // rows the scale may leave behind (they survive against everybody)

// histogram of the exponents of the finite squared norms of rows [r0, r1) into misc[8 ..]
__global__ void __launch_bounds__(256) k_tc_nrm_hist(const double *__restrict__ NRM, uint64_t r0, uint64_t r1,
                                                     unsigned long long *__restrict__ misc)
{
    __shared__ unsigned int h[HIST_BINS];
    for (uint32_t b = threadIdx.x; b < HIST_BINS; b += blockDim.x) h[b] = 0;
    __syncthreads();
    for (uint64_t i = r0 + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < r1; i += (uint64_t)gridDim.x * blockDim.x) {
        const double v = NRM[i];
        if (isfinite(v)) atomicAdd(&h[v > 0.0 ? (uint32_t)(ilogb(v) + 1075) : 0u], 1u);
    }
    __syncthreads();
    for (uint32_t b = threadIdx.x; b < HIST_BINS; b += blockDim.x)
        if (h[b]) atomicAdd(misc + 8 + b, (unsigned long long)h[b]);
}

// Power-of-two scale that brings the largest finite magnitude into [2^(11-headroom), 2^(12-headroom)).
// misc[0] = largest magnitude seen (bits), misc[1] = the scale (double bits), misc[2] = rows whose scaled
// magnitude reached the limit, misc[3] = tiles of the norm band, misc[4] = rows with a non-finite norm,
// misc[8 ..] = histogram of the squared-norm exponents.
// A handful of rows many decades above the rest would push everybody else into the flushed range of fp16 (every
// pair a survivor). If at most MAX_OUTLIERS rows sit at least 12 binades of squared norm (6 of magnitude) above all
// others, the scale is taken from the others instead: |v| <= |row| < 2^((E+1)/2) for a row whose squared norm has
// exponent E; the rows left behind exceed the limit in k_tc_prep and are treated like rows with a non-finite norm.
__global__ void __launch_bounds__(256) k_tc_fix_scale(unsigned long long *misc, int headroom)
{
    __shared__ int s_hi;
    if (threadIdx.x == 0) s_hi = -1;
    __syncthreads();
    for (int b = threadIdx.x + 1; b < (int)HIST_BINS; b += blockDim.x)   // highest populated bin, all threads
        if (misc[8 + b]) atomicMax(&s_hi, b);
    __syncthreads();
    if (threadIdx.x != 0) return;
    const double maxabs = __longlong_as_double((long long)misc[0]);
    double s = 1.0;
    if (maxabs > 0.0) {
        int top = ilogb(maxabs);  // exponent the scale is built on
        const int e_hi = s_hi;
        if (e_hi > 0) {
            unsigned long long above = 0;
            for (int b = e_hi; b > 0; b--) {
                above += misc[8 + b];
                if (above > MAX_OUTLIERS) break;
                int nb = b - 1;  // next populated bin below
                while (nb > 0 && !misc[8 + nb]) nb--;
                if (nb > 0 && b - nb >= 12) {
                    // rows in bins >= b are left behind; everybody else has |v| < 2^((E+1)/2), E = nb - 1075
                    const int E = nb - 1075;
                    const int cap = (E + 1 + (E + 1 >= 0 ? 1 : 0)) / 2;  // ceil((E + 1) / 2)
                    if (cap - 1 < top) top = cap - 1;                     // as if the largest magnitude were just below 2^cap
                    break;
                }
            }
        }
        int se = 11 - headroom - top;
        se = max(-1000, min(1000, se));
        s = scalbn(1.0, se);
    }
    misc[1] = (unsigned long long)__double_as_longlong(s);
}

// fp16 rounding with subnormal results flushed to zero: the operands never contain an fp16 subnormal, so
// whether the tensor core would flush them itself does not matter (the error bound budgets 2^-14 per element)
__device__ __forceinline__ double h16z(double v)
{
    const float f = __half2float(__double2half(v));
    return fabsf(f) < 6.103515625e-05f ? 0.0 : (double)f;
}

// pass 2: one warp per row. Writes the row's hi and lo fp16 slices, chunk by chunk (64 columns each; the last
// chunk has at most 60 data columns and 4 columns carrying the row term -h_i, split three ways against the
// constants P = 2^15 and Q = 2^3 on the other operand), into the A-flavoured and the B-flavoured copy, already in
// the swizzled shared-memory image.
//   A hi: [x0 x1 P Q]   A lo: [0 x2 0 0]        B hi: [P Q x0 x1]   B lo: [0 0 0 x2]
// so that  A_hi.B_hi + A_lo.B_hi + A_hi.B_lo  adds  (P x0 + Q x1 + Q x2)_i + (P x0 + Q x1 + Q x2)_j = -h_i - h_j
// (to 2^-33 |h| + 2^-11; with the hi slices alone the x2 terms drop out: 2^-22 |h| + 2^-11).
__global__ void __launch_bounds__(256) k_tc_prep(const double *__restrict__ S, uint64_t n, uint64_t r0, uint64_t r1, uint32_t K,
                                                 uint32_t nc, uint32_t slices, double vmax, const double *__restrict__ NRM,
                                                 unsigned long long *__restrict__ misc, double T0, double cguard,
                                                 const uint32_t *__restrict__ perm, const double *__restrict__ centre, uint32_t compact,
                                                 uint32_t vec, unsigned char *__restrict__ HA, unsigned char *__restrict__ HB)
{
    const uint64_t row = r0 + (uint64_t)blockIdx.x * 8 + (threadIdx.x >> 5);  // position in the operand copies
    const int lane = threadIdx.x & 31;
    if (row >= r1) return;
    const double s = __longlong_as_double((long long)misc[1]);
    const bool real = row < n;
    const uint64_t src = real && perm ? perm[row] : row;                     // row of S (norm-band mode: sorted order)
    const bool wild = real && !isfinite(NRM[src]);
    const bool data = real && !wild;
    // Lane l owns the ADJACENT columns 2l and 2l + 1 of every 64-column chunk (K = 6 P is even, so a pair never straddles
    // the end of the row): one 16-byte load per pair and pass, one 4-byte store per pair and copy.
    // norm of the scaled row; a row beyond the range the scale was chosen for (possible only when the scale was
    // fixed before every row had been seen) gets no fp16 image and survives against everybody, like a row with
    // a non-finite norm
    auto load2 = [&](uint32_t kd, double &v0, double &v1) {   // scaled, centred columns kd, kd + 1 (0 beyond the row)
        v0 = v1 = 0.0;
        if (kd + 1 < K) {
            double2 x, m;
            if (vec) { x = *reinterpret_cast<const double2 *>(S + src * K + kd); m = *reinterpret_cast<const double2 *>(centre + kd); }
            else { x = make_double2(S[src * K + kd], S[src * K + kd + 1]); m = make_double2(centre[kd], centre[kd + 1]); }
            v0 = __dsub_rn(x.x, m.x) * s;
            v1 = __dsub_rn(x.y, m.y) * s;
        } else if (kd < K) {
            v0 = __dsub_rn(S[src * K + kd], centre[kd]) * s;
        }
    };
    double nrm = 0.0, first0 = 0.0, first1 = 0.0;
    bool big = false;
    if (data)
        for (uint32_t c = 0; c < nc; c++) {
            double v0, v1;
            load2(c * 64 + 2 * lane, v0, v1);
            if (c == 0) { first0 = v0; first1 = v1; }
            nrm = fma(v0, v0, nrm);
            nrm = fma(v1, v1, nrm);
            big |= fabs(v0) >= vmax || fabs(v1) >= vmax;
        }
    const bool too_big = __any_sync(0xffffffffu, big);
    if (too_big && lane == 0) atomicAdd(misc + 2, 1ull);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) nrm += __shfl_xor_sync(0xffffffffu, nrm, o);
    if (too_big) nrm = 0.0;
    // row term
    const double P = 32768.0, Q = 8.0;
    const double T0s = (T0 * s) * s;
    const double e0 = (double)K * 0.0078125;  // K 2^-7: flushed fp16 subnormals (data and fold slices)
    const double h = 0.5 * (nrm * (1.0 - cguard) - T0s * (0.5 + 2.0 * cguard) - e0);
    double x0, x1, x2;
    if (!real) { x0 = -65504.0; x1 = x2 = 0.0; }                              // padding row: never a survivor
    else if (wild || too_big || !(-h <= 32768.0 * P)) { x0 = 65504.0; x1 = x2 = 0.0; }  // always a survivor
    else {
        x0 = h16z(-h / P);
        x1 = h16z((-h - P * x0) / Q);
        x2 = h16z((-h - P * x0 - Q * x1) / Q);
    }
    const uint64_t blk = row / ROWS;
    const uint32_t r = (uint32_t)(row % ROWS);
    const bool two = slices != 1;  // the one-slice kernel never reads the lo halves: neither computed nor written
    for (uint32_t c = 0; c < nc; c++) {
        const uint64_t base = (blk * nc + c) * (compact ? SLICE_BYTES : BLOCK_BYTES) + (uint64_t)r * 128;
        const uint32_t k = 2 * lane;       // columns k, k + 1 of the chunk
        double v0 = 0.0, v1 = 0.0;
        if (data && !too_big) {
            if (c == 0) { v0 = first0; v1 = first1; }
            else load2(c * 64 + k, v0, v1);
        }
        const double hi0 = h16z(v0), hi1 = h16z(v1);
        __half2 ahi = __halves2half2(__double2half(hi0), __double2half(hi1)), bhi = ahi;
        __half2 alo = __halves2half2(__double2half(0.0), __double2half(0.0)), blo = alo;
        if (two) alo = blo = __halves2half2(__double2half(h16z(v0 - hi0)), __double2half(h16z(v1 - hi1)));
        if (c == nc - 1 && k >= KMAX) {
            // fold columns 60..63:  A hi [x0 x1 | P Q], A lo [0 x2 | 0 0];  B hi [P Q | x0 x1], B lo [0 0 | 0 x2]
            const __half z = __double2half(0.0);
            if (k == KMAX) {
                ahi = __halves2half2(__double2half(x0), __double2half(x1));
                bhi = __halves2half2(__double2half(P), __double2half(Q));
                alo = __halves2half2(z, __double2half(x2));
                blo = __halves2half2(z, z);
            } else {
                ahi = __halves2half2(__double2half(P), __double2half(Q));
                bhi = __halves2half2(__double2half(x0), __double2half(x1));
                alo = __halves2half2(z, z);
                blo = __halves2half2(z, __double2half(x2));
            }
        }
        const uint32_t off = ((((k >> 3) ^ (r & 7u)) << 4) | ((k & 7u) << 1));  // swizzled 16-byte chunk, pair inside it
        *reinterpret_cast<__half2 *>(HA + base + off) = ahi;
        if (!compact) *reinterpret_cast<__half2 *>(HB + base + off) = bhi;  // compact: B is derived from the gathered A image
        if (two) {
            *reinterpret_cast<__half2 *>(HA + base + SLICE_BYTES + off) = alo;
            *reinterpret_cast<__half2 *>(HB + base + SLICE_BYTES + off) = blo;
        }
    }
}

// ---- projected operands (DESIGN.md "K2-TC", projection) -------------------------------------------
// Rows of the orthonormalised basis P^ (FP64, zero beyond K), passed by value: every thread reads them as uniform operands.
struct Basis {
    double p[PROJ_R][KMAX];
};

// Second moments about the centre m of the same <= CENTRE_SAMPLE rows k_tc_centre_median reads: one block per entry
// (i <= j), every thread a fixed stride of the sample, a fixed-order tree in shared memory; no atomics, so every GPU
// derives the same bits from the same rows. Entries that are not finite, or whose product is not, are skipped.
__global__ void __launch_bounds__(256) k_tc_cov(const double *__restrict__ S, uint64_t r0, uint64_t r1, uint32_t K,
                                                const double *__restrict__ centre, double *__restrict__ cov)
{
    __shared__ double red[256];
    uint32_t b = blockIdx.x, i = 0;
    while (b >= K - i) { b -= K - i; i++; }
    const uint32_t j = i + b;
    const uint64_t n = r1 - r0;
    const uint64_t ns = n < CENTRE_SAMPLE ? n : CENTRE_SAMPLE;
    double acc = 0.0;
    for (uint64_t t = threadIdx.x; t < ns; t += blockDim.x) {
        const uint64_t row = r0 + t * (n / ns);
        const double p = __dmul_rn(__dsub_rn(S[row * K + i], centre[i]), __dsub_rn(S[row * K + j], centre[j]));
        if (isfinite(p)) acc = __dadd_rn(acc, p);
    }
    red[threadIdx.x] = acc;
    __syncthreads();
    for (uint32_t h = blockDim.x / 2; h > 0; h >>= 1) {
        if (threadIdx.x < h) red[threadIdx.x] = __dadd_rn(red[threadIdx.x], red[threadIdx.x + h]);
        __syncthreads();
    }
    if (threadIdx.x == 0) { cov[i * K + j] = red[0]; cov[j * K + i] = red[0]; }
}

// y = P^ a', rho = |a' - P^T y| (computed directly: |a'|^2 - |y|^2 cancels when the row lies in the span), FP64, fixed order.
// a' has K <= KMAX entries, zero beyond.
__device__ __forceinline__ void proj_row(const Basis &B, const double (&x)[KMAX], double (&y)[PROJ_R], double &rho)
{
#pragma unroll
    for (uint32_t k = 0; k < PROJ_R; k++) {
        double t = 0.0;
#pragma unroll
        for (uint32_t c = 0; c < KMAX; c++) t = fma(B.p[k][c], x[c], t);
        y[k] = t;
    }
    double r2 = 0.0;
#pragma unroll
    for (uint32_t c = 0; c < KMAX; c++) {
        double r = x[c];
#pragma unroll
        for (uint32_t k = 0; k < PROJ_R; k++) r = fma(-B.p[k][c], y[k], r);
        r2 = fma(r, r, r2);
    }
    rho = sqrt(r2);
}

// One thread per row (operand position): the 16-column fp16 image, A [y0 .. y10 rho | x0 x1 P Q] and B [y .. rho | P Q x0 x1],
// both K-major SWIZZLE_32B. The scale is the centred rows' scale s (k_tc_fix_scale) divided by 8: |y_k|, rho <= |a'| (1 + delta)
// <= sqrt(60) max_k |a'_k|, so the magnitudes k_tc_prep keeps below 2^12 stay below it here. The fold column carries
//   h = (|z|^2 (1 - c) - cproj |a'|^2 - T0 (1/2 + 2c) - e0) / 2,   z = (y, rho) scaled, |a'|^2 scaled (NRM s^2),
// T0 passed with the projection's relative term already in it (tc_prepare). One slice: no lo halves.
__global__ void __launch_bounds__(128) k_tc_prep_proj(const double *__restrict__ S, uint64_t n, uint64_t r0, uint64_t r1, uint32_t K,
                                                      const Basis B, const double *__restrict__ NRM,
                                                      unsigned long long *__restrict__ misc, double T0, double cguard, double cproj,
                                                      const double *__restrict__ centre, unsigned char *__restrict__ HA,
                                                      unsigned char *__restrict__ HB)
{
    const uint64_t row = r0 + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= r1) return;
    const double s = __longlong_as_double((long long)misc[1]) * 0.125;
    const bool real = row < n;
    const bool wild = real && !isfinite(NRM[row]);
    const bool data = real && !wild;
    double y[PROJ_R], rho = 0.0;
#pragma unroll
    for (uint32_t k = 0; k < PROJ_R; k++) y[k] = 0.0;
    bool too_big = false;
    double nz = 0.0;
    if (data) {
        double x[KMAX];
#pragma unroll
        for (uint32_t c = 0; c < KMAX; c++) x[c] = c < K ? __dsub_rn(S[row * K + c], centre[c]) : 0.0;
        proj_row(B, x, y, rho);
#pragma unroll
        for (uint32_t k = 0; k < PROJ_R; k++) {
            y[k] *= s;
            too_big |= !(fabs(y[k]) < 4096.0);
            nz = fma(y[k], y[k], nz);
        }
        rho *= s;
        too_big |= !(rho < 4096.0);
        nz = fma(rho, rho, nz);
        if (too_big) {
            atomicAdd(misc + 2, 1ull);
            nz = 0.0;
        }
    }
    const double P = 32768.0, Q = 8.0;
    const double T0s = (T0 * s) * s;
    const double e0 = (double)K * 0.0078125;
    const double nfull = data ? (NRM[row] * s) * s : 0.0;
    const double h = 0.5 * (nz * (1.0 - cguard) - cproj * nfull - T0s * (0.5 + 2.0 * cguard) - e0);
    double x0, x1;
    if (!real) { x0 = -65504.0; x1 = 0.0; }                                           // padding row: never a survivor
    else if (wild || too_big || !(-h <= 32768.0 * P)) { x0 = 65504.0; x1 = 0.0; }     // always a survivor
    else {
        x0 = h16z(-h / P);
        x1 = h16z((-h - P * x0) / Q);
    }
    __align__(16) __half va[16], vb[16];
#pragma unroll
    for (uint32_t k = 0; k < PROJ_R; k++) va[k] = vb[k] = __double2half(too_big ? 0.0 : h16z(y[k]));
    va[PROJ_R] = vb[PROJ_R] = __double2half(too_big ? 0.0 : h16z(rho));
    va[12] = __double2half(x0); va[13] = __double2half(x1); va[14] = __double2half(P); va[15] = __double2half(Q);
    vb[12] = __double2half(P); vb[13] = __double2half(Q); vb[14] = __double2half(x0); vb[15] = __double2half(x1);
    const uint32_t r = (uint32_t)(row % ROWS), sw = (r >> 2) & 1u;
    const uint64_t base = (row / ROWS) * NBLOCK_BYTES + (uint64_t)r * NROW_BYTES;
    const uint4 *pa = reinterpret_cast<const uint4 *>(va), *pb = reinterpret_cast<const uint4 *>(vb);
#pragma unroll
    for (uint32_t c = 0; c < 2; c++) {
        *reinterpret_cast<uint4 *>(HA + base + 16 * (c ^ sw)) = pa[c];
        *reinterpret_cast<uint4 *>(HB + base + 16 * (c ^ sw)) = pb[c];
    }
}

// ---- survivor-density estimate ---------------------------------------------------------------------
// PLAN_SAMPLE pseudo-random pairs, one warp each, in FP64: would the pair survive the one-slice filter, the two-slice
// filter — each with centred and with raw operand copies — the FP64 DMMA filter and (proj != 0) the projected filter?
// plan[0..5] receive the six counts, plan[6] one per launch; the host turns them into survivor estimates and picks the variant BEFORE the first launch (tc_choose),
// instead of finding out by overflowing the queue.
// Criterion (DESIGN.md "K2-TC"): acc >= 0  <=>  d^2 <= c (|a'|^2 + |b'|^2) + T0 (1 + 4c) + 2 e0 / s^2, a' = a - m.
constexpr uint32_t PLAN_SAMPLE = 8192;
__device__ __forceinline__ uint64_t plan_mix(uint64_t z)
{
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}
__global__ void __launch_bounds__(256) k_tc_plan_sample(const double *__restrict__ S, const double *__restrict__ NRM, uint64_t r0,
                                                        uint64_t n, uint32_t K, double T0, unsigned long long *__restrict__ misc,
                                                        const double *__restrict__ basis, const double *__restrict__ centre, double T0p,
                                                        double cproj)
{
    const uint32_t t = blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (t >= PLAN_SAMPLE) return;
    if (t == 0 && lane == 0) atomicAdd(misc + PLAN_WORD + 6, 1ull);   // plan[6]: samples taken (a sharded prepare sums the shards')
    // pairs among the n rows starting at r0
    const uint64_t i = r0 + plan_mix(0x5ce3a0000ull + 2 * t) % n, j = r0 + plan_mix(0x5ce3a0001ull + 2 * t) % n;
    if (i == j) return;
    double d2 = 0.0, ua = 0.0, ub = 0.0;
    for (uint32_t k = lane; k < K; k += 32) {
        const double a = S[i * K + k], b = S[j * K + k];
        const double d = a - b;
        d2 = fma(d, d, d2);
        ua = fma(a, a, ua);
        ub = fma(b, b, ub);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        d2 += __shfl_xor_sync(0xffffffffu, d2, o);
        ua += __shfl_xor_sync(0xffffffffu, ua, o);
        ub += __shfl_xor_sync(0xffffffffu, ub, o);
    }
    // projected criterion of k_tc_prep_proj: the warp computes z = (P^ a', |a' - P^T P^ a'|) of both rows
    // (basis: PROJ_R x KMAX in global memory, nullptr = no projected count)
    double dz = 0.0, nz = 0.0;
    const bool proj = basis != nullptr;
    auto BP = [&](uint32_t k, uint32_t c) { return basis[k * KMAX + c]; };
    if (proj) {
        double ya[PROJ_R], yb[PROJ_R];
#pragma unroll
        for (uint32_t k = 0; k < PROJ_R; k++) {
            double ta = 0.0, tb = 0.0;
            for (uint32_t c = lane; c < K; c += 32) {
                ta = fma(BP(k, c), S[i * K + c] - centre[c], ta);
                tb = fma(BP(k, c), S[j * K + c] - centre[c], tb);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                ta += __shfl_xor_sync(0xffffffffu, ta, o);
                tb += __shfl_xor_sync(0xffffffffu, tb, o);
            }
            ya[k] = ta;
            yb[k] = tb;
        }
        double ra = 0.0, rb = 0.0;
        for (uint32_t c = lane; c < K; c += 32) {
            double xa = S[i * K + c] - centre[c], xb = S[j * K + c] - centre[c];
#pragma unroll
            for (uint32_t k = 0; k < PROJ_R; k++) { xa = fma(-BP(k, c), ya[k], xa); xb = fma(-BP(k, c), yb[k], xb); }
            ra = fma(xa, xa, ra);
            rb = fma(xb, xb, rb);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            ra += __shfl_xor_sync(0xffffffffu, ra, o);
            rb += __shfl_xor_sync(0xffffffffu, rb, o);
        }
        ra = sqrt(ra);
        rb = sqrt(rb);
#pragma unroll
        for (uint32_t k = 0; k < PROJ_R; k++) {
            dz = fma(ya[k] - yb[k], ya[k] - yb[k], dz);
            nz = fma(ya[k], ya[k], fma(yb[k], yb[k], nz));
        }
        dz = fma(ra - rb, ra - rb, dz);
        nz = fma(ra, ra, fma(rb, rb, nz));
    }
    if (lane != 0) return;
    const double s = __longlong_as_double((long long)misc[1]);
    const double nn = NRM[i] + NRM[j];            // centred squared norms (raw ones: ua + ub)
    const double e0 = 2.0 * (double)K * 0.0078125 / (s * s);
    const double c1 = 0.001953125, c2 = 0.0001220703125;
    unsigned long long *plan = misc + PLAN_WORD;
    // anything non-finite survives every filter
    if (!(d2 > c1 * nn + T0 * (1.0 + 4.0 * c1) + e0)) atomicAdd(plan + 0, 1ull);
    if (!(d2 > c2 * nn + T0 * (1.0 + 4.0 * c2) + e0)) atomicAdd(plan + 1, 1ull);
    if (!(d2 > c1 * (ua + ub) + T0 * (1.0 + 4.0 * c1) + e0)) atomicAdd(plan + 2, 1ull);
    if (!(d2 > c2 * (ua + ub) + T0 * (1.0 + 4.0 * c2) + e0)) atomicAdd(plan + 3, 1ull);
    if (!(d2 > T0 + (4.0 * K + 64.0) * 1.1102230246251565e-16 * 4.0 * (ua + ub))) atomicAdd(plan + 4, 1ull);
    if (proj && !(dz > c1 * nz + cproj * nn + T0p * (1.0 + 4.0 * c1) + 64.0 * e0)) atomicAdd(plan + 5, 1ull);  // scale s / 8
}

// ---- norm-band mode -------------------------------------------------------------------------------
__global__ void k_tc_iota(uint32_t *v, uint64_t n)
{
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v[i] = (uint32_t)i;
}

// One block. snrm2: squared norms in ascending order (non-finite ones last). For every row tile I (rows_per_tile rows)
// the first column tile (256 rows) that no pair of the two can share an edge with: all its norms exceed the
// row tile's largest norm by more than the threshold plus the rounding of the norms themselves. Then the
// exclusive scan of the strips per row tile. misc[3] receives the number of tiles in the band.
__global__ void __launch_bounds__(1024) k_tc_band_plan(const double *__restrict__ snrm2, uint64_t n, uint32_t rows_per_tile,
                                                       uint32_t n_row_tiles, uint32_t n_col_tiles, double thr, double keps,
                                                       uint32_t S, uint32_t *__restrict__ jend, uint32_t *__restrict__ item_start,
                                                       unsigned long long *__restrict__ misc)
{
    __shared__ unsigned long long s_sum[1024];
    const uint32_t rpc = 256 / rows_per_tile;
    unsigned long long tiles = 0;
    for (uint32_t I = threadIdx.x; I < n_row_tiles; I += blockDim.x) {
        const uint64_t last = min((uint64_t)(I + 1) * rows_per_tile, n) - 1;
        const double hi2 = snrm2[last];
        uint32_t je = n_col_tiles;
        if (isfinite(hi2)) {
            const double hi = sqrt(hi2);
            // smallest J > I / rpc whose first (= smallest) norm is out of reach; norms ascend, so bisect
            uint32_t lo_j = I / rpc, hi_j = n_col_tiles;  // tile lo_j is always in the band
            while (hi_j - lo_j > 1) {
                const uint32_t mid = (lo_j + hi_j) >> 1;
                const double l2 = snrm2[(uint64_t)mid * 256];
                const double l = sqrt(l2);
                const bool out = isfinite(l2) && (l - hi > thr * (1.0 + 4.0 * keps) + 4.0 * keps * l + 1e-150);
                if (out) hi_j = mid; else lo_j = mid;
            }
            je = hi_j;
        }
        jend[I] = je;
        tiles += je - I / rpc;
    }
    // strips per row tile -> exclusive prefix: every thread scans a contiguous run of row tiles, thread 0 the 1024 run sums
    __shared__ unsigned int s_items[1024];
    const uint32_t per = (n_row_tiles + blockDim.x - 1) / blockDim.x;
    const uint32_t i0 = min(threadIdx.x * per, n_row_tiles), i1 = min(i0 + per, n_row_tiles);
    __syncthreads();  // jend[] of the whole block is visible
    unsigned int run = 0;
    for (uint32_t I = i0; I < i1; I++) run += (jend[I] - I / rpc + S - 1) / S;
    s_items[threadIdx.x] = run;
    s_sum[threadIdx.x] = tiles;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t = 0;
        unsigned int acc = 0;
        for (uint32_t q = 0; q < blockDim.x; q++) {
            t += s_sum[q];
            const unsigned int r = s_items[q];
            s_items[q] = acc;
            acc += r;
        }
        misc[3] = t;
        item_start[n_row_tiles] = acc;
    }
    __syncthreads();
    unsigned int acc = s_items[threadIdx.x];
    for (uint32_t I = i0; I < i1; I++) {
        item_start[I] = acc;
        acc += (jend[I] - I / rpc + S - 1) / S;
    }
}

}  // namespace tc

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
// 64-column chunks of a K-column row: the last one keeps 4 columns for the row term
static uint32_t tc_chunks(uint32_t K) { return (K + 4 + 63) / 64; }
// binades the scale gives up so that |row|^2 stays below 2^30 (the fold columns hold h / 2^15 in fp16)
static int tc_k_headroom(uint32_t K) { return K <= 64 ? 0 : K <= 256 ? 1 : 2; }
// up to 10 chunks (K <= 636): the one-slice A tile of a row block (160 KB) plus two B stages still fit one SM
bool tc_supported(const scema_ctx *ctx) { return ctx->K >= 1 && tc_chunks(ctx->K) <= 10; }
// more than one chunk: hi slices only (the two-slice A tile would not fit next to a B ring)
bool tc_two_slices_possible(const scema_ctx *ctx) { return tc_chunks(ctx->K) == 1; }
// the projected filter: rows of one chunk that are wider than its 16 columns
bool tc_proj_possible(uint32_t K) { return K >= 16 && K <= tc::KMAX; }
static constexpr double TC_CPROJ = 1.0 / 4294967296.0;       // 2^-32: FP64 rounding of y and rho, relative to |a'|^2
static constexpr double TC_DELTA_MAX = 1.0 / 4294967296.0;   // largest |P P^T - I|_F the bound accepts
static constexpr double TC_T0_PROJ = 1.0 + 1.0 / 1073741824.0; // T0 (1 + 2^-30) covers (1 + 2 delta) d^2 on an edge

// cyclic Jacobi on a symmetric m x m matrix H (row-major, destroyed): eigenvalues on its diagonal, eigenvectors the columns of W
static void jacobi_sym(uint32_t m, std::vector<double> &H, std::vector<double> &W)
{
    W.assign((size_t)m * m, 0.0);
    for (uint32_t i = 0; i < m; i++) W[i * m + i] = 1.0;
    for (int sweep = 0; sweep < 64; sweep++) {
        double off = 0.0, dia = 0.0;
        for (uint32_t p = 0; p < m; p++) {
            dia += H[p * m + p] * H[p * m + p];
            for (uint32_t q = p + 1; q < m; q++) off += H[p * m + q] * H[p * m + q];
        }
        if (!(off > 1e-32 * dia)) break;   // off-diagonal below 1e-16 of the diagonal: the order of the Ritz values is settled
        const double small = 1e-18 * std::sqrt(dia);
        for (uint32_t p = 0; p < m; p++)
            for (uint32_t q = p + 1; q < m; q++) {
                const double apq = H[p * m + q];
                if (!(std::fabs(apq) > small)) continue;
                const double theta = 0.5 * (H[q * m + q] - H[p * m + p]) / apq;
                double t = 1.0 / (std::fabs(theta) + std::sqrt(1.0 + theta * theta));
                if (theta < 0.0) t = -t;
                const double c = 1.0 / std::sqrt(1.0 + t * t), sn = t * c;
                for (uint32_t k = 0; k < m; k++) {
                    const double hkp = H[k * m + p], hkq = H[k * m + q];
                    H[k * m + p] = c * hkp - sn * hkq;
                    H[k * m + q] = sn * hkp + c * hkq;
                }
                for (uint32_t k = 0; k < m; k++) {
                    const double hpk = H[p * m + k], hqk = H[q * m + k];
                    H[p * m + k] = c * hpk - sn * hqk;
                    H[q * m + k] = sn * hpk + c * hqk;
                }
                H[p * m + q] = H[q * m + p] = 0.0;
                for (uint32_t k = 0; k < m; k++) {
                    const double wkp = W[k * m + p], wkq = W[k * m + q];
                    W[k * m + p] = c * wkp - sn * wkq;
                    W[k * m + q] = sn * wkp + c * wkq;
                }
            }
    }
}

// modified Gram-Schmidt on the m vectors of length K in V (vector j at V[j * K]); a vector with (almost) nothing left
// is replaced by the unit vector that keeps the most of itself against the ones before it
static void mgs(uint32_t m, uint32_t K, std::vector<double> &V)
{
    for (uint32_t j = 0; j < m; j++) {
        double *v = &V[(size_t)j * K];
        double before = 0.0;
        for (uint32_t c = 0; c < K; c++) before += v[c] * v[c];
        for (int attempt = 0;; attempt++) {
            for (uint32_t i = 0; i < j; i++) {
                const double *u = &V[(size_t)i * K];
                double r = 0.0;
                for (uint32_t c = 0; c < K; c++) r += u[c] * v[c];
                for (uint32_t c = 0; c < K; c++) v[c] -= r * u[c];
            }
            double nn = 0.0;
            for (uint32_t c = 0; c < K; c++) nn += v[c] * v[c];
            if (attempt == 0 && nn > 1e-24 * before && nn > 0.0) {
                const double f = 1.0 / std::sqrt(nn);
                for (uint32_t c = 0; c < K; c++) v[c] *= f;
                break;
            }
            if (attempt > 0) {
                const double f = 1.0 / std::sqrt(nn);
                for (uint32_t c = 0; c < K; c++) v[c] *= f;
                break;
            }
            // degenerate: the unit vector e_b with the largest component outside span(V[0 .. j))
            uint32_t best = 0;
            double bres = -1.0;
            for (uint32_t b = 0; b < K; b++) {
                double res = 1.0;
                for (uint32_t i = 0; i < j; i++) res -= V[(size_t)i * K + b] * V[(size_t)i * K + b];
                if (res > bres) { bres = res; best = b; }
            }
            for (uint32_t c = 0; c < K; c++) v[c] = c == best ? 1.0 : 0.0;
        }
    }
}

// Orthonormal basis (PROJ_R rows, basis[k * KMAX + c], zero beyond K) of the leading principal directions of the second
// moments C [K][K] of the centred sample: block subspace iteration on 16 vectors from a fixed pseudo-random start, then a
// Rayleigh-Ritz step (Jacobi on the 16 x 16 projection), Ritz vectors by descending Ritz value, each signed so that its
// largest-magnitude component (first such) is positive, orthonormalised twice by modified Gram-Schmidt. Fixed
// operation order and no threads: the same C gives the same bits on every host. *delta = |P P^T - I|_F. The filter's
// bound holds for any basis with a small delta (DESIGN.md "K2-TC"); how well it fits the data only decides how many
// pairs survive. False when C is not finite, K is outside [16, KMAX] or delta exceeds TC_DELTA_MAX.
bool tc_basis_from_moments(const double *C, uint32_t K, double *basis, double *delta)
{
    constexpr uint32_t M = 16, ITER = 3, R = tc::PROJ_R;
    *delta = INFINITY;
    if (!tc_proj_possible(K)) return false;
    for (uint32_t i = 0; i < K * K; i++)
        if (!std::isfinite(C[i])) return false;
    std::vector<double> Q((size_t)M * K), Z((size_t)M * K);
    uint64_t z = 0x9e3779b97f4a7c15ull;
    for (auto &q : Q) {
        z += 0x9e3779b97f4a7c15ull;
        uint64_t x = z;
        x = (x ^ (x >> 30)) * 0xbf58476d1ce4e5b9ull;
        x = (x ^ (x >> 27)) * 0x94d049bb133111ebull;
        x ^= x >> 31;
        q = (double)(x >> 11) * 0x1.0p-52 - 1.0;
    }
    mgs(M, K, Q);
    auto mul = [&](const std::vector<double> &in, std::vector<double> &out) {   // out_j = C in_j, column by column (C = C^T)
        for (uint32_t j = 0; j < M; j++) {
            double *o = &out[(size_t)j * K];
            for (uint32_t r = 0; r < K; r++) o[r] = 0.0;
            for (uint32_t c = 0; c < K; c++) {
                const double x = in[(size_t)j * K + c];
                for (uint32_t r = 0; r < K; r++) o[r] += C[c * K + r] * x;
            }
        }
    };
    for (uint32_t it = 0; it < ITER; it++) {
        mul(Q, Z);
        Q.swap(Z);
        mgs(M, K, Q);
    }
    mul(Q, Z);
    std::vector<double> H((size_t)M * M), W;
    for (uint32_t a = 0; a < M; a++)
        for (uint32_t b = a; b < M; b++) {
            double t = 0.0;
            for (uint32_t c = 0; c < K; c++) t += Q[(size_t)a * K + c] * Z[(size_t)b * K + c] + Q[(size_t)b * K + c] * Z[(size_t)a * K + c];
            H[a * M + b] = H[b * M + a] = 0.5 * t;
        }
    jacobi_sym(M, H, W);
    std::vector<uint32_t> ord(M);
    for (uint32_t i = 0; i < M; i++) ord[i] = i;
    std::stable_sort(ord.begin(), ord.end(), [&](uint32_t a, uint32_t b) { return H[a * M + a] > H[b * M + b]; });
    std::vector<double> U((size_t)R * K, 0.0);
    for (uint32_t k = 0; k < R; k++) {
        double *u = &U[(size_t)k * K];
        for (uint32_t j = 0; j < M; j++) {
            const double w = W[j * M + ord[k]];
            for (uint32_t c = 0; c < K; c++) u[c] += w * Q[(size_t)j * K + c];
        }
    }
    mgs(R, K, U);
    mgs(R, K, U);
    for (uint32_t k = 0; k < R; k++) {
        double *u = &U[(size_t)k * K];
        uint32_t big = 0;
        for (uint32_t c = 1; c < K; c++)
            if (std::fabs(u[c]) > std::fabs(u[big])) big = c;
        if (u[big] < 0.0)
            for (uint32_t c = 0; c < K; c++) u[c] = -u[c];
    }
    double f2 = 0.0;
    for (uint32_t a = 0; a < R; a++)
        for (uint32_t b = 0; b < R; b++) {
            double t = 0.0;
            for (uint32_t c = 0; c < K; c++) t += U[(size_t)a * K + c] * U[(size_t)b * K + c];
            t -= a == b ? 1.0 : 0.0;
            f2 += t * t;
        }
    *delta = std::sqrt(f2);
    for (uint32_t k = 0; k < R; k++)
        for (uint32_t c = 0; c < tc::KMAX; c++) basis[k * tc::KMAX + c] = c < K ? U[(size_t)k * K + c] : 0.0;
    return *delta <= TC_DELTA_MAX;
}

// Operand preparation in three steps so that the host-buffer pipeline can run it range by range:
//   tc_prepare_begin : buffers, threshold constants, guard band of the slice count
//   tc_stats_rows    : norms of rows [r0, r1) (and, if wanted, their largest magnitude into the scale input)
//   tc_fix_scale     : freeze the power-of-two scale (headroom = binades left for rows not seen yet)
//   tc_prep_rows     : fp16 operand copies of rows [r0, r1) (r1 may run into the padding)
int tc_prepare_begin(scema_ctx *ctx, double thr, uint32_t slices)
{
    const uint64_t n = ctx->n;
    const uint32_t K = ctx->K;
    const uint64_t n_pad = (n + tc::COLT - 1) / tc::COLT * tc::COLT;
    ctx->tc_valid = false;
    ctx->tc_compact = false;  // [hi | lo] blocks unless a sharded prepare (tc_shard_*) asks for the hi-only layout
    ctx->shard_phase = 0;     // any prepare ends a sharded one in progress
    ctx->tc_band = false;  // row order unless tc_prepare sorts by norm afterwards
    ctx->tc_proj = false;  // 64-column copies unless tc_prepare chooses the projection
    const uint32_t nc = tc_chunks(K);
    if (nc > 1 && slices != 1) return fail(ctx, SCEMA_ERR_INVALID, "tensor-core filter: rows wider than 60 columns run with one slice");
    SCEMA_CUDA(ctx, ctx->d_tc_a.reserve(n_pad * 256 * nc));
    SCEMA_CUDA(ctx, ctx->d_tc_b.reserve(n_pad * 256 * nc));
    SCEMA_CUDA(ctx, ctx->d_tc_nrm.reserve(n_pad * sizeof(double)));
    SCEMA_CUDA(ctx, ctx->d_tc_misc.reserve(tc::MISC_WORDS * sizeof(unsigned long long)));
    SCEMA_CUDA(ctx, cudaMemsetAsync(ctx->d_tc_misc.p, 0, tc::MISC_WORDS * sizeof(unsigned long long), ctx->stream));
    // centre vector [K]; all zero until tc_centre_rows has run
    SCEMA_CUDA(ctx, ctx->d_tc_centre.reserve((size_t)std::max<uint32_t>(K, 1) * sizeof(double)));
    SCEMA_CUDA(ctx, cudaMemsetAsync(ctx->d_tc_centre.p, 0, (size_t)std::max<uint32_t>(K, 1) * sizeof(double), ctx->stream));
    const double eps = 1.1102230246251565e-16;  // 2^-53
    // The operands are rescaled, so the reference's underflow must be budgeted explicitly: each squared
    // difference of compare_L2_norm may lose up to half a subnormal ulp, i.e. the reference's sum can sit
    // K 2^-1075 below d^2 (and thr * thr itself rounds there too).
    ctx->tc_T0 = thr * thr * (1.0 + (2.0 * K + 16.0) * eps) * (1.0 + 4.0 * eps) + (2.0 * K + 4.0) * 4.9406564584124654e-324;
    // Guard band (DESIGN.md "K2-TC"): relative to |a_i|^2 + |a_j|^2 the computed accumulator is off by at most
    //   two slices: 3.1 2^-22 (slicing) + 13 2^-18 (12 MMA steps, fp32 accumulate)          < 2^-14
    //   one slice : 2^-11 (dropping a_lo, b_lo) + (4 nc + 1) 2^-18 (4 steps per chunk, nc <= 10) + 2^-23 (two-slice fold)
    //               < 2^-10.6
    // and the band must be twice that. Centring (a' = fl(a - m), relative error 2^-53 per element) moves d^2 by at most
    // 2 d 2^-53 (|a'| + |b'|) <= 2^-53 d^2 + 2^-52 (|a'|^2 + |b'|^2): the first term sits in the slack of T0 (the
    // reference needs (K + 4) eps of its (2K + 16) eps), the second is 2^-39 of the band.
    ctx->tc_cguard = slices == 1 ? 0.001953125 : 0.0001220703125;  // 2^-9, 2^-13
    ctx->tc_thr = thr;
    ctx->tc_n = n;
    ctx->tc_K = K;
    ctx->tc_slices = slices;
    ctx->tc_for_version = ctx->spline_version;
    return SCEMA_OK;
}

// Centre of the filter copies from a sample of the rows [r0, r1) (SCEMA_TC_CENTRE=0 leaves it at zero).
int tc_centre_rows(scema_ctx *ctx, uint64_t r0, uint64_t r1)
{
    static const char *env = getenv("SCEMA_TC_CENTRE");
    if (r1 <= r0 || ctx->K == 0 || (env && atoi(env) == 0)) return SCEMA_OK;
    tc::k_tc_centre_median<<<ctx->K, 256, 0, ctx->stream>>>(ctx->d_spline, r0, r1, ctx->K, ctx->d_tc_centre.as<double>());
    ctx->launches++;
    SCEMA_CUDA(ctx, cudaGetLastError());
    return SCEMA_OK;
}

int tc_stats_rows(scema_ctx *ctx, uint64_t r0, uint64_t r1, bool into_scale)
{
    if (r1 <= r0) return SCEMA_OK;
    tc::k_tc_rowstats<<<(unsigned)((r1 - r0 + 7) / 8), 256, 0, ctx->stream>>>(
        ctx->d_spline, ctx->d_tc_centre.as<double>(), r0, r1, ctx->K, ctx->d_tc_nrm.as<double>(),
        into_scale ? ctx->d_tc_misc.as<unsigned long long>() : nullptr);
    ctx->launches++;
    if (into_scale) {
        const unsigned grid = (unsigned)std::min<uint64_t>((uint64_t)ctx->sm_count * 4, (r1 - r0 + 255) / 256);
        tc::k_tc_nrm_hist<<<grid, 256, 0, ctx->stream>>>(ctx->d_tc_nrm.as<double>(), r0, r1, ctx->d_tc_misc.as<unsigned long long>());
        ctx->launches++;
    }
    SCEMA_CUDA(ctx, cudaGetLastError());
    return SCEMA_OK;
}

int tc_fix_scale(scema_ctx *ctx, int headroom)
{
    tc::k_tc_fix_scale<<<1, 256, 0, ctx->stream>>>(ctx->d_tc_misc.as<unsigned long long>(), headroom + tc_k_headroom(ctx->K));
    ctx->launches++;
    SCEMA_CUDA(ctx, cudaGetLastError());
    return SCEMA_OK;
}

int tc_prep_rows(scema_ctx *ctx, uint64_t r0, uint64_t r1)
{
    if (r1 <= r0) return SCEMA_OK;
    if (ctx->tc_proj) {
        tc::Basis B;
        std::copy(ctx->tc_basis_h, ctx->tc_basis_h + tc::PROJ_R * tc::KMAX, &B.p[0][0]);
        tc::k_tc_prep_proj<<<(unsigned)((r1 - r0 + 127) / 128), 128, 0, ctx->stream>>>(
            ctx->d_spline, ctx->n, r0, r1, ctx->K, B, ctx->d_tc_nrm.as<double>(), ctx->d_tc_misc.as<unsigned long long>(),
            ctx->tc_T0 * TC_T0_PROJ, ctx->tc_cguard, TC_CPROJ, ctx->d_tc_centre.as<double>(), ctx->d_tc_a.as<unsigned char>(),
            ctx->d_tc_b.as<unsigned char>());
        ctx->launches++;
        SCEMA_CUDA(ctx, cudaGetLastError());
        return SCEMA_OK;
    }
    tc::k_tc_prep<<<(unsigned)((r1 - r0 + 7) / 8), 256, 0, ctx->stream>>>(
        ctx->d_spline, ctx->n, r0, r1, ctx->K, tc_chunks(ctx->K), ctx->tc_slices, ldexp(1.0, 12 - tc_k_headroom(ctx->K)),
        ctx->d_tc_nrm.as<double>(),
        ctx->d_tc_misc.as<unsigned long long>(), ctx->tc_T0, ctx->tc_cguard, ctx->tc_band ? ctx->d_tc_perm.as<uint32_t>() : nullptr,
        ctx->d_tc_centre.as<double>(), ctx->tc_compact ? 1u : 0u,
        (reinterpret_cast<uintptr_t>(ctx->d_spline) % 16 == 0 && ctx->K % 2 == 0) ? 1u : 0u,   // 16-byte loads of column pairs
        ctx->d_tc_a.as<unsigned char>(), ctx->d_tc_b.as<unsigned char>());
    ctx->launches++;
    SCEMA_CUDA(ctx, cudaGetLastError());
    return SCEMA_OK;
}

// Basis of the projected filter from the centred sample of rows [r0, r1) (the rows k_tc_centre_median read): second
// moments on the device (k_tc_cov), basis on the host (tc_basis_from_moments) while the device computes the row
// statistics that were enqueued behind the copy (`then`), basis back to the device for the survivor sample.
// *ok = false: no usable basis (the 64-column copies stay).
template <class F>
static int tc_basis_rows(scema_ctx *ctx, uint64_t r0, uint64_t r1, bool *ok, F then)
{
    const uint32_t K = ctx->K;
    *ok = false;
    SCEMA_CUDA(ctx, ctx->d_tc_cov.reserve((size_t)K * K * sizeof(double)));
    SCEMA_CUDA(ctx, ctx->d_tc_basis.reserve(sizeof(ctx->tc_basis_h)));
    if (!ctx->h_tc_cov) SCEMA_CUDA(ctx, cudaMallocHost(&ctx->h_tc_cov, 60 * 60 * sizeof(double)));
    tc::k_tc_cov<<<K * (K + 1) / 2, 256, 0, ctx->stream>>>(ctx->d_spline, r0, r1, K, ctx->d_tc_centre.as<double>(), ctx->d_tc_cov.as<double>());
    ctx->launches++;
    SCEMA_CUDA(ctx, cudaGetLastError());
    SCEMA_CUDA(ctx, cudaMemcpyAsync(ctx->h_tc_cov, ctx->d_tc_cov.p, (size_t)K * K * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    cudaEvent_t ev;
    SCEMA_CUDA(ctx, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    cudaError_t e = cudaEventRecord(ev, ctx->stream);
    int rc = e == cudaSuccess ? then() : SCEMA_OK;
    if (e == cudaSuccess) e = cudaEventSynchronize(ev);
    cudaEventDestroy(ev);
    if (e != cudaSuccess) return fail(ctx, SCEMA_ERR_CUDA, std::string("tc basis: ") + cudaGetErrorString(e));
    if (rc) return rc;
    double delta = 0.0;
    *ok = tc_basis_from_moments(ctx->h_tc_cov, K, ctx->tc_basis_h, &delta);
    if (*ok)
        SCEMA_CUDA(ctx, cudaMemcpyAsync(ctx->d_tc_basis.p, ctx->tc_basis_h, sizeof(ctx->tc_basis_h), cudaMemcpyHostToDevice, ctx->stream));
    return SCEMA_OK;
}

int tc_basis_range(scema_ctx *ctx, uint64_t r0, uint64_t r1, bool *ok)
{
    return tc_basis_rows(ctx, r0, r1, ok, [] { return SCEMA_OK; });
}

// Which filter should evaluate `pairs` pairs of rows of K columns, given how many of `sample` random pairs would survive
// the one-slice / two-slice tcgen05 filter with centred copies (counts[0], [1]), with raw copies (counts[2], [3]), the
// DMMA filter (counts[4]) and (proj_ok) the projected filter (counts[5])? Cost model in seconds on one B200 (measured rates, DESIGN.md section 6): filter time + exact
// recompute of the estimated survivors; a queue that would not fit `mem_budget` bytes rules an option out; raw copies
// must beat the centred ones by 20 % to be taken. Fewer than four hits in the sample are noise as far as SIZING a queue
// goes (one hit in 8192 stands for 6e7 survivors at 1M rows). Pure host logic (scema_tc_choose: CPU tests).
//   -> choice: 1 / 2 = tcgen05 with that many slices, 3 = the projected tcgen05 filter (centred), 0 = SCEMA_PAIRS_DMMA,
//      -1 = SCEMA_PAIRS_EXACT; centred: which copies; est_survivors: queue entries to expect for the choice.
void tc_choose(uint64_t pairs, uint32_t K, const uint64_t counts[6], uint64_t sample, uint64_t mem_budget, bool tc_ok, bool proj_ok,
               int *choice, int *centred, uint64_t *est_survivors)
{
    const uint32_t nc = tc_chunks(K);
    const double P = (double)pairs, kf = 60.0 / (double)std::max<uint32_t>(K, 1);
    const double R1 = RATE_TC1 / nc, R2 = RATE_TC2, RD = RATE_DMMA * kf, RE = RATE_EXACT * kf, RQ = RATE_QUEUE * kf;
    double best = P / RE;
    *choice = -1;
    *centred = 1;
    *est_survivors = 0;
    auto consider = [&](int ch, int cen, double rate, uint64_t count) {
        const double surv = (double)count / (double)sample * P;
        const double sized = count >= 4 ? surv : 0.0;
        if (sized * 8.0 > (double)mem_budget) return;
        const double t = (P / rate + surv / RQ) * (cen || ch == 0 ? 1.0 : 1.25);
        if (t < best) { best = t; *choice = ch; *centred = cen; *est_survivors = (uint64_t)sized; }
    };
    consider(0, 1, RD, counts[4]);
    if (tc_ok && nc == 1) consider(2, 0, R2, counts[3]);
    if (tc_ok) consider(1, 0, R1, counts[2]);
    if (tc_ok && nc == 1) consider(2, 1, R2, counts[1]);
    if (tc_ok) consider(1, 1, R1, counts[0]);
    if (tc_ok && proj_ok && nc == 1 && tc_proj_possible(K)) consider(3, 1, RATE_TCP, counts[5]);
}

// Builds (or reuses) the fp16 operand copies for the current spline matrix and threshold.
// slices: 1 or 2 pins the number of fp16 slices, 3 the projected filter (one slice of 16 columns; 1 slice where the rows
// do not allow it); 0 = decide from a sample of the pairs (k_tc_plan_sample, tc_choose):
// *choice then returns what was decided (1 / 2 slices, 3: projected, 0: the caller should take SCEMA_PAIRS_DMMA, -1: SCEMA_PAIRS_EXACT —
// no operand copies are built in those two cases) and *est_survivors the estimate behind it. `pairs` = pairs this
// context will evaluate (its shard). want_band: sort the rows by norm first (operand copies in sorted order,
// ctx->d_tc_perm maps a position back to its row) so that the launch can restrict itself to the band of tiles the
// triangle inequality cannot rule out; refused (dense order instead) when a row has a non-finite norm or the rows
// are wider than one chunk.
int tc_prepare(scema_ctx *ctx, double thr, uint32_t slices, bool want_band, uint64_t pairs, int *choice, uint64_t *est_survivors)
{
    const uint64_t n = ctx->n;
    const uint64_t n_pad = (n + tc::COLT - 1) / tc::COLT * tc::COLT;
    if (choice) *choice = (int)slices;
    if (est_survivors) *est_survivors = 0;
    if (ctx->tc_for_version == ctx->spline_version && ctx->tc_thr == thr && ctx->tc_n == n && ctx->tc_K == ctx->K &&
        (slices == 0 || (slices == 3 ? ctx->tc_proj : !ctx->tc_proj && ctx->tc_slices == slices)) && ctx->tc_valid &&
        ctx->tc_band_wanted == want_band) {
        if (choice) *choice = ctx->tc_proj ? 3 : (int)ctx->tc_slices;   // the same rows and threshold: the earlier decision stands
        return SCEMA_OK;
    }
    const bool two_ok = tc_two_slices_possible(ctx);
    // the projection needs rows of 16 .. 60 columns and row order (the norm-band mode sorts the 64-column copies)
    bool proj_ok = (slices == 0 || slices == 3) && !want_band && tc_proj_possible(ctx->K) && n >= 2;
    int rc = wait_rows(ctx);   // a full prepare reads every row
    if (rc) return rc;
    rc = tc_prepare_begin(ctx, thr, slices == 0 || slices == 3 ? 1 : slices);
    ctx->tc_band = false;
    ctx->tc_band_wanted = want_band;
    if (!rc) rc = tc_centre_rows(ctx, 0, n);
    auto stats = [&]() {
        int r = tc_stats_rows(ctx, 0, n, true);
        return r ? r : tc_fix_scale(ctx, 0);
    };
    if (!rc) rc = proj_ok ? tc_basis_rows(ctx, 0, n, &proj_ok, stats) : stats();
    if (rc) return rc;
    if (slices == 3) slices = 1;   // pinned projection: one slice, 16 columns (64 where the rows do not allow it)
    else if (slices != 0) proj_ok = false;
    unsigned long long misc[8] = {};
    bool have_misc = false;
    if (slices == 0 && n >= 2) {
        uint64_t counts[6];
        rc = tc_plan_rows(ctx, n, counts, proj_ok);
        if (rc) return rc;
        int ch = 1, centred = 1;
        uint64_t est = 0;
        tc_choose(pairs, ctx->K, counts, tc::PLAN_SAMPLE, (uint64_t)ctx->mem_budget, true, proj_ok, &ch, &centred, &est);
        if (ch == 2 && !two_ok) ch = 1;
        if (choice) *choice = ch;
        if (est_survivors) *est_survivors = est;
        if (ch <= 0) return SCEMA_OK;  // the caller takes the DMMA / the filter-free kernel
        proj_ok = ch == 3;
        slices = ch == 3 ? 1u : (uint32_t)ch;
        ctx->tc_slices = slices;
        ctx->tc_cguard = slices == 1 ? 0.001953125 : 0.0001220703125;
        if (!centred) {
            // the raw rows filter better than the centred ones (a centre far from most rows): statistics and scale again
            SCEMA_CUDA(ctx, cudaMemsetAsync(ctx->d_tc_centre.p, 0, (size_t)ctx->K * sizeof(double), ctx->stream));
            SCEMA_CUDA(ctx, cudaMemsetAsync(ctx->d_tc_misc.p, 0, tc::MISC_WORDS * sizeof(unsigned long long), ctx->stream));
            rc = tc_stats_rows(ctx, 0, n, true);
            if (!rc) rc = tc_fix_scale(ctx, 0);
            if (rc) return rc;
        }
    } else if (slices == 0) {
        slices = 1;
        proj_ok = false;
    }
    ctx->tc_proj = proj_ok;
    if (proj_ok && choice) *choice = 3;
    if (want_band && tc_chunks(ctx->K) == 1) {
        if (!have_misc) {
            SCEMA_CUDA(ctx, cudaMemcpyAsync(misc, ctx->d_tc_misc.p, sizeof(misc), cudaMemcpyDeviceToHost, ctx->stream));
            SCEMA_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        }
        if (misc[4] == 0) {
            // ascending squared norms (non-negative doubles order as unsigned integers) and the permutation
            SCEMA_CUDA(ctx, ctx->d_tc_perm.reserve(n_pad * sizeof(uint32_t)));
            SCEMA_CUDA(ctx, ctx->d_tc_iota.reserve(n_pad * sizeof(uint32_t)));
            SCEMA_CUDA(ctx, ctx->d_tc_snrm.reserve(n_pad * sizeof(double)));
            tc::k_tc_iota<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(ctx->d_tc_iota.as<uint32_t>(), n);
            size_t tmp = 0;
            SCEMA_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, tmp, ctx->d_tc_nrm.as<uint64_t>(), ctx->d_tc_snrm.as<uint64_t>(),
                                                            ctx->d_tc_iota.as<uint32_t>(), ctx->d_tc_perm.as<uint32_t>(), (int64_t)n, 0, 64,
                                                            ctx->stream));
            SCEMA_CUDA(ctx, ctx->d_sort_tmp.reserve(tmp));
            SCEMA_CUDA(ctx, cub::DeviceRadixSort::SortPairs(ctx->d_sort_tmp.p, tmp, ctx->d_tc_nrm.as<uint64_t>(),
                                                            ctx->d_tc_snrm.as<uint64_t>(), ctx->d_tc_iota.as<uint32_t>(),
                                                            ctx->d_tc_perm.as<uint32_t>(), (int64_t)n, 0, 64, ctx->stream));
            ctx->launches += 10;
            ctx->tc_band = true;
        }
    }
    rc = tc_prep_rows(ctx, 0, n_pad);
    if (rc) return rc;
    ctx->tc_valid = true;
    return SCEMA_OK;
}

// Survivor-density sample over the rows [0, r1) (all rows; host-buffer pipeline: the first range, after its statistics
// and scale). counts = pairs of tc::PLAN_SAMPLE that would survive one slice / two slices with centred copies, the same
// with raw copies, the DMMA filter, the projected filter (proj: with the basis tc_basis_rows left on the device; 0
// otherwise). One host synchronisation.
int tc_plan_rows(scema_ctx *ctx, uint64_t r1, uint64_t counts[6], bool proj)
{
    for (int i = 0; i < 6; i++) counts[i] = 0;
    if (r1 < 2) return SCEMA_OK;
    unsigned long long *d_plan = ctx->d_tc_misc.as<unsigned long long>() + tc::PLAN_WORD, plan[8];
    SCEMA_CUDA(ctx, cudaMemsetAsync(d_plan, 0, 8 * sizeof(unsigned long long), ctx->stream));
    tc::k_tc_plan_sample<<<tc::PLAN_SAMPLE / 8, 256, 0, ctx->stream>>>(
        ctx->d_spline, ctx->d_tc_nrm.as<double>(), 0, r1, ctx->K, ctx->tc_T0, ctx->d_tc_misc.as<unsigned long long>(),
        proj ? ctx->d_tc_basis.as<double>() : nullptr, ctx->d_tc_centre.as<double>(), ctx->tc_T0 * TC_T0_PROJ, TC_CPROJ);
    ctx->launches++;
    SCEMA_CUDA(ctx, cudaMemcpyAsync(plan, d_plan, sizeof(plan), cudaMemcpyDeviceToHost, ctx->stream));
    SCEMA_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < 6; i++) ctx->tc_plan_counts[i] = counts[i] = plan[i];
    return SCEMA_OK;
}
uint32_t tc_plan_sample_size() { return tc::PLAN_SAMPLE; }

// ------------------------------------------------------------------------------------------------
// Sharded prepare (one context per GPU, rows split between them): every GPU builds the operand copies of ITS OWN rows
// only and the GPUs all-gather the fp16 images (128 bytes per row and chunk instead of 8 K bytes of FP64 rows), so the
// filter can start while the FP64 rows — which only the exact recompute needs — are still travelling. Centre and scale
// must be the same everywhere:
//   tc_shard_begin   own rows [r0, r1): centre candidate (column medians of the own sample)       -> all-gather, take rank 0's
//   tc_shard_stats   with the agreed centre: norms, magnitude, exponent histogram, survivor sample -> all-gather the packets
//   tc_shard_finish  packets of all GPUs reduced (max / sums) -> same scale and same choice of filter on every GPU; if that is
//                    "one slice, centred copies": hi-only A image of the own rows, in place          -> all-gather the images
//   tc_shard_commit  B image derived from A (fold columns swapped), operand copies declared valid; the exact recompute of
//                    the following scema_compare waits for `rows_ready` (the event behind the FP64 all-gather)
// Any other choice (two slices, raw copies, DMMA, ...) is reported to the caller, which then takes the ordinary path.
// ------------------------------------------------------------------------------------------------
namespace tc {
__global__ void __launch_bounds__(256) k_tc_reduce_packets(const unsigned long long *__restrict__ packets, uint32_t G,
                                                           unsigned long long *__restrict__ misc)
{
    for (uint32_t w = blockIdx.x * blockDim.x + threadIdx.x; w < MISC_WORDS; w += gridDim.x * blockDim.x) {
        unsigned long long acc = 0;
        for (uint32_t g = 0; g < G; g++) {
            const unsigned long long v = packets[(uint64_t)g * MISC_WORDS + w];
            if (w == 0) acc = v > acc ? v : acc;   // largest magnitude: non-negative doubles order as integers
            else acc += v;
        }
        if (w == 1 || w == 2 || w == 3) acc = 0;    // scale (set by k_tc_fix_scale), rows beyond the scale, band tiles
        misc[w] = acc;
    }
}
// B image from the A image (hi slices, compact layout): same data columns, fold columns [x0 x1 P Q] -> [P Q x0 x1]
__global__ void __launch_bounds__(256) k_tc_derive_b(const uint4 *__restrict__ HA, uint4 *__restrict__ HB, uint64_t n_chunks16, uint32_t nc)
{
    const uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;   // 16-byte chunk index
    if (q >= n_chunks16) return;
    uint4 v = HA[q];
    // chunk q: row = (q / 8) % 128 of slice (q / 1024); stored position p = q % 8 holds logical chunk p ^ (row & 7)
    const uint32_t row = (uint32_t)((q >> 3) & 127u), logical = (uint32_t)(q & 7u) ^ (row & 7u);
    const uint32_t c = (uint32_t)((q >> 10) % nc);
    if (c == nc - 1 && logical == 7u) { const uint32_t t0 = v.z; v.z = v.w; v.w = t0; }  // halves 60,61 <-> 62,63
    HB[q] = v;
}
}  // namespace tc

int tc_shard_begin(scema_ctx *ctx, double thr, uint64_t r0, uint64_t r1, const double **centre_dev)
{
    if (!ctx->have_spline) return fail(ctx, SCEMA_ERR_STATE, "Spline is not up to date.");
    // a share is whole 128-row blocks of the image, the last one ending at n; an empty share (the ranks past the end of
    // a split into equal shares) may sit at any row: it builds nothing and takes no sample
    const bool aligned = r0 == r1 || (r0 % 128 == 0 && (r1 % 128 == 0 || r1 == ctx->n));
    if (!tc_supported(ctx) || r0 > r1 || r1 > ctx->n || !aligned) return fail(ctx, SCEMA_ERR_INVALID, "tc_shard_begin: bad row range or row width");
    int rc = tc_prepare_begin(ctx, thr, 1);
    if (rc) return rc;
    ctx->tc_band_wanted = false;
    ctx->tc_compact = true;
    ctx->shard_r0 = r0;
    ctx->shard_r1 = r1;
    rc = tc_centre_rows(ctx, r0, r1);
    if (rc) return rc;
    ctx->shard_phase = 1;
    if (centre_dev) *centre_dev = ctx->d_tc_centre.as<double>();
    return SCEMA_OK;
}

int tc_shard_stats(scema_ctx *ctx, const double *centre_dev, const unsigned long long **packet_dev, uint64_t *packet_words)
{
    if (ctx->shard_phase != 1) return fail(ctx, SCEMA_ERR_STATE, "tc_shard_stats: call scema_tc_shard_begin first");
    if (centre_dev && centre_dev != ctx->d_tc_centre.as<double>())
        SCEMA_CUDA(ctx, cudaMemcpyAsync(ctx->d_tc_centre.p, centre_dev, (size_t)ctx->K * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    const uint64_t r0 = ctx->shard_r0, r1 = ctx->shard_r1;
    int rc = tc_stats_rows(ctx, r0, r1, true);
    if (!rc) rc = tc_fix_scale(ctx, 0);   // the local scale only feeds the (negligible) e0 term of the sample
    if (rc) return rc;
    if (r1 - r0 >= 2) {
        tc::k_tc_plan_sample<<<tc::PLAN_SAMPLE / 8, 256, 0, ctx->stream>>>(ctx->d_spline, ctx->d_tc_nrm.as<double>(), r0, r1 - r0, ctx->K,
                                                                         ctx->tc_T0, ctx->d_tc_misc.as<unsigned long long>(), nullptr,
                                                                         nullptr, 0.0, 0.0);
        ctx->launches++;
        SCEMA_CUDA(ctx, cudaGetLastError());
    }
    ctx->shard_phase = 2;
    if (packet_dev) *packet_dev = ctx->d_tc_misc.as<unsigned long long>();
    if (packet_words) *packet_words = tc::MISC_WORDS;
    return SCEMA_OK;
}

// optimistic != 0: do not wait for the sample (no host synchronisation in the middle of the step): the image is built on
// the assumption that the choice is again "one slice, centred copies"; tc_shard_check, called after the compare has
// synchronised anyway, says whether that was right (if not, the caller repeats the step on the ordinary path).
int tc_shard_finish(scema_ctx *ctx, const unsigned long long *packets_dev, uint32_t G, uint64_t pairs, int optimistic, int *choice,
                    const void **image_dev, uint64_t *image_bytes_per_row)
{
    if (ctx->shard_phase != 2) return fail(ctx, SCEMA_ERR_STATE, "tc_shard_finish: call scema_tc_shard_stats first");
    if (!packets_dev || G == 0 || !choice) return fail(ctx, SCEMA_ERR_INVALID, "tc_shard_finish: null pointer or no shards");
    unsigned long long *misc = ctx->d_tc_misc.as<unsigned long long>();
    if (!ctx->h_plan) SCEMA_CUDA(ctx, cudaMallocHost(&ctx->h_plan, 8 * sizeof(uint64_t)));
    tc::k_tc_reduce_packets<<<(tc::MISC_WORDS + 255) / 256, 256, 0, ctx->stream>>>(packets_dev, G, misc);
    ctx->launches++;
    SCEMA_CUDA(ctx, cudaMemcpyAsync(ctx->h_plan, misc + tc::PLAN_WORD, 8 * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    ctx->plan_pending = true;
    ctx->plan_pairs = pairs;
    uint64_t est = 0;
    if (!optimistic) {
        SCEMA_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        int rc0 = tc_shard_check(ctx, choice, &est);
        if (rc0) return rc0;
    } else {
        *choice = 1;
    }
    if (*choice != 1) { ctx->tc_compact = false; ctx->shard_phase = 0; return SCEMA_OK; }
    ctx->tc_slices = 1;
    ctx->tc_cguard = 0.001953125;
    ctx->cand_cap = std::max<uint64_t>(ctx->cand_cap, std::max<uint64_t>(std::max<uint64_t>(1ull << 20, 32 * ctx->n), est + est / 4));
    int rc = tc_fix_scale(ctx, 0);
    const uint64_t n_pad = (ctx->n + tc::COLT - 1) / tc::COLT * tc::COLT;
    // the share that ends at n also writes the padding rows up to n_pad; an empty share writes nothing
    if (!rc && ctx->shard_r1 > ctx->shard_r0) rc = tc_prep_rows(ctx, ctx->shard_r0, ctx->shard_r1 == ctx->n ? n_pad : ctx->shard_r1);
    if (rc) return rc;
    ctx->shard_phase = 3;
    if (image_dev) *image_dev = ctx->d_tc_a.p;
    if (image_bytes_per_row) *image_bytes_per_row = (uint64_t)tc_chunks(ctx->K) * 128;
    return SCEMA_OK;
}

// The choice the (by now arrived) sample of the last tc_shard_finish stands for: 1 = one slice with centred copies, anything
// else = the ordinary path should have been taken. Call after a host synchronisation of the context's stream.
int tc_shard_check(scema_ctx *ctx, int *choice, uint64_t *est_survivors)
{
    if (!ctx->plan_pending || !ctx->h_plan) return fail(ctx, SCEMA_ERR_STATE, "tc_shard_check: no sharded prepare to check");
    // the sharded prepare all-gathers 64-column images: the projected filter is never a candidate here
    uint64_t counts[6];
    for (int i = 0; i < 6; i++) ctx->tc_plan_counts[i] = counts[i] = i < 5 ? ctx->h_plan[i] : 0;
    ctx->plan_pending = false;
    // h_plan[6]: shares that took a sample (an empty or one-row share takes none and must not dilute the estimate)
    const uint64_t sampled = std::max<uint64_t>(ctx->h_plan[6], 1);
    int ch = 1, centred = 1;
    uint64_t est = 0;
    tc_choose(ctx->plan_pairs, ctx->K, counts, (uint64_t)tc::PLAN_SAMPLE * sampled, (uint64_t)ctx->mem_budget, true, false, &ch, &centred,
              &est);
    *choice = (ch == 1 && centred) ? 1 : (ch == 1 ? 3 : ch);   // 3: one slice but raw copies -> ordinary path
    if (est_survivors) *est_survivors = est;
    return SCEMA_OK;
}

int tc_shard_commit(scema_ctx *ctx, void *rows_ready_event)
{
    if (ctx->shard_phase != 3) return fail(ctx, SCEMA_ERR_STATE, "tc_shard_commit: no image of a sharded prepare to commit");
    ctx->shard_phase = 0;
    const uint64_t n_pad = (ctx->n + tc::COLT - 1) / tc::COLT * tc::COLT;
    const uint32_t nc = tc_chunks(ctx->K);
    const uint64_t chunks16 = n_pad * nc * 8;
    tc::k_tc_derive_b<<<(unsigned)((chunks16 + 255) / 256), 256, 0, ctx->stream>>>(ctx->d_tc_a.as<uint4>(), ctx->d_tc_b.as<uint4>(), chunks16, nc);
    ctx->launches++;
    SCEMA_CUDA(ctx, cudaGetLastError());
    ctx->rows_ready_event = rows_ready_event;
    ctx->tc_valid = true;
    return SCEMA_OK;
}

template <int CG, bool DBG, bool WIDE, bool BAND, bool NARROW = false>
static int tc_launch_t(scema_ctx *ctx, const tc::Args &a, uint64_t items)
{
    auto kern = tc::k_filter_tc<CG, DBG, WIDE, BAND, NARROW>;
    const size_t smem = (size_t)a.data_bytes + tc::Smem<CG>::tail;
    if (smem > ctx->smem_optin) return fail(ctx, SCEMA_ERR_CUDA, "tensor-core filter: shared memory exceeds device limit");
    SCEMA_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    uint64_t units = std::min<uint64_t>((uint64_t)ctx->sm_count / CG, std::max<uint64_t>(items, 1));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(units * CG));
    cfg.blockDim = dim3(384);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CG;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    SCEMA_CUDA(ctx, cudaLaunchKernelEx(&cfg, kern, a));
    ctx->launches++;
    return SCEMA_OK;
}

// Shared-memory plan of k_filter_tc (pure host logic, also reachable through scema_tc_plan for the CPU tests):
// A = all chunks of the row tile, double-buffered over items when that still leaves a deep B ring; B ring = a
// power-of-two number of stages of one chunk of a column tile; data_bytes = what is actually used (the rest of the
// SM stays L1). False when even one A buffer and two B stages do not fit 224 KB.
bool tc_smem_plan(uint32_t nc, uint32_t slices, uint32_t cg, uint32_t *a_bytes, uint32_t *n_abuf, uint32_t *lg_nst,
                  uint32_t *stage_bytes, uint32_t *data_bytes)
{
    const uint32_t b_rows = tc::COLT / cg;
    *stage_bytes = (slices == 1 ? 1u : 2u) * b_rows * 128u;
    *a_bytes = nc * (slices == 1 ? tc::SLICE_BYTES : tc::BLOCK_BYTES);
    const uint32_t data = 224u * 1024u;
    if (nc == 1) {
        // one chunk: two A buffers at a 32 KB stride, the B ring in what the 192 KB budget leaves (compile-time plan
        // of the WIDE = false kernel)
        *a_bytes = tc::BLOCK_BYTES;
        *n_abuf = 2;
        *lg_nst = slices == 1 ? (cg == 2 ? 3u : 2u) : (cg == 2 ? 2u : 1u);
    } else {
        auto lg_stages = [&](uint32_t nb) -> int {  // log2 of the B stages left next to nb A buffers, -1: does not fit
            if (nb * *a_bytes + 2u * *stage_bytes > data) return -1;
            const uint32_t room = (data - nb * *a_bytes) / *stage_bytes;
            return room >= 8 ? 3 : room >= 4 ? 2 : 1;
        };
        const int lg2 = lg_stages(2), lg1 = lg_stages(1);
        if (lg1 < 0) return false;
        // a deep B ring hides the TMA round trip on every tile, a second A buffer only the reload at item boundaries
        *n_abuf = (lg2 < 0 || (lg2 < 3 && lg1 > lg2)) ? 1u : 2u;
        *lg_nst = (uint32_t)(*n_abuf == 2 ? lg2 : lg1);
    }
    *data_bytes = *n_abuf * *a_bytes + (*stage_bytes << *lg_nst);
    return true;
}

uint32_t tc_chunks_for(uint32_t K) { return tc_chunks(K); }

// Filter the pairs of the row tiles [I0, I1) (256-row units) that belong to this shard; survivors go
// to the candidate queue (cand_count is d_counters[0]). dbg != nullptr selects the instrumented kernel.
int tc_launch(scema_ctx *ctx, uint32_t I0, uint32_t I1, uint32_t C0, uint32_t C1, uint32_t shard, uint32_t n_shards,
              unsigned long long *cand_count, float *dbg, uint64_t dbg_ld)
{
    tc::Args a;
    a.HA = ctx->d_tc_a.as<unsigned char>();
    a.HB = ctx->d_tc_b.as<unsigned char>();
    a.cand_count = cand_count;
    a.cand = ctx->d_cand.as<uint64_t>();
    a.cand_cap = ctx->cand_cap;
    a.n = ctx->n;
    a.NT = (uint32_t)((ctx->n + tc::COLT - 1) / tc::COLT);
    a.I0 = I0;
    a.I1 = std::min<uint32_t>(I1, a.NT);
    a.C0 = C0;
    a.C1 = std::min<uint32_t>(C1, a.NT);
    a.shard = shard;
    a.n_shards = n_shards;
    a.slices = ctx->tc_slices;
    a.dbg = dbg;
    a.dbg_ld = dbg_ld;
    a.nc = tc_chunks(ctx->K);
    a.compact = ctx->tc_compact ? 1u : 0u;
    a.band_item_start = a.band_jend = a.perm = nullptr;
    a.band_row_tiles = 0;
    static const char *cg_env = getenv("SCEMA_TC_CG");
    // cta_group::2 pairs (the default): each SM of a pair fetches half of every B tile, which halves the L2 -> SM traffic
    // and the shared-memory reads per SM. With the issue loops out of the way (round 2) the single-CTA kernel sits on
    // the L2 -> SM rate for wide rows (config-5 shape 14.6 vs 13.6 ms) and draws more power for the same work at
    // config 4 (37.0 vs 36.7 ms, both power-capped); SCEMA_TC_CG=1 selects it.
    const int cg = cg_env && atoi(cg_env) == 1 ? 1 : 2;
    // strips: long enough to amortise the A tile, short enough to leave every cluster many items
    const uint64_t rows = a.I1 > a.I0 ? a.I1 - a.I0 : 0;
    const uint64_t cols = a.C1 > a.C0 ? a.C1 - a.C0 : 0;
    const uint64_t tiles = rows * cols;  // upper bound
    const uint64_t units = (uint64_t)ctx->sm_count / cg;
    a.strip_len = (uint32_t)std::min<uint64_t>(32, std::max<uint64_t>(1, tiles / (units * 32 * std::max<uint32_t>(n_shards, 1))));
    if (rows == 0 || cols == 0) return SCEMA_OK;
    // items of this shard (upper bound is enough to size the grid)
    const uint64_t n_strips = (cols + a.strip_len - 1) / a.strip_len + 1;
    const uint64_t items = std::max<uint64_t>(1, rows * (2 / cg) * n_strips / std::max<uint32_t>(n_shards, 1));
    if (ctx->tc_proj) {
        // projected operands: 4 KB A buffers, a 16-deep ring of B stages (one column tile each: 4 KB per CTA of a pair)
        a.a_bytes = tc::NBLOCK_BYTES;
        a.n_abuf = 2;
        a.lg_nst = 4;
        a.stage_bytes = (tc::COLT / (uint32_t)cg) * tc::NROW_BYTES;
        a.data_bytes = a.n_abuf * a.a_bytes + (a.stage_bytes << a.lg_nst);
        if (cg == 1) return dbg ? tc_launch_t<1, true, false, false, true>(ctx, a, items) : tc_launch_t<1, false, false, false, true>(ctx, a, items);
        return dbg ? tc_launch_t<2, true, false, false, true>(ctx, a, items) : tc_launch_t<2, false, false, false, true>(ctx, a, items);
    }
    if (!tc_smem_plan(a.nc, a.slices, (uint32_t)cg, &a.a_bytes, &a.n_abuf, &a.lg_nst, &a.stage_bytes, &a.data_bytes))
        return fail(ctx, SCEMA_ERR_INVALID, "tensor-core filter: row tile does not fit shared memory");
    if (ctx->tc_band && !dbg && a.nc == 1) {
        // band plan for this kernel flavour: last column tile per row tile, strips per row tile, their prefix
        const uint32_t rpt = 128u * (uint32_t)cg;
        const uint64_t n_pad = (uint64_t)a.NT * tc::COLT;
        a.band_row_tiles = (uint32_t)(n_pad / rpt);
        a.strip_len = 8;
        SCEMA_CUDA(ctx, ctx->d_tc_band.reserve((2ull * a.band_row_tiles + 2) * sizeof(uint32_t)));
        uint32_t *jend = ctx->d_tc_band.as<uint32_t>(), *item_start = jend + a.band_row_tiles;
        const double keps = (ctx->K + 8.0) * 2.220446049250313e-16;
        tc::k_tc_band_plan<<<1, 1024, 0, ctx->stream>>>(ctx->d_tc_snrm.as<double>(), ctx->n, rpt, a.band_row_tiles, a.NT, ctx->tc_thr, keps,
                                                      a.strip_len, jend, item_start, ctx->d_tc_misc.as<unsigned long long>());
        ctx->launches++;
        a.band_item_start = item_start;
        a.band_jend = jend;
        a.perm = ctx->d_tc_perm.as<uint32_t>();
        a.I0 = 0; a.I1 = a.NT; a.C0 = 0; a.C1 = a.NT;
        return cg == 1 ? tc_launch_t<1, false, false, true>(ctx, a, ctx->sm_count) : tc_launch_t<2, false, false, true>(ctx, a, ctx->sm_count);
    }
    if (ctx->tc_band) return fail(ctx, SCEMA_ERR_STATE, "tensor-core filter: operands are in norm order, this launch needs row order");
    if (a.nc > 1) return cg == 1 ? tc_launch_t<1, false, true, false>(ctx, a, items) : tc_launch_t<2, false, true, false>(ctx, a, items);
    if (cg == 1) return dbg ? tc_launch_t<1, true, false, false>(ctx, a, items) : tc_launch_t<1, false, false, false>(ctx, a, items);
    return dbg ? tc_launch_t<2, true, false, false>(ctx, a, items) : tc_launch_t<2, false, false, false>(ctx, a, items);
}

// Debug / validation entry (scema_tc_debug): runs the instrumented kernel over the whole pair matrix
// and returns every accumulator (acc_host[row * ld + col], ld >= n_pad) and the operand copies, so a
// test can redo the sliced contraction in FP64 and check the layout, the fold columns and the
// accumulation-error model against the hardware. slices = 3: the projected filter (operand copies of
// n_pad x 32 bytes).
int tc_debug_run(scema_ctx *ctx, double thr, uint32_t slices, float *acc_host, uint64_t ld, unsigned char *ha_host,
                 unsigned char *hb_host)
{
    if (slices < 1 || slices > 3) return fail(ctx, SCEMA_ERR_INVALID, "tc_debug: slices must be 1, 2 or 3");
    if (!ctx->have_spline) return fail(ctx, SCEMA_ERR_STATE, "Spline is not up to date.");
    if (!tc_supported(ctx) || !tc_two_slices_possible(ctx)) return fail(ctx, SCEMA_ERR_INVALID, "tc_debug needs 1 <= K <= 60");
    if (slices == 3 && !tc_proj_possible(ctx->K)) return fail(ctx, SCEMA_ERR_INVALID, "tc_debug: the projected filter needs 16 <= K <= 60");
    const uint64_t n_pad = (ctx->n + tc::COLT - 1) / tc::COLT * tc::COLT;
    if (ld < n_pad) return fail(ctx, SCEMA_ERR_INVALID, "tc_debug: ld < padded n");
    if (n_pad > 8192) return fail(ctx, SCEMA_ERR_INVALID, "tc_debug: at most 8192 rows");
    int rc = tc_prepare(ctx, thr, slices, false, 0, nullptr, nullptr);
    if (rc) return rc;
    if (slices == 3 && !ctx->tc_proj) return fail(ctx, SCEMA_ERR_STATE, "tc_debug: no usable basis for the projected filter");
    const uint64_t img = n_pad * (ctx->tc_proj ? tc::NROW_BYTES : 256u);
    SCEMA_CUDA(ctx, ctx->d_counters.reserve(8 * sizeof(uint64_t)));
    SCEMA_CUDA(ctx, cudaMemsetAsync(ctx->d_counters.p, 0, 8 * sizeof(uint64_t), ctx->stream));
    if (ctx->cand_cap == 0) ctx->cand_cap = 1ull << 20;
    SCEMA_CUDA(ctx, ctx->d_cand.reserve(ctx->cand_cap * sizeof(uint64_t)));
    DevBuf dbg;
    SCEMA_CUDA(ctx, dbg.reserve(n_pad * n_pad * sizeof(float)));
    SCEMA_CUDA(ctx, cudaMemsetAsync(dbg.p, 0xFF, n_pad * n_pad * sizeof(float), ctx->stream));  // NaN = never written
    rc = tc_launch(ctx, 0, (uint32_t)(n_pad / tc::COLT), 0, (uint32_t)(n_pad / tc::COLT), 0, 1,
                   ctx->d_counters.as<unsigned long long>(), dbg.as<float>(), n_pad);
    if (rc) { dbg.release(); return rc; }
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e == cudaSuccess && acc_host)
        e = cudaMemcpy2D(acc_host, ld * sizeof(float), dbg.p, n_pad * sizeof(float), n_pad * sizeof(float), n_pad, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && ha_host) e = cudaMemcpy(ha_host, ctx->d_tc_a.p, img, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && hb_host) e = cudaMemcpy(hb_host, ctx->d_tc_b.p, img, cudaMemcpyDeviceToHost);
    dbg.release();
    if (e != cudaSuccess) return fail(ctx, SCEMA_ERR_CUDA, std::string("tc_debug: ") + cudaGetErrorString(e));
    return SCEMA_OK;
}

}  // namespace scema
