// Modulated 3x3 convolution as a shared-weight implicit GEMM on the 5th-gen tensor cores (sm_100a).
//   ModulatedConv2d.forward   scf/networks/stylegan2/model.py:237-278
//   StyledConv.forward        model.py:336-342   (noise + bias + leaky ReLU fused into the epilogue)
//
//   y[b,o,p] = d[b,o] * sum_{t,i} Ws[t,o,i] * xs[b,p+t,i],   xs = s[b,i]*x[b,i,p]  (pre-scaled by the producer)
//
// GEMM view: M = pixels (128 per tile), N = Cout (BN per tile), K = taps*Cin in BK-wide chunks (BK = 64, or 32 for
// layers with 32 input channels).
//   A tile  : per-tap kernel (modconv_tc_kernel): one TMA im2col load of 128 consecutive pixels of the flattened
//             (b, y, x) output grid per (tap, K chunk), shifted by the tap offset; the conv's zero padding is the
//             tensor map's out-of-bounds fill.  Halo kernels: one tiled TMA load of the halo of a spatial output tile
//             per K chunk, which all taps read through shifted operand descriptors.
//   B tile  : one TMA 3-D box {BK ch, BN (/2 per CTA of a pair), 1 tap} of the [tap][Cout][Cin] weight pack (shared by
//             all samples).
//   MMA     : tcgen05.mma kind::f16, M = 128 (single CTA) or 256 (CTA pair, cta_group::2), N = BN, K = 16, operands
//             straight from swizzled shared memory, fp32 accumulator in TMEM (double-buffered: 2 x BN columns).
//   Precision: 3-term bf16 split (hi*hi + hi*lo + lo*hi) into the same accumulator (SURVEY.md §7: single-pass
//             bf16/tf32 operands cannot meet the label criterion; the 3-term split gives ~1e-4 max abs error).
//   Epilogue: tcgen05.ld 32x32b -> x demod -> + noise -> + bias -> lrelu*sqrt2 -> fp32 NCHW capture + the next
//             conv's pre-scaled bf16 hi/lo NHWC planes (plain conv); or x demod -> fp32 NHWC scratch at the
//             phase position (transposed conv; blur + activation follow in blur_act_split_kernel).
//   The stride-2 transposed conv (model.py:251-259) is 4 output-phase sub-GEMMs with 4/2/2/1 taps (no wasted
//   FLOPs): out[2y'+py, 2x'+px] = sum_{ky = py (mod 2)...} W[ky,kx] x[y' - ky/2, x' - kx/2].
// Warp roles (320 threads, persistent, static round-robin tile schedule): warp 0 = TMA producer, warp 1 = MMA
// issuer + TMEM allocator, warps 2-9 = epilogue (TMEM lane quarter = warp_id % 4, two warps per quarter).
#include <cuda.h>
#include <cstring>
#include "common.cuh"
#include "kernels.h"
#include "modconv_tc.h"

namespace sis {

using bf16 = __nv_bfloat16;

// ------------------------------------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// One lane of a converged warp (PTX elect.sync).  A branch on this predicate is a pattern the compiler knows: inside it
// the single-thread tcgen05 / TMA instructions are issued once with warp-uniform operands, without a per-lane loop.
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(pred));
    return pred != 0;
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
// The producer / MMA loops of the warp-specialised kernels are executed by the WHOLE warp with warp-uniform control flow
// and operands; the single-thread instructions sit in `if (elect_one())` blocks, so their descriptors live in uniform
// registers and the UTCHMMA / UTMALDG instructions issue back to back.  (Wrapping the whole loop in `if (lane == 0)`
// makes every descriptor a per-thread value: the compiler then emits an ELECT + 5 x R2UR.BROADCAST + BRA.U.ANY
// "waterfall" around every UTCHMMA, ~95 clk per MMA whatever its shape -- measured: N = 64 layers at 32 % tensor-active,
// N = 32 at 17 %, N = 128 at 63 %.  A lane predicate inside the asm block (`pred`, kept for single call sites) still
// costs an ELECT loop per instruction: 42 % / 17 % / 78 %.)
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes, uint32_t pred = 1u) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\t@q mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n\t}"
                 ::"r"(smem_u32(bar)), "r"(bytes), "r"(pred) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred P1;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, P1;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug must never hang the GPU.  ~4e9 cycles (about 2 s) then record + trap.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, unsigned int* error, unsigned int code) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 4000000000ll) {
            if (error) *(volatile unsigned int*)error = code;      // mapped host word (watchdog_word): readable after the trap
            __threadfence_system();
            asm volatile("trap;");
        }
    }
}

__device__ __forceinline__ void tma_load_4d(const void* map, uint64_t* bar, void* dst, int c0, int c1, int c2, int c3, uint32_t pred = 1u) {
    asm volatile(
        "{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %7, 0;\n\t"
        "@q cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];\n\t}"
        ::"r"(smem_u32(dst)), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(pred) : "memory");
}
__device__ __forceinline__ void tma_load_3d(const void* map, uint64_t* bar, void* dst, int c0, int c1, int c2, uint32_t pred = 1u) {
    asm volatile(
        "{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %6, 0;\n\t"
        "@q cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];\n\t}"
        ::"r"(smem_u32(dst)), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(pred) : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const void* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)map) : "memory");
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate,
                                          uint32_t pred = 1u) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "setp.ne.b32 q, %5, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(pred) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar, uint32_t pred = 1u) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %1, 0;\n\t"
                 "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(smem_u32(bar)), "r"(pred) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major swizzled operand tile whose rows are ROW_BYTES (= swizzle width: 128 or 64) long: 8-row atoms of
// 8*ROW_BYTES (SBO), LBO unused (=1), descriptor version 1, layout type SWIZZLE_128B (2) / SWIZZLE_64B (4).
template <int ROW_BYTES>
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
    static_assert(ROW_BYTES == 128 || ROW_BYTES == 64, "swizzle width");
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)1 << 16;                             // leading byte offset (16 B units), ignored for swizzled K-major
    d |= (uint64_t)((8 * ROW_BYTES) >> 4) << 32;        // stride byte offset between 8-row groups
    d |= (uint64_t)1 << 46;                             // version = 1 (Blackwell)
    d |= (uint64_t)(ROW_BYTES == 128 ? 2 : 4) << 61;
    return d;
}

// ------------------------------------------------------------------------------------------------ kernel
// One sub-GEMM of a launch: the plain conv (one), the 4 output phases of a transposed conv, or its 4 border strips.
struct TcSubProblem {
    int ntaps;
    short dy[9], dx[9];         // tap offsets (may carry a sub-problem origin: border strips of the transposed conv)
    signed char widx[9];        // weight pack tap of every tap
    signed char phase[9];       // 4-phase halo kernels (transposed conv, Cout <= 64): output phase py*2+px of every tap
    int oh, ow;                 // extent of this sub-problem's output grid
    int ostride, ooff_y, ooff_x;   // output pixel = (y * ostride + ooff_y, x * ostride + ooff_x)
    int tiles_y, tiles_x;       // halo kernels: spatial output tiles of HALO_TH x HALO_TW
    int tile_begin;             // first tile of this sub-problem (sub-problems one after another, not interleaved)
    int base_dy, base_dx;       // per-tap kernel: smallest tap offset (the im2col traversal box starts there)
    int m_tiles;                // per-tap kernel: ceil(B*oh*ow / 128) im2col runs of 128 flattened pixels
};

// A-operand tensor maps: one (hi, lo) pair per sub-problem (the im2col maps of the 4 transposed-conv phases have
// different traversal boxes; the halo kernels use pair 0) and the weight pack maps.
struct TcMaps {
    CUtensorMap a[4][2];
    CUtensorMap w[2];
};

struct TcKernelArgs {
    TcSubProblem sub[4];
    int nsub, total_tiles;      // total_tiles counts tiles (single CTAs) or pair tiles (CTA pairs)
    int batch, cin, cout, b_tiles, kchunks;
    int mode;                   // 0 plain (fused noise + bias [+ activation]), 1 transposed-conv phase (demod only)
    int act;                    // mode 0: apply lrelu(0.2)*sqrt2 (StyledConv) or not (bare ModulatedConv2d)
    int interleave_units;       // > 0: the 4 transposed-conv phases are interleaved, each padded to this many (pair) tiles
    const float* demod; const float* noise; int64_t noise_bstride; float noise_w; const float* bias;
    float* out_f32; int out_h, out_w;
    const float* s_next; bf16* next_hi; bf16* next_lo;
    unsigned int* error;
};

constexpr int BM = 128, UMMA_K = 16;
constexpr int TC_EPI_WARPS = 8;                        // two per TMEM lane quarter
constexpr int TC_THREADS = 32 * (2 + TC_EPI_WARPS);   // warp 0: TMA, warp 1: MMA, warps 2..9: epilogue
// output tile of the halo kernels (16 x 8 pixels = one M = 128 tile; see modconv_tc_halo_kernel)
constexpr int HALO_TH = 16, HALO_TW = 8, HALO_W = HALO_TW + 2, HALO_H = HALO_TH + 2;

// BK = K elements per pipeline stage = one swizzle row (64 -> 128 B rows, 32 -> 64 B rows; measured: the 64 B rows
// are slower, the L2 -> SM path is request-bound).  CG = tcgen05 cta_group: with CG = 2 a CTA pair computes a
// 256 x BN tile: each CTA stages its own 128 pixel rows of A but only HALF of the weight tile (BN/2 rows), and the
// pair's MMA (M = 256, issued by the even CTA) reads B from both CTAs' shared memory.  That cuts the L2 -> SM bytes
// per MMA by a third (BN = 256: 96 -> 64 KB per K-step), which is what bounds the 1-CTA kernel (~40 B/clk/SM).
template <int BN, int BK, int CG> struct TcCfg {
    static constexpr int A_TILE_BYTES = BM * BK * 2;
    static constexpr int B_ROWS = BN / CG;                       // weight rows staged by this CTA
    static constexpr int B_TILE_BYTES = B_ROWS * BK * 2;
    static constexpr int STAGE_BYTES = 2 * A_TILE_BYTES + 2 * B_TILE_BYTES;
    static constexpr int STAGES = (216 * 1024) / STAGE_BYTES > 8 ? 8 : (216 * 1024) / STAGE_BYTES;
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/;
    static constexpr int TMEM_COLS = (2 * BN <= 32) ? 32 : (2 * BN <= 64) ? 64 : (2 * BN <= 128) ? 128 : (2 * BN <= 256) ? 256 : 512;
};

struct TileCoord { int sub, b0, y0, x0, n0; int p0; bool dummy; bool skip; };

// Tile t of this CTA.  CG = 1: t is a tile index.  CG = 2: t is a PAIR index and `rank` selects the m-tile of the pair
// (2*mp + rank); an odd m-tile count leaves rank 1 of the last pair with a dummy tile (it recomputes rank 0's tile and
// stores nothing).  HALO: m-tiles are HALO_TH x HALO_TW spatial tiles; otherwise im2col runs of 128 flattened pixels.
template <int BN, bool HALO, int CG>
__device__ __forceinline__ TileCoord decode_tile(const TcKernelArgs& a, int t, int rank) {
    TileCoord c;
    c.skip = false;
    int p = 0, local;
    if (!HALO && a.interleave_units) {
        // transposed conv, im2col mode: the 4 phase sub-GEMMs walk the image together (phase fastest, rotated so a
        // CTA's static stride does not lock onto one phase), so the input planes are read from DRAM once, not 4 times.
        // All phases are padded to the same number of units; the surplus tiles are skipped by every role alike.
        const int per_n = 4 * a.interleave_units;
        const int r = t % per_n, u = r >> 2;
        p = (u + (r & 3)) & 3;
        local = (t / per_n) * a.interleave_units + u;          // n * units + u; decoded below with m_units := interleave_units
    } else {
#pragma unroll
        for (int i = 1; i < 4; ++i)
            if (i < a.nsub && t >= a.sub[i].tile_begin) p = i;
        local = t - a.sub[p].tile_begin;
    }
    const TcSubProblem& s = a.sub[p];
    const int m_tiles = HALO ? a.b_tiles * s.tiles_y * s.tiles_x : s.m_tiles;
    const int m_units = (!HALO && a.interleave_units) ? a.interleave_units : (m_tiles + CG - 1) / CG;
    int m = (local % m_units) * CG + rank;
    const int n = local / m_units;
    if (!HALO && a.interleave_units && (local % m_units) * CG >= m_tiles) c.skip = true;
    c.dummy = m >= m_tiles;
    if (c.dummy) m = m_tiles - 1;
    c.sub = p;
    if (HALO) {
        c.p0 = 0;
        c.x0 = (m % s.tiles_x) * HALO_TW;
        c.y0 = ((m / s.tiles_x) % s.tiles_y) * HALO_TH;
        c.b0 = m / (s.tiles_x * s.tiles_y);
    } else {
        c.p0 = m * BM;                              // first flattened pixel of the run
        c.x0 = c.p0 % s.ow;
        c.y0 = (c.p0 / s.ow) % s.oh;
        c.b0 = c.p0 / (s.ow * s.oh);
    }
    c.n0 = n * BN;
    return c;
}

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// address of the same shared-memory location in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_to_cta(uint32_t saddr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    // default semantics (.release.cta), as CUTLASS' ClusterBarrier::arrive(cta_id): a cluster-scope release would make the
    // epilogue wait for its global stores to be acknowledged by L2 before every accumulator hand-back; the accumulator
    // reads themselves are ordered by tcgen05.wait::ld + tcgen05.fence::before_thread_sync
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;   // clears the CTA-pair bit of a shared::cluster address -> even CTA

template <int CG>
__device__ __forceinline__ void tma_load_4d_cg(const void* map, uint64_t* bar, void* dst, int c0, int c1, int c2, int c3, uint32_t pred = 1u) {
    if (CG == 1) {
        tma_load_4d(map, bar, dst, c0, c1, c2, c3, pred);
    } else {
        asm volatile(
            "{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %7, 0;\n\t"
            "@q cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];\n\t}"
            ::"r"(smem_u32(dst)), "l"((uint64_t)map), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(pred) : "memory");
    }
}
// TMA im2col mode: 128 consecutive pixels (W fastest, then H, then N) of the traversal box starting at the base pixel
// (c1, c2, c3), each shifted by the filter offset (off_w, off_h); pixels outside the tensor are zero-filled.
template <int CG>
__device__ __forceinline__ void tma_load_im2col_cg(const void* map, uint64_t* bar, void* dst, int c0, int c1, int c2, int c3,
                                                   unsigned short off_w, unsigned short off_h, uint32_t pred = 1u) {
    if (CG == 1) {
        asm volatile(
            "{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %9, 0;\n\t"
            "@q cp.async.bulk.tensor.4d.shared::cluster.global.im2col.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2], {%7, %8};\n\t}"
            ::"r"(smem_u32(dst)), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "h"(off_w), "h"(off_h), "r"(pred) : "memory");
    } else {
        asm volatile(
            "{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %9, 0;\n\t"
            "@q cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.im2col.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2], {%7, %8};\n\t}"
            ::"r"(smem_u32(dst)), "l"((uint64_t)map), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "h"(off_w), "h"(off_h), "r"(pred) : "memory");
    }
}
template <int CG>
__device__ __forceinline__ void tma_load_3d_cg(const void* map, uint64_t* bar, void* dst, int c0, int c1, int c2, uint32_t pred = 1u) {
    if (CG == 1) {
        tma_load_3d(map, bar, dst, c0, c1, c2, pred);
    } else {
        asm volatile(
            "{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %6, 0;\n\t"
            "@q cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];\n\t}"
            ::"r"(smem_u32(dst)), "l"((uint64_t)map), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1), "r"(c2), "r"(pred) : "memory");
    }
}
template <int CG>
__device__ __forceinline__ void umma_bf16_cg(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate,
                                             uint32_t pred = 1u) {
    if (CG == 1) {
        umma_bf16(tmem_d, adesc, bdesc, idesc, accumulate, pred);
    } else {
        asm volatile(
            "{\n\t.reg .pred p, q;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "setp.ne.b32 q, %5, 0;\n\t"
            "@q tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(pred) : "memory");
    }
}
// tcgen05.commit: arrive on `bar` when all previously issued MMAs retire; CG = 2 arrives on the barrier at the same
// offset in BOTH CTAs of the pair.
template <int CG>
__device__ __forceinline__ void umma_commit_cg(uint64_t* bar, uint32_t pred = 1u) {
    if (CG == 1) {
        umma_commit(bar, pred);
    } else {
        asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\t"
                     "@q tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n\t}"
                     ::"r"(smem_u32(bar)), "h"((uint16_t)3), "r"(pred) : "memory");
    }
}

// Epilogue warps (2..9): TMEM accumulator -> demodulate [-> noise + bias + lrelu] -> fp32 capture (+ the next conv's
// pre-scaled bf16 hi/lo planes), shared by the per-tap and the halo kernels.
// 32 consecutive per-channel constants (demodulation factors, bias, next style) as 8 x 128-bit loads when aligned
__device__ __forceinline__ void load32(const float* p, float (&o)[32]) {
    if ((reinterpret_cast<uintptr_t>(p) & 15) == 0) {
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const float4 v = __ldg(reinterpret_cast<const float4*>(p) + q);
            o[4 * q] = v.x; o[4 * q + 1] = v.y; o[4 * q + 2] = v.z; o[4 * q + 3] = v.w;
        }
    } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) o[j] = __ldg(p + j);
    }
}

// UP4: the accumulator holds the FOUR output phases of a transposed conv side by side (4 x BN columns; phase p of pixel
// (yy, xx) goes to scratch position (2yy + py, 2xx + px); the py = 1 / px = 1 phases are one row / column shorter).
template <int BN, bool HALO, int CG, bool UP4 = false>
__device__ __forceinline__ void tc_epilogue(const TcKernelArgs& a, uint64_t* tfull_bar, uint64_t* tempty_bar, uint32_t tmem_base,
                                            int rank, int warp, int lane, int unit0, int unit_stride) {
        // ============================== epilogue (warps 2..9) ==============================
        const int quarter = warp & 3;                   // TMEM lane quarter this warp may access
        const int chalf = (warp - 2) >> 2;              // the two warps of a quarter take alternate 32-column chunks
        const int row = quarter * 32 + lane;            // GEMM row = pixel of the tile
        const int tw = row % HALO_TW, th = row / HALO_TW;
        const uint32_t tempty_leader = (CG == 2) ? map_to_cta(smem_u32(&tempty_bar[0]), 0) : 0u;
        int acc = 0; uint32_t acc_phase = 0;
        for (int t = unit0; t < a.total_tiles; t += unit_stride) {
            const TileCoord c = decode_tile<BN, HALO, CG>(a, t, rank);
            if (c.skip) continue;
            const TcSubProblem& s = a.sub[c.sub];
            int b, yy, xx;
            if (HALO) {
                b = c.b0; yy = c.y0 + th; xx = c.x0 + tw;
            } else {
                const int p = c.p0 + row;
                xx = p % s.ow; yy = (p / s.ow) % s.oh; b = p / (s.ow * s.oh);
            }
            const bool valid0 = !c.dummy && b < a.batch && yy < s.oh && xx < s.ow;
            const int oy0 = yy * s.ostride + s.ooff_y, ox0 = xx * s.ostride + s.ooff_x;
            mbar_wait(&tfull_bar[acc], acc_phase, a.error, 0x400 + acc);
            tc_fence_after();
            constexpr int ACC_COLS = (UP4 ? 4 : 1) * BN;
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * ACC_COLS);
            const float* dm = a.demod + (int64_t)(valid0 ? b : 0) * a.cout + c.n0;
            float nz = 0.0f;
            if (!UP4 && a.mode == 0 && valid0 && a.noise) nz = __fmul_rn(a.noise_w, a.noise[(int64_t)b * a.noise_bstride + (int64_t)oy0 * a.out_w + ox0]);
#pragma unroll 1
            for (int k = chalf; k < ACC_COLS / 32; k += 2) {       // this warp's 32-column chunks
                const int call = k * 32;
                const int ph = UP4 ? call / BN : 0;
                const int c0 = UP4 ? call - ph * BN : call;
                const bool valid = UP4 ? (valid0 && yy < s.oh - (ph >> 1) && xx < s.ow - (ph & 1)) : valid0;
                const int oy = UP4 ? oy0 + (ph >> 1) : oy0, ox = UP4 ? ox0 + (ph & 1) : ox0;
                uint32_t r[32];
                tmem_ld_32x32(taddr + (uint32_t)call, r);
                tmem_ld_wait();
                if (valid) {
                    float v[32], cst[32];
                    load32(dm + c0, cst);
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = __fmul_rn(__uint_as_float(r[j]), cst[j]);
                    if (!UP4 && a.mode == 0) {
                        // NoiseInjection + FusedLeakyReLU (model.py:292, fused_bias_act_kernel.cu:26-47)
                        const int64_t plane = (int64_t)a.out_h * a.out_w;
                        float* dst = a.out_f32 + ((int64_t)b * a.cout + c.n0 + c0) * plane + (int64_t)oy * a.out_w + ox;
                        if (a.bias) load32(a.bias + c.n0 + c0, cst);
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            float x = __fadd_rn(v[j], nz);
                            if (a.bias) x = __fadd_rn(x, cst[j]);
                            if (a.act) x = lrelu_scale(x, 0.2f, 1.41421356237309504880f);
                            v[j] = x;
                            dst[(int64_t)j * plane] = x;       // lanes = consecutive x: coalesced per channel
                        }
                        if (a.s_next) {
                            load32(a.s_next + (int64_t)b * a.cout + c.n0 + c0, cst);
                            const float* sn = cst;
                            const int64_t off = (((int64_t)b * a.out_h + oy) * a.out_w + ox) * a.cout + c.n0 + c0;
                            uint4* ph_ = reinterpret_cast<uint4*>(a.next_hi + off);
                            uint4* pl = reinterpret_cast<uint4*>(a.next_lo + off);
#pragma unroll
                            for (int q = 0; q < 4; ++q) {
                                uint32_t wh[4], wl[4];
#pragma unroll
                                for (int e = 0; e < 4; ++e) {
                                    const int j = q * 8 + e * 2;
                                    const float x0 = __fmul_rn(v[j], sn[j]), x1 = __fmul_rn(v[j + 1], sn[j + 1]);
                                    const bf16 h0 = __float2bfloat16_rn(x0), h1 = __float2bfloat16_rn(x1);
                                    const bf16 l0 = __float2bfloat16_rn(x0 - __bfloat162float(h0));
                                    const bf16 l1 = __float2bfloat16_rn(x1 - __bfloat162float(h1));
                                    wh[e] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
                                    wl[e] = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
                                }
                                ph_[q] = make_uint4(wh[0], wh[1], wh[2], wh[3]);
                                pl[q] = make_uint4(wl[0], wl[1], wl[2], wl[3]);
                            }
                        }
                    } else {
                        // transposed-conv phase: demodulated fp32, NHWC scratch [B][out_h][out_w][cout]
                        float4* dst = reinterpret_cast<float4*>(
                            a.out_f32 + (((int64_t)b * a.out_h + oy) * a.out_w + ox) * a.cout + c.n0 + c0);
#pragma unroll
                        for (int q = 0; q < 8; ++q) dst[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if (CG == 1) mbar_arrive(&tempty_bar[acc]);
                else mbar_arrive_cluster(tempty_leader + (uint32_t)(acc * 8));   // the even CTA's MMA thread waits on it
            }
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    }

// Per-tap kernel: one im2col A tile per (tap, K chunk).
template <int BN, int BK, int CG>
__global__ void __launch_bounds__(TC_THREADS, 1)
modconv_tc_kernel(const __grid_constant__ TcMaps maps, const __grid_constant__ TcKernelArgs a) {
    static_assert(CG == 1 || CG == 2, "cta_group");
    using Cfg = TcCfg<BN, BK, CG>;
    constexpr int STAGES = Cfg::STAGES;
    constexpr int A_TILE_BYTES = Cfg::A_TILE_BYTES;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = (uint64_t*)(smem + STAGES * Cfg::STAGE_BYTES);
    uint64_t* full_bar = bars;                 // [STAGES]  (CG = 2: only the even CTA's are used)
    uint64_t* empty_bar = bars + STAGES;       // [STAGES]
    uint64_t* tfull_bar = bars + 2 * STAGES;   // [2]
    uint64_t* tempty_bar = bars + 2 * STAGES + 2;  // [2]       (CG = 2: only the even CTA's are used)
    uint32_t* tmem_ptr_smem = (uint32_t*)(bars + 2 * STAGES + 4);

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // provably warp-uniform
    const int rank = (CG == 2) ? (int)cluster_ctarank() : 0;
    const bool leader = rank == 0;
    const int unit0 = (CG == 2) ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;        // first tile (pair) of this CTA
    const int unit_stride = (CG == 2) ? (int)(gridDim.x >> 1) : (int)gridDim.x;

    if (warp == 0 && lane == 0) {
        for (int i = 0; i < a.nsub; ++i) { tma_prefetch_desc(&maps.a[i][0]); tma_prefetch_desc(&maps.a[i][1]); }
        tma_prefetch_desc(&maps.w[0]); tma_prefetch_desc(&maps.w[1]);
        for (int i = 0; i < STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], TC_EPI_WARPS * CG); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        if (CG == 1) {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        } else {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        }
    }
    tc_fence_before();
    if (CG == 2) cluster_sync_all(); else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;

    if (warp == 0) {
        // ============================== TMA producer (both CTAs of a pair; whole warp, lane 0 issues) ==============================
        {
            int stage = 0; uint32_t phase = 0;
            for (int t = unit0; t < a.total_tiles; t += unit_stride) {
                const TileCoord c = decode_tile<BN, false, CG>(a, t, rank);
                if (c.skip) continue;
                const TcSubProblem& s = a.sub[c.sub];
                const int wrow = c.n0 + rank * Cfg::B_ROWS;
                const CUtensorMap* ma_hi = &maps.a[c.sub][0];
                const CUtensorMap* ma_lo = &maps.a[c.sub][1];
                for (int tap = 0; tap < s.ntaps; ++tap) {
                    const int wi = s.widx[tap];
                    const unsigned short ow_ = (unsigned short)(s.dx[tap] - s.base_dx), oh_ = (unsigned short)(s.dy[tap] - s.base_dy);
                    for (int kc = 0; kc < a.kchunks; ++kc) {
                        mbar_wait(&empty_bar[stage], phase ^ 1, a.error, 0x100 + stage);
                        uint8_t* st = smem + stage * Cfg::STAGE_BYTES;
                        if (elect_one()) {
                            // one arming per stage: the even CTA expects the bytes of BOTH CTAs on its barrier
                            if (leader) mbar_expect_tx(&full_bar[stage], CG * Cfg::STAGE_BYTES);
                            tma_load_im2col_cg<CG>(ma_hi, &full_bar[stage], st, kc * BK, c.x0 + s.base_dx, c.y0 + s.base_dy, c.b0, ow_, oh_);
                            tma_load_im2col_cg<CG>(ma_lo, &full_bar[stage], st + A_TILE_BYTES, kc * BK, c.x0 + s.base_dx, c.y0 + s.base_dy, c.b0, ow_, oh_);
                            tma_load_3d_cg<CG>(&maps.w[0], &full_bar[stage], st + 2 * A_TILE_BYTES, kc * BK, wrow, wi);
                            tma_load_3d_cg<CG>(&maps.w[1], &full_bar[stage], st + 2 * A_TILE_BYTES + Cfg::B_TILE_BYTES, kc * BK, wrow, wi);
                        }
                        __syncwarp();
                        if (++stage == STAGES) { stage = 0; phase ^= 1; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ============================== MMA issuer (even CTA of a pair only; whole warp, lane 0 issues) ==============================
        if (leader) {
            // instruction descriptor: D=f32, A=B=bf16, both K-major, N=BN, M=128*CG
            constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)((BM * CG) >> 4) << 24);
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            for (int t = unit0; t < a.total_tiles; t += unit_stride) {
                const TileCoord c = decode_tile<BN, false, CG>(a, t, 0);
                if (c.skip) continue;
                const int kblocks = a.sub[c.sub].ntaps * a.kchunks;
                mbar_wait(&tempty_bar[acc], acc_phase ^ 1, a.error, 0x200 + acc);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
                for (int kb = 0; kb < kblocks; ++kb) {
                    mbar_wait(&full_bar[stage], phase, a.error, 0x300 + stage);
                    tc_fence_after();
                    const uint32_t sa = smem_u32(smem + stage * Cfg::STAGE_BYTES);
                    const uint64_t d_ah = make_smem_desc<BK * 2>(sa), d_al = make_smem_desc<BK * 2>(sa + A_TILE_BYTES);
                    const uint64_t d_bh = make_smem_desc<BK * 2>(sa + 2 * A_TILE_BYTES);
                    const uint64_t d_bl = make_smem_desc<BK * 2>(sa + 2 * A_TILE_BYTES + Cfg::B_TILE_BYTES);
                    if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < BK / UMMA_K; ++k) {
                            const uint64_t koff = (uint64_t)((k * UMMA_K * 2) >> 4);   // +32 B per K step inside the swizzle row
                            umma_bf16_cg<CG>(d_tmem, d_ah + koff, d_bh + koff, idesc, (kb | k) ? 1u : 0u);
                            umma_bf16_cg<CG>(d_tmem, d_ah + koff, d_bl + koff, idesc, 1u);
                            umma_bf16_cg<CG>(d_tmem, d_al + koff, d_bh + koff, idesc, 1u);
                        }
                        umma_commit_cg<CG>(&empty_bar[stage]);      // frees this smem stage (in both CTAs) when the MMAs retire
                        if (kb == kblocks - 1) umma_commit_cg<CG>(&tfull_bar[acc]);   // accumulator complete -> epilogue (both CTAs)
                    }
                    __syncwarp();
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        tc_epilogue<BN, false, CG>(a, tfull_bar, tempty_bar, tmem_base, rank, warp, lane, unit0, unit_stride);
    }
    tc_fence_before();
    if (CG == 2) cluster_sync_all(); else __syncthreads();   // CG = 2: the peer may still read this CTA's smem / TMEM
    if (warp == 1) {
        __syncwarp();
        tc_fence_after();
        if (CG == 1)
            asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
        else
            asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
    }
}

// ------------------------------------------------------------------------------- halo-reuse variant
// Plain 3x3 layers with H >= 16: instead of one A tile per (tap, K chunk), the producer loads ONE 18 x 10 pixel halo of
// the 16 x 8 output tile per K chunk and the 9 taps read it through shifted operand descriptors: tap (dy, dx) starts
// at halo pixel (dy+1)*10 + (dx+1) and its sixteen 8-pixel row groups are one halo row (10 pixels = 1280 B) apart.
// SWIZZLE_128B is a function of the absolute shared-memory address (bits 4-6 ^= bits 7-9), so any 128 B-aligned start
// inside a 1024 B-aligned TMA-written buffer reads back consistently with base_offset 0 (scripts/exp_halo_desc.cu
// verifies this on the B200).  A traffic drops from 9 x 32 KB to 45 KB per K chunk; the weights stream per tap through
// their own ring.  With Cout = 128 that takes the L2 -> SM fill from ~62 to ~27 B/clk/SM, i.e. back under the tensor pipe.
// BK = 64: 128 B operand rows (SWIZZLE_128B); BK = 32 (layers with 32 input channels): 64 B rows (SWIZZLE_64B), as the
// transposed halo kernel below uses them.
// UP4 (transposed conv with Cout <= 64): the 9 taps of a stride-2 transposed conv fall into 4 output phases with 4/2/2/1
// taps whose offsets are all in {-1, 0}: one halo per K chunk serves ALL FOUR phases of the spatial tile, each phase
// accumulating into its own BN columns of a 4 x BN accumulator (double-buffered: 8 x BN <= 512 TMEM columns).  The
// per-tap kernel re-fetches an A tile per (phase, tap, K chunk): with N <= 64 that is ~85 B/clk/SM of L2 -> SM fill for
// MMAs that need 40-48 clk each, i.e. fill-bound at about half the MMA rate.
template <int BN, int CG, int BK = 64, bool UP4 = false> struct TcHaloCfg {
    static constexpr int ROW = BK * 2;
    static constexpr int A_BYTES = HALO_H * HALO_W * ROW;                    // 23040 (BK 64): bytes one halo load delivers
    static constexpr int A_PAD = (A_BYTES + 1023) / 1024 * 1024;             // hi / lo planes stay 1024 B aligned
    static constexpr int A_STAGE = 2 * A_PAD;
    static constexpr int NA = 2;
    static constexpr int B_ROWS = BN / CG;
    static constexpr int B_TILE_BYTES = B_ROWS * ROW;
    static constexpr int B_STAGE = 2 * B_TILE_BYTES;
    static constexpr int BUDGET = 227 * 1024 - 1024 - 512;
    static constexpr int NB_RAW = (BUDGET - NA * A_STAGE) / B_STAGE;
    static constexpr int NB = NB_RAW > 8 ? 8 : NB_RAW;
    static constexpr int SMEM_BYTES = NA * A_STAGE + NB * B_STAGE + 1024 /*align*/ + 512 /*barriers*/;
    static constexpr int ACC_COLS = (UP4 ? 4 : 1) * BN;
    static constexpr int TMEM_COLS = (2 * ACC_COLS <= 32) ? 32 : (2 * ACC_COLS <= 64) ? 64 : (2 * ACC_COLS <= 128) ? 128 : (2 * ACC_COLS <= 256) ? 256 : 512;
    static_assert(NB >= 2, "weight ring too shallow");
    static_assert(2 * ACC_COLS <= 512, "accumulators exceed TMEM");
};

template <int ROW>
__device__ __forceinline__ uint64_t make_halo_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)((HALO_W * ROW) >> 4) << 32;         // 8-pixel row groups are one halo row apart
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)(ROW == 128 ? 2 : 4) << 61;          // SWIZZLE_128B / SWIZZLE_64B, base_offset 0
    return d;
}

template <int BN, int CG, int BK, bool UP4>
__global__ void __launch_bounds__(TC_THREADS, 1)
modconv_tc_halo_kernel(const __grid_constant__ TcMaps maps, const __grid_constant__ TcKernelArgs a) {
    using Cfg = TcHaloCfg<BN, CG, BK, UP4>;
    constexpr int NA = Cfg::NA, ROW = Cfg::ROW;
    constexpr int NB = Cfg::NB;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* smem_b = smem + NA * Cfg::A_STAGE;
    uint64_t* bars = (uint64_t*)(smem_b + NB * Cfg::B_STAGE);
    uint64_t* full_bar = bars;                       // [NB] weights   (CG = 2: only the even CTA's full barriers are used)
    uint64_t* empty_bar = bars + NB;                 // [NB]
    uint64_t* afull_bar = bars + 2 * NB;             // [NA] halo tiles
    uint64_t* aempty_bar = bars + 2 * NB + NA;       // [NA]
    uint64_t* tfull_bar = bars + 2 * NB + 2 * NA;    // [2]
    uint64_t* tempty_bar = tfull_bar + 2;            // [2]
    uint32_t* tmem_ptr_smem = (uint32_t*)(tempty_bar + 2);

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // provably warp-uniform
    const int rank = (CG == 2) ? (int)cluster_ctarank() : 0;
    const bool leader = rank == 0;
    const int unit0 = (CG == 2) ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
    const int unit_stride = (CG == 2) ? (int)(gridDim.x >> 1) : (int)gridDim.x;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&maps.a[0][0]); tma_prefetch_desc(&maps.a[0][1]);
        tma_prefetch_desc(&maps.w[0]); tma_prefetch_desc(&maps.w[1]);
        for (int i = 0; i < NB; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
        for (int i = 0; i < NA; ++i) { mbar_init(&afull_bar[i], 1); mbar_init(&aempty_bar[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], TC_EPI_WARPS * CG); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        if (CG == 1) {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        } else {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        }
    }
    tc_fence_before();
    if (CG == 2) cluster_sync_all(); else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;
    const TcSubProblem& s = a.sub[0];

    if (warp == 0) {
        // ============================== TMA producer (both CTAs of a pair; whole warp, lane 0 issues) ==============================
        {
            int as = 0; uint32_t aphase = 0;
            int bs = 0; uint32_t bphase = 0;
            for (int t = unit0; t < a.total_tiles; t += unit_stride) {
                const TileCoord c = decode_tile<BN, true, CG>(a, t, rank);
                const int wrow = c.n0 + rank * Cfg::B_ROWS;
                for (int kc = 0; kc < a.kchunks; ++kc) {
                    mbar_wait(&aempty_bar[as], aphase ^ 1, a.error, 0x500 + as);
                    uint8_t* sa = smem + as * Cfg::A_STAGE;
                    if (elect_one()) {
                        if (leader) mbar_expect_tx(&afull_bar[as], CG * 2 * Cfg::A_BYTES);
                        tma_load_4d_cg<CG>(&maps.a[0][0], &afull_bar[as], sa, kc * BK, c.x0 - 1, c.y0 - 1, c.b0);
                        tma_load_4d_cg<CG>(&maps.a[0][1], &afull_bar[as], sa + Cfg::A_PAD, kc * BK, c.x0 - 1, c.y0 - 1, c.b0);
                    }
                    __syncwarp();
                    if (++as == NA) { as = 0; aphase ^= 1; }
                    for (int tap = 0; tap < s.ntaps; ++tap) {
                        mbar_wait(&empty_bar[bs], bphase ^ 1, a.error, 0x100 + bs);
                        uint8_t* sb = smem_b + bs * Cfg::B_STAGE;
                        if (elect_one()) {
                            if (leader) mbar_expect_tx(&full_bar[bs], CG * Cfg::B_STAGE);
                            tma_load_3d_cg<CG>(&maps.w[0], &full_bar[bs], sb, kc * BK, wrow, s.widx[tap]);
                            tma_load_3d_cg<CG>(&maps.w[1], &full_bar[bs], sb + Cfg::B_TILE_BYTES, kc * BK, wrow, s.widx[tap]);
                        }
                        __syncwarp();
                        if (++bs == NB) { bs = 0; bphase ^= 1; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ============================== MMA issuer (even CTA of a pair only; whole warp, lane 0 issues) ==============================
        if (leader) {
            constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)((BM * CG) >> 4) << 24);
            int as = 0; uint32_t aphase = 0;
            int bs = 0; uint32_t bphase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            for (int t = unit0; t < a.total_tiles; t += unit_stride) {
                mbar_wait(&tempty_bar[acc], acc_phase ^ 1, a.error, 0x200 + acc);
                tc_fence_after();
                const uint32_t d_tile = tmem_base + (uint32_t)(acc * Cfg::ACC_COLS);
                uint32_t started = 0;                       // UP4: phases whose accumulator has been written in this tile
                for (int kc = 0; kc < a.kchunks; ++kc) {
                    mbar_wait(&afull_bar[as], aphase, a.error, 0x600 + as);
                    const uint32_t sa = smem_u32(smem + as * Cfg::A_STAGE);
                    for (int tap = 0; tap < s.ntaps; ++tap) {
                        mbar_wait(&full_bar[bs], bphase, a.error, 0x300 + bs);
                        tc_fence_after();
                        const uint32_t aoff = (uint32_t)(((s.dy[tap] + 1) * HALO_W + (s.dx[tap] + 1)) * ROW);
                        const uint64_t d_ah = make_halo_desc<ROW>(sa + aoff), d_al = make_halo_desc<ROW>(sa + Cfg::A_PAD + aoff);
                        const uint32_t sb = smem_u32(smem_b + bs * Cfg::B_STAGE);
                        const uint64_t d_bh = make_smem_desc<ROW>(sb), d_bl = make_smem_desc<ROW>(sb + Cfg::B_TILE_BYTES);
                        const int ph = UP4 ? s.phase[tap] : 0;
                        const uint32_t d_tmem = d_tile + (uint32_t)(ph * BN);
                        const uint32_t fresh = UP4 ? (((started >> ph) & 1u) ^ 1u) : ((kc | tap) ? 0u : 1u);
                        started |= 1u << ph;
                        if (elect_one()) {
#pragma unroll
                            for (int k = 0; k < BK / UMMA_K; ++k) {
                                const uint64_t koff = (uint64_t)((k * UMMA_K * 2) >> 4);
                                umma_bf16_cg<CG>(d_tmem, d_ah + koff, d_bh + koff, idesc, (fresh && k == 0) ? 0u : 1u);
                                umma_bf16_cg<CG>(d_tmem, d_ah + koff, d_bl + koff, idesc, 1u);
                                umma_bf16_cg<CG>(d_tmem, d_al + koff, d_bh + koff, idesc, 1u);
                            }
                            umma_commit_cg<CG>(&empty_bar[bs]);
                            if (tap == s.ntaps - 1) {
                                umma_commit_cg<CG>(&aempty_bar[as]);    // halo stage free (in both CTAs) once its taps retire
                                if (kc == a.kchunks - 1) umma_commit_cg<CG>(&tfull_bar[acc]);
                            }
                        }
                        __syncwarp();
                        if (++bs == NB) { bs = 0; bphase ^= 1; }
                    }
                    if (++as == NA) { as = 0; aphase ^= 1; }
                }
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        tc_epilogue<BN, true, CG, UP4>(a, tfull_bar, tempty_bar, tmem_base, rank, warp, lane, unit0, unit_stride);
    }
    tc_fence_before();
    if (CG == 2) cluster_sync_all(); else __syncthreads();
    if (warp == 1) {
        __syncwarp();
        tc_fence_after();
        if (CG == 1)
            asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
        else
            asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
    }
}

// ------------------------------------------------------------------------------- halo kernel with resident weights
// The 32-output-channel layers of the 1024^2 model (32 -> 32 plain, 64 -> 32 up): an MMA with N = 32 needs 40 clk of
// operand fetch for 16 clk of math, a tap is only 6-12 of them, and a weight tile is 2-4 KB -- streaming the weights per
// (tile, tap) through a barrier ring makes the producer and the per-tap barrier round trips the bottleneck (measured:
// 83 clk per MMA).  Here all 9 taps of the (single) K chunk stay in shared memory for the life of the CTA (36-72 KB),
// the producer only streams halos (ring of up to 4), and the MMA warp issues the 54-108 MMAs of a tile in ONE elected
// block behind a single barrier wait.
template <int BN, int BK, bool UP4> struct TcHaloRwCfg {
    static constexpr int ROW = BK * 2;
    static constexpr int A_BYTES = HALO_H * HALO_W * ROW;
    static constexpr int A_PAD = (A_BYTES + 1023) / 1024 * 1024;
    static constexpr int A_STAGE = 2 * A_PAD;
    static constexpr int W_TILE = BN * ROW;                                  // one plane of one tap
    static constexpr int W_TAP = 2 * W_TILE;
    static constexpr int W_BYTES = 9 * W_TAP;
    static constexpr int BUDGET = 227 * 1024 - 1024 - 512;
    static constexpr int NA_RAW = (BUDGET - W_BYTES) / A_STAGE;
    static constexpr int NA = NA_RAW > 4 ? 4 : NA_RAW;
    static constexpr int SMEM_BYTES = W_BYTES + NA * A_STAGE + 1024 + 512;
    static constexpr int ACC_COLS = (UP4 ? 4 : 1) * BN;
    static constexpr int TMEM_COLS = (2 * ACC_COLS <= 32) ? 32 : (2 * ACC_COLS <= 64) ? 64 : (2 * ACC_COLS <= 128) ? 128 : (2 * ACC_COLS <= 256) ? 256 : 512;
    static_assert(NA >= 2, "halo ring too shallow");
    static_assert(W_TILE % 1024 == 0, "weight tiles must stay swizzle-aligned");
};

template <int BN, int BK, bool UP4>
__global__ void __launch_bounds__(TC_THREADS, 1)
modconv_tc_halo_rw_kernel(const __grid_constant__ TcMaps maps, const __grid_constant__ TcKernelArgs a) {
    using Cfg = TcHaloRwCfg<BN, BK, UP4>;
    constexpr int NA = Cfg::NA, ROW = Cfg::ROW;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem_w = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* smem_a = smem_w + Cfg::W_BYTES;
    uint64_t* bars = (uint64_t*)(smem_a + NA * Cfg::A_STAGE);
    uint64_t* afull_bar = bars;                      // [NA]
    uint64_t* aempty_bar = bars + NA;                // [NA]
    uint64_t* tfull_bar = bars + 2 * NA;             // [2]
    uint64_t* tempty_bar = tfull_bar + 2;            // [2]
    uint64_t* wfull_bar = tempty_bar + 2;            // [1]
    uint32_t* tmem_ptr_smem = (uint32_t*)(wfull_bar + 1);

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const int unit0 = (int)blockIdx.x, unit_stride = (int)gridDim.x;
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&maps.a[0][0]); tma_prefetch_desc(&maps.a[0][1]);
        tma_prefetch_desc(&maps.w[0]); tma_prefetch_desc(&maps.w[1]);
        for (int i = 0; i < NA; ++i) { mbar_init(&afull_bar[i], 1); mbar_init(&aempty_bar[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], TC_EPI_WARPS); }
        mbar_init(wfull_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;
    const TcSubProblem& s = a.sub[0];

    if (warp == 0) {
        // ============================== TMA producer (whole warp, one elected lane issues) ==============================
        if (elect_one()) {
            mbar_expect_tx(wfull_bar, Cfg::W_BYTES);
            for (int tap = 0; tap < 9; ++tap) {
                tma_load_3d(&maps.w[0], wfull_bar, smem_w + tap * Cfg::W_TAP, 0, 0, s.widx[tap]);
                tma_load_3d(&maps.w[1], wfull_bar, smem_w + tap * Cfg::W_TAP + Cfg::W_TILE, 0, 0, s.widx[tap]);
            }
        }
        __syncwarp();
        int as = 0; uint32_t aphase = 0;
        for (int t = unit0; t < a.total_tiles; t += unit_stride) {
            const TileCoord c = decode_tile<BN, true, 1>(a, t, 0);
            mbar_wait(&aempty_bar[as], aphase ^ 1, a.error, 0x500 + as);
            uint8_t* sa = smem_a + as * Cfg::A_STAGE;
            if (elect_one()) {
                mbar_expect_tx(&afull_bar[as], 2 * Cfg::A_BYTES);
                tma_load_4d(&maps.a[0][0], &afull_bar[as], sa, 0, c.x0 - 1, c.y0 - 1, c.b0);
                tma_load_4d(&maps.a[0][1], &afull_bar[as], sa + Cfg::A_PAD, 0, c.x0 - 1, c.y0 - 1, c.b0);
            }
            __syncwarp();
            if (++as == NA) { as = 0; aphase ^= 1; }
        }
    } else if (warp == 1) {
        // ============================== MMA issuer (whole warp, one elected lane issues) ==============================
        constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
        int as = 0; uint32_t aphase = 0;
        int acc = 0; uint32_t acc_phase = 0;
        mbar_wait(wfull_bar, 0, a.error, 0x700);
        const uint32_t sw0 = smem_u32(smem_w);
        for (int t = unit0; t < a.total_tiles; t += unit_stride) {
            mbar_wait(&tempty_bar[acc], acc_phase ^ 1, a.error, 0x200 + acc);
            mbar_wait(&afull_bar[as], aphase, a.error, 0x600 + as);
            tc_fence_after();
            const uint32_t d_tile = tmem_base + (uint32_t)(acc * Cfg::ACC_COLS);
            const uint32_t sa = smem_u32(smem_a + as * Cfg::A_STAGE);
            if (elect_one()) {
                uint32_t started = 0;
#pragma unroll 1
                for (int tap = 0; tap < 9; ++tap) {
                    const uint32_t aoff = (uint32_t)(((s.dy[tap] + 1) * HALO_W + (s.dx[tap] + 1)) * ROW);
                    const uint64_t d_ah = make_halo_desc<ROW>(sa + aoff), d_al = make_halo_desc<ROW>(sa + Cfg::A_PAD + aoff);
                    const uint32_t sb = sw0 + (uint32_t)(tap * Cfg::W_TAP);
                    const uint64_t d_bh = make_smem_desc<ROW>(sb), d_bl = make_smem_desc<ROW>(sb + Cfg::W_TILE);
                    const int ph = UP4 ? s.phase[tap] : 0;
                    const uint32_t d_tmem = d_tile + (uint32_t)(ph * BN);
                    const uint32_t fresh = UP4 ? (((started >> ph) & 1u) ^ 1u) : (tap ? 0u : 1u);
                    started |= 1u << ph;
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; ++k) {
                        const uint64_t koff = (uint64_t)((k * UMMA_K * 2) >> 4);
                        umma_bf16(d_tmem, d_ah + koff, d_bh + koff, idesc, (fresh && k == 0) ? 0u : 1u);
                        umma_bf16(d_tmem, d_ah + koff, d_bl + koff, idesc, 1u);
                        umma_bf16(d_tmem, d_al + koff, d_bh + koff, idesc, 1u);
                    }
                }
                umma_commit(&aempty_bar[as]);
                umma_commit(&tfull_bar[acc]);
            }
            __syncwarp();
            if (++as == NA) { as = 0; aphase ^= 1; }
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    } else {
        tc_epilogue<BN, true, 1, UP4>(a, tfull_bar, tempty_bar, tmem_base, 0, warp, lane, unit0, unit_stride);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        __syncwarp();
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
    }
}

// ------------------------------------------------------------------------------- transposed halo variant (Cout = 128)
// An M=128 x N=128 MMA fetches (128 + 128) rows x 32 B of operands for 64 clk of math: exactly the 128 B/clk the SM's
// shared memory delivers (scripts/exp_mma_rate.cu), so the Cout = 128 layers run at ~2/3 of the tensor rate.  This
// variant computes the TRANSPOSED product: the weights are the M = 128 operand, 256 pixels (a 32 x 8 tile) the N operand,
// D[channel][pixel] -> (128 + 256) x 32 B per 128 clk = 96 B/clk, the same slack the Cout >= 256 layers have.
// The pixels come from one 34 x 10 halo per 32-channel K chunk (64 B rows, SWIZZLE_64B, shifted descriptors with a
// 640 B group stride: exp_halo_desc.cu covers this case), the weights stream per tap.  TMEM lanes are output channels, so
// the epilogue thread owns ONE channel and 32 consecutive tile pixels per chunk: demod / bias are per-thread scalars, the
// noise row is shared by the warp, and the fp32 NCHW capture is written as 32 B row segments.  Used for plain layers with
// Cout = 128 and H a multiple of 32 (128 -> 128 at 256^2); when a conv follows, the epilogue also emits its pre-scaled
// bf16 hi/lo NHWC planes (lane pairs trade values: one bf16x2 store per lane and pixel pair).
constexpr int HT_TH = 32, HT_TW = 8, HT_W = HT_TW + 2, HT_H = HT_TH + 2, HT_BK = 32, HT_N = HT_TH * HT_TW;
struct TcHaloTCfg {
    static constexpr int ROW = HT_BK * 2;                                        // 64 B operand rows
    static constexpr int A_BYTES = HT_H * HT_W * ROW;                            // 21760 bytes per halo plane
    static constexpr int A_PAD = (A_BYTES + 1023) / 1024 * 1024;                 // 22528
    static constexpr int A_STAGE = 2 * A_PAD;
    static constexpr int NA = 2;
    static constexpr int W_TILE_BYTES = 128 * ROW;                               // 8192 per plane
    static constexpr int W_STAGE = 2 * W_TILE_BYTES;
    static constexpr int NW = 8;
    static constexpr int SMEM_BYTES = NA * A_STAGE + NW * W_STAGE + 1024 + 512;
    static constexpr int TMEM_COLS = 512;
};

__device__ __forceinline__ uint64_t make_halo_t_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)((HT_W * TcHaloTCfg::ROW) >> 4) << 32;   // 8-pixel row groups are one halo row (640 B) apart
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)4 << 61;                                 // SWIZZLE_64B
    return d;
}

__global__ void __launch_bounds__(TC_THREADS, 1)
modconv_tc_halo_t_kernel(const __grid_constant__ TcMaps maps, const __grid_constant__ TcKernelArgs a) {
    using Cfg = TcHaloTCfg;
    constexpr int NA = Cfg::NA, NW = Cfg::NW, BK = HT_BK;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* smem_w = smem + NA * Cfg::A_STAGE;
    uint64_t* bars = (uint64_t*)(smem_w + NW * Cfg::W_STAGE);
    uint64_t* full_bar = bars;                       // [NW] weights
    uint64_t* empty_bar = bars + NW;                 // [NW]
    uint64_t* afull_bar = bars + 2 * NW;             // [NA] halo tiles
    uint64_t* aempty_bar = bars + 2 * NW + NA;       // [NA]
    uint64_t* tfull_bar = bars + 2 * NW + 2 * NA;    // [2]
    uint64_t* tempty_bar = tfull_bar + 2;            // [2]
    uint32_t* tmem_ptr_smem = (uint32_t*)(tempty_bar + 2);

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // provably warp-uniform
    // tiles: n-tile slowest, then spatial tile, then (transposed conv) the 4 output phases, rotated by the spatial index so
    // that a CTA's static stride (148 = 4 * 37) does not lock onto one phase (they have 4 / 2 / 2 / 1 taps)
    const int tiles_x = a.sub[0].ow / HT_TW, tiles_y = a.sub[0].oh / HT_TH;
    const int m_tiles = a.batch * tiles_y * tiles_x;
    const int per = a.nsub;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&maps.a[0][0]); tma_prefetch_desc(&maps.a[0][1]);
        tma_prefetch_desc(&maps.w[0]); tma_prefetch_desc(&maps.w[1]);
        for (int i = 0; i < NW; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
        for (int i = 0; i < NA; ++i) { mbar_init(&afull_bar[i], 1); mbar_init(&aempty_bar[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], TC_EPI_WARPS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;

    if (warp == 0) {
        // ============================== TMA producer (whole warp, lane 0 issues) ==============================
        {
            int as = 0; uint32_t aphase = 0;
            int ws = 0; uint32_t wphase = 0;
            for (int t = blockIdx.x; t < a.total_tiles; t += gridDim.x) {
                const int rt = t % (m_tiles * per), n0 = (t / (m_tiles * per)) * 128;
                const int m = rt / per;
                const TcSubProblem& s = a.sub[per == 1 ? 0 : ((rt % per) + m) & 3];
                const int x0 = (m % tiles_x) * HT_TW, y0 = ((m / tiles_x) % tiles_y) * HT_TH, b = m / (tiles_x * tiles_y);
                for (int kc = 0; kc < a.kchunks; ++kc) {
                    mbar_wait(&aempty_bar[as], aphase ^ 1, a.error, 0x500 + as);
                    uint8_t* sa = smem + as * Cfg::A_STAGE;
                    if (elect_one()) {
                        mbar_expect_tx(&afull_bar[as], 2 * Cfg::A_BYTES);
                        tma_load_4d(&maps.a[0][0], &afull_bar[as], sa, kc * BK, x0 - 1, y0 - 1, b);
                        tma_load_4d(&maps.a[0][1], &afull_bar[as], sa + Cfg::A_PAD, kc * BK, x0 - 1, y0 - 1, b);
                    }
                    __syncwarp();
                    if (++as == NA) { as = 0; aphase ^= 1; }
                    for (int tap = 0; tap < s.ntaps; ++tap) {
                        mbar_wait(&empty_bar[ws], wphase ^ 1, a.error, 0x100 + ws);
                        uint8_t* sw = smem_w + ws * Cfg::W_STAGE;
                        if (elect_one()) {
                            mbar_expect_tx(&full_bar[ws], Cfg::W_STAGE);
                            tma_load_3d(&maps.w[0], &full_bar[ws], sw, kc * BK, n0, s.widx[tap]);
                            tma_load_3d(&maps.w[1], &full_bar[ws], sw + Cfg::W_TILE_BYTES, kc * BK, n0, s.widx[tap]);
                        }
                        __syncwarp();
                        if (++ws == NW) { ws = 0; wphase ^= 1; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ============================== MMA issuer (whole warp, lane 0 issues) ==============================
        {
            // D[128 channels][256 pixels] = W[128][K] . X[256][K]^T : A = weights, B = pixels, both K-major
            constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(HT_N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
            int as = 0; uint32_t aphase = 0;
            int ws = 0; uint32_t wphase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            for (int t = blockIdx.x; t < a.total_tiles; t += gridDim.x) {
                const int rt = t % (m_tiles * per);
                const TcSubProblem& s = a.sub[per == 1 ? 0 : ((rt % per) + rt / per) & 3];
                mbar_wait(&tempty_bar[acc], acc_phase ^ 1, a.error, 0x200 + acc);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * HT_N);
                for (int kc = 0; kc < a.kchunks; ++kc) {
                    mbar_wait(&afull_bar[as], aphase, a.error, 0x600 + as);
                    const uint32_t sa = smem_u32(smem + as * Cfg::A_STAGE);
                    for (int tap = 0; tap < s.ntaps; ++tap) {
                        mbar_wait(&full_bar[ws], wphase, a.error, 0x300 + ws);
                        tc_fence_after();
                        const uint32_t xoff = (uint32_t)(((s.dy[tap] + 1) * HT_W + (s.dx[tap] + 1)) * Cfg::ROW);
                        const uint64_t d_xh = make_halo_t_desc(sa + xoff), d_xl = make_halo_t_desc(sa + Cfg::A_PAD + xoff);
                        const uint32_t sw = smem_u32(smem_w + ws * Cfg::W_STAGE);
                        const uint64_t d_wh = make_smem_desc<Cfg::ROW>(sw), d_wl = make_smem_desc<Cfg::ROW>(sw + Cfg::W_TILE_BYTES);
                        if (elect_one()) {
#pragma unroll
                            for (int k = 0; k < BK / UMMA_K; ++k) {
                                const uint64_t koff = (uint64_t)((k * UMMA_K * 2) >> 4);
                                umma_bf16(d_tmem, d_wh + koff, d_xh + koff, idesc, (kc | tap | k) ? 1u : 0u);
                                umma_bf16(d_tmem, d_wl + koff, d_xh + koff, idesc, 1u);
                                umma_bf16(d_tmem, d_wh + koff, d_xl + koff, idesc, 1u);
                            }
                            umma_commit(&empty_bar[ws]);
                            if (tap == s.ntaps - 1) {
                                umma_commit(&aempty_bar[as]);
                                if (kc == a.kchunks - 1) umma_commit(&tfull_bar[acc]);
                            }
                        }
                        __syncwarp();
                        if (++ws == NW) { ws = 0; wphase ^= 1; }
                    }
                    if (++as == NA) { as = 0; aphase ^= 1; }
                }
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // ============================== epilogue: one output channel per thread ==============================
        const int quarter = warp & 3;
        const int chalf = (warp - 2) >> 2;
        int acc = 0; uint32_t acc_phase = 0;
        for (int t = blockIdx.x; t < a.total_tiles; t += gridDim.x) {
            const int rt = t % (m_tiles * per), n0 = (t / (m_tiles * per)) * 128;
            const int m = rt / per;
            const TcSubProblem& s = a.sub[per == 1 ? 0 : ((rt % per) + m) & 3];
            const int x0 = (m % tiles_x) * HT_TW, y0 = ((m / tiles_x) % tiles_y) * HT_TH, b = m / (tiles_x * tiles_y);
            const int ch = n0 + quarter * 32 + lane;
            const float d = __ldg(a.demod + (int64_t)b * a.cout + ch);
            const float bias = a.bias ? __ldg(a.bias + ch) : 0.0f;
            const float sn = a.s_next ? __ldg(a.s_next + (int64_t)b * a.cout + ch) : 0.0f;
            float* plane = a.out_f32 + ((int64_t)b * a.cout + ch) * ((int64_t)a.out_h * a.out_w);
            const float* nzp = a.noise ? a.noise + (int64_t)b * a.noise_bstride : nullptr;
            mbar_wait(&tfull_bar[acc], acc_phase, a.error, 0x400 + acc);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * HT_N);
#pragma unroll 1
            for (int c0 = chalf * 32; c0 < HT_N; c0 += 64) {
                uint32_t r[32];
                tmem_ld_32x32(taddr + (uint32_t)c0, r);
                tmem_ld_wait();
                if (a.mode == 1) {
                    // transposed-conv phase: demodulated fp32 into the NHWC scratch at (2y + py, 2x + px); for every pixel
                    // the warp writes 32 consecutive channels = one 128 B line
#pragma unroll
                    for (int rr = 0; rr < 4; ++rr) {
                        const int oy = (y0 + c0 / HT_TW + rr) * s.ostride + s.ooff_y;
                        float* row = a.out_f32 + (((int64_t)b * a.out_h + oy) * a.out_w + x0 * s.ostride + s.ooff_x) * a.cout + ch;
#pragma unroll
                        for (int j = 0; j < 8; ++j) row[(int64_t)j * s.ostride * a.cout] = __fmul_rn(__uint_as_float(r[rr * 8 + j]), d);
                    }
                    continue;
                }
#pragma unroll
                for (int rr = 0; rr < 4; ++rr) {            // 32 columns = 4 tile rows of 8 pixels
                    const int y = y0 + c0 / HT_TW + rr;
                    float nz[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                    if (nzp) {
                        const float4 n0v = __ldg(reinterpret_cast<const float4*>(nzp + (int64_t)y * a.out_w + x0));
                        const float4 n1v = __ldg(reinterpret_cast<const float4*>(nzp + (int64_t)y * a.out_w + x0) + 1);
                        nz[0] = n0v.x; nz[1] = n0v.y; nz[2] = n0v.z; nz[3] = n0v.w; nz[4] = n1v.x; nz[5] = n1v.y; nz[6] = n1v.z; nz[7] = n1v.w;
                    }
                    float v[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        float x = __fmul_rn(__uint_as_float(r[rr * 8 + j]), d);
                        x = __fadd_rn(x, __fmul_rn(a.noise_w, nz[j]));
                        if (a.bias) x = __fadd_rn(x, bias);
                        if (a.act) x = lrelu_scale(x, 0.2f, 1.41421356237309504880f);
                        v[j] = x;
                    }
                    float4* dst = reinterpret_cast<float4*>(plane + (int64_t)y * a.out_w + x0);
                    dst[0] = make_float4(v[0], v[1], v[2], v[3]);
                    dst[1] = make_float4(v[4], v[5], v[6], v[7]);
                    if (a.s_next) {
                        // the next conv's pre-scaled bf16 hi/lo NHWC planes: per pixel the warp writes 32 consecutive
                        // channels (64 B); lane pairs trade values so that every lane stores a bf16x2 for half of the pixels
                        const int64_t off = (((int64_t)b * a.out_h + y) * a.out_w + x0) * a.cout + (ch & ~1);
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const float xs = __fmul_rn(v[j], sn);
                            const float other = __shfl_xor_sync(0xffffffffu, xs, 1);
                            if ((j & 1) == (lane & 1)) {
                                const float c0v = (lane & 1) ? other : xs, c1v = (lane & 1) ? xs : other;   // channels ch&~1, ch|1
                                const bf16 h0 = __float2bfloat16_rn(c0v), h1 = __float2bfloat16_rn(c1v);
                                const bf16 l0 = __float2bfloat16_rn(c0v - __bfloat162float(h0)), l1 = __float2bfloat16_rn(c1v - __bfloat162float(h1));
                                *reinterpret_cast<uint32_t*>(a.next_hi + off + (int64_t)j * a.cout) =
                                    (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
                                *reinterpret_cast<uint32_t*>(a.next_lo + off + (int64_t)j * a.cout) =
                                    (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
                            }
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty_bar[acc]);
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        __syncwarp();
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
    }
}

// ------------------------------------------------------------------------------- blur + activation + split
// Second half of the up-sampling StyledConv: Blur(4x4, pad (1,1)) + noise + bias + lrelu*sqrt2 over the NHWC fp32
// scratch, writing the fp32 NCHW capture and the next conv's pre-scaled bf16 hi/lo NHWC planes in one pass.
struct BlurSplitArgs {
    const float* in; int IH, IW;          // [B][IH][IW][C]
    float* out_f32; int OH, OW, C, batch; // [B][C][OH][OW]
    const float* blur_k; const float* noise; int64_t noise_bstride; float noise_w; const float* bias;
    const float* s_next; bf16* next_hi; bf16* next_lo;   // [B][OH][OW][C]
    int act;                              // apply lrelu(0.2)*sqrt2 (StyledConv) or blur only (bare ModulatedConv2d)
};
// Tile geometry by channel block CB: 64 channels -> 8 x 16 output pixels, a warp owns one column pair (32 lanes x 2
// channels); 32 channels (the 1024^2 layer) -> 8 x 32 output pixels, a warp owns TWO column pairs (16 lanes x 2 channels
// each), so no lane idles and the NCHW capture is written as full 128 B rows.
constexpr int BS_TH = 8, BS_IH = BS_TH + 3;
template <int CB> struct BlurGeo {
    static constexpr int LPG = CB / 2;                       // lanes per column-pair group
    static constexpr int GROUPS = 32 / LPG;                  // column pairs per warp
    static constexpr int TW = 8 * GROUPS * 2;                // 16 / 32 output columns per block (8 warps)
    static constexpr int IW = TW + 3;
    static constexpr int OPITCH = BS_TH * TW + 1;            // transposing writes are 2-way conflicted at worst
    static constexpr int SMEM = BS_IH * IW * CB * 4;         // 53,504 B (CB 64) / 49,280 B (CB 32)
    static_assert(CB * OPITCH * 4 <= SMEM, "the transposed output must fit in the input tile");
};

// packed fp32x2 arithmetic (sm_100: FFMA2 / FADD2 / FMUL2): two channels per lane per instruction
using u64 = unsigned long long;
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
    float2 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(reinterpret_cast<u64&>(d)) : "l"(reinterpret_cast<u64&>(a)), "l"(reinterpret_cast<u64&>(b)), "l"(reinterpret_cast<u64&>(c)));
    return d;
}
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
    float2 d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(reinterpret_cast<u64&>(d)) : "l"(reinterpret_cast<u64&>(a)), "l"(reinterpret_cast<u64&>(b)));
    return d;
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) {
    float2 d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(reinterpret_cast<u64&>(d)) : "l"(reinterpret_cast<u64&>(a)), "l"(reinterpret_cast<u64&>(b)));
    return d;
}
__device__ __forceinline__ float2 splat2(float v) { return make_float2(v, v); }
// explicit shared-space accesses by 32-bit address: the tile pointer is picked from a ring at run time, and through a
// generic pointer every access becomes LD.E / ST.E with 64-bit address arithmetic (measured: ~250 extra integer instructions
// per tile and generic-path loads in a kernel that is co-limited by issue)
__device__ __forceinline__ float2 lds_f2(uint32_t addr) {
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ float lds_f1(uint32_t addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts_f1(uint32_t addr, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory"); }

// Block = 8 x TW output pixels x CB channels, 8 warps; lane = 2 channels (LDS.64, packed fp32x2 math, 32-bit bf16x2
// stores).  A column-pair group of lanes owns the output columns (px, px+1) and walks down the rows, sharing the 5 input
// columns the pair needs.  Separable taps (the reference's [1,3,3,1] outer product always is): a horizontal 4-tap pass per
// input row, then a vertical 4-tap pass over a sliding register window = 8 FMAs per output instead of 16; a non-separable
// `blur.kernel` takes the generic 16-tap path.  The bf16 hi/lo NHWC planes are written straight from registers; the fp32
// NCHW capture goes through a shared-memory transpose that re-uses the input tile's storage.  All index arithmetic is
// hoisted out of the per-element loops: the kernel is HBM-bound only if its instruction count is small.
// The input tile comes from ONE TMA box load (fp32 NHWC scratch, out-of-bounds rows / columns / channels are zero-filled
// by the tensor map) into a ring of two, issued a tile ahead by thread 0: no per-thread staging instructions and the load
// of tile i+1 overlaps the math and stores of tile i.
template <bool SEP, int CB>
__global__ void __launch_bounds__(256, 2) blur_act_split_kernel(BlurSplitArgs a, const __grid_constant__ CUtensorMap in_map) {
    using G = BlurGeo<CB>;
    constexpr int TW = G::TW, IW = G::IW, LPG = G::LPG, OPITCH = G::OPITCH, TILE_BYTES = G::SMEM;
    extern __shared__ __align__(128) float stile_raw[];    // 2 x [11*IW][CB] fp32; a slot is re-used as sout[CB][OPITCH]
    __shared__ float sk[16], skx[4], sky[4];
    __shared__ float snz[BS_TH * TW];
    __shared__ uint64_t tma_bar[2];
    float* const ring0 = (float*)(((uintptr_t)stile_raw + 127) & ~(uintptr_t)127);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int grp = lane / LPG, cl = lane - grp * LPG;      // column-pair group of this lane, channel pair inside the block
    if (tid < 16) sk[tid] = a.blur_k[(3 - tid / 4) * 4 + (3 - tid % 4)];   // flipped taps
    __syncthreads();
    if (tid < 4) { sky[tid] = sk[tid * 4]; skx[tid] = SEP ? sk[tid] / sk[0] : 0.0f; }   // k[i][j] = sky[i] * skx[j]
    const int tiles_x = (a.OW + TW - 1) / TW, tiles_y = (a.OH + BS_TH - 1) / BS_TH;
    const int cgroups = (a.C + CB - 1) / CB;
    const int64_t total = (int64_t)a.batch * tiles_y * tiles_x * cgroups;
    auto tile_coords = [&](int64_t tile, int& b, int& y0, int& x0, int& c0) {
        const int cg = (int)(tile % cgroups);
        int64_t r = tile / cgroups;
        const int tx = (int)(r % tiles_x); r /= tiles_x;
        const int ty = (int)(r % tiles_y);
        b = (int)(r / tiles_y); y0 = ty * BS_TH; x0 = tx * TW; c0 = cg * CB;
    };
    if (tid == 0) {
        mbar_init(&tma_bar[0], 1); mbar_init(&tma_bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        if ((int64_t)blockIdx.x < total) {
            int b, y0, x0, c0;
            tile_coords(blockIdx.x, b, y0, x0, c0);
            mbar_expect_tx(&tma_bar[0], TILE_BYTES);
            tma_load_4d(&in_map, &tma_bar[0], ring0, c0, x0 - 1, y0 - 1, b);
        }
    }
    int it = 0;
    for (int64_t tile = blockIdx.x; tile < total; tile += gridDim.x, ++it) {
        int b, y0, x0, c0;
        tile_coords(tile, b, y0, x0, c0);
        float* const stile = ring0 + (it & 1) * (TILE_BYTES / 4);
        const uint32_t stile_u32 = smem_u32(stile);                    // tile: [pix][CB / 2 lanes] float2
        __syncthreads();     // previous tile's transpose reads are done (and the tap tables are visible)
        // the other ring slot held the previous tile (its transposed output was just consumed): refill it a tile ahead
        if (tid == 0 && tile + gridDim.x < total) {
            int nb, ny0, nx0, nc0;
            tile_coords(tile + gridDim.x, nb, ny0, nx0, nc0);
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // generic-proxy accesses of that slot are done
            mbar_expect_tx(&tma_bar[(it + 1) & 1], TILE_BYTES);
            tma_load_4d(&in_map, &tma_bar[(it + 1) & 1], ring0 + ((it + 1) & 1) * (TILE_BYTES / 4), nc0, nx0 - 1, ny0 - 1, nb);
        }
        if (tid < BS_TH * TW) {
            const int oy = y0 + tid / TW, ox = x0 + tid % TW;
            snz[tid] = (a.noise && oy < a.OH && ox < a.OW) ? a.noise_w * __ldg(a.noise + (int64_t)b * a.noise_bstride + (int64_t)oy * a.OW + ox) : 0.0f;
        }
        mbar_wait(&tma_bar[it & 1], (uint32_t)((it >> 1) & 1), nullptr, 0);
        __syncthreads();

        // ---- blur: column pair (px, px+1), rows top to bottom
        float2 res[2][BS_TH];
        const int px = (warp * G::GROUPS + grp) * 2;
        const uint32_t in_base = stile_u32 + (uint32_t)(px * LPG + cl) * 8u;
        {
            const bool chok = c0 + 2 * cl < a.C;
            const float2 bias = (chok && a.bias) ? *reinterpret_cast<const float2*>(a.bias + c0 + 2 * cl) : make_float2(0.f, 0.f);
            const float2 sn = (a.s_next && chok) ? *reinterpret_cast<const float2*>(a.s_next + (int64_t)b * a.C + c0 + 2 * cl) : make_float2(0.f, 0.f);
            const bool colok0 = chok && x0 + px < a.OW, colok1 = chok && x0 + px + 1 < a.OW;
            // NHWC element offset of (b, y0, x0+px, c0+2*cl); advances by OW*C per row, C per column
            const int64_t off0 = (((int64_t)b * a.OH + y0) * a.OW + x0 + px) * a.C + c0 + 2 * cl;
            // plane pointers of this lane's first pixel, in bf16x2 units: + C/2 per column, + OW*C/2 per row.  (Only
            // dereferenced when the planes are wanted; the stores below are predicated, not branched around.)
            __nv_bfloat162* ph = reinterpret_cast<__nv_bfloat162*>(a.next_hi + off0);
            __nv_bfloat162* pl = reinterpret_cast<__nv_bfloat162*>(a.next_lo + off0);
            const int c2 = a.C >> 1;
            const int64_t rs2 = ((int64_t)a.OW * a.C) >> 1;
            const bool st0 = a.s_next != nullptr && colok0, st1 = a.s_next != nullptr && colok1;
            float2 win[2][4][SEP ? 1 : 4];
#pragma unroll
            for (int rr = 0; rr < BS_IH; ++rr) {
                float2 in5[5];
#pragma unroll
                for (int j = 0; j < 5; ++j) in5[j] = lds_f2(in_base + (uint32_t)((rr * IW + j) * LPG) * 8u);
#pragma unroll
                for (int cx = 0; cx < 2; ++cx) {
#pragma unroll
                    for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                        for (int kx = 0; kx < (SEP ? 1 : 4); ++kx) win[cx][ky][kx] = win[cx][ky + 1][kx];
                    if (SEP) {
                        float2 h = make_float2(0.f, 0.f);
#pragma unroll
                        for (int kx = 0; kx < 4; ++kx) h = ffma2(in5[cx + kx], splat2(skx[kx]), h);
                        win[cx][3][0] = h;
                    } else {
#pragma unroll
                        for (int kx = 0; kx < 4; ++kx) win[cx][3][kx] = in5[cx + kx];
                    }
                }
                if (rr >= 3) {
                    const int py = rr - 3;
                    const bool rowok = y0 + py < a.OH;
#pragma unroll
                    for (int cx = 0; cx < 2; ++cx) {
                        float2 v = make_float2(0.f, 0.f);
                        if (SEP) {
#pragma unroll
                            for (int ky = 0; ky < 4; ++ky) v = ffma2(win[cx][ky][0], splat2(sky[ky]), v);
                        } else {
#pragma unroll
                            for (int ky = 0; ky < 4; ++ky)
#pragma unroll
                                for (int kx = 0; kx < 4; ++kx) v = ffma2(win[cx][ky][kx], splat2(sk[ky * 4 + kx]), v);
                        }
                        v = fadd2(fadd2(v, splat2(snz[py * TW + px + cx])), bias);
                        // lrelu(x)*sqrt2 = max(x*sqrt2, x*0.2*sqrt2)
                        if (a.act) {
                            const float2 p = fmul2(v, splat2(1.41421356237309504880f)), q = fmul2(v, splat2(0.2f * 1.41421356237309504880f));
                            v = make_float2(fmaxf(p.x, q.x), fmaxf(p.y, q.y));
                        }
                        res[cx][py] = v;
                        const float2 xs = fmul2(v, sn);
                        const __nv_bfloat162 h = __floats2bfloat162_rn(xs.x, xs.y);
                        const float2 hf = __bfloat1622float2(h);
                        const __nv_bfloat162 l = __floats2bfloat162_rn(xs.x - hf.x, xs.y - hf.y);
                        if (rowok && (cx ? st1 : st0)) {
                            ph[cx * c2] = h;
                            pl[cx * c2] = l;
                        }
                    }
                    ph += rs2;
                    pl += rs2;
                }
            }
        }
        __syncthreads();     // everyone is done reading the input tile
        // sout = the tile's storage again, [CB][OPITCH] fp32
        {
            const uint32_t w0 = stile_u32 + (uint32_t)((2 * cl) * OPITCH + px) * 4u;
#pragma unroll
            for (int cx = 0; cx < 2; ++cx)
#pragma unroll
                for (int py = 0; py < BS_TH; ++py) {
                    sts_f1(w0 + (uint32_t)(py * TW + cx) * 4u, res[cx][py].x);
                    sts_f1(w0 + (uint32_t)(OPITCH + py * TW + cx) * 4u, res[cx][py].y);
                }
        }
        __syncthreads();
        // ---- NCHW capture: warp -> channels warp, warp+8, ...; a pass of the 32 lanes covers 32 / TW rows of TW pixels
        {
            constexpr int RPP = 32 / TW;                    // rows per pass: 2 (TW 16) or 1 (TW 32)
            const int ox = x0 + (lane % TW), oyb = y0 + lane / TW;
            const bool colok = ox < a.OW;
            const int64_t plane = (int64_t)a.OH * a.OW;
            float* dst = a.out_f32 + ((int64_t)b * a.C + c0 + warp) * plane + (int64_t)oyb * a.OW + ox;
            uint32_t sp = stile_u32 + (uint32_t)(warp * OPITCH + lane) * 4u;
#pragma unroll
            for (int j = 0; j < CB / 8; ++j) {
                if (c0 + warp + 8 * j >= a.C) break;
#pragma unroll
                for (int i = 0; i < BS_TH / RPP; ++i)
                    if (colok && oyb + RPP * i < a.OH) dst[(int64_t)(RPP * i) * a.OW] = lds_f1(sp + (uint32_t)(32 * i) * 4u);
                dst += 8 * plane;
                sp += (uint32_t)(8 * OPITCH) * 4u;
            }
        }
    }
}

// NCHW fp32 * s -> NHWC bf16 hi/lo (only used for the 4x4 constant input; tiny)
__global__ void __launch_bounds__(256) prescale_split_kernel(bf16* __restrict__ hi, bf16* __restrict__ lo, const float* __restrict__ x,
                                                             const float* __restrict__ s, int batch, int C, int64_t hw) {
    const int64_t total = (int64_t)batch * hw * C;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % C);
        const int64_t p = (i / C) % hw;
        const int b = (int)(i / (C * hw));
        const float v = __fmul_rn(x[((int64_t)b * C + c) * hw + p], s[(int64_t)b * C + c]);
        const bf16 h = __float2bfloat16_rn(v);
        hi[i] = h;
        lo[i] = __float2bfloat16_rn(v - __bfloat162float(h));
    }
}

// NCHW fp32 plane set -> a channel slice [c_off, c_off + C) of an NHWC bf16 hi/lo plane pair with c_total channels
// (unscaled), through a shared-memory transpose.  Used by the DatasetGAN labeller to stack the captures of one resolution along K.
__global__ void __launch_bounds__(256) nchw_to_nhwc_split_kernel(bf16* __restrict__ hi, bf16* __restrict__ lo, const float* __restrict__ x,
                                                                 int C, int64_t hw, int c_total, int c_off) {
    // 64 channels x 64 pixels per block: 128-bit loads along the pixels (when hw is a multiple of 4), 128 B stores along
    // the channels
    __shared__ float tile[64][65];
    const int b = blockIdx.z, c0 = blockIdx.y * 64;
    const int64_t p0 = (int64_t)blockIdx.x * 64;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const bool vec = (hw & 3) == 0;
    if (vec) {
        for (int i = threadIdx.x; i < 64 * 16; i += 256) {
            const int cc = i >> 4, q = i & 15;
            const int c = c0 + cc;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (c < C && p0 + 4 * q < hw) v = __ldg(reinterpret_cast<const float4*>(x + ((int64_t)b * C + c) * hw + p0) + q);
            tile[cc][4 * q] = v.x; tile[cc][4 * q + 1] = v.y; tile[cc][4 * q + 2] = v.z; tile[cc][4 * q + 3] = v.w;
        }
    } else {
        for (int i = threadIdx.x; i < 64 * 64; i += 256) {
            const int cc = i >> 6, pp = i & 63;
            const int c = c0 + cc;
            tile[cc][pp] = (c < C && p0 + pp < hw) ? __ldg(x + ((int64_t)b * C + c) * hw + p0 + pp) : 0.0f;
        }
    }
    __syncthreads();
    for (int pp = w; pp < 64; pp += 8) {
        const int64_t p = p0 + pp;
        const int c = c0 + 2 * lane;
        if (p >= hw || c >= C) continue;
        const float v0 = tile[2 * lane][pp], v1 = tile[2 * lane + 1][pp];
        const bf16 h0 = __float2bfloat16_rn(v0), h1 = __float2bfloat16_rn(v1);
        const bf16 l0 = __float2bfloat16_rn(v0 - __bfloat162float(h0)), l1 = __float2bfloat16_rn(v1 - __bfloat162float(h1));
        const int64_t o = ((int64_t)b * hw + p) * c_total + c_off + c;
        *reinterpret_cast<uint32_t*>(hi + o) = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
        *reinterpret_cast<uint32_t*>(lo + o) = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
    }
}

// W [N][k_total] fp32 (row-major), columns [k_off, k_off + K) -> columns [out_off, out_off + K) of hi/lo [N][out_total] bf16
__global__ void __launch_bounds__(256) pack_matrix_split_kernel(bf16* __restrict__ hi, bf16* __restrict__ lo, const float* __restrict__ w,
                                                                int N, int K, int k_total, int k_off, int out_total, int out_off) {
    const int64_t total = (int64_t)N * K;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int n = (int)(i / K), k = (int)(i - (int64_t)n * K);
        const float v = w[(int64_t)n * k_total + k_off + k];
        const bf16 h = __float2bfloat16_rn(v);
        const int64_t o = (int64_t)n * out_total + out_off + k;
        hi[o] = h;
        lo[o] = __float2bfloat16_rn(v - __bfloat162float(h));
    }
}

// scale*W [Cout][Cin][9] fp32 -> hi/lo [9][Cout][Cin] bf16
__global__ void __launch_bounds__(256) pack_weights_kernel(bf16* __restrict__ hi, bf16* __restrict__ lo, const float* __restrict__ w,
                                                           float scale, int cout, int cin) {
    const int64_t total = (int64_t)9 * cout * cin;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int ci = (int)(i % cin);
        const int o = (int)((i / cin) % cout);
        const int t = (int)(i / ((int64_t)cin * cout));
        const float v = __fmul_rn(w[((int64_t)o * cin + ci) * 9 + t], scale);
        const bf16 h = __float2bfloat16_rn(v);
        hi[i] = h;
        lo[i] = __float2bfloat16_rn(v - __bfloat162float(h));
    }
}

// ------------------------------------------------------------------------------------------------- host
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_fn() {
    static PFN_encodeTiled fn = nullptr;
    if (fn) return fn;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) return nullptr;
    fn = (PFN_encodeTiled)p;
    return fn;
}

// fp32 tensor, no swizzle (the blur kernel's input tiles)
static int make_map_f32(CUtensorMap* map, const void* base, int rank, const uint64_t* dims, const uint32_t* box) {
    PFN_encodeTiled enc = get_encode_fn();
    if (!enc) { set_error("cuTensorMapEncodeTiled entry point not available"); return SIS_ERR_CUDA; }
    cuuint64_t gdim[5]; cuuint64_t gstride[4]; cuuint32_t bdim[5]; cuuint32_t estr[5];
    uint64_t stride = 4;
    for (int i = 0; i < rank; ++i) {
        gdim[i] = dims[i]; bdim[i] = box[i]; estr[i] = 1;
        stride *= dims[i];
        if (i < rank - 1) gstride[i] = stride;
    }
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, (cuuint32_t)rank, const_cast<void*>(base), gdim, gstride, bdim, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled (fp32) failed with CUresult %d", (int)r); return SIS_ERR_CUDA; }
    return SIS_OK;
}

static int make_map(CUtensorMap* map, void* base, int rank, const uint64_t* dims, const uint32_t* box, int swizzle_bytes) {
    PFN_encodeTiled enc = get_encode_fn();
    if (!enc) { set_error("cuTensorMapEncodeTiled entry point not available"); return SIS_ERR_CUDA; }
    cuuint64_t gdim[5]; cuuint64_t gstride[4]; cuuint32_t bdim[5]; cuuint32_t estr[5];
    uint64_t stride = 2;
    for (int i = 0; i < rank; ++i) {
        gdim[i] = dims[i]; bdim[i] = box[i]; estr[i] = 1;
        stride *= dims[i];
        if (i < rank - 1) gstride[i] = stride;    // byte stride of dimension i+1
    }
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, base, gdim, gstride, bdim, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed with CUresult %d (rank %d)", (int)r, rank); return SIS_ERR_CUDA; }
    return SIS_OK;
}

typedef CUresult (*PFN_encodeIm2col)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                     const int*, const int*, cuuint32_t, cuuint32_t, const cuuint32_t*, CUtensorMapInterleave,
                                     CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeIm2col get_encode_im2col_fn() {
    static PFN_encodeIm2col fn = nullptr;
    if (fn) return fn;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) return nullptr;
    fn = (PFN_encodeIm2col)p;
    return fn;
}

// NHWC bf16 plane [B][H][W][C] as an im2col tensor map: traversal box [lower, dim-1+upper] in W and H, 128 pixels x
// `channels` per load (corner arrays in W, H order as CUTLASS passes them).
static int make_im2col_map(CUtensorMap* map, void* base, int C, int W, int H, int B, int lower_w, int lower_h, int upper_w, int upper_h,
                           int channels, int swizzle_bytes) {
    PFN_encodeIm2col enc = get_encode_im2col_fn();
    if (!enc) { set_error("cuTensorMapEncodeIm2col entry point not available"); return SIS_ERR_CUDA; }
    const cuuint64_t gdim[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
    const cuuint64_t gstride[3] = {(cuuint64_t)C * 2, (cuuint64_t)C * 2 * W, (cuuint64_t)C * 2 * W * H};
    const int lower[2] = {lower_w, lower_h}, upper[2] = {upper_w, upper_h};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, base, gdim, gstride, lower, upper, (cuuint32_t)channels, (cuuint32_t)BM, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeIm2col failed with CUresult %d", (int)r); return SIS_ERR_CUDA; }
    return SIS_OK;
}

int tc_pack_weights(TcConvWeights& w, const float* d_weight, int cin, int cout, bool up, float scale, cudaStream_t stream) {
    (void)up;
    const size_t bytes = (size_t)9 * cin * cout * sizeof(bf16);
    if (w.cin != cin || w.cout != cout || !w.hi) {
        tc_free_weights(w);
        SIS_CHECK_CUDA(cudaMalloc(&w.hi, bytes));
        SIS_CHECK_CUDA(cudaMalloc(&w.lo, bytes));
        w.cin = cin; w.cout = cout;
    }
    int64_t total = (int64_t)9 * cin * cout;
    int grid = (int)std::min<int64_t>(ceil_div64(total, 256), (int64_t)kNumSMs * 8);
    pack_weights_kernel<<<grid, 256, 0, stream>>>((bf16*)w.hi, (bf16*)w.lo, d_weight, scale, cout, cin);
    SIS_CHECK_LAUNCH();
    return SIS_OK;
}

void tc_free_weights(TcConvWeights& w) {
    if (w.hi) cudaFree(w.hi);
    if (w.lo) cudaFree(w.lo);
    w.hi = w.lo = nullptr; w.cin = w.cout = 0;
}

int tc_ensure_workspace(TcWorkspace& ws, int batch, int size, int c4, const std::map<int, int>& channels) {
    if (ws.batch == batch) return SIS_OK;
    size_t max_elems = (size_t)batch * c4 * 16;
    for (int res = 8; res <= size; res *= 2) max_elems = std::max(max_elems, (size_t)batch * channels.at(res) * res * res);
    const size_t bytes = max_elems * sizeof(bf16);
    if (bytes > ws.a_bytes) {
        for (int i = 0; i < 2; ++i) {
            if (ws.a_hi[i]) cudaFree(ws.a_hi[i]);
            if (ws.a_lo[i]) cudaFree(ws.a_lo[i]);
            ws.a_hi[i] = ws.a_lo[i] = nullptr;
        }
        ws.a_bytes = 0;
        for (int i = 0; i < 2; ++i) {
            SIS_CHECK_CUDA(cudaMalloc(&ws.a_hi[i], bytes));
            SIS_CHECK_CUDA(cudaMalloc(&ws.a_lo[i], bytes));
        }
        ws.a_bytes = bytes;
    }
    if (!ws.d_error) ws.d_error = watchdog_word();
    ws.batch = batch;
    return SIS_OK;
}

void tc_free_workspace(TcWorkspace& ws) {
    for (int i = 0; i < 2; ++i) {
        if (ws.a_hi[i]) cudaFree(ws.a_hi[i]);
        if (ws.a_lo[i]) cudaFree(ws.a_lo[i]);
        ws.a_hi[i] = ws.a_lo[i] = nullptr;
    }
    ws.d_error = nullptr; ws.a_bytes = 0; ws.batch = -1;      // the watchdog word belongs to the library
}

int tc_check_error(TcWorkspace& ws, cudaStream_t stream) {
    // The stream is drained first; a fired watchdog has trapped, so this synchronise fails -- the code is read from
    // the mapped host word either way.
    const cudaError_t sync = cudaStreamSynchronize(stream);
    const unsigned int h = ws.d_error ? *(volatile unsigned int*)ws.d_error : 0u;
    if (h) { set_error("tcgen05 conv watchdog fired: code 0x%x (%s)", h, cudaGetErrorString(sync)); return SIS_ERR_CUDA; }
    if (sync != cudaSuccess) { set_error("cudaStreamSynchronize failed: %s", cudaGetErrorString(sync)); return SIS_ERR_CUDA; }
    return SIS_OK;
}

int tc_prescale_split(TcWorkspace& ws, int slot, const float* x, const float* s, int batch, int c, int h, int w, cudaStream_t stream) {
    const int64_t total = (int64_t)batch * c * h * w;
    SIS_REQUIRE((size_t)total * sizeof(bf16) <= ws.a_bytes, "tc_prescale_split: workspace too small");
    int grid = (int)std::min<int64_t>(ceil_div64(total, 256), (int64_t)kNumSMs * 8);
    prescale_split_kernel<<<grid, 256, 0, stream>>>((bf16*)ws.a_hi[slot], (bf16*)ws.a_lo[slot], x, s, batch, c, (int64_t)h * w);
    SIS_CHECK_LAUNCH();
    return SIS_OK;
}

// Weight pack maps: boxes of {BK channels, `rows` output channels, 1 tap} of the [taps][Cout][Cin] hi / lo packs.
static int make_weight_maps(TcMaps& maps, const void* hi, const void* lo, int cin, int cout, int taps, int BK, int rows) {
    const uint64_t wdims[3] = {(uint64_t)cin, (uint64_t)cout, (uint64_t)taps};
    const uint32_t wbox[3] = {(uint32_t)BK, (uint32_t)rows, 1};
    SIS_PROPAGATE(make_map(&maps.w[0], const_cast<void*>(hi), 3, wdims, wbox, BK * 2));
    SIS_PROPAGATE(make_map(&maps.w[1], const_cast<void*>(lo), 3, wdims, wbox, BK * 2));
    return SIS_OK;
}

// Halo maps of the conv's input planes: boxes of {BK channels, hw x hh pixels, 1 sample}; the out-of-bounds zero fill is
// the conv's padding.
static int make_halo_maps(TcMaps& maps, const TcWorkspace& ws, const TcConvCall& call, int BK, int hw, int hh) {
    const uint64_t adims[4] = {(uint64_t)call.cin, (uint64_t)call.res_in, (uint64_t)call.res_in, (uint64_t)call.batch};
    const uint32_t abox[4] = {(uint32_t)BK, (uint32_t)hw, (uint32_t)hh, 1};
    SIS_PROPAGATE(make_map(&maps.a[0][0], ws.a_hi[call.in_slot], 4, adims, abox, BK * 2));
    SIS_PROPAGATE(make_map(&maps.a[0][1], ws.a_lo[call.in_slot], 4, adims, abox, BK * 2));
    return SIS_OK;
}

// im2col maps of sub-problem i over the conv's input planes: the base pixels of its runs span the traversal box
// [base_d, base_d + extent - 1] = [lower, dim - 1 + upper].
static int make_im2col_maps(TcMaps& maps, int i, const TcSubProblem& s, const TcWorkspace& ws, const TcConvCall& call, int BK) {
    const int H = call.res_in;
    const int lw = s.base_dx, lh = s.base_dy, uw = s.base_dx + s.ow - H, uh = s.base_dy + s.oh - H;
    SIS_PROPAGATE(make_im2col_map(&maps.a[i][0], ws.a_hi[call.in_slot], call.cin, H, H, call.batch, lw, lh, uw, uh, BK, BK * 2));
    SIS_PROPAGATE(make_im2col_map(&maps.a[i][1], ws.a_lo[call.in_slot], call.cin, H, H, call.batch, lw, lh, uw, uh, BK, BK * 2));
    return SIS_OK;
}

// Taps of the plain 3x3 conv: tap t = ky*3 + kx reads the input at offset (ky - 1, kx - 1).
static void set_conv_taps(TcSubProblem& s) {
    s.ntaps = 9;
    for (int ky = 0; ky < 3; ++ky)
        for (int kx = 0; kx < 3; ++kx) { const int t = ky * 3 + kx; s.dy[t] = (short)(ky - 1); s.dx[t] = (short)(kx - 1); s.widx[t] = (signed char)t; }
}

// Appends the taps of output phase (py, px) of the stride-2 transposed conv.  F.conv_transpose2d(stride 2, pad 0),
// model.py:259: out[2i+k] += x[i]*W[k], so phase p = o mod 2 takes the taps ky = py, kx = px (mod 2) at input offset
// (-ky/2, -kx/2), shifted by the sub-problem's origin (y0, x0) when it starts inside the grid (the border strips).
static void add_phase_taps(TcSubProblem& s, int py, int px, int y0 = 0, int x0 = 0) {
    for (int ky = py; ky < 3; ky += 2)
        for (int kx = px; kx < 3; kx += 2) {
            s.dy[s.ntaps] = (short)(y0 - ky / 2); s.dx[s.ntaps] = (short)(x0 - kx / 2);
            s.widx[s.ntaps] = (signed char)(ky * 3 + kx); s.phase[s.ntaps] = (signed char)(py * 2 + px); s.ntaps++;
        }
}

// im2col runs of a per-tap sub-problem: 128 flattened output pixels each; the traversal box starts at the smallest tap offset.
static void set_im2col_runs(TcSubProblem& s, int batch) {
    s.m_tiles = (int)ceil_div64((int64_t)batch * s.oh * s.ow, BM);
    s.base_dy = s.dy[0]; s.base_dx = s.dx[0];
    for (int t = 1; t < s.ntaps; ++t) { s.base_dy = std::min<int>(s.base_dy, s.dy[t]); s.base_dx = std::min<int>(s.base_dx, s.dx[t]); }
}

// Arguments shared by the launches of one conv call.  Plain layers (mode 0) write the capture and the next conv's planes;
// up-convs (mode 1) write the demodulated phases to the fp32 NHWC scratch that the blur pass reads.
static TcKernelArgs conv_args(const TcWorkspace& ws, const TcConvCall& call, int BK) {
    TcKernelArgs a;
    memset(&a, 0, sizeof(a));
    const int H = call.res_in;
    a.batch = call.batch; a.cin = call.cin; a.cout = call.cout; a.kchunks = call.cin / BK; a.b_tiles = call.batch;
    a.demod = call.demod; a.error = ws.d_error;
    if (call.up) {
        a.mode = 1;
        a.out_f32 = call.upconv_tmp; a.out_h = 2 * H + 1; a.out_w = 2 * H + 1;
    } else {
        a.mode = 0; a.act = call.act ? 1 : 0;
        a.noise = call.noise; a.noise_bstride = call.noise_bstride; a.noise_w = call.noise_w; a.bias = call.bias;
        a.out_f32 = call.out_f32; a.out_h = H; a.out_w = H;
        a.s_next = call.s_next; a.next_hi = (bf16*)ws.a_hi[call.out_slot]; a.next_lo = (bf16*)ws.a_lo[call.out_slot];
    }
    return a;
}

// Persistent launch of a GEMM kernel: one CTA (CG = 1) or CTA pair (CG = 2) per SM (pair), at most one per tile;
// a.total_tiles counts tiles resp. pair tiles.
template <auto Kernel, int SMEM_BYTES, int CG = 1>
static int launch_persistent(const TcMaps& maps, const TcKernelArgs& a, cudaStream_t stream) {
    static bool configured = false;
    if (!configured) {
        SIS_CHECK_CUDA(cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
        configured = true;
    }
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(a.total_tiles * CG < kNumSMs ? a.total_tiles * CG : kNumSMs);
    cfg.blockDim = dim3(TC_THREADS); cfg.dynamicSmemBytes = SMEM_BYTES; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CG; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    SIS_CHECK_CUDA(cudaLaunchKernelEx(&cfg, Kernel, maps, a));
    SIS_CHECK_LAUNCH();
    return SIS_OK;
}

// Per-tap kernel by N tile.  CTA pairs are only chosen with BN >= 64 (each CTA's half of the weight tile must be a legal
// UMMA N), so BN = 32 exists for single CTAs only.
template <int BK, int CG>
static int launch_tc(int BN, const TcMaps& maps, const TcKernelArgs& a, cudaStream_t stream) {
    if (BN == 256) return launch_persistent<modconv_tc_kernel<256, BK, CG>, TcCfg<256, BK, CG>::SMEM_BYTES, CG>(maps, a, stream);
    if (BN == 128) return launch_persistent<modconv_tc_kernel<128, BK, CG>, TcCfg<128, BK, CG>::SMEM_BYTES, CG>(maps, a, stream);
    if (BN == 64) return launch_persistent<modconv_tc_kernel<64, BK, CG>, TcCfg<64, BK, CG>::SMEM_BYTES, CG>(maps, a, stream);
    if constexpr (CG == 1) {
        if (BN == 32) return launch_persistent<modconv_tc_kernel<32, BK, 1>, TcCfg<32, BK, 1>::SMEM_BYTES>(maps, a, stream);
    }
    set_error("tc_modconv: no per-tap kernel for BN %d with CG %d", BN, CG);
    return SIS_ERR_UNSUPPORTED;
}

// Halo kernel of the plain conv by N tile and K chunk (32-channel K chunks only for the narrow layers that have them).
template <int CG>
static int launch_tc_halo(int BN, int BK, const TcMaps& maps, const TcKernelArgs& a, cudaStream_t stream) {
    if (BK == 32) {
        if (BN == 64) return launch_persistent<modconv_tc_halo_kernel<64, CG, 32, false>, TcHaloCfg<64, CG, 32, false>::SMEM_BYTES, CG>(maps, a, stream);
        if constexpr (CG == 1) {
            if (BN == 32) return launch_persistent<modconv_tc_halo_kernel<32, 1, 32, false>, TcHaloCfg<32, 1, 32, false>::SMEM_BYTES>(maps, a, stream);
        }
    } else {
        if (BN == 256) return launch_persistent<modconv_tc_halo_kernel<256, CG, 64, false>, TcHaloCfg<256, CG, 64, false>::SMEM_BYTES, CG>(maps, a, stream);
        if (BN == 128) return launch_persistent<modconv_tc_halo_kernel<128, CG, 64, false>, TcHaloCfg<128, CG, 64, false>::SMEM_BYTES, CG>(maps, a, stream);
        if (BN == 64) return launch_persistent<modconv_tc_halo_kernel<64, CG, 64, false>, TcHaloCfg<64, CG, 64, false>::SMEM_BYTES, CG>(maps, a, stream);
        if constexpr (CG == 1) {
            if (BN == 32) return launch_persistent<modconv_tc_halo_kernel<32, 1, 64, false>, TcHaloCfg<32, 1, 64, false>::SMEM_BYTES>(maps, a, stream);
        }
    }
    set_error("tc_modconv: no halo kernel for BN %d, BK %d with CG %d", BN, BK, CG);
    return SIS_ERR_UNSUPPORTED;
}

// 4-phase halo kernel of the transposed conv with Cout <= 64 (BN = Cout; CTA pairs for BN = 64 only)
static int launch_tc_halo_up4(int BN, int BK, int CG, const TcMaps& maps, const TcKernelArgs& a, cudaStream_t stream) {
    if (BN == 64 && CG == 2) {
        if (BK == 64) return launch_persistent<modconv_tc_halo_kernel<64, 2, 64, true>, TcHaloCfg<64, 2, 64, true>::SMEM_BYTES, 2>(maps, a, stream);
        return launch_persistent<modconv_tc_halo_kernel<64, 2, 32, true>, TcHaloCfg<64, 2, 32, true>::SMEM_BYTES, 2>(maps, a, stream);
    }
    if (BN == 64) {
        if (BK == 64) return launch_persistent<modconv_tc_halo_kernel<64, 1, 64, true>, TcHaloCfg<64, 1, 64, true>::SMEM_BYTES>(maps, a, stream);
        return launch_persistent<modconv_tc_halo_kernel<64, 1, 32, true>, TcHaloCfg<64, 1, 32, true>::SMEM_BYTES>(maps, a, stream);
    }
    if (BK == 64) return launch_persistent<modconv_tc_halo_kernel<32, 1, 64, true>, TcHaloCfg<32, 1, 64, true>::SMEM_BYTES>(maps, a, stream);
    return launch_persistent<modconv_tc_halo_kernel<32, 1, 32, true>, TcHaloCfg<32, 1, 32, true>::SMEM_BYTES>(maps, a, stream);
}

// Second half of an up-sampling layer: Blur(4x4, pad 1) + noise + bias + lrelu over the fp32 NHWC scratch.
template <int CB>
static int launch_blur_split(const BlurSplitArgs& bs, bool sep, cudaStream_t stream) {
    using G = BlurGeo<CB>;
    static int blocks_per_sm[2] = {0, 0};                  // by `sep`
    const size_t smem = 2 * (size_t)G::SMEM + 128;         // the ring of two input tiles + alignment
    auto kern = sep ? blur_act_split_kernel<true, CB> : blur_act_split_kernel<false, CB>;
    int& bps = blocks_per_sm[sep ? 1 : 0];
    if (!bps) {
        SIS_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        SIS_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, kern, 256, smem));
        if (bps < 1) bps = 1;
    }
    CUtensorMap in_map;
    memset(&in_map, 0, sizeof(in_map));
    const uint64_t dims[4] = {(uint64_t)bs.C, (uint64_t)bs.IW, (uint64_t)bs.IH, (uint64_t)bs.batch};
    const uint32_t box[4] = {(uint32_t)CB, (uint32_t)G::IW, (uint32_t)BS_IH, 1};
    SIS_PROPAGATE(make_map_f32(&in_map, bs.in, 4, dims, box));
    const int64_t total = (int64_t)bs.batch * ceil_div(bs.OH, BS_TH) * ceil_div(bs.OW, G::TW) * ceil_div(bs.C, CB);
    const int grid = (int)std::min<int64_t>(total, (int64_t)kNumSMs * bps);   // exactly one resident wave
    ProfScope prof(PROF_BLUR_SPLIT, stream);
    kern<<<grid, 256, smem, stream>>>(bs, in_map);
    SIS_CHECK_LAUNCH();
    return SIS_OK;
}

// Second half of an up-sampling layer: Blur(4x4, pad 1) + noise + bias + lrelu over the fp32 NHWC scratch.
static int tc_blur_after_upconv(TcWorkspace& ws, const TcConvCall& call, cudaStream_t stream) {
    const int B = call.batch, H = call.res_in;
    BlurSplitArgs bs;
    bs.in = call.upconv_tmp; bs.IH = 2 * H + 1; bs.IW = 2 * H + 1;
    bs.out_f32 = call.out_f32; bs.OH = call.res_out; bs.OW = call.res_out; bs.C = call.cout; bs.batch = B;
    bs.blur_k = call.blur_k; bs.noise = call.noise; bs.noise_bstride = call.noise_bstride; bs.noise_w = call.noise_w; bs.bias = call.bias;
    bs.s_next = call.s_next; bs.next_hi = (bf16*)ws.a_hi[call.out_slot]; bs.next_lo = (bf16*)ws.a_lo[call.out_slot];
    bs.act = call.act ? 1 : 0;
    SIS_REQUIRE(bs.C % 32 == 0, "tc_modconv: the blur pass needs Cout %% 32 == 0 (got %d)", bs.C);
    // 32-channel blocks when the channel count is an odd multiple of 32 (the 1024^2 layer): no idle lanes
    if (bs.C % 64 != 0 && bs.OW >= 32) return launch_blur_split<32>(bs, call.blur_separable, stream);
    return launch_blur_split<64>(bs, call.blur_separable, stream);
}

int tc_modconv(TcWorkspace& ws, const TcConvWeights& w, const TcConvCall& call, cudaStream_t stream) {
    // layers with Cout <= 64 are timed apart: SURVEY §8(d)'s ridge check reports them against HBM, not the tensor peak
    const int conv_cat = call.cout <= 64 ? PROF_CONV_TC_NARROW : PROF_CONV_TC;
    SIS_REQUIRE(w.hi && w.cin == call.cin && w.cout == call.cout, "tc_modconv: weights not packed for this layer");
    const int B = call.batch, H = call.res_in;
    // transposed halo kernel: Cout = 128 plain layers whose image holds whole 32 x 8 tiles
    if (!call.up && call.cout == 128 && call.cin % HT_BK == 0 && H % HT_TH == 0) {
        TcKernelArgs a = conv_args(ws, call, HT_BK);
        a.nsub = 1;
        TcSubProblem& s = a.sub[0];
        set_conv_taps(s);
        s.oh = H; s.ow = H; s.ostride = 1;
        a.total_tiles = B * (H / HT_TH) * (H / HT_TW);
        TcMaps maps;
        memset(&maps, 0, sizeof(maps));
        SIS_PROPAGATE(make_halo_maps(maps, ws, call, HT_BK, HT_W, HT_H));
        SIS_PROPAGATE(make_weight_maps(maps, w.hi, w.lo, call.cin, call.cout, 9, HT_BK, 128));
        ProfScope prof(conv_cat, stream);
        return launch_persistent<modconv_tc_halo_t_kernel, TcHaloTCfg::SMEM_BYTES>(maps, a, stream);
    }
    // Cout = 128 up-convs: the interior H x H of the four phase grids on the transposed halo kernel (exact 32 x 8 tiles),
    // the one extra row / column of the (H+1)-extent phases as four thin strips on the per-tap kernel
    if (call.up && call.cout == 128 && call.cin % 64 == 0 && H % HT_TH == 0 && H <= 128 /* im2col box corners are 8-bit */) {
        TcKernelArgs a = conv_args(ws, call, HT_BK);
        a.nsub = 4;
        for (int p = 0; p < 4; ++p) {
            TcSubProblem& s = a.sub[p];
            add_phase_taps(s, p >> 1, p & 1);
            s.oh = H; s.ow = H; s.ostride = 2; s.ooff_y = p >> 1; s.ooff_x = p & 1;
        }
        a.total_tiles = B * (H / HT_TH) * (H / HT_TW) * 4;
        TcMaps maps;
        memset(&maps, 0, sizeof(maps));
        SIS_PROPAGATE(make_halo_maps(maps, ws, call, HT_BK, HT_W, HT_H));
        SIS_PROPAGATE(make_weight_maps(maps, w.hi, w.lo, call.cin, call.cout, 9, HT_BK, 128));
        {
            ProfScope prof(conv_cat, stream);
            SIS_PROPAGATE((launch_persistent<modconv_tc_halo_t_kernel, TcHaloTCfg::SMEM_BYTES>(maps, a, stream)));
        }
        // strips: (py=0) row yy = H of phases (0,0) [xx 0..H] and (0,1) [xx 0..H-1]; (px=0) column xx = H of phases
        // (0,0) and (1,0) [yy 0..H-1].  Origins are folded into the tap offsets and the output offsets.
        TcKernelArgs b = conv_args(ws, call, 64);
        b.nsub = 4;
        struct Strip { int py, px, y0, x0, oh, ow; };
        const Strip strips[4] = {{0, 0, H, 0, 1, H + 1}, {0, 1, H, 0, 1, H}, {0, 0, 0, H, H, 1}, {1, 0, 0, H, H, 1}};
        TcMaps mb;
        memset(&mb, 0, sizeof(mb));
        int tiles = 0;
        for (int i = 0; i < 4; ++i) {
            const Strip& sp = strips[i];
            TcSubProblem& s = b.sub[i];
            add_phase_taps(s, sp.py, sp.px, sp.y0, sp.x0);
            s.oh = sp.oh; s.ow = sp.ow; s.ostride = 2; s.ooff_y = 2 * sp.y0 + sp.py; s.ooff_x = 2 * sp.x0 + sp.px;
            set_im2col_runs(s, B);
            s.tile_begin = tiles;
            tiles += s.m_tiles;
            SIS_PROPAGATE(make_im2col_maps(mb, i, s, ws, call, 64));
        }
        b.total_tiles = tiles;
        SIS_PROPAGATE(make_weight_maps(mb, w.hi, w.lo, call.cin, call.cout, 9, 64, 128));
        {
            ProfScope prof(conv_cat, stream);
            SIS_PROPAGATE((launch_tc<64, 1>(128, mb, b, stream)));
        }
        return tc_blur_after_upconv(ws, call, stream);
    }
    // Cout <= 64 up-convs (the 512^2 / 1024^2 models): all four output phases of a spatial tile from ONE halo per K chunk
    if (call.up && (call.cout == 64 || call.cout == 32) && call.cin % 32 == 0 && H >= 8) {
        const int BN = call.cout, BK = call.cin % 64 == 0 ? 64 : 32;
        TcKernelArgs a = conv_args(ws, call, BK);
        a.nsub = 1;
        TcSubProblem& s = a.sub[0];
        for (int p = 0; p < 4; ++p) add_phase_taps(s, p >> 1, p & 1);
        // tiles cover the (H+1)^2 grid of the py = px = 0 phase; the other phases' last row / column is masked in the epilogue
        s.oh = H + 1; s.ow = H + 1; s.ostride = 2;
        s.tiles_y = ceil_div(H + 1, HALO_TH); s.tiles_x = ceil_div(H + 1, HALO_TW);
        const int64_t m_tiles = (int64_t)B * s.tiles_y * s.tiles_x;
        const int CG = (BN == 64 && m_tiles >= 2 * kNumSMs) ? 2 : 1;
        a.total_tiles = (int)ceil_div64(m_tiles, CG);
        TcMaps maps;
        memset(&maps, 0, sizeof(maps));
        SIS_PROPAGATE(make_halo_maps(maps, ws, call, BK, HALO_W, HALO_H));
        SIS_PROPAGATE(make_weight_maps(maps, w.hi, w.lo, call.cin, call.cout, 9, BK, BN / CG));
        {
            ProfScope prof(conv_cat, stream);
            // 64 -> 32: all nine weight tiles stay resident in shared memory
            if (BN == 32 && BK == 64 && a.kchunks == 1)
                SIS_PROPAGATE((launch_persistent<modconv_tc_halo_rw_kernel<32, 64, true>, TcHaloRwCfg<32, 64, true>::SMEM_BYTES>(maps, a, stream)));
            else
                SIS_PROPAGATE(launch_tc_halo_up4(BN, BK, CG, maps, a, stream));
        }
        return tc_blur_after_upconv(ws, call, stream);
    }
    // halo reuse: plain 3x3 layers whose image holds whole 16 x 8 tiles; K chunks of 64 channels (128 B rows), or of 32
    // (64 B rows) for the narrow layers with 32 input channels.  Everything else runs on the per-tap kernel.
    const bool halo = !call.up && H >= HALO_TH && H % HALO_TH == 0 && (call.cin % 64 == 0 || (call.cin % 32 == 0 && call.cout <= 64));
    const int BK = call.cin % 64 == 0 ? 64 : 32;
    SIS_REQUIRE(call.cin % BK == 0, "tc_modconv: Cin must be a multiple of 32 (got %d)", call.cin);
    SIS_REQUIRE(call.cout % 32 == 0, "tc_modconv: Cout must be a multiple of 32 (got %d)", call.cout);
    // N tile: as wide as possible (fewest re-reads of the A tile) while the launch still fills the 148 SMs; the 4x4 and
    // 8x8 layers only have a handful of pixel tiles, so they run narrow N tiles on many CTAs instead of 8 fat ones
    const int64_t m_tiles_all = halo ? (int64_t)B * ceil_div(H, HALO_TH) * ceil_div(H, HALO_TW)
                                     : ceil_div64((int64_t)B * (call.up ? (2 * H + 1) * (2 * H + 1) : H * H), BM);
    int BN = 32;
    for (int cand = 256; cand >= 32; cand /= 2) {
        if (call.cout % cand) continue;
        if (m_tiles_all * (call.cout / cand) >= kNumSMs || cand == 32) { BN = cand; break; }
    }
    if (!call.up && !halo && m_tiles_all * (call.cout / BN) < 4 * kNumSMs) {
        // the 4^2 / 8^2 plain layers have a handful of pixel tiles, and the rule above can land on 1.x waves of narrow
        // tiles.  Pick the N tile by a small cost model instead: waves x per-K-block time, the latter the larger of the
        // MMA time (12 instructions of max(BN/2, (128 + BN)/4) clk: math, or operand fetch from shared memory at
        // 128 B/clk) and the L2 -> SM fill of the stage (A 32 KB + B BN x 256 B at ~60 B/clk/SM).  Measured: 8^2 layer
        // 89 -> 51 us.  (Applied to the plain per-tap kernel only; it mispredicts the halo and the 4-phase layers.)
        double best = 1e30;
        for (int cand = 256; cand >= 32; cand /= 2) {
            if (call.cout % cand) continue;
            const int64_t tiles_c = m_tiles_all * (call.cout / cand);
            const double waves = (double)((tiles_c + kNumSMs - 1) / kNumSMs);
            const double mma = 12.0 * std::max(cand / 2.0, (128.0 + cand) / 4.0);
            const double cost = waves * std::max(mma, (32768.0 + 256.0 * cand) / 60.0);
            if (cost < best) { best = cost; BN = cand; }
        }
    }
    SIS_REQUIRE(call.cout % BN == 0, "tc_modconv: unsupported Cout %d", call.cout);
    const int n_tiles = call.cout / BN;
    // CTA pairs only when there is at least one full wave of pair tiles and each CTA's weight half is a legal UMMA N
    const int CG = (BN >= 64 && m_tiles_all * n_tiles >= 2 * kNumSMs) ? 2 : 1;

    TcKernelArgs a = conv_args(ws, call, BK);
    if (!call.up) {
        a.nsub = 1;
        TcSubProblem& s = a.sub[0];
        set_conv_taps(s);
        s.oh = H; s.ow = H; s.ostride = 1;
        if (halo) {
            s.tiles_y = ceil_div(H, HALO_TH); s.tiles_x = ceil_div(H, HALO_TW);
            a.total_tiles = ceil_div(B * s.tiles_y * s.tiles_x, CG) * n_tiles;
        } else {
            set_im2col_runs(s, B);
            a.total_tiles = ceil_div(s.m_tiles, CG) * n_tiles;
        }
    } else {
        // the 4 phase sub-GEMMs walk the image together (see decode_tile), each padded to the largest one's (pair) tiles
        a.nsub = 4;
        int umax = 0;
        for (int p = 0; p < 4; ++p) {
            TcSubProblem& s = a.sub[p];
            const int py = p >> 1, px = p & 1;
            add_phase_taps(s, py, px);
            s.oh = H + (py == 0 ? 1 : 0); s.ow = H + (px == 0 ? 1 : 0);
            s.ostride = 2; s.ooff_y = py; s.ooff_x = px;
            set_im2col_runs(s, B);
            umax = std::max(umax, ceil_div(s.m_tiles, CG));
        }
        a.interleave_units = umax;
        a.total_tiles = 4 * umax * n_tiles;
    }

    TcMaps maps;
    memset(&maps, 0, sizeof(maps));
    if (halo) SIS_PROPAGATE(make_halo_maps(maps, ws, call, BK, HALO_W, HALO_H));
    else
        for (int i = 0; i < a.nsub; ++i) SIS_PROPAGATE(make_im2col_maps(maps, i, a.sub[i], ws, call, BK));
    SIS_PROPAGATE(make_weight_maps(maps, w.hi, w.lo, call.cin, call.cout, 9, BK, BN / CG));     // CG = 2: each CTA stages half the rows
    {
        ProfScope prof(conv_cat, stream);
        if (halo && BN == 32 && BK == 32 && CG == 1 && a.kchunks == 1 && n_tiles == 1)          // 32 -> 32: resident weights
            SIS_PROPAGATE((launch_persistent<modconv_tc_halo_rw_kernel<32, 32, false>, TcHaloRwCfg<32, 32, false>::SMEM_BYTES>(maps, a, stream)));
        else if (halo)
            SIS_PROPAGATE(CG == 2 ? launch_tc_halo<2>(BN, BK, maps, a, stream) : launch_tc_halo<1>(BN, BK, maps, a, stream));
        else if (CG == 2)
            SIS_PROPAGATE((BK == 64 ? launch_tc<64, 2>(BN, maps, a, stream) : launch_tc<32, 2>(BN, maps, a, stream)));
        else
            SIS_PROPAGATE((BK == 64 ? launch_tc<64, 1>(BN, maps, a, stream) : launch_tc<32, 1>(BN, maps, a, stream)));
    }
    if (call.up) SIS_PROPAGATE(tc_blur_after_upconv(ws, call, stream));
    return SIS_OK;
}

// ------------------------------------------------------------------------------- 1x1 GEMM (DatasetGAN labeller)
int tc_nchw_to_nhwc_split(void* hi, void* lo, const float* x, int batch, int c, int64_t hw, int c_total, int c_off, cudaStream_t stream) {
    SIS_REQUIRE(c % 2 == 0 && c_off % 2 == 0 && c_total % 2 == 0, "nchw_to_nhwc_split: channel counts must be even");
    dim3 grid((unsigned)ceil_div64(hw, 64), (unsigned)ceil_div(c, 64), (unsigned)batch);
    ProfScope prof(PROF_OTHER, stream);
    nchw_to_nhwc_split_kernel<<<grid, 256, 0, stream>>>((bf16*)hi, (bf16*)lo, x, c, hw, c_total, c_off);
    SIS_CHECK_LAUNCH();
    return SIS_OK;
}

int tc_pack_matrix_split(void* hi, void* lo, const float* w, int n, int k, int k_total, int k_off, int out_total, int out_off, cudaStream_t stream) {
    const int64_t total = (int64_t)n * k;
    int grid = (int)std::min<int64_t>(ceil_div64(total, 256), (int64_t)kNumSMs * 8);
    pack_matrix_split_kernel<<<grid, 256, 0, stream>>>((bf16*)hi, (bf16*)lo, w, n, k, k_total, k_off, out_total, out_off);
    SIS_CHECK_LAUNCH();
    return SIS_OK;
}

// out[b, n, y, x] = sum_k W[n, k] * A[b, y, x, k]: the conv GEMM with a single tap and the plain epilogue without
// noise / bias / activation (`ones` [B, cout] stands in for the demodulation factors); fp32 NCHW out, or NHWC
// [B][res][res][cout] with `out_nhwc`.
int tc_conv1x1(const void* a_hi, const void* a_lo, const void* w_hi, const void* w_lo, int batch, int res, int cin, int cout,
               const float* ones, float* out, bool out_nhwc, unsigned int* d_error, cudaStream_t stream) {
    SIS_REQUIRE(cin % 32 == 0, "tc_conv1x1: K must be a multiple of 32 (got %d)", cin);
    SIS_REQUIRE(cout % 32 == 0, "tc_conv1x1: N must be a multiple of 32 (got %d)", cout);
    const int BK = (cin % 64 == 0) ? 64 : 32;
    const int64_t m_tiles = ceil_div64((int64_t)batch * res * res, BM);
    int BN = 32;
    for (int cand = 256; cand >= 32; cand /= 2) {
        if (cout % cand) continue;
        if (m_tiles * (cout / cand) >= kNumSMs || cand == 32) { BN = cand; break; }
    }
    const int n_tiles = cout / BN;
    const int CG = (BN >= 64 && m_tiles * n_tiles >= 2 * kNumSMs) ? 2 : 1;
    TcKernelArgs a;
    memset(&a, 0, sizeof(a));
    a.batch = batch; a.cin = cin; a.cout = cout; a.kchunks = cin / BK;
    a.b_tiles = batch;
    a.demod = ones; a.error = d_error; a.act = 0; a.mode = out_nhwc ? 1 : 0; a.nsub = 1;
    TcSubProblem& s = a.sub[0];
    s.ntaps = 1; s.dy[0] = 0; s.dx[0] = 0; s.widx[0] = 0;
    s.oh = res; s.ow = res; s.ostride = 1; s.ooff_y = 0; s.ooff_x = 0;
    s.m_tiles = (int)m_tiles; s.base_dy = 0; s.base_dx = 0;
    a.total_tiles = ceil_div((int)m_tiles, CG) * n_tiles;
    a.out_f32 = out; a.out_h = res; a.out_w = res;
    TcMaps maps;
    memset(&maps, 0, sizeof(maps));
    SIS_PROPAGATE(make_im2col_map(&maps.a[0][0], const_cast<void*>(a_hi), cin, res, res, batch, 0, 0, 0, 0, BK, BK * 2));
    SIS_PROPAGATE(make_im2col_map(&maps.a[0][1], const_cast<void*>(a_lo), cin, res, res, batch, 0, 0, 0, 0, BK, BK * 2));
    SIS_PROPAGATE(make_weight_maps(maps, w_hi, w_lo, cin, cout, 1, BK, BN / CG));
    ProfScope prof(PROF_CONV_TC, stream);
    if (CG == 2) return (BK == 64) ? launch_tc<64, 2>(BN, maps, a, stream) : launch_tc<32, 2>(BN, maps, a, stream);
    return (BK == 64) ? launch_tc<64, 1>(BN, maps, a, stream) : launch_tc<32, 1>(BN, maps, a, stream);
}

}  // namespace sis
