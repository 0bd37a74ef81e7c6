// K2 -- implicit-GEMM convolution + bias + SiLU (+ residual, + channel-offset write) on the
// 5th-generation tensor cores: tcgen05.mma with the accumulator in TMEM, operands staged in
// shared memory by TMA, one elected lane issuing the MMAs.
//
// Replaces every Conv(+folded BN)+Sigmoid*Mul node onnxruntime executes inside
// `session.run` (reference call sites simple_detector.py:474, :666; _script/gpu_handler.py:165).
//
// GEMM view:  D[M = pixels, N = Cout] = sum over taps (kh,kw) and 64-channel chunks of
//             A_tap[M, 64] * W_tap[N, 64]^T
//   * activations are NHWC bf16.  An M tile is a box of bw x bh pixels of bn images = 128 rows,
//     row m = (y * bn + n) * bw + x.  `mt` (1, 2 or 4) M tiles form one *round*: they share every
//     weight stage (B is fetched once per round, not once per tile), sit side by side in one TMEM
//     accumulator stage and pay the per-round epilogue synchronisation once.
//   * three ways to feed A:
//       generic  one TMA box per (tap, chunk): the same box shifted by the tap offset; the zero
//                padding of the convolution is TMA's out-of-bounds fill.  Stride-2 convs read four
//                "phase" maps (even/odd rows x columns), each again a dense tiled map.
//       halo     3x3 stride-1 convs on 8-pixel-wide tiles: the (bw+2) x (bh+2) halo of a chunk is
//                fetched once and the nine taps are nine MMAs over it, the A descriptor starting at
//                halo row kh*bn*(bw+2) + kw with (bw+2) rows between 8-row groups.  A traffic /6.
//       stem     the 4-channel network input (8 B per pixel): one un-swizzled box per tile, read as
//                the no-swizzle K-major layout (space-to-depth for stride 2, pixel pairs for stride 1,
//                see conv_tc_stem2_kernel); weights stay resident.
//   * weights are pre-packed [Cout][kh][kw][Cin_pad] (K contiguous), fetched by 2-D TMA loads.
//   * operands are K-major SWIZZLE_128B; a short last chunk is zero-filled by TMA and its unused
//     K=16 sub-steps are skipped.
//   * epilogue: tcgen05.ld the fp32 accumulator, + bias (smem), SiLU with one MUFU op, + residual
//     (TMA-loaded into the staging slab), round to bf16 (or keep fp32 for head outputs), write the
//     slab in the TMA swizzle pattern, TMA-store at the channel offset of the destination buffer:
//     Concat / Split never run as ops, partial tiles and padded channels are clipped by TMA.
//
// Kernel shape: persistent, one CTA per SM.  Warps: 0 TMA producer | 1 MMA issuer | 2 TMEM
// allocator | 3 store | 4-11 or 4-15 epilogue (warp % 4 = TMEM lane quarter, two or three warps per
// quarter; the fused depthwise + pointwise kernel: 4-7 epilogue, 8-15 depthwise).  Control loops run
// warp-uniformly and elect one lane around the asynchronous instructions.  Pipelines: smem ring
// (full/empty mbarriers) TMA -> MMA; two TMEM accumulator stages (tmem_full/tmem_empty) MMA ->
// epilogue; one or two staging slabs epilogue -> TMA store.
//
// CTA pairs: the generic and halo kernels have a second form (template argument PAIR = 1) for wide output tiles, in which the
// two CTAs of a cluster compute two M tiles with one stream of cta_group::2 MMAs (M = 256) issued by the leader, each CTA
// loading its own A and half of every weight box.  The forms share their main loops; what differs is written as
// `if constexpr (PAIR)` or as the PAIR form of a PTX wrapper.  RoundSched is the one description of which rounds and tiles
// a CTA computes, used by every role of every kernel.
#include "common.cuh"

#include <cudaTypedefs.h>
#include <stdlib.h>
#include <string.h>
#include <vector>

namespace {

constexpr int kThreads = 512;         // 4 control warps + up to 12 epilogue warps (ConvTcParams::epi_parts per TMEM lane quarter)
constexpr int kTileM = 128;
constexpr int kMaxStages = 9;         // 9: a 3x3 layer with one K chunk keeps all nine weight taps resident (b_res)

// ---- PTX wrappers -----------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive_u32(uint32_t addr) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(addr) : "memory");
}
__device__ __forceinline__ void mbar_wait_u32(uint32_t addr, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred P1;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}" ::"r"(addr), "r"(parity) : "memory");
}
// PAIR = 1 selects the CTA-pair form of an instruction (see cluster_ctarank below): here `addr` is a shared::cluster address
template <int PAIR = 0>
__device__ __forceinline__ void mbar_expect_tx_u32(uint32_t addr, uint32_t bytes) {
    if constexpr (PAIR) asm volatile("mbarrier.arrive.expect_tx.shared::cluster.b64 _, [%0], %1;" ::"r"(addr), "r"(bytes) : "memory");
    else asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(addr), "r"(bytes) : "memory");
}
// one lane of a converged warp (always the same one for a full mask)
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t"
        ".reg .pred P;\n\t"
        "elect.sync _|P, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, P;\n\t"
        "}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// PAIR: `bar` is the leader's barrier (a shared::cluster address), the completion is signalled there
template <int PAIR = 0>
__device__ __forceinline__ void tma_load_4d(const CUtensorMap* map, uint32_t bar, uint32_t dst_smem, int c0, int c1, int c2, int c3) {
    if constexpr (PAIR)
        asm volatile(
            "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(dst_smem),
            "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
            : "memory");
    else
        asm volatile(
            "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(dst_smem),
            "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
            : "memory");
}
template <int PAIR = 0>
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint32_t bar, uint32_t dst_smem, int c0, int c1) {
    if constexpr (PAIR)
        asm volatile(
            "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst_smem),
            "l"(map), "r"(bar), "r"(c0), "r"(c1)
            : "memory");
    else
        asm volatile(
            "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst_smem),
            "l"(map), "r"(bar), "r"(c0), "r"(c1)
            : "memory");
}
// 4-D activation box at channel c, pixel (x, y) of image n: the map's last two dimensions are (image, y) when `perm`
// (tiles spanning several images, see encode_act_map)
template <int PAIR = 0>
__device__ __forceinline__ void tma_load_act(const CUtensorMap* map, uint32_t bar, uint32_t dst_smem, int c, int x, int y, int n, bool perm) {
    tma_load_4d<PAIR>(map, bar, dst_smem, c, x, perm ? n : y, perm ? y : n);
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, uint32_t src_smem, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(map), "r"(src_smem),
                 "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

template <int PAIR = 0>
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t cols) {
    if constexpr (PAIR) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
}
template <int PAIR = 0>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    if constexpr (PAIR) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// PAIR: arrives on the barrier at this offset in both CTAs
template <int PAIR = 0>
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    if constexpr (PAIR)
        asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"((uint16_t)3) : "memory");
    else
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, bf16 x bf16 -> fp32 (PAIR: M = 256 over the two CTAs)
template <int PAIR = 0>
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    if constexpr (PAIR)
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
            "}" ::"r"(d_tmem),
            "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
            : "memory");
    else
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
            "}" ::"r"(d_tmem),
            "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
            : "memory");
}
// ---- CTA pairs (cta_group::2): one MMA spans the two SMs of a 2-CTA cluster (M = 256), each CTA holding its own 128 A
// rows and half of the B rows; the leader (cluster rank 0) issues, barriers that gate it live in its smem.
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t mapa_u32(uint32_t smem_addr, uint32_t rank) {   // shared::cta address -> shared::cluster address in CTA `rank`
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ uint4 lds128(uint32_t a) {
    uint4 v;
    asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts128(uint32_t a, uint4 v) {
    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ float4 lds_f4(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ void pair_sync(int q) { asm volatile("bar.sync %0, 64;" ::"r"(q + 1) : "memory"); }

// High word of a K-major SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit
// layout): stride byte offset (distance between 8-row groups) at [32,46), version 1 at [46,48),
// layout SWIZZLE_128B = 2 at [61,64).  The low word is (address >> 4) | LBO(=1, unused) << 16.
__device__ __forceinline__ uint32_t desc_hi(uint32_t sbo_bytes) { return (sbo_bytes >> 4) | (1u << 14) | (2u << 29); }
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr) { return ((saddr & 0x3FFFFu) >> 4) | (1u << 16); }
__device__ __forceinline__ uint64_t desc64(uint32_t hi, uint32_t lo) { return ((uint64_t)hi << 32) | (uint64_t)lo; }
// K-major descriptor WITHOUT swizzle (layout type 0, "interleave"): a core matrix is 8 rows x 16 bytes stored as 128 contiguous
// bytes; LBO = bytes between the two core matrices of one K = 16 step, SBO = bytes between 8-row groups
// (canonical layout ((8,m),(T,2)):((1T,SBO),(1,LBO)) of cute's UMMA::make_umma_desc).
__device__ __forceinline__ uint32_t desc_hi_ns(uint32_t sbo_bytes) { return (sbo_bytes >> 4) | (1u << 14); }
__device__ __forceinline__ uint32_t desc_lo_ns(uint32_t saddr, uint32_t lbo_bytes) { return ((saddr & 0x3FFFFu) >> 4) | ((lbo_bytes >> 4) << 16); }

struct TileCoord { int nt, x0, y0, n0; };
template <int V> struct KConst { static constexpr int value = V; };
// fn(KConst<km>{}) for a runtime count km of K = 16 steps (1-4): the MMA issue loops keep the count a compile-time constant,
// since a per-MMA `k < km` test costs ~13 cycles per MMA on the single issuing thread (tools/ubench/mma_issue.cu, variants 32 / 33)
template <typename Fn>
__device__ __forceinline__ void with_ksteps(int km, Fn&& fn) {
    if (km == 4) fn(KConst<4>{});
    else if (km == 3) fn(KConst<3>{});
    else if (km == 2) fn(KConst<2>{});
    else fn(KConst<1>{});
}

// t -> (nt, x tile, y tile, image group) without hardware division: q = umulhi(t, ceil(2^32 / d)) is exact
// for t * d < 2^32 (tile counts are far below that); the reciprocals are computed on the host.
__device__ __forceinline__ TileCoord decode_tile(const ConvTcParams& p, int t) {
    TileCoord c;
    uint32_t m = (uint32_t)t;
    if (p.n_tiles_n > 1) {
        const uint32_t q = __umulhi(m, p.rcp_nn);
        c.nt = (int)(m - q * (uint32_t)p.n_tiles_n);
        m = q;
    } else {
        c.nt = 0;
    }
    if (p.rev_last >= 0) m = (uint32_t)p.rev_last - m;     // walk the M tiles backwards (see conv_tc_launch)
    const uint32_t qx = p.tiles_x > 1 ? __umulhi(m, p.rcp_tx) : m;
    const uint32_t tx = m - qx * (uint32_t)p.tiles_x;
    const uint32_t qy = p.tiles_y > 1 ? __umulhi(qx, p.rcp_ty) : qx;
    const uint32_t ty = qx - qy * (uint32_t)p.tiles_y;
    c.x0 = (int)tx * p.bw;
    c.y0 = (int)ty * p.bh;
    c.n0 = (int)qy * p.bn;
    return c;
}

// The round schedule of a CTA, shared by every role of every kernel.  A single CTA takes rounds blockIdx.x, + gridDim.x, ...;
// round rd is the mt tiles from rd * mt on (the last round may be short).  A CTA pair (PAIR, mt == 1) takes rounds
// blockIdx.x / 2, + gridDim.x / 2, ...; its round rd is two M tiles of one output-channel tile nt, one per CTA (rank 0 / 1),
// and an odd last M tile is computed (and stored, identically) by both.  Tile index t = m * n_tiles_n + nt as everywhere else.
template <int PAIR>
struct RoundSched {
    const ConvTcParams& p;
    int total, mt, rounds;
    uint32_t rank;                                   // cluster rank of this CTA (PAIR), else 0
    __device__ __forceinline__ RoundSched(const ConvTcParams& p_, int total_tiles) : p(p_), total(total_tiles) {
        if constexpr (PAIR) {
            rank = cluster_ctarank();
            mt = 1;
            rounds = ((total / p.n_tiles_n + 1) >> 1) * p.n_tiles_n;
        } else {
            rank = 0;
            mt = p.mt;
            rounds = (total + mt - 1) / mt;
        }
    }
    // this CTA's first round and the step to its next one
    __device__ __forceinline__ int rd0() const { return PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x; }
    __device__ __forceinline__ int step() const { return PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x; }
    // the first tile of round rd (a pair: this CTA's tile)
    __device__ __forceinline__ int tile0(int rd) const {
        if constexpr (PAIR) {
            const int nn = p.n_tiles_n;
            const int mp = nn == 1 ? rd : (int)__umulhi((uint32_t)rd, p.rcp_nn), nt = rd - mp * nn;
            return min(2 * mp + (int)rank, total / nn - 1) * nn + nt;
        } else {
            return rd * mt;
        }
    }
    // the tiles of round rd this CTA computes
    __device__ __forceinline__ int tiles(int rd) const { return PAIR ? 1 : min(mt, total - rd * mt); }
};

// Debug trace (build with -DB2D_ENABLE_TRACE, run with B2D_TRACE=1): CTA 0 records clock64() at role
// events of its first kTraceTiles rounds.  Compiled out of product builds.
constexpr int kTraceTiles = 24, kTraceEvents = 4, kTraceRoles = 4;   // roles: 0 producer, 1 MMA, 2 epilogue warp 4, 3 = warp 4's cycles per round in: TMEM-load waits, slab / residual waits, epi_unit, fence + hand-off
__device__ __forceinline__ void trace(const ConvTcParams& p, int role, int it, int ev) {
#ifdef B2D_ENABLE_TRACE
    if (p.trace && blockIdx.x == 0 && it < kTraceTiles) p.trace[(role * kTraceTiles + it) * kTraceEvents + ev] = clock64();
#endif
}

// Packed fp32 arithmetic (Blackwell FADD2 / FMUL2 / FFMA2: two fp32 lanes per instruction, each component rounded
// exactly like the scalar op).  The epilogue is bound by the FMA pipe -- a 3-register FFMA issues every other cycle
// per scheduler -- so bias, SiLU and the residual add run on register pairs: about 4 FMA-pipe instructions per output
// element instead of 7, with the same results bit for bit.
__device__ __forceinline__ uint64_t pk2(float lo, float hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ uint64_t pk2u(uint32_t lo, uint32_t hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi));
    return r;
}
__device__ __forceinline__ void upk2(uint64_t v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ void upk2u(uint64_t v, uint32_t& lo, uint32_t& hi) { asm("mov.b64 {%0, %1}, %2;" : "=r"(lo), "=r"(hi) : "l"(v)); }
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ uint64_t sub2(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ uint64_t mul2(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}

// SiLU of two values, v = 2h given as h:  v * sigmoid(v) = h + h * tanh(h).  One MUFU.TANH per element plus one FFMA2 per
// pair; the halving is folded into the bias step (h = 0.5 * acc + 0.5 * bias, exact scaling).  Measured on B200
// (tools/ubench/silu_acc.cu, 4M points in [-16, 16] against double precision): absolute error <= 1.1e-5 everywhere,
// relative error <= 4.3e-6 for v > 0 -- hundreds of times below the bf16 rounding that follows -- at 15.4 outputs/clk/SM
// with eight warps, the MUFU limit, against 7.0 for exp2 + Newton reciprocal and 7.8 for exp2 + rcp
// (tools/ubench/silu_rate.cu).  The epilogue's throughput bounds every short-K layer of the network.
__device__ __forceinline__ uint64_t silu2_h(uint64_t h) {
    float h0, h1, t0, t1;
    upk2(h, h0, h1);
    asm("tanh.approx.f32 %0, %1;" : "=f"(t0) : "f"(h0));
    asm("tanh.approx.f32 %0, %1;" : "=f"(t1) : "f"(h1));
    return fma2(h, pk2(t0, t1), h);
}
// (tanh.approx.f16x2 does not help: sm_100a lowers it to two MUFU.TANH.F16, one per half -- same MUFU count, less accuracy.)
__device__ __forceinline__ void lds_b64x2(uint32_t a, uint64_t& x, uint64_t& y) {
    asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];" : "=l"(x), "=l"(y) : "r"(a));
}
__device__ __forceinline__ void sts_b64x2(uint32_t a, uint64_t x, uint64_t y) {
    asm volatile("st.shared.v2.b64 [%0], {%1, %2};" ::"r"(a), "l"(x), "l"(y) : "memory");
}

// ===================== epilogue (warps 4-11), shared by all kernels =====================
// NC accumulator columns of this thread's row (already in registers) -> staging slab, in three steps so that the
// caller can run two 16-column units side by side (sixteen independent SiLU chains in flight per thread instead of
// eight: with only two epilogue warps per scheduler the dependent FFMA2 / MUFU latencies are otherwise exposed).
// `base` is the swizzled address of the unit's first 16-byte piece; the others are base ^ (j << 4).
// `scale2` = the accumulator scale of the layer in both lanes: 0.5 for SiLU layers (the halving of silu2_h), 1 otherwise,
// times ConvTcParams::acc_scale (1/255 in the stem, whose input is the raw 0..255 pixel value; 1 elsewhere).  fma(acc, 1, b)
// rounds exactly like acc + b.
template <int ACT, int NC>
__device__ __forceinline__ void epi_bias(const uint32_t (&r)[16], uint32_t bias_addr, uint64_t (&v)[8], uint64_t scale2) {
#pragma unroll
    for (int j = 0; j < NC / 4; ++j) {
        uint64_t b0, b1;
        lds_b64x2(bias_addr + 16 * j, b0, b1);          // ACT layers keep 0.5 * bias in shared memory (prologue)
        v[2 * j] = fma2(pk2u(r[4 * j], r[4 * j + 1]), scale2, b0);
        v[2 * j + 1] = fma2(pk2u(r[4 * j + 2], r[4 * j + 3]), scale2, b1);
    }
}
// Split-fp16 storage (B2D_PREC_FP16X2): a value v is kept as hi = fp16(v) and lo = fp16(v - hi), ~22 mantissa bits.  Eight
// channels form one 32-byte group [hi x 8 | lo x 8]; a convolution reads the pair as 16 K positions against the same
// weight twice, so the tensor core computes w * hi + w * lo with exact products and fp32 accumulation.
__device__ __forceinline__ void split2(uint64_t v, uint32_t& hi, uint32_t& lo) {      // two values -> packed hi pair, packed lo pair
    float a, b;
    upk2(v, a, b);
    const __half2 h = __floats2half2_rn(a, b);
    const float2 hf = __half22float2(h);
    const __half2 l = __floats2half2_rn(__fsub_rn(a, hf.x), __fsub_rn(b, hf.y));
    hi = *(const uint32_t*)&h;
    lo = *(const uint32_t*)&l;
}
__device__ __forceinline__ uint64_t join2(uint32_t hi, uint32_t lo) {                  // packed hi pair + packed lo pair -> two fp32 values
    const float2 a = __half22float2(*(const __half2*)&hi), b = __half22float2(*(const __half2*)&lo);
    return pk2(__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y));
}
template <int RES, int F32, int NC>
__device__ __forceinline__ void epi_store(uint64_t (&v)[8], uint32_t base, int f16) {
    if (F32 == 2) {             // split fp16: per 8 columns one 16-byte piece of high parts, then one of low parts
#pragma unroll
        for (int j = 0; j < NC / 8; ++j) {
            const uint32_t a_hi = base ^ (uint32_t)((2 * j) << 4), a_lo = base ^ (uint32_t)((2 * j + 1) << 4);
            if (RES) {
                const uint4 xh = lds128(a_hi), xl = lds128(a_lo);
                v[4 * j] = add2(v[4 * j], join2(xh.x, xl.x));
                v[4 * j + 1] = add2(v[4 * j + 1], join2(xh.y, xl.y));
                v[4 * j + 2] = add2(v[4 * j + 2], join2(xh.z, xl.z));
                v[4 * j + 3] = add2(v[4 * j + 3], join2(xh.w, xl.w));
            }
            uint32_t h[4], l[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) split2(v[4 * j + i], h[i], l[i]);
            sts128(a_hi, make_uint4(h[0], h[1], h[2], h[3]));
            sts128(a_lo, make_uint4(l[0], l[1], l[2], l[3]));
        }
    } else if (F32) {
#pragma unroll
        for (int j = 0; j < NC / 4; ++j) sts_b64x2(base ^ (uint32_t)(j << 4), v[2 * j], v[2 * j + 1]);
    } else {
#pragma unroll
        for (int j = 0; j < NC / 8; ++j) {
            const uint32_t a0 = base ^ (uint32_t)(j << 4);
            if (RES) {
                const uint4 x = lds128(a0);
                const uint32_t w[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    if (f16) {
                        const float2 f = __half22float2(*(const __half2*)&w[i]);
                        v[4 * j + i] = add2(v[4 * j + i], pk2(f.x, f.y));
                    } else {
                        v[4 * j + i] = add2(v[4 * j + i], pk2u(w[i] << 16, w[i] & 0xFFFF0000u));
                    }
                }
            }
            uint32_t w[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                float lo, hi;
                upk2(v[4 * j + i], lo, hi);
                if (f16) {
                    __half2 h = __floats2half2_rn(lo, hi);
                    w[i] = *(uint32_t*)&h;
                } else {
                    __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
                    w[i] = *(uint32_t*)&h;
                }
            }
            sts128(a0, make_uint4(w[0], w[1], w[2], w[3]));
        }
    }
}
template <int ACT, int RES, int F32, int NC = 16>
__device__ __forceinline__ void epi_unit(const uint32_t (&r)[16], uint32_t bias_addr, uint32_t base, int f16, uint64_t scale2) {
    uint64_t v[8];
    epi_bias<ACT, NC>(r, bias_addr, v, scale2);
    if (ACT) {
#pragma unroll
        for (int i = 0; i < NC / 2; ++i) v[i] = silu2_h(v[i]);
    }
    epi_store<RES, F32, NC>(v, base, f16);
}

// The epilogue chunk format: a tile row of `row_bytes` is cut into chunks of 128 / 64 / 32 bytes, one tensor map per width
// (tmO / tmR [0], [1], [2]): full 128-byte chunks first, then at most one 64-byte and one 32-byte chunk.  The planner encodes
// the maps and bounds the chunk count with it, the kernels lay out the staging slabs with it.
struct EpiChunks {
    uint32_t n128, has64, has32;
};
__host__ __device__ __forceinline__ EpiChunks epi_chunks(uint32_t row_bytes) {
    return {row_bytes >> 7, (row_bytes >> 6) & 1u, (row_bytes >> 5) & 1u};
}

// Geometry of the staging slabs, shared by the epilogue warps and the store warp: a tile's slab holds, chunk after chunk
// (epi_chunks), all 128 rows x chunk width.  One TMA store (or residual load) moves a whole chunk of a tile: the box of the
// maps is the M tile itself.
template <int F32>      // 0: 16-bit outputs, 1: fp32 outputs, 2: split fp16 (hi | lo) -- 4 bytes per output column like fp32
struct EpiGeom {
    static constexpr int esize = F32 ? 4 : 2;
    uint32_t row_bytes, tile_bytes, base, n128, has64, has32;
    int nb;
    __device__ __forceinline__ EpiGeom(const ConvTcParams& p, uint8_t* stg_base) {
        row_bytes = (uint32_t)(p.n_tile * esize);
        tile_bytes = 128u * row_bytes;                                          // staging bytes of one M tile
        base = smem_u32(stg_base);                                              // slab 0
        nb = p.stg_bufs;
        const EpiChunks c = epi_chunks(row_bytes);
        n128 = c.n128; has64 = c.has64; has32 = c.has32;
    }
    // TMA boxes of one tile's slab: fn(map index, byte offset in the slab, first column)
    template <typename Fn>
    __device__ __forceinline__ void for_each_chunk(Fn&& fn) const {
        constexpr int cols128 = 128 / esize, cols64 = 64 / esize;
        for (uint32_t k = 0; k < n128; ++k) fn(0, k * 16384u, (int)k * cols128);
        if (has64) fn(1, n128 * 16384u, (int)n128 * cols128);
        if (has32) fn(2, n128 * 16384u + has64 * 8192u, (int)n128 * cols128 + (int)has64 * cols64);
    }
};

// Store warp (warp 3), one elected lane.  The staging area is a ring of S = stg_bufs * mt one-tile slabs.  For every tile, in
// the order the epilogue produces them, the lane waits for the slab to be written by all epilogue warps (sfull), issues one
// TMA store per chunk of the tile, waits until the TMA unit has read the slab, hands it back (sempty) and -- for residual
// layers -- starts the residual loads of the tile that will use this slab next, so they have S tiles of time to land.
// Issuing a TMA instruction costs its thread ~200 cycles; taking that, the slab wait and the residual latency out of the
// epilogue warps' loop is what the layers with epilogue-bound rounds needed.
// (Until round 2 four lanes served one TMEM lane quarter each with quarter-sized boxes: 4 x the TMA instructions, and UTMASTG
// takes uniform registers, so the compiler serialised the four lanes in a loop around every one of them -- ncu showed the
// warp 100 % busy with 62 % of its samples in those loops and the epilogue warps waiting for free slabs on the stem.)
template <int RES, int F32, int PAIR = 0>
__device__ __forceinline__ void store_loop(const ConvTcParams& p, int total_tiles, uint64_t* sfull_bar, uint64_t* sempty_bar,
                                           uint64_t* res_bar, uint8_t* stg_base, int lane) {
    if (!elect_one()) return;
    (void)lane;
    const EpiGeom<F32> g(p, stg_base);
    const int mt = p.mt, n_tile = p.n_tile;
    const int S = g.nb * mt, s_shift = 31 - __clz(S);                          // S is 1, 2, 4 or 8
    const uint32_t sfull_u32 = smem_u32(sfull_bar), sempty_u32 = smem_u32(sempty_bar), rbar_u32 = smem_u32(res_bar);
    const RoundSched<PAIR> rs(p, total_tiles);
    const int rd0 = rs.rd0(), rd_step = rs.step();
    const bool perm = p.perm != 0;
    // TMA boxes of tile t: residual loads into / stores out of slab `slab`
    auto tile_io = [&](int t, int slab, bool load) {
        const TileCoord tc = decode_tile(p, t);
        const int c0 = tc.nt * n_tile, c1 = tc.x0;
        const int c2 = perm ? tc.n0 : tc.y0, c3 = perm ? tc.y0 : tc.n0;
        const uint32_t sa = g.base + (uint32_t)slab * g.tile_bytes;
        if (load) {
            const uint32_t bar = rbar_u32 + (uint32_t)slab * 8u;
            mbar_expect_tx_u32(bar, g.tile_bytes);
            g.for_each_chunk([&](int map, uint32_t off, int col0) { tma_load_4d(&p.tmR[map], bar, sa + off, c0 + col0, c1, c2, c3); });
        } else {
            g.for_each_chunk([&](int map, uint32_t off, int col0) { tma_store_4d(&p.tmO[map], sa + off, c0 + col0, c1, c2, c3); });
        }
    };
    if (RES) {                                                                 // the first S tiles' residuals: every slab is free
        for (int c = 0; c < S; ++c) {
            const int rd = rd0 + (c / mt) * rd_step, m = c % mt;
            if (rd < rs.rounds && m < rs.tiles(rd)) tile_io(rs.tile0(rd) + m, c, true);
        }
    }
    // Layers without a residual keep one store group in flight: tile c's stores are issued before the lane waits for tile c - 1's
    // slab to be read, so the read latency of the TMA unit is not paid once per tile (stem 180 -> 147 us).
    int it = 0;
    int pend_slab = -1, pend_next = -1;                                        // slab whose stores are in flight; residual tile to load into it (or -1)
    auto release = [&](bool last) {
        if (pend_slab < 0) return;
        if (last) tma_store_wait_read0(); else tma_store_wait_read1();      // the TMA unit has read the pending slab
        mbar_arrive_u32(sempty_u32 + (uint32_t)pend_slab * 8u);
        if (RES && pend_next >= 0) tile_io(pend_next, pend_slab, true);
        pend_slab = -1;
    };
    for (int rd = rd0; rd < rs.rounds; rd += rd_step, ++it) {
        const int t0 = rs.tile0(rd), nv = rs.tiles(rd);
        const int rdn = rd + g.nb * rd_step;                                  // the round whose tile m reuses tile m's slab
        const int nvn = rdn < rs.rounds ? rs.tiles(rdn) : 0;
        for (int m = 0; m < nv; ++m) {
            const int c = it * mt + m, slab = c & (S - 1);
            const uint32_t use = (uint32_t)(c >> s_shift);
            mbar_wait_u32(sfull_u32 + (uint32_t)slab * 8u, use & 1u);
            tile_io(t0 + m, slab, false);
            tma_store_commit();
            if (RES || S < 4) {                          // residual layers: the slab's next residual must start loading as early as possible
                pend_slab = slab;                        // (measured: +11 us on the 96-channel residual layers when it waits a tile longer);
                pend_next = (RES && m < nvn) ? rs.tile0(rdn) + m : -1;         // with fewer than four slabs a pending one starves the epilogue (+2-4 us)
                release(true);
            } else {
                release(false);
                pend_slab = slab;
                pend_next = -1;
            }
        }
    }
    release(true);
    tma_store_wait_all();
}

// Eight epilogue warps: warp w serves TMEM lane quarter q = w % 4 (a hardware rule) and, of that quarter's
// 16-column units, the ones with unit % 2 == (w - 4) / 4.  The two warps of a quarter share the quarter's ring of
// one-tile staging slabs; a slab is handed to the store warp and back through the sfull / sempty mbarriers (no named
// barriers, no TMA instruction on this path).  A round's mt tiles are drained back to back as one flat list of work
// items, the TMEM load of the next item always in flight behind the math of the current one.
template <int ACT, int RES, int F32, int PAIR = 0>
__device__ __forceinline__ void epilogue_loop(const ConvTcParams& p, int total_tiles, uint32_t tmem_base, const float* bias_s,
                                              uint64_t* tfull_bar, uint64_t* tempty_bar, uint64_t* sfull_bar, uint64_t* sempty_bar,
                                              uint64_t* res_bar, uint8_t* stg_base, int warp, int lane) {
    const int q = warp & 3;
    const int half = (warp - 4) >> 2;                  // this warp's part of the quarter's column units: 0 .. epi_parts - 1
    const int nparts = p.epi_parts;
    if (half >= nparts) return;                        // a layer with two parts per quarter leaves warps 12-15 idle
    const EpiGeom<F32> g(p, stg_base);
    constexpr int esize = F32 ? 4 : 2;
    const int n_tile = p.n_tile, mt = p.mt;
    const int S = g.nb * mt, s_shift = 31 - __clz(S);
    const uint32_t tile_bytes = g.tile_bytes;
    const uint32_t sfull_u32 = smem_u32(sfull_bar), sempty_u32 = smem_u32(sempty_bar), rbar_u32 = smem_u32(res_bar);
    const uint32_t bias_base = smem_u32(bias_s);
    const uint32_t tfull_u32 = smem_u32(tfull_bar), tempty_u32 = smem_u32(tempty_bar);
    // 16-column units alternate between the two warps of a quarter; an odd last unit is split 8 + 8 so both warps carry
    // the same load (n_tile = 16, 48, 144 would otherwise leave one warp idle for a unit)
    // With three parts (n_tile a multiple of 48) every warp takes the units part, part + 3, ... and nothing is split.
    const int nunits = n_tile >> 4;
    const bool split_last = nparts == 2 && (nunits & 1) != 0;
    const int my_units = nparts == 1 ? nunits : nparts == 3 ? nunits / 3 : split_last ? (nunits - 1) >> 1 : (nunits - half + 1) >> 1;     // full units half, half + nparts, ...
    const int ipt = my_units + (split_last ? 1 : 0);                                    // work items per tile
    // Swizzled slab address of this lane's row (row q * 32 + lane of the tile) for the 16-column unit starting at byte `b` of the row.
    const uint32_t n128 = g.n128, has64 = g.has64;
    const uint32_t trow = (uint32_t)(q * 32 + lane);
    const uint32_t row128 = g.base + trow * 128u, sw128 = (uint32_t)(lane & 7);
    const uint32_t row64 = g.base + n128 * 16384u + trow * 64u, sw64 = (uint32_t)((lane >> 1) & 3);
    const uint32_t row32 = g.base + n128 * 16384u + has64 * 8192u + trow * 32u, sw32 = (uint32_t)((lane >> 2) & 1);
    auto unit_base = [&](uint32_t b) -> uint32_t {
        if (b < (n128 << 7)) return row128 + (b >> 7) * 16384u + ((((b & 127u) >> 4) ^ sw128) << 4);
        const uint32_t rem = b - (n128 << 7);
        if (has64 && rem < 64u) return row64 + (((rem >> 4) ^ sw64) << 4);
        return row32 + ((((rem >> 4) & 1u) ^ sw32) << 4);
    };
    const uint32_t ubytes = 16u * esize;               // bytes of one unit in a row
    // Each path below sets up its own round schedule: kept next to the path's other loop invariants, the single-CTA
    // instantiations compile to the same instructions as when each path spelled the schedule out.
    int it = 0;
    if (my_units <= 2 && !split_last && p.n_tiles_n == 1) {
        // Narrow tiles (n_tile = 32, 48, 64, 96: the stem, the 160^2 stage, the 96-channel 3x3 layers, the head's box branch): a warp
        // owns the same one or two 16-column units of every tile, so the staging addresses and the bias pointers are loop
        // invariants and a tile is one straight-line block -- TMEM loads of the next tile in flight behind the SiLU of this
        // one -- instead of the general path's per-item bookkeeping (~180 instructions per 16 columns at ~7 cycles each).
        const bool two = my_units == 2;
        const uint32_t ub0 = unit_base((uint32_t)half * ubytes), ub1 = two ? unit_base((uint32_t)(half + nparts) * ubytes) : ub0;
        const uint32_t baddr0 = bias_base + (uint32_t)(half * 16) * 4u, baddr1 = baddr0 + (uint32_t)nparts * 64u;
        const RoundSched<PAIR> rs(p, total_tiles);
        const int rd0 = rs.rd0(), rd_step = rs.step();
        const uint32_t tempty_arrive = PAIR ? mapa_u32(tempty_u32, 0) : tempty_u32;
        const int f16 = p.f16;
        const float sc = (ACT ? 0.5f : 1.0f) * p.acc_scale;
        const uint64_t scale2 = pk2(sc, sc);
        const uint32_t col0 = (uint32_t)(half * 16), col1 = col0 + (uint32_t)nparts * 16u;
        for (int rd = rd0; rd < rs.rounds; rd += rd_step, ++it) {
            const int as = it & 1;
            const int nv = rs.tiles(rd);
            if (warp == 4 && lane == 0) trace(p, 2, it, 0);
            mbar_wait_u32(tfull_u32 + as * 8, (uint32_t)((it >> 1) & 1));
            tc_fence_after();
            if (warp == 4 && lane == 0) trace(p, 2, it, 1);
            const uint32_t tq = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * mt * n_tile);
            uint32_t ra[16], rb[16];
            tmem_ld16(tq + col0, ra);
            if (two) tmem_ld16(tq + col1, rb);
#pragma unroll 1
            for (int m = 0; m < nv; ++m) {
                const int c = it * mt + m, slab = c & (S - 1);
                const uint32_t use = (uint32_t)(c >> s_shift);
                mbar_wait_u32(sempty_u32 + (uint32_t)slab * 8u, (use & 1u) ^ 1u);      // the tile's slab is free ...
                if (RES) mbar_wait_u32(rbar_u32 + (uint32_t)slab * 8u, use & 1u);     // ... and its residual has landed in it
                const uint32_t moff = (uint32_t)slab * tile_bytes;
                uint64_t v0[8], v1[8];
                tmem_ld_wait();
                epi_bias<ACT, 16>(ra, baddr0, v0, scale2);
                if (two) epi_bias<ACT, 16>(rb, baddr1, v1, scale2);
                if (m + 1 < nv) {                                                      // next tile's accumulators while this one's SiLU runs
                    tmem_ld16(tq + (uint32_t)((m + 1) * n_tile) + col0, ra);
                    if (two) tmem_ld16(tq + (uint32_t)((m + 1) * n_tile) + col1, rb);
                }
                if (ACT) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) v0[i] = silu2_h(v0[i]);
                }
                epi_store<RES, F32, 16>(v0, ub0 + moff, f16);
                if (two) {
                    if (ACT) {
#pragma unroll
                        for (int i = 0; i < 8; ++i) v1[i] = silu2_h(v1[i]);
                    }
                    epi_store<RES, F32, 16>(v1, ub1 + moff, f16);
                }
                fence_proxy_async();                                                   // generic-proxy slab writes -> visible to the TMA store
                __syncwarp();
                if (lane == 0) mbar_arrive_u32(sfull_u32 + (uint32_t)slab * 8u);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if constexpr (PAIR) mbar_arrive_cluster(tempty_arrive + as * 8);     // the leader's barrier gates the pair's MMAs
                else mbar_arrive_u32(tempty_u32 + as * 8);
            }
            if (warp == 4 && lane == 0) trace(p, 2, it, 2);
        }
        return;
    }
    if (!split_last) {
        // Tile-structured path (everything except the 8 + 8 split of an odd last unit): a warp's 16-column units are the same
        // columns of every tile, a tile is one block of straight-line code per pair of units -- bias step of the pair, TMEM loads
        // of the next pair (of this tile or the next) issued behind it, SiLU + pack + staging stores -- with one slab wait in
        // front and one hand-off behind.  The item-list form below spends ~180 instructions per 16 columns, most of them
        // bookkeeping, and a warp issues about one instruction per six cycles.
        const RoundSched<PAIR> rs(p, total_tiles);
        const int rd0 = rs.rd0(), rd_step = rs.step();
        const uint32_t tempty_arrive = PAIR ? mapa_u32(tempty_u32, 0) : tempty_u32;
        const int f16 = p.f16;
        const float sc = (ACT ? 0.5f : 1.0f) * p.acc_scale;
        const uint64_t scale2 = pk2(sc, sc);
        const uint32_t col0 = (uint32_t)(half * 16), ustep = (uint32_t)nparts * 16u;
        for (int rd = rd0; rd < rs.rounds; rd += rd_step, ++it) {
            const int as = it & 1;
            const int t0 = rs.tile0(rd), nv = rs.tiles(rd);
            if (warp == 4 && lane == 0) trace(p, 2, it, 0);
            mbar_wait_u32(tfull_u32 + as * 8, (uint32_t)((it >> 1) & 1));
            tc_fence_after();
            if (warp == 4 && lane == 0) trace(p, 2, it, 1);
            const int ch_base = p.n_tiles_n > 1 ? (int)((uint32_t)t0 - __umulhi((uint32_t)t0, p.rcp_nn) * (uint32_t)p.n_tiles_n) * n_tile : 0;   // n_tiles_n > 1 implies mt == 1
            const uint32_t baddr = bias_base + (uint32_t)ch_base * 4u + col0 * 4u;
            const uint32_t tq = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * mt * n_tile) + col0;
            uint32_t ra[16], rb[16];
            tmem_ld16(tq, ra);
            if (my_units > 1) tmem_ld16(tq + ustep, rb);
#pragma unroll 1
            for (int m = 0; m < nv; ++m) {
                const int c = it * mt + m, slab = c & (S - 1);
                const uint32_t use = (uint32_t)(c >> s_shift);
                mbar_wait_u32(sempty_u32 + (uint32_t)slab * 8u, (use & 1u) ^ 1u);      // the tile's slab is free ...
                if (RES) mbar_wait_u32(rbar_u32 + (uint32_t)slab * 8u, use & 1u);     // ... and its residual has landed in it
                const uint32_t moff = (uint32_t)slab * tile_bytes;
                const uint32_t tm = tq + (uint32_t)(m * n_tile);
#pragma unroll 1
                for (int u = 0; u < my_units; u += 2) {
                    const bool two = u + 1 < my_units;
                    uint64_t v0[8], v1[8];
                    tmem_ld_wait();
                    epi_bias<ACT, 16>(ra, baddr + (uint32_t)u * ustep * 4u, v0, scale2);
                    if (two) epi_bias<ACT, 16>(rb, baddr + (uint32_t)(u + 1) * ustep * 4u, v1, scale2);
                    {   // the next pair's accumulators while this pair's SiLU runs: same tile, or the first pair of the next tile
                        const bool same = u + 2 < my_units;
                        const uint32_t tn = same ? tm + (uint32_t)(u + 2) * ustep : tm + (uint32_t)n_tile;
                        const int un = same ? u + 2 : 0;
                        if (same || m + 1 < nv) {
                            tmem_ld16(tn, ra);
                            if (un + 1 < my_units) tmem_ld16(tn + ustep, rb);
                        }
                    }
                    if (ACT) {
#pragma unroll
                        for (int i = 0; i < 8; ++i) v0[i] = silu2_h(v0[i]);
                    }
                    epi_store<RES, F32, 16>(v0, unit_base((col0 + (uint32_t)u * ustep) * esize) + moff, f16);
                    if (two) {
                        if (ACT) {
#pragma unroll
                            for (int i = 0; i < 8; ++i) v1[i] = silu2_h(v1[i]);
                        }
                        epi_store<RES, F32, 16>(v1, unit_base((col0 + (uint32_t)(u + 1) * ustep) * esize) + moff, f16);
                    }
                }
                fence_proxy_async();                                                   // generic-proxy slab writes -> visible to the TMA store
                __syncwarp();
                if (lane == 0) mbar_arrive_u32(sfull_u32 + (uint32_t)slab * 8u);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if constexpr (PAIR) mbar_arrive_cluster(tempty_arrive + as * 8);     // the leader's barrier gates the pair's MMAs
                else mbar_arrive_u32(tempty_u32 + as * 8);
            }
            if (warp == 4 && lane == 0) trace(p, 2, it, 2);
        }
        return;
    }
    // Item-list path: the 8 + 8 split of an odd last unit (n_tile 16, 80, 112 ...).
    const RoundSched<PAIR> rs(p, total_tiles);
    const int rd0 = rs.rd0(), rd_step = rs.step();
    const uint32_t tempty_arrive = PAIR ? mapa_u32(tempty_u32, 0) : tempty_u32;
    const int f16 = p.f16;
    const float sc = (ACT ? 0.5f : 1.0f) * p.acc_scale;
    const uint64_t scale2 = pk2(sc, sc);
    const int split_col = (nunits - 1) * 16 + half * 8;
    for (int rd = rd0; rd < rs.rounds; rd += rd_step, ++it) {
        const int as = it & 1;
        const uint32_t aphase = (it >> 1) & 1;
        const int t0 = rs.tile0(rd), nv = rs.tiles(rd);
        if (warp == 4 && lane == 0) trace(p, 2, it, 0);
        mbar_wait_u32(tfull_u32 + as * 8, aphase);
        tc_fence_after();
        if (warp == 4 && lane == 0) trace(p, 2, it, 1);
        const int ch_base = p.n_tiles_n > 1 ? (int)((uint32_t)t0 - __umulhi((uint32_t)t0, p.rcp_nn) * (uint32_t)p.n_tiles_n) * n_tile : 0;   // n_tiles_n > 1 implies mt == 1
        const uint32_t baddr = bias_base + (uint32_t)(ch_base + half * 16) * 4u;
        const uint32_t ustep = (uint32_t)nparts * 16u;                             // columns between this warp's consecutive units
        const uint32_t tq = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * mt * n_tile);
        const int c_base = it * mt;
        auto item_ld = [&](int m, int u, uint32_t (&rb)[16]) {
            if (u < my_units) tmem_ld16(tq + (uint32_t)(m * n_tile + half * 16) + (uint32_t)u * ustep, rb);
            else tmem_ld8(tq + (uint32_t)(m * n_tile + split_col), rb);
        };
#ifdef B2D_ENABLE_TRACE
        long long w_ld = 0, w_slab = 0, w_math = 0, w_hand = 0, w0 = 0;
#define B2D_TICK() (w0 = clock64())
#define B2D_TOCK(acc) (acc += clock64() - w0)
#else
#define B2D_TICK() ((void)0)
#define B2D_TOCK(acc) ((void)0)
#endif
        auto item_do = [&](int m, int u, const uint32_t (&rb)[16]) {
            const int c = c_base + m, slab = c & (S - 1);
            const uint32_t use = (uint32_t)(c >> s_shift);
            if (u == 0) {                                                      // first item of a tile: its slab must be free (and the residual in it)
                B2D_TICK();
                mbar_wait_u32(sempty_u32 + (uint32_t)slab * 8u, (use & 1u) ^ 1u);
                if (RES) mbar_wait_u32(rbar_u32 + (uint32_t)slab * 8u, use & 1u);
                B2D_TOCK(w_slab);
            }
            const uint32_t moff = (uint32_t)slab * tile_bytes;
            B2D_TICK();
            if (u < my_units) epi_unit<ACT, RES, F32, 16>(rb, baddr + (uint32_t)u * ustep * 4u, unit_base((uint32_t)(half + nparts * u) * ubytes) + moff, f16, scale2);
            else epi_unit<ACT, RES, F32, 8>(rb, bias_base + (uint32_t)(ch_base + split_col) * 4u, unit_base((uint32_t)split_col * esize) + moff, f16, scale2);
            B2D_TOCK(w_math);
            if (u == ipt - 1) {                                                // last item: hand the slab to the store warp (one arrival per warp of the quarter)
                B2D_TICK();
                fence_proxy_async();                                           // generic-proxy slab writes -> visible to the TMA store
                __syncwarp();
                if (lane == 0) mbar_arrive_u32(sfull_u32 + (uint32_t)slab * 8u);
                B2D_TOCK(w_hand);
            }
        };
        const int nitems = nv * ipt;
        uint32_t rbuf[2][16];
        int m0 = 0, u0 = 0;
        item_ld(0, 0, rbuf[0]);
#pragma unroll 1
        for (int j = 0; j < nitems; j += 2) {
            int m1 = m0, u1 = u0 + 1;
            if (u1 == ipt) { u1 = 0; ++m1; }
            B2D_TICK();
            tmem_ld_wait();
            B2D_TOCK(w_ld);
            if (j + 1 < nitems) item_ld(m1, u1, rbuf[1]);
            item_do(m0, u0, rbuf[0]);
            if (j + 1 < nitems) {
                int m2 = m1, u2 = u1 + 1;
                if (u2 == ipt) { u2 = 0; ++m2; }
                B2D_TICK();
                tmem_ld_wait();
                B2D_TOCK(w_ld);
                if (j + 2 < nitems) item_ld(m2, u2, rbuf[0]);
                item_do(m1, u1, rbuf[1]);
                m0 = m2; u0 = u2;
            }
        }
        // accumulator stage free: all tcgen05.ld of this round have completed (tcgen05.wait::ld is warp-wide).  ONE lane per
        // warp arrives: 32 arrivals of a warp on one mbarrier are 32 serialised shared-memory atomics (~9 cycles each, measured:
        // with 384 arrivals per round on tempty and 96 per tile and quarter on sfull an empty epilogue still took ~3 500 cycles
        // per round on every layer, profiles/r2_ablation_handoff.txt)
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
            if constexpr (PAIR) mbar_arrive_cluster(tempty_arrive + as * 8);     // the leader's barrier gates the pair's MMAs
            else mbar_arrive_u32(tempty_u32 + as * 8);
        }
        if (warp == 4 && lane == 0) trace(p, 2, it, 2);
#ifdef B2D_ENABLE_TRACE
        if (p.trace && blockIdx.x == 0 && warp == 4 && lane == 0 && it < kTraceTiles) {       // durations, stored relative to the first stamp
            long long* tr = p.trace + (3 * kTraceTiles + it) * kTraceEvents;
            const long long base = p.trace[0] ? p.trace[0] : p.trace[kTraceTiles * kTraceEvents];
            tr[0] = base + w_ld; tr[1] = base + w_slab; tr[2] = base + w_math; tr[3] = base + w_hand;
        }
#endif
    }
#undef B2D_TICK
#undef B2D_TOCK
}

// barrier block shared by all kernels (offsets in 8-byte units from bar_off)
struct Bars {
    uint64_t *full, *empty, *tfull, *tempty, *hfull, *hempty, *afull, *aempty, *res, *sfull, *sempty;   // res / sfull / sempty: one per slab (stg_bufs * mt one-tile slabs); afull / aempty: the fused depthwise + pointwise kernel's A tiles
    uint32_t* tmem_slot;
    float* bias_s;
};
__device__ __forceinline__ Bars carve_bars(uint8_t* smem, const ConvTcParams& p) {
    Bars b;
    b.full = (uint64_t*)(smem + p.bar_off);
    b.empty = b.full + kMaxStages;
    b.tfull = b.empty + kMaxStages;
    b.tempty = b.tfull + 2;
    b.hfull = b.tempty + 2;
    b.hempty = b.hfull + 2;
    b.afull = b.hempty + 2;
    b.aempty = b.afull + 2;
    b.res = b.aempty + 2;
    const int nslab = p.stg_bufs * p.mt;                // one per slab; the residual barriers exist only for residual layers
    b.sfull = b.res + (p.has_res ? nslab : 0);
    b.sempty = b.sfull + nslab;
    b.tmem_slot = (uint32_t*)(((uintptr_t)(b.sempty + nslab) + 15) & ~(uintptr_t)15);   // keeps bias_s 16-byte aligned for any slab count
    b.bias_s = (float*)(b.tmem_slot + 4);
    return b;
}
// common prologue: barrier init (warp 1), TMEM allocation (warp 2), bias to smem (everyone).  In a CTA pair the barriers
// that gate the leader's MMAs (full, hfull, tempty) count the arrivals of both CTAs; the leader's copies are the ones waited on.
template <int PAIR = 0>
__device__ __forceinline__ uint32_t prologue(const ConvTcParams& p, const Bars& b, int warp, int lane, uint32_t issuers = 1,
                                             uint32_t hempty_count = 0, uint32_t afull_count = 0) {
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < p.stages; ++i) {
            mbar_init(&b.full[i], PAIR ? 2 : 1);             // one arrive.expect_tx per CTA
            mbar_init(&b.empty[i], issuers);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&b.tfull[i], issuers);
            mbar_init(&b.tempty[i], (PAIR ? 8 : 4) * p.epi_parts);     // one elected lane of every active epilogue warp
            mbar_init(&b.hfull[i], PAIR ? 2 : 1);
            mbar_init(&b.hempty[i], hempty_count ? hempty_count : issuers);
            if (afull_count) {
                mbar_init(&b.afull[i], afull_count);
                mbar_init(&b.aempty[i], 1);
            }
        }
        for (int i = 0; i < p.stg_bufs * p.mt; ++i) {
            if (p.has_res) mbar_init(&b.res[i], 1);
            mbar_init(&b.sfull[i], 4 * p.epi_parts);          // every active epilogue warp, one arrival each
            mbar_init(&b.sempty[i], 1);
        }
        fence_barrier_init();
    }
    if (warp == 2) tmem_alloc<PAIR>(b.tmem_slot, p.tmem_cols);
    for (int i = threadIdx.x; i < p.n_tile * p.n_tiles_n; i += blockDim.x) b.bias_s[i] = p.act ? 0.5f * p.bias[i] : p.bias[i];   // see epi_bias
    tc_fence_before();
    if constexpr (PAIR) cluster_sync_all();             // barriers of both CTAs initialised before anyone signals them
    else __syncthreads();
    tc_fence_after();
    return *b.tmem_slot;
}
template <int PAIR = 0>
__device__ __forceinline__ void epilogue_exit(const ConvTcParams& p, uint32_t tmem_base, int warp) {
    tc_fence_before();
    if constexpr (PAIR) cluster_sync_all();             // the peer may still signal this CTA's barriers / read its smem until here
    else __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc<PAIR>(tmem_base, p.tmem_cols);
    }
}

// ---------------------------------------------------------------------------------------------
// generic kernel: one A box per (tap, chunk) and tile, one B box per (tap, chunk) and round.
// PAIR (1x1 and stride-2 layers with n_tile >= 128 and a short reduction, see conv_tc_plan): the two CTAs of a cluster run ONE
// stream of cta_group::2 MMAs (M = 256), issued by the leader.  Each CTA loads the A box of its own M tile and HALF of every
// weight box into the same stage slot, so per SM the weight traffic from L2 and the B-operand reads are halved: these layers
// run N = 192 tiles, where a single SM needs ~105 bytes of operands per clock to keep its tensor pipe busy and L2 delivers
// about half of that.  Barriers: full / tempty live in the leader (both CTAs arrive), empty / tfull are signalled in both CTAs
// by the leader's multicast commits.
// ---------------------------------------------------------------------------------------------
template <int ACT, int RES, int F32, int PAIR>
__global__ void __launch_bounds__(kThreads, 1) conv_tc_kernel(const __grid_constant__ ConvTcParams p, int nimg) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const Bars b = carve_bars(smem, p);
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int total_tiles = p.tiles_x * p.tiles_y * ((nimg + p.bn - 1) / p.bn) * p.n_tiles_n;
    const RoundSched<PAIR> rs(p, total_tiles);
    const int mt = rs.mt;
    const int ksteps = p.taps * p.chunks;
    const uint32_t stage_bytes = (uint32_t)mt * p.a_bytes + p.b_bytes;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&p.tmA[0]);
        if (p.stride == 2) {
            tma_prefetch_desc(&p.tmA[1]);
            tma_prefetch_desc(&p.tmA[2]);
            tma_prefetch_desc(&p.tmA[3]);
        }
        tma_prefetch_desc(&p.tmB);
    }
    const uint32_t tmem_base = prologue<PAIR>(p, b, warp, lane);
    const uint32_t smem_base = smem_u32(smem);
    const uint32_t full_u32 = smem_u32(b.full), empty_u32 = smem_u32(b.empty);

    if (warp == 0) {
        // ===================== TMA producer (a pair: in both CTAs) =====================
        int stage = 0;
        uint32_t phase = 0;
        const int pad = p.ksz >> 1;
        const int nstages = p.stages, taps = p.taps, chunks = p.chunks, ksz = p.ksz, n_tile = p.n_tile;
        const int cin_pad = chunks * 64;
        const uint32_t a_bytes = p.a_bytes;
        const bool s2 = (p.stride == 2), perm = p.perm != 0;
        const uint32_t full_bar = PAIR ? mapa_u32(full_u32, 0) : full_u32;     // a pair's loads complete on the leader's barrier
        int pit = 0;
        for (int rd = rs.rd0(); rd < rs.rounds; rd += rs.step(), ++pit) {
            const int t0 = rs.tile0(rd);
            const int nv = rs.tiles(rd);
            const TileCoord tc0 = decode_tile(p, t0);
            const TileCoord tc1 = decode_tile(p, nv > 1 ? t0 + 1 : t0);
            const int bn0 = tc0.nt * n_tile + (PAIR ? (int)rs.rank * (n_tile >> 1) : 0);   // a pair: this CTA's half of the weight rows
            const uint32_t tx_bytes = (uint32_t)nv * p.a_tx_bytes + p.b_tx_bytes;
            int kh = 0, kw = 0;
            trace(p, 0, pit, 0);
            for (int tap = 0; tap < taps; ++tap) {
                const CUtensorMap* mapA = &p.tmA[0];
                int ox = kw - pad, oy = kh - pad;
                if (s2) {
                    // input pixel = 2*o + d, d in {-1,0,1}: odd phase for d = +-1, even for 0
                    const int dy = kh - 1, dx = kw - 1;
                    const int py = dy & 1, px = dx & 1;
                    mapA = &p.tmA[py * 2 + px];
                    ox = (dx - px) / 2;
                    oy = (dy - py) / 2;
                }
                const int kb = tap * cin_pad;
                for (int ch = 0; ch < chunks; ++ch) {
                    mbar_wait_u32(empty_u32 + stage * 8, phase ^ 1);
                    if (elect_one()) {
                        const uint32_t sa = smem_base + (uint32_t)stage * stage_bytes, fb = full_bar + stage * 8;
                        mbar_expect_tx_u32<PAIR>(fb, tx_bytes);
                        {
                            const int cy = tc0.y0 + oy;
                            tma_load_act<PAIR>(mapA, fb, sa, ch * 64, tc0.x0 + ox, cy, tc0.n0, perm);
                        }
                        if (nv > 1) {
                            const int cy = tc1.y0 + oy;
                            tma_load_act(mapA, fb, sa + a_bytes, ch * 64, tc1.x0 + ox, cy, tc1.n0, perm);
                        }
                        tma_load_2d<PAIR>(&p.tmB, fb, sa + (uint32_t)mt * a_bytes, kb + ch * 64, bn0);
                    }
                    if (++stage == nstages) { stage = 0; phase ^= 1; }
                }
                if (++kw == ksz) { kw = 0; ++kh; }
            }
            trace(p, 0, pit, 1);
        }
    } else if (warp == 1 && (!PAIR || rs.rank == 0)) {
        // ===================== MMA issuer (a pair: the leader CTA only) =====================
        // One lane issues; it is elected once, and the loop body is kept to a handful of instructions per MMA: the issue
        // interval of a lone thread (~8 cycles per dependent instruction), not the tensor pipe, bounds narrow layers.
        int stage = 0;
        uint32_t phase = 0;
        int it = 0;
        const bool leader = elect_one();
        const uint32_t hi = desc_hi(1024);
        const uint32_t lo_base = desc_lo(smem_base);
        const uint32_t stage_units = stage_bytes >> 4, a_units = p.a_bytes >> 4;
        const uint32_t idesc = p.idesc;
        const int nstages = p.stages, n_tile = p.n_tile, chunks = p.chunks;
        const int last_kmmas = (p.cin - (chunks - 1) * 64 + 15) >> 4;      // K=16 MMAs that carry data in the last chunk
        const int taps = p.taps;
        const uint32_t tfull_u32 = smem_u32(b.tfull), tempty_u32 = smem_u32(b.tempty);
        for (int rd = rs.rd0(); rd < rs.rounds; rd += rs.step(), ++it) {
            const int as = it & 1;
            const uint32_t aphase = (it >> 1) & 1;
            const bool two = rs.tiles(rd) > 1;
            trace(p, 1, it, 0);
            mbar_wait_u32(tempty_u32 + as * 8, aphase ^ 1);
            tc_fence_after();
            trace(p, 1, it, 1);
            const uint32_t d_tmem = tmem_base + (uint32_t)(as * mt * n_tile);
            // one (tap, chunk) step: KM K=16 MMAs per tile (+32 B each), KM a compile-time constant -- the full chunks run
            // without any per-MMA test, only a tap's last (possibly short, zero-padded) chunk picks its count
            int ks = 0;
            auto step = [&](auto KM) {
                mbar_wait_u32(full_u32 + stage * 8, phase);
                tc_fence_after();
                if (ks == 0) trace(p, 1, it, 2);
                if (leader) {
                    const uint32_t a_lo = lo_base + (uint32_t)stage * stage_units;
                    const uint32_t b_lo = a_lo + (uint32_t)mt * a_units;
                    const uint32_t acc0 = (uint32_t)(ks != 0);
#pragma unroll
                    for (int k = 0; k < decltype(KM)::value; ++k)
                        umma_bf16<PAIR>(d_tmem, desc64(hi, a_lo + 2 * k), desc64(hi, b_lo + 2 * k), idesc, k == 0 ? acc0 : 1u);
                    if (two) {
#pragma unroll
                        for (int k = 0; k < decltype(KM)::value; ++k)
                            umma_bf16(d_tmem + (uint32_t)n_tile, desc64(hi, a_lo + a_units + 2 * k), desc64(hi, b_lo + 2 * k), idesc, k == 0 ? acc0 : 1u);
                    }
                    umma_commit<PAIR>(empty_u32 + stage * 8);                 // frees the smem slot (a pair: in both CTAs) when these MMAs retire
                    if (ks == ksteps - 1) umma_commit<PAIR>(tfull_u32 + as * 8);     // accumulators complete
                }
                ++ks;
                if (++stage == nstages) { stage = 0; phase ^= 1; }
            };
            for (int tap = 0; tap < taps; ++tap) {
                for (int ch = 0; ch < chunks - 1; ++ch) step(KConst<4>{});
                with_ksteps(last_kmmas, step);
            }
            trace(p, 1, it, 3);
        }
    } else if (warp == 3) {
        store_loop<RES, F32, PAIR>(p, total_tiles, b.sfull, b.sempty, b.res, smem + p.stg_off, lane);
    } else if (warp >= 4) {
        epilogue_loop<ACT, RES, F32, PAIR>(p, total_tiles, tmem_base, b.bias_s, b.tfull, b.tempty, b.sfull, b.sempty, b.res, smem + p.stg_off, warp, lane);
    }
    epilogue_exit<PAIR>(p, tmem_base, warp);
}

// ---------------------------------------------------------------------------------------------
// halo kernel: 3x3 stride-1 convs on 8-pixel-wide tiles.  Per round and chunk, one halo box per tile
// (double buffered) and nine weight boxes through the stage ring.
// PAIR (wide layers, n_tile >= 128): the two CTAs of a cluster work on two neighbouring M tiles with ONE stream of MMAs
// (cta_group::2, M = 256) issued by the leader.  Each CTA loads its own halo and only half of every weight tile, so per SM the
// weight fill and the B-operand reads are halved and each MMA instruction carries twice the work -- what keeps the tensor pipe
// fed where a single SM's issue rate and smem bandwidth could not.  One tile per CTA and round, weights never resident.
// Barriers: full / hfull / tempty live in the leader (both CTAs arrive), empty / hempty / tfull are signalled in both CTAs by
// the leader's multicast commits.
// ---------------------------------------------------------------------------------------------
template <int ACT, int RES, int F32, int PAIR>
__global__ void __launch_bounds__(kThreads, 1) conv_tc_halo_kernel(const __grid_constant__ ConvTcParams p, int nimg) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const Bars b = carve_bars(smem, p);
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int total_tiles = p.tiles_x * p.tiles_y * ((nimg + p.bn - 1) / p.bn) * p.n_tiles_n;
    const RoundSched<PAIR> rs(p, total_tiles);
    const int mt = rs.mt;

    if (warp == 0 && lane == 0) { tma_prefetch_desc(&p.tmA[0]); tma_prefetch_desc(&p.tmB); }
    const uint32_t tmem_base = prologue<PAIR>(p, b, warp, lane);
    const uint32_t halo_bytes = p.halo_bytes;
    const uint32_t smem_a = smem_u32(smem), smem_b = smem_a + 2u * (uint32_t)mt * halo_bytes;   // [2][mt] halos, then the B ring
    const uint32_t full_u32 = smem_u32(b.full), empty_u32 = smem_u32(b.empty);
    const uint32_t hfull_u32 = smem_u32(b.hfull), hempty_u32 = smem_u32(b.hempty);

    if (warp == 0) {
        // ===================== weight producer: nine boxes per chunk through the stage ring =====================
        int stage = 0;
        uint32_t phase = 0;
        const int nstages = p.stages, chunks = p.chunks, n_tile = p.n_tile;
        const int cin_pad = chunks * 64;
        const uint32_t b_tx = p.b_tx_bytes, b_bytes = p.b_bytes;
        const uint32_t full_bar = PAIR ? mapa_u32(full_u32, 0) : full_u32;     // a pair's loads complete on the leader's barrier
        int pit = 0;
        for (int rd = rs.rd0(); rd < rs.rounds; rd += rs.step(), ++pit) {
            if (!PAIR && p.b_res && pit > 0) break;      // resident weights: the ring holds every (chunk, tap) and is filled once
            // a pair (one output-channel tile): this CTA's half of the weight rows
            const int bn0 = PAIR ? (int)rs.rank * (n_tile >> 1) : decode_tile(p, rs.tile0(rd)).nt * n_tile;
            for (int ch = 0; ch < chunks; ++ch) {
                for (int tap = 0; tap < 9; ++tap) {
                    mbar_wait_u32(empty_u32 + stage * 8, phase ^ 1);
                    if (elect_one()) {
                        mbar_expect_tx_u32<PAIR>(full_bar + stage * 8, b_tx);
                        tma_load_2d<PAIR>(&p.tmB, full_bar + stage * 8, smem_b + (uint32_t)stage * b_bytes, tap * cin_pad + ch * 64, bn0);
                    }
                    if (++stage == nstages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 2) {
        // ===================== halo producer (the TMEM allocator warp, idle after the prologue) =====================
        // Its own warp, so the next round's halos are requested the moment a halo buffer frees up instead of queueing
        // behind the weight ring: the MMA warp used to wait ~2000 cycles per round for its first operand.
        int hb = 0;
        uint32_t hphase = 0;
        const int chunks = p.chunks;
        const bool perm = p.perm != 0;
        const uint32_t hfull_bar = PAIR ? mapa_u32(hfull_u32, 0) : hfull_u32;
        int pit = 0;
        for (int rd = rs.rd0(); rd < rs.rounds; rd += rs.step(), ++pit) {
            const int t0 = rs.tile0(rd);
            const int nv = rs.tiles(rd);
            const TileCoord tc0 = decode_tile(p, t0);
            const TileCoord tc1 = decode_tile(p, nv > 1 ? t0 + 1 : t0);
            trace(p, 0, pit, 0);
            for (int ch = 0; ch < chunks; ++ch) {
                mbar_wait_u32(hempty_u32 + hb * 8, hphase ^ 1);
                if (ch == 0) trace(p, 0, pit, 1);
                if (elect_one()) {
                    const uint32_t hbar = hfull_bar + hb * 8, dst = smem_a + (uint32_t)(hb * mt) * halo_bytes;
                    mbar_expect_tx_u32<PAIR>(hbar, (uint32_t)nv * p.a_tx_bytes);
                    tma_load_act<PAIR>(&p.tmA[0], hbar, dst, ch * 64, tc0.x0 - 1, tc0.y0 - 1, tc0.n0, perm);
                    if (nv > 1) tma_load_act(&p.tmA[0], hbar, dst + halo_bytes, ch * 64, tc1.x0 - 1, tc1.y0 - 1, tc1.n0, perm);
                }
                if (++hb == 2) { hb = 0; hphase ^= 1; }
            }
            trace(p, 0, pit, 2);
        }
    } else if (warp == 1 && (!PAIR || rs.rank == 0)) {
        int stage = 0, hb = 0, it = 0;
        uint32_t phase = 0, hphase = 0;
        const bool leader = elect_one();                 // elected once; see conv_tc_kernel for why the loop is this lean
        // B: canonical SW128 K-major, 8-row groups 1024 B apart.  A: 8-row groups one halo row (bw + 2 pixels) apart.
        const uint32_t hi_b = desc_hi(1024), hi_a = desc_hi((uint32_t)p.halo_w * 128u);
        const uint32_t b_units = p.b_bytes >> 4, halo_units = halo_bytes >> 4, kh_units = (p.halo_kh_rows * 128u) >> 4;
        const uint32_t a_lo0 = desc_lo(smem_a), b_lo0 = desc_lo(smem_b);
        const uint32_t idesc = p.idesc;
        const int nstages = p.stages, n_tile = p.n_tile, chunks = p.chunks;
        const int last_kmmas = (p.cin - (chunks - 1) * 64 + 15) >> 4;
        const uint32_t tfull_u32 = smem_u32(b.tfull), tempty_u32 = smem_u32(b.tempty);
        for (int rd = rs.rd0(); rd < rs.rounds; rd += rs.step(), ++it) {
            const int as = it & 1;
            const uint32_t aphase = (it >> 1) & 1;
            const bool two = rs.tiles(rd) > 1;
            const bool b_res = !PAIR && p.b_res != 0, b_wait = !b_res || it == 0;
            trace(p, 1, it, 0);
            mbar_wait_u32(tempty_u32 + as * 8, aphase ^ 1);
            tc_fence_after();
            trace(p, 1, it, 1);
            const uint32_t d_tmem = tmem_base + (uint32_t)(as * mt * n_tile);
            for (int ch = 0; ch < chunks; ++ch) {
                mbar_wait_u32(hfull_u32 + hb * 8, hphase);
                tc_fence_after();
                if (ch == 0) trace(p, 1, it, 2);
                const uint32_t a_lo_h = a_lo0 + (uint32_t)(hb * mt) * halo_units;
                const bool last = ch == chunks - 1;
                const int km = last ? last_kmmas : 4;                        // skip the zero-padded tail of the last chunk
                auto taps = [&](auto KM) {
#pragma unroll
                    for (int tap = 0; tap < 9; ++tap) {
                        if (b_wait) {                    // resident weights: only the first round waits for (and never releases) a stage
                            mbar_wait_u32(full_u32 + stage * 8, phase);
                            tc_fence_after();
                        }
                        if (leader) {
                            const uint32_t b_lo = b_lo0 + (uint32_t)stage * b_units;
                            const uint32_t a_lo = a_lo_h + (uint32_t)(tap / 3) * kh_units + (uint32_t)(tap % 3) * 8u;
                            const uint32_t acc0 = tap == 0 ? (uint32_t)(ch != 0) : 1u;
#pragma unroll
                            for (int k = 0; k < decltype(KM)::value; ++k)
                                umma_bf16<PAIR>(d_tmem, desc64(hi_a, a_lo + 2 * k), desc64(hi_b, b_lo + 2 * k), idesc, k == 0 ? acc0 : 1u);
                            if (two) {
#pragma unroll
                                for (int k = 0; k < decltype(KM)::value; ++k)
                                    umma_bf16(d_tmem + (uint32_t)n_tile, desc64(hi_a, a_lo + halo_units + 2 * k), desc64(hi_b, b_lo + 2 * k), idesc, k == 0 ? acc0 : 1u);
                            }
                            if (!b_res) umma_commit<PAIR>(empty_u32 + stage * 8);
                            if (tap == 8) {
                                umma_commit<PAIR>(hempty_u32 + hb * 8);                   // halo tiles free once their MMAs retire
                                if (last) umma_commit<PAIR>(tfull_u32 + as * 8);
                            }
                        }
                        if (++stage == nstages) { stage = 0; phase ^= 1; }
                    }
                };
                with_ksteps(km, taps);
                if (++hb == 2) { hb = 0; hphase ^= 1; }
            }
            trace(p, 1, it, 3);
        }
    } else if (warp == 3) {
        store_loop<RES, F32, PAIR>(p, total_tiles, b.sfull, b.sempty, b.res, smem + p.stg_off, lane);
    } else if (warp >= 4) {
        epilogue_loop<ACT, RES, F32, PAIR>(p, total_tiles, tmem_base, b.bias_s, b.tfull, b.tempty, b.sfull, b.sempty, b.res, smem + p.stg_off, warp, lane);
    }
    epilogue_exit<PAIR>(p, tmem_base, warp);
}

// ---------------------------------------------------------------------------------------------
// depthwise kernel: 3x3 stride-1 depthwise conv (Ultralytics 8.3.x cls branch) on the tensor cores.
// Channels are cut into groups of 16; for a group the depthwise filter is a dense 16 -> 16 conv whose
// weight matrix per tap is diagonal, i.e. one M128 x N16 x K16 MMA per (tap, group): A = the halo
// tile of the group's 64-channel chunk at K offset 32 B x (group % 4), B = a 16 x 16 diagonal block,
// D = the group's 16 accumulator columns.  15/16 of the multiplies hit zeros, which is irrelevant:
// the tensor pipe is otherwise idle here and the kernel stays bound by its output like every other
// narrow layer, while the CUDA-core version was bound by FMA issue and L2 re-reads.
// Weights: per 64-channel chunk one 18 KB stage = [tap][16 rows][64 k] bf16, SWIZZLE_128B: row n of tap t
// holds the four groups' diagonal entries side by side (k = group * 16 + n), so a group's block is the
// same 16 rows at K offset 32 B x group -- 144 full 128-byte TMA rows instead of 576 32-byte ones.
// ---------------------------------------------------------------------------------------------
// Split-fp16 storage (OUT == 2): a 64-channel storage chunk holds 32 real channels as four [hi x 8 | lo x 8] groups; real
// channels 16 g2 .. 16 g2 + 15 (storage groups 2 g2 and 2 g2 + 1) share one block of 16 accumulator columns, filled by two
// K = 16 MMAs per tap whose B blocks carry the channel's weight at both its hi and its lo position.
template <int ACT, int OUT>
__global__ void __launch_bounds__(kThreads, 1) conv_tc_dw_kernel(const __grid_constant__ ConvTcParams p, int nimg) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const Bars b = carve_bars(smem, p);
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int total_tiles = p.tiles_x * p.tiles_y * ((nimg + p.bn - 1) / p.bn) * p.n_tiles_n;
    const RoundSched<0> rs(p, total_tiles);
    const int mt = rs.mt;

    if (warp == 0 && lane == 0) { tma_prefetch_desc(&p.tmA[0]); tma_prefetch_desc(&p.tmB); }
    const uint32_t tmem_base = prologue(p, b, warp, lane, 2);
    const uint32_t halo_bytes = p.halo_bytes;
    const uint32_t smem_a = smem_u32(smem), smem_b = smem_a + 2u * (uint32_t)mt * halo_bytes;
    const uint32_t full_u32 = smem_u32(b.full), empty_u32 = smem_u32(b.empty);
    const uint32_t hfull_u32 = smem_u32(b.hfull), hempty_u32 = smem_u32(b.hempty);
    const int chunks = p.chunks;                 // 64-channel (storage) chunks per n_tile

    if (warp == 0) {
        int stage = 0, hb = 0;
        uint32_t phase = 0, hphase = 0;
        const int nstages = p.stages;
        const uint32_t b_tx = p.b_tx_bytes, b_bytes = p.b_bytes;
        const bool perm = p.perm != 0;
        int pit = 0;
        for (int rd = rs.rd0(); rd < rs.rounds; rd += rs.step(), ++pit) {
            const int t0 = rs.tile0(rd);
            const int nv = rs.tiles(rd);
            const TileCoord tc0 = decode_tile(p, t0);
            const TileCoord tc1 = decode_tile(p, nv > 1 ? t0 + 1 : t0);
            trace(p, 0, pit, 0);
            for (int ch = 0; ch < chunks; ++ch) {
                const int gch = tc0.nt * chunks + ch;                    // chunk index in the whole channel range
                mbar_wait_u32(empty_u32 + stage * 8, phase ^ 1);
                if (elect_one()) {
                    mbar_expect_tx_u32(full_u32 + stage * 8, b_tx);
                    tma_load_2d(&p.tmB, full_u32 + stage * 8, smem_b + (uint32_t)stage * b_bytes, 0, gch * 144);
                }
                if (++stage == nstages) { stage = 0; phase ^= 1; }
                mbar_wait_u32(hempty_u32 + hb * 8, hphase ^ 1);
                if (elect_one()) {
                    const uint32_t hbar = hfull_u32 + hb * 8, dst = smem_a + (uint32_t)(hb * mt) * halo_bytes;
                    mbar_expect_tx_u32(hbar, (uint32_t)nv * p.a_tx_bytes);
                    tma_load_act(&p.tmA[0], hbar, dst, gch * 64, tc0.x0 - 1, tc0.y0 - 1, tc0.n0, perm);
                    if (nv > 1) tma_load_act(&p.tmA[0], hbar, dst + halo_bytes, gch * 64, tc1.x0 - 1, tc1.y0 - 1, tc1.n0, perm);
                }
                if (++hb == 2) { hb = 0; hphase ^= 1; }
            }
            trace(p, 0, pit, 1);
        }
    } else if (warp == 1 || warp == 2) {
        // Two MMA issuers (warps 1 and 2, the latter idle after allocating TMEM): an N = 16 MMA occupies its issuing
        // thread for ~55 cycles whatever its size, two threads together sustain one per ~39 (tools/ubench/mma_rate.cu).
        // Issuer i takes the 16-channel groups j with j % 2 == i -- disjoint accumulator columns, no ordering between
        // them -- and commits for its own MMAs; empty / hempty / tfull therefore expect two arrivals in this kernel.
        const int isu = warp - 1;
        int stage = 0, hb = 0, it = 0;
        uint32_t phase = 0, hphase = 0;
        const uint32_t hi_b = desc_hi(1024), hi_a = desc_hi((uint32_t)p.halo_w * 128u);
        const uint32_t b_units = p.b_bytes >> 4;
        const uint32_t idesc = p.idesc;                                   // M128 x N16
        const int nstages = p.stages, n_tile = p.n_tile;
        const uint32_t kh_bytes = p.halo_kh_rows * 128u;
        const uint32_t tfull_u32 = smem_u32(b.tfull), tempty_u32 = smem_u32(b.tempty);
        for (int rd = rs.rd0(); rd < rs.rounds; rd += rs.step(), ++it) {
            const int as = it & 1;
            const uint32_t aphase = (it >> 1) & 1;
            const int nv = rs.tiles(rd);
            if (isu == 0) trace(p, 1, it, 0);
            mbar_wait_u32(tempty_u32 + as * 8, aphase ^ 1);
            tc_fence_after();
            if (isu == 0) trace(p, 1, it, 1);
            const uint32_t d_tmem = tmem_base + (uint32_t)(as * mt * n_tile);
            for (int ch = 0; ch < chunks; ++ch) {
                mbar_wait_u32(full_u32 + stage * 8, phase);
                mbar_wait_u32(hfull_u32 + hb * 8, hphase);
                tc_fence_after();
                if (ch == 0 && isu == 0) trace(p, 1, it, 2);
                const uint32_t a_base = smem_a + (uint32_t)(hb * mt) * halo_bytes;
                const int ngroups = min(4, ((OUT == 2 ? 2 * n_tile : n_tile) - ch * 64) >> 4);      // 16-channel (storage) groups in this chunk
                if (elect_one()) {
                    const uint32_t b_lo = desc_lo(smem_b) + (uint32_t)stage * b_units;
                    for (int m = 0; m < nv; ++m) {
#pragma unroll
                        for (int tap = 0; tap < 9; ++tap) {
                            const uint32_t a_lo = desc_lo(a_base + (uint32_t)m * halo_bytes + (uint32_t)(tap / 3) * kh_bytes + (uint32_t)(tap % 3) * 128u);
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                if (OUT == 2) {      // storage groups 2 g2, 2 g2 + 1 -> accumulator block g2 (one issuer per block: the two MMAs are ordered)
                                    if (j < ngroups && ((j >> 1) & 1) == isu)
                                        umma_bf16(d_tmem + (uint32_t)(m * n_tile + ch * 32 + (j >> 1) * 16), desc64(hi_a, a_lo + 2 * j),
                                                  desc64(hi_b, b_lo + (uint32_t)(tap * 128 + 2 * j)), idesc, (uint32_t)(tap != 0 || (j & 1) != 0));
                                } else if (j < ngroups && (j & 1) == isu) {
                                    umma_bf16(d_tmem + (uint32_t)(m * n_tile + ch * 64 + j * 16), desc64(hi_a, a_lo + 2 * j),
                                              desc64(hi_b, b_lo + (uint32_t)(tap * 128 + 2 * j)), idesc, (uint32_t)(tap != 0));
                                }
                            }
                        }
                    }
                    umma_commit(empty_u32 + stage * 8);
                    umma_commit(hempty_u32 + hb * 8);
                    if (ch == chunks - 1) umma_commit(tfull_u32 + as * 8);
                }
                if (++stage == nstages) { stage = 0; phase ^= 1; }
                if (++hb == 2) { hb = 0; hphase ^= 1; }
            }
            if (isu == 0) trace(p, 1, it, 3);
        }
    } else if (warp == 3) {
        store_loop<0, OUT>(p, total_tiles, b.sfull, b.sempty, b.res, smem + p.stg_off, lane);
    } else if (warp >= 4) {
        epilogue_loop<ACT, 0, OUT>(p, total_tiles, tmem_base, b.bias_s, b.tfull, b.tempty, b.sfull, b.sempty, b.res, smem + p.stg_off, warp, lane);
    }
    epilogue_exit(p, tmem_base, warp);
}

// ---------------------------------------------------------------------------------------------
// stride-2 stem kernel (YOLOv8 model.0: 3x3 stride 2 on the 4-channel network input), fed by TMA.
// Seen through a 2 x 2 space-to-depth lens the layer is a 2 x 2 stride-1 convolution over blocks of 2 x 2 input pixels
// with 16 channels each (row phase, column phase, 4 channels): output (i, j) reads input rows 2i-1 .. 2i+1 = block row i-1
// (phase 1 only) and block row i (both phases), the same for columns.  The NHWC4 input needs no repacking for that view: the
// two pixels of a block row phase are 16 contiguous bytes, so a 4-D tensor map (8 pixels-pairs of a row | row phase | block
// row | image) with an UN-swizzled box of (bw+1) x 2 x (bh+1) lands in shared memory as
//     [block row][row phase][block column][16 B]
// which IS the no-swizzle K-major operand layout: eight consecutive block columns = one 8-row x 16-byte core matrix, the
// second core matrix of a K = 16 step (row phase 1) LBO = (bw+1) * 16 bytes further, the next 8-row group (next output row)
// SBO = 2 * LBO further.  The four taps (di, dj) are four descriptor offsets (di * SBO + dj * 16) into the one box: four
// K = 16 MMAs per tile against resident weights whose k index is tap * 16 + row phase * 8 + column phase * 4 + channel, with
// zeros where the 3x3 filter has no entry.  No warp builds operands, so warps 4-15 are free for the epilogue (three per
// TMEM lane quarter when the tile width splits into thirds).  Out-of-image blocks (the zero padding) are TMA's out-of-bounds fill.  The stride-1 stem runs here in its
// pixel-pair form (see conv_tc_plan).
// ---------------------------------------------------------------------------------------------
template <int ACT, int OUT>
__global__ void __launch_bounds__(kThreads, 1) conv_tc_stem2_kernel(const __grid_constant__ ConvTcParams p, int nimg) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const Bars b = carve_bars(smem, p);
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int total_tiles = p.tiles_x * p.tiles_y * nimg;                // bn == 1
    const RoundSched<0> rs(p, total_tiles);
    const int mt = rs.mt;
    const uint32_t tile_bytes = p.a_bytes, stage_bytes = (uint32_t)mt * tile_bytes;
    uint8_t* wres = smem + (size_t)p.stages * stage_bytes;               // resident weights [n_tile][64] 16-bit, SWIZZLE_128B

    if (warp == 0 && lane == 0) tma_prefetch_desc(&p.tmA[0]);
    const bool s1 = p.stride == 1;                                        // pair-pixel form of the stride-1 stem (see conv_tc_plan)
    const int wchunks = s1 ? 2 : 1;
    const uint32_t wchunk_bytes = p.b_bytes / (uint32_t)wchunks;
    {
        const uint4* wg = (const uint4*)p.w_raw;
        const uint32_t wbase = smem_u32(wres);
        const int per_chunk = p.n_tile * 8;
        for (int i = threadIdx.x; i < per_chunk * wchunks; i += kThreads) {
            const int ch = i >= per_chunk ? 1 : 0, r = i - ch * per_chunk, n = r >> 3, j = r & 7;
            sts128(wbase + (uint32_t)ch * wchunk_bytes + (uint32_t)n * 128u + (uint32_t)((j ^ (n & 7)) << 4), __ldg(wg + n * 8 * wchunks + ch * 8 + j));
        }
        fence_proxy_async();
    }
    const uint32_t tmem_base = prologue(p, b, warp, lane);
    const uint32_t smem_base = smem_u32(smem);
    const uint32_t full_u32 = smem_u32(b.full), empty_u32 = smem_u32(b.empty);

    if (warp == 0) {
        // ===================== TMA producer: one box per tile =====================
        int stage = 0, pit = 0;
        uint32_t phase = 0;
        const int nstages = p.stages;
        for (int rd = rs.rd0(); rd < rs.rounds; rd += rs.step(), ++pit) {
            const int t0 = rs.tile0(rd), nv = rs.tiles(rd);
            trace(p, 0, pit, 0);
            mbar_wait_u32(empty_u32 + stage * 8, phase ^ 1);
            if (elect_one()) {
                const uint32_t fb = full_u32 + stage * 8, sa = smem_base + (uint32_t)stage * stage_bytes;
                mbar_expect_tx_u32(fb, (uint32_t)nv * p.a_tx_bytes);
                for (int m = 0; m < nv; ++m) {
                    const TileCoord tc = decode_tile(p, t0 + m);
                    if (s1) tma_load_4d(&p.tmA[0], fb, sa + (uint32_t)m * tile_bytes, (2 * tc.x0 - 2) * 4, tc.y0 - 1, tc.n0, 0);
                    else tma_load_4d(&p.tmA[0], fb, sa + (uint32_t)m * tile_bytes, (tc.x0 - 1) * 8, 0, tc.y0 - 1, tc.n0);
                }
            }
            trace(p, 0, pit, 1);
            if (++stage == nstages) { stage = 0; phase ^= 1; }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer: four taps per tile =====================
        int stage = 0, it = 0;
        uint32_t phase = 0;
        const bool leader = elect_one();
        const uint32_t lbo = s1 ? 16u : (uint32_t)p.halo_w * 16u, sbo = s1 ? (uint32_t)p.halo_w * 8u : 2u * lbo;
        const uint32_t wchunk_units = wchunk_bytes >> 4;
        const uint32_t hi_a = desc_hi_ns(sbo), hi_b = desc_hi(1024);
        const uint32_t b_lo = desc_lo(smem_u32(wres));
        const uint32_t idesc = p.idesc;
        const int nstages = p.stages, n_tile = p.n_tile;
        const uint32_t tfull_u32 = smem_u32(b.tfull), tempty_u32 = smem_u32(b.tempty);
        for (int rd = rs.rd0(); rd < rs.rounds; rd += rs.step(), ++it) {
            const int as = it & 1;
            const int nv = rs.tiles(rd);
            trace(p, 1, it, 0);
            mbar_wait_u32(tempty_u32 + as * 8, ((it >> 1) & 1) ^ 1);
            trace(p, 1, it, 1);
            mbar_wait_u32(full_u32 + stage * 8, phase);
            tc_fence_after();
            trace(p, 1, it, 2);
            if (leader) {
                const uint32_t d_tmem = tmem_base + (uint32_t)(as * mt * n_tile);
                const uint32_t sa = smem_base + (uint32_t)stage * stage_bytes;
                for (int m = 0; m < nv; ++m) {
                    const uint32_t a0 = sa + (uint32_t)m * tile_bytes;
                    if (s1) {            // filter row kh = t >> 1, K half t & 1: input pixels x - 2 .. x + 1 / x + 2 .. x + 5 of box line y + kh
#pragma unroll
                        for (int t = 0; t < 6; ++t)
                            umma_bf16(d_tmem + (uint32_t)(m * n_tile), desc64(hi_a, desc_lo_ns(a0 + (uint32_t)(t >> 1) * sbo + (uint32_t)(t & 1) * 32u, lbo)),
                                      desc64(hi_b, b_lo + (uint32_t)(t >> 2) * wchunk_units + 2 * (t & 3)), idesc, (uint32_t)(t != 0));
                    } else {
#pragma unroll
                        for (int t = 0; t < 4; ++t)
                            umma_bf16(d_tmem + (uint32_t)(m * n_tile), desc64(hi_a, desc_lo_ns(a0 + (uint32_t)(t >> 1) * sbo + (uint32_t)(t & 1) * 16u, lbo)),
                                      desc64(hi_b, b_lo + 2 * t), idesc, (uint32_t)(t != 0));
                    }
                }
                umma_commit(empty_u32 + stage * 8);
                umma_commit(tfull_u32 + as * 8);
            }
            trace(p, 1, it, 3);
            if (++stage == nstages) { stage = 0; phase ^= 1; }
        }
    } else if (warp == 3) {
        store_loop<0, OUT>(p, total_tiles, b.sfull, b.sempty, b.res, smem + p.stg_off, lane);
    } else if (warp >= 4) {
        epilogue_loop<ACT, 0, OUT>(p, total_tiles, tmem_base, b.bias_s, b.tfull, b.tempty, b.sfull, b.sempty, b.res, smem + p.stg_off, warp, lane);
    }
    epilogue_exit(p, tmem_base, warp);
}

// ---------------------------------------------------------------------------------------------
// fused depthwise 3x3 + pointwise 1x1 kernel (Ultralytics 8.3.x cls branch: DWConv(c, c, 3) -> Conv(c, c3, 1), each with
// bias + SiLU).  The depthwise result never leaves the SM: four warps compute it on the CUDA cores straight from the TMA-loaded
// halo tile of a 64-channel chunk -- thread (x, 4 channels) walks the tile's pixel lines with a three-line register window, fp32
// FFMA2 accumulation, bias, SiLU -- round it to the 16-bit storage format exactly where the unfused pair rounds its stored
// intermediate, and write it as the K-major SWIZZLE_128B A operand of the pointwise GEMM, whose weights stream through (or
// stay in) a ring of 64-channel stages.  Per chunk: TMA halo -> depthwise warps -> A tile -> four K = 16 MMAs into the
// tile's accumulator; epilogue and stores are the shared ones.  Against the two separate launches this removes one write and
// one read of the c-channel map (157 MB each at 80 x 80 x 192 x 64 images), the depthwise-as-N=16-MMA kernel that was bound
// by its single issuing thread, and a launch.
// Warps: 0 halo producer | 1 MMA issuer | 2 TMEM allocator, then weight producer | 3 store | 4-7 epilogue (one per TMEM lane
// quarter) | 8-15 depthwise: the depthwise stage is ~1 000 CUDA-core instructions per thread and chunk and a warp issues about one
// instruction every five cycles, so it gets two warps per scheduler.
// ---------------------------------------------------------------------------------------------
template <int F16>
__device__ __forceinline__ void dw_cvt(uint32_t u, uint64_t& out) {      // two packed 16-bit values -> two fp32
    if (F16) {
        const float2 f = __half22float2(*(const __half2*)&u);
        out = pk2(f.x, f.y);
    } else {
        out = pk2u(u << 16, u & 0xFFFF0000u);
    }
}
// the three pixels x .. x + 2 of one halo line, this thread's four channels: six fp32 pairs.  The halo tile is NOT swizzled
// (rows of 64 channels = 128 bytes; the sixteen lanes of a pixel read one whole row, so the plain layout is conflict-free):
// `a` = address of pixel x's four channels, the neighbours are +128 and +256 bytes.
template <int F16>
__device__ __forceinline__ void dw_load_line(uint32_t a, uint64_t (&r)[6]) {
    uint32_t u0, u1, u2, u3, u4, u5;
    asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(u0), "=r"(u1) : "r"(a));
    asm volatile("ld.shared.v2.b32 {%0, %1}, [%2+128];" : "=r"(u2), "=r"(u3) : "r"(a));
    asm volatile("ld.shared.v2.b32 {%0, %1}, [%2+256];" : "=r"(u4), "=r"(u5) : "r"(a));
    dw_cvt<F16>(u0, r[0]); dw_cvt<F16>(u1, r[1]);
    dw_cvt<F16>(u2, r[2]); dw_cvt<F16>(u3, r[3]);
    dw_cvt<F16>(u4, r[4]); dw_cvt<F16>(u5, r[5]);
}
// Two output lines (y, y + 1) of this thread's pixel column and four channels from four input lines.  Twelve independent
// three-FMA chains (2 lines x 2 channel pairs x 3 filter rows), then the sums: one warp per scheduler does this work, so the
// instruction-level parallelism inside a thread is what hides the FMA and MUFU latencies.
template <int F16>
__device__ __forceinline__ uint2 dw_finish(uint64_t a0, uint64_t a1, int act) {
    if (act) { a0 = silu2_h(a0); a1 = silu2_h(a1); }       // weights and bias carry the halving (see silu2_h)
    float x0, x1, x2, x3;
    upk2(a0, x0, x1);
    upk2(a1, x2, x3);
    uint2 o;
    if (F16) {
        const __half2 h0 = __floats2half2_rn(x0, x1), h1 = __floats2half2_rn(x2, x3);
        o.x = *(const uint32_t*)&h0; o.y = *(const uint32_t*)&h1;
    } else {
        const __nv_bfloat162 h0 = __floats2bfloat162_rn(x0, x1), h1 = __floats2bfloat162_rn(x2, x3);
        o.x = *(const uint32_t*)&h0; o.y = *(const uint32_t*)&h1;
    }
    return o;
}
// filter row kh (weights w[6 kh ..]) over the three pixels of one input line: a three-FMA chain per channel pair, started from `c`
__device__ __forceinline__ void dw_row(const uint64_t (&l)[6], const uint64_t (&w)[18], int kh, uint64_t c0, uint64_t c1, uint64_t& r0, uint64_t& r1) {
    r0 = fma2(w[6 * kh], l[0], c0);          r1 = fma2(w[6 * kh + 1], l[1], c1);
    r0 = fma2(w[6 * kh + 2], l[2], r0);      r1 = fma2(w[6 * kh + 3], l[3], r1);
    r0 = fma2(w[6 * kh + 4], l[4], r0);      r1 = fma2(w[6 * kh + 5], l[5], r1);
}
template <int F16>
__device__ __forceinline__ void dw_out2(const uint64_t (&la)[6], const uint64_t (&lb)[6], const uint64_t (&lc)[6], const uint64_t (&ld)[6],
                                        const uint64_t (&w)[18], uint64_t b0, uint64_t b1, int act, uint32_t dst, uint32_t line_bytes) {
    uint64_t p[12];
    dw_row(la, w, 0, b0, b1, p[0], p[1]);          // line y: rows a, b, c
    dw_row(lb, w, 1, 0ull, 0ull, p[2], p[3]);
    dw_row(lc, w, 2, 0ull, 0ull, p[4], p[5]);
    dw_row(lb, w, 0, b0, b1, p[6], p[7]);          // line y + 1: rows b, c, d
    dw_row(lc, w, 1, 0ull, 0ull, p[8], p[9]);
    dw_row(ld, w, 2, 0ull, 0ull, p[10], p[11]);
    const uint2 o0 = dw_finish<F16>(add2(add2(p[0], p[2]), p[4]), add2(add2(p[1], p[3]), p[5]), act);
    const uint2 o1 = dw_finish<F16>(add2(add2(p[6], p[8]), p[10]), add2(add2(p[7], p[9]), p[11]), act);
    asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(dst), "r"(o0.x), "r"(o0.y) : "memory");
    asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(dst + line_bytes), "r"(o1.x), "r"(o1.y) : "memory");
}
// one 64-channel chunk of one tile: halo tile (SWIZZLE_128B rows of 64 channels) -> A tile (128 rows x 64 channels, SWIZZLE_128B).
// Thread (x, 4 channels) walks its pixel column two lines at a time with a four-line register window (no register moves: the
// loop body is two steps with the window halves swapped).  bh is even for every 8-pixel-wide tile (bh * bn = 16).
template <int F16>
__device__ __forceinline__ void dw_chunk(const ConvTcParams& p, uint32_t halo_base, uint32_t a_base, uint32_t w_addr, uint32_t b_addr, int tid) {
    const uint32_t c4 = (uint32_t)(tid & 15);
    const int x = (tid >> 4) & 7;                            // 0 .. 7 (bw == 8)
    const int seg = tid >> 7;                                // 256 threads: each half takes eight of the tile's sixteen pixel lines
    const int bn = p.bn, bh = p.bh, act = p.dw_act;
    const int n_lo = bn >= 2 ? seg * (bn >> 1) : 0, n_hi = bn >= 2 ? n_lo + (bn >> 1) : 1;     // several images: half of them each ...
    const int y_lo = bn >= 2 ? 0 : seg * (bh >> 1), ny = bn >= 2 ? bh : bh >> 1;               // ... one image: half of its lines each
    uint64_t w[18], b0, b1;
#pragma unroll
    for (int t = 0; t < 9; ++t) lds_b64x2(w_addr + (uint32_t)t * 256u + c4 * 16u, w[2 * t], w[2 * t + 1]);
    lds_b64x2(b_addr + c4 * 16u, b0, b1);
    // halo pixel (line l, column x): row l * halo_w + x of 128 bytes; lines y and y + 1 of one image are bn * halo_w rows apart
    const uint32_t hline = (uint32_t)(p.halo_w * 128), hstep = hline * (uint32_t)bn;
    const uint32_t src0 = halo_base + (uint32_t)x * 128u + c4 * 8u;
    // A tile row m = (y * bn + n) * 8 + x: 16-byte piece (c4 >> 1) ^ (m & 7) = (c4 >> 1) ^ x, 8 bytes at (c4 & 1) * 8
    const uint32_t dst0 = a_base + (uint32_t)x * 128u + ((((c4 >> 1) ^ (uint32_t)x)) << 4) + ((c4 & 1u) << 3);
    const uint32_t line_bytes = (uint32_t)bn * 1024u;        // A tile bytes between lines y and y + 1 of one image
    const int steps = ny >> 1;
    for (int n = n_lo; n < n_hi; ++n) {
        uint64_t L[4][6];
        uint32_t src = src0 + (uint32_t)(y_lo * bn + n) * hline;
        uint32_t dst = dst0 + (uint32_t)(y_lo * bn + n) * 1024u;
        dw_load_line<F16>(src, L[0]);
        dw_load_line<F16>(src + hstep, L[1]);
        src += 2u * hstep;
#pragma unroll 1
        for (int st = 0; st < steps; st += 2) {
            dw_load_line<F16>(src, L[2]);
            dw_load_line<F16>(src + hstep, L[3]);
            dw_out2<F16>(L[0], L[1], L[2], L[3], w, b0, b1, act, dst, line_bytes);
            if (st + 1 < steps) {
                dw_load_line<F16>(src + 2u * hstep, L[0]);
                dw_load_line<F16>(src + 3u * hstep, L[1]);
                dw_out2<F16>(L[2], L[3], L[0], L[1], w, b0, b1, act, dst + 2u * line_bytes, line_bytes);
            }
            src += 4u * hstep;
            dst += 4u * line_bytes;
        }
    }
}

template <int ACT, int OUT>
__global__ void __launch_bounds__(kThreads, 1) conv_tc_dwpw_kernel(const __grid_constant__ ConvTcParams p, int nimg) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const Bars b = carve_bars(smem, p);
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int total_tiles = p.tiles_x * p.tiles_y * ((nimg + p.bn - 1) / p.bn);     // mt == 1, one output-channel tile
    const int chunks = p.chunks;
    const uint32_t halo_bytes = p.halo_bytes;
    const uint32_t smem_h = smem_u32(smem), smem_at = smem_h + 2u * halo_bytes, smem_w = smem_at + 2u * p.a_bytes;
    const uint32_t smem_dw = smem_u32(smem + p.dw_off);              // [chunk][tap][64] fp32 weights, then [chunks * 64] fp32 bias

    if (warp == 0 && lane == 0) { tma_prefetch_desc(&p.tmA[0]); tma_prefetch_desc(&p.tmB); }
    {   // depthwise weights and bias -> shared memory (plain loads: they are constants of the plan, not produced by the previous kernel)
        const float4* src = (const float4*)p.dw_w;
        const int n4 = chunks * (9 * 64 + 64) / 4;
        for (int i = threadIdx.x; i < n4; i += kThreads) {
            const float4 v = __ldg(src + i);
            asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(smem_dw + (uint32_t)i * 16u), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
        }
    }
    const uint32_t tmem_base = prologue(p, b, warp, lane, 1, 8, 8);    // hempty / afull: one arrival per depthwise warp
    const uint32_t full_u32 = smem_u32(b.full), empty_u32 = smem_u32(b.empty);
    const uint32_t hfull_u32 = smem_u32(b.hfull), hempty_u32 = smem_u32(b.hempty);
    const uint32_t afull_u32 = smem_u32(b.afull), aempty_u32 = smem_u32(b.aempty);
    const bool perm = p.perm != 0;

    if (warp == 0) {
        // ===================== halo producer =====================
        int hb = 0;
        uint32_t hphase = 0;
        for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
            const TileCoord tc = decode_tile(p, t);
            for (int ch = 0; ch < chunks; ++ch) {
                mbar_wait_u32(hempty_u32 + hb * 8, hphase ^ 1);
                if (elect_one()) {
                    const uint32_t hbar = hfull_u32 + hb * 8;
                    mbar_expect_tx_u32(hbar, p.a_tx_bytes);
                    tma_load_act(&p.tmA[0], hbar, smem_h + (uint32_t)hb * halo_bytes, ch * 64, tc.x0 - 1, tc.y0 - 1, tc.n0, perm);
                }
                if (++hb == 2) { hb = 0; hphase ^= 1; }
            }
        }
    } else if (warp == 2) {
        // ===================== pointwise-weight producer: one [n_tile x 64] box per chunk through the ring =====================
        int stage = 0, it = 0;
        uint32_t phase = 0;
        const int nstages = p.stages;
        for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++it) {
            if (p.b_res && it > 0) break;                // resident: the ring holds every chunk and is filled once
            for (int ch = 0; ch < chunks; ++ch) {
                mbar_wait_u32(empty_u32 + stage * 8, phase ^ 1);
                if (elect_one()) {
                    mbar_expect_tx_u32(full_u32 + stage * 8, p.b_tx_bytes);
                    tma_load_2d(&p.tmB, full_u32 + stage * 8, smem_w + (uint32_t)stage * p.b_bytes, ch * 64, 0);
                }
                if (++stage == nstages) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer: four K = 16 steps per chunk =====================
        int stage = 0, ab = 0, it = 0;
        uint32_t phase = 0, aphase_b = 0;
        const bool leader = elect_one();
        const uint32_t hi = desc_hi(1024);
        const uint32_t a_lo0 = desc_lo(smem_at), b_lo0 = desc_lo(smem_w);
        const uint32_t a_units = p.a_bytes >> 4, b_units = p.b_bytes >> 4;
        const uint32_t idesc = p.idesc;
        const int nstages = p.stages, n_tile = p.n_tile;
        const uint32_t tfull_u32 = smem_u32(b.tfull), tempty_u32 = smem_u32(b.tempty);
        const bool b_res = p.b_res != 0;
        for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++it) {
            const int as = it & 1;
            mbar_wait_u32(tempty_u32 + as * 8, ((it >> 1) & 1) ^ 1);
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + (uint32_t)(as * n_tile);
            for (int ch = 0; ch < chunks; ++ch) {
                if (!b_res || it == 0) mbar_wait_u32(full_u32 + stage * 8, phase);
                mbar_wait_u32(afull_u32 + ab * 8, aphase_b);
                tc_fence_after();
                if (leader) {
                    const uint32_t a_lo = a_lo0 + (uint32_t)ab * a_units, b_lo = b_lo0 + (uint32_t)stage * b_units;
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        umma_bf16(d_tmem, desc64(hi, a_lo + 2 * k), desc64(hi, b_lo + 2 * k), idesc, (uint32_t)((ch | k) != 0));
                    umma_commit(aempty_u32 + ab * 8);
                    if (!b_res) umma_commit(empty_u32 + stage * 8);
                    if (ch == chunks - 1) umma_commit(tfull_u32 + as * 8);
                }
                if (++stage == nstages) { stage = 0; phase ^= 1; }
                if (++ab == 2) { ab = 0; aphase_b ^= 1; }
            }
        }
    } else if (warp == 3) {
        store_loop<0, OUT>(p, total_tiles, b.sfull, b.sempty, b.res, smem + p.stg_off, lane);
    } else if (warp >= 8) {
        // ===================== depthwise warps (8-15) =====================
        const int tid = threadIdx.x - 256;
        int hb = 0, ab = 0;
        uint32_t hphase = 0, aphase_b = 0;
        for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
            for (int ch = 0; ch < chunks; ++ch) {
                mbar_wait_u32(hfull_u32 + hb * 8, hphase);                   // the chunk's halo has landed
                mbar_wait_u32(aempty_u32 + ab * 8, aphase_b ^ 1);            // the MMAs that read this A tile have retired
                const uint32_t hbase = smem_h + (uint32_t)hb * halo_bytes, abase = smem_at + (uint32_t)ab * p.a_bytes;
                const uint32_t w_addr = smem_dw + (uint32_t)ch * (9u * 256u), b_addr = smem_dw + (uint32_t)chunks * (9u * 256u) + (uint32_t)ch * 256u;
                if (p.f16) dw_chunk<1>(p, hbase, abase, w_addr, b_addr, tid);
                else dw_chunk<0>(p, hbase, abase, w_addr, b_addr, tid);
                fence_proxy_async();                                         // generic-proxy A tile writes -> visible to the MMA's reads
                __syncwarp();
                if (lane == 0) {
                    mbar_arrive_u32(afull_u32 + ab * 8);
                    mbar_arrive_u32(hempty_u32 + hb * 8);                    // halo buffer read completely by this warp
                }
                if (++hb == 2) { hb = 0; hphase ^= 1; }
                if (++ab == 2) { ab = 0; aphase_b ^= 1; }
            }
        }
    } else if (warp >= 4) {
        epilogue_loop<ACT, 0, OUT>(p, total_tiles, tmem_base, b.bias_s, b.tfull, b.tempty, b.sfull, b.sempty, b.res, smem + p.stg_off, warp, lane);
    }
    epilogue_exit(p, tmem_base, warp);
}

// ---------------------------------------------------------------------------------------------
// stride-2 halo kernel: 3x3 stride-2 convs with one K chunk (cin <= 64) on 8-pixel-wide one-image tiles, weights resident.
// The generic kernel feeds a stride-2 layer nine shifted boxes per tile -- every input pixel 2.25 times -- plus the nine weight
// boxes of every round, and ncu shows model.1 (48 -> 96 at 160 x 160) pulling 2.6 GB through L2 for 0.31 GB of input: it runs
// at the 11 TB/s the L2 delivers, not at the HBM rate.  Here a tile fetches each of the four even / odd phase maps ONCE as a
// (bw + 1) x (bh + 1) halo box (input row 2 oy + kh - 1 is row oy - 1 or oy of the odd-row phase, row oy of the even one) and
// the nine taps are descriptor offsets into the box of their phase, exactly as in the stride-1 halo kernel; the 9 weight
// boxes are loaded once per CTA.  Operand traffic per tile: 4 x 153 rows instead of 9 x 128 + 9 weight boxes.
// Ring of phase boxes in the order P11, P10, P01, P00 (taps: 4, 2, 2, 1); a slot is released as soon as its taps have retired.
// Warps: 0 phase-box producer | 1 MMA issuer | 2 TMEM allocator, then the one-time weight load | 3 store | 4-15 epilogue.
// ---------------------------------------------------------------------------------------------
template <int ACT, int RES, int F32>
__global__ void __launch_bounds__(kThreads, 1) conv_tc_s2halo_kernel(const __grid_constant__ ConvTcParams p, int nimg) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const Bars b = carve_bars(smem, p);
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int total_tiles = p.tiles_x * p.tiles_y * nimg;            // bn == 1, mt == 1, one output-channel tile
    const int nslots = p.stages;
    const uint32_t box_bytes = p.halo_bytes;
    const uint32_t smem_a = smem_u32(smem), smem_w = smem_a + (uint32_t)nslots * box_bytes;

    if (warp == 0 && lane == 0) {
        for (int i = 0; i < 4; ++i) tma_prefetch_desc(&p.tmA[i]);
        tma_prefetch_desc(&p.tmB);
    }
    const uint32_t tmem_base = prologue(p, b, warp, lane);
    const uint32_t full_u32 = smem_u32(b.full), empty_u32 = smem_u32(b.empty);
    const uint32_t wbar = smem_u32(b.hfull);                          // "weights have landed"

    if (warp == 0) {
        // ===================== phase-box producer =====================
        int slot = 0;
        uint32_t phase = 0;
        for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
            const TileCoord tc = decode_tile(p, t);
#pragma unroll 1
            for (int ph = 0; ph < 4; ++ph) {                          // P11, P10, P01, P00
                mbar_wait_u32(empty_u32 + slot * 8, phase ^ 1);
                if (elect_one()) {
                    const uint32_t fb = full_u32 + slot * 8;
                    mbar_expect_tx_u32(fb, p.a_tx_bytes);
                    tma_load_4d(&p.tmA[3 - ph], fb, smem_a + (uint32_t)slot * box_bytes, 0, tc.x0 - 1, tc.y0 - 1, tc.n0);
                }
                if (++slot == nslots) { slot = 0; phase ^= 1; }
            }
        }
    } else if (warp == 2) {
        // ===================== resident weights: nine boxes, once =====================
        if (elect_one()) {
            mbar_expect_tx_u32(wbar, 9u * p.b_tx_bytes);
            for (int tap = 0; tap < 9; ++tap) tma_load_2d(&p.tmB, wbar, smem_w + (uint32_t)tap * p.b_bytes, tap * 64, 0);
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        int slot = 0, it = 0;
        uint32_t phase = 0;
        const bool leader = elect_one();
        const uint32_t hi_b = desc_hi(1024), hi_a = desc_hi((uint32_t)p.halo_w * 128u);
        const uint32_t a_lo0 = desc_lo(smem_a), b_lo0 = desc_lo(smem_w);
        const uint32_t box_units = box_bytes >> 4, b_units = p.b_bytes >> 4, row_units = ((uint32_t)p.halo_w * 128u) >> 4;
        const uint32_t idesc = p.idesc;
        const int n_tile = p.n_tile;
        const int kmmas = (p.cin + 15) >> 4;
        const uint32_t tfull_u32 = smem_u32(b.tfull), tempty_u32 = smem_u32(b.tempty);
        mbar_wait_u32(wbar, 0);
        for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++it) {
            const int as = it & 1;
            mbar_wait_u32(tempty_u32 + as * 8, ((it >> 1) & 1) ^ 1);
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + (uint32_t)(as * n_tile);
            auto tile = [&](auto KM) {
                bool first = true;
#pragma unroll
                for (int ph = 0; ph < 4; ++ph) {
                    // phase ph = (py, px) = (1,1), (1,0), (0,1), (0,0): filter rows kh with (kh + 1) & 1 == py ... i.e. py = 1: kh in {0, 2}, py = 0: kh = 1
                    const int py = ph < 2 ? 1 : 0, px = (ph & 1) ? 0 : 1;
                    mbar_wait_u32(full_u32 + slot * 8, phase);
                    tc_fence_after();
                    if (leader) {
                        const uint32_t a_box = a_lo0 + (uint32_t)slot * box_units;
#pragma unroll
                        for (int kh = 0; kh < 3; ++kh) {
                            if (((kh + 1) & 1) != py) continue;
#pragma unroll
                            for (int kw = 0; kw < 3; ++kw) {
                                if (((kw + 1) & 1) != px) continue;
                                const uint32_t dy = kh == 0 ? 0u : 1u, dx = kw == 0 ? 0u : 1u;
                                const uint32_t a_lo = a_box + dy * row_units + dx * 8u;
                                const uint32_t b_lo = b_lo0 + (uint32_t)(kh * 3 + kw) * b_units;
#pragma unroll
                                for (int k = 0; k < decltype(KM)::value; ++k)
                                    umma_bf16(d_tmem, desc64(hi_a, a_lo + 2 * k), desc64(hi_b, b_lo + 2 * k), idesc, (first && k == 0) ? 0u : 1u);
                                first = false;
                            }
                        }
                        umma_commit(empty_u32 + slot * 8);
                        if (ph == 3) umma_commit(tfull_u32 + as * 8);
                    }
                    if (++slot == nslots) { slot = 0; phase ^= 1; }
                }
            };
            with_ksteps(kmmas, tile);
        }
    } else if (warp == 3) {
        store_loop<RES, F32>(p, total_tiles, b.sfull, b.sempty, b.res, smem + p.stg_off, lane);
    } else if (warp >= 4) {
        epilogue_loop<ACT, RES, F32>(p, total_tiles, tmem_base, b.bias_s, b.tfull, b.tempty, b.sfull, b.sempty, b.res, smem + p.stg_off, warp, lane);
    }
    epilogue_exit(p, tmem_base, warp);
}

// ---- host side ----------------------------------------------------------------------------
PFN_cuTensorMapEncodeTiled_v12000 get_encode() {
    static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
    if (!fn) {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = (PFN_cuTensorMapEncodeTiled_v12000)ptr;
    }
    return fn;
}

int encode_map(CUtensorMap* map, void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes, const uint32_t* box,
               uint32_t swizzle_bytes, bool f32 = false, CUtensorMapL2promotion promo = CU_TENSOR_MAP_L2_PROMOTION_L2_256B) {
    auto enc = get_encode();
    B2D_CHECK(enc != nullptr, "cuTensorMapEncodeTiled entry point not available");
    cuuint64_t gd[5], gs[4];
    cuuint32_t bx[5], es[5];
    for (int i = 0; i < rank; ++i) { gd[i] = dims[i]; bx[i] = box[i]; es[i] = 1; }
    for (int i = 0; i < rank - 1; ++i) gs[i] = strides_bytes[i];
    CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                          : swizzle_bytes == 64  ? CU_TENSOR_MAP_SWIZZLE_64B
                          : swizzle_bytes == 32  ? CU_TENSOR_MAP_SWIZZLE_32B
                                                 : CU_TENSOR_MAP_SWIZZLE_NONE;
    CUresult r = enc(map, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, rank, base, gd, gs, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                     promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    B2D_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed: CUresult %d (rank %d dims %llu %llu %llu %llu box %u %u %u %u)", (int)r, rank,
              (unsigned long long)dims[0], (unsigned long long)dims[1], (unsigned long long)(rank > 2 ? dims[2] : 0),
              (unsigned long long)(rank > 3 ? dims[3] : 0), box[0], box[1], rank > 2 ? box[2] : 0, rank > 3 ? box[3] : 0);
    return 0;
}

// 4-D activation map over an NHWC slice: dims (C, W, H, N), or (C, W, N, H) when `perm` (tiles spanning several
// images keep an image's rows of one y together, see the header).
int encode_act_map(CUtensorMap* map, void* base, int c, int w, int h, int n, uint64_t pix_bytes, uint64_t row_bytes, uint64_t img_bytes,
                   uint32_t bc, uint32_t bw, uint32_t bh, uint32_t bn, bool perm, uint32_t swizzle, bool f32 = false) {
    // L2 promotion widens every request to an aligned 64/128/256-byte block.  On a dense tensor (the slice is the whole
    // pixel) that is a free prefetch of the neighbouring pixel; on a channel slice of a wider concat buffer it drags in
    // the other producers' channels -- measured 3.3x the algorithmic DRAM reads on the 48-of-192-channel slices.
    const CUtensorMapL2promotion promo = (uint64_t)c * (f32 ? 4u : 2u) == pix_bytes ? CU_TENSOR_MAP_L2_PROMOTION_L2_256B : CU_TENSOR_MAP_L2_PROMOTION_NONE;
    if (perm) {
        uint64_t dims[4] = {(uint64_t)c, (uint64_t)w, (uint64_t)n, (uint64_t)h};
        uint64_t str[3] = {pix_bytes, img_bytes, row_bytes};
        uint32_t box[4] = {bc, bw, bn, bh};
        return encode_map(map, base, 4, dims, str, box, swizzle, f32, promo);
    }
    uint64_t dims[4] = {(uint64_t)c, (uint64_t)w, (uint64_t)h, (uint64_t)n};
    uint64_t str[3] = {pix_bytes, row_bytes, img_bytes};
    uint32_t box[4] = {bc, bw, bh, bn};
    return encode_map(map, base, 4, dims, str, box, swizzle, f32, promo);
}

uint16_t f2h(float f) {
    const __half h = __float2half_rn(f);
    uint16_t u;
    memcpy(&u, &h, 2);
    return u;
}

uint16_t f2bf(float f) {
    uint32_t u;
    memcpy(&u, &f, 4);
    u = (u + 0x7FFFu + ((u >> 16) & 1u)) >> 16;
    return (uint16_t)u;
}

// pick (bw, bh, bn), bw*bh*bn == 128, maximising useful rows; ties -> squarer spatial box, smaller bn
void pick_tile(int W, int H, int N, int* bw, int* bh, int* bn, bool need_w8 = false) {
    double best = -1.0;
    int best_halo = 1 << 30;
    for (int w = 1; w <= 32; w *= 2)
        for (int h = 1; w * h <= 128; h *= 2) {
            int n = 128 / (w * h);
            if (w * n < 8) continue;             // an 8-row operand group must not straddle two y rows
            if (need_w8 && w != 8) continue;     // halo-fed kernels need 8-pixel-wide tiles
            long long tiles = (long long)ceil_div(W, w) * ceil_div(H, h) * ceil_div(N, n);
            double eff = (double)W * H * N / (double)(tiles * 128);
            int halo = (w + 2) * (h + 2) * n;
            if (eff > best + 1e-9 || (eff > best - 1e-9 && halo < best_halo)) {
                best = eff; best_halo = halo; *bw = w; *bh = h; *bn = n;
            }
        }
}

int env_int(const char* name, int dflt) {
    const char* e = getenv(name);
    return e ? atoi(e) : dflt;
}

}  // namespace

int conv_tc_supported(int cin, int ksz, int stride) {
    if (cin % 8 != 0) return 0;
    if (!((ksz == 1 && stride == 1) || (ksz == 3 && (stride == 1 || stride == 2)))) return 0;
    return 1;
}

// depthwise 3x3 stride 1 with 16-channel groups on the tensor cores
int conv_tc_dw_supported(int cin, int cout, int ksz, int stride, int dst_f32, int has_res) {
    return cin == cout && cin % 16 == 0 && ksz == 3 && stride == 1 && !dst_f32 && !has_res;
}

// the network input: 4-channel NHWC buffer of which the first `cin` (<= 4) carry weights, 3x3, 16-bit output, one output-channel
// tile (the stride-1 form computes two pixels per GEMM row: N = 2 * cout).  conv_tc_plan checks what depends on the buffers:
// an even input size (stride 2), an even-width output buffer of its own (stride 1), a one-image 8-pixel-wide tile.
int conv_tc_stem_supported(int src_cs, int cin, int ksz, int stride, int cout, int dst_f32, int has_res) {
    return src_cs == 4 && cin <= 4 && ksz == 3 && (stride == 2 || (stride == 1 && cout % 8 == 0 && 2 * cout <= 256)) && cout <= 256 &&
           !dst_f32 && !has_res;
}

// fused depthwise + pointwise: c a multiple of 64 (whole K chunks), one output-channel tile, 16-bit unsplit storage
int conv_tc_dwpw_supported(int c, int cout, int dst_f32, int x2) {
    return c % 64 == 0 && c / 64 <= kMaxStages && cout % 16 == 0 && cout <= 256 && !dst_f32 && !x2;
}

int conv_tc_plan(ConvTcPlan* plan, int sm_count, int max_batch, const __nv_bfloat16* src, int src_h, int src_w, int src_cs,
                 int src_c0, int cin, void* dst, int dst_h, int dst_w, int dst_cs, int dst_c0, int cout, int dst_f32, int ksz,
                 int stride, int act, const float* w_host, const float* b_host, const __nv_bfloat16* res, int res_cs,
                 int res_c0, int depthwise, int f16, int x2, float acc_scale, const DwFuse* fuse) {
    // Channel arguments are REAL channel counts.  In split-fp16 storage (x2) a 16-bit buffer keeps 2 x 16 bits per channel
    // ([hi x 8 | lo x 8] groups, see split2): the A operand then has K = 2 * cin storage channels against weights packed twice,
    // and 16-bit outputs / residuals are 4 bytes per channel like fp32 ones.  The network input (stem) is never split.
    *plan = ConvTcPlan{};
    const bool dw = depthwise != 0;
    const bool fused = fuse != nullptr;       // this 1x1 conv reads the depthwise 3x3 of fuse->src computed in the same kernel (src is unused)
    B2D_CHECK(!x2 || f16, "conv_tc: split storage is fp16");
    if (fused) {
        B2D_CHECK(!dw && ksz == 1 && stride == 1 && !res && conv_tc_dwpw_supported(cin, cout, dst_f32, x2), "conv_tc: unsupported fused depthwise + pointwise shape");
        B2D_CHECK(fuse->src_cs % 8 == 0 && fuse->src_c0 % 8 == 0, "conv_tc: fused source slice must be 16-byte aligned");
        src = fuse->src; src_cs = fuse->src_cs; src_c0 = fuse->src_c0;
    }
    if (dw) B2D_CHECK(conv_tc_dw_supported(cin, cout, ksz, stride, dst_f32, res != nullptr), "conv_tc: unsupported depthwise shape");
    const bool stem = !dw && conv_tc_stem_supported(src_cs, cin, ksz, stride, cout, dst_f32, res != nullptr) && src_c0 == 0;
    if (!stem) {
        B2D_CHECK(conv_tc_supported(cin, ksz, stride), "conv_tc: unsupported shape cin=%d k=%d s=%d", cin, ksz, stride);
        B2D_CHECK(src_cs % 8 == 0 && src_c0 % 8 == 0, "conv_tc: source slice must be 16-byte aligned (cs=%d c0=%d)", src_cs, src_c0);
    }
    B2D_CHECK(stride == 1 || (src_h % 2 == 0 && src_w % 2 == 0), "conv_tc: stride-2 input must have even size");
    // Stride-1 3x3 stem (YOLOv7 model.0) through TMA: two horizontally adjacent output pixels form ONE GEMM row.  For an even x the
    // inputs of pixels x and x + 1 (input pixels x - 1 .. x + 2) lie inside the 64 contiguous, 16-byte-aligned bytes of input pixels
    // x - 2 .. x + 5 of each of the three input rows, consecutive pairs are 16 bytes apart -- the no-swizzle K-major layout again
    // (a core matrix = 8 pairs x 16 B, LBO = 16 B, SBO = one box line) -- and the pair's outputs, 2 x cout channels, are contiguous
    // in the NHWC output.  So the layer is planned as a conv with N = 2 * cout over an image of W / 2 pair-pixels: six K = 16 MMAs
    // per tile (3 filter rows x 32 input values) against weights that hold every filter tap twice, once per pixel of the pair.
    const int cout_real = cout;
    const bool stem1 = stem && stride == 1;
    B2D_CHECK(!stem1 || (dst_c0 == 0 && dst_cs == cout && dst_w % 2 == 0 && 2 * cout <= (x2 ? 128 : 256)),
              "conv_tc: the stride-1 stem writes an even-width buffer of its own (%d of %d channels at %d, width %d)", cout, dst_cs, dst_c0, dst_w);
    if (stem1) { cout *= 2; dst_cs *= 2; dst_w /= 2; }
    ConvTcParams& p = plan->p;
    plan->sm_count = sm_count;
    const int kmul = (x2 && !stem) ? 2 : 1;        // storage channels per real input channel
    const int kin = cin * kmul, src_cs_s = src_cs * kmul, src_c0_s = src_c0 * kmul;
    p.W = dst_w; p.H = dst_h; p.cin = kin; p.cout = cout;
    p.ksz = ksz; p.taps = ksz * ksz; p.stride = stride;
    p.act = act; p.out_f32 = dst_f32;
    p.x2 = x2; p.acc_scale = acc_scale;
    p.chunks = stem ? 1 : ceil_div(kin, 64);       // a short last chunk is zero-filled by TMA (A) and zero-padded in the packed weights (B)
    const int cout_pad = ceil_div(cout, 16) * 16;
    int split = 1;
    const int n_max = x2 && !dst_f32 ? 128 : 256;      // split outputs are 4 bytes per column: a 256-column staging tile alone would be 128 KB
    while (cout_pad % split != 0 || (cout_pad / split) % 16 != 0 || cout_pad / split > n_max || (dw && split > 1 && (kmul * cout_pad / split) % 64 != 0)) {
        ++split;
        B2D_CHECK(split <= cout_pad / 16, "conv_tc: %d output channels cannot be tiled (depthwise layers wider than %d need whole 64-channel chunks)", cout, n_max);
    }
    p.n_tile = cout_pad / split;
    p.n_tiles_n = split;
    if (dw) p.chunks = ceil_div(kmul * p.n_tile, 64);     // depthwise: storage chunks of one channel tile
    // the stem (conv_tc_stem2_kernel: space-to-depth for stride 2, pixel pairs for stride 1) and the fused and depthwise
    // kernels need 8-pixel-wide tiles, the stem one-image ones
    pick_tile(dst_w, dst_h, max_batch, &p.bw, &p.bh, &p.bn, stem || dw || fused);
    B2D_CHECK(!stem || p.bn == 1, "conv_tc: the stem needs a one-image tile (tile %dx%dx%d)", p.bw, p.bh, p.bn);
    // 3x3 stride-2 layers with one K chunk: the stride-2 halo kernel when an 8-pixel-wide one-image tile fits (decided below with the
    // shared-memory budget: its nine weight boxes stay resident)
    bool s2halo = !stem && !dw && !fused && ksz == 3 && stride == 2 && kin <= 64 && cout_pad <= 256;
    if (s2halo) {
        int w8, h8, n8;
        pick_tile(dst_w, dst_h, max_batch, &w8, &h8, &n8, true);
        if (n8 == 1) { p.bw = w8; p.bh = h8; p.bn = n8; }
        else s2halo = false;
    }
    p.perm = p.bn > 1 ? 1 : 0;
    p.tiles_x = ceil_div(dst_w, p.bw);
    p.tiles_y = ceil_div(dst_h, p.bh);
    auto rcp32 = [](int d) { return d <= 1 ? 0u : (uint32_t)(((1ull << 32) + (uint64_t)d - 1) / (uint64_t)d); };   // d == 1 handled below
    p.rcp_nn = rcp32(split);
    p.rcp_tx = rcp32(p.tiles_x);
    p.rcp_ty = rcp32(p.tiles_y);
    const int total_tiles = p.tiles_x * p.tiles_y * ceil_div(max_batch, p.bn) * split;
    p.a_bytes = kTileM * 64 * 2;
    p.a_tx_bytes = p.a_bytes;
    if (stem1) {        // one tile's box: (bh + 2) input rows x (2 bw + 6) pixels x 8 bytes (the last pair's K = 32 run ends at pixel
                        // x + 5: its two zero-weighted pixels must still be finite numbers, so they are fetched); two 64-value weight chunks
        p.halo_w = 2 * p.bw + 6;
        p.a_tx_bytes = (uint32_t)((p.bh + 2) * p.halo_w * 8);
        p.a_bytes = (p.a_tx_bytes + 1023u) & ~1023u;
    } else if (stem) {        // one tile's box: (bh + 1) block rows x 2 row phases x (bw + 1) block columns x 16 bytes
        p.halo_w = p.bw + 1;
        p.a_tx_bytes = (uint32_t)((p.bh + 1) * 2 * (p.bw + 1) * 16);
        p.a_bytes = (p.a_tx_bytes + 1023u) & ~1023u;
    }
    p.b_tx_bytes = dw ? 144 * 128 : p.n_tile * 64 * 2;      // depthwise: [9 taps][16 rows] x 128 B per 64-channel chunk
    p.b_bytes = (p.b_tx_bytes + 1023u) & ~1023u;
    if (stem1) p.b_bytes *= 2;                              // two 64-value weight chunks per output row
    const int esize = (dst_f32 || x2) ? 4 : 2;     // bytes per output column in the destination buffer
    const int esize_r = x2 ? 4 : 2;                // ... and per residual column
    B2D_CHECK(!(dst_f32 && res), "conv_tc: residual with fp32 output is not supported");
    B2D_CHECK(((size_t)dst_cs * esize) % 16 == 0 && ((size_t)dst_c0 * esize) % 16 == 0,
              "conv_tc: destination slice must be 16-byte aligned (cs=%d c0=%d)", dst_cs, dst_c0);
    B2D_CHECK(!res || (res_cs % 8 == 0 && res_c0 % 8 == 0), "conv_tc: residual slice must be 16-byte aligned");
    B2D_CHECK(p.bw <= 32 && 32 % p.bw == 0 && p.bw * p.bn >= 8, "conv_tc: unsupported tile %dx%dx%d", p.bw, p.bh, p.bn);
    B2D_CHECK(!stem || split == 1, "conv_tc: stem with %d output channels", cout);
    const uint32_t row_bytes = (uint32_t)p.n_tile * esize;
    const uint32_t tile_stg = 128u * row_bytes;
    const uint32_t tail_fixed = 256 /*pipeline barriers + tmem slot*/ + (uint32_t)cout_pad * 4 /*bias*/;
    // slab hand-off barriers: sfull + sempty (+ residual) per quarter and one-tile slab
    auto slab_bars = [&](int mt, int bufs) { return (uint32_t)((res ? 3 : 2) * mt * bufs * 8); };
    const uint32_t avail = 226 * 1024 - 1024 /*align slack*/ - tail_fixed;

    // ---- kind, tiles per round, stages, staging buffers ----
    // halo: 3x3 stride 1 on 8-pixel-wide tiles (uniform (bw+2)-row stride between 8-row groups)
    const bool halo_ok = !stem && ksz == 3 && stride == 1 && p.bw == 8;
    B2D_CHECK(!dw || halo_ok, "conv_tc: depthwise needs an 8-pixel-wide tile");
    B2D_CHECK(!fused || (p.bw == 8 && p.bh % 2 == 0 && (p.bn == 1 ? p.bh % 4 == 0 : p.bn % 2 == 0)), "conv_tc: fused depthwise + pointwise needs an 8-pixel-wide tile that splits into two even halves");
    if (!stem) p.halo_w = p.bw + 2;
    p.halo_kh_rows = (uint32_t)(p.bn * p.halo_w);
    const uint32_t halo_rows = (uint32_t)(p.halo_w * p.bn * (p.bh + 2));
    p.halo_bytes = (halo_rows * 128u + 1023u) & ~1023u;
    // test hooks: B2D_MT caps the M tiles per round and lifts the balance rule, B2D_PAIR = 2 forces CTA pairs (0 forbids them),
    // so that small batches run the variants the planner picks at large ones
    const int mt_env = env_int("B2D_MT", 0), pair_env = env_int("B2D_PAIR", 1);
    const bool force_pair = pair_env == 2;
    const int mt_cap = stem ? 4 : 2;
    bool planned = false;
    ConvKind best_kind = CONV_GENERIC;
    int best_mt = 1, best_stages = 0, best_bufs = 1, best_bres = 0;
    const uint32_t dw_bytes = fused ? (((uint32_t)p.chunks * (9 * 64 + 64) * 4 + 1023u) & ~1023u) : 0u;   // depthwise weights + bias in shared memory
    if (s2halo) {
        // resident weights (nine boxes), two staging buffers if they fit, the rest phase-box slots (at least the four of one tile)
        const uint32_t box = ((uint32_t)((p.bw + 1) * (p.bh + 1)) * 128u + 1023u) & ~1023u;
        const uint32_t wres = 9u * p.b_bytes;
        int bufs = 2;
        while (bufs >= 1 && avail < wres + (uint32_t)bufs * tile_stg + slab_bars(1, bufs) + 4u * box) --bufs;
        if (bufs >= 1 && split == 1) {
            int slots = (int)((avail - wres - (uint32_t)bufs * tile_stg - slab_bars(1, bufs)) / box);
            if (slots > 8) slots = 8;
            planned = true; best_kind = CONV_S2HALO; best_mt = 1; best_stages = slots; best_bufs = bufs; best_bres = 1;
            p.halo_w = p.bw + 1;
            p.halo_bytes = box;
        } else {
            s2halo = false;                      // does not fit: the generic kernel runs the layer (its tile choice is redone here)
            pick_tile(dst_w, dst_h, max_batch, &p.bw, &p.bh, &p.bn, false);
            p.perm = p.bn > 1 ? 1 : 0;
            p.tiles_x = ceil_div(dst_w, p.bw);
            p.tiles_y = ceil_div(dst_h, p.bh);
            p.rcp_tx = rcp32(p.tiles_x);
            p.rcp_ty = rcp32(p.tiles_y);
        }
    }
    if (fused) {
        // two halo buffers, two A tiles, the depthwise constants, one staging buffer (two if they fit), the rest weight stages
        const uint32_t fixed = 2u * p.halo_bytes + 2u * p.a_bytes + dw_bytes;
        B2D_CHECK(avail > fixed + tile_stg + slab_bars(1, 1) + 2u * p.b_bytes, "conv_tc: fused depthwise + pointwise does not fit shared memory (c %d cout %d)", cin, cout);
        int st = (int)((avail - fixed - tile_stg - slab_bars(1, 1)) / p.b_bytes);
        if (st >= p.chunks) { st = p.chunks; best_bres = 1; }
        if (st > kMaxStages) st = kMaxStages;
        best_bufs = avail >= fixed + 2u * tile_stg + slab_bars(1, 2) + (uint32_t)st * p.b_bytes ? 2 : 1;
        planned = true; best_kind = CONV_DWPW; best_mt = 1; best_stages = st;
    }
    // the halo kernel falls back to the generic one when its buffers do not fit
    const ConvKind first_kind = stem ? CONV_STEM : dw ? CONV_DEPTHWISE : halo_ok ? CONV_HALO : CONV_GENERIC;
    const int nkinds = first_kind == CONV_HALO ? 2 : 1;
    for (int mt = mt_cap; mt >= 1 && !planned; mt >>= 1) {
        if (mt_env > 0 && mt > mt_env) continue;
        if (mt > 1 && (split > 1 || 2 * mt * p.n_tile > 512)) continue;
        if (mt > 1 && !stem && mt_env == 0 && total_tiles < 4 * mt * sm_count) continue;   // keep enough rounds per SM for balance (B2D_MT forces)
        for (int ki = 0; ki < nkinds && !planned; ++ki) {
            const ConvKind kind = ki == 0 ? first_kind : CONV_GENERIC;
            for (int bufs = 2; bufs >= 1 && !planned; --bufs) {
                const uint32_t stg = (uint32_t)bufs * mt * tile_stg + slab_bars(mt, bufs);
                if (stg + 4096 > avail) continue;
                const uint32_t room = avail - stg;
                int stages = 0, min_stages = 0;
                bool bres = false;
                if (kind == CONV_GENERIC) {
                    const uint32_t sb = (uint32_t)mt * p.a_bytes + p.b_bytes;
                    stages = (int)(room / sb);
                    const int ksteps = p.taps * p.chunks;
                    if (stages > ksteps * 2) stages = ksteps * 2;
                    // a second staging buffer is worth more than a deep ring when a round has few k-steps (memory-bound 1x1 layers)
                    min_stages = (bufs == 2 || mt > 1) ? 4 : 2;
                    if (ksteps < min_stages) min_stages = ksteps < 2 ? 2 : ksteps;
                } else if (kind == CONV_HALO || kind == CONV_DEPTHWISE) {
                    const uint32_t fixed = 2u * mt * p.halo_bytes;
                    stages = room > fixed ? (int)((room - fixed) / p.b_bytes) : 0;
                    min_stages = (bufs == 2 || mt > 1) ? 4 : 3;
                    // resident weights: every (chunk, tap) weight box gets its own stage, loaded once per CTA.  The narrow 3x3
                    // layers are bound by the TMA unit's request rate and the per-round weight refetch was a third of it.
                    bres = kind == CONV_HALO && split == 1 && 9 * p.chunks <= kMaxStages && stages >= 9 * p.chunks;
                    if (bres) stages = 9 * p.chunks;
                } else {                                // CONV_STEM: resident weights
                    const uint32_t sb = (uint32_t)mt * p.a_bytes;
                    stages = room > p.b_bytes ? (int)((room - p.b_bytes) / sb) : 0;
                    if (stages > 4) stages = 4;
                    min_stages = 2;
                }
                if (stages > kMaxStages) stages = kMaxStages;
                if (stages < min_stages) continue;
                planned = true; best_kind = kind; best_mt = mt; best_stages = stages; best_bufs = bufs; best_bres = bres ? 1 : 0;
            }
        }
    }
    B2D_CHECK(planned, "conv_tc: no shared-memory configuration fits (n_tile %d)", p.n_tile);
    p.kind = best_kind; p.mt = best_mt; p.stages = best_stages; p.stg_bufs = best_bufs; p.b_res = best_bres;
    // CTA pairs (the PAIR forms of the halo and generic kernels) for layers with wide output tiles and enough tiles for 2 x 148
    // SMs: a stage holds half a weight tile per CTA, so the ring gets deeper.
    //   halo: 192-channel 3x3 layers and wider, n_tile a multiple of 32.
    //   generic (1x1, stride 2), one tile per round and a SHORT reduction.  Measured per op at batch 64
    //   (profiles/r2_pair_generic_per_op.txt): K = cin * taps < 576 gains 5-18 % (the weight tile is a large share of a short
    //   round's operand traffic), K >= 576 loses 1-6 % (the leader's barrier round trip through the cluster per K step is no
    //   longer hidden), so the planner pairs only the short ones ... and the 3x3 stride-1 layers that run here because their
    //   tiles are not 8 pixels wide (288 -> 288 at 20 x 20, two N = 144 tiles): 41.6 -> 35 us each with the pair's halved weight
    //   traffic, N / 2 = 72 rows per CTA.
    const bool pair_short_k = cin * p.taps < 576 || (stride == 2 && cin <= 96) || (ksz == 3 && stride == 1);
    const bool pair_kind = p.kind == CONV_HALO ? split == 1 && p.n_tile % 32 == 0
                         : p.kind == CONV_GENERIC && p.n_tile % 16 == 0 && p.mt == 1 && (pair_short_k || force_pair);
    p.pair = pair_kind && p.n_tile >= 128 && (total_tiles >= 2 * sm_count || force_pair) && pair_env != 0 ? 1 : 0;
    if (p.pair) {
        // what differs between the kinds: the halo kernel keeps its two halo buffers outside the ring, whose stages hold weights
        // only, and keeps six of them before it takes a second staging buffer; the generic ring holds A + B and needs four
        // stages, at most two rounds' worth
        const bool halo = p.kind == CONV_HALO;
        p.mt = 1;
        p.b_res = 0;
        p.b_tx_bytes = (uint32_t)(p.n_tile / 2) * 128u;
        p.b_bytes = (p.b_tx_bytes + 1023u) & ~1023u;
        const uint32_t fixed = halo ? 2u * p.halo_bytes : 0u, sb = halo ? p.b_bytes : p.a_bytes + p.b_bytes, min_st = halo ? 6u : 4u;
        if (avail > 2u * tile_stg + fixed + min_st * sb + slab_bars(1, 2)) p.stg_bufs = 2;
        const uint32_t room = avail - (uint32_t)p.stg_bufs * tile_stg - fixed - slab_bars(1, p.stg_bufs);
        int st = (int)(room / sb);
        if (!halo && st > 2 * p.taps * p.chunks) st = 2 * p.taps * p.chunks;
        p.stages = st > kMaxStages ? kMaxStages : st;
    }
    const uint32_t stg_bytes = (uint32_t)p.stg_bufs * p.mt * tile_stg;
    uint32_t operand_bytes = 0;
    switch (p.kind) {
        case CONV_GENERIC: operand_bytes = (uint32_t)p.stages * ((uint32_t)p.mt * p.a_bytes + p.b_bytes); break;
        case CONV_HALO:
        case CONV_DEPTHWISE:
            p.a_tx_bytes = halo_rows * 128u;
            operand_bytes = 2u * p.mt * p.halo_bytes + (uint32_t)p.stages * p.b_bytes;
            break;
        case CONV_STEM: operand_bytes = (uint32_t)p.stages * p.mt * p.a_bytes + p.b_bytes; break;
        case CONV_DWPW:
            p.a_tx_bytes = halo_rows * 128u;
            operand_bytes = 2u * p.halo_bytes + 2u * p.a_bytes + (uint32_t)p.stages * p.b_bytes + dw_bytes;
            break;
        case CONV_S2HALO:
            p.a_tx_bytes = (uint32_t)((p.bw + 1) * (p.bh + 1)) * 128u;
            operand_bytes = (uint32_t)p.stages * p.halo_bytes + 9u * p.b_bytes;
            break;
    }
    p.stg_off = operand_bytes;                                   // 1 KiB aligned: every operand slot is a multiple of 1 KiB
    p.dw_off = operand_bytes - dw_bytes;
    p.bar_off = p.stg_off + stg_bytes;
    plan->smem_bytes = (size_t)p.bar_off + tail_fixed + slab_bars(p.mt, p.stg_bufs) + 1024 /*align slack*/;
    B2D_CHECK(plan->smem_bytes <= 227 * 1024, "conv_tc: %zu bytes of shared memory needed", plan->smem_bytes);
    // epilogue chunks (epi_chunks): at most six, which bounds fp32 tiles at 192 columns
    const EpiChunks epi = epi_chunks(row_bytes);
    B2D_CHECK(epi.n128 + epi.has64 + epi.has32 <= 6, "conv_tc: n_tile %d needs too many epilogue chunks", p.n_tile);
    B2D_CHECK(row_bytes % 32 == 0, "conv_tc: n_tile %d is not a multiple of 32 bytes", p.n_tile);
    p.has_res = res ? 1 : 0;
    // Epilogue warps per TMEM lane quarter.  A warp's epilogue is a chain of dependent instructions (TMEM load -> bias FMA ->
    // MUFU.TANH -> FMA -> pack -> shared store) that issues about one instruction per six cycles; with two warps per scheduler
    // the epilogue ran at 3-4.5 outputs per clock per SM against 15 for the same code with eight warps per scheduler
    // (role traces, profiles/r2_role_traces.txt).  A third warp per quarter takes every third 16-column unit when the tile
    // width allows an even split (48, 96, 144, 192 ...).
    p.epi_parts = fused ? 1 : (p.n_tile >> 4) % 3 == 0 ? 3 : 2;   // fused: warps 8-15 compute the depthwise stage
    p.trace = nullptr;
    if (getenv("B2D_TRACE")) {
        if (plan->trace_dev.reserve(sizeof(long long) * kTraceRoles * kTraceTiles * kTraceEvents)) return -2;
        p.trace = plan->trace_dev.get();
    }
    uint32_t cols = 32;
    while (cols < (uint32_t)(2 * p.mt * p.n_tile)) cols *= 2;
    p.tmem_cols = cols;
    // kind::f16 instruction descriptor: D=f32, A=B=bf16, both K-major, N>>3 at [17,23), M>>4 at [24,29)
    p.f16 = f16;
    p.idesc = (1u << 4) | (f16 ? 0u : (1u << 7) | (1u << 10)) |        // D fp32; A / B format: 1 = bf16, 0 = fp16 (also the split storage)
              ((uint32_t)((dw ? 16 : p.n_tile) >> 3) << 17) | ((uint32_t)((p.pair ? 2 * kTileM : kTileM) >> 4) << 24);

    // ---- weights: fp32 [cout][cin][k][k] -> bf16 [cout_pad][kh][kw][cin_pad] (zero padded) ----
    const int cin_pad = p.chunks * 64;
    const size_t ktot = stem1 ? 128 : stem ? 64 : (size_t)p.taps * cin_pad;     // stem: one or two 128-byte rows per output channel
    const int dw_chunks = p.chunks * split;                       // depthwise: 64-channel chunks over all channels
    std::vector<uint16_t> wp(dw ? (size_t)dw_chunks * 9 * 16 * 64 : (size_t)cout_pad * ktot, 0);
    if (dw && x2) {
        // a 64-channel storage chunk = 32 real channels; real channel r of the chunk -> accumulator block g2 = r / 16, column
        // n = r % 16, storage K group q = 2 g2 + n / 8, K positions j = n % 8 (its hi) and j + 8 (its lo)
        for (int c = 0; c < cout; ++c)
            for (int t = 0; t < 9; ++t) {
                const int chunk = c / 32, r = c % 32, g2 = r / 16, n = r % 16, q = 2 * g2 + n / 8, j = n % 8;
                const size_t row = ((size_t)chunk * 9 + t) * 16 + n;
                const uint16_t v = f2h(w_host[(size_t)c * 9 + t]);
                wp[row * 64 + q * 16 + j] = v;
                wp[row * 64 + q * 16 + j + 8] = v;
            }
    } else if (dw) {
        // row (chunk * 9 + tap) * 16 + n, 64 k each: k = group * 16 + n carries w[chunk * 64 + group * 16 + n][tap]
        for (int c = 0; c < cout; ++c)
            for (int t = 0; t < 9; ++t) {
                const int chunk = c / 64, g = (c % 64) / 16, d = c % 16;
                const size_t row = ((size_t)chunk * 9 + t) * 16 + d;
                wp[row * 64 + g * 16 + d] = f16 ? f2h(w_host[(size_t)c * 9 + t]) : f2bf(w_host[(size_t)c * 9 + t]);
            }
    } else {
        for (int o = 0; o < cout_real; ++o)
            for (int c = 0; c < cin; ++c)
                for (int t = 0; t < p.taps; ++t) {
                    const uint16_t v = f16 ? f2h(w_host[((size_t)o * cin + c) * p.taps + t]) : f2bf(w_host[((size_t)o * cin + c) * p.taps + t]);
                    if (stem1) {      // row half * cout + o (half = pixel of the pair), k = kh * 32 + (kw + 1 + half) * 4 + c
                        const int kh = t / 3, kw = t % 3;
                        for (int half = 0; half < 2; ++half)
                            wp[(size_t)(half * cout_real + o) * ktot + (size_t)(kh * 32 + (kw + 1 + half) * 4 + c)] = v;
                    } else if (stem) {      // tap (kh, kw) -> block (di, dj), phase (rp, px): k = (di * 2 + dj) * 16 + rp * 8 + px * 4 + c
                        const int kh = t / 3, kw = t % 3;
                        const int di = kh == 0 ? 0 : 1, rp = kh == 1 ? 0 : 1, dj = kw == 0 ? 0 : 1, px = kw == 1 ? 0 : 1;
                        wp[(size_t)o * ktot + (size_t)((di * 2 + dj) * 16 + rp * 8 + px * 4 + c)] = v;
                    } else if (kmul == 2) {      // the weight sits under the channel's hi and lo position
                        const size_t k = (size_t)t * cin_pad + 16 * (c / 8) + (c % 8);
                        wp[(size_t)o * ktot + k] = v;
                        wp[(size_t)o * ktot + k + 8] = v;
                    } else {
                        wp[(size_t)o * ktot + (size_t)t * cin_pad + c] = v;
                    }
                }
    }
    std::vector<float> bp(cout_pad, 0.f);
    for (int o = 0; o < cout; ++o) bp[o] = b_host ? b_host[o % cout_real] : 0.f;      // stride-1 stem: both pixels of a pair
    if (plan->w_dev.reserve(wp.size() * 2)) return -2;
    B2D_CUDA(cudaMemcpy(plan->w_dev.get(), wp.data(), wp.size() * 2, cudaMemcpyHostToDevice));
    if (plan->bias_dev.reserve(bp.size() * 4)) return -2;
    B2D_CUDA(cudaMemcpy(plan->bias_dev.get(), bp.data(), bp.size() * 4, cudaMemcpyHostToDevice));
    p.bias = plan->bias_dev.get();
    p.w_raw = plan->w_dev.get();
    if (fused) {
        // [chunk][tap][64] fp32 then [chunks * 64] bias; values rounded to the 16-bit weight format like every packed weight, and
        // halved for SiLU layers (silu2_h takes v / 2; the scaling is exact)
        std::vector<float> dwc((size_t)p.chunks * (9 * 64 + 64), 0.f);
        const float hs = fuse->act ? 0.5f : 1.0f;
        for (int c = 0; c < cin; ++c) {
            for (int t = 0; t < 9; ++t) {
                const uint16_t v = f16 ? f2h(fuse->w[(size_t)c * 9 + t]) : f2bf(fuse->w[(size_t)c * 9 + t]);
                float wf;
                if (f16) { __half h; memcpy(&h, &v, 2); wf = __half2float(h); }
                else { uint32_t u = (uint32_t)v << 16; memcpy(&wf, &u, 4); }
                dwc[((size_t)(c / 64) * 9 + t) * 64 + c % 64] = hs * wf;
            }
            dwc[(size_t)p.chunks * 9 * 64 + c] = hs * (fuse->b ? fuse->b[c] : 0.f);
        }
        if (plan->dw_dev.reserve(dwc.size() * 4)) return -2;
        B2D_CUDA(cudaMemcpy(plan->dw_dev.get(), dwc.data(), dwc.size() * 4, cudaMemcpyHostToDevice));
        p.dw_w = plan->dw_dev.get();
        p.dw_act = fuse->act;
    }

    // ---- tensor maps ----
    const bool perm = p.perm != 0;
    if (!stem) {
        if (dw) {
            uint64_t dims[2] = {64u, (uint64_t)dw_chunks * 9 * 16};
            uint64_t str[1] = {128u};
            uint32_t box[2] = {64u, 144u};
            if (encode_map(&p.tmB, plan->w_dev.get(), 2, dims, str, box, 128)) return -1;
        } else {
            uint64_t dims[2] = {(uint64_t)ktot, (uint64_t)cout_pad};
            uint64_t str[1] = {(uint64_t)ktot * 2};
            uint32_t box[2] = {64u, (uint32_t)(p.pair ? p.n_tile / 2 : p.n_tile)};
            if (encode_map(&p.tmB, plan->w_dev.get(), 2, dims, str, box, 128)) return -1;
        }
        const uint64_t pix = (uint64_t)src_cs_s * 2, rowb = (uint64_t)src_w * pix, imgb = (uint64_t)src_h * rowb;
        if (p.kind == CONV_HALO || p.kind == CONV_DEPTHWISE || p.kind == CONV_DWPW) {
            if (encode_act_map(&p.tmA[0], (void*)(src + src_c0_s), kin, src_w, src_h, max_batch, pix, rowb, imgb, 64u, (uint32_t)p.halo_w,
                               (uint32_t)(p.bh + 2), (uint32_t)p.bn, perm, p.kind == CONV_DWPW ? 0 : 128))    // fused: read by threads, plain rows
                return -1;
        } else if (stride == 1) {
            if (encode_act_map(&p.tmA[0], (void*)(src + src_c0_s), kin, src_w, src_h, max_batch, pix, rowb, imgb, 64u, (uint32_t)p.bw, (uint32_t)p.bh,
                               (uint32_t)p.bn, perm, 128))
                return -1;
        } else {
            const uint32_t hb = p.kind == CONV_S2HALO ? 1u : 0u;           // stride-2 halo kernel: one more column and row per phase box
            for (int py = 0; py < 2; ++py)
                for (int px = 0; px < 2; ++px) {
                    const __nv_bfloat16* base = src + ((size_t)py * src_w + px) * src_cs_s + src_c0_s;
                    if (encode_act_map(&p.tmA[py * 2 + px], (void*)base, kin, src_w / 2, src_h / 2, max_batch, 2 * pix, 2 * rowb, imgb, 64u,
                                       (uint32_t)p.bw + hb, (uint32_t)p.bh + hb, (uint32_t)p.bn, perm, 128))
                        return -1;
                }
        }
    }
    if (stem1) {        // (8-byte pixels of an input row as 16-bit elements | row | image | 1), un-swizzled box of (bh + 2) rows
        uint64_t dims[4] = {(uint64_t)src_w * 4, (uint64_t)src_h, (uint64_t)max_batch, 1u};
        uint64_t str[3] = {(uint64_t)src_w * 8, (uint64_t)src_h * src_w * 8, (uint64_t)src_h * src_w * 8 * (uint64_t)max_batch};
        uint32_t box[4] = {(uint32_t)p.halo_w * 4u, (uint32_t)(p.bh + 2), 1u, 1u};
        if (encode_map(&p.tmA[0], (void*)src, 4, dims, str, box, 0)) return -1;
    } else if (stem) {        // (8-byte pixels of one input row as 16-bit elements | row phase | block row | image), un-swizzled box
        uint64_t dims[4] = {(uint64_t)src_w * 4, 2u, (uint64_t)src_h / 2, (uint64_t)max_batch};
        uint64_t str[3] = {(uint64_t)src_w * 8, (uint64_t)src_w * 16, (uint64_t)src_h * src_w * 8};
        uint32_t box[4] = {(uint32_t)(p.bw + 1) * 8u, 2u, (uint32_t)(p.bh + 1), 1u};
        if (encode_map(&p.tmA[0], (void*)src, 4, dims, str, box, 0)) return -1;
    }
    {   // output / residual maps: the box is one M tile, one map per chunk width
        const uint32_t sbn = (uint32_t)p.bn, sbh = (uint32_t)p.bh;
        const uint32_t spans[3] = {128, 64, 32};
        const bool used[3] = {epi.n128 > 0, epi.has64 != 0, epi.has32 != 0};
        const uint64_t pix = (uint64_t)dst_cs * esize, rowb = (uint64_t)dst_w * pix, imgb = (uint64_t)dst_h * rowb;
        for (int si = 0; si < 3; ++si) {
            if (!used[si]) continue;
            if (encode_act_map(&p.tmO[si], (uint8_t*)dst + (size_t)dst_c0 * esize, cout, dst_w, dst_h, max_batch, pix, rowb, imgb,
                               spans[si] / (uint32_t)esize, (uint32_t)p.bw, sbh, sbn, perm, spans[si], esize == 4))
                return -1;
            if (res) {
                const uint64_t rpix = (uint64_t)res_cs * esize_r, rrow = (uint64_t)dst_w * rpix, rimg = (uint64_t)dst_h * rrow;
                if (encode_act_map(&p.tmR[si], (void*)((const uint8_t*)res + (size_t)res_c0 * esize_r), cout, dst_w, dst_h, max_batch, rpix, rrow, rimg,
                                   spans[si] / (uint32_t)esize_r, (uint32_t)p.bw, sbh, sbn, perm, spans[si], esize_r == 4))
                    return -1;
            }
        }
    }
    return 0;
}

namespace {
typedef void (*ConvKernel)(const ConvTcParams, int);
// (kind, act, res, out) -> instantiation; out: 0 16-bit, 1 fp32 (never with a residual), 2 split fp16
ConvKernel pick_kernel(ConvKind kind, int pair, int act, int res, int out) {
    // K<act, res, out ...>, the trailing arguments (`, pair`) for the kernels with a CTA-pair form
#define B2D_PICK(K, ...)                                                                        \
    if (out == 1) return act ? K<1, 0, 1 __VA_ARGS__> : K<0, 0, 1 __VA_ARGS__>;                 \
    if (out == 2 && res) return act ? K<1, 1, 2 __VA_ARGS__> : K<0, 1, 2 __VA_ARGS__>;          \
    if (out == 2) return act ? K<1, 0, 2 __VA_ARGS__> : K<0, 0, 2 __VA_ARGS__>;                 \
    if (res) return act ? K<1, 1, 0 __VA_ARGS__> : K<0, 1, 0 __VA_ARGS__>;                      \
    return act ? K<1, 0, 0 __VA_ARGS__> : K<0, 0, 0 __VA_ARGS__>;
    if (kind == CONV_S2HALO) { B2D_PICK(conv_tc_s2halo_kernel, ) }
    if (kind == CONV_DWPW) return act ? conv_tc_dwpw_kernel<1, 0> : conv_tc_dwpw_kernel<0, 0>;
    if (kind == CONV_STEM) return out == 2 ? (act ? conv_tc_stem2_kernel<1, 2> : conv_tc_stem2_kernel<0, 2>) : (act ? conv_tc_stem2_kernel<1, 0> : conv_tc_stem2_kernel<0, 0>);
    if (kind == CONV_DEPTHWISE) return out == 2 ? (act ? conv_tc_dw_kernel<1, 2> : conv_tc_dw_kernel<0, 2>) : (act ? conv_tc_dw_kernel<1, 0> : conv_tc_dw_kernel<0, 0>);
    if (kind == CONV_HALO) {
        if (pair) { B2D_PICK(conv_tc_halo_kernel, , 1) }
        B2D_PICK(conv_tc_halo_kernel, , 0)
    }
    if (pair) { B2D_PICK(conv_tc_kernel, , 1) }
    B2D_PICK(conv_tc_kernel, , 0)
#undef B2D_PICK
}
}  // namespace

int conv_tc_launch(const ConvTcPlan* plan, int n, cudaStream_t stream) {
    ConvTcParams p = plan->p;
    const int tiles = p.tiles_x * p.tiles_y * ceil_div(n, p.bn) * p.n_tiles_n;
    // Every other op of the graph walks its tiles backwards: what the previous kernel wrote last (the part of its output
    // still resident in the 126 MB L2) is what this kernel reads first, before its own traffic evicts it.
    p.rev_last = p.rev ? tiles / p.n_tiles_n - 1 : -1;
    const int rounds = ceil_div(tiles, p.mt);
    int grid = rounds < plan->sm_count ? rounds : plan->sm_count;
    if (grid < 1) return 0;
    if (p.pair) {
        const int prs = ceil_div(tiles / p.n_tiles_n, 2) * p.n_tiles_n;      // rounds of a pair (see RoundSched)
        grid = 2 * (prs < plan->sm_count / 2 ? prs : plan->sm_count / 2);
    }
    ConvKernel k = pick_kernel(p.kind, p.pair, p.act, p.has_res, p.out_f32 ? 1 : p.x2 ? 2 : 0);
    if (b2d_func_smem_optin((const void*)k, 227 * 1024)) return -2;
    if (p.trace) B2D_CUDA(cudaMemsetAsync(p.trace, 0, sizeof(long long) * kTraceRoles * kTraceTiles * kTraceEvents, stream));
    {
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3((unsigned)grid);
        cfg.blockDim = dim3(kThreads);
        cfg.dynamicSmemBytes = plan->smem_bytes;
        cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        if (p.pair) {
            attr[0].id = cudaLaunchAttributeClusterDimension;
            attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        }
        cfg.attrs = attr;
        cfg.numAttrs = p.pair ? 1 : 0;
        B2D_CUDA(cudaLaunchKernelEx(&cfg, k, p, n));
    }
    if (p.trace && getenv("B2D_TRACE_DUMP")) {
        static long long h[kTraceRoles * kTraceTiles * kTraceEvents];
        B2D_CUDA(cudaStreamSynchronize(stream));
        B2D_CUDA(cudaMemcpy(h, p.trace, sizeof(h), cudaMemcpyDeviceToHost));
        long long t0 = h[0] ? h[0] : h[kTraceTiles * kTraceEvents];
        const char* names[kTraceRoles] = {"load", "mma ", "epi ", "epi: ld-wait slab-wait math hand-off"};
        fprintf(stderr, "trace (cycles from first stamp; load: first issue, last issue | mma: start, tmem free, first operand, last commit | epi: slab free, acc ready, math done, store issued)\n");
        for (int it = 0; it < kTraceTiles; ++it) {
            fprintf(stderr, "round %2d", it);
            for (int r = 0; r < kTraceRoles; ++r) {
                fprintf(stderr, " | %s", names[r]);
                for (int e = 0; e < kTraceEvents; ++e) {
                    long long v = h[(r * kTraceTiles + it) * kTraceEvents + e];
                    if (v) fprintf(stderr, " %7lld", v - t0); else fprintf(stderr, "       -");
                }
            }
            fprintf(stderr, "\n");
        }
    }
    B2D_LAUNCH_CHECK();
    return 0;
}

int conv_tc_describe(const ConvTcPlan* plan, char* buf, int buflen) {
    const ConvTcParams& p = plan->p;
    const char* name = "";
    switch (p.kind) {
        case CONV_GENERIC: name = p.pair ? "-pair" : ""; break;
        case CONV_HALO: name = p.pair ? "-halo-pair" : "-halo"; break;
        case CONV_DEPTHWISE: name = "-depthwise"; break;
        case CONV_STEM: name = p.stride == 1 ? "-stem-pairs" : "-stem-s2d"; break;
        case CONV_DWPW: name = "-dw3x3+pw"; break;
        case CONV_S2HALO: name = "-s2halo"; break;
    }
    const int cin = p.x2 && p.kind != CONV_STEM ? p.cin / 2 : p.cin;     // split storage doubles K, except on the network input
    return snprintf(buf, buflen, "tcgen05%s conv k%d s%d cin %d cout %d -> %dx%d | tile %dx%dx%d x%d n_tile %d x%d stages %d%s stg %d tmem %u smem %zu",
                    name, p.ksz, p.stride, cin, p.cout, p.H, p.W, p.bw, p.bh, p.bn, p.mt, p.n_tile, p.n_tiles_n, p.stages,
                    p.b_res ? " (resident)" : "", p.stg_bufs, p.tmem_cols, plan->smem_bytes);
}
