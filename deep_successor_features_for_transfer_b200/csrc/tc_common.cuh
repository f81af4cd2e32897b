// Blackwell (sm_100a) primitives used by the tensor-core path: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 MMA with
// TMEM accumulators, UMMA shared-memory / instruction descriptors.  Raw PTX, no CUTLASS.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include "common.cuh"

namespace sfgpi {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// Bounded spin: a protocol bug must end in a trap (reported CUDA error), never in a hung GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    long long t0 = 0;
    for (uint32_t spin = 0; !done; ++spin) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (!done && (spin & 1023) == 1023) {
            const long long now = clock64();
            if (t0 == 0) t0 = now;
            else if (now - t0 > 4000000000ll) __trap();       // ~2 s: a healthy wait is microseconds
        }
    }
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const void *tmap) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
// 2-D tiled load: box -> smem, completion counted in bytes on `bar`.  crd0 = innermost (contiguous) coordinate.
__device__ __forceinline__ void tma_load_2d(uint32_t smem_dst, const void *tmap, uint32_t bar, int crd0, int crd1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(crd0), "r"(crd1)
        : "memory");
}

// 3-D tiled load (crd2 = outermost): used for the [slab][row][col] activation / dZ tensors so that a row tile is clipped
// (zero-filled) at the end of ITS slab instead of running into the next one.
__device__ __forceinline__ void tma_load_3d(uint32_t smem_dst, const void *tmap, uint32_t bar, int crd0, int crd1, int crd2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(crd0), "r"(crd1), "r"(crd2)
        : "memory");
}

// Tiled store shared -> global (bulk async-group completion).  The source tile must be visible to the async proxy
// (fence.proxy.async by its writers + a barrier) and must not be overwritten before bulk_wait_read0() returns in the issuer.
__device__ __forceinline__ void tma_store_3d(const void *tmap, uint32_t smem_src, int crd0, int crd1, int crd2) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
                 ::"l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_src), "r"(crd0), "r"(crd1), "r"(crd2)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }   // all but the newest
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ---------------------------------------------------------------- TMEM / tcgen05
__device__ __forceinline__ void tmem_alloc(uint32_t smem_result, uint32_t ncols) {      // whole warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_result), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {          // whole warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem], bf16 inputs, fp32 accumulate; issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// ---- warp-uniform issue: the WHOLE warp runs the issue loop (so every operand is provably warp-uniform and lives in uniform
// registers) and only the instruction itself is predicated on the elected lane.  Issuing from inside `if (lane == 0)` makes
// ptxas treat the descriptors as per-thread values: every UTCHMMA / UTMALDG is then wrapped in an ELECT + 7x R2UR "waterfall"
// loop that costs ~170 cycles per MMA (measured: in-kernel clock64 timeline), 2.6x the 64-cycle MMA it feeds.
__device__ __forceinline__ uint32_t elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred;
}
__device__ __forceinline__ void umma_bf16_e(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate,
                                            uint32_t leader) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "setp.ne.b32 q, %5, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(leader)
        : "memory");
}
__device__ __forceinline__ void umma_commit_e(uint32_t bar, uint32_t leader) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "setp.ne.b32 q, %1, 0;\n\t"
        "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}"
        ::"r"(bar), "r"(leader)
        : "memory");
}
// whole-warp wait without the clock-based watchdog (keeps the loop's control flow value-uniform); bounded by a spin count
__device__ __forceinline__ void mbar_wait_warp(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    for (uint32_t spin = 0; !done; ++spin) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (spin > (1u << 26)) __trap();
    }
}
__device__ __forceinline__ void mbar_arrive_expect_tx_e(uint32_t bar, uint32_t bytes, uint32_t leader) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "setp.ne.b32 q, %2, 0;\n\t"
        "@q mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n\t}"
        ::"r"(bar), "r"(bytes), "r"(leader)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d_e(uint32_t smem_dst, const void *tmap, uint32_t bar, int crd0, int crd1, uint32_t leader) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "setp.ne.b32 q, %5, 0;\n\t"
        "@q cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n\t}"
        ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(crd0), "r"(crd1), "r"(leader)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d_e(uint32_t smem_dst, const void *tmap, uint32_t bar, int crd0, int crd1, int crd2,
                                              uint32_t leader) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "setp.ne.b32 q, %6, 0;\n\t"
        "@q cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];\n\t}"
        ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(crd0), "r"(crd1), "r"(crd2), "r"(leader)
        : "memory");
}

// mbarrier arrives once all previously issued MMAs of this thread have completed (implies fence::before_thread_sync)
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (thread = TMEM lane = output row)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}

// 32 lanes x 8 consecutive fp32 columns (compact epilogue loops: small code beats wide loads when the loop body is cold)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr)
                 : "memory");
}

// ---------------------------------------------------------------- descriptors
// K-major operand tile in the canonical 128B-swizzled layout: row r at byte r*128, 16-byte chunk j stored at j ^ (r & 7);
// 8-row groups 1024 B apart (SBO).  Bits: [0,14) addr>>4, [16,30) LBO>>4 (unused for swizzled K-major), [32,46) SBO>>4,
// [46,48) version = 1 (Blackwell), [61,64) layout type 2 = SWIZZLE_128B.  (cute/arch/mma_sm100_desc.hpp bitfields.)
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t smem_addr) {
    return (uint64_t)((smem_addr & 0x3FFFF) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) |
           ((uint64_t)2 << 61);
}
// MN-major operand tile (the reduction index k is the ROW of the source matrix, the M/N index is contiguous) in the canonical
// 128B-swizzled layout  ((8,n),(8,k)) : ((1,LBO),(8,SBO))  in 16-byte units (cute/atom/mma_traits_sm100.hpp): one atom =
// 64 M/N-elements (one 128 B row) x 8 k-rows; 8-row k groups SBO = 1024 B apart; 64-wide M/N blocks LBO bytes apart.
// This is exactly what a TMA box {64 elements, R rows} with SWIZZLE_128B of a row-major [k][mn] matrix produces
// (LBO = R * 128 when consecutive boxes hold consecutive 64-wide column blocks).  A K=16 step advances the address by 2048 B.
__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes) {
    return (uint64_t)((smem_addr & 0x3FFFF) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(1024 >> 4) << 32) |
           ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
// kind::f16 instruction descriptor: c_format F32 (1) @4, a/b format BF16 (1) @7/@10, K-major A and B, N>>3 @17, M>>4 @24.
__device__ __forceinline__ uint32_t umma_idesc_bf16(uint32_t M, uint32_t N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

// same with explicit operand majors (bit 15: A is MN-major, bit 16: B is MN-major)
__device__ __forceinline__ uint32_t umma_idesc_bf16_major(uint32_t M, uint32_t N, uint32_t a_mn, uint32_t b_mn) {
    return umma_idesc_bf16(M, N) | (a_mn << 15) | (b_mn << 16);
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);       // .x = lo (low 16 bits)
    return *reinterpret_cast<uint32_t *>(&h);
}
__device__ __forceinline__ float bf16_round(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }

constexpr int kTM = 128;                 // rows per tile (UMMA M)
constexpr int kH = 256;                  // hidden width == K of every hidden MMA layer (the shipped configs' MLP width)
constexpr int kKB = 64;                  // k elements per stage (one 128B swizzle span of bf16)

// explicit shared-space accesses (32-bit shared addresses; keeps everything on LDS/STS instead of generic LD/ST)
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ float lds32(uint32_t addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts32(uint32_t addr, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory"); }

// byte offset of the 16-byte chunk holding columns [c, c+8) of row r inside a [128][256] bf16 K-major SW128 operand
__device__ __forceinline__ uint32_t a_chunk_off(int r, int c) {
    const int kb = c >> 6, j = (c & 63) >> 3;
    return (uint32_t)(kb * (kTM * 128) + r * 128 + ((j ^ (r & 7)) << 4));
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static inline EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *sym = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(sym);
    }
    return fn;
}

// Host-side cache of encoded tensor maps (per translation unit).  A train step needs ~15 maps whose arguments never change from
// one step to the next; cuTensorMapEncodeTiled costs ~0.5-1 us each and the forward's nine sit on the host's critical path
// between the prologue launch and the forward launch (4.7 us hand-over in an isolated step, profiles/r02_forward_chain.md).
// Key = every argument of the encode call; 64 entries, round-robin replacement.  outer_stride: byte stride of the outermost
// dimension when it is not the packed one (0 = packed).
struct TmapKey {
    const void *base;
    uint64_t dims[3];
    uint32_t box[3];
    int rank, dtype, swizzle;
    uint64_t outer_stride;
    bool operator==(const TmapKey &o) const {
        return base == o.base && rank == o.rank && dtype == o.dtype && swizzle == o.swizzle && dims[0] == o.dims[0] && dims[1] == o.dims[1] &&
               dims[2] == o.dims[2] && box[0] == o.box[0] && box[1] == o.box[1] && box[2] == o.box[2] && outer_stride == o.outer_stride;
    }
};
static inline bool tmap_cache_get(const TmapKey &k, CUtensorMap *out, bool store) {
    static TmapKey keys[64];
    static CUtensorMap maps[64];
    static int used = 0, next = 0;
    if (!store) {
        for (int i = 0; i < used; ++i)
            if (keys[i] == k) { *out = maps[i]; return true; }
        return false;
    }
    const int slot = used < 64 ? used++ : (next++ & 63);
    keys[slot] = k;
    maps[slot] = *out;
    return true;
}

}  // namespace tc
}  // namespace sfgpi
