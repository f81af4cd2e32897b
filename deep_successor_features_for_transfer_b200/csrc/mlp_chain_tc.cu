// Fused ensemble psi-MLP forward on tcgen05, layer-pipelined inside ONE row tile ("chain" kernel; bf16 operands, fp32 TMEM
// accumulation).  Same jobs, arguments, shadow layout and bit-identical results as mlp_forward_tc.cu (tests/test_gpu_bf16.py::
// test_bf16_chain_and_pair_kernels_agree_bit_for_bit); what differs is how a CTA overlaps the tensor pipe with the epilogue.
//
// mlp_forward_tc.cu overlaps the epilogue of tile X with the MMAs of a second tile Y (ping-pong pairs).  A CTA with a single
// tile has nothing to ping-pong with: its 4-layer chain is MMA (~2-4 k cycles), then epilogue (~2 k), per layer.  Here the
// overlap is INSIDE the tile.  Output columns [64 j, 64 j + 64) of layer l are exactly k-block j of layer l+1's A operand, so
// the epilogue hands the next operand over in four quarters (barriers A_READY[j]) and the MMA warp issues k-block j of layer
// l+1 while the epilogue warps still drain the later columns of layer l.  The two accumulators (TMEM columns 0-255 / 256-511)
// alternate between consecutive layers; the A operand is rewritten IN PLACE (layer l's MMAs have completed when its
// accumulator is handed to the epilogue), which leaves room for an 8-stage weight ring: a whole 256 x 256 layer is in flight,
// so layer l+1's weights are resident before its first k-block may issue.  The next tile's state rows and biases are prefetched
// with cp.async during the current tile and staged as soon as its last accumulator is complete, so the next input layer runs
// under the current output epilogue.
//
// Measured on B200 (in-kernel clock64 timeline, SFGPI_TIMELINE=1; profiles/r02_forward_chain.md): the epilogue drains an
// accumulator at TMEM's ~64 B/cycle (2 k cycles per 128 x 256 fp32), the MMA phase of a layer runs at ~230 cycles per
// N = 256, K = 16 MMA while an epilogue shares the shared-memory ports (3-3.7 k cycles per layer: operand reads 192 KB + weight
// stages 128 KB + epilogue writes 64 KB per tile-layer against 128 B/cycle), and a layer of the chain costs ~5 k cycles = first
// quarter of the epilogue + MMA phase + completion latency.  That beats a lone tile of the pair kernel (84 vs 90 us per B = 32
// train step) but not a ping-pong pair, which hides the whole MMA phase behind the OTHER tile's epilogue (3.1 k cycles per
// tile-layer; 50 vs 52 us for the 384-tile headline launch).  sfgpi_mlp_forward_tc_jobs therefore picks this kernel for launches
// of <= 148 tiles (one wave) and the pair kernel beyond; sfgpi_set_option("forward_chain", ...) overrides.
//
// Code size matters: whatever runs once per tile is instruction-fetch bound (an unrolled 36-column GPI scan cost 8-10 k cycles
// per tile, measured), so the once-per-tile paths are rolled loops and the helpers exist once (__noinline__).
//
//   warps 0-3   TMA producers (ring of 8 x 16 KB stages, stage s owned by warp s & 3)
//   warp 4      MMA issuer
//   warps 5-12  epilogue: thread = TMEM lane = state row; group g = (warp - 5) / 4 takes columns [64 j + 32 g, +32) of quarter j
#include "forward_tc.cuh"
#include <limits.h>
#include <stdlib.h>

namespace sfgpi {
namespace tc {

constexpr int kRing = 8;                             // ring stages (16 KB each): one full hidden layer
constexpr int kXsFloats = 2560;                      // prefetched fp32 state tile [128][S], S <= 20
constexpr int kBiasHalf = kBiasFloatsMax / 2;        // double-buffered biases when every job needs <= 3072 floats

__device__ __forceinline__ void cp_async4(uint32_t smem_dst, const void *gsrc, bool valid) {      // 4 bytes, zero-filled if !valid
    const uint32_t n = valid ? 4u : 0u;
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(smem_dst), "l"(gsrc), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_async_commit_all() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

struct ChainSmem { uint32_t a, ring, bias, xs, bar; };
__device__ __forceinline__ uint32_t bar_w_full(const ChainSmem &s, int i) { return s.bar + 8u * i; }
__device__ __forceinline__ uint32_t bar_w_empty(const ChainSmem &s, int i) { return s.bar + 8u * (kRing + i); }
__device__ __forceinline__ uint32_t bar_a_ready(const ChainSmem &s, int j) { return s.bar + 8u * (2 * kRing + j); }
__device__ __forceinline__ uint32_t bar_acc_full(const ChainSmem &s, int a) { return s.bar + 8u * (2 * kRing + 4 + a); }
__device__ __forceinline__ uint32_t bar_acc_empty(const ChainSmem &s, int a) { return s.bar + 8u * (2 * kRing + 6 + a); }

// work unit g = one row tile: job, policy slot, tile
__device__ __forceinline__ void chain_unit(const TcMulti &m, int g, int &jb, int &pl, int &tile) {
    jb = 0;
    while (jb + 1 < m.n_jobs && g >= m.pair_start[jb + 1]) ++jb;
    const int t = g - m.pair_start[jb];
    pl = t / m.job[jb].tiles_per_policy;
    tile = t - pl * m.job[jb].tiles_per_policy;
}

// ---- prefetch of a unit's inputs (all 256 epilogue threads): state rows -> xs (fp32), biases -> bias buffer `buf` ----
__device__ __noinline__ void chain_prefetch(const TcMulti &m, int g, int buf, int et, ChainSmem sm) {
    int jb, pl, tile;
    chain_unit(m, g, jb, pl, tile);
    const TcParams &p = m.job[jb];
    const sfgpi_forward_args &a = p.a;
    const sfgpi_net_desc &net = a.net;
    const int S = net.dims[0], B = a.B, L = net.n_layers, AD = net.n_actions * net.n_features;
    if (128 * S <= kXsFloats) {
        const int row_first = tile * kTM;
        for (int e = et; e < 128 * S; e += 256) {
            const bool ok = row_first + e / S < B;
            cp_async4(sm.xs + 4u * e, a.x + (ok ? (size_t)row_first * S + e : 0), ok);
        }
    }
    const float *P = a.params + (size_t)(a.policy_lo + pl) * net.row_stride;
    const int nh = (1 + p.Lh) * kH, n_bias = nh + p.n_final;
    const uint32_t dst = sm.bias + 4u * (uint32_t)(buf * kBiasHalf);
    for (int e = et; e < n_bias; e += 256) {
        const float *src = P;
        bool ok = true;
        if (e < nh) src = P + net.b_off[e >> 8] + (e & 255);
        else {
            const int c = e - nh;
            if (p.gpi) src = p.bq + (size_t)pl * p.n_final + c;
            else { ok = c < AD; src = P + net.b_off[L - 1] + (ok ? c : 0); }
        }
        cp_async4(dst + 4u * e, src, ok);
    }
    cp_async_commit_all();
}

// ---- staging (all 256 epilogue threads): the prefetched state rows become the input layer's A operand (bf16, K padded to
// 16 * ks0), in place: every MMA that read the previous operand has completed (the caller saw the last ACC_FULL) ----
__device__ __noinline__ void chain_stage(const TcMulti &m, int g, int et, int r, ChainSmem sm) {
    int jb, pl, tile;
    chain_unit(m, g, jb, pl, tile);
    const TcParams &p = m.job[jb];
    const sfgpi_forward_args &a = p.a;
    const int S = a.net.dims[0], B = a.B;
    cp_async_wait_all();
    epi_bar();
    if (et < 128) {
        const int b = tile * kTM + r;
        const bool pre = 128 * S <= kXsFloats;
        const float *xr = a.x + (size_t)b * S;
        for (int c = 0; c < p.ks0 * 16; c += 8) {
            float xv[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                xv[i] = 0.0f;
                if (c + i < S) xv[i] = pre ? lds32(sm.xs + 4u * (uint32_t)(r * S + c + i)) : (b < B ? xr[c + i] : 0.0f);
            }
            sts128(sm.a + a_chunk_off(r, c), pack_bf16x2(xv[0], xv[1]), pack_bf16x2(xv[2], xv[3]), pack_bf16x2(xv[4], xv[5]),
                   pack_bf16x2(xv[6], xv[7]));
        }
        fence_proxy_async();
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) mbar_arrive(bar_a_ready(sm, j));
    epi_bar();                                       // xs consumed: the next prefetch may overwrite it
}

// ---- hidden / input layer epilogue of one row: 4 quarters of 64 columns, this thread's 32 of each (columns 64 j + 32 g),
// bias + activation -> bf16 -> the next layer's A operand in place, quarter j handed to the MMA warp as soon as it is written.
// Rolled over pairs of quarters (two TMEM loads in flight, half the code of a fully unrolled row).
template <int ACT, bool MASK>
__device__ __forceinline__ void chain_hidden_epilogue(uint32_t t_acc, uint32_t bias, uint32_t A, int r, int group, uint32_t *mask_out,
                                                      const ChainSmem &sm) {
    uint32_t v[2][32];
    tmem_ld32(t_acc + 32u * group, v[0]);
#pragma unroll 1
    for (int jj = 0; jj < 4; jj += 2) {
#pragma unroll
        for (int u2 = 0; u2 < 2; ++u2) {
            const int j = jj + u2, c0 = 64 * j + 32 * group;
            tmem_wait_ld();
            if (u2 == 0) tmem_ld32(t_acc + (uint32_t)(c0 + 64), v[1]);
            else if (jj == 0) tmem_ld32(t_acc + (uint32_t)(c0 + 64), v[0]);
            const uint32_t(&u)[32] = v[u2];
            uint32_t pk[16];
            uint32_t mb = 0;
#pragma unroll
            for (int g4 = 0; g4 < 8; ++g4) {
                const float4 bv = lds128(bias + 4u * (c0 + 4 * g4));
                float h0, h1, h2, h3;
                add_f32x2(__uint_as_float(u[4 * g4]), __uint_as_float(u[4 * g4 + 1]), bv.x, bv.y, h0, h1);
                add_f32x2(__uint_as_float(u[4 * g4 + 2]), __uint_as_float(u[4 * g4 + 3]), bv.z, bv.w, h2, h3);
                if (ACT == SFGPI_ACT_RELU) {
                    if (MASK)
                        mb |= (h0 > 0.f ? 1u : 0u) << (4 * g4) | (h1 > 0.f ? 2u : 0u) << (4 * g4) | (h2 > 0.f ? 4u : 0u) << (4 * g4) |
                              (h3 > 0.f ? 8u : 0u) << (4 * g4);
                    pk[2 * g4] = pack_bf16x2_relu(h0, h1);
                    pk[2 * g4 + 1] = pack_bf16x2_relu(h2, h3);
                } else {
                    if (ACT == SFGPI_ACT_TANH) { h0 = tanhf(h0); h1 = tanhf(h1); h2 = tanhf(h2); h3 = tanhf(h3); }
                    pk[2 * g4] = pack_bf16x2(h0, h1);
                    pk[2 * g4 + 1] = pack_bf16x2(h2, h3);
                }
            }
#pragma unroll
            for (int g4 = 0; g4 < 4; ++g4)
                sts128(A + a_chunk_off(r, c0 + 8 * g4), pk[4 * g4], pk[4 * g4 + 1], pk[4 * g4 + 2], pk[4 * g4 + 3]);
            fence_proxy_async();
            mbar_arrive(bar_a_ready(sm, j));
            if (MASK && mask_out != nullptr) mask_out[c0 >> 5] = mb;      // 1 bit per activation: all the backward needs of a ReLU layer
        }
    }
}

__global__ void __launch_bounds__(kThreadsTc, 1)
mlp_chain_tc_kernel(const __grid_constant__ TcMulti m, const __grid_constant__ TmapSet maps, const int bias_dbl) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    pdl_launch_dependents(SFGPI_TR_FWD);
    if (m.timeline != nullptr && blockIdx.x == 0 && threadIdx.x == 0) m.timeline[255] = clock64();      // kernel entry
    const long long cta_t0 = clock64();
    if (m.timeline != nullptr && threadIdx.x == 0) { unsigned long long gt; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt)); m.timeline[768 + blockIdx.x] = (long long)gt; }

    // ---- carve-up: [A operand 64K][weight ring 8 x 16K][biases 24K][state tile 10K][barriers] ----
    ChainSmem sm;
    sm.a = smem_u32(smem_raw);
    sm.ring = sm.a + kABytes;
    sm.bias = sm.ring + kRing * kStageBytes;
    sm.xs = sm.bias + kBiasFloatsMax * 4;
    sm.bar = sm.xs + kXsFloats * 4;
    const uint32_t holder_addr = sm.bar + 8u * (2 * kRing + 8);

    if (threadIdx.x == 0) {
        for (int s = 0; s < kRing; ++s) { mbar_init(bar_w_full(sm, s), 1); mbar_init(bar_w_empty(sm, s), 1); }
        for (int j = 0; j < 4; ++j) mbar_init(bar_a_ready(sm, j), 256);
        for (int s = 0; s < 2; ++s) { mbar_init(bar_acc_full(sm, s), 1); mbar_init(bar_acc_empty(sm, s), 256); }
        fence_mbar_init();
        for (int j = 0; j < m.n_jobs; ++j) {
            tma_prefetch_desc(&maps.w[j]);
            if (m.job[j].gpi) tma_prefetch_desc(&maps.q[j]);
        }
    }
    if (warp == kMmaWarp) tmem_alloc(holder_addr, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(holder_addr));
    pdl_wait(SFGPI_TR_FWD);                                  // set-up above overlapped the predecessor's tail

    const int unit0 = (int)blockIdx.x, unit_stride = (int)gridDim.x;

    if (warp < 4) {
        // =========================== TMA producers ===========================
        const uint32_t leader = elect_one();
        uint32_t n = 0;
        int tlc = 0;
        for (int g = unit0; g < m.total_pairs; g += unit_stride) {
            int jb, pl, tile;
            chain_unit(m, g, jb, pl, tile);
            const TcParams &p = m.job[jb];
            const int row0 = (p.a.policy_lo + pl) * p.rows_per_policy;
            for (int it = 0; it < p.n_items; ++it) {
                const ItemInfo ii = item_info(p, it);
                const int nblocks = (ii.n_cols + kNB - 1) / kNB;
                const bool folded = ii.kind == 2 && p.gpi;
                const void *tm = folded ? (const void *)&maps.q[jb] : (const void *)&maps.w[jb];
                const int rbase = folded ? pl * p.n_final + ii.row_base : row0 + ii.row_base;
                for (int kb = 0; kb < ii.n_kb; ++kb)
                    for (int nb = 0; nb < nblocks; ++nb, ++n) {
                        const int s = n & (kRing - 1);
                        if ((s & 3) != warp) continue;
                        mbar_wait_warp(bar_w_empty(sm, s), ((n / kRing) & 1) ^ 1);
                        if (warp == 0 && leader) TL_STAMP(2, tlc);
                        mbar_arrive_expect_tx_e(bar_w_full(sm, s), kStageBytes, leader);
                        tma_load_2d_e(sm.ring + s * kStageBytes, tm, bar_w_full(sm, s), kb * kKB, rbase + nb * kNB, leader);
                    }
            }
        }
    } else if (warp == kMmaWarp) {
        // =========================== MMA issuer ===========================
        const uint32_t leader = elect_one();
        uint32_t n = 0, q = 0, f = 0;                       // ring stage counter, item counter, A-operand production counter
        int tlc = 0;
        const uint64_t adesc0 = umma_desc_k_sw128(sm.a), bdesc0 = umma_desc_k_sw128(sm.ring);
        const uint32_t idesc_wide = umma_idesc_bf16(kTM, 256), idesc_full = umma_idesc_bf16(kTM, kNB);
        for (int g = unit0; g < m.total_pairs; g += unit_stride) {
            int jb, pl, tile;
            chain_unit(m, g, jb, pl, tile);
            const TcParams &p = m.job[jb];
            for (int it = 0; it < p.n_items; ++it, ++q) {
                const ItemInfo ii = item_info(p, it);
                const int nblocks = (ii.n_cols + kNB - 1) / kNB;
                const uint32_t idesc_last = umma_idesc_bf16(kTM, (uint32_t)(ii.n_cols - (nblocks - 1) * kNB));
                const uint32_t d_base = tmem_base + (q & 1u) * 256u;
                const bool fresh = ii.kind != 2 || ii.col0 == 0;          // consumes a newly produced A operand
                // the accumulator's previous contents (item q - 2) have been read by the epilogue
                mbar_wait_warp(bar_acc_empty(sm, q & 1), ((q >> 1) & 1) ^ 1);
                tc_fence_after();
                const bool wide = nblocks == 2 && ii.n_cols == 256;
                for (int kb = 0; kb < 4; ++kb) {
                    if (fresh) {                                          // k-block kb <- quarter kb of the producer's epilogue
                        mbar_wait_warp(bar_a_ready(sm, kb), f & 1);
                        tc_fence_after();
                        if (leader && (kb == 0 || kb == 3)) TL_STAMP(1, tlc);
                    }
                    if (kb >= ii.n_kb) continue;                          // (input layer: K fits k-block 0; the phases are consumed all the same)
                    const uint64_t ad = adesc0 + (uint64_t)(kb * ((kTM * 128) >> 4));
                    if (wide) {
                        const int s = n & (kRing - 1);
                        mbar_wait_warp(bar_w_full(sm, s), (n / kRing) & 1);
                        mbar_wait_warp(bar_w_full(sm, s + 1), (n / kRing) & 1);
                        tc_fence_after();
                        const uint64_t bd = bdesc0 + (uint64_t)((s * kStageBytes) >> 4);
                        for (int k16 = 0; k16 < ii.n_k16; ++k16)
                            umma_bf16_e(d_base, ad + 2 * k16, bd + 2 * k16, idesc_wide, (kb | k16) ? 1u : 0u, leader);
                        umma_commit_e(bar_w_empty(sm, s), leader);
                        umma_commit_e(bar_w_empty(sm, s + 1), leader);
                        n += 2;
                        continue;
                    }
                    for (int nb = 0; nb < nblocks; ++nb, ++n) {
                        const int s = n & (kRing - 1);
                        mbar_wait_warp(bar_w_full(sm, s), (n / kRing) & 1);
                        tc_fence_after();
                        const uint32_t idesc = (nb == nblocks - 1) ? idesc_last : idesc_full;
                        const uint64_t bd = bdesc0 + (uint64_t)((s * kStageBytes) >> 4);
                        const uint32_t d = d_base + nb * kNB;
                        for (int k16 = 0; k16 < ii.n_k16; ++k16)
                            umma_bf16_e(d, ad + 2 * k16, bd + 2 * k16, idesc, (kb | k16) ? 1u : 0u, leader);
                        umma_commit_e(bar_w_empty(sm, s), leader);
                    }
                }
                umma_commit_e(bar_acc_full(sm, q & 1), leader);
                if (leader) TL_STAMP(1, tlc);
                if (fresh) ++f;
            }
        }
    } else {
        // =========================== epilogue warps ===========================
        const int group = (warp - kEpiWarp0) >> 2;          // warps 5-8 -> 0, 9-12 -> 1
        const int quad = warp & 3;                          // TMEM lane quadrant this warp may access
        const int r = quad * 32 + lane;                     // row inside the tile == TMEM lane
        const int et = threadIdx.x - kEpiWarp0 * 32;        // 0..255
        const uint32_t t_lane0 = tmem_base + ((uint32_t)(quad * 32) << 16);
        uint32_t q = 0;
        bool store_pending = false;                          // a bulk store of the A operand may still be reading it (uniform)
        int tlc = 0;
        const int tl_role = (et == 0) ? 0 : ((et == 128) ? 3 : -1);
#define TL_EPI() do { if (tl_role >= 0) TL_STAMP(tl_role, tlc); } while (0)
        TL_EPI();
        int ubuf = 0;                                        // bias buffer of the current unit
        bool need_stage = unit0 < m.total_pairs;
        if (need_stage) chain_prefetch(m, unit0, 0, et, sm);
        for (int g = unit0; g < m.total_pairs; g += unit_stride) {
            if (need_stage) {                                // first unit, or large bias sets (one buffer: no overlap with the previous unit)
                if (store_pending) { if (et == 0) bulk_wait_read0(); store_pending = false; }
                chain_stage(m, g, et, r, sm);
                need_stage = false;
                TL_EPI();
            }
            int jb, pl, tile;
            chain_unit(m, g, jb, pl, tile);
            const TcParams &p = m.job[jb];
            const sfgpi_forward_args &a = p.a;
            const sfgpi_net_desc &net = a.net;
            const int B = a.B, A_ = net.n_actions, D = net.n_features, AD = A_ * D;
            const int b = tile * kTM + r;
            const bool row_ok = b < B;
            const bool has_next = g + unit_stride < m.total_pairs;
            const bool saving = a.acts_bf16_out != nullptr;
            const uint32_t bias_u = sm.bias + 4u * (uint32_t)(ubuf * kBiasHalf);
            // every epilogue of the previous unit is done: its bias buffer (the next unit's, when double-buffered) and xs are free
            if (has_next && bias_dbl) chain_prefetch(m, g + unit_stride, ubuf ^ 1, et, sm);
            int sel_base = -(1 << 30);
            if (a.sel_out != nullptr && row_ok) {
                const int sidx = a.sel_actions ? (int)a.sel_actions[b] : (int)key_index(a.sel_keys[(size_t)pl * a.sel_key_stride + b]);
                sel_base = sidx * D;
            }
#pragma unroll 1
            for (int it = 0; it < p.n_items; ++it, ++q) {
                const ItemInfo ii = item_info(p, it);
                const uint32_t t_acc = t_lane0 + (q & 1u) * 256u;
                mbar_wait(bar_acc_full(sm, q & 1), (q >> 1) & 1);
                tc_fence_after();
                TL_EPI();
                if (ii.kind != 2) {
                    // ------ input / hidden layer ------
                    const uint32_t bias = bias_u + 4u * (uint32_t)(it * kH);
                    const int act = net.acts[it];
                    uint32_t *mask_out = (a.relu_mask_out && row_ok)
                        ? reinterpret_cast<uint32_t *>(a.relu_mask_out) + (((size_t)it * a.n_pol + pl) * B + b) * 8 : nullptr;
                    if (store_pending) {                     // the previous layer's bulk store has finished reading the operand
                        if (et == 0) bulk_wait_read0();
                        store_pending = false;
                        epi_bar();
                    }
                    if (act == SFGPI_ACT_RELU) {
                        if (a.relu_mask_out) chain_hidden_epilogue<SFGPI_ACT_RELU, true>(t_acc, bias, sm.a, r, group, mask_out, sm);
                        else chain_hidden_epilogue<SFGPI_ACT_RELU, false>(t_acc, bias, sm.a, r, group, nullptr, sm);
                    } else if (act == SFGPI_ACT_NONE) chain_hidden_epilogue<SFGPI_ACT_NONE, false>(t_acc, bias, sm.a, r, group, nullptr, sm);
                    else chain_hidden_epilogue<SFGPI_ACT_TANH, false>(t_acc, bias, sm.a, r, group, nullptr, sm);
                    tc_fence_before();
                    mbar_arrive(bar_acc_empty(sm, q & 1));
                    if (saving) {                            // the complete bf16 tile in the A operand IS the saved activation block
                        epi_bar();
                        if (et == 0) {
#pragma unroll
                            for (int kb = 0; kb < kH / kKB; ++kb)
                                tma_store_3d(&maps.acts[jb], sm.a + kb * (kTM * 128), kb * kKB, tile * kTM, it * a.n_pol + pl);
                            bulk_commit();
                        }
                        store_pending = true;
                    }
                } else {
                    // ------ output layer chunk ------
                    if (it == p.n_items - 1 && has_next && bias_dbl) {       // every MMA of this tile has completed: the operand is free
                        if (store_pending) { if (et == 0) bulk_wait_read0(); store_pending = false; }
                        chain_stage(m, g + unit_stride, et, r, sm);          // the next input layer runs under this epilogue
                    }
                    const uint32_t bias = bias_u + 4u * (uint32_t)((1 + p.Lh) * kH);       // bias of folded / psi column 0
                    const int n_cols_it = ii.n_cols, col0_it = ii.col0, n_pol_job = a.n_pol;
                    if (p.gpi) {
                        const int nw = p.nw, wblk = gpi_wblock(nw), ncol = gpi_ncols(nw, A_);
                        const uint32_t kstep = a.w_diag ? 0u : (uint32_t)B;
                        long long *ka = a.key_action ? reinterpret_cast<long long *>(a.key_action) + (a.w_diag ? (size_t)pl * B : 0) + b : nullptr;
                        long long *kt = a.key_task ? reinterpret_cast<long long *>(a.key_task) + (a.w_diag ? (size_t)pl * B : 0) + b : nullptr;
                        float *q_row = (a.q_out != nullptr && row_ok) ? a.q_out + ((size_t)b * n_pol_job + pl) * A_ : nullptr;
                        const uint32_t tid_ = (uint32_t)(a.task_base + pl);
                        const int c_hi = min(col0_it + n_cols_it, ncol);
                        // each group scans one 128-column half of the chunk (1-3 reward vectors: plain order, group 0 scans it all)
                        const int cb = wblk > 1 ? col0_it + group * 128 : (group == 0 ? col0_it : c_hi);
                        const int ce = wblk > 1 ? min(cb + 128, c_hi) : c_hi;
                        if (cb < ce) {
                            if (wblk == 8) gpi_scan_rolled<8>(t_acc, bias, col0_it, cb, ce, A_, nw, ka, kt, kstep, row_ok, tid_, q_row);
                            else if (wblk == 4) gpi_scan_rolled<4>(t_acc, bias, col0_it, cb, ce, A_, nw, ka, kt, kstep, row_ok, tid_, q_row);
                            else gpi_scan_rolled<1>(t_acc, bias, col0_it, cb, ce, A_, nw, ka, kt, kstep, row_ok, tid_, q_row);
                        }
                    } else {
                        float *const psi_out = a.psi_out, *const sel_out = a.sel_out;
                        const int sb = sel_base;
#pragma unroll 1
                        for (int c0 = group * 8; c0 < n_cols_it; c0 += 16) {
                            uint32_t v[8];
                            tmem_ld8(t_acc + (uint32_t)c0, v);
                            const int colb = col0_it + c0;
                            const float4 b0 = lds128(bias + 4u * colb), b1 = lds128(bias + 4u * (colb + 4));
                            const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
                            tmem_wait_ld();
                            float val[8];
#pragma unroll
                            for (int i = 0; i < 8; ++i) val[i] = __uint_as_float(v[i]) + bv[i];
                            if (row_ok) {
                                if (psi_out != nullptr) {
                                    float *po = psi_out + ((size_t)b * n_pol_job + pl) * AD + colb;
                                    if ((AD & 3) == 0) {
                                        if (colb < AD) *reinterpret_cast<float4 *>(po) = make_float4(val[0], val[1], val[2], val[3]);
                                        if (colb + 4 < AD) *reinterpret_cast<float4 *>(po + 4) = make_float4(val[4], val[5], val[6], val[7]);
                                    } else {
#pragma unroll
                                        for (int i = 0; i < 8; ++i)
                                            if (colb + i < AD) po[i] = val[i];
                                    }
                                }
                                if ((unsigned)(colb + 7 - sb) < (unsigned)(D + 7)) {
                                    float *so = sel_out + ((size_t)pl * B + b) * D;
#pragma unroll
                                    for (int i = 0; i < 8; ++i) {
                                        const unsigned off = (unsigned)(colb + i - sb);
                                        if (off < (unsigned)D) so[off] = val[i];
                                    }
                                }
                            }
                        }
                    }
                    tc_fence_before();
                    mbar_arrive(bar_acc_empty(sm, q & 1));
                }
                TL_EPI();
            }
            if (has_next) {
                if (!bias_dbl) { chain_prefetch(m, g + unit_stride, 0, et, sm); need_stage = true; }
                else ubuf ^= 1;
            }
        }
        if (et == 0) bulk_wait0();                           // outstanding activation stores complete before the CTA retires
    }

    // ---- teardown ----
    if (m.timeline != nullptr && threadIdx.x == 0) {
        m.timeline[512 + blockIdx.x] = clock64() - cta_t0;   // per-CTA busy cycles
        unsigned long long gt; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt)); m.timeline[1024 + blockIdx.x] = (long long)gt;
    }
    tc_fence_before();
    __syncthreads();
    if (warp == kMmaWarp) {
        __syncwarp();
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
    trace_exit(SFGPI_TR_FWD);
}

// The chain kernel covers every cta_group::1 launch except fp32 activation saves and staged keys (callers of those get the
// ping-pong kernel).
bool forward_chain_supported(const TcMulti &m) {
    for (int j = 0; j < m.n_jobs; ++j) {
        const sfgpi_forward_args &a = m.job[j].a;
        for (int l = 0; l < SFGPI_MAX_LAYERS; ++l)
            if (a.acts_out[l] != nullptr) return false;
    }
    return true;
}

int launch_forward_chain(TcMulti &m, const TmapSet &maps, int total_tiles, cudaStream_t st) {
    trace_bind();
    m.total_pairs = 0;
    m.paired = 0;
    m.sched = 0;
    int bias_dbl = 1;
    for (int j = 0; j < m.n_jobs; ++j) {
        TcParams &p = m.job[j];
        p.paired = 0;
        p.pairs_per_policy = p.tiles_per_policy;
        p.total_pairs = p.tiles_per_policy * p.a.n_pol;
        m.pair_start[j] = m.total_pairs;
        m.total_pairs += p.total_pairs;
        if ((1 + p.Lh) * kH + p.n_final > kBiasHalf) bias_dbl = 0;
    }
    for (int j = m.n_jobs; j <= kMaxJobs; ++j) m.pair_start[j] = m.total_pairs;
    const int smem_bytes = kABytes + kRing * kStageBytes + kBiasFloatsMax * 4 + kXsFloats * 4 + 256;
    static bool cfg = false;
    if (!cfg) {
        cudaFuncSetAttribute(mlp_chain_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
        cfg = true;
    }
    const int grid = total_tiles < 148 ? total_tiles : 148;
    launch_pdl(mlp_chain_tc_kernel, dim3(grid), dim3(kThreadsTc), smem_bytes, st, m, maps, bias_dbl);
    return grid;
}

}  // namespace tc
}  // namespace sfgpi
