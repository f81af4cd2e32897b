// Backward of the psi MLP on the 5th-gen tensor cores (bf16 operands, fp32 accumulation in TMEM).  Two kernels:
//
// (1) mlp_dgrad_tc_kernel -- the dZ chain dZ_{L-1} -> dZ_{L-2} -> ... -> dZ_0 for one 128-row tile per slot, same persistent
//     warp-specialised structure as the forward kernel (4 TMA producer warps, 1 MMA-issuer warp, 2 x 4 epilogue warps, two
//     tiles ping-ponging on 2 x 256 TMEM columns).  dA_{l-1}[b][k] = sum_n dZ_l[b][n] W_l[n][k]: A = dZ_l is K-major in
//     shared memory exactly like a forward activation; B = W_l is read from the SAME bf16 shadow as the forward, as an
//     MN-major operand (its rows are the reduction index), so no transposed copy of the weights exists.  The last layer's
//     dZ is D-sparse in the train step (sfdqn.py:334-335: only psi(s)[b, a_b, :] is in the loss); the epilogue threads expand
//     d_out[b][D] into the dense row on the fly.  Autograd through PackedSFLibrary.psi passes a dense dZ instead (actions
//     NULL, d_out [B][n_pol][A*D]): the same threads read it and convert it to bf16 (the kDense instantiation).  Each epilogue multiplies by the activation derivative (from the bf16 activations the forward
//     saved), writes the next A operand in place and the row-major bf16 dZ_l to HBM for the wgrad kernel.
//
// (2) mlp_wgrad_tc_kernel -- dW_l[n][k] = sum_b dZ_l[b][n] in_l[b][k] and db_l[n] = sum_b dZ_l[b][n], split-K over the batch.
//     Both operands are MN-major (the reduction index b is the row of the row-major [B][width] tensors), TMA-loaded as
//     {64 x 64} 128B-swizzled boxes straight from the tensors the forward / dgrad kernels wrote.  One CTA = (policy, layer,
//     128-row tile of dW_l, batch split): acc[128][256] in TMEM, plus 64 auxiliary columns against xo = [x | 1 | 0..] that
//     yield the bias gradient (the ones column) and, for layer 0, dW_0 itself.  fp32 partials go to grad_part, which the
//     Adam kernel sums in a fixed order (deterministic).
#include "tc_common.cuh"
#include <stdlib.h>

namespace sfgpi {
namespace tc {

constexpr int kNB = 128;                            // N columns per dgrad weight stage
constexpr int kStageBytes = kNB * kKB * 2;          // 16 KB = two {64 x 64} boxes
constexpr int kBoxBytes = 64 * 64 * 2;              // 8 KB
constexpr int kNStage = 4;
constexpr int kABytes = kTM * kH * 2;               // 64 KB per tile slot
constexpr int kThreadsDg = 416;                     // 4 producer warps + 1 MMA warp + 2 x 4 epilogue warps
constexpr int kMmaWarp = 4, kEpiWarp0 = 5;
constexpr int kXoCols = 64;                         // width of the auxiliary operand xo = [x | 1 | 0 ...]

struct DgParams {
    sfgpi_net_desc net;
    int policy_lo, n_pol, B;
    const long long *actions;        // [B]
    const float *d_out;              // [n_pol][B][D]; dense (kDense): [B][n_pol][AD]
    const __nv_bfloat16 *acts;       // [L-1][n_pol][B][256]
    const uint32_t *masks;           // [L-1][n_pol][B][8] ReLU sign bits written by the forward (NULL: derive from acts)
    __nv_bfloat16 *dz;               // [L-1][n_pol][B][256]
    __nv_bfloat16 *dzo;              // [n_pol][B][ADp]
    int rows_per_policy, L, AD, AD16, ADp, n_chunks, n_items;
    int tiles_per_policy, pairs_per_policy, total_pairs, paired;
    int n_main;                      // CTAs running the dgrad tile loop; CTAs [n_main, gridDim.x) are riders (see ex)
};

// Rolled form of dgrad_epilogue for the hot shapes (no activation, or ReLU gated by the forward's mask words), activation at RUN
// time: one copy of the code for every layer.  The fully unrolled template cost 17 k cycles on a CTA's first call (instruction
// fetch: ~150 cycles per 128-byte line of straight-line code) against 5.5 k warm -- and with one tile per CTA there are only three
// calls.  Body = two 32-column chunks (two TMEM loads in flight), looped over n_pairs.  Same arithmetic (bit-identical).
__device__ __forceinline__ void dgrad_epilogue_rolled(uint32_t t_lane, uint32_t Arow, int r, bool row_ok, const uint32_t *mask_row, bool relu,
                                                      int cbase, int n_pairs) {
    uint32_t v[2][32];
    uint4 mq = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
    if (relu && row_ok) mq = __ldg(reinterpret_cast<const uint4 *>(mask_row + (cbase >> 5)));
    if (!row_ok) mq = make_uint4(0u, 0u, 0u, 0u);              // rows past the batch contribute zeros
    tmem_ld32(t_lane + cbase, v[0]);
#pragma unroll 1
    for (int jp = 0; jp < n_pairs; ++jp) {
        const uint32_t mlo = jp ? mq.z : mq.x, mhi = jp ? mq.w : mq.y;
#pragma unroll
        for (int u2 = 0; u2 < 2; ++u2) {
            const int c0 = cbase + (2 * jp + u2) * 32;
            tmem_wait_ld();
            if (u2 == 0) tmem_ld32(t_lane + c0 + 32, v[1]);
            else if (jp + 1 < n_pairs) tmem_ld32(t_lane + c0 + 32, v[0]);
            const uint32_t(&u)[32] = v[u2];
            const uint32_t mword = u2 ? mhi : mlo;
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                float hv[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) hv[i] = ((mword >> (8 * g + i)) & 1u) ? __uint_as_float(u[8 * g + i]) : 0.0f;      // threshold_backward
                sts128(Arow + a_chunk_off(r, c0 + 8 * g), pack_bf16x2(hv[0], hv[1]), pack_bf16x2(hv[2], hv[3]), pack_bf16x2(hv[4], hv[5]),
                       pack_bf16x2(hv[6], hv[7]));
            }
        }
    }
}

// developer aid (env SFGPI_TIMELINE): clock64 stamps of CTA 0 -- [0, 32) epilogue thread 0, [32, 64) MMA issuer, [64] entry, [65] exit
static __device__ long long g_dg_tl[66];
static __device__ int g_dg_tl_on = 0;
#define DG_STAMP(base, cnt) do { if (g_dg_tl_on && blockIdx.x == 0 && (cnt) < 32) g_dg_tl[(base) + (cnt)++] = clock64(); } while (0)

struct DgItem { int row_base, K; };                 // shadow row of the first reduction index, reduction length (mult. of 16)

__device__ __forceinline__ DgItem dg_item(const DgParams &p, int it) {
    DgItem r;
    if (it < p.n_chunks) { r.row_base = (p.L - 1) * kH + it * 256; r.K = min(256, p.AD16 - it * 256); }
    else { const int l = p.L - 2 - (it - p.n_chunks); r.row_base = l * kH; r.K = kH; }
    return r;
}

// Expanded dense chunk c of this row's dZ_{L-1}: columns [256c, 256c+256) of a row that is zero except d_out[0..D) at
// [sel, sel+D) -- or, kDense, the row drow[0..AD) itself, zero past AD.  Written to the A slot (K-major SW128) and, as the
// wgrad operand, to dzo (row-major bf16).
template <bool kDense>
__device__ __forceinline__ void build_dzo_chunk(const DgParams &p, int c, uint32_t Arow, int r, bool row_ok, int sel,
                                                const float *drow, __nv_bfloat16 *dzo_row, int j0, int jstep) {
    const int D = p.net.n_features;
    const int cend = min(256, p.ADp - c * 256);
#pragma unroll 1
    for (int j = j0; j * 8 < cend; j += jstep) {
        const int col0 = c * 256 + j * 8;
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            if constexpr (kDense) {
                v[i] = (row_ok && col0 + i < p.AD) ? drow[col0 + i] : 0.0f;
            } else {
                const unsigned off = (unsigned)(col0 + i - sel);
                v[i] = (row_ok && off < (unsigned)D) ? drow[off] : 0.0f;
            }
        }
        const uint32_t q0 = pack_bf16x2(v[0], v[1]), q1 = pack_bf16x2(v[2], v[3]), q2 = pack_bf16x2(v[4], v[5]),
                       q3 = pack_bf16x2(v[6], v[7]);
        sts128(Arow + a_chunk_off(r, j * 8), q0, q1, q2, q3);      // the tile is stored to dzo by TMA (see the epilogue)
    }
}

// dZ_lo = acc * act'(act_lo): 256 accumulator columns of one row -> bf16 -> next A operand (in place) + HBM row.
// dZ_lo = acc * act'(act_lo) for NCH 32-column chunks starting at cbase: bf16 -> A slot (next layer's operand AND the tile that a
// bulk tensor store writes to dz[lo]).  ReLU: the sign bits come from the forward's mask words (16 bytes per thread);
// tanh: from the saved activations (slow path: 16-byte loads at a 512-byte pitch).
template <int ACT, int NCH>
__device__ __forceinline__ void dgrad_epilogue(uint32_t t_lane, uint32_t Arow, int r, bool row_ok, const uint4 *act_row,
                                               const uint32_t *mask_row, int cbase) {
    uint32_t v[2][32];
    uint4 am[2][4] = {};
    uint32_t mw[4] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu};
    const bool use_mask = (ACT == SFGPI_ACT_RELU) && mask_row != nullptr;
    if (ACT == SFGPI_ACT_RELU && use_mask && row_ok) {
        const uint4 q = __ldg(reinterpret_cast<const uint4 *>(mask_row + (cbase >> 5)));
        mw[0] = q.x; mw[1] = q.y; mw[2] = q.z; mw[3] = q.w;
    }
    const bool need_vals = (ACT == SFGPI_ACT_TANH) || (ACT == SFGPI_ACT_RELU && !use_mask);
    if (need_vals && row_ok) {
#pragma unroll
        for (int g = 0; g < 4; ++g) am[0][g] = __ldg(act_row + (cbase >> 3) + g);
    }
    tmem_ld32(t_lane + cbase, v[0]);
#pragma unroll
    for (int cb = 0; cb < NCH; ++cb) {
        const int c0 = cbase + cb * 32;
        tmem_wait_ld();
        if (cb + 1 < NCH) {
            tmem_ld32(t_lane + c0 + 32, v[(cb + 1) & 1]);
            if (need_vals && row_ok) {
#pragma unroll
                for (int g = 0; g < 4; ++g) am[(cb + 1) & 1][g] = __ldg(act_row + ((c0 + 32) >> 3) + g);
            }
        }
        const uint32_t(&u)[32] = v[cb & 1];
        const uint32_t mword = mw[cb & 3];
#pragma unroll
        for (int g = 0; g < 4; ++g) {
            const uint4 aq = am[cb & 1][g];
            const uint32_t aw[4] = {aq.x, aq.y, aq.z, aq.w};
            float h[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                float gv = row_ok ? __uint_as_float(u[8 * g + i]) : 0.0f;
                if (ACT == SFGPI_ACT_RELU && use_mask) {
                    gv = ((mword >> (8 * g + i)) & 1u) ? gv : 0.0f;                                   // threshold_backward
                } else if (ACT != SFGPI_ACT_NONE) {
                    const uint32_t ab = (i & 1) ? (aw[i >> 1] >> 16) : (aw[i >> 1] & 0xFFFFu);      // bf16 bits of act[col]
                    if (ACT == SFGPI_ACT_RELU) gv = ((short)ab > 0) ? gv : 0.0f;
                    else { const float av = __uint_as_float(ab << 16); gv *= (1.0f - av * av); }      // tanh_backward
                }
                h[i] = gv;
            }
            sts128(Arow + a_chunk_off(r, c0 + 8 * g), pack_bf16x2(h[0], h[1]), pack_bf16x2(h[2], h[3]), pack_bf16x2(h[4], h[5]),
                   pack_bf16x2(h[6], h[7]));
        }
    }
}

template <bool kDense>
__global__ void __launch_bounds__(kThreadsDg, 1)
mlp_dgrad_tc_kernel(const __grid_constant__ DgParams p, const __grid_constant__ CUtensorMap tmap_w,
                    const __grid_constant__ CUtensorMap tmap_dz, const __grid_constant__ CUtensorMap tmap_dzo,
                    const __grid_constant__ sfgpi_td_args ex, int ex_nclu) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    pdl_launch_dependents(SFGPI_TR_DGRAD);
    if (g_dg_tl_on && blockIdx.x == 0 && threadIdx.x == 0) g_dg_tl[64] = clock64();
    if ((int)blockIdx.x >= p.n_main) {
        // Rider CTAs: the TSF expand of the TD step (one policy each).  It depends only on the TD kernel -- this launch's
        // predecessor -- and only the Adam kernel consumes it, so instead of a launch of its own on the step's dependent chain
        // it runs here, on SMs the dgrad tile loop leaves idle, concurrently with the dgrad CTAs.
        pdl_wait();
        tsf_expand_cta(ex, (int)blockIdx.x - p.n_main, ex_nclu, reinterpret_cast<float *>(smem_raw), threadIdx.x, kThreadsDg);
        return;
    }
    const sfgpi_net_desc &net = p.net;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    // ---- carve-up: [A slot X 64K][A slot Y 64K][weight ring 4 x 16K][barriers] ----
    const uint32_t sbase = smem_u32(smem_raw);
    const uint32_t W_addr = sbase + 2 * kABytes;
    const uint32_t bar0 = W_addr + kNStage * kStageBytes;
    // one-tile mode (p.paired == 0): slot Y's 64 KB are 4 more weight stages and both epilogue groups share the tile (see the
    // forward kernel).  Stage s lives at W_addr + (s < 4 ? s : s - 8) * 16 KB.
    const int ns_log = p.paired ? 2 : 3, ns_mask = (1 << ns_log) - 1;
    auto W_FULL = [&](int s) { return bar0 + 8u * s; };
    auto W_EMPTY = [&](int s) { return bar0 + 8u * (8 + s); };
    auto SLOT_READY = [&](int s) { return bar0 + 8u * (16 + s); };
    auto ACC_FULL = [&](int s) { return bar0 + 8u * (18 + s); };
    auto stage_off = [&](int s) { return (s - ((s & 4) << 1)) * kStageBytes; };
    const uint32_t holder_addr = bar0 + 8u * 20;

    if (threadIdx.x == 0) {
        for (int s = 0; s < 8; ++s) { mbar_init(W_FULL(s), 1); mbar_init(W_EMPTY(s), 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(SLOT_READY(s), 256); mbar_init(ACC_FULL(s), 1); }
        fence_mbar_init();
        tma_prefetch_desc(&tmap_w);
    }
    if (warp == kMmaWarp) tmem_alloc(holder_addr, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(holder_addr));
    pdl_wait(SFGPI_TR_DGRAD);

    const int B = p.B, D = net.n_features;

    if (warp < kNStage) {
        // =========================== TMA producers (ring stage s is owned by producer warp s) ===========================
        {
            const uint32_t leader = elect_one();             // whole-warp loop, elected issue (tc_common.cuh)
            uint32_t n = 0;
            for (int pair = blockIdx.x; pair < p.total_pairs; pair += p.n_main) {
                const int pl = pair / p.pairs_per_policy, pip = pair - pl * p.pairs_per_policy;
                const int row0 = (p.policy_lo + pl) * p.rows_per_policy;
                const bool has_y = p.paired && (2 * pip + 1 < p.tiles_per_policy);
                for (int it = 0; it < p.n_items; ++it) {
                    const DgItem ii = dg_item(p, it);
                    const int n_kb = (ii.K + kKB - 1) / kKB;
                    for (int slot = 0; slot < (has_y ? 2 : 1); ++slot)
                        for (int kb = 0; kb < n_kb; ++kb)
                            for (int nb = 0; nb < kH / kNB; ++nb, ++n) {
                                const int s = n & ns_mask;
                                if ((s & 3) != warp) continue;
                                mbar_wait_warp(W_EMPTY(s), ((n >> ns_log) & 1) ^ 1);
                                mbar_arrive_expect_tx_e(W_FULL(s), kStageBytes, leader);
                                const int wrow = row0 + ii.row_base + kb * kKB;       // 64 reduction rows of W
                                tma_load_2d_e(W_addr + stage_off(s), &tmap_w, W_FULL(s), nb * kNB, wrow, leader);
                                tma_load_2d_e(W_addr + stage_off(s) + kBoxBytes, &tmap_w, W_FULL(s), nb * kNB + 64, wrow, leader);
                            }
                }
            }
        }
    } else if (warp == kMmaWarp) {
        // =========================== MMA issuer ===========================
        {
            const uint32_t leader = elect_one();
            uint32_t n = 0, ready_cnt[2] = {0, 0};
            int tlm = 0;
            const uint64_t adesc_x = umma_desc_k_sw128(sbase), adesc_y = umma_desc_k_sw128(sbase + kABytes);
            const uint64_t bdesc0 = umma_desc_mn_sw128(W_addr, kBoxBytes);
            const uint32_t idesc = umma_idesc_bf16_major(kTM, kNB, 0u, 1u);
            for (int pair = blockIdx.x; pair < p.total_pairs; pair += p.n_main) {
                const int pip = pair % p.pairs_per_policy;
                const bool has_y = p.paired && (2 * pip + 1 < p.tiles_per_policy);
                for (int it = 0; it < p.n_items; ++it) {
                    const DgItem ii = dg_item(p, it);
                    const int n_kb = (ii.K + kKB - 1) / kKB;
                    const bool fresh = (it == 0) || (it >= p.n_chunks);          // output-layer chunks 1.. accumulate
                    for (int slot = 0; slot < (has_y ? 2 : 1); ++slot) {
                        mbar_wait_warp(SLOT_READY(slot), ready_cnt[slot] & 1);
                        ++ready_cnt[slot];
                        tc_fence_after();
                        if (leader) DG_STAMP(32, tlm);
                        const uint32_t d_base = tmem_base + (uint32_t)slot * 256u;
                        // N = 256 MMAs over a pair of adjacent ring stages (four 64-column blocks, LBO apart): half the instructions
                        const bool wide = !(n & 1);
                        const uint32_t idesc_wide = umma_idesc_bf16_major(kTM, 256, 0u, 1u);
                        for (int kb = 0; kb < n_kb; ++kb) {
                            const uint64_t ad = (slot ? adesc_y : adesc_x) + (uint64_t)(kb * ((kTM * 128) >> 4));
                            const int n_k16 = min(4, (ii.K - kb * kKB) >> 4);
                            const uint32_t acc0 = (!fresh || kb) ? 1u : 0u;
                            if (wide) {
                                const int s = n & ns_mask;
                                mbar_wait_warp(W_FULL(s), (n >> ns_log) & 1);
                                mbar_wait_warp(W_FULL(s + 1), (n >> ns_log) & 1);
                                tc_fence_after();
                                const uint64_t bd = bdesc0 + (uint64_t)(int64_t)(stage_off(s) >> 4);
                                if (n_k16 == 4) {
                                    umma_bf16_e(d_base, ad, bd, idesc_wide, acc0, leader);
                                    umma_bf16_e(d_base, ad + 2, bd + 128, idesc_wide, 1u, leader);
                                    umma_bf16_e(d_base, ad + 4, bd + 256, idesc_wide, 1u, leader);
                                    umma_bf16_e(d_base, ad + 6, bd + 384, idesc_wide, 1u, leader);
                                } else {
                                    for (int k16 = 0; k16 < n_k16; ++k16)
                                        umma_bf16_e(d_base, ad + 2 * k16, bd + 128 * k16, idesc_wide, (acc0 || k16) ? 1u : 0u, leader);
                                }
                                umma_commit_e(W_EMPTY(s), leader);
                                umma_commit_e(W_EMPTY(s + 1), leader);
                                n += 2;
                                continue;
                            }
                            for (int nb = 0; nb < kH / kNB; ++nb, ++n) {
                                const int s = n & ns_mask;
                                mbar_wait_warp(W_FULL(s), (n >> ns_log) & 1);
                                tc_fence_after();
                                const uint64_t bd = bdesc0 + (uint64_t)(int64_t)(stage_off(s) >> 4);
                                const uint32_t d = d_base + nb * kNB;
                                if (n_k16 == 4) {
                                    umma_bf16_e(d, ad, bd, idesc, acc0, leader);
                                    umma_bf16_e(d, ad + 2, bd + 128, idesc, 1u, leader);
                                    umma_bf16_e(d, ad + 4, bd + 256, idesc, 1u, leader);
                                    umma_bf16_e(d, ad + 6, bd + 384, idesc, 1u, leader);
                                } else {
                                    for (int k16 = 0; k16 < n_k16; ++k16)
                                        umma_bf16_e(d, ad + 2 * k16, bd + 128 * k16, idesc, (acc0 || k16) ? 1u : 0u, leader);
                                }
                                umma_commit_e(W_EMPTY(s), leader);
                            }
                        }
                        umma_commit_e(ACC_FULL(slot), leader);
                        if (leader) DG_STAMP(32, tlm);
                    }
                }
            }
        }
    } else {
        // =========================== epilogue groups ===========================
        // Both groups (8 warps) drain ONE accumulator at a time, each half of the columns, alternating between the two tile
        // slots -- same reasoning as in the forward kernel (a TMEM drain needs 8 warps in flight to run at its 2048-cycle floor).
        const int group = (warp - kEpiWarp0) >> 2;
        const int quad = warp & 3;
        const int r = quad * 32 + lane;
        const int et = threadIdx.x - kEpiWarp0 * 32;
        const uint32_t t_lane0 = tmem_base + ((uint32_t)(quad * 32) << 16);
        uint32_t full_cnt[2] = {0, 0};
        int tle = 0;
#define DG_EPI() do { if (et == 0) DG_STAMP(0, tle); } while (0)
        DG_EPI();
        // Every tile this kernel produces (the dense dZ_{L-1} chunk, each dZ_lo) is left in the A slot in TMA's swizzled box
        // layout and written to HBM by ONE thread with bulk tensor stores; see the forward kernel for the reasoning and the
        // guard protocol (a slot is rewritten only after its pending store has finished reading it).
        bool store_pending[2] = {false, false};
        auto a_slot_guard = [&](bool all) {
            if (et == 0) { if (all) bulk_wait_read0(); else bulk_wait_read1(); }
            asm volatile("bar.sync 1, 256;" ::: "memory");
        };
        auto guard_slot = [&](int slot) {
            if (store_pending[slot]) { a_slot_guard(!store_pending[slot ^ 1]); store_pending[slot] = false; }
        };

        for (int pair = blockIdx.x; pair < p.total_pairs; pair += p.n_main) {
            const int pl = pair / p.pairs_per_policy, pip = pair - pl * p.pairs_per_policy;
            const int n_slots = (p.paired && (2 * pip + 1 < p.tiles_per_policy)) ? 2 : 1;
            int bs[2];
            // tile complete in shared memory (fenced by its writers) -> barrier, one thread stores nbox 64-column boxes
            auto store_tile = [&](const CUtensorMap *tm, int slot, int nbox, int col0, int slab) {
                asm volatile("bar.sync 1, 256;" ::: "memory");
                if (et == 0) {
                    const uint32_t Arow = sbase + (uint32_t)slot * kABytes;
                    const int row0 = (p.paired ? 2 * pip + slot : pip) * kTM;
                    for (int j = 0; j < nbox; ++j) tma_store_3d(tm, Arow + j * (kTM * 128), col0 + j * kKB, row0, slab);
                    bulk_commit();
                }
                store_pending[slot] = true;
            };
#pragma unroll 1
            for (int slot = 0; slot < n_slots; ++slot) {
                const int b = (p.paired ? 2 * pip + slot : pip) * kTM + r;
                bs[slot] = b;
                const bool row_ok = b < B;
                const size_t prow = (size_t)pl * B + (row_ok ? b : 0);
                const int sel = (!kDense && row_ok) ? (int)p.actions[b] * D : 0;
                const float *drow = kDense ? p.d_out + ((size_t)(row_ok ? b : 0) * p.n_pol + pl) * p.AD : p.d_out + prow * D;
                guard_slot(slot);
                build_dzo_chunk<kDense>(p, 0, sbase + (uint32_t)slot * kABytes, r, row_ok, sel, drow, p.dzo + prow * p.ADp,
                                        group, 2);
                fence_proxy_async();
                mbar_arrive(SLOT_READY(slot));
                store_tile(&tmap_dzo, slot, (min(256, p.ADp) + kKB - 1) / kKB, 0, pl);
                DG_EPI();
            }

            for (int it = 0; it < p.n_items; ++it) {
#pragma unroll 1
                for (int slot = 0; slot < n_slots; ++slot) {
                    const int b = bs[slot];
                    const bool row_ok = b < B;
                    const uint32_t t_lane = t_lane0 + (uint32_t)slot * 256u;
                    const uint32_t Arow = sbase + (uint32_t)slot * kABytes;
                    mbar_wait(ACC_FULL(slot), full_cnt[slot] & 1);
                    ++full_cnt[slot];
                    tc_fence_after();
                    DG_EPI();
                    guard_slot(slot);
                    if (it + 1 < p.n_chunks) {                   // more output-layer chunks: refill the A slot
                        const size_t prow = (size_t)pl * B + (row_ok ? b : 0);
                        const int sel = (!kDense && row_ok) ? (int)p.actions[b] * D : 0;
                        const float *drow = kDense ? p.d_out + ((size_t)(row_ok ? b : 0) * p.n_pol + pl) * p.AD : p.d_out + prow * D;
                        build_dzo_chunk<kDense>(p, it + 1, Arow, r, row_ok, sel, drow, p.dzo + prow * p.ADp, group, 2);
                        fence_proxy_async();
                        mbar_arrive(SLOT_READY(slot));
                        store_tile(&tmap_dzo, slot, (min(256, p.ADp - (it + 1) * 256) + kKB - 1) / kKB, (it + 1) * 256, pl);
                        continue;
                    }
                    const int lo = (it < p.n_chunks) ? p.L - 2 : p.L - 3 - (it - p.n_chunks);    // produces dZ_lo
                    const int act = net.acts[lo];
                    const size_t rowi = ((size_t)lo * p.n_pol + pl) * B + (row_ok ? b : 0);
                    const uint4 *act_row = reinterpret_cast<const uint4 *>(p.acts + rowi * kH);
                    const uint32_t *mask_row = p.masks ? p.masks + rowi * 8 : nullptr;
                    if (act == SFGPI_ACT_NONE || (act == SFGPI_ACT_RELU && mask_row != nullptr))
                        dgrad_epilogue_rolled(t_lane, Arow, r, row_ok, mask_row, act == SFGPI_ACT_RELU, group * 128, 2);
                    else if (act == SFGPI_ACT_RELU) dgrad_epilogue<SFGPI_ACT_RELU, 4>(t_lane, Arow, r, row_ok, act_row, mask_row, group * 128);
                    else if (act == SFGPI_ACT_NONE) dgrad_epilogue<SFGPI_ACT_NONE, 4>(t_lane, Arow, r, row_ok, act_row, mask_row, group * 128);
                    else dgrad_epilogue<SFGPI_ACT_TANH, 4>(t_lane, Arow, r, row_ok, act_row, mask_row, group * 128);
                    tc_fence_before();
                    fence_proxy_async();
                    if (lo > 0) mbar_arrive(SLOT_READY(slot));   // dZ_lo is the next MMA's A operand
                    store_tile(&tmap_dz, slot, kH / kKB, 0, lo * p.n_pol + pl);
                    DG_EPI();
                }
            }
        }
        if (et == 0) bulk_wait0();                               // outstanding stores complete before the CTA retires
    }

    tc_fence_before();
    __syncthreads();
    if (warp == kMmaWarp) {
        __syncwarp();
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
    if (g_dg_tl_on && blockIdx.x == 0 && threadIdx.x == 0) g_dg_tl[65] = clock64();
    trace_exit(SFGPI_TR_DGRAD);
}

// ------------------------------------------------------------------------------------------------------------------------
// wgrad
// ------------------------------------------------------------------------------------------------------------------------
// One TMA-issuing thread sustains ~27 B/cycle and issuers in different warps add up (DESIGN.md section 3): a 56 KB stage per
// producer warp, four of them (224 KB of the 227 KB an SM has).
constexpr int kWgThreads = 288;                     // 4 producer warps + 1 MMA warp + 4 epilogue warps
constexpr int kWgStages = 4;
constexpr int kWgMmaWarp = kWgStages;
constexpr int kWgABytes = 2 * kBoxBytes;            // dZ tile: 64 b x 128 n
constexpr int kWgBBytes = 4 * kBoxBytes;            // in tile: 64 b x 256 k
constexpr int kWgXBytes = kBoxBytes;                // xo tile: 64 b x 64
constexpr int kWgStageBytes = kWgABytes + kWgBBytes + kWgXBytes;      // 56 KB

struct WgParams {
    sfgpi_net_desc net;
    int n_pol, B, L, AD, S;
    int n_split, bs;                 // batch rows per split (multiple of 64)
    int mt_out, items_per_policy;    // 128-row tiles of the output layer's dW; mt_out + 2 * (L - 1) items per policy
    float *grad_part;                // [n_pol][n_split][row_stride]
};

// Store maps of dW_l (l >= 1) inside grad_part: fp32 {256 k, N_l rows, n_pol * n_split partial rows}, box {32, 128, 1},
// 128B-swizzled.  A 128-row tile of dW_l is one contiguous range of a partial row; the map clips rows past N_l.
struct WgStoreMaps { CUtensorMap w[SFGPI_MAX_LAYERS - 1]; };

// developer aid (env SFGPI_TIMELINE): clock64 stamps of the policy-0, split-0 CTA of the first hidden layer's tile 0 --
// [0] entry, [1] accumulator complete, [2] dW tile handed to the bulk stores, [3] stores complete, [4] exit
static __device__ long long g_wg_tl[5];
static __device__ int g_wg_tl_on = 0;

__global__ void __launch_bounds__(kWgThreads, 1)
mlp_wgrad_tc_kernel(const __grid_constant__ WgParams p, const __grid_constant__ CUtensorMap tmap_dz,
                    const __grid_constant__ CUtensorMap tmap_dzo, const __grid_constant__ CUtensorMap tmap_acts,
                    const __grid_constant__ CUtensorMap tmap_xo, const __grid_constant__ WgStoreMaps smaps) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    pdl_launch_dependents(SFGPI_TR_WGRAD);
    const bool tl = g_wg_tl_on && blockIdx.x == p.mt_out && blockIdx.y == 0;
    if (tl && threadIdx.x == 0) g_wg_tl[0] = clock64();
    const sfgpi_net_desc &net = p.net;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t sbase = smem_u32(smem_raw);
    const uint32_t bar0 = sbase + kWgStages * kWgStageBytes;
    auto FULL = [&](int s) { return bar0 + 8u * s; };
    auto EMPTY = [&](int s) { return bar0 + 8u * (kWgStages + s); };
    const uint32_t ACC_FULL = bar0 + 8u * (2 * kWgStages);
    const uint32_t holder_addr = ACC_FULL + 8u;

    // ---- decode the work item: (policy, layer l, 128-row tile mt of dW_l, batch split) ----
    const int pl = blockIdx.y;
    const int split = blockIdx.x / p.items_per_policy;
    int t = blockIdx.x - split * p.items_per_policy;
    int l, mt;
    if (t < p.mt_out) { l = p.L - 1; mt = t; }
    else { t -= p.mt_out; l = p.L - 2 - (t >> 1); mt = t & 1; }       // hidden layers L-2 .. 1, then layer 0
    const bool main_mma = l >= 1;                                       // layer 0's input is x itself: only the aux MMA
    const int b_lo = split * p.bs, b_hi = min(p.B, b_lo + p.bs);
    const int n_kb = (b_hi - b_lo + 63) / 64;

    if (threadIdx.x == 0) {
        for (int s = 0; s < kWgStages; ++s) { mbar_init(FULL(s), 1); mbar_init(EMPTY(s), 1); }
        mbar_init(ACC_FULL, 1);
        fence_mbar_init();
        tma_prefetch_desc(&tmap_dz); tma_prefetch_desc(&tmap_dzo); tma_prefetch_desc(&tmap_acts); tma_prefetch_desc(&tmap_xo);
    }
    if (warp == kWgMmaWarp) tmem_alloc(holder_addr, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(holder_addr));
    pdl_wait(SFGPI_TR_WGRAD);

    if (warp < kWgStages) {
        {
            const uint32_t leader = elect_one();
            const uint32_t bytes = kWgABytes + kWgXBytes + (main_mma ? kWgBBytes : 0);
            for (int kb = warp; kb < n_kb; kb += kWgStages) {
                const int s = warp;                                      // stage s is owned by producer warp s
                mbar_wait_warp(EMPTY(s), ((kb / kWgStages) & 1) ^ 1);
                mbar_arrive_expect_tx_e(FULL(s), bytes, leader);
                const uint32_t st = sbase + s * kWgStageBytes;
                const int b0 = b_lo + kb * 64;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    if (l == p.L - 1) tma_load_3d_e(st + h * kBoxBytes, &tmap_dzo, FULL(s), mt * 128 + h * 64, b0, pl, leader);
                    else tma_load_3d_e(st + h * kBoxBytes, &tmap_dz, FULL(s), mt * 128 + h * 64, b0, l * p.n_pol + pl, leader);
                }
                if (main_mma) {
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        tma_load_3d_e(st + kWgABytes + j * kBoxBytes, &tmap_acts, FULL(s), j * 64, b0, (l - 1) * p.n_pol + pl, leader);
                }
                tma_load_2d_e(st + kWgABytes + kWgBBytes, &tmap_xo, FULL(s), 0, b0, leader);
            }
        }
    } else if (warp == kWgMmaWarp) {
        {
            const uint32_t leader = elect_one();
            const uint32_t idesc_main = umma_idesc_bf16_major(kTM, 256, 1u, 1u);
            const uint32_t idesc_aux = umma_idesc_bf16_major(kTM, kXoCols, 1u, 1u);
            for (int kb = 0; kb < n_kb; ++kb) {
                const int s = kb % kWgStages;
                mbar_wait_warp(FULL(s), (kb / kWgStages) & 1);
                tc_fence_after();
                const uint32_t st = sbase + s * kWgStageBytes;
                const uint64_t ad = umma_desc_mn_sw128(st, kBoxBytes);
                const uint64_t bd = umma_desc_mn_sw128(st + kWgABytes, kBoxBytes);
                const uint64_t xd = umma_desc_mn_sw128(st + kWgABytes + kWgBBytes, kBoxBytes);
#pragma unroll
                for (int k16 = 0; k16 < 4; ++k16) {
                    const uint32_t accum = (kb | k16) ? 1u : 0u;
                    if (main_mma) umma_bf16_e(tmem_base, ad + 128 * k16, bd + 128 * k16, idesc_main, accum, leader);
                    umma_bf16_e(tmem_base + 256u, ad + 128 * k16, xd + 128 * k16, idesc_aux, accum, leader);
                }
                umma_commit_e(EMPTY(s), leader);
            }
            umma_commit_e(ACC_FULL, leader);
        }
    } else {
        // ---- epilogue: thread = TMEM lane = one row n of dW_l ----
        const int quad = warp & 3;
        const int n_loc = quad * 32 + lane;
        const int n = mt * 128 + n_loc;
        const int N_l = net.dims[l + 1];
        const bool et0 = threadIdx.x == (kWgMmaWarp + 1) * 32;
        const uint32_t t_lane = tmem_base + ((uint32_t)(quad * 32) << 16);
        float *gp = p.grad_part + ((size_t)pl * p.n_split + split) * net.row_stride;
        mbar_wait(ACC_FULL, 0);
        tc_fence_after();
        if (tl && et0) g_wg_tl[1] = clock64();
        const bool ok = n < N_l;
        if (main_mma) {
            // The ring stages are free once the accumulator is complete: the fp32 tile goes there as eight 128B-swizzled
            // {32 columns x 128 rows} boxes (conflict-free 16-byte stores: the lanes of a quarter-warp hit 8 different chunks),
            // and one thread writes each box to grad_part with a bulk tensor store as soon as all rows have written it, so the
            // stores run under the rest of the drain.  Per-row float4 stores to global memory at a 1 KB pitch touch 32 rows per
            // warp instruction.
#pragma unroll 1
            for (int cb = 0; cb < kH / 32; ++cb) {
                uint32_t v[32];
                tmem_ld32(t_lane + cb * 32, v);
                tmem_wait_ld();
                const uint32_t box = sbase + (uint32_t)(cb * (kTM * 128));
#pragma unroll
                for (int g = 0; g < 8; ++g)
                    sts128(box + n_loc * 128 + ((g ^ (n_loc & 7)) << 4), v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]);
                fence_proxy_async();
                asm volatile("bar.sync 1, 128;" ::: "memory");
                if (et0) tma_store_3d(&smaps.w[l - 1], box, cb * 32, mt * 128, pl * p.n_split + split);
            }
            if (et0) {
                bulk_commit();
                if (tl) g_wg_tl[2] = clock64();
            }
        }
        // aux columns: [0,S) = sum_b dZ[b][n] x[b][s] (dW_0 when l == 0), column S = sum_b dZ[b][n] (bias gradient)
#pragma unroll 1
        for (int c0 = 0; c0 <= p.S; c0 += 32) {
            uint32_t v[32];
            tmem_ld32(t_lane + 256u + c0, v);
            tmem_wait_ld();
            if (ok) {
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    const int c = c0 + i;
                    if (c == p.S) gp[net.b_off[l] + n] = __uint_as_float(v[i]);
                    else if (c < p.S && l == 0) gp[net.w_off[0] + (size_t)n * p.S + c] = __uint_as_float(v[i]);
                }
            }
        }
        tc_fence_before();
        if (main_mma && et0) {
            bulk_wait0();                                               // the dW tile is written before the CTA retires
            if (tl) g_wg_tl[3] = clock64();
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == kWgMmaWarp) {
        __syncwarp();
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
    if (tl && threadIdx.x == 0) g_wg_tl[4] = clock64();
    trace_exit(SFGPI_TR_WGRAD);
}

// xo[b][c] = x[b][c] for c < S, 1 for c == S, 0 otherwise  (bf16 [B][64])
__global__ void build_xo_kernel(const float *__restrict__ x, int B, int S, __nv_bfloat16 *__restrict__ xo) {
    pdl_launch_dependents();
    pdl_wait();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * kXoCols) return;
    const int b = i / kXoCols, c = i - b * kXoCols;
    xo[i] = __float2bfloat16_rn(c < S ? x[(size_t)b * S + c] : (c == S ? 1.0f : 0.0f));
}

static int make_tmap_bf16(CUtensorMap *tm, const void *base, int rank, const uint64_t *dims, const uint32_t *box) {
    TmapKey key = {base, {0, 0, 0}, {0, 0, 0}, rank, 0, 0};
    for (int i = 0; i < rank; ++i) { key.dims[i] = dims[i]; key.box[i] = box[i]; }
    if (tmap_cache_get(key, tm, false)) return SFGPI_OK;
    EncodeTiledFn encode = get_encode_fn();
    if (!encode) { set_error("cuTensorMapEncodeTiled entry point not found"); return SFGPI_E_CUDA; }
    cuuint64_t gdim[3], gstride[2];
    cuuint32_t bx[3], estride[3] = {1, 1, 1};
    uint64_t pitch = 2;
    for (int i = 0; i < rank; ++i) {
        gdim[i] = dims[i];
        bx[i] = box[i];
        pitch *= dims[i];
        if (i + 1 < rank) gstride[i] = pitch;
    }
    CUresult cr = encode(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void *>(base), gdim, gstride, bx, estride,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed (%d)", (int)cr); return SFGPI_E_CUDA; }
    tmap_cache_get(key, tm, true);
    return SFGPI_OK;
}

// store map of one weight matrix W_l [rows][256] in every partial row of grad_part (see WgStoreMaps)
static int make_tmap_wpart(CUtensorMap *tm, const float *base, int rows, int n_part, int row_stride) {
    const uint64_t pitch = (uint64_t)row_stride * sizeof(float);
    TmapKey key = {base, {(uint64_t)kH, (uint64_t)rows, (uint64_t)n_part}, {32, (uint32_t)kTM, 1}, 3, 1, 0, pitch};
    if (tmap_cache_get(key, tm, false)) return SFGPI_OK;
    EncodeTiledFn encode = get_encode_fn();
    if (!encode) { set_error("cuTensorMapEncodeTiled entry point not found"); return SFGPI_E_CUDA; }
    const cuuint64_t gdim[3] = {(cuuint64_t)kH, (cuuint64_t)rows, (cuuint64_t)n_part}, gstride[2] = {kH * sizeof(float), pitch};
    const cuuint32_t bx[3] = {32, (cuuint32_t)kTM, 1}, estride[3] = {1, 1, 1};
    CUresult cr = encode(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float *>(base), gdim, gstride, bx, estride,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed for grad_part (%d)", (int)cr); return SFGPI_E_CUDA; }
    tmap_cache_get(key, tm, true);
    return SFGPI_OK;
}

}  // namespace tc
}  // namespace sfgpi

using namespace sfgpi;
using namespace sfgpi::tc;

extern "C" int sfgpi_bwd_tc_out_pad(const sfgpi_net_desc *net) { return (net->n_actions * net->n_features + 63) & ~63; }

extern "C" int sfgpi_bwd_tc_splits(int32_t B, int32_t want) {
    if (B <= 0) return 1;
    if (want < 1) want = 1;
    const int bs = (((B + want - 1) / want) + 63) & ~63;
    return (B + bs - 1) / bs;
}

extern "C" int sfgpi_mlp_backward_tc(const sfgpi_backward_tc_args *args, void *stream) {
    trace_bind();
    const sfgpi_backward_tc_args &a = *args;
    const sfgpi_net_desc &net = a.net;
    const int L = net.n_layers;
    if (L < 3 || L > SFGPI_MAX_LAYERS || net.dims[0] > kXoCols - 1 || net.acts[L - 1] != SFGPI_ACT_NONE ||
        net.dims[L] != net.n_actions * net.n_features) {
        set_error("sfgpi_mlp_backward_tc: needs >= 3 Linear layers, S <= 63, a linear output layer");
        return SFGPI_E_INVALID;
    }
    for (int l = 1; l < L; ++l)
        if (net.dims[l] != kH) { set_error("sfgpi_mlp_backward_tc: every hidden width must be 256"); return SFGPI_E_INVALID; }
    if (a.B < 0 || a.n_pol < 0 || a.n_split < 1) { set_error("sfgpi_mlp_backward_tc: invalid sizes"); return SFGPI_E_INVALID; }
    if (a.B == 0 || a.n_pol == 0) return SFGPI_OK;
    if (!a.d_out) { set_error("sfgpi_mlp_backward_tc: d_out is NULL"); return SFGPI_E_INVALID; }
    const bool dense = a.actions == nullptr;                        // d_out [B][n_pol][A*D] instead of [n_pol][B][D]
    if (sfgpi_bwd_tc_splits(a.B, a.n_split) != a.n_split) {
        set_error("sfgpi_mlp_backward_tc: n_split %d leaves empty batch splits for B=%d (use sfgpi_bwd_tc_splits)", a.n_split, a.B);
        return SFGPI_E_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int AD = net.n_actions * net.n_features, ADp = sfgpi_bwd_tc_out_pad(&net), S = net.dims[0];

    int rc = SFGPI_OK;
    if (!a.xo_ready) {
        launch_pdl(build_xo_kernel, dim3((a.B * kXoCols + 255) / 256), dim3(256), 0, st, a.x, a.B, S, reinterpret_cast<__nv_bfloat16 *>(a.xo_bf16));
        rc = check_launch("sfgpi_mlp_backward_tc(xo)");
        if (rc) return rc;
    }

    // ---------------- dgrad chain ----------------
    DgParams dp;
    dp.net = net;
    dp.policy_lo = a.policy_lo; dp.n_pol = a.n_pol; dp.B = a.B;
    dp.actions = reinterpret_cast<const long long *>(a.actions);
    dp.d_out = a.d_out;
    dp.acts = reinterpret_cast<const __nv_bfloat16 *>(a.acts_bf16);
    dp.masks = reinterpret_cast<const uint32_t *>(a.relu_masks);
    dp.dz = reinterpret_cast<__nv_bfloat16 *>(a.dz_bf16);
    dp.dzo = reinterpret_cast<__nv_bfloat16 *>(a.dzo_bf16);
    dp.rows_per_policy = sfgpi_bf16_rows_per_policy(&net);
    dp.L = L; dp.AD = AD; dp.AD16 = (AD + 15) & ~15; dp.ADp = ADp;
    dp.n_chunks = (dp.AD16 + 255) / 256;
    dp.n_items = dp.n_chunks + (L - 2);
    dp.tiles_per_policy = (a.B + kTM - 1) / kTM;
    const int total_tiles = dp.tiles_per_policy * a.n_pol;
    dp.paired = total_tiles > 148 ? 1 : 0;
    dp.pairs_per_policy = dp.paired ? (dp.tiles_per_policy + 1) / 2 : dp.tiles_per_policy;
    dp.total_pairs = dp.pairs_per_policy * a.n_pol;
    CUtensorMap tmap_w;
    {
        const uint64_t dims[2] = {(uint64_t)kH, (uint64_t)a.n_policies_total * dp.rows_per_policy};
        const uint32_t box[2] = {64, 64};
        rc = make_tmap_bf16(&tmap_w, a.params_bf16, 2, dims, box);
        if (rc) return rc;
    }
    CUtensorMap tm_dz_st, tm_dzo_st;                                 // store maps: box = {64 columns, 128 rows, 1 slab}
    {
        const uint64_t d3[3] = {(uint64_t)kH, (uint64_t)a.B, (uint64_t)(L - 1) * a.n_pol};
        const uint64_t do3[3] = {(uint64_t)ADp, (uint64_t)a.B, (uint64_t)a.n_pol};
        const uint32_t box[3] = {64, 128, 1};
        if ((rc = make_tmap_bf16(&tm_dz_st, a.dz_bf16, 3, d3, box))) return rc;
        if ((rc = make_tmap_bf16(&tm_dzo_st, a.dzo_bf16, 3, do3, box))) return rc;
    }
    const int dg_smem = 2 * kABytes + kNStage * kStageBytes + 256;
    static bool cfg = false;
    if (!cfg) {
        cudaFuncSetAttribute(mlp_dgrad_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, dg_smem);
        cudaFuncSetAttribute(mlp_dgrad_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, dg_smem);
        cfg = true;
    }
    dp.n_main = dp.total_pairs < 148 ? dp.total_pairs : 148;
    sfgpi_td_args ex = {};
    int ex_nclu = 0, riders = 0;
    if (a.expand_td != nullptr) {                                    // deferred TSF expand (sfgpi_td_args.defer_expand)
        ex = *reinterpret_cast<const sfgpi_td_args *>(a.expand_td);
        if (ex.variant != 2 || ex.n_pol < 1 || !ex.tsf_part || !ex.aux_grad_part || !ex.g || !ex.h ||
            (size_t)tsf_expand_smem_floats(ex.D, ex.S, ex.G, ex.n_flows) * sizeof(float) > (size_t)dg_smem) {
            set_error("sfgpi_mlp_backward_tc: expand_td is not a variant-2 TD step that fits the dgrad launch");
            return SFGPI_E_INVALID;
        }
        ex_nclu = sfgpi_td_partials(ex.B);
        riders = ex.n_pol;
    }
    static const bool dg_tl = getenv("SFGPI_TIMELINE") != nullptr;
    if (dg_tl) {
        const int on = 1;
        long long z[66] = {0};
        cudaMemcpyToSymbol(g_dg_tl_on, &on, sizeof(on));
        cudaMemcpyToSymbol(g_dg_tl, z, sizeof(z));
    }
    if (dense) launch_pdl(mlp_dgrad_tc_kernel<true>, dim3(dp.n_main + riders), dim3(kThreadsDg), dg_smem, st, dp, tmap_w, tm_dz_st, tm_dzo_st, ex, ex_nclu);
    else launch_pdl(mlp_dgrad_tc_kernel<false>, dim3(dp.n_main + riders), dim3(kThreadsDg), dg_smem, st, dp, tmap_w, tm_dz_st, tm_dzo_st, ex, ex_nclu);
    rc = check_launch("sfgpi_mlp_backward_tc(dgrad)");
    if (rc) return rc;
    if (dg_tl) {                                                 // developer aid: CTA 0's timeline (cycles since its entry)
        long long h[66];
        cudaStreamSynchronize(st);
        cudaMemcpyFromSymbol(h, g_dg_tl, sizeof(h));
        fprintf(stderr, "[sfgpi dgrad timeline] tiles=%d grid=%d %s; exit %lld\n  epi :", dp.total_pairs, dp.n_main, dp.paired ? "paired" : "one-tile", h[65] - h[64]);
        for (int i = 0; i < 32 && h[i]; ++i) fprintf(stderr, " %lld", h[i] - h[64]);
        fprintf(stderr, "\n  mma :");
        for (int i = 32; i < 64 && h[i]; ++i) fprintf(stderr, " %lld", h[i] - h[64]);
        fprintf(stderr, "\n");
    }

    // ---------------- wgrad ----------------
    WgParams wp;
    wp.net = net;
    wp.n_pol = a.n_pol; wp.B = a.B; wp.L = L; wp.AD = AD; wp.S = S;
    wp.n_split = a.n_split;
    wp.bs = (((a.B + a.n_split - 1) / a.n_split) + 63) & ~63;
    wp.mt_out = (AD + 127) / 128;
    wp.items_per_policy = wp.mt_out + 2 * (L - 1);
    wp.grad_part = a.grad_part;
    CUtensorMap tm_dz, tm_dzo, tm_acts, tm_xo;
    {
        const uint64_t d3[3] = {(uint64_t)kH, (uint64_t)a.B, (uint64_t)(L - 1) * a.n_pol};
        const uint64_t do3[3] = {(uint64_t)ADp, (uint64_t)a.B, (uint64_t)a.n_pol};
        const uint64_t dx[2] = {(uint64_t)kXoCols, (uint64_t)a.B};
        const uint32_t box3[3] = {64, 64, 1}, box2[2] = {64, 64};
        if ((rc = make_tmap_bf16(&tm_dz, a.dz_bf16, 3, d3, box3))) return rc;
        if ((rc = make_tmap_bf16(&tm_dzo, a.dzo_bf16, 3, do3, box3))) return rc;
        if ((rc = make_tmap_bf16(&tm_acts, a.acts_bf16, 3, d3, box3))) return rc;
        if ((rc = make_tmap_bf16(&tm_xo, a.xo_bf16, 2, dx, box2))) return rc;
    }
    WgStoreMaps smaps;
    memset(&smaps, 0, sizeof(smaps));
    for (int l = 1; l < L; ++l)
        if ((rc = make_tmap_wpart(&smaps.w[l - 1], a.grad_part + net.w_off[l], net.dims[l + 1], a.n_pol * a.n_split, net.row_stride))) return rc;
    const int wg_smem = kWgStages * kWgStageBytes + 256;
    static bool cfg2 = false;
    if (!cfg2) { cudaFuncSetAttribute(mlp_wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, wg_smem); cfg2 = true; }
    if (dg_tl) {
        const int on = 1;
        long long z[5] = {0};
        cudaMemcpyToSymbol(g_wg_tl_on, &on, sizeof(on));
        cudaMemcpyToSymbol(g_wg_tl, z, sizeof(z));
    }
    dim3 grid(wp.items_per_policy * a.n_split, a.n_pol);
    launch_pdl(mlp_wgrad_tc_kernel, grid, dim3(kWgThreads), wg_smem, st, wp, tm_dz, tm_dzo, tm_acts, tm_xo, smaps);
    rc = check_launch("sfgpi_mlp_backward_tc(wgrad)");
    if (rc == SFGPI_OK && dg_tl) {                               // developer aid: one hidden-layer CTA's epilogue (cycles)
        long long h[5];
        cudaStreamSynchronize(st);
        cudaMemcpyFromSymbol(h, g_wg_tl, sizeof(h));
        fprintf(stderr, "[sfgpi wgrad timeline] grid=%dx%d; accumulator %lld, epilogue %lld (tile handed to TMA %lld), exit %lld\n",
                grid.x, grid.y, h[1] - h[0], h[3] - h[1], h[2] - h[1], h[4] - h[0]);
    }
    return rc;
}
