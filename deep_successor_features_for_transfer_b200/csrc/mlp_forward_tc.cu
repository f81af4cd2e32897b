// Fused ensemble psi-MLP forward on the 5th-gen tensor cores (mode 1: bf16 operands, fp32 accumulation in TMEM).
//
// Persistent, warp-specialised kernel, one CTA per SM:
//   warps 0-3   TMA producers: stream the policy's bf16 weights (K-major, 128B-swizzled boxes of 128 rows x 64 k = 16 KB)
//               through a 4-stage mbarrier ring, one stage per producer warp;
//   warp 4      MMA issuer: one thread issues tcgen05.mma (M=128, N<=128, K=16) into TMEM, commits free the ring stages;
//   warps 5-8   epilogue group of tile slot X, warps 9-12 of tile slot Y: thread = TMEM lane = one state (row).  They stage
//               the bf16 state tile, and after every MMA layer read the accumulator with tcgen05.ld, apply bias +
//               activation, round to bf16 and write the next layer's A operand straight into shared memory in the UMMA
//               K-major SWIZZLE_128B layout (activations never touch HBM).
// Two 128-row tiles (X, Y) of the same policy are in flight per CTA and ping-pong: while the epilogue group of X drains
// its accumulator, the tensor core runs Y's layer, so the pipe stays busy.  TMEM: 2 x 256 fp32 columns.
//
// Every Linear layer runs on the tensor core, including the K=S input layer (states rounded to bf16, K padded to 16).
// Output layer, two forms:
//   psi form  : N = A*D columns (padded to 16), epilogue = psi store and / or gather of the selected action's D columns;
//   GPI form  : q = psi . w is folded into the weights beforehand (sfgpi_fold_gpi: Wq[w,a,:] = sum_d w[d] W_out[a*D+d,:]),
//               so the layer has only n_w * A columns and the epilogue is a running (max, argmax) per reward vector --
//               psi[B,N,A,D] is never formed, not even on chip.  (GPI_w, sfdqn.py:215-240.)
#include "forward_tc.cuh"
#include <limits.h>
#include <stdlib.h>
#include <string.h>

namespace sfgpi {
namespace tc {


__device__ __forceinline__ int job_of_pair(const TcMulti &m, int pair) {
    int j = 0;
    while (j + 1 < m.n_jobs && pair >= m.pair_start[j + 1]) ++j;
    return j;
}

__global__ void __launch_bounds__(kThreadsTc, 1)
mlp_forward_tc_kernel(const __grid_constant__ TcMulti m, const __grid_constant__ TmapSet maps, const __grid_constant__ UnitTable ut) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int unit0 = (int)blockIdx.x, unit_stride = (int)gridDim.x;
    // work unit g -> job, policy slot, the tile this CTA handles in slot X (slot Y: tile0 + 1), whether it has a Y slot
    auto unit_at = [&](int g) {
        Unit u;
        if (m.sched) {
            const uint32_t e = ut.u[g];
            u.jb = (int)(e >> 30); u.has_y = (e >> 29) & 1u; u.pl = (int)((e >> 16) & 0x1FFFu); u.tile0 = (int)(e & 0xFFFFu);
            return u;
        }
        u.jb = job_of_pair(m, g);
        const TcParams &p = m.job[u.jb];
        const int pair = g - m.pair_start[u.jb];
        u.pl = pair / p.pairs_per_policy;
        const int pip = pair - u.pl * p.pairs_per_policy;
        u.tile0 = p.paired ? 2 * pip : pip;
        u.has_y = p.paired && (2 * pip + 1 < p.tiles_per_policy);
        return u;
    };
    pdl_launch_dependents(SFGPI_TR_FWD);
    if (m.timeline != nullptr && blockIdx.x == 0 && threadIdx.x == 0) m.timeline[255] = clock64();      // kernel entry
    const long long cta_t0 = clock64();
    if (m.timeline != nullptr && threadIdx.x == 0) { unsigned long long gt; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt)); m.timeline[768 + blockIdx.x] = (long long)gt; }

    // ---- carve-up: [A slot X 64K][A slot Y 64K][weight ring 4 x 16K][biases 24K][barriers] ----
    const uint32_t sbase = smem_u32(smem_raw);
    const uint32_t W_addr = sbase + 2 * kABytes;
    const uint32_t bias_addr = W_addr + kNStage * kStageBytes;
    const uint32_t bar0 = bias_addr + kBiasFloatsMax * 4;
    // barriers: [0,4) w_full, [4,8) w_empty, [8,10) slot_ready, [10,12) acc_full ; then the TMEM base holder
    // One-tile-per-CTA mode (launches of <= 148 tiles): the idle Y slot's 64 KB become 4 more weight stages (an 8-deep ring holds
    // a whole 256x256 layer, so the next layer streams in during the current epilogue) and BOTH epilogue groups work on the one
    // tile, each on half of the columns.  Stage s lives at W_addr + (s < 4 ? s : s - 8) * 16 KB (s >= 4: inside slot Y).
    const int ns_log = m.paired ? 2 : 3, ns_mask = (1 << ns_log) - 1;
    auto W_FULL = [&](int s) { return bar0 + 8u * s; };
    auto W_EMPTY = [&](int s) { return bar0 + 8u * (8 + s); };
    auto SLOT_READY = [&](int s) { return bar0 + 8u * (16 + s); };
    auto ACC_FULL = [&](int s) { return bar0 + 8u * (18 + s); };
    auto stage_off = [&](int s) { return (s - ((s & 4) << 1)) * kStageBytes; };      // signed byte offset from W_addr
    const uint32_t holder_addr = bar0 + 8u * 20;

    if (threadIdx.x == 0) {
        for (int s = 0; s < 8; ++s) { mbar_init(W_FULL(s), 1); mbar_init(W_EMPTY(s), 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(SLOT_READY(s), 256); mbar_init(ACC_FULL(s), 1); }
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


    if (warp < kNStage) {
        // =========================== TMA producers ===========================
        // One issuing thread sustains only ~27 B/cycle of 128-row boxes (its bulk-tensor copies do not overlap: scripts/
        // tma_bench.cu), well below the 64 B/cycle the MMA consumes; issuers in different warps scale linearly.  So ring stage
        // s is owned by producer warp s.
        {
            const uint32_t leader = elect_one();
            uint32_t n = 0;
            int tlc = 0;
            for (int gpair = unit0; gpair < m.total_pairs; gpair += unit_stride) {
                const Unit un = unit_at(gpair);
                const int jb = un.jb, pl = un.pl;
                const TcParams &p = m.job[jb];
                const sfgpi_forward_args &a = p.a;
                const int row0 = (a.policy_lo + pl) * p.rows_per_policy;
                const bool has_y = un.has_y;
                for (int it = 0; it < p.n_items; ++it) {
                    const ItemInfo ii = item_info(p, it);
                    const int nblocks = (ii.n_cols + kNB - 1) / kNB;
                    const bool folded = ii.kind == 2 && p.gpi;
                    const void *tm = folded ? (const void *)&maps.q[jb] : (const void *)&maps.w[jb];
                    const int rbase = folded ? pl * p.n_final + ii.row_base : row0 + ii.row_base;
                    for (int slot = 0; slot < (has_y ? 2 : 1); ++slot)
                        for (int kb = 0; kb < ii.n_kb; ++kb)
                            for (int nb = 0; nb < nblocks; ++nb, ++n) {
                                const int s = n & ns_mask;
                                if ((s & 3) != warp) continue;
                                mbar_wait_warp(W_EMPTY(s), ((n >> ns_log) & 1) ^ 1);
                                if (warp == 0 && leader) TL_STAMP(2, tlc);
                                mbar_arrive_expect_tx_e(W_FULL(s), kStageBytes, leader);
                                tma_load_2d_e(W_addr + stage_off(s), tm, W_FULL(s), kb * kKB, rbase + nb * kNB, leader);
                            }
                }
            }
        }
    } else if (warp == kMmaWarp) {
        // =========================== MMA issuer ===========================
        // Whole warp runs the loop (operands stay in uniform registers), the elected lane issues: see tc_common.cuh.
        const uint32_t leader = elect_one();
        uint32_t n = 0, ready_cnt[2] = {0, 0};
        int tlc = 0;
        const uint64_t adesc_x = umma_desc_k_sw128(sbase), adesc_y = umma_desc_k_sw128(sbase + kABytes);
        const uint64_t bdesc0 = umma_desc_k_sw128(W_addr);
        for (int gpair = unit0; gpair < m.total_pairs; gpair += unit_stride) {
            const Unit un = unit_at(gpair);
            const int jb = un.jb;
            const TcParams &p = m.job[jb];
            const bool has_y = un.has_y;
            for (int it = 0; it < p.n_items; ++it) {
                const ItemInfo ii = item_info(p, it);
                const int nblocks = (ii.n_cols + kNB - 1) / kNB;
                const uint32_t idesc_full = umma_idesc_bf16(kTM, kNB);
                const uint32_t idesc_last = umma_idesc_bf16(kTM, (uint32_t)(ii.n_cols - (nblocks - 1) * kNB));
                for (int slot = 0; slot < (has_y ? 2 : 1); ++slot) {
                    mbar_wait_warp(SLOT_READY(slot), ready_cnt[slot] & 1);
                    ++ready_cnt[slot];
                    tc_fence_after();
                    if (leader) TL_STAMP(1, tlc);                         // slot ready
                    const uint32_t d_base = tmem_base + (uint32_t)slot * 256u;
                    // A full 256-column layer is issued as N=256 MMAs over a PAIR of adjacent ring stages (rows 0-127 | 128-255
                    // of the weight block are contiguous in shared memory): half as many instructions for the same math --
                    // the single issuing thread needs ~107 cycles per tcgen05.mma, more than the 64 an N=128 MMA executes.
                    const bool wide = nblocks == 2 && ii.n_cols == 256 && !(n & 1);
                    const uint32_t idesc_wide = umma_idesc_bf16(kTM, 256);
                    for (int kb = 0; kb < ii.n_kb; ++kb) {
                        const uint64_t ad = (slot ? adesc_y : adesc_x) + (uint64_t)(kb * ((kTM * 128) >> 4));
                        if (wide) {
                            const int s = n & ns_mask;
                            mbar_wait_warp(W_FULL(s), (n >> ns_log) & 1);
                            mbar_wait_warp(W_FULL(s + 1), (n >> ns_log) & 1);
                            tc_fence_after();
                            if (leader && kb == 0) TL_STAMP(1, tlc);              // first weight stages landed
                            const uint64_t bd = bdesc0 + (uint64_t)(int64_t)(stage_off(s) >> 4);
                            if (ii.n_k16 == 4) {
                                umma_bf16_e(d_base, ad, bd, idesc_wide, kb ? 1u : 0u, leader);
                                umma_bf16_e(d_base, ad + 2, bd + 2, idesc_wide, 1u, leader);
                                umma_bf16_e(d_base, ad + 4, bd + 4, idesc_wide, 1u, leader);
                                umma_bf16_e(d_base, ad + 6, bd + 6, idesc_wide, 1u, leader);
                            } else {
                                for (int k16 = 0; k16 < ii.n_k16; ++k16)
                                    umma_bf16_e(d_base, ad + 2 * k16, bd + 2 * k16, idesc_wide, (kb | k16) ? 1u : 0u, leader);
                            }
                            umma_commit_e(W_EMPTY(s), leader);
                            umma_commit_e(W_EMPTY(s + 1), leader);
                            n += 2;
                            continue;
                        }
                        for (int nb = 0; nb < nblocks; ++nb, ++n) {
                            const int s = n & ns_mask;
                            mbar_wait_warp(W_FULL(s), (n >> ns_log) & 1);
                            tc_fence_after();
                            if (leader && kb == 0 && nb == 0) TL_STAMP(1, tlc);   // first weight stage landed
                            const uint32_t idesc = (nb == nblocks - 1) ? idesc_last : idesc_full;
                            const uint64_t bd = bdesc0 + (uint64_t)(int64_t)(stage_off(s) >> 4);
                            const uint32_t d = d_base + nb * kNB;
                            if (ii.n_k16 == 4) {
                                umma_bf16_e(d, ad, bd, idesc, kb ? 1u : 0u, leader);
                                umma_bf16_e(d, ad + 2, bd + 2, idesc, 1u, leader);
                                umma_bf16_e(d, ad + 4, bd + 4, idesc, 1u, leader);
                                umma_bf16_e(d, ad + 6, bd + 6, idesc, 1u, leader);
                            } else {
                                for (int k16 = 0; k16 < ii.n_k16; ++k16)
                                    umma_bf16_e(d, ad + 2 * k16, bd + 2 * k16, idesc, (kb | k16) ? 1u : 0u, leader);
                            }
                            umma_commit_e(W_EMPTY(s), leader);           // stage free once these MMAs have read it
                        }
                    }
                    umma_commit_e(ACC_FULL(slot), leader);                // accumulator of this item complete
                    if (leader) TL_STAMP(1, tlc);                         // all MMAs of the item issued
                }
            }
        }
    } else {
        // =========================== epilogue groups ===========================
        // All 8 epilogue warps work on ONE accumulator at a time, each group on half of the columns: draining a 128 x 256 fp32
        // accumulator is TMEM-read-bound (~2048 cycles, as long as the MMAs that produced it) only with 8 warps in flight;
        // 4 warps need 3100-4100 cycles (measured, clock64 timeline) and would pace the whole kernel.  With two tiles per
        // CTA the groups alternate X, Y, X, ... while the tensor core works on the other slot.
        const int group = (warp - kEpiWarp0) >> 2;          // warps 5-8 -> group 0, 9-12 -> group 1
        const int quad = warp & 3;                          // TMEM lane quadrant this warp may access
        const int r = quad * 32 + lane;                     // row inside the tile == TMEM lane
        const int et = threadIdx.x - kEpiWarp0 * 32;        // 0..255 among epilogue threads
        const uint32_t t_lane0 = tmem_base + ((uint32_t)(quad * 32) << 16);
        uint32_t full_cnt[2] = {0, 0};
        int cur_policy = -1;
        bool store_pending[2] = {false, false};              // (uniform over the 256 epilogue threads)
        int tlc = 0;
        const int tl_role = (et == 0) ? 0 : ((et == 128) ? 3 : -1);
#define TL_EPI() do { if (tl_role >= 0) TL_STAMP(tl_role, tlc); } while (0)
        TL_EPI();                                            // set-up done

        for (int gpair = unit0; gpair < m.total_pairs; gpair += unit_stride) {
            const Unit un = unit_at(gpair);
            const int jb = un.jb;
            const TcParams &p = m.job[jb];
            const sfgpi_forward_args &a = p.a;
            const sfgpi_net_desc &net = a.net;
            const int B = a.B, L = net.n_layers, A_ = net.n_actions, D = net.n_features, AD = A_ * D;
            const int S = net.dims[0];
            const int n_bias = (1 + p.Lh) * kH + p.n_final;     // [b_0 | b_1..b_Lh | b_final]
            const int pl = un.pl;
            const int n_slots = un.has_y ? 2 : 1;
            const float *P = a.params + (size_t)(a.policy_lo + pl) * net.row_stride;

            // Saved activations (training forward): the bf16 tile a hidden epilogue leaves in the A slot IS the row-major
            // activation block in TMA's 128B-swizzled box layout, so one thread stores it with 4 bulk tensor copies while the
            // next layer's MMAs read the same tile -- per-thread 16-byte stores at a 512-byte row pitch cost one L1 wavefront per
            // lane (~8000 cycles per tile-layer, measured) against ~2000 for everything else in the epilogue.
            const bool saving = a.acts_bf16_out != nullptr;
            // before a write to A slot s: its pending bulk store has finished READING it.  Stores are issued in (item, slot)
            // order, so with two slots in flight the newest group belongs to the other slot and may stay pending.
            auto a_slot_guard = [&](bool all) {
                if (et == 0) { if (all) bulk_wait_read0(); else bulk_wait_read1(); }
                asm volatile("bar.sync 1, 256;" ::: "memory");
            };
            if (store_pending[0] || store_pending[1]) { a_slot_guard(true); store_pending[0] = store_pending[1] = false; }

            // Biases of a new (job, policy): the global loads are ISSUED here, ahead of the state staging, and land in shared memory
            // after it -- one memory round trip for both instead of two back to back (~2 k cycles per work unit).
            const bool new_bias = jb * 65536 + pl != cur_policy;
            const bool bias_pre = new_bias && n_bias <= 4 * 256;
            float bias_v[4] = {0.0f, 0.0f, 0.0f, 0.0f};
            auto bias_load = [&](int e) {
                float v = 0.0f;
                if (e < (1 + p.Lh) * kH) v = P[net.b_off[e >> 8] + (e & 255)];
                else if (e < n_bias) {
                    const int c = e - (1 + p.Lh) * kH;
                    v = p.gpi ? p.bq[(size_t)pl * p.n_final + c] : (c < AD ? P[net.b_off[L - 1] + c] : 0.0f);
                }
                return v;
            };
            if (bias_pre) {
#pragma unroll
                for (int u = 0; u < 4; ++u) bias_v[u] = bias_load(et + u * 256);
            }
            int bs[2], sel_base[2];
            // ---------------- stage the state tiles as the input layer's A operands (bf16, K padded to 16*ks0) ----------------
            // Every global load of the unit's head is ISSUED before the first one is consumed: the gather indices of both slots
            // and (states of <= 8 features) both slots' state rows.  Consumed one after the other -- row, index, next slot's row,
            // its index -- they were four dependent memory round trips, ~4.4 k cycles at the head of every work unit (stamps).
            int sidx_v[2] = {0, 0};
            float xf[2][8];
            const bool x_pre = S <= 8;
#pragma unroll
            for (int slot = 0; slot < 2; ++slot) {
                if (slot >= n_slots) break;
                const int b = (un.tile0 + slot) * kTM + r;                             // global state index of this thread's row
                bs[slot] = b;
                if (a.sel_out != nullptr && b < B)
                    sidx_v[slot] = a.sel_actions ? (int)a.sel_actions[b] : (int)key_index(a.sel_keys[(size_t)pl * a.sel_key_stride + b]);
                if (group == 0 && x_pre) {
                    const float *xr = a.x + (size_t)b * S;
#pragma unroll
                    for (int i = 0; i < 8; ++i) xf[slot][i] = (b < B && i < S) ? xr[i] : 0.0f;
                }
            }
#pragma unroll
            for (int slot = 0; slot < 2; ++slot) {
                if (slot >= n_slots) break;
                const int b = bs[slot];
                const bool row_ok = b < B;
                if (group == 0) {
                    const float *xr = a.x + (size_t)b * S;
                    const uint32_t Arow = sbase + (uint32_t)slot * kABytes;
                    for (int c = 0; c < p.ks0 * 16; c += 8) {
                        float xv[8];
#pragma unroll
                        for (int i = 0; i < 8; ++i) xv[i] = x_pre ? (c == 0 ? xf[slot][i] : 0.0f) : ((row_ok && c + i < S) ? xr[c + i] : 0.0f);
                        sts128(Arow + a_chunk_off(r, c), pack_bf16x2(xv[0], xv[1]), pack_bf16x2(xv[2], xv[3]),
                               pack_bf16x2(xv[4], xv[5]), pack_bf16x2(xv[6], xv[7]));
                    }
                    fence_proxy_async();                      // generic-proxy smem writes -> visible to the UMMA (async proxy)
                }
                mbar_arrive(SLOT_READY(slot));
                sel_base[slot] = (a.sel_out != nullptr && row_ok) ? sidx_v[slot] * D : -(1 << 30);
            }
            TL_EPI();                                         // state tiles staged

            // Biases AFTER the state tiles were handed to the MMA warp: their global-load latency hides behind the input layer.
            if (new_bias) {                                  // per-(job, policy) biases -> smem (all 256 epilogue threads)
                asm volatile("bar.sync 1, 256;" ::: "memory");
                if (bias_pre) {
#pragma unroll
                    for (int u = 0; u < 4; ++u)
                        if (et + u * 256 < n_bias) sts32(bias_addr + 4u * (et + u * 256), bias_v[u]);
                } else {
                    for (int e0 = et; e0 < n_bias; e0 += 4 * 256) {       // 4 independent loads in flight per thread
                        float v[4];
#pragma unroll
                        for (int u = 0; u < 4; ++u) v[u] = bias_load(e0 + u * 256);
#pragma unroll
                        for (int u = 0; u < 4; ++u)
                            if (e0 + u * 256 < n_bias) sts32(bias_addr + 4u * (e0 + u * 256), v[u]);
                    }
                }
                asm volatile("bar.sync 1, 256;" ::: "memory");
                cur_policy = jb * 65536 + pl;
            }

            // GPI output chunks: the generic item loop below spends as long on its per-(chunk, slot) set-up -- job fields re-read
            // through register-indexed constant loads, slot-indexed state in local memory, a page of straight-line code that runs
            // once per chunk and is therefore never in the 32 KB instruction cache -- as on the scan itself (ncu source page at 256
            // reward vectors: the once-per-chunk instructions collect as many stall samples as the scan's inner loop; in-kernel
            // stamps at 4 vectors: 3.3 k cycles of set-up ahead of a 5-trip scan).  GPI jobs that write action / task keys only
            // take their output chunks through the lean loop further down: everything chunk-invariant in registers, slots unrolled.
            const int Lh_u = p.Lh, n_items_u = p.n_items;
            const bool lean_gpi = p.gpi != 0 && !a.w_diag && a.q_out == nullptr;
            const bool lean_psi = p.gpi == 0;
            for (int it = 0; it < n_items_u; ++it) {
                if (lean_gpi && it == 1 + Lh_u) {
                    const int nw_u = p.nw, n_final_u = p.n_final, wblk_u = gpi_wblock(nw_u), ncol_u = gpi_ncols(nw_u, A_);
                    const bool wide_u = wblk_u == 8 && ncol_u >= m.wide_min;
                    const uint32_t bias_u = bias_addr + 4u * ((1 + Lh_u) * kH);        // folded biases, indexed by absolute column
                    const uint32_t tid_u = (uint32_t)(a.task_base + pl), kstep_u = (uint32_t)B;
                    long long *const ka_u = reinterpret_cast<long long *>(a.key_action), *const kt_u = reinterpret_cast<long long *>(a.key_task);
                    const int b0_u = bs[0], b1_u = n_slots > 1 ? bs[1] : 0;
#pragma unroll 1
                    for (int col0 = 0; col0 < n_final_u; col0 += 256) {
                        const int c_hi = min(min(col0 + 256, n_final_u), ncol_u);
                        const bool more = col0 + 256 < n_final_u;
#pragma unroll
                        for (int slot = 0; slot < 2; ++slot) {
                            if (slot >= n_slots) break;
                            // blocked column orders: each epilogue group takes one 128-column half of the chunk (every emission is an
                            // atomicMax, so a block cut by the boundary merges); plain order (< 4 vectors): group g scans slot g
                            // (a chunk of <= 128 columns -- the headline's 36 -- is shared as well: half of its 8-column trips each)
                            const int half = c_hi - col0 > 128 ? 128 : ((c_hi - col0 + 15) >> 4) << 3;
                            const int cb = wblk_u > 1 ? col0 + group * half : (group == slot ? col0 : c_hi);
                            const int ce = wblk_u > 1 ? min(cb + half, c_hi) : c_hi;
                            const int cm = (wide_u && cb < ce) ? cb + ((ce - cb) & ~31) : cb;      // whole 32-column windows: gpi_scan_wide8
                            const int b = slot ? b1_u : b0_u;
                            const uint32_t t_lane = t_lane0 + (uint32_t)slot * 256u;
                            long long *const ka_b = ka_u ? ka_u + b : nullptr, *const kt_b = kt_u ? kt_u + b : nullptr;
                            mbar_wait(ACC_FULL(slot), full_cnt[slot] & 1);
                            ++full_cnt[slot];
                            tc_fence_after();
                            TL_EPI();
                            if (cb < cm) gpi_scan_wide8(t_lane, bias_u, col0, cb, cm, A_, nw_u, ka_b, kt_b, kstep_u, b < B, tid_u);
                            if (cm < ce) {
                                if (wblk_u == 8) gpi_scan_rolled<8>(t_lane, bias_u, col0, cm, ce, A_, nw_u, ka_b, kt_b, kstep_u, b < B, tid_u, nullptr);
                                else if (wblk_u == 4) gpi_scan_rolled<4>(t_lane, bias_u, col0, cm, ce, A_, nw_u, ka_b, kt_b, kstep_u, b < B, tid_u, nullptr);
                                else gpi_scan_rolled<1>(t_lane, bias_u, col0, cm, ce, A_, nw_u, ka_b, kt_b, kstep_u, b < B, tid_u, nullptr);
                            }
                            tc_fence_before();
                            if (more) mbar_arrive(SLOT_READY(slot));                                     // next chunk may overwrite the accumulator
                            TL_EPI();
                        }
                    }
                    break;
                }
                if (lean_psi && it == 1 + Lh_u) {
                    // psi-form output chunks (online job: the gathered rows; target job: the full psi rows), same lean shape
                    const int n_final_u = p.n_final, n_pol_u = a.n_pol;
                    const uint32_t bias_u = bias_addr + 4u * ((1 + Lh_u) * kH);
                    float *const psi_u = a.psi_out, *const sel_u = a.sel_out;
                    const int b0_u = bs[0], b1_u = n_slots > 1 ? bs[1] : 0;
                    const int sb0_u = sel_base[0], sb1_u = n_slots > 1 ? sel_base[1] : -(1 << 30);
#pragma unroll 1
                    for (int col0 = 0; col0 < n_final_u; col0 += 256) {
                        const int n_cols = min(256, n_final_u - col0);
                        const bool more = col0 + 256 < n_final_u;
#pragma unroll
                        for (int slot = 0; slot < 2; ++slot) {
                            if (slot >= n_slots) break;
                            const int b = slot ? b1_u : b0_u;
                            const uint32_t t_lane = t_lane0 + (uint32_t)slot * 256u;
                            mbar_wait(ACC_FULL(slot), full_cnt[slot] & 1);
                            ++full_cnt[slot];
                            tc_fence_after();
                            TL_EPI();
                            psi_out_rolled(t_lane, bias_u + 4u * (uint32_t)col0, col0, n_cols, group * 8,
                                           psi_u ? psi_u + ((size_t)b * n_pol_u + pl) * AD : nullptr, AD,
                                           sel_u ? sel_u + ((size_t)pl * B + b) * D : nullptr, slot ? sb1_u : sb0_u, D, b < B);
                            tc_fence_before();
                            if (more) mbar_arrive(SLOT_READY(slot));                                     // next chunk may overwrite the accumulator
                            TL_EPI();
                        }
                    }
                    break;
                }
                const ItemInfo ii = item_info(p, it);
#pragma unroll 1
                for (int slot = 0; slot < n_slots; ++slot) {
                    const int b = bs[slot];
                    const bool row_ok = b < B;
                    const uint32_t t_lane = t_lane0 + (uint32_t)slot * 256u;
                    const uint32_t Arow = sbase + (uint32_t)slot * kABytes;
                    mbar_wait(ACC_FULL(slot), full_cnt[slot] & 1);
                    ++full_cnt[slot];
                    tc_fence_after();
                    TL_EPI();                                 // accumulator of (item, slot) complete
                    if (ii.kind != 2) {
                        // ------ input / hidden layer: bias + act, bf16, write next A operand (in place), optional save ------
                        const uint32_t bias = bias_addr + 4u * (it * kH);
                        const int act = net.acts[it];
                        float *save = (a.acts_out[it] && row_ok) ? a.acts_out[it] + ((size_t)pl * B + b) * kH : nullptr;
                        uint32_t *mask_out = (a.relu_mask_out && row_ok)
                            ? reinterpret_cast<uint32_t *>(a.relu_mask_out) + (((size_t)it * a.n_pol + pl) * B + b) * 8
                            : nullptr;
                        if (store_pending[slot]) { a_slot_guard(!store_pending[slot ^ 1]); store_pending[slot] = false; }
                        // An opaque copy of the row index: ptxas then derives the swizzled store addresses inside each epilogue
                        // instead of keeping values of r live across the work-unit loop (measured on B200, 1000 W: 52 instead of
                        // 80 B of spills, forward 37.6 instead of 38.6 us at the bench's headline size).
                        int rr = r;
                        asm volatile("" : "+r"(rr));
                        if (act == SFGPI_ACT_RELU) {
                            if (a.relu_mask_out) hidden_epilogue<SFGPI_ACT_RELU, 4, true>(t_lane, bias, Arow, rr, save, mask_out, group * 128);
                            else hidden_epilogue<SFGPI_ACT_RELU, 4, false>(t_lane, bias, Arow, rr, save, nullptr, group * 128);
                        } else if (act == SFGPI_ACT_NONE) hidden_epilogue<SFGPI_ACT_NONE, 4, false>(t_lane, bias, Arow, rr, save, nullptr, group * 128);
                        else hidden_epilogue<SFGPI_ACT_TANH, 4, false>(t_lane, bias, Arow, rr, save, nullptr, group * 128);
                        tc_fence_before();
                        fence_proxy_async();
                        mbar_arrive(SLOT_READY(slot));
                        if (saving) {                         // tile complete in shared memory -> one thread stores it
                            asm volatile("bar.sync 1, 256;" ::: "memory");
                            if (et == 0) {
                                const int row0 = (un.tile0 + slot) * kTM;
#pragma unroll
                                for (int kb = 0; kb < kH / kKB; ++kb)
                                    tma_store_3d(&maps.acts[jb], Arow + kb * (kTM * 128), kb * kKB, row0, it * a.n_pol + pl);
                                bulk_commit();
                            }
                            store_pending[slot] = true;
                        }
                    } else {
                        // ------ output layer chunk, GPI form (psi-form chunks always take the lean loop above) ------
                        // Rolled 8-column scan (gpi_scan_rolled, forward_tc.cuh): this code runs once per tile, so it is
                        // instruction-FETCH bound -- unrolled 32-column windows cost 9-13 k cycles per tile for 36 columns
                        // (profiles/r02_forward_chain.md), the rolled loop ~2.5 k.  Every emission is an atomicMax, so a chunk
                        // needs no state from the previous one and each group takes one 128-column half.
                        const uint32_t bias = bias_addr + 4u * ((1 + p.Lh) * kH + ii.col0);
                        const int col0_it = ii.col0, ncol = gpi_ncols(p.nw, A_), wblk = gpi_wblock(p.nw);
                        const uint32_t kstep = a.w_diag ? 0u : (uint32_t)B;
                        float *const q_row = (a.q_out != nullptr && row_ok) ? a.q_out + ((size_t)b * a.n_pol + pl) * A_ : nullptr;
                        long long *ka = a.key_action ? reinterpret_cast<long long *>(a.key_action) + (a.w_diag ? (size_t)pl * B : 0) + b : nullptr;
                        long long *kt = a.key_task ? reinterpret_cast<long long *>(a.key_task) + (a.w_diag ? (size_t)pl * B : 0) + b : nullptr;
                        const int c_hi = min(col0_it + ii.n_cols, ncol);
                        const int cb = wblk > 1 ? col0_it + group * 128 : (group == slot ? col0_it : c_hi);
                        const int ce = wblk > 1 ? min(cb + 128, c_hi) : c_hi;
                        const uint32_t tid_ = (uint32_t)(a.task_base + pl);
                        if (cb < ce) {
                            if (wblk == 8) gpi_scan_rolled<8>(t_lane, bias - 4u * col0_it, col0_it, cb, ce, A_, p.nw, ka, kt, kstep, row_ok, tid_, q_row);
                            else if (wblk == 4) gpi_scan_rolled<4>(t_lane, bias - 4u * col0_it, col0_it, cb, ce, A_, p.nw, ka, kt, kstep, row_ok, tid_, q_row);
                            else gpi_scan_rolled<1>(t_lane, bias - 4u * col0_it, col0_it, cb, ce, A_, p.nw, ka, kt, kstep, row_ok, tid_, q_row);
                        }
                        tc_fence_before();
                        if (it + 1 < p.n_items) mbar_arrive(SLOT_READY(slot));                  // next chunk may overwrite the accumulator
                    }
                    TL_EPI();                                 // epilogue of (item, slot) done
                }
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

// fp32 library rows -> bf16 shadow [n_pol][rows_per_policy][256]:
//   rows [0,256) W_0 (columns >= S zero), then hidden W_1..W_Lh, then W_out padded to n3pad rows.
__global__ void pack_bf16_kernel(sfgpi_net_desc net, const float *__restrict__ params, int policy_lo, int n_pol,
                                 __nv_bfloat16 *__restrict__ out, int rows_per_policy, int Lh) {
    pdl_launch_dependents();
    pdl_wait();
    const int AD = net.n_actions * net.n_features, L = net.n_layers, S = net.dims[0];
    const size_t total = (size_t)n_pol * rows_per_policy * kH;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int k = (int)(i % kH);
        const size_t rr = i / kH;
        const int row = (int)(rr % rows_per_policy), pl = (int)(rr / rows_per_policy);
        const float *P = params + (size_t)(policy_lo + pl) * net.row_stride;
        float v = 0.0f;
        if (row < kH) {
            if (k < S) v = P[net.w_off[0] + row * S + k];
        } else if (row < (1 + Lh) * kH) {
            const int l = row / kH, n = row % kH;
            v = P[net.w_off[l] + n * kH + k];
        } else {
            const int n = row - (1 + Lh) * kH;
            if (n < AD) v = P[net.w_off[L - 1] + n * kH + k];
        }
        out[((size_t)(policy_lo + pl) * rows_per_policy + row) * kH + k] = __float2bfloat16_rn(v);
    }
}

// GPI fold: Wq[pl][row(wi, act)][k] = sum_d w[wi][d] * W_out[pl][act*D + d][k]   (fp32 accumulate, bf16 out; row order: gpi_scan.cuh)
//           bq[pl][row(wi, act)]    = sum_d w[wi][d] * b_out[pl][act*D + d]
// One block per UNIT = (policy, action, up to kFoldBlocksPerUnit consecutive blocks of reward vectors), 256 threads = k: the
// D rows of W_out that belong to the action are read once (registers for D <= 16) and every folded row of the unit is D fused
// multiply-adds and one store.  (Round 1 had one block per folded ROW: at BASELINE config 4 -- 256 policies x 2304 rows --
// that is 590 k blocks of 12 multiply-adds per thread, and the step's prologue took 1.84 ms of a 7.1 ms step at the block
// scheduler's rate.)  One more unit per policy zeroes the padding rows [n_w-blocks * A, nqpad).
// Small folds (the headline step: 4 policies x 48 rows) keep one block per row (fold_row): there
// the serial loop over a unit's rows would only lengthen the step's dependent chain.  Both give the same bits: every output is
// the same fmaf chain over d = 0 .. D-1.
constexpr int kFoldBlocksPerUnit = 32;
constexpr int kFoldUnitMinRows = 4096;                        // folds with fewer rows in total: one block per row
__host__ __device__ inline int fold_units_per_policy(int nw, int A) {
    const int wb = gpi_wblock(nw), nblk = (nw + wb - 1) / wb;
    return A * ((nblk + kFoldBlocksPerUnit - 1) / kFoldBlocksPerUnit) + 1;
}
__device__ __forceinline__ void fold_row(const sfgpi_net_desc &net, const float *__restrict__ P, const float *__restrict__ w, int nw,
                                         int w_diag, int pl, int row, int k, __nv_bfloat16 *__restrict__ wq_pl, float *__restrict__ bq_pl) {
    const int A_ = net.n_actions, D = net.n_features, L = net.n_layers;
    float acc = 0.0f, bacc = 0.0f;
    int wi, act;
    gpi_row_to_wa(row, nw, A_, wi, act);
    if (row < gpi_ncols(nw, A_) && wi < nw) {
        const float *wv = w + (size_t)(w_diag ? pl : wi) * D;
        const float *Wo = P + net.w_off[L - 1] + (size_t)act * D * kH;
        const float *bo = P + net.b_off[L - 1] + act * D;
        for (int d = 0; d < D; ++d) {
            const float wd = wv[d];
            acc = fmaf(wd, Wo[d * kH + k], acc);
            bacc = fmaf(wd, bo[d], bacc);
        }
    }
    wq_pl[(size_t)row * kH + k] = __float2bfloat16_rn(acc);
    if (k == 0) bq_pl[row] = bacc;
}
__device__ __forceinline__ void fold_unit(const sfgpi_net_desc &net, const float *__restrict__ P, const float *__restrict__ w, int nw,
                                          int w_diag, int pl, int nqpad, int unit, int tid, __nv_bfloat16 *__restrict__ wq_pl,
                                          float *__restrict__ bq_pl) {
    __shared__ __align__(16) float w_s[kFoldBlocksPerUnit * 8][16];       // the unit's reward vectors, zero-padded to 16 features
    const int A_ = net.n_actions, D = net.n_features, L = net.n_layers;
    const int wb = gpi_wblock(nw), wlog = wb == 8 ? 3 : (wb == 4 ? 2 : 0);
    const int nblk = (nw + wb - 1) / wb, nchunk = (nblk + kFoldBlocksPerUnit - 1) / kFoldBlocksPerUnit;
    const int k4 = (tid & 63) * 4, rl = tid >> 6;            // 4 consecutive k of every 4th row
    if (unit == A_ * nchunk) {                                // padding rows
        for (int row = nblk * wb * A_ + rl; row < nqpad; row += 4) {
            *reinterpret_cast<uint2 *>(wq_pl + (size_t)row * kH + k4) = make_uint2(0u, 0u);
            if (k4 == 0) bq_pl[row] = 0.0f;
        }
        return;
    }
    const int act = unit / nchunk, b0 = (unit - act * nchunk) * kFoldBlocksPerUnit, b1 = min(b0 + kFoldBlocksPerUnit, nblk);
    const int i0 = b0 * wb, i1 = b1 * wb;                    // reward vectors [i0, i1) (padded count)
    const float *Wo = P + net.w_off[L - 1] + (size_t)act * D * kH + k4;
    const float *bo = P + net.b_off[L - 1] + act * D;
    const bool small_d = D <= 16;
    float4 wr[16];
    if (small_d) {
#pragma unroll 4
        for (int e = tid; e < (i1 - i0) * 16; e += 256) {
            const int i = i0 + (e >> 4), d = e & 15;
            w_s[e >> 4][d] = (i < nw && d < D) ? w[(size_t)(w_diag ? pl : i) * D + d] : 0.0f;
        }
#pragma unroll
        for (int d = 0; d < 16; ++d) wr[d] = d < D ? *reinterpret_cast<const float4 *>(Wo + d * kH) : make_float4(0.f, 0.f, 0.f, 0.f);
        __syncthreads();
    }
    float bor[16];                                           // the action's output biases (every thread: a uniform load each)
#pragma unroll
    for (int d = 0; d < 16; ++d) bor[d] = (small_d && d < D) ? bo[d] : 0.0f;
    for (int i = i0 + rl; i < i1; i += 4) {
        const int blk = i >> wlog, ws = i & (wb - 1), row = (blk * A_ + act) * wb + ws;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        float bacc = 0.0f;
        if (i < nw) {                                         // (vectors beyond n_w pad the last block: zero rows)
            const float *wv = w + (size_t)(w_diag ? pl : i) * D;
            if (small_d) {
                const float4 *ws4 = reinterpret_cast<const float4 *>(&w_s[i - i0][0]);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    if (4 * q < D) {
                        const float4 wq4 = ws4[q];
                        const float wd[4] = {wq4.x, wq4.y, wq4.z, wq4.w};
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            if (4 * q + u < D) {                  // same fmaf chain over d = 0 .. D-1 as fold_row
                                acc.x = fmaf(wd[u], wr[4 * q + u].x, acc.x); acc.y = fmaf(wd[u], wr[4 * q + u].y, acc.y);
                                acc.z = fmaf(wd[u], wr[4 * q + u].z, acc.z); acc.w = fmaf(wd[u], wr[4 * q + u].w, acc.w);
                                bacc = fmaf(wd[u], bor[4 * q + u], bacc);
                            }
                        }
                    }
                }
            } else {
                for (int d = 0; d < D; ++d) {
                    const float wd = __ldg(wv + d);
                    const float4 wo = *reinterpret_cast<const float4 *>(Wo + d * kH);
                    acc.x = fmaf(wd, wo.x, acc.x); acc.y = fmaf(wd, wo.y, acc.y);
                    acc.z = fmaf(wd, wo.z, acc.z); acc.w = fmaf(wd, wo.w, acc.w);
                    bacc = fmaf(wd, bo[d], bacc);
                }
            }
        }
        *reinterpret_cast<uint2 *>(wq_pl + (size_t)row * kH + k4) = make_uint2(pack_bf16x2(acc.x, acc.y), pack_bf16x2(acc.z, acc.w));
        if (k4 == 0) bq_pl[row] = bacc;
    }
}

// trace_slot: SFGPI_TR_PREP when the launch is the second half of a step's prologue (sfgpi_step_prep), else -1
__global__ void __launch_bounds__(256) fold_gpi_kernel(sfgpi_net_desc net, const float *__restrict__ params, int policy_lo,
                                                       const float *__restrict__ w, int nw, int w_diag, int nqpad, int by_unit, int trace_slot,
                                                       __nv_bfloat16 *__restrict__ wq, float *__restrict__ bq) {
    pdl_launch_dependents(trace_slot);
    pdl_wait(trace_slot);
    const int pl = blockIdx.y;
    const float *P = params + (size_t)(policy_lo + pl) * net.row_stride;
    if (by_unit) fold_unit(net, P, w, nw, w_diag, pl, nqpad, blockIdx.x, threadIdx.x, wq + (size_t)pl * nqpad * kH, bq + (size_t)pl * nqpad);
    else fold_row(net, P, w, nw, w_diag, pl, blockIdx.x, threadIdx.x, wq + (size_t)pl * nqpad * kH, bq + (size_t)pl * nqpad);
    if (trace_slot >= 0) trace_exit(trace_slot);
}

// ---- step prologue in ONE launch ---------------------------------------------------------------------------------------------
// Everything a tensor-core train step needs before its first GEMM is independent elementwise work on different buffers: the two
// bf16 shadow packs (online, target), the GPI key fill, the GPI fold and the backward pass's [x | 1 | 0] operand.  As five
// launches they cost five launch latencies on the step's dependent chain (~2-6 us each); here they are block ranges of one
// grid.  Same arithmetic as pack_bf16_kernel / keys_fill_kernel / fold_gpi_kernel / build_xo_kernel (bit-identical outputs),
// with 128-bit loads and stores in the packs.
struct PrepParams {
    sfgpi_step_prep_args a;
    int rows_per_policy, Lh, nqpad;
    int blk_end[6];                  // exclusive prefix ends of the block ranges: pack 0, pack 1, keys, fold, xo, TSF M / c
    int copy_end[SFGPI_PREP_COPIES]; // ... preceded by the staging copies' ranges (blocks [0, copy_end[5]))
    const void *copy_src_dev[SFGPI_PREP_COPIES];      // device-visible addresses of the (pinned host) sources
};

__device__ __forceinline__ void prep_pack8(const sfgpi_net_desc &net, const float *__restrict__ params, int policy_lo, long long item,
                                           __nv_bfloat16 *__restrict__ out, int rpp, int Lh) {
    const int AD = net.n_actions * net.n_features, L = net.n_layers, S = net.dims[0];
    const int k0 = (int)(item & 31) * 8;
    const long long rr = item >> 5;
    const int row = (int)(rr % rpp), pl = (int)(rr / rpp);
    const float *P = params + (size_t)(policy_lo + pl) * net.row_stride;
    float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (row < kH) {
#pragma unroll
        for (int i = 0; i < 8; ++i)
            if (k0 + i < S) v[i] = P[net.w_off[0] + row * S + k0 + i];
    } else {
        const float *src = nullptr;
        if (row < (1 + Lh) * kH) src = P + net.w_off[row / kH] + (size_t)(row % kH) * kH + k0;
        else if (row - (1 + Lh) * kH < AD) src = P + net.w_off[L - 1] + (size_t)(row - (1 + Lh) * kH) * kH + k0;
        if (src != nullptr) {
            if ((reinterpret_cast<uintptr_t>(src) & 15) == 0) {
                const float4 lo = *reinterpret_cast<const float4 *>(src), hi = *reinterpret_cast<const float4 *>(src + 4);
                v[0] = lo.x; v[1] = lo.y; v[2] = lo.z; v[3] = lo.w; v[4] = hi.x; v[5] = hi.y; v[6] = hi.z; v[7] = hi.w;
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] = src[i];
            }
        }
    }
    *reinterpret_cast<uint4 *>(out + ((size_t)(policy_lo + pl) * rpp + row) * kH + k0) =
        make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
}

__global__ void __launch_bounds__(256) step_prep_kernel(const __grid_constant__ PrepParams pp) {
    pdl_launch_dependents(SFGPI_TR_PREP);
    pdl_wait(SFGPI_TR_PREP);
    const sfgpi_step_prep_args &a = pp.a;
    const int tid = threadIdx.x;
    int bid = blockIdx.x;
    if (bid < a.tsf_n) {                                      // ---- TSF: M = Wh Wg, c = 2 (Wh bg + bh) of one policy (csrc/td.cu) ----
        // first in the grid (the longest chain of the launch: staging, then D*(S+1) dot products of length G)
        extern __shared__ __align__(16) float tsf_sm[];
        const int pl = bid, S = a.net.dims[0], D = a.net.n_features, G = a.tsf_G;
        float *Wg_s = tsf_sm, *bg_s = Wg_s + G * S, *Wh_s = bg_s + G, *bh_s = Wh_s + D * G;
        const float *gp = a.tsf_g + (size_t)(a.tsf_lo + pl) * a.tsf_g_stride;
        const uint32_t d0 = smem_u32(tsf_sm);
        for (int e = tid; e < G * S + G; e += 256)
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d0 + 4u * e), "l"(gp + e) : "memory");
        for (int e = tid; e < D * G + D; e += 256)
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d0 + 4u * (G * S + G + e)), "l"(a.tsf_h + e) : "memory");
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();
        float *mc = a.tsf_mc + (size_t)pl * (D * S + D);
        for (int o = tid; o < D * (S + 1); o += 256) {               // same dot products, same order as the TD kernel's own derivation
            const int d = o / (S + 1), sx = o - d * (S + 1);
            const float *wh = Wh_s + d * G;
            float acc = 0.0f;
            if (sx < S) {
                for (int g = 0; g < G; ++g) acc = fmaf(wh[g], Wg_s[g * S + sx], acc);
                mc[d * S + sx] = acc;
            } else {
                for (int g = 0; g < G; ++g) acc = fmaf(wh[g], bg_s[g], acc);
                mc[D * S + d] = 2.0f * (acc + bh_s[d]);
            }
        }
        trace_exit(SFGPI_TR_PREP);
        return;
    }
    bid -= a.tsf_n;
    if (bid < pp.copy_end[SFGPI_PREP_COPIES - 1]) {           // ---- staging copies (pinned host -> HBM over PCIe), first in the grid ----
        int j = 0;
        while (bid >= pp.copy_end[j]) ++j;
        const long long off = ((long long)(bid - (j ? pp.copy_end[j - 1] : 0)) * 256 + tid) * 16;
        const char *src = reinterpret_cast<const char *>(pp.copy_src_dev[j]);
        char *dst = reinterpret_cast<char *>(a.copy_dst[j]);
        const long long n = a.copy_bytes[j];
        if (off + 16 <= n && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0)
            *reinterpret_cast<uint4 *>(dst + off) = *reinterpret_cast<const uint4 *>(src + off);
        else
            for (long long q = off; q < min(off + 16, n); ++q) dst[q] = src[q];
        trace_exit(SFGPI_TR_PREP);
        return;
    }
    bid -= pp.copy_end[SFGPI_PREP_COPIES - 1];
    if (bid < pp.blk_end[1]) {                                // ---- bf16 shadow packs: 8 consecutive k per thread ----
        const int j = bid < pp.blk_end[0] ? 0 : 1;
        const long long item = (long long)(bid - (j ? pp.blk_end[0] : 0)) * 256 + tid;
        if (item < (long long)a.pack_n[j] * pp.rows_per_policy * 32)
            prep_pack8(a.net, a.pack_params[j], a.pack_lo[j], item, reinterpret_cast<__nv_bfloat16 *>(a.pack_out[j]), pp.rows_per_policy, pp.Lh);
    } else if (bid < pp.blk_end[2]) {                         // ---- GPI keys <- INT64_MIN, 2 per thread ----
        const long long i = ((long long)(bid - pp.blk_end[1]) * 256 + tid) * 2;
        long long *k = reinterpret_cast<long long *>(a.keys);
        if (i + 1 < a.n_keys && (reinterpret_cast<uintptr_t>(k) & 15) == 0) *reinterpret_cast<longlong2 *>(k + i) = make_longlong2(LLONG_MIN, LLONG_MIN);
        else {
            if (i < a.n_keys) k[i] = LLONG_MIN;
            if (i + 1 < a.n_keys) k[i + 1] = LLONG_MIN;
        }
    } else if (bid < pp.blk_end[3]) {                         // ---- GPI fold, small folds: one block per folded row (large ones: their own launch) ----
        const int u = bid - pp.blk_end[2];
        const int pl = u / pp.nqpad, row = u - pl * pp.nqpad;
        fold_row(a.net, a.fold_params + (size_t)(a.fold_lo + pl) * a.net.row_stride, a.w, a.w_diag ? 1 : a.n_w, a.w_diag, pl, row, tid,
                 reinterpret_cast<__nv_bfloat16 *>(a.wq) + (size_t)pl * pp.nqpad * kH, a.bq + (size_t)pl * pp.nqpad);
    } else {                                                  // ---- xo[b] = [x[b] | 1 | 0 ...] bf16 [B][64], 8 columns per thread ----
        const int i = (bid - pp.blk_end[3]) * 256 + tid;
        const int b = i >> 3, c0 = (i & 7) * 8, S = a.net.dims[0];
        if (b < a.B) {
            float v[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) v[q] = (c0 + q < S) ? a.x[(size_t)b * S + c0 + q] : ((c0 + q == S) ? 1.0f : 0.0f);
            *reinterpret_cast<uint4 *>(reinterpret_cast<__nv_bfloat16 *>(a.xo_bf16) + (size_t)b * 64 + c0) =
                make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
        }
    }
    trace_exit(SFGPI_TR_PREP);
}

static int make_tmap(CUtensorMap *tm, const void *base, uint64_t rows) {
    const TmapKey key = {base, {(uint64_t)kH, rows, 0}, {(uint32_t)kKB, (uint32_t)kNB, 0}, 2, 0, 0};
    if (tmap_cache_get(key, tm, false)) return SFGPI_OK;
    EncodeTiledFn encode = get_encode_fn();
    if (!encode) { set_error("cuTensorMapEncodeTiled entry point not found"); return SFGPI_E_CUDA; }
    const cuuint64_t gdim[2] = {(cuuint64_t)kH, (cuuint64_t)rows};
    const cuuint64_t gstride[1] = {(cuuint64_t)kH * 2};
    const cuuint32_t box[2] = {(cuuint32_t)kKB, (cuuint32_t)kNB};
    const cuuint32_t estride[2] = {1, 1};
    CUresult cr = encode(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void *>(base), gdim, gstride, box, estride,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed (%d)", (int)cr); return SFGPI_E_CUDA; }
    tmap_cache_get(key, tm, true);
    return SFGPI_OK;
}

// 3-D map of a [slabs][rows][256] bf16 tensor, box = {64 columns, 128 rows, 1 slab}: rows past the end of a slab are clipped
static int make_tmap_acts(CUtensorMap *tm, const void *base, uint64_t slabs, uint64_t rows) {
    const TmapKey key = {base, {(uint64_t)kH, rows, slabs}, {(uint32_t)kKB, (uint32_t)kTM, 1}, 3, 0, 0};
    if (tmap_cache_get(key, tm, false)) return SFGPI_OK;
    EncodeTiledFn encode = get_encode_fn();
    if (!encode) { set_error("cuTensorMapEncodeTiled entry point not found"); return SFGPI_E_CUDA; }
    const cuuint64_t gdim[3] = {(cuuint64_t)kH, (cuuint64_t)rows, (cuuint64_t)slabs};
    const cuuint64_t gstride[2] = {(cuuint64_t)kH * 2, (cuuint64_t)kH * 2 * rows};
    const cuuint32_t box[3] = {(cuuint32_t)kKB, (cuuint32_t)kTM, 1};
    const cuuint32_t estride[3] = {1, 1, 1};
    CUresult cr = encode(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void *>(base), gdim, gstride, box, estride,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(acts) failed (%d)", (int)cr); return SFGPI_E_CUDA; }
    tmap_cache_get(key, tm, true);
    return SFGPI_OK;
}

static int g_forward_chain = 1;
static int g_wide_min = 256;

// developer aid (SFGPI_TIMELINE=1): dump CTA 0's role timelines (cycles since the first stamp)
static void dump_timeline(long long *tl_buf, cudaStream_t st, int n_jobs, int units, int grid, const char *mode) {
    long long h[1280];
    cudaStreamSynchronize(st);
    cudaMemcpy(h, tl_buf, sizeof(h), cudaMemcpyDeviceToHost);
    long long t0 = 0;
    for (int i = 0; i < 512; ++i) if (h[i] && (!t0 || h[i] < t0)) t0 = h[i];
    if (h[256]) { fprintf(stderr, "  detail:"); for (int i = 256; i < 512 && h[i]; ++i) fprintf(stderr, " %lld", h[i] - t0); fprintf(stderr, "\n"); }
    { long long g0 = 0, g1 = 0, gs = 0; for (int i = 0; i < grid && i < 256; ++i) { if (!g0 || h[768 + i] < g0) g0 = h[768 + i]; if (h[768 + i] > gs) gs = h[768 + i]; if (h[1024 + i] > g1) g1 = h[1024 + i]; }
      fprintf(stderr, "  globaltimer: first CTA start -> last CTA start %lld ns, -> last CTA end %lld ns; CTA 0: %lld cycles in %lld ns = %.0f MHz\n", gs - g0, g1 - g0,
              h[512], h[1024] - h[768], 1000.0 * (double)h[512] / (double)(h[1024] - h[768])); }
    fprintf(stderr, "  per-CTA busy cycles (k):");
    for (int i = 0; i < grid && i < 256; ++i) fprintf(stderr, " %lld", h[512 + i] / 1000);
    fprintf(stderr, "\n");
    static const char *role[4] = {"epiX", "mma", "tma0", "epiY"};
    fprintf(stderr, "[sfgpi timeline] jobs=%d units=%d grid=%d %s\n", n_jobs, units, grid, mode);
    for (int r = 0; r < 4; ++r) {
        fprintf(stderr, "  %-4s:", role[r]);
        for (int i = 0; i < 64 && h[r * 64 + i]; ++i) fprintf(stderr, " %lld", h[r * 64 + i] - t0);
        fprintf(stderr, "\n");
    }
}

static bool tc_shape_ok(const sfgpi_net_desc &net, const char **why) {
    if (net.n_layers < 3) { *why = "needs >= 3 Linear layers"; return false; }
    for (int l = 1; l < net.n_layers; ++l)
        if (net.dims[l] != kH) { *why = "every hidden width must be 256"; return false; }
    if (net.dims[0] > 64) { *why = "state dimension must be <= 64"; return false; }
    if (net.acts[net.n_layers - 1] != SFGPI_ACT_NONE) { *why = "output layer must be linear"; return false; }
    return true;
}

}  // namespace tc
}  // namespace sfgpi

using namespace sfgpi;
using namespace sfgpi::tc;

// Runtime options of the tensor-core forward.  Each moves a choice between two code paths that give the same bits, which the
// code otherwise makes from the launch size, so that tests can run the other path and compare.  Returns the previous value,
// or -1 for an unknown option.
extern "C" int sfgpi_set_option(const char *name, int32_t value) {
    if (name != nullptr && strcmp(name, "forward_chain") == 0) {      // 0: never, 1 (default): launches of <= 148 tiles, 2: always
        const int old = g_forward_chain;
        g_forward_chain = value;
        return old;
    }
    if (name != nullptr && strcmp(name, "gpi_wide_min") == 0) {       // folded GPI columns from which the output chunks take the lean loop (gpi_scan_wide8)
        const int old = g_wide_min;
        g_wide_min = value;
        return old;
    }
    set_error("sfgpi_set_option: unknown option");
    return -1;
}

extern "C" int sfgpi_bf16_rows_per_policy(const sfgpi_net_desc *net) {
    const int AD = net->n_actions * net->n_features;
    return (net->n_layers - 1) * kH + ((AD + 15) & ~15);
}

extern "C" int sfgpi_gpi_fold_rows(const sfgpi_net_desc *net, int32_t n_w) { return (gpi_ncols(n_w, net->n_actions) + 15) & ~15; }

extern "C" int sfgpi_pack_bf16(const sfgpi_net_desc *net, const float *params, int32_t policy_lo, int32_t n_pol, void *out_bf16,
                               void *stream) {
    const char *why = "";
    if (!tc_shape_ok(*net, &why)) { set_error("sfgpi_pack_bf16: tensor-core path %s", why); return SFGPI_E_INVALID; }
    if (n_pol <= 0) return SFGPI_OK;
    const int Lh = net->n_layers - 2;
    const int rpp = sfgpi_bf16_rows_per_policy(net);
    const size_t total = (size_t)n_pol * rpp * kH;
    int blocks = (int)((total + 255) / 256);
    if (blocks > 148 * 16) blocks = 148 * 16;
    launch_pdl(pack_bf16_kernel, dim3(blocks), dim3(256), 0, (cudaStream_t)stream, *net, params, policy_lo, n_pol,
               reinterpret_cast<__nv_bfloat16 *>(out_bf16), rpp, Lh);
    return check_launch("sfgpi_pack_bf16");
}

// Folds reward vectors into the output layer for the GPI form.  wq_out: bf16 [n_pol][nqpad][256], bq_out: fp32 [n_pol][nqpad],
// nqpad = sfgpi_gpi_fold_rows(net, n_w) (n_w = 1 when w_diag).  w: [n_w][D] (w_diag: [n_pol][D], row p for policy slot p).
extern "C" int sfgpi_fold_gpi(const sfgpi_net_desc *net, const float *params, int32_t policy_lo, int32_t n_pol, const float *w,
                              int32_t n_w, int32_t w_diag, void *wq_out, float *bq_out, void *stream) {
    const char *why = "";
    if (!tc_shape_ok(*net, &why)) { set_error("sfgpi_fold_gpi: tensor-core path %s", why); return SFGPI_E_INVALID; }
    if (n_pol <= 0) return SFGPI_OK;
    const int nw = w_diag ? 1 : n_w;
    if (nw < 1) { set_error("sfgpi_fold_gpi: n_w must be >= 1"); return SFGPI_E_INVALID; }
    const int nqpad = sfgpi_gpi_fold_rows(net, nw);
    const int by_unit = (long long)nqpad * n_pol >= kFoldUnitMinRows ? 1 : 0;
    dim3 grid(by_unit ? fold_units_per_policy(nw, net->n_actions) : nqpad, n_pol);
    launch_pdl(fold_gpi_kernel, grid, dim3(256), 0, (cudaStream_t)stream, *net, params, policy_lo, w, nw, w_diag, nqpad, by_unit, -1,
               reinterpret_cast<__nv_bfloat16 *>(wq_out), bq_out);
    return check_launch("sfgpi_fold_gpi");
}

// Kernels one sfgpi_step_prep call launches: 2 when the GPI fold is large enough to run as its own launch, else 1.
extern "C" int sfgpi_step_prep_launches(const sfgpi_step_prep_args *args) {
    if (!args || args->fold_n <= 0) return 1;
    const int nw = args->w_diag ? 1 : args->n_w;
    return (long long)sfgpi_gpi_fold_rows(&args->net, nw) * args->fold_n >= kFoldUnitMinRows ? 2 : 1;
}

extern "C" int sfgpi_step_prep(const sfgpi_step_prep_args *args, void *stream) {
    trace_bind();
    if (!args) { set_error("sfgpi_step_prep: null args"); return SFGPI_E_INVALID; }
    PrepParams pp;
    pp.a = *args;
    const sfgpi_step_prep_args &a = pp.a;
    const char *why = "";
    if (!tc_shape_ok(a.net, &why)) { set_error("sfgpi_step_prep: tensor-core path %s", why); return SFGPI_E_INVALID; }
    pp.Lh = a.net.n_layers - 2;
    pp.rows_per_policy = sfgpi_bf16_rows_per_policy(&a.net);
    const int nw = a.w_diag ? 1 : a.n_w;
    pp.nqpad = a.fold_n > 0 ? sfgpi_gpi_fold_rows(&a.net, nw) : 0;
    const bool fold_apart = a.fold_n > 0 && (long long)pp.nqpad * a.fold_n >= kFoldUnitMinRows;       // large fold: its own launch, below
    if (a.fold_n > 0 && (nw < 1 || !a.fold_params || !a.w || !a.wq || !a.bq)) { set_error("sfgpi_step_prep: incomplete fold arguments"); return SFGPI_E_INVALID; }
    if (a.x != nullptr && (a.B < 0 || !a.xo_bf16 || a.net.dims[0] > 63)) { set_error("sfgpi_step_prep: invalid xo arguments"); return SFGPI_E_INVALID; }
    long long nc = 0;
    for (int j = 0; j < SFGPI_PREP_COPIES; ++j) {
        pp.copy_src_dev[j] = nullptr;
        if (a.copy_bytes[j] > 0) {
            if (!a.copy_src[j] || !a.copy_dst[j]) { set_error("sfgpi_step_prep: incomplete staging copy %d", j); return SFGPI_E_INVALID; }
            cudaPointerAttributes at;
            if (cudaPointerGetAttributes(&at, a.copy_src[j]) != cudaSuccess || at.type == cudaMemoryTypeUnregistered || !at.devicePointer) {
                // pageable host memory: the kernel cannot read it -> a plain stream-ordered copy ahead of the launch
                cudaGetLastError();
                if (cudaMemcpyAsync(a.copy_dst[j], a.copy_src[j], (size_t)a.copy_bytes[j], cudaMemcpyHostToDevice, (cudaStream_t)stream) != cudaSuccess)
                    return check_launch("sfgpi_step_prep(pageable staging copy)");
                if (a.x == a.copy_src[j]) pp.a.x = reinterpret_cast<const float *>(a.copy_dst[j]);
            } else {
                pp.copy_src_dev[j] = at.devicePointer;
                if (a.x == a.copy_src[j]) pp.a.x = reinterpret_cast<const float *>(at.devicePointer);
                nc += ((a.copy_bytes[j] + 15) / 16 + 255) / 256;
            }
        }
        pp.copy_end[j] = (int)nc;
    }
    long long n = 0;
    for (int j = 0; j < 2; ++j) {
        if (a.pack_n[j] > 0 && (!a.pack_params[j] || !a.pack_out[j])) { set_error("sfgpi_step_prep: incomplete pack arguments"); return SFGPI_E_INVALID; }
        if (a.pack_n[j] > 0) n += ((long long)a.pack_n[j] * pp.rows_per_policy * 32 + 255) / 256;
        pp.blk_end[j] = (int)n;
    }
    if (a.keys != nullptr && a.n_keys > 0) n += ((a.n_keys + 1) / 2 + 255) / 256;
    pp.blk_end[2] = (int)n;
    if (a.fold_n > 0 && !fold_apart) n += (long long)pp.nqpad * a.fold_n;
    pp.blk_end[3] = (int)n;
    if (a.x != nullptr && a.B > 0) n += ((long long)a.B * 8 + 255) / 256;
    pp.blk_end[4] = (int)n;
    size_t tsf_bytes = 0;
    if (a.tsf_n < 0) { set_error("sfgpi_step_prep: tsf_n < 0"); return SFGPI_E_INVALID; }
    if (a.tsf_n > 0) {
        if (!a.tsf_g || !a.tsf_h || !a.tsf_mc || a.tsf_G < 1) { set_error("sfgpi_step_prep: incomplete TSF M / c arguments"); return SFGPI_E_INVALID; }
        tsf_bytes = ((size_t)a.tsf_G * a.net.dims[0] + a.tsf_G + (size_t)a.net.n_features * a.tsf_G + a.net.n_features) * sizeof(float);
        if (tsf_bytes > 48 * 1024) { set_error("sfgpi_step_prep: g / h too large for the M / c blocks (%zu B)", tsf_bytes); return SFGPI_E_SMEM; }
        n += a.tsf_n;
    }
    pp.blk_end[5] = (int)n;
    n += nc;
    if (n > 0x7fffffffLL) { set_error("sfgpi_step_prep: too many blocks"); return SFGPI_E_INVALID; }
    if (n > 0) launch_pdl(step_prep_kernel, dim3((unsigned)n), dim3(256), tsf_bytes, (cudaStream_t)stream, pp);
    if (fold_apart) {
        // Large folds (BASELINE config 4: 256 policies x 2304 folded rows) run as a second launch of the prologue: fold units keep
        // 16 rows of the output layer in registers (fold_unit), which inside step_prep_kernel would cost the packs their occupancy.
        launch_pdl(fold_gpi_kernel, dim3(fold_units_per_policy(nw, a.net.n_actions), a.fold_n), dim3(256), 0, (cudaStream_t)stream, a.net,
                   a.fold_params, a.fold_lo, a.w, nw, a.w_diag, pp.nqpad, 1, (int)SFGPI_TR_PREP, reinterpret_cast<__nv_bfloat16 *>(a.wq), a.bq);
    }
    return check_launch("sfgpi_step_prep");
}

// mode-1 forward, up to 3 independent jobs in one launch.  Per job: `params_bf16` = shadow produced by sfgpi_pack_bf16 for
// the same `params` (n_policies_total row sets); GPI form (args.w != NULL) additionally needs wq / bq from sfgpi_fold_gpi for
// the same (policy_lo, n_pol, w).
extern "C" int sfgpi_mlp_forward_tc_jobs(const sfgpi_forward_tc_job *jobs, int32_t n_jobs, void *stream) {
    if (n_jobs < 1 || n_jobs > kMaxJobs) { set_error("sfgpi_mlp_forward_tc_jobs: 1..%d jobs per launch", kMaxJobs); return SFGPI_E_INVALID; }
    trace_bind();
    TcMulti m;
    TmapSet maps;
    m.n_jobs = 0;
    int total_tiles = 0;
    for (int j = 0; j < n_jobs; ++j) {
        const sfgpi_forward_args &a = jobs[j].args;
        const sfgpi_net_desc &net = a.net;
        const char *why = "";
        if (!tc_shape_ok(net, &why)) { set_error("sfgpi_mlp_forward_tc: tensor-core path %s", why); return SFGPI_E_INVALID; }
        if (a.B < 0 || a.n_pol < 0 || net.dims[net.n_layers] != net.n_actions * net.n_features) {
            set_error("sfgpi_mlp_forward_tc: invalid sizes");
            return SFGPI_E_INVALID;
        }
        if (a.B == 0 || a.n_pol == 0) continue;
        TcParams &p = m.job[m.n_jobs];
        p.a = a;
        p.gpi = a.w != nullptr ? 1 : 0;
        if (p.gpi && (a.psi_out || a.sel_out)) {
            set_error("sfgpi_mlp_forward_tc: the GPI form cannot also emit psi / gathered rows (use a separate job)");
            return SFGPI_E_INVALID;
        }
        if (p.gpi && (!jobs[j].wq || !jobs[j].bq)) { set_error("sfgpi_mlp_forward_tc: GPI form needs the folded weights"); return SFGPI_E_INVALID; }
        p.nw = p.gpi ? (a.w_diag ? 1 : a.n_w) : 0;
        p.Lh = net.n_layers - 2;
        p.rows_per_policy = sfgpi_bf16_rows_per_policy(&net);
        p.n_final = p.gpi ? sfgpi_gpi_fold_rows(&net, p.nw) : ((net.n_actions * net.n_features + 15) & ~15);
        p.n_items = 1 + p.Lh + (p.n_final + 255) / 256;
        p.ks0 = (net.dims[0] + 15) / 16;
        p.bq = jobs[j].bq;
        if ((1 + p.Lh) * kH + p.n_final > kBiasFloatsMax) {
            set_error("sfgpi_mlp_forward_tc: %d bias floats exceed the shared-memory budget", (1 + p.Lh) * kH + p.n_final);
            return SFGPI_E_SMEM;
        }
        p.tiles_per_policy = (a.B + kTM - 1) / kTM;
        total_tiles += p.tiles_per_policy * a.n_pol;
        int rc = make_tmap(&maps.w[m.n_jobs], jobs[j].params_bf16, (uint64_t)jobs[j].n_policies_total * p.rows_per_policy);
        if (rc) return rc;
        if (p.gpi) {
            rc = make_tmap(&maps.q[m.n_jobs], jobs[j].wq, (uint64_t)a.n_pol * p.n_final);
            if (rc) return rc;
        } else {
            maps.q[m.n_jobs] = maps.w[m.n_jobs];
        }
        maps.acts[m.n_jobs] = maps.w[m.n_jobs];
        if (a.acts_bf16_out != nullptr) {                        // [L-1][n_pol][B][256] bf16, stored tile by tile with TMA
            rc = make_tmap_acts(&maps.acts[m.n_jobs], a.acts_bf16_out, (uint64_t)(net.n_layers - 1) * a.n_pol, (uint64_t)a.B);
            if (rc) return rc;
        }
        ++m.n_jobs;
    }
    if (m.n_jobs == 0) return SFGPI_OK;
    static long long *tl_buf = nullptr;
    static const bool tl_on = getenv("SFGPI_TIMELINE") != nullptr;
    if (tl_on && !tl_buf) cudaMalloc(&tl_buf, 1280 * sizeof(long long));
    if (tl_on) cudaMemsetAsync(tl_buf, 0, 1280 * sizeof(long long), (cudaStream_t)stream);
    m.timeline = tl_on ? tl_buf : nullptr;
    m.wide_min = g_wide_min;
    const int paired = total_tiles > 148 ? 1 : 0;                // small launches: one tile per CTA, no ping-pong partner
    // Launches that fit in ONE wave (<= 148 row tiles: every CTA has a single tile, nothing to ping-pong with) take the layer-
    // pipelined single-tile kernel (mlp_chain_tc.cu): measured 84 vs 90 us per B = 32 step.  Larger launches keep the ping-pong
    // pairs: with the MMA phase shared-memory-bound at ~3 k cycles per tile-layer, overlapping it with ANOTHER tile's epilogue
    // (3.1 k per tile-layer) beats overlapping it with its own tile's previous epilogue (~5 k), 50 vs 52 us at 384 tiles.
    // sfgpi_set_option("forward_chain", 0 / 1 / 2) = never / one-wave launches (default) / always.
    if (g_forward_chain && (g_forward_chain > 1 || total_tiles <= 148) && forward_chain_supported(m)) {
        for (int j = m.n_jobs; j < kMaxJobs; ++j) { m.job[j] = m.job[0]; maps.w[j] = maps.w[0]; maps.q[j] = maps.q[0]; maps.acts[j] = maps.acts[0]; }
        const int grid = launch_forward_chain(m, maps, total_tiles, (cudaStream_t)stream);
        if (tl_on) dump_timeline(tl_buf, (cudaStream_t)stream, m.n_jobs, m.total_pairs, grid, "chain (one tile, layer-pipelined)");
        return check_launch("sfgpi_mlp_forward_tc(chain)");
    }
    m.total_pairs = 0;
    m.paired = paired;
    for (int j = 0; j < m.n_jobs; ++j) {
        TcParams &p = m.job[j];
        p.paired = paired;
        p.pairs_per_policy = paired ? (p.tiles_per_policy + 1) / 2 : p.tiles_per_policy;
        p.total_pairs = p.pairs_per_policy * p.a.n_pol;
        m.pair_start[j] = m.total_pairs;
        m.total_pairs += p.total_pairs;
    }
    for (int j = m.n_jobs; j <= kMaxJobs; ++j) m.pair_start[j] = m.total_pairs;
    // Balanced schedule (see UnitTable): r = floor(tiles / 2G) full rounds of pairs, and when the remainder fits in ONE more
    // round of single tiles (<= G) it runs as singles instead of as pairs on a few CTAs.  Pairs are listed cheapest first
    // and singles dearest first (jobs that save activations have the longer epilogues), so CTA c -- which takes units
    // c, c + G, ... -- combines a cheap pair with a single, and the dear pairs at the end of the round get no second unit.
    static UnitTable ut;                                         // (host scratch; the launch copies it into the kernel parameters)
    m.sched = 0;
    {
        const int G = 148, rounds = total_tiles / (2 * G), left = total_tiles - 2 * rounds * G;
        int q_total = 0;
        for (int j = 0; j < m.n_jobs; ++j) q_total += m.job[j].a.n_pol;
        if (paired && rounds >= 1 && left > 0 && left <= G && q_total <= 0x1FFF) {
            const int p_target = rounds * G;
            int order[kMaxJobs], nj = m.n_jobs;
            for (int j = 0; j < nj; ++j) order[j] = j;
            auto dear = [&](int j) { return m.job[j].a.acts_bf16_out != nullptr ? 1 : 0; };
            for (int i = 0; i < nj; ++i)                      // cheapest jobs first (stable)
                for (int k = i + 1; k < nj; ++k)
                    if (dear(order[k]) < dear(order[i])) { int t = order[i]; order[i] = order[k]; order[k] = t; }
            int n_units = 0;
            bool ok = true;
            // Which tiles run as singles: a lone tile costs ~1.6x a paired one (nothing hides its MMA phase) and the jobs that save
            // activations have the longer epilogues, so the singles are taken from the CHEAPEST jobs first and every other tile
            // is paired.
            static int np_buf[0x2000];
            int qi = 0, given = 0;
            int singles_left = total_tiles - 2 * p_target;
            for (int oi = 0; oi < nj && ok; ++oi) {
                const TcParams &p = m.job[order[oi]];
                if (p.tiles_per_policy > 0xFFFF) { ok = false; break; }
                for (int pl = 0; pl < p.a.n_pol; ++pl, ++qi) {
                    int s1 = singles_left < p.tiles_per_policy ? singles_left : p.tiles_per_policy;
                    if ((p.tiles_per_policy - s1) & 1) s1 += (s1 < p.tiles_per_policy) ? 1 : -1;      // the rest pairs up
                    singles_left -= s1;
                    const int share = (p.tiles_per_policy - s1) / 2;
                    np_buf[qi] = share;
                    given += share;
                }
            }
            const int singles = total_tiles - 2 * given;
            if (ok && given + singles <= kMaxUnits) {
                qi = 0;
                for (int oi = 0; oi < nj; ++oi) {             // pairs, cheapest job first
                    const int j = order[oi];
                    for (int pl = 0; pl < m.job[j].a.n_pol; ++pl, ++qi)
                        for (int k = 0; k < np_buf[qi]; ++k)
                            ut.u[n_units++] = ((uint32_t)j << 30) | (1u << 29) | ((uint32_t)pl << 16) | (uint32_t)(2 * k);
                }
                for (int oi = nj - 1; oi >= 0; --oi) {        // singles, dearest job first
                    const int j = order[oi];
                    int qj = 0;
                    for (int o2 = 0; o2 < oi; ++o2) qj += m.job[order[o2]].a.n_pol;
                    for (int pl = 0; pl < m.job[j].a.n_pol; ++pl)
                        for (int t = 2 * np_buf[qj + pl]; t < m.job[j].tiles_per_policy; ++t)
                            ut.u[n_units++] = ((uint32_t)j << 30) | ((uint32_t)pl << 16) | (uint32_t)t;
                }
                m.sched = 1;
                m.total_pairs = n_units;
            }
        }
    }
    for (int j = m.n_jobs; j < kMaxJobs; ++j) { m.job[j] = m.job[0]; maps.w[j] = maps.w[0]; maps.q[j] = maps.q[0]; maps.acts[j] = maps.acts[0]; }
    const int smem_bytes = 2 * kABytes + kNStage * kStageBytes + kBiasFloatsMax * 4 + 256;
    static bool cfg = false;
    if (!cfg) {
        cudaFuncSetAttribute(mlp_forward_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
        cfg = true;
    }
    const int grid = m.total_pairs < 148 ? m.total_pairs : 148;
    launch_pdl(mlp_forward_tc_kernel, dim3(grid), dim3(kThreadsTc), smem_bytes, (cudaStream_t)stream, m, maps, ut);
    if (tl_on) dump_timeline(tl_buf, (cudaStream_t)stream, m.n_jobs, m.total_pairs, grid, m.sched ? "pairs + singles (unit table)" : (paired ? "paired" : "one-tile"));
    return check_launch("sfgpi_mlp_forward_tc");
}

extern "C" int sfgpi_mlp_forward_tc(const sfgpi_forward_args *args, const void *params_bf16, int32_t n_policies_total,
                                    const void *wq, const float *bq, void *stream) {
    sfgpi_forward_tc_job job;
    job.args = *args;
    job.params_bf16 = params_bf16;
    job.n_policies_total = n_policies_total;
    job.wq = wq;
    job.bq = bq;
    return sfgpi_mlp_forward_tc_jobs(&job, 1, stream);
}
