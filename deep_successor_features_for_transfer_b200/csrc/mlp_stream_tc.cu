// Ensemble psi-MLP forward on the tensor cores at the REFERENCE's precision: tcgen05.mma kind::tf32 on fp32 operands,
// one pass (TF32, stated tolerance 2e-3) or the 3-pass split a_hi.b_hi + a_hi.b_lo + a_lo.b_hi (TF32X3: the 1e-5 parity mode),
// fp32 accumulation in TMEM.  See stream_tc.cuh for the measured numerics.
//
// fp32 operands are twice as wide as bf16 and the split needs a hi AND a lo copy of each, so a whole 128 x 256 activation tile
// (hi + lo = 256 KB) can no longer sit in shared memory as the next layer's A operand the way the bf16 kernel
// (mlp_forward_tc.cu) keeps it.  This kernel therefore STREAMS the layer chain by k-blocks of 32 columns:
//
//   epilogue warps (8)   drain 32 accumulator columns of layer l (tcgen05.ld), add bias, activate, split into hi / lo and write
//                        them as ONE k-block of layer l+1's A operand (K-major SWIZZLE_128B, 16 KB per part) into a small ring;
//   MMA warp             as soon as A k-block kb and the matching weight k-block have landed, issues layer l+1's MMAs for
//                        that k-block into the OTHER accumulator (TMEM: 2 x 256 columns, ping-pong between layers);
//   TMA producer warps   stream the fp32 hi / lo weight k-blocks (256 rows x 32 k per part).
//
// So layer l+1's tensor-core work overlaps layer l's epilogue k-block by k-block, the A operand never exists as a whole, and
// shared memory holds 2 (TF32X3) or 4 (TF32) ring stages of (A 16 KB + B 32 KB) per part.  In TF32X3 a k-block costs
// 12 MMAs x 128 cycles = 1536 tensor cycles against ~400 epilogue cycles: the pipe stays busy with ONE tile per CTA.
// Output layer in more than one 256-column chunk (Hopper psi: 1350 columns; folded GPI with many reward vectors): every chunk
// goes to the same accumulator and the epilogue RE-produces the A k-blocks from the last hidden layer's accumulator, which
// stays in TMEM untouched -- no activation scratch in HBM.
#include "stream_tc.cuh"
#include "gpi_scan.cuh"
#include <limits.h>
#include <stdlib.h>

namespace sfgpi {
namespace tc {

constexpr int kSThreads = 416;                       // 4 producer warps + 1 MMA warp + 8 epilogue warps
constexpr int kSMmaWarp = 4, kSEpiWarp0 = 5;
constexpr int kAPart = kTM * 128;                    // 16 KB: 128 rows x 32 fp32 of an A k-block (one part)
constexpr int kBBox = 128 * 128;                     // 16 KB: 128 weight rows x 32 fp32 (one TMA box)
constexpr int kBPart = 2 * kBBox;                    // 32 KB: up to 256 weight rows of a B k-block (one part)
constexpr int kSBiasFloats = 6144;
constexpr int kSMaxJobs = 3;

struct SJob {
    sfgpi_forward_args a;
    int rows_per_policy;     // rows of the fp32 shadow per policy = (1 + Lh) * 256 + n3pad
    int n_final;             // output columns computed (padded to 16)
    int Lh, n_items, ks0, gpi, nw;
    int tiles_per_policy, unit_start;
    int w_part_rows, q_part_rows;        // rows per part in the w / q tensor maps
    const float *bq;
};
struct SMulti {
    int n_jobs, total_units;
    SJob job[kSMaxJobs];
};
struct SMaps { CUtensorMap w[kSMaxJobs]; CUtensorMap q[kSMaxJobs]; CUtensorMap acts[kSMaxJobs]; };

struct SItem { int row_base, n_cols, col0, n_kb, n_k8; bool folded; };

__device__ __forceinline__ SItem s_item(const SJob &p, int it) {
    SItem r;
    r.folded = false;
    if (it == 0) { r.row_base = 0; r.n_cols = kH; r.col0 = 0; r.n_kb = 1; r.n_k8 = p.ks0; }
    else if (it <= p.Lh) { r.row_base = it * kH; r.n_cols = kH; r.col0 = 0; r.n_kb = kH / kK32; r.n_k8 = 4; }
    else {
        const int c = it - 1 - p.Lh;
        r.col0 = c * 256;
        r.n_cols = min(256, p.n_final - r.col0);
        r.row_base = (p.gpi ? 0 : (1 + p.Lh) * kH) + r.col0;
        r.n_kb = kH / kK32; r.n_k8 = 4;
        r.folded = p.gpi != 0;
    }
    return r;
}

__device__ __forceinline__ int s_job_of_unit(const SMulti &m, int g) {
    int j = 0;
    while (j + 1 < m.n_jobs && g >= m.job[j + 1].unit_start) ++j;
    return j;
}

// Barriers of the streaming pipeline (byte offsets from bar0)
struct SBars {
    uint32_t b0;
    __device__ __forceinline__ uint32_t a_full(int s) const { return b0 + 8u * s; }
    __device__ __forceinline__ uint32_t a_empty(int s) const { return b0 + 8u * (4 + s); }
    __device__ __forceinline__ uint32_t b_full(int s) const { return b0 + 8u * (8 + s); }
    __device__ __forceinline__ uint32_t b_empty(int s) const { return b0 + 8u * (12 + s); }
    __device__ __forceinline__ uint32_t acc_full(int a) const { return b0 + 8u * (16 + a); }
    __device__ __forceinline__ uint32_t acc_empty(int a) const { return b0 + 8u * (18 + a); }
    __device__ __forceinline__ uint32_t holder() const { return b0 + 8u * 20; }
};

__device__ __forceinline__ void s_bars_init(const SBars &bars) {
    for (int s = 0; s < 4; ++s) {
        mbar_init(bars.a_full(s), 1); mbar_init(bars.a_empty(s), 1);
        mbar_init(bars.b_full(s), 4); mbar_init(bars.b_empty(s), 1);
    }
    for (int a = 0; a < 2; ++a) { mbar_init(bars.acc_full(a), 1); mbar_init(bars.acc_empty(a), 1); }
    fence_mbar_init();
}

// ---- MMA issue for one k-block: A stage x B stage -> accumulator d (whole warp, elected lane issues) ----
template <int PARTS>
__device__ __forceinline__ void s_issue_kblock(uint32_t d, uint32_t a_stage, uint32_t b_stage, uint32_t idesc, int n_k8, bool first,
                                               uint32_t leader) {
    const uint64_t ah = umma_desc_k_sw128(a_stage), bh = umma_desc_k_sw128(b_stage);
    if (PARTS == 2) {
        const uint64_t al = umma_desc_k_sw128(a_stage + kAPart), bl = umma_desc_k_sw128(b_stage + kBPart);
        for (int k8 = 0; k8 < n_k8; ++k8) {               // small terms first, the hi.hi product last
            umma_tf32_e(d, al + 2 * k8, bh + 2 * k8, idesc, (first && k8 == 0) ? 0u : 1u, leader);
            umma_tf32_e(d, ah + 2 * k8, bl + 2 * k8, idesc, 1u, leader);
            umma_tf32_e(d, ah + 2 * k8, bh + 2 * k8, idesc, 1u, leader);
        }
    } else {
        for (int k8 = 0; k8 < n_k8; ++k8) umma_tf32_e(d, ah + 2 * k8, bh + 2 * k8, idesc, (first && k8 == 0) ? 0u : 1u, leader);
    }
}

// ---- epilogue: 16 accumulator columns of one row -> bias + activation -> hi / lo -> A k-block stage ----
// v: raw accumulator words; cb = first column inside the 32-column k-block (0 or 16); returns the sign bits (h > 0).
template <int PARTS>
__device__ __forceinline__ uint32_t s_write_a16(const float (&h)[16], uint32_t stage, int r, int cb) {
    uint32_t bits = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        float hi[4], lo[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float x = h[4 * q + i];
            bits |= (x > 0.f ? 1u : 0u) << (4 * q + i);
            hi[i] = tf32_rna(x);
            lo[i] = tf32_rna(x - hi[i]);          // exactly representable: the tensor core's truncation of lo is then a no-op
        }
        const uint32_t off = a32_chunk_off(r, cb + 4 * q);
        sts128(stage + off, __float_as_uint(hi[0]), __float_as_uint(hi[1]), __float_as_uint(hi[2]), __float_as_uint(hi[3]));
        if (PARTS == 2)
            sts128(stage + kAPart + off, __float_as_uint(lo[0]), __float_as_uint(lo[1]), __float_as_uint(lo[2]), __float_as_uint(lo[3]));
    }
    return bits;
}

template <int PARTS>
__global__ void __launch_bounds__(kSThreads, 1)
mlp_forward_stream_kernel(const __grid_constant__ SMulti m, const __grid_constant__ SMaps maps) {
    constexpr int NS = PARTS == 2 ? 2 : 4;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    pdl_launch_dependents();
    const uint32_t sbase = smem_u32(smem_raw);
    const uint32_t A_addr = sbase, B_addr = sbase + NS * PARTS * kAPart;
    const uint32_t bias_addr = B_addr + NS * PARTS * kBPart;
    SBars bars;
    bars.b0 = bias_addr + kSBiasFloats * 4;
    if (threadIdx.x == 0) {
        s_bars_init(bars);
        for (int j = 0; j < m.n_jobs; ++j) {
            tma_prefetch_desc(&maps.w[j]);
            if (m.job[j].gpi) tma_prefetch_desc(&maps.q[j]);
        }
    }
    if (warp == kSMmaWarp) tmem_alloc(bars.holder(), 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(bars.holder()));
    pdl_wait();

    auto unit_decode = [&](int g, int &jb, int &pl, int &tile) {
        jb = s_job_of_unit(m, g);
        const int u = g - m.job[jb].unit_start;
        pl = u / m.job[jb].tiles_per_policy;
        tile = u - pl * m.job[jb].tiles_per_policy;
    };

    if (warp < 4) {
        // =========================== TMA producers: the weight k-blocks ===========================
        // A stage holds PARTS x up to 2 boxes of 128 rows; box b = warp is issued by producer warp `warp` (<= 4 boxes per stage),
        // every producer warp arrives once per stage (with or without bytes), so B_FULL counts 4.
        const uint32_t leader = elect_one();
        uint32_t n = 0;
        for (int g = blockIdx.x; g < m.total_units; g += gridDim.x) {
            int jb, pl, tile;
            unit_decode(g, jb, pl, tile);
            const SJob &p = m.job[jb];
            for (int it = 0; it < p.n_items; ++it) {
                const SItem ii = s_item(p, it);
                const int nblocks = (ii.n_cols + 127) / 128;
                const void *tm = ii.folded ? (const void *)&maps.q[jb] : (const void *)&maps.w[jb];
                const int part_rows = ii.folded ? p.q_part_rows : p.w_part_rows;
                const int part = warp % PARTS, nb = warp / PARTS;
                const bool has_box = warp < PARTS * nblocks;
                const int row = part * part_rows + (ii.folded ? pl * p.n_final : (p.a.policy_lo + pl) * p.rows_per_policy) + ii.row_base + nb * 128;
                for (int kb = 0; kb < ii.n_kb; ++kb, ++n) {
                    const int s = n % NS;
                    mbar_wait_warp(bars.b_empty(s), ((n / NS) & 1) ^ 1);
                    if (has_box) {
                        mbar_arrive_expect_tx_e(bars.b_full(s), kBBox, leader);
                        tma_load_2d_e(B_addr + (s * PARTS + part) * kBPart + nb * kBBox, tm, bars.b_full(s), kb * kK32, row, leader);
                    } else if (leader) {
                        mbar_arrive(bars.b_full(s));
                    }
                }
            }
        }
    } else if (warp == kSMmaWarp) {
        // =========================== MMA issuer ===========================
        const uint32_t leader = elect_one();
        uint32_t n = 0, acc_use[2] = {0, 0};
        for (int g = blockIdx.x; g < m.total_units; g += gridDim.x) {
            int jb, pl, tile;
            unit_decode(g, jb, pl, tile);
            const SJob &p = m.job[jb];
            for (int it = 0; it < p.n_items; ++it) {
                const SItem ii = s_item(p, it);
                const int dst = (it <= p.Lh ? it : p.Lh + 1) & 1;
                mbar_wait_warp(bars.acc_empty(dst), (acc_use[dst] & 1) ^ 1);          // the epilogue has drained this accumulator
                ++acc_use[dst];
                tc_fence_after();
                const uint32_t d = tmem_base + (uint32_t)dst * 256u;
                const uint32_t idesc = idesc_tf32(kTM, (uint32_t)ii.n_cols, 0u, 0u);
                for (int kb = 0; kb < ii.n_kb; ++kb, ++n) {
                    const int s = n % NS;
                    mbar_wait_warp(bars.a_full(s), (n / NS) & 1);
                    mbar_wait_warp(bars.b_full(s), (n / NS) & 1);
                    tc_fence_after();
                    s_issue_kblock<PARTS>(d, A_addr + s * PARTS * kAPart, B_addr + s * PARTS * kBPart, idesc, ii.n_k8, kb == 0, leader);
                    umma_commit_e(bars.a_empty(s), leader);
                    umma_commit_e(bars.b_empty(s), leader);
                }
                umma_commit_e(bars.acc_full(dst), leader);
            }
        }
    } else {
        // =========================== epilogue warps ===========================
        const int group = (warp - kSEpiWarp0) >> 2;         // column half inside a k-block
        const int quad = warp & 3;                          // TMEM lane quadrant this warp may access
        const int r = quad * 32 + lane;                     // row inside the tile == TMEM lane
        const int et = threadIdx.x - kSEpiWarp0 * 32;       // 0..255
        const uint32_t t_lane0 = tmem_base + ((uint32_t)(quad * 32) << 16);
        uint32_t n = 0, full_cnt[2] = {0, 0};
        int cur_policy = -1;
        bool store_in_flight = false;
        auto bar_epi = [&]() { asm volatile("bar.sync 1, 256;" ::: "memory"); };
        // hand a finished A k-block (stage s) to the MMA warp; saving: also bulk-store its parts to the activation tensor
        auto publish = [&](int s, const CUtensorMap *tm, int c0, int row0, int slab0, int slab_part_stride) {
            fence_proxy_async();
            if (et == 0 && store_in_flight) bulk_wait_read0();      // the previous k-block's store has finished reading ITS stage
            bar_epi();
            if (et == 0) {
                mbar_arrive(bars.a_full(s));
                if (tm != nullptr) {
#pragma unroll
                    for (int part = 0; part < PARTS; ++part)
                        tma_store_3d(tm, A_addr + (s * PARTS + part) * kAPart, c0, row0, slab0 + part * slab_part_stride);
                    bulk_commit();
                }
            }
            store_in_flight = tm != nullptr;
        };
        auto release_acc = [&](int a) {
            tc_fence_before();
            bar_epi();
            if (et == 0) mbar_arrive(bars.acc_empty(a));
        };

        for (int g = blockIdx.x; g < m.total_units; g += gridDim.x) {
            int jb, pl, tile;
            unit_decode(g, jb, pl, tile);
            const SJob &p = m.job[jb];
            const sfgpi_forward_args &a = p.a;
            const sfgpi_net_desc &net = a.net;
            const int B = a.B, L = net.n_layers, A_ = net.n_actions, D = net.n_features, AD = A_ * D, S = net.dims[0];
            const int n_bias = (1 + p.Lh) * kH + p.n_final;
            const float *P = a.params + (size_t)(a.policy_lo + pl) * net.row_stride;
            const int b = tile * kTM + r;
            const bool row_ok = b < B;

            // ---- item 0's A operand: the state tile (k-block 0, columns [0, 8 ks0), zero-padded) ----
            {
                const int s = n % NS;
                mbar_wait(bars.a_empty(s), ((n / NS) & 1) ^ 1);
                if (group == 0) {
                    const float *xr = a.x + (size_t)b * S;
                    const uint32_t stage = A_addr + s * PARTS * kAPart;
                    for (int c = 0; c < p.ks0 * 8; c += 4) {
                        float hi[4], lo[4];
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const float x = (row_ok && c + i < S) ? xr[c + i] : 0.0f;
                            hi[i] = tf32_rna(x);
                            lo[i] = tf32_rna(x - hi[i]);          // exactly representable: the tensor core's truncation of lo is then a no-op
                        }
                        const uint32_t off = a32_chunk_off(r, c);
                        sts128(stage + off, __float_as_uint(hi[0]), __float_as_uint(hi[1]), __float_as_uint(hi[2]), __float_as_uint(hi[3]));
                        if (PARTS == 2)
                            sts128(stage + kAPart + off, __float_as_uint(lo[0]), __float_as_uint(lo[1]), __float_as_uint(lo[2]), __float_as_uint(lo[3]));
                    }
                }
                publish(s, nullptr, 0, 0, 0, 0);
                ++n;
            }
            int sel_base = -(1 << 30);
            if (a.sel_out != nullptr && row_ok) {
                const int sidx = a.sel_actions ? (int)a.sel_actions[b] : (int)key_index(a.sel_keys[(size_t)pl * a.sel_key_stride + b]);
                sel_base = sidx * D;
            }
            // biases of this (job, policy) -> shared memory (their latency hides behind the input layer's MMAs)
            if (jb * 65536 + pl != cur_policy) {
                bar_epi();
                for (int e = et; e < n_bias; e += 256) {
                    float v = 0.0f;
                    if (e < (1 + p.Lh) * kH) v = P[net.b_off[e >> 8] + (e & 255)];
                    else {
                        const int c = e - (1 + p.Lh) * kH;
                        v = p.gpi ? p.bq[(size_t)pl * p.n_final + c] : (c < AD ? P[net.b_off[L - 1] + c] : 0.0f);
                    }
                    sts32(bias_addr + 4u * e, v);
                }
                bar_epi();
                cur_policy = jb * 65536 + pl;
            }

            // GPI running state (folded form)
            float best = -INFINITY;
            int best_a = 0, wi = 0, act_i = 0;
            float bb[8];
            int ba[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) { bb[i] = -INFINITY; ba[i] = 0; }
            const bool saving = a.acts_bf16_out != nullptr;

            for (int it = 1; it < p.n_items; ++it) {
                const int src = min(it - 1, p.Lh), src_acc = src & 1;
                const bool first_prod = it - 1 <= p.Lh;          // first production from this accumulator (later ones: re-production)
                if (first_prod) {
                    mbar_wait(bars.acc_full(src_acc), full_cnt[src_acc] & 1);
                    ++full_cnt[src_acc];
                    tc_fence_after();
                }
                const int act = net.acts[src];
                const uint32_t t_src = t_lane0 + (uint32_t)src_acc * 256u;
                const bool save_here = saving && first_prod;
                uint16_t *mask_row = (first_prod && a.relu_mask_out && row_ok && act == SFGPI_ACT_RELU)
                    ? reinterpret_cast<uint16_t *>(reinterpret_cast<uint32_t *>(a.relu_mask_out) + (((size_t)src * a.n_pol + pl) * B + b) * 8)
                    : nullptr;
                // ------ 8 k-blocks of the next A operand from the 256 accumulator columns of layer `src` ------
#pragma unroll 1
                for (int kb = 0; kb < kH / kK32; ++kb, ++n) {
                    const int s = n % NS;
                    mbar_wait(bars.a_empty(s), ((n / NS) & 1) ^ 1);
                    uint32_t v[16];
                    const int c0 = kb * kK32 + group * 16;
                    tmem_ld16(t_src + c0, v);
                    float h[16];
                    const uint32_t bias = bias_addr + 4u * (src * kH + c0);
                    tmem_wait_ld();
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const float4 bv = lds128(bias + 16u * q);
                        h[4 * q] = __uint_as_float(v[4 * q]) + bv.x; h[4 * q + 1] = __uint_as_float(v[4 * q + 1]) + bv.y;
                        h[4 * q + 2] = __uint_as_float(v[4 * q + 2]) + bv.z; h[4 * q + 3] = __uint_as_float(v[4 * q + 3]) + bv.w;
                    }
                    if (act == SFGPI_ACT_RELU) {
#pragma unroll
                        for (int i = 0; i < 16; ++i) h[i] = fmaxf(h[i], 0.f);
                    } else if (act == SFGPI_ACT_TANH) {
#pragma unroll
                        for (int i = 0; i < 16; ++i) h[i] = tanhf(h[i]);
                    }
                    const uint32_t bits = s_write_a16<PARTS>(h, A_addr + s * PARTS * kAPart, r, group * 16);
                    if (mask_row != nullptr) mask_row[kb * 2 + group] = (uint16_t)bits;
                    publish(s, save_here ? &maps.acts[jb] : nullptr, kb * kK32, tile * kTM, src * a.n_pol + pl, (L - 1) * a.n_pol);
                }
                if (it <= p.Lh || it == p.n_items - 1) release_acc(src_acc);      // last reader of this accumulator
                if (it <= p.Lh) continue;

                // ------ output layer chunk: drain the destination accumulator ------
                const SItem ii = s_item(p, it);
                const int dst = (p.Lh + 1) & 1;
                mbar_wait(bars.acc_full(dst), full_cnt[dst] & 1);
                ++full_cnt[dst];
                tc_fence_after();
                const uint32_t t_lane = t_lane0 + (uint32_t)dst * 256u;
                const uint32_t bias = bias_addr + 4u * ((1 + p.Lh) * kH + ii.col0);
                const bool gpi_form = p.gpi != 0;
                const int c_first = gpi_form ? (group == 0 ? 0 : ii.n_cols) : group * 8;
                const int c_step = gpi_form ? 8 : 16;
                const int ncol = gpi_form ? gpi_ncols(p.nw, A_) : 0;
                const int wblk = gpi_form ? gpi_wblock(p.nw) : 1;
                const int n_cols_it = ii.n_cols, col0_it = ii.col0, n_pol_job = a.n_pol, task_base = a.task_base;
                float *const q_out = a.q_out, *const psi_out = a.psi_out, *const sel_out = a.sel_out;
                uint32_t kstep = 0;
                bool k_has = false, t_has = false;
                long long *kp = nullptr, *tp = nullptr;
                if (gpi_form) {
                    kstep = a.w_diag ? 0u : (uint32_t)B;
                    k_has = a.key_action != nullptr;
                    t_has = a.key_task != nullptr;
                    kp = reinterpret_cast<long long *>(a.key_action) + (a.w_diag ? (size_t)pl * B : 0) + (size_t)(wi * wblk) * kstep + b;
                    tp = reinterpret_cast<long long *>(a.key_task) + (a.w_diag ? (size_t)pl * B : 0) + (size_t)(wi * wblk) * kstep + b;
                }
                const int nw_job = p.nw;
                float *const q_row = (q_out != nullptr && row_ok) ? q_out + ((size_t)b * n_pol_job + pl) * A_ : nullptr;
                if (gpi_form && wblk > 1) {
                    if (group == 0) {
                        const uint32_t tid_ = (uint32_t)(task_base + pl);
#pragma unroll 1
                        for (int c0 = 0; c0 < n_cols_it; c0 += 32) {
                            uint32_t v[32];
                            tmem_ld32(t_lane + c0, v);
                            tmem_wait_ld();
#define SFGPI_SCAN(WB, OFF)                                                                                                            \
    do {                                                                                                                                \
        const float4 b0_ = lds128(bias + 4u * (c0 + OFF)), b1_ = lds128(bias + 4u * (c0 + OFF + 4));                                    \
        const float bv_[8] = {b0_.x, b0_.y, b0_.z, b0_.w, b1_.x, b1_.y, b1_.z, b1_.w};                                                  \
        gpi_scan_blocked<WB, OFF>(v, bv_, col0_it + c0 + OFF, ncol, A_, nw_job, bb, ba, act_i, wi, kp, tp, kstep, k_has,                \
                                  t_has, row_ok, tid_, q_row);                                                                          \
    } while (0)
                            if (wblk == 8) { SFGPI_SCAN(8, 0); SFGPI_SCAN(8, 8); SFGPI_SCAN(8, 16); SFGPI_SCAN(8, 24); }
                            else { SFGPI_SCAN(4, 0); SFGPI_SCAN(4, 8); SFGPI_SCAN(4, 16); SFGPI_SCAN(4, 24); }
#undef SFGPI_SCAN
                        }
                    }
                } else {
#pragma unroll 1
                    for (int c0 = c_first; c0 < n_cols_it; c0 += c_step) {
                        uint32_t v[8];
                        tmem_ld8(t_lane + c0, v);
                        const float4 b0 = lds128(bias + 4u * c0), b1 = lds128(bias + 4u * (c0 + 4));
                        const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
                        tmem_wait_ld();
                        if (gpi_form) {
                            // folded GPI, plain column order (n_w < 4): column = wi * A + act
#pragma unroll
                            for (int i = 0; i < 8; ++i) {
                                if (col0_it + c0 + i < ncol) {
                                    const float q = __uint_as_float(v[i]) + bv[i];
                                    if (wi == 0 && q_row != nullptr) q_row[act_i] = q;
                                    if (q > best) { best = q; best_a = act_i; }
                                    if (++act_i == A_) {
                                        if (row_ok) {
                                            if (k_has) atomicMax(kp, pack_key(best, (uint32_t)best_a));
                                            if (t_has) atomicMax(tp, pack_key(best, (uint32_t)(task_base + pl)));
                                        }
                                        kp += kstep; tp += kstep;
                                        act_i = 0; ++wi; best = -INFINITY; best_a = 0;
                                    }
                                }
                            }
                        } else {
                            const int colb = col0_it + c0;
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
                                if ((unsigned)(colb + 7 - sel_base) < (unsigned)(D + 7)) {
                                    float *so = sel_out + ((size_t)pl * B + b) * D;
#pragma unroll
                                    for (int i = 0; i < 8; ++i) {
                                        const unsigned off = (unsigned)(colb + i - sel_base);
                                        if (off < (unsigned)D) so[off] = val[i];
                                    }
                                }
                            }
                        }
                    }
                }
                release_acc(dst);
            }
        }
        if (et == 0) bulk_wait0();                           // outstanding activation stores complete before the CTA retires
    }

    tc_fence_before();
    __syncthreads();
    if (warp == kSMmaWarp) {
        __syncwarp();
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// ------------------------------------------------------------------------------------------------------------------------
// dgrad chain in the same streaming structure: dZ_{L-1} (the D-sparse d_out of the TD step, expanded on the fly, or with kDense
// the dense d_out [B][n_pol][A*D] of a general loss, read as it is) -> dZ_{L-2} ->
// ... -> dZ_0 for one 128-row tile.  dA_{l-1}[b][k] = sum_n dZ_l[b][n] W_l[n][k]: A = dZ_l k-blocks (produced by the epilogue
// threads exactly like forward activations), B = W_l^T read K-major from the TRANSPOSED operand shadows that sfgpi_pack_f32
// writes next to the forward ones (so the forward's verified operand path is reused; fp32 MN-major would need the BASE32B
// layout and eight 4 KB boxes per k-block).  Every dZ k-block is also bulk-stored (hi / lo) as the wgrad kernel's operand.
// The last product of the chain, dZ_0, has no consumer MMA: the issuer warp acknowledges its stages without issuing.
// ------------------------------------------------------------------------------------------------------------------------
struct SDg {
    sfgpi_net_desc net;
    int policy_lo, n_pol, B;
    const long long *actions;        // [B]
    const float *d_out;              // [n_pol][B][D]; dense (kDense): [B][n_pol][AD]
    const uint32_t *masks;           // [L-1][n_pol][B][8] ReLU sign bits written by the forward
    const float *acts;               // fp32 [parts][L-1][n_pol][B][256] (tanh layers: derivative from the stored outputs)
    int L, Lh, AD, ADp, n_kb0;       // ADp = A*D padded to 32, n_kb0 = ADp / 32
    int tiles_per_policy, total_units;
    int wt_part_rows, wo_part_rows;  // rows per part of the two weight maps
    int acts_part_stride;            // floats between the hi and lo activation tensors
};

template <int PARTS, bool kDense>
__global__ void __launch_bounds__(kSThreads, 1)
mlp_dgrad_stream_kernel(const __grid_constant__ SDg p, const __grid_constant__ CUtensorMap tmap_wt, const __grid_constant__ CUtensorMap tmap_wo,
                        const __grid_constant__ CUtensorMap tmap_dz, const __grid_constant__ CUtensorMap tmap_dzo) {
    constexpr int NS = PARTS == 2 ? 2 : 4;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    pdl_launch_dependents();
    const uint32_t sbase = smem_u32(smem_raw);
    const uint32_t A_addr = sbase, B_addr = sbase + NS * PARTS * kAPart;
    SBars bars;
    bars.b0 = B_addr + NS * PARTS * kBPart;
    if (threadIdx.x == 0) {
        s_bars_init(bars);
        tma_prefetch_desc(&tmap_wt);
        tma_prefetch_desc(&tmap_wo);
    }
    if (warp == kSMmaWarp) tmem_alloc(bars.holder(), 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(bars.holder()));
    pdl_wait();
    const sfgpi_net_desc &net = p.net;
    const int n_items = p.L - 1;                            // item i uses W_{L-1-i} and yields dZ_{L-2-i}

    if (warp < 4) {
        const uint32_t leader = elect_one();
        uint32_t n = 0;
        const int part = warp % PARTS, nb = warp / PARTS;
        const bool has_box = warp < PARTS * 2;
        for (int g = blockIdx.x; g < p.total_units; g += gridDim.x) {
            const int pl = g / p.tiles_per_policy;
            for (int it = 0; it < n_items; ++it) {
                const void *tm = it == 0 ? (const void *)&tmap_wo : (const void *)&tmap_wt;
                const int row = it == 0 ? part * p.wo_part_rows + (p.policy_lo + pl) * kH + nb * 128
                                        : part * p.wt_part_rows + ((p.policy_lo + pl) * p.Lh + (p.L - 2 - it)) * kH + nb * 128;
                const int n_kb = it == 0 ? p.n_kb0 : kH / kK32;
                for (int kb = 0; kb < n_kb; ++kb, ++n) {
                    const int s = n % NS;
                    mbar_wait_warp(bars.b_empty(s), ((n / NS) & 1) ^ 1);
                    if (has_box) {
                        mbar_arrive_expect_tx_e(bars.b_full(s), kBBox, leader);
                        tma_load_2d_e(B_addr + (s * PARTS + part) * kBPart + nb * kBBox, tm, bars.b_full(s), kb * kK32, row, leader);
                    } else if (leader) {
                        mbar_arrive(bars.b_full(s));
                    }
                }
            }
        }
    } else if (warp == kSMmaWarp) {
        const uint32_t leader = elect_one();
        uint32_t na = 0, nb_ = 0, acc_use[2] = {0, 0};
        const uint32_t idesc = idesc_tf32(kTM, 256u, 0u, 0u);
        for (int g = blockIdx.x; g < p.total_units; g += gridDim.x) {
            for (int it = 0; it < n_items; ++it) {
                const int dst = it & 1;
                mbar_wait_warp(bars.acc_empty(dst), (acc_use[dst] & 1) ^ 1);
                ++acc_use[dst];
                tc_fence_after();
                const uint32_t d = tmem_base + (uint32_t)dst * 256u;
                const int n_kb = it == 0 ? p.n_kb0 : kH / kK32;
                for (int kb = 0; kb < n_kb; ++kb, ++na, ++nb_) {
                    const int sa = na % NS, sb = nb_ % NS;
                    mbar_wait_warp(bars.a_full(sa), (na / NS) & 1);
                    mbar_wait_warp(bars.b_full(sb), (nb_ / NS) & 1);
                    tc_fence_after();
                    s_issue_kblock<PARTS>(d, A_addr + sa * PARTS * kAPart, B_addr + sb * PARTS * kBPart, idesc, 4, kb == 0, leader);
                    umma_commit_e(bars.a_empty(sa), leader);
                    umma_commit_e(bars.b_empty(sb), leader);
                }
                umma_commit_e(bars.acc_full(dst), leader);
            }
            // dZ_0's k-blocks pass through the A ring only to be bulk-stored: acknowledge them
            for (int kb = 0; kb < kH / kK32; ++kb, ++na) {
                const int sa = na % NS;
                mbar_wait_warp(bars.a_full(sa), (na / NS) & 1);
                if (leader) mbar_arrive(bars.a_empty(sa));
            }
        }
    } else {
        const int group = (warp - kSEpiWarp0) >> 2;
        const int quad = warp & 3;
        const int r = quad * 32 + lane;
        const int et = threadIdx.x - kSEpiWarp0 * 32;
        const uint32_t t_lane0 = tmem_base + ((uint32_t)(quad * 32) << 16);
        uint32_t n = 0, full_cnt[2] = {0, 0};
        bool store_in_flight = false;
        auto bar_epi = [&]() { asm volatile("bar.sync 1, 256;" ::: "memory"); };
        auto publish = [&](int s, const CUtensorMap *tm, int c0, int row0, int slab0, int slab_part_stride) {
            fence_proxy_async();
            if (et == 0 && store_in_flight) bulk_wait_read0();
            bar_epi();
            if (et == 0) {
                mbar_arrive(bars.a_full(s));
#pragma unroll
                for (int part = 0; part < PARTS; ++part)
                    tma_store_3d(tm, A_addr + (s * PARTS + part) * kAPart, c0, row0, slab0 + part * slab_part_stride);
                bulk_commit();
            }
            store_in_flight = true;
        };
        const int B = p.B, D = net.n_features;
        for (int g = blockIdx.x; g < p.total_units; g += gridDim.x) {
            const int pl = g / p.tiles_per_policy, tile = g - pl * p.tiles_per_policy;
            const int b = tile * kTM + r;
            const bool row_ok = b < B;
            const int sel = (!kDense && row_ok) ? (int)p.actions[b] * D : 0;
            const float *drow = kDense ? p.d_out + ((size_t)(row_ok ? b : 0) * p.n_pol + pl) * p.AD
                                       : p.d_out + ((size_t)pl * B + (row_ok ? b : 0)) * D;
            // ---- item 0's A operand: the expanded dense dZ_{L-1} row, zero except d_out[0..D) at [sel, sel + D) (kDense: the
            //      row of the dense d_out, zero past AD) ----
#pragma unroll 1
            for (int kb = 0; kb < p.n_kb0; ++kb, ++n) {
                const int s = n % NS;
                mbar_wait(bars.a_empty(s), ((n / NS) & 1) ^ 1);
                float h[16];
                const int col0 = kb * kK32 + group * 16;
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    if constexpr (kDense) {
                        h[i] = (row_ok && col0 + i < p.AD) ? drow[col0 + i] : 0.0f;
                    } else {
                        const unsigned off = (unsigned)(col0 + i - sel);
                        h[i] = (row_ok && off < (unsigned)D) ? drow[off] : 0.0f;
                    }
                }
                s_write_a16<PARTS>(h, A_addr + s * PARTS * kAPart, r, group * 16);
                publish(s, &tmap_dzo, kb * kK32, tile * kTM, pl, p.n_pol);
            }
            for (int it = 0; it < n_items; ++it) {
                const int lo = p.L - 2 - it, src_acc = it & 1;            // produces dZ_lo
                mbar_wait(bars.acc_full(src_acc), full_cnt[src_acc] & 1);
                ++full_cnt[src_acc];
                tc_fence_after();
                const int act = net.acts[lo];
                const uint32_t t_src = t_lane0 + (uint32_t)src_acc * 256u;
                const size_t rowi = ((size_t)lo * p.n_pol + pl) * B + (row_ok ? b : 0);
                const uint16_t *mask_row = (act == SFGPI_ACT_RELU) ? reinterpret_cast<const uint16_t *>(p.masks + rowi * 8) : nullptr;
                const float *act_row = p.acts + rowi * kH;
#pragma unroll 1
                for (int kb = 0; kb < kH / kK32; ++kb, ++n) {
                    const int s = n % NS;
                    mbar_wait(bars.a_empty(s), ((n / NS) & 1) ^ 1);
                    uint32_t v[16];
                    const int c0 = kb * kK32 + group * 16;
                    tmem_ld16(t_src + c0, v);
                    uint32_t bits = 0xFFFFu;
                    if (mask_row != nullptr) bits = row_ok ? (uint32_t)__ldg(mask_row + kb * 2 + group) : 0u;
                    float h[16];
                    tmem_wait_ld();
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        float gv = row_ok ? __uint_as_float(v[i]) : 0.0f;
                        if (act == SFGPI_ACT_RELU) gv = ((bits >> i) & 1u) ? gv : 0.0f;                       // threshold_backward
                        else if (act == SFGPI_ACT_TANH && row_ok) {
                            float av = act_row[c0 + i];
                            if (PARTS == 2) av += act_row[p.acts_part_stride + c0 + i];
                            gv *= (1.0f - av * av);                                                           // tanh_backward
                        }
                        h[i] = gv;
                    }
                    s_write_a16<PARTS>(h, A_addr + s * PARTS * kAPart, r, group * 16);
                    publish(s, &tmap_dz, kb * kK32, tile * kTM, lo * p.n_pol + pl, (p.L - 1) * p.n_pol);
                }
                tc_fence_before();
                bar_epi();
                if (et == 0) mbar_arrive(bars.acc_empty(src_acc));
            }
        }
        if (et == 0) bulk_wait0();
    }

    tc_fence_before();
    __syncthreads();
    if (warp == kSMmaWarp) {
        __syncwarp();
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// xo[part][b][c] = hi / lo of (x[b][c] for c < S, 1 for c == S, 0 otherwise): fp32 [parts][B][32], the wgrad kernel's auxiliary operand
__global__ void build_xo_f32_kernel(const float *__restrict__ x, int B, int S, int parts, float *__restrict__ xo) {
    pdl_launch_dependents();
    pdl_wait();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * 32) return;
    const int b = i >> 5, c = i & 31;
    const float v = c < S ? x[(size_t)b * S + c] : (c == S ? 1.0f : 0.0f);
    const float hi = tf32_rna(v);
    xo[i] = hi;
    if (parts == 2) xo[(size_t)B * 32 + i] = tf32_rna(v - hi);
}

// ---- fp32 library rows -> hi / lo operand shadows ---------------------------------------------------------------------------
// shadow  [parts][n_total][rows_per_policy][256]: W_0 (columns >= S zero), hidden W_1..W_Lh, W_out padded (the forward's B operands)
// shadow_t[parts][n_total][Lh][256][256]        : W_l^T, l = 1..Lh (dgrad's B operands: rows = the forward's input index)
// wout_t  [parts][n_total][256][ADp]            : W_out^T, columns >= A*D zero
// parts = 1: hi only (TF32: rounded to nearest, the tensor core itself would truncate); parts = 2: hi, lo = v - hi (TF32X3).
// One block = one 32 x 32 tile of one matrix; the transposes go through shared memory so that both sides are coalesced.
__global__ void __launch_bounds__(256) pack_f32_kernel(sfgpi_net_desc net, const float *__restrict__ params, int policy_lo, int n_total,
                                                       int parts, float *__restrict__ shadow, float *__restrict__ shadow_t,
                                                       float *__restrict__ wout_t, int rpp, int Lh, int ADp, int tiles_out) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ float t[32][33];
    const int AD = net.n_actions * net.n_features, L = net.n_layers, S = net.dims[0];
    const int pl = policy_lo + blockIdx.y;
    const float *P = params + (size_t)pl * net.row_stride;
    // tile index -> (matrix, tile row, tile col): W_0 has 8 row tiles x 1 col tile; hidden 8 x 8 each; output tiles_out x 8
    int tix = blockIdx.x, mat, tr, tc_;
    if (tix < 8) { mat = 0; tr = tix; tc_ = 0; }
    else if (tix < 8 + Lh * 64) { tix -= 8; mat = 1 + tix / 64; tr = (tix % 64) / 8; tc_ = tix % 8; }
    else { tix -= 8 + Lh * 64; mat = L - 1; tr = tix / 8; tc_ = tix % 8; }
    const int n_rows = mat == L - 1 ? AD : kH, n_in = mat == 0 ? S : kH;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;           // 32 x 8 threads
    const size_t part_stride = (size_t)n_total * rpp * kH;
    const int row_base = mat == 0 ? 0 : (mat == L - 1 ? (1 + Lh) * kH : mat * kH);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int rr = tr * 32 + ty + 8 * q, cc = tc_ * 32 + tx;
        float v = 0.0f;
        if (rr < n_rows && cc < n_in) v = P[net.w_off[mat] + (size_t)rr * n_in + cc];
        t[ty + 8 * q][tx] = v;
        const float hi = tf32_rna(v);
        const int rows_here = mat == L - 1 ? ((AD + 15) & ~15) : kH;
        if (rr < rows_here) {
            float *dst = shadow + ((size_t)pl * rpp + row_base + rr) * kH + cc;
            dst[0] = hi;
            if (parts == 2) dst[part_stride] = tf32_rna(v - hi);
        }
    }
    if (mat == 0 || (shadow_t == nullptr && wout_t == nullptr)) return;
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        // transposed element: row = input index (tc_ * 32 + ty + 8q), column = output index (tr * 32 + tx)
        const int kk = tc_ * 32 + ty + 8 * q, nn = tr * 32 + tx;
        const float v = t[tx][ty + 8 * q];
        const float hi = tf32_rna(v);
        if (mat < L - 1) {
            if (shadow_t != nullptr) {
                float *dst = shadow_t + (((size_t)pl * Lh + (mat - 1)) * kH + kk) * kH + nn;
                dst[0] = hi;
                if (parts == 2) dst[(size_t)n_total * Lh * kH * kH] = tf32_rna(v - hi);
            }
        } else if (wout_t != nullptr && nn < ADp) {
            float *dst = wout_t + ((size_t)pl * kH + kk) * ADp + nn;
            dst[0] = hi;
            if (parts == 2) dst[(size_t)n_total * kH * ADp] = tf32_rna(v - hi);
        }
    }
}

// GPI fold in fp32 hi / lo: Wq[part][pl][row][k], bq[pl][row]  (row order: gpi_scan.cuh)
__global__ void __launch_bounds__(256) fold_gpi_f32_kernel(sfgpi_net_desc net, const float *__restrict__ params, int policy_lo,
                                                           const float *__restrict__ w, int nw, int w_diag, int nqpad, int n_pol, int parts,
                                                           float *__restrict__ wq, float *__restrict__ bq) {
    pdl_launch_dependents();
    pdl_wait();
    const int pl = blockIdx.y, row = blockIdx.x, k = threadIdx.x;
    const int A_ = net.n_actions, D = net.n_features, L = net.n_layers;
    const float *P = params + (size_t)(policy_lo + pl) * net.row_stride;
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
    const float hi = tf32_rna(acc);
    const size_t o = ((size_t)pl * nqpad + row) * kH + k;
    wq[o] = hi;
    if (parts == 2) wq[o + (size_t)n_pol * nqpad * kH] = tf32_rna(acc - hi);
    if (k == 0) bq[(size_t)pl * nqpad + row] = bacc;
}

static bool stream_shape_ok(const sfgpi_net_desc &net, const char **why) {
    if (net.n_layers < 3) { *why = "needs >= 3 Linear layers"; return false; }
    for (int l = 1; l < net.n_layers; ++l)
        if (net.dims[l] != kH) { *why = "every hidden width must be 256"; return false; }
    if (net.dims[0] > 31) { *why = "state dimension must be <= 31"; return false; }
    if (net.acts[net.n_layers - 1] != SFGPI_ACT_NONE) { *why = "output layer must be linear"; return false; }
    return true;
}

}  // namespace tc
}  // namespace sfgpi

using namespace sfgpi;
using namespace sfgpi::tc;

extern "C" int sfgpi_f32_out_pad(const sfgpi_net_desc *net) { return (net->n_actions * net->n_features + 31) & ~31; }

static int parts_of(int32_t precision) { return precision == kPrecTf32x3 ? 2 : (precision == kPrecTf32 ? 1 : 0); }

extern "C" int sfgpi_pack_f32(const sfgpi_net_desc *net, const float *params, int32_t policy_lo, int32_t n_pol, int32_t n_policies_total,
                              int32_t precision, float *shadow, float *shadow_t, float *wout_t, void *stream) {
    const char *why = "";
    if (!stream_shape_ok(*net, &why)) { set_error("sfgpi_pack_f32: tensor-core path %s", why); return SFGPI_E_INVALID; }
    const int parts = parts_of(precision);
    if (!parts || !params || !shadow || policy_lo < 0 || n_pol < 0 || policy_lo + n_pol > n_policies_total) {
        set_error("sfgpi_pack_f32: invalid arguments");
        return SFGPI_E_INVALID;
    }
    if (n_pol == 0) return SFGPI_OK;
    const int Lh = net->n_layers - 2, AD = net->n_actions * net->n_features;
    const int tiles_out = (((AD + 15) & ~15) + 31) / 32;
    dim3 grid(8 + Lh * 64 + tiles_out * 8, n_pol);
    launch_pdl(pack_f32_kernel, grid, dim3(256), 0, (cudaStream_t)stream, *net, params, policy_lo, n_policies_total, parts, shadow, shadow_t,
               wout_t, sfgpi_bf16_rows_per_policy(net), Lh, sfgpi_f32_out_pad(net), tiles_out);
    return check_launch("sfgpi_pack_f32");
}

extern "C" int sfgpi_fold_gpi_f32(const sfgpi_net_desc *net, const float *params, int32_t policy_lo, int32_t n_pol, const float *w,
                                  int32_t n_w, int32_t w_diag, int32_t precision, float *wq_out, float *bq_out, void *stream) {
    const char *why = "";
    if (!stream_shape_ok(*net, &why)) { set_error("sfgpi_fold_gpi_f32: tensor-core path %s", why); return SFGPI_E_INVALID; }
    const int parts = parts_of(precision);
    if (!parts) { set_error("sfgpi_fold_gpi_f32: precision must be SFGPI_PREC_TF32 or SFGPI_PREC_TF32X3"); return SFGPI_E_INVALID; }
    if (n_pol <= 0) return SFGPI_OK;
    const int nw = w_diag ? 1 : n_w;
    if (nw < 1) { set_error("sfgpi_fold_gpi_f32: n_w must be >= 1"); return SFGPI_E_INVALID; }
    const int nqpad = sfgpi_gpi_fold_rows(net, nw);
    launch_pdl(fold_gpi_f32_kernel, dim3(nqpad, n_pol), dim3(256), 0, (cudaStream_t)stream, *net, params, policy_lo, w, nw, w_diag, nqpad,
               (int)n_pol, parts, wq_out, bq_out);
    return check_launch("sfgpi_fold_gpi_f32");
}

// Same job semantics as sfgpi_mlp_forward_tc_jobs; params_bf16 -> the fp32 shadow of sfgpi_pack_f32, wq -> sfgpi_fold_gpi_f32's
// output, args.acts_bf16_out -> fp32 [parts][L-1][n_pol][B][256].
extern "C" int sfgpi_mlp_forward_stream(const sfgpi_forward_tc_job *jobs, int32_t n_jobs, int32_t precision, void *stream) {
    const int parts = parts_of(precision);
    if (!parts) { set_error("sfgpi_mlp_forward_stream: precision must be SFGPI_PREC_TF32 or SFGPI_PREC_TF32X3"); return SFGPI_E_INVALID; }
    if (n_jobs < 1 || n_jobs > kSMaxJobs) { set_error("sfgpi_mlp_forward_stream: 1..%d jobs per launch", kSMaxJobs); return SFGPI_E_INVALID; }
    SMulti m;
    SMaps maps;
    m.n_jobs = 0;
    m.total_units = 0;
    for (int j = 0; j < n_jobs; ++j) {
        const sfgpi_forward_args &a = jobs[j].args;
        const sfgpi_net_desc &net = a.net;
        const char *why = "";
        if (!stream_shape_ok(net, &why)) { set_error("sfgpi_mlp_forward_stream: tensor-core path %s", why); return SFGPI_E_INVALID; }
        if (a.B < 0 || a.n_pol < 0 || net.dims[net.n_layers] != net.n_actions * net.n_features) {
            set_error("sfgpi_mlp_forward_stream: invalid sizes");
            return SFGPI_E_INVALID;
        }
        if (a.B == 0 || a.n_pol == 0) continue;
        SJob &p = m.job[m.n_jobs];
        p.a = a;
        p.gpi = a.w != nullptr ? 1 : 0;
        if (p.gpi && (a.psi_out || a.sel_out)) {
            set_error("sfgpi_mlp_forward_stream: the GPI form cannot also emit psi / gathered rows (use a separate job)");
            return SFGPI_E_INVALID;
        }
        if (p.gpi && (!jobs[j].wq || !jobs[j].bq)) { set_error("sfgpi_mlp_forward_stream: GPI form needs the folded weights"); return SFGPI_E_INVALID; }
        p.nw = p.gpi ? (a.w_diag ? 1 : a.n_w) : 0;
        p.Lh = net.n_layers - 2;
        p.rows_per_policy = sfgpi_bf16_rows_per_policy(&net);
        p.n_final = p.gpi ? sfgpi_gpi_fold_rows(&net, p.nw) : ((net.n_actions * net.n_features + 15) & ~15);
        p.n_items = 1 + p.Lh + (p.n_final + 255) / 256;
        p.ks0 = (net.dims[0] + 7) / 8;
        p.bq = jobs[j].bq;
        if ((1 + p.Lh) * kH + p.n_final > kSBiasFloats) {
            set_error("sfgpi_mlp_forward_stream: %d bias floats exceed the shared-memory budget", (1 + p.Lh) * kH + p.n_final);
            return SFGPI_E_SMEM;
        }
        p.tiles_per_policy = (a.B + kTM - 1) / kTM;
        p.unit_start = m.total_units;
        m.total_units += p.tiles_per_policy * a.n_pol;
        p.w_part_rows = jobs[j].n_policies_total * p.rows_per_policy;
        p.q_part_rows = a.n_pol * p.n_final;
        const uint32_t box[2] = {(uint32_t)kK32, 128u};
        {
            const uint64_t dims[2] = {(uint64_t)kH, (uint64_t)parts * p.w_part_rows};
            int rc = make_tmap_f32(&maps.w[m.n_jobs], jobs[j].params_bf16, 2, dims, box, false);
            if (rc) return rc;
        }
        maps.q[m.n_jobs] = maps.w[m.n_jobs];
        if (p.gpi) {
            const uint64_t dims[2] = {(uint64_t)kH, (uint64_t)parts * p.q_part_rows};
            int rc = make_tmap_f32(&maps.q[m.n_jobs], jobs[j].wq, 2, dims, box, false);
            if (rc) return rc;
        }
        maps.acts[m.n_jobs] = maps.w[m.n_jobs];
        if (a.acts_bf16_out != nullptr) {                        // fp32 [parts][L-1][n_pol][B][256], stored k-block by k-block with TMA
            const uint64_t d3[3] = {(uint64_t)kH, (uint64_t)a.B, (uint64_t)parts * (net.n_layers - 1) * a.n_pol};
            const uint32_t b3[3] = {(uint32_t)kK32, (uint32_t)kTM, 1u};
            int rc = make_tmap_f32(&maps.acts[m.n_jobs], a.acts_bf16_out, 3, d3, b3, false);
            if (rc) return rc;
        }
        ++m.n_jobs;
    }
    if (m.n_jobs == 0) return SFGPI_OK;
    for (int j = m.n_jobs; j < kSMaxJobs; ++j) { m.job[j] = m.job[0]; m.job[j].unit_start = m.total_units; maps.w[j] = maps.w[0]; maps.q[j] = maps.q[0]; maps.acts[j] = maps.acts[0]; }
    const int NS = parts == 2 ? 2 : 4;
    const int smem_bytes = NS * parts * (kAPart + kBPart) + kSBiasFloats * 4 + 256;
    static bool cfg = false;
    if (!cfg) {
        cudaFuncSetAttribute(mlp_forward_stream_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
        cudaFuncSetAttribute(mlp_forward_stream_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
        cfg = true;
    }
    const int grid = m.total_units < 148 ? m.total_units : 148;
    if (parts == 2) launch_pdl(mlp_forward_stream_kernel<2>, dim3(grid), dim3(kSThreads), smem_bytes, (cudaStream_t)stream, m, maps);
    else launch_pdl(mlp_forward_stream_kernel<1>, dim3(grid), dim3(kSThreads), smem_bytes, (cudaStream_t)stream, m, maps);
    return check_launch("sfgpi_mlp_forward_stream");
}

int sfgpi_wgrad_tf32_launch(const sfgpi_net_desc &net, int parts, int n_pol, int B, const float *dz, const float *dzo, const float *acts,
                            const float *xo, int ADp, float *grad_part, int n_split, cudaStream_t st);

extern "C" int sfgpi_mlp_backward_stream(const sfgpi_backward_stream_args *args, void *stream) {
    if (!args) { set_error("sfgpi_mlp_backward_stream: null args"); return SFGPI_E_INVALID; }
    const sfgpi_backward_stream_args &a = *args;
    const sfgpi_net_desc &net = a.net;
    const int L = net.n_layers;
    const char *why = "";
    if (!stream_shape_ok(net, &why) || net.dims[L] != net.n_actions * net.n_features) {
        set_error("sfgpi_mlp_backward_stream: tensor-core path %s", why);
        return SFGPI_E_INVALID;
    }
    const int parts = parts_of(a.precision);
    if (!parts) { set_error("sfgpi_mlp_backward_stream: precision must be SFGPI_PREC_TF32 or SFGPI_PREC_TF32X3"); return SFGPI_E_INVALID; }
    if (a.B < 0 || a.n_pol < 0 || a.n_split < 1) { set_error("sfgpi_mlp_backward_stream: invalid sizes"); return SFGPI_E_INVALID; }
    if (a.B == 0 || a.n_pol == 0) return SFGPI_OK;
    if (sfgpi_bwd_tc_splits(a.B, a.n_split) != a.n_split) {
        set_error("sfgpi_mlp_backward_stream: n_split %d leaves empty batch splits for B=%d (use sfgpi_bwd_tc_splits)", a.n_split, a.B);
        return SFGPI_E_INVALID;
    }
    bool relu = false;
    for (int l = 0; l < L - 1; ++l) relu = relu || net.acts[l] == SFGPI_ACT_RELU;
    if (!a.shadow_t || !a.wout_t || !a.x || !a.acts || !a.d_out || !a.dz || !a.dzo || !a.xo || !a.grad_part || (relu && !a.relu_masks)) {
        set_error("sfgpi_mlp_backward_stream: missing buffers");
        return SFGPI_E_INVALID;
    }
    const bool dense = a.actions == nullptr;                          // d_out [B][n_pol][A*D] instead of [n_pol][B][D]
    cudaStream_t st = (cudaStream_t)stream;
    const int S = net.dims[0], AD = net.n_actions * net.n_features, ADp = sfgpi_f32_out_pad(&net), Lh = L - 2;
    launch_pdl(build_xo_f32_kernel, dim3((a.B * 32 + 255) / 256), dim3(256), 0, st, a.x, a.B, S, parts, a.xo);
    int rc = check_launch("sfgpi_mlp_backward_stream(xo)");
    if (rc) return rc;

    SDg dp;
    dp.net = net;
    dp.policy_lo = a.policy_lo; dp.n_pol = a.n_pol; dp.B = a.B;
    dp.actions = reinterpret_cast<const long long *>(a.actions);
    dp.d_out = a.d_out;
    dp.masks = reinterpret_cast<const uint32_t *>(a.relu_masks);
    dp.acts = a.acts;
    dp.L = L; dp.Lh = Lh; dp.AD = AD; dp.ADp = ADp; dp.n_kb0 = ADp / kK32;
    dp.tiles_per_policy = (a.B + kTM - 1) / kTM;
    dp.total_units = dp.tiles_per_policy * a.n_pol;
    dp.wt_part_rows = a.n_policies_total * Lh * kH;
    dp.wo_part_rows = a.n_policies_total * kH;
    dp.acts_part_stride = (L - 1) * a.n_pol * a.B * kH;
    CUtensorMap tm_wt, tm_wo, tm_dz, tm_dzo;
    {
        const uint32_t box[2] = {(uint32_t)kK32, 128u};
        const uint64_t dwt[2] = {(uint64_t)kH, (uint64_t)parts * dp.wt_part_rows};
        const uint64_t dwo[2] = {(uint64_t)ADp, (uint64_t)parts * dp.wo_part_rows};
        if ((rc = make_tmap_f32(&tm_wt, a.shadow_t, 2, dwt, box, false))) return rc;
        if ((rc = make_tmap_f32(&tm_wo, a.wout_t, 2, dwo, box, false))) return rc;
        const uint64_t d3[3] = {(uint64_t)kH, (uint64_t)a.B, (uint64_t)parts * (L - 1) * a.n_pol};
        const uint64_t do3[3] = {(uint64_t)ADp, (uint64_t)a.B, (uint64_t)parts * a.n_pol};
        const uint32_t b3[3] = {(uint32_t)kK32, (uint32_t)kTM, 1u};
        if ((rc = make_tmap_f32(&tm_dz, a.dz, 3, d3, b3, false))) return rc;
        if ((rc = make_tmap_f32(&tm_dzo, a.dzo, 3, do3, b3, false))) return rc;
    }
    const int NS = parts == 2 ? 2 : 4;
    const int smem = NS * parts * (kAPart + kBPart) + 256;
    static bool cfg = false;
    if (!cfg) {
        cudaFuncSetAttribute(mlp_dgrad_stream_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        cudaFuncSetAttribute(mlp_dgrad_stream_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        cudaFuncSetAttribute(mlp_dgrad_stream_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        cudaFuncSetAttribute(mlp_dgrad_stream_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        cfg = true;
    }
    const int grid = dp.total_units < 148 ? dp.total_units : 148;
    auto kern = parts == 2 ? (dense ? mlp_dgrad_stream_kernel<2, true> : mlp_dgrad_stream_kernel<2, false>)
                           : (dense ? mlp_dgrad_stream_kernel<1, true> : mlp_dgrad_stream_kernel<1, false>);
    launch_pdl(kern, dim3(grid), dim3(kSThreads), smem, st, dp, tm_wt, tm_wo, tm_dz, tm_dzo);
    rc = check_launch("sfgpi_mlp_backward_stream(dgrad)");
    if (rc) return rc;
    return sfgpi_wgrad_tf32_launch(net, parts, a.n_pol, a.B, a.dz, a.dzo, a.acts, a.xo, ADp, a.grad_part, a.n_split, st);
}
