// TD target, the two MSE losses and every gradient that does not flow through the psi MLP, fused in one kernel
// (sfdqn.py:330-345; tsfdqn.py:621-645; features/deep.py:112-121).  Elementwise work per transition plus small reductions:
// HBM-bound on the [B][D] operands, deterministic reductions.
//
// TSF (variant 2): g_i = Linear(S,G) and h = Linear(G,D) are applied back to back with NO nonlinearity between them
// (tsfdqn.py:621-623), so aff = h(g(s)) + h(g(s')) = M (s + s') + c with M = Wh Wg [D][S], c = 2 (Wh bg + bh), and every g / h
// gradient is a linear image of two tiny per-policy sums over the batch,
//     T[d][s] = sum_b daff[b][d] (s + s')[b][s]        t[d] = sum_b daff[b][d]        (daff = dLoss/daff)
//     dWh = T Wg^T + 2 t bg^T     dbh = 2 t     dWg = Wh^T T     dbg = 2 Wh^T t
// The TD kernel therefore reduces only D*S + 2D numbers per policy (not G*S + G + D*G + D), and tsf_expand_kernel applies the
// linear maps once per policy after the reduction.  Same mathematics as autograd through u = g(s)+g(s'), different summation
// order (within the 1e-5 parity bound; tests/test_gpu_parity.py).
//
// Thread-block clusters: 8 CTAs (8 x 32 transitions) form a cluster and sum their partials through distributed shared memory in
// a fixed rank order before anything is written: ceil(B/256) partials per policy reach global memory.
#include <cooperative_groups.h>
#include "peer.cuh"

namespace cg = cooperative_groups;

namespace sfgpi {

constexpr int kTdRows = 32;       // transitions per CTA
constexpr int kTdThreads = 128;
constexpr int kTdCluster = 8;     // CTAs per cluster (portable maximum)


__global__ void __cluster_dims__(kTdCluster, 1, 1) __launch_bounds__(kTdThreads)
td_kernel(const __grid_constant__ sfgpi_td_args a, const __grid_constant__ sfgpi_peer_keys_args pk) {
    extern __shared__ __align__(16) float sm[];
    __shared__ int astar_s[kTdRows];                        // a*_b of this CTA's rows, decoded from the GPI keys
    pdl_launch_dependents(SFGPI_TR_TD);
    pdl_wait(SFGPI_TR_TD);
    cg::cluster_group cluster = cg::this_cluster();
    const int tid = threadIdx.x;
    const int B = a.B, S = a.S, D = a.D, G = a.G;
    const int pl = blockIdx.y, blk = blockIdx.x;
    const int clu = blk / kTdCluster, nclu = gridDim.x / kTdCluster;
    const int row0 = blk * kTdRows;
    const int rows = max(0, min(kTdRows, B - row0));         // the grid is padded to whole clusters: trailing CTAs add zeros
    const bool tsf = a.variant == 2, reward = a.variant >= 1;
    const int K = tsf ? a.n_flows : 0, nfl = tsf_flow_len(S, K);      // normalising-flow g: K planar flows ahead of the Linear
    const int n_red = tsf ? tsf_red_len(D, S, K) : (reward ? D : 0);      // gradient partials of this variant
    const int n_acc = n_red + 2;                             // [partials | sum diff^2 | sum e^2]

    // carve-up
    float *w_s = sm;                              // [D]
    float *phi_s = w_s + D;                       // [32][D]  phi (raw)
    float *tphi_s = phi_s + kTdRows * D;          // [32][D]  phi~ (transformed)
    float *diff_s = tphi_s + kTdRows * D;         // [32][D]  then reused as daff
    float *e_s = diff_s + kTdRows * D;            // [32]
    float *red_s = e_s + kTdRows;                 // [8] block-reduction scratch
    float *gacc_s = red_s + 8;                    // [n_acc] this CTA's partials, summed across the cluster
    float *cur_s = gacc_s + n_acc;                // [32][D]  psi(s)[a]
    float *gam_s = cur_s + kTdRows * D;           // [32] gammas | [32] rewards
    float *rs_s = gam_s + kTdRows;
    float *M_s = rs_s + kTdRows;                  // [D][S]   (tsf only from here)
    float *c_s = M_s + D * S;                     // [D]
    float *ss_s = c_s + D;                        // [32][S]  s, then s + s'
    float *sn_s = ss_s + kTdRows * S;             // [32][S]  s'
    float *Wg_s = sn_s + kTdRows * S;             // [G][S] | bg [G] | Wh [D][G] | bh [D]   staging for M, c (only without a.tsf_mc)
    float *bg_s = Wg_s + G * S, *Wh_s = bg_s + G, *bh_s = Wh_s + D * G;
    const bool own_mc = tsf && a.tsf_mc == nullptr;
    float *fl_s = own_mc ? bh_s + D : Wg_s;       // (flows only) [K][weight S | bias | scale S]
    float *zh_s = fl_s + nfl;                     // [64][K + 1][S]  z_0 .. z_K of (branch, row): branch 0 = s, 1 = s'
    float *th_s = zh_s + 2 * kTdRows * (K + 1) * S;          // [64][K]  tanh of every flow's activation
    float *fw_s = th_s + 2 * kTdRows * K;         // [2][nfl] the two warps' sums of the flows' gradients

    for (int e = tid; e < n_acc; e += kTdThreads) gacc_s[e] = 0.0f;

    // Everything this CTA reads that does not depend on a*, in ONE memory round trip: the GPI key of each row into a register,
    // all the rest straight into shared memory with cp.async (fire and forget), one wait at the end.  As plain load -> store
    // loops these were 6-7 dependent round trips (each loop's first store waits for its loads) of a kernel that is nothing but
    // latency: 512 CTAs in one wave, 4 MB of data.
    long long key_r = 0;
    const bool sharded = a.next_psi != nullptr && pk.ctx.world > 0;
    if (a.next_psi != nullptr && !sharded && tid < rows) key_r = a.next_keys[(size_t)pl * a.next_key_stride + row0 + tid];

    const float *cur = a.cur_sel + (size_t)pl * B * D;
    const float *nxt = a.next_sel + (size_t)pl * B * D;
    float *dout = a.d_out + (size_t)pl * B * D;
    auto stage = [&](float *dst, const float *src, int n_valid, int n_total) {       // dst[e] = e < n_valid ? src[e] : 0
        const uint32_t d0 = (uint32_t)__cvta_generic_to_shared(dst);
        for (int e = tid; e < n_total; e += kTdThreads) {
            const uint32_t nb = e < n_valid ? 4u : 0u;
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(d0 + 4u * e), "l"(src + (e < n_valid ? e : 0)), "r"(nb) : "memory");
        }
    };
    if (reward) stage(w_s, a.w + (size_t)pl * a.w_stride, D, D);
    stage(phi_s, a.phis + (size_t)row0 * D, rows * D, kTdRows * D);
    stage(cur_s, cur + (size_t)row0 * D, rows * D, kTdRows * D);
    stage(gam_s, a.gammas + row0, rows, kTdRows);
    if (reward) stage(rs_s, a.rs + row0, rows, kTdRows);
    if (tsf) {
        stage(ss_s, a.states + (size_t)row0 * S, rows * S, kTdRows * S);
        stage(sn_s, a.next_states + (size_t)row0 * S, rows * S, kTdRows * S);
        if (own_mc) {
            stage(Wg_s, a.g + (size_t)pl * a.g_stride, G * S + G, G * S + G);            // Wg | bg (contiguous in the row)
            stage(Wh_s, a.h, D * G + D, D * G + D);                                      // Wh | bh
        } else {
            stage(M_s, a.tsf_mc + (size_t)pl * (D * S + D), D * S + D, D * S + D);       // M | c (contiguous, like M_s | c_s)
        }
        if (K > 0) stage(fl_s, a.g + (size_t)pl * a.g_stride + G * S + G, nfl, nfl);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");

    if (a.next_psi != nullptr) {
        // next actions: one key per row.  Sharded over peer memory, the key is the MAX over ranks of the rows this rank owns,
        // pulled here from the peers' arenas (csrc/peer.cu) once every rank has signalled that its forward pass is complete.
        if (sharded) {
            peer_signal_and_wait(pk.ctx, SFGPI_PEER_CH_KEYS, (unsigned long long)pk.epoch, blockIdx.x == 0 && blockIdx.y == 0);
            if (tid < rows) {
                const size_t off = (size_t)(pk.row_lo + pl) * B + row0 + tid;
                long long kv[SFGPI_MAX_PEERS];                 // all peers' loads in flight at once (one NVLink round trip, not world)
#pragma unroll
                for (int r = 0; r < SFGPI_MAX_PEERS; ++r)
                    if (r < pk.ctx.world) kv[r] = ld_peer_i64(reinterpret_cast<const long long *>(pk.keys_all[r]) + off);
                long long k = kv[0];
#pragma unroll
                for (int r = 1; r < SFGPI_MAX_PEERS; ++r)
                    if (r < pk.ctx.world) k = max(k, kv[r]);
                astar_s[tid] = (int)key_index(k);
                if (pk.keys_out != nullptr) pk.keys_out[(size_t)pl * B + row0 + tid] = k;
            }
        } else if (tid < rows) {
            astar_s[tid] = (int)key_index(key_r);
        }
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();

    if (K > 0) {
        // normalising-flow g (tsfdqn_nf.py:347-349): both state rows of every transition run through the K planar flows,
        // z <- z + scale_k * tanh(z . weight_k + bias_k); thread t < 64 owns (branch t / 32, row t % 32) and keeps z_0 .. z_K and
        // the tanh values for the backward sweep below.  h(g(.)) stays affine in the FLOWED states: aff = M (z + z') + c.
        if (tid < 2 * kTdRows) {
            const float *src = (tid < kTdRows ? ss_s : sn_s) + (tid & (kTdRows - 1)) * S;
            float *z = zh_s + (size_t)tid * (K + 1) * S;
            for (int s_ = 0; s_ < S; ++s_) z[s_] = src[s_];
            for (int k = 0; k < K; ++k) {
                const float *fw = fl_s + k * (2 * S + 1), *fsc = fw + S + 1;
                float act = fw[S];
                for (int s_ = 0; s_ < S; ++s_) act = fmaf(z[s_], fw[s_], act);
                const float th = tanhf(act);
                th_s[tid * K + k] = th;
                for (int s_ = 0; s_ < S; ++s_) z[S + s_] = fmaf(fsc[s_], th, z[s_]);
                z += S;
            }
        }
        __syncthreads();
        for (int e = tid; e < 2 * kTdRows * S; e += kTdThreads) {                        // ss_s <- z_K(s), sn_s <- z_K(s')
            const int t = e / S, s_ = e - t * S;
            (t < kTdRows ? ss_s : sn_s)[(t & (kTdRows - 1)) * S + s_] = zh_s[((size_t)t * (K + 1) + K) * S + s_];
        }
        __syncthreads();
    }
    if (tsf) {
        for (int e = tid; e < kTdRows * S; e += kTdThreads) ss_s[e] += sn_s[e];           // s + s'
        if (own_mc) {
            // M = Wh Wg, c = 2 (Wh bg + bh): D*(S+1) dot products of length G
            for (int o = tid; o < D * (S + 1); o += kTdThreads) {
                const int d = o / (S + 1), s = o - d * (S + 1);
                const float *wh = Wh_s + d * G;
                float acc = 0.0f;
                if (s < S) {
                    for (int g = 0; g < G; ++g) acc = fmaf(wh[g], Wg_s[g * S + s], acc);
                    M_s[d * S + s] = acc;
                } else {
                    for (int g = 0; g < G; ++g) acc = fmaf(wh[g], bg_s[g], acc);
                    c_s[d] = 2.0f * (acc + bh_s[d]);
                }
            }
        }
        __syncthreads();
    }

    // phi~, target, diff, d_out, l1 partial                                    (tsfdqn.py:623-633 / sfdqn.py:330-335)
    const float c1 = 2.0f / ((float)B * (float)a.A * (float)D);
    float l1_acc = 0.0f;
    for (int e = tid; e < kTdRows * D; e += kTdThreads) {
        const int r = e / D, d = e - r * D;
        float tphi = phi_s[e], df = 0.0f;
        if (tsf) {
            float aff = c_s[d];
            for (int s = 0; s < S; ++s) aff = fmaf(M_s[d * S + s], ss_s[r * S + s], aff);
            tphi *= aff;
        }
        if (r < rows) {
            const size_t gi = (size_t)row0 * D + e;
            float nv;
            if (a.next_psi != nullptr) {                 // gather psi^-(s')[a*] from the full target output by the GPI key
                const int astar = astar_s[r];
                nv = a.next_psi[((size_t)(row0 + r) * a.n_pol + pl) * ((size_t)a.A * D) + (size_t)astar * D + d];
            } else {
                nv = nxt[gi];
            }
            const float target = fmaf(gam_s[r], nv, tphi);
            df = cur_s[e] - target;
            dout[gi] = c1 * df;
            l1_acc = fmaf(df, df, l1_acc);
        }
        tphi_s[e] = tphi;
        diff_s[e] = df;
    }
    __syncthreads();

    // reward head: e = w . phi~ - r, l2 partial                                (sfdqn.py:339-341 / tsfdqn.py:638-642)
    float l2_acc = 0.0f;
    if (reward) {
        if (tid < kTdRows) {
            float ev = 0.0f;
            if (tid < rows) {
                for (int d = 0; d < D; ++d) ev = fmaf(w_s[d], tphi_s[tid * D + d], ev);
                ev -= rs_s[tid];
                l2_acc = ev * ev;
            }
            e_s[tid] = ev;
        }
        __syncthreads();
    }

    // loss partials (deterministic tree inside the CTA)
    {
        float s1 = warp_sum(l1_acc), s2 = warp_sum(l2_acc);
        if ((tid & 31) == 0) { red_s[tid >> 5] = s1; red_s[4 + (tid >> 5)] = s2; }
        __syncthreads();
        if (tid == 0) {
            gacc_s[n_red] = (red_s[0] + red_s[1]) + (red_s[2] + red_s[3]);
            gacc_s[n_red + 1] = (red_s[4] + red_s[5]) + (red_s[6] + red_s[7]);
        }
    }
    const float c2 = 2.0f * a.beta / (float)B;           // variant 1: beta == 1

    if (reward) {
        // dL/dw[d] = c2 * sum_b e_b * phi~[b][d]
        for (int d = tid; d < D; d += kTdThreads) {
            float acc = 0.0f;
            for (int r = 0; r < kTdRows; ++r) acc = fmaf(e_s[r], tphi_s[r * D + d], acc);
            gacc_s[d] = c2 * acc;
        }
    }
    if (tsf) {
        // daff = (dL/dphi~) * phi,  dL/dphi~ = -c1*diff + c2*e*w                   (targets carry grad, tsfdqn.py:629)
        __syncthreads();
        for (int e = tid; e < kTdRows * D; e += kTdThreads) {
            const int r = e / D, d = e - r * D;
            diff_s[e] = (c2 * e_s[r] * w_s[d] - c1 * diff_s[e]) * phi_s[e];
        }
        __syncthreads();
        const float *daff_s = diff_s;
        float *T = gacc_s + D, *tv = T + D * S;
        for (int o = tid; o < D * (S + 1); o += kTdThreads) {
            const int d = o / (S + 1), s = o - d * (S + 1);
            float acc = 0.0f;
            if (s < S) {
                for (int r = 0; r < kTdRows; ++r) acc = fmaf(daff_s[r * D + d], ss_s[r * S + s], acc);
                T[d * S + s] = acc;
            } else {
                for (int r = 0; r < kTdRows; ++r) acc += daff_s[r * D + d];
                tv[d] = acc;
            }
        }
        if (K > 0) {
            // backward sweep through the flows: dL/dz_K = M^T daff for both branches, then per flow (t = tanh, a = its argument)
            //   dscale = dz * t,  da = (dz . scale) (1 - t^2),  dweight = da * z_in,  dbias = da,  dz_in = dz + da * weight.
            // Every contribution is summed over the 32 rows of a branch by a fixed butterfly, the two branches are added in order.
            float *fgrad = tv + D;                       // [nfl] behind [dw | T | t]
            if (tid < 2 * kTdRows) {
                const int r = tid & (kTdRows - 1), wp = tid >> 5, ln = tid & 31;
                float *zrow = zh_s + (size_t)tid * (K + 1) * S;
                float *dz = zrow + K * S;                 // z_K is not needed any more: its slot holds dz
                for (int s_ = 0; s_ < S; ++s_) {
                    float acc = 0.0f;
                    for (int d = 0; d < D; ++d) acc = fmaf(M_s[d * S + s_], daff_s[r * D + d], acc);
                    dz[s_] = acc;
                }
                for (int k = K - 1; k >= 0; --k) {
                    const float *fw = fl_s + k * (2 * S + 1), *fsc = fw + S + 1;
                    const float *zin = zrow + k * S;
                    float *out = fw_s + wp * nfl + k * (2 * S + 1);
                    const float th = th_s[tid * K + k];
                    float dt = 0.0f;
                    for (int s_ = 0; s_ < S; ++s_) {
                        const float v = warp_sum(dz[s_] * th);
                        if (ln == 0) out[S + 1 + s_] = v;
                        dt = fmaf(dz[s_], fsc[s_], dt);
                    }
                    const float da = dt * (1.0f - th * th);
                    for (int s_ = 0; s_ < S; ++s_) {
                        const float v = warp_sum(da * zin[s_]);
                        if (ln == 0) out[s_] = v;
                        dz[s_] = fmaf(da, fw[s_], dz[s_]);
                    }
                    const float vb = warp_sum(da);
                    if (ln == 0) out[S] = vb;
                }
            }
            __syncthreads();
            for (int e = tid; e < nfl; e += kTdThreads) fgrad[e] = fw_s[e] + fw_s[nfl + e];
        }
    }

    // ---- cluster reduction through distributed shared memory: rank r sums slice r of the 8 CTAs' partials, rank order ----
    float *out_part = tsf ? a.tsf_part + ((size_t)pl * nclu + clu) * n_red
                          : a.aux_grad_part + ((size_t)pl * nclu + clu) * a.aux_len;
    cluster.sync();
    {
        const unsigned rk = cluster.block_rank();
        const int per = (n_acc + kTdCluster - 1) / kTdCluster;
        const int e_lo = rk * per, e_hi = min(n_acc, e_lo + per);
        const float *remote[kTdCluster];
#pragma unroll
        for (int q = 0; q < kTdCluster; ++q) remote[q] = cluster.map_shared_rank(gacc_s, q);
        for (int e = e_lo + tid; e < e_hi; e += kTdThreads) {
            float v[kTdCluster];
#pragma unroll
            for (int q = 0; q < kTdCluster; ++q) v[q] = remote[q][e];
            const float sum = ((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]));
            if (e < n_red) out_part[e] = sum;
            else a.loss_part[((size_t)pl * nclu + clu) * 2 + (e - n_red)] = sum;
        }
    }
    cluster.sync();                                          // nobody leaves while its shared memory is still being read
    trace_exit(SFGPI_TR_TD);
}

__global__ void __launch_bounds__(256) tsf_expand_kernel(const __grid_constant__ sfgpi_td_args a, int nclu) {
    extern __shared__ __align__(16) float sm[];
    pdl_launch_dependents();
    pdl_wait();
    tsf_expand_cta(a, blockIdx.x, nclu, sm, threadIdx.x, 256);
}

}  // namespace sfgpi

using namespace sfgpi;

extern "C" int sfgpi_td_partials(int32_t B) { return B <= 0 ? 1 : (B + kTdRows * kTdCluster - 1) / (kTdRows * kTdCluster); }

extern "C" int sfgpi_td_step(const sfgpi_td_args *args, void *stream) {
    const sfgpi_td_args &a = *args;
    trace_bind();
    if (a.variant < 0 || a.variant > 2 || a.B < 0 || a.n_pol < 0 || a.D < 1) { set_error("sfgpi_td_step: invalid arguments"); return SFGPI_E_INVALID; }
    if (a.B == 0 || a.n_pol == 0) return SFGPI_OK;
    const bool tsf = a.variant == 2;
    const int want_aux = a.variant == 0 ? 0 : (tsf ? a.D + a.G * a.S + a.G + tsf_flow_len(a.S, a.n_flows) + a.D * a.G + a.D : a.D);
    if (a.aux_len < want_aux) { set_error("sfgpi_td_step: aux_len %d < %d", a.aux_len, want_aux); return SFGPI_E_INVALID; }
    if (tsf && a.tsf_part == nullptr) { set_error("sfgpi_td_step: variant 2 needs the tsf_part scratch buffer"); return SFGPI_E_INVALID; }
    const int K = tsf ? a.n_flows : 0;
    if (K < 0) { set_error("sfgpi_td_step: n_flows < 0"); return SFGPI_E_INVALID; }
    const int n_red = tsf ? tsf_red_len(a.D, a.S, K) : a.D;
    size_t fl = a.D + 4 * (size_t)kTdRows * a.D + 3 * kTdRows + 8 + (size_t)n_red + 2;
    if (tsf) fl += (size_t)a.D * a.S + a.D + 2 * (size_t)kTdRows * a.S + (a.tsf_mc ? 0 : (size_t)a.G * a.S + a.G + (size_t)a.D * a.G + a.D);
    if (K > 0) fl += 3 * (size_t)tsf_flow_len(a.S, K) + 2 * (size_t)kTdRows * ((size_t)(K + 1) * a.S + K);
    const size_t bytes = fl * sizeof(float);
    const int nclu = sfgpi_td_partials(a.B);
    dim3 grid(nclu * kTdCluster, a.n_pol);
    sfgpi_peer_keys_args pk = {};
    if (a.peer_keys != nullptr) {
        pk = *reinterpret_cast<const sfgpi_peer_keys_args *>(a.peer_keys);
        if (a.next_psi == nullptr || pk.ctx.world < 1 || pk.ctx.world > SFGPI_MAX_PEERS || pk.ctx.rank < 0 || pk.ctx.rank >= pk.ctx.world ||
            pk.epoch <= 0 || pk.B != a.B || pk.n_rows < a.n_pol) {
            set_error("sfgpi_td_step: peer_keys does not describe this step (needs next_psi, same B, n_rows >= n_pol, epoch > 0)");
            return SFGPI_E_INVALID;
        }
        for (int r = 0; r < pk.ctx.world; ++r)
            if (!pk.ctx.flags[r] || !pk.keys_all[r]) { set_error("sfgpi_td_step: peer arena of rank %d not mapped", r); return SFGPI_E_INVALID; }
    }
    // every argument is checked before the first CUDA call; both launches' shared memory before the first launch
    const size_t ebytes = ((size_t)n_red + (size_t)a.G * a.S + a.G + (size_t)a.D * a.G) * sizeof(float);
    static int td_static = -1, expand_static = -1;
    if (int rc = smem_opt_in(td_kernel, bytes, &td_static, "sfgpi_td_step (D/G too large)")) return rc;
    if (tsf && !a.defer_expand)
        if (int rc = smem_opt_in(tsf_expand_kernel, ebytes, &expand_static, "sfgpi_td_step(expand)")) return rc;
    launch_pdl(td_kernel, grid, dim3(kTdThreads), bytes, (cudaStream_t)stream, a, pk);
    int rc = check_launch("sfgpi_td_step");
    if (rc || !tsf || a.defer_expand) return rc;              // deferred: the expand rides in sfgpi_mlp_backward_tc's dgrad launch
    launch_pdl(tsf_expand_kernel, dim3(a.n_pol), dim3(256), ebytes, (cudaStream_t)stream, a, nclu);
    return check_launch("sfgpi_td_step(expand)");
}
