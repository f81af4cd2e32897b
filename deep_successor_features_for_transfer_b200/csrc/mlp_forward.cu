// Fused ensemble psi-MLP forward, fp32 CUDA-core path (mode 0: the 1e-5 parity mode).
//
// One CTA = one (policy, 64-state tile).  The whole chain Linear -> act -> ... -> Linear runs inside the CTA: activations
// ping-pong between two shared-memory tiles and never touch HBM; weights stream L2 -> smem through a 2-stage cp.async
// pipeline.  The last layer is produced in column chunks whose epilogue is one of
//   (a) store psi  (get_successors, sfdqn.py:295-301)
//   (b) GPI: q = psi . w, per-state (max, argmax) folded into packed int64 keys with atomicMax (GPI_w, sfdqn.py:215-240)
//   (c) gather psi[b, a_b, :] for the TD target / current value (sfdqn.py:328-335)
// and hidden layers can additionally be saved for the backward pass.
#include "common.cuh"

namespace sfgpi {

struct FwdSmem {
    int lda;            // activation tile row stride (floats)
    int off_act1;       // float offsets into dynamic smem
    int off_ws;
    int off_w;          // reward vectors [n_w][D]
    int off_sel;        // int[BM] selected action per row
    int total_bytes;
};

__host__ __device__ inline FwdSmem fwd_smem_layout(const sfgpi_net_desc &net, bool gpi, int n_w) {
    int maxw = 0;
    for (int l = 0; l < net.n_layers; ++l) maxw = max(maxw, net.dims[l]);
    maxw = (maxw + 3) & ~3;
    if (gpi) maxw = max(maxw, kNC);
    FwdSmem s;
    s.lda = maxw + 4;
    s.off_act1 = kBM * s.lda;
    s.off_ws = 2 * kBM * s.lda;
    s.off_w = s.off_ws + 2 * kWsFloats;
    s.off_sel = s.off_w + ((gpi ? n_w * net.n_features : 0) + 3 & ~3);
    s.total_bytes = (s.off_sel + kBM) * 4;
    return s;
}

__global__ void __launch_bounds__(kThreads, 1) mlp_forward_kernel(const __grid_constant__ sfgpi_forward_args a) {
    extern __shared__ __align__(16) float smem[];
    const sfgpi_net_desc &net = a.net;
    const int tid = threadIdx.x, tx = tid & 31, ty = tid >> 5;
    const int L = net.n_layers, A = net.n_actions, D = net.n_features, AD = A * D;
    const bool gpi = (a.w != nullptr);
    const FwdSmem lay = fwd_smem_layout(net, gpi, a.w_diag ? 1 : a.n_w);
    const int lda = lay.lda;
    float *cur = smem, *nxt = smem + lay.off_act1, *Ws = smem + lay.off_ws, *w_s = smem + lay.off_w;
    int *sel_s = reinterpret_cast<int *>(smem + lay.off_sel);

    const int pl = blockIdx.y;                         // local policy slot
    const int row0 = blockIdx.x * kBM;
    const int B = a.B;
    const float *P = a.params + (size_t)(a.policy_lo + pl) * net.row_stride;

    // ---- stage the input tile (zero-padded to a multiple of 4 columns and to 64 rows), w and the gather selectors ----
    {
        const int S = net.dims[0], S4 = (S + 3) & ~3;
        for (int e = tid; e < kBM * S4; e += kThreads) {
            int r = e / S4, k = e - r * S4;
            cur[r * lda + k] = (k < S && row0 + r < B) ? a.x[(size_t)(row0 + r) * S + k] : 0.0f;
        }
        if (gpi) {
            const float *wsrc = a.w_diag ? a.w + (size_t)pl * D : a.w;      // diag: only this policy's own reward vector
            const int nw = a.w_diag ? 1 : a.n_w;
            for (int e = tid; e < nw * D; e += kThreads) w_s[e] = wsrc[e];
        }
        if (a.sel_out != nullptr && tid < kBM) {
            int b = row0 + tid, s = 0;
            if (b < B) {
                if (a.sel_actions != nullptr) s = (int)a.sel_actions[b];
                else s = (int)key_index(a.sel_keys[(size_t)pl * a.sel_key_stride + b]);
            }
            sel_s[tid] = s;
        }
    }
    __syncthreads();

    for (int l = 0; l < L; ++l) {
        const int K = net.dims[l], N = net.dims[l + 1];
        const bool last = (l == L - 1);
        const float *W = P + net.w_off[l];
        const float *bias = P + net.b_off[l];
        const int act = net.acts[l];
        const int chunk = (last && gpi) ? (kNC / D) * D : kNC;      // GPI epilogue needs whole actions per chunk
        for (int n0 = 0; n0 < N; n0 += chunk) {
            const int ncols = min(chunk, N - n0);
            const int nc8 = (ncols + 31) >> 5;
            float acc[8][8];
#pragma unroll
            for (int r = 0; r < 8; ++r)
#pragma unroll
                for (int c = 0; c < 8; ++c) acc[r][c] = 0.0f;
            cta_gemm_nt(acc, cur, lda, W + (size_t)n0 * K, K, ncols, Ws);

            // bias + activation
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const int n = n0 + c * 32 + tx;
                if (c < nc8 && c * 32 + tx < ncols) {
                    const float bv = bias[n];
#pragma unroll
                    for (int r = 0; r < 8; ++r) acc[r][c] = apply_act(acc[r][c] + bv, act);
                }
            }

            if (!last) {
                float *save = a.acts_out[l] ? a.acts_out[l] + (size_t)pl * B * N : nullptr;
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const int cc = c * 32 + tx, n = n0 + cc;
                    if (c < nc8 && cc < ncols) {
#pragma unroll
                        for (int r = 0; r < 8; ++r) {
                            const int row = ty * 8 + r;
                            nxt[row * lda + n] = acc[r][c];
                            if (save && row0 + row < B) save[(size_t)(row0 + row) * N + n] = acc[r][c];
                        }
                    }
                }
                continue;
            }

            // ---------------- last layer epilogues ----------------
            if (a.psi_out != nullptr) {
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const int cc = c * 32 + tx;
                    if (c < nc8 && cc < ncols) {
#pragma unroll
                        for (int r = 0; r < 8; ++r) {
                            const int b = row0 + ty * 8 + r;
                            if (b < B) a.psi_out[((size_t)b * a.n_pol + pl) * AD + n0 + cc] = acc[r][c];
                        }
                    }
                }
            }
            if (a.sel_out != nullptr) {
#pragma unroll
                for (int r = 0; r < 8; ++r) {
                    const int row = ty * 8 + r, b = row0 + row;
                    const int base = sel_s[row] * D;
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        const int cc = c * 32 + tx;
                        const unsigned off = (unsigned)(n0 + cc - base);
                        if (c < nc8 && cc < ncols && off < (unsigned)D && b < B)
                            a.sel_out[((size_t)pl * B + b) * D + off] = acc[r][c];
                    }
                }
            }
            if (gpi) {
                // tile -> smem (the idle activation buffer), then 4 lanes per state reduce q over their share of actions
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const int cc = c * 32 + tx;
                    if (c < nc8 && cc < ncols) {
#pragma unroll
                        for (int r = 0; r < 8; ++r) nxt[(ty * 8 + r) * lda + cc] = acc[r][c];
                    }
                }
                __syncthreads();
                const int na = ncols / D, a0 = n0 / D;
                const int row = tid >> 2, sub = tid & 3, b = row0 + row;
                const float *trow = nxt + row * lda;
                const int nw = a.w_diag ? 1 : a.n_w;
                for (int wl = 0; wl < nw; ++wl) {
                    const float *wv = w_s + wl * D;
                    const int wi = a.w_diag ? pl : wl;                      // key row
                    // (-inf, the chunk's first action): a chunk emits a key even when no q beats -inf (all NaN / -inf), so
                    // such a state decodes to action 0 as in the tensor-core scans, never to the unwritten key's index
                    float best = -INFINITY;
                    int best_a = a0;
                    for (int al = sub; al < na; al += 4) {
                        const float *pv = trow + al * D;
                        float q = 0.0f;
                        for (int d = 0; d < D; ++d) q = fmaf(pv[d], wv[d], q);
                        if (a.q_out != nullptr && wl == 0 && b < B)
                            a.q_out[((size_t)b * a.n_pol + pl) * A + a0 + al] = q;
                        if (q > best) { best = q; best_a = a0 + al; }         // ascending a: first max wins
                    }
#pragma unroll
                    for (int o = 1; o < 4; o <<= 1) {
                        const float ob = __shfl_xor_sync(0xffffffffu, best, o);
                        const int oa = __shfl_xor_sync(0xffffffffu, best_a, o);
                        if (ob > best || (ob == best && oa < best_a)) { best = ob; best_a = oa; }
                    }
                    if (sub == 0 && b < B) {
                        if (a.key_action) atomicMax(reinterpret_cast<long long *>(a.key_action) + (size_t)wi * B + b,
                                                    pack_key(best, (uint32_t)best_a));
                        if (a.key_task) atomicMax(reinterpret_cast<long long *>(a.key_task) + (size_t)wi * B + b,
                                                  pack_key(best, (uint32_t)(a.task_base + pl)));
                    }
                }
                __syncthreads();
            }
        }
        if (!last) {
            // zero the K-padding columns of the next layer's input, then swap the ping-pong tiles
            const int N4 = (N + 3) & ~3;
            if (N4 != N)
                for (int e = tid; e < kBM * (N4 - N); e += kThreads) {
                    int r = e / (N4 - N), k = N + (e - r * (N4 - N));
                    nxt[r * lda + k] = 0.0f;
                }
            __syncthreads();
            float *t = cur; cur = nxt; nxt = t;
        }
    }
}

}  // namespace sfgpi

using namespace sfgpi;

extern "C" int sfgpi_mlp_forward(const sfgpi_forward_args *args, void *stream) {
    const sfgpi_forward_args &a = *args;
    const sfgpi_net_desc &net = a.net;
    if (net.n_layers < 1 || net.n_layers > SFGPI_MAX_LAYERS || a.B < 0 || a.n_pol < 0 ||
        net.dims[net.n_layers] != net.n_actions * net.n_features) {
        set_error("sfgpi_mlp_forward: invalid network descriptor / sizes");
        return SFGPI_E_INVALID;
    }
    if (a.mode != 0) { set_error("sfgpi_mlp_forward: mode %d not built into this entry point", a.mode); return SFGPI_E_INVALID; }
    if (a.B == 0 || a.n_pol == 0) return SFGPI_OK;
    const bool gpi = a.w != nullptr;
    if (gpi && (net.n_features > kNC || a.n_w < 1)) {
        set_error("sfgpi_mlp_forward: fused GPI needs 1 <= D <= %d and n_w >= 1", kNC);
        return SFGPI_E_INVALID;
    }
    if (a.sel_out && !a.sel_actions && !a.sel_keys) { set_error("sfgpi_mlp_forward: sel_out without selectors"); return SFGPI_E_INVALID; }
    const FwdSmem lay = fwd_smem_layout(net, gpi, a.w_diag ? 1 : a.n_w);
    if (lay.total_bytes > kMaxSmem) {
        set_error("sfgpi_mlp_forward: layer width / n_w*D needs %d B of shared memory (> %d)", lay.total_bytes, kMaxSmem);
        return SFGPI_E_SMEM;
    }
    static int configured = 0;
    if (configured < lay.total_bytes) {
        cudaFuncSetAttribute(mlp_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem);
        configured = kMaxSmem;
    }
    dim3 grid((a.B + kBM - 1) / kBM, a.n_pol);
    mlp_forward_kernel<<<grid, kThreads, lay.total_bytes, (cudaStream_t)stream>>>(a);
    return check_launch("sfgpi_mlp_forward");
}
