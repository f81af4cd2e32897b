// Backward of the psi MLP, fp32 CUDA-core path: (1) fused dgrad chain, (2) split-K wgrad + bias grad.
//
// The TD loss touches psi(s)[b, a_b, :] only (sfdqn.py:334-335: merge[indices, actions,:] = targets), so dZ of the last layer
// is D-sparse per row; it is kept as d_out [n_pol][B][D] in HBM and expanded on the fly while staging shared-memory chunks.
// A general loss (autograd through PackedSFLibrary.psi) has a dense dZ of the last layer: actions == NULL, d_out is
// [B][n_pol][A*D] (the forward's psi_out layout).  Both are template instantiations (kDense), so the sparse kernels are
// exactly the train step's.
#include "common.cuh"

namespace sfgpi {

// acc[r][c] += sum_n A[row ty*8+r][n] * W[n][kout0 + c*32+tx],  n in [0, nred)   (NN: reduction index = weight row)
// dense:  A = As (smem tile, stride lda).   sparse (last layer): A[row][n] = dsel[row][n - sel[row]*D] inside the action's
// D columns, else 0 -- materialised per 32-wide chunk into dzc.  kDense (last layer of a dense d_out): A[row][n] =
// dsel[row * dld + n] for the rows_ok rows inside the batch, dsel pointing into d_out in global memory.
template <bool kDense>
__device__ __forceinline__ void cta_gemm_nn(float (&acc)[8][8], const float *As, int lda, int nred,
                                            const float *__restrict__ W, int ldw, int kcols, float *Ws, bool sparse,
                                            float *dzc, const float *dsel, const int *sel_s, int D,
                                            size_t dld, int rows_ok) {
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5, tid = threadIdx.x;
    const int nc8 = (kcols + 31) >> 5;
    const bool aligned = ((ldw & 3) == 0) && ((reinterpret_cast<uintptr_t>(W) & 15) == 0);
    const int nchunks = (nred + kKC - 1) / kKC;
    {
        int nlen = min(kKC, nred);
        stage_rows(Ws, kWsNN, W, ldw, nlen, (nlen + 3) & ~3, kcols, nc8 * 32, aligned);
        cp_async_commit();
    }
    for (int ch = 0; ch < nchunks; ++ch) {
        const int n0 = ch * kKC;
        const int nlen = min(kKC, nred - n0), nlen4 = (nlen + 3) & ~3;
        if (ch + 1 < nchunks) {
            int n1 = n0 + kKC, nl1 = min(kKC, nred - n1);
            stage_rows(Ws + ((ch + 1) & 1) * kWsFloats, kWsNN, W + (size_t)n1 * ldw, ldw, nl1, (nl1 + 3) & ~3, kcols,
                       nc8 * 32, aligned);
            cp_async_commit();
        }
        if (sparse) {
            for (int e = tid; e < kBM * nlen4; e += kThreads) {
                int r = e / nlen4, nn = e - r * nlen4;
                if constexpr (kDense) {
                    dzc[r * kWsNT + nn] = (nn < nlen && r < rows_ok) ? dsel[(size_t)r * dld + n0 + nn] : 0.0f;
                } else {
                    unsigned off = (unsigned)(n0 + nn - sel_s[r] * D);
                    dzc[r * kWsNT + nn] = (nn < nlen && off < (unsigned)D) ? dsel[r * D + off] : 0.0f;
                }
            }
        }
        if (ch + 1 < nchunks) cp_async_wait<1>(); else cp_async_wait<0>();
        __syncthreads();
        const float *Wb = Ws + (ch & 1) * kWsFloats + tx;
        const float *Ab = sparse ? dzc + (ty * 8) * kWsNT : As + (ty * 8) * lda + n0;
        const int astr = sparse ? kWsNT : lda;
        for (int nn = 0; nn < nlen4; nn += 4) {
            float4 a[8];
#pragma unroll
            for (int r = 0; r < 8; ++r) a[r] = *reinterpret_cast<const float4 *>(Ab + r * astr + nn);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float *wr = Wb + (nn + j) * kWsNN;
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    if (c < nc8) {
                        const float b = wr[c * 32];
#pragma unroll
                        for (int r = 0; r < 8; ++r) {
                            const float av = j == 0 ? a[r].x : (j == 1 ? a[r].y : (j == 2 ? a[r].z : a[r].w));
                            acc[r][c] = fmaf(av, b, acc[r][c]);
                        }
                    }
                }
            }
        }
        __syncthreads();
    }
}

struct BwdSmem { int lda, off_act1, off_ws, off_dzc, off_dsel, off_sel, total_bytes; };

__host__ __device__ inline BwdSmem bwd_smem_layout(const sfgpi_net_desc &net) {
    int maxw = 4;
    for (int l = 1; l < net.n_layers; ++l) maxw = max(maxw, net.dims[l]);
    maxw = (maxw + 3) & ~3;
    BwdSmem s;
    s.lda = maxw + 4;
    s.off_act1 = kBM * s.lda;
    s.off_ws = 2 * kBM * s.lda;
    s.off_dzc = s.off_ws + 2 * kWsFloats;
    s.off_dsel = s.off_dzc + kBM * kWsNT;
    s.off_sel = s.off_dsel + ((kBM * net.n_features + 3) & ~3);
    s.total_bytes = (s.off_sel + kBM) * 4;
    return s;
}

// ---- (1) dgrad chain: dZ_{L-1} (sparse or dense) -> dZ_{L-2} -> ... -> dZ_0, all inside one CTA per (policy, 64-row tile) ----
template <bool kDense>
__global__ void __launch_bounds__(kThreads, 1) mlp_dgrad_kernel(const __grid_constant__ sfgpi_backward_args a) {
    extern __shared__ __align__(16) float smem[];
    const sfgpi_net_desc &net = a.net;
    const int tid = threadIdx.x, tx = tid & 31, ty = tid >> 5;
    const int L = net.n_layers, D = net.n_features, B = a.B;
    const BwdSmem lay = bwd_smem_layout(net);
    const int lda = lay.lda;
    float *cur = smem, *nxt = smem + lay.off_act1, *Ws = smem + lay.off_ws, *dzc = smem + lay.off_dzc,
          *dsel = smem + lay.off_dsel;
    int *sel_s = reinterpret_cast<int *>(smem + lay.off_sel);
    const int pl = blockIdx.y, row0 = blockIdx.x * kBM;
    const float *P = a.params + (size_t)(a.policy_lo + pl) * net.row_stride;

    const int AD = net.dims[L];
    const float *dsrc = dsel;
    if constexpr (kDense) {
        dsrc = a.d_out + ((size_t)row0 * a.n_pol + pl) * AD;
    } else {
        for (int e = tid; e < kBM * D; e += kThreads) {
            int r = e / D;
            dsel[e] = (row0 + r < B) ? a.d_out[((size_t)pl * B + row0) * D + e] : 0.0f;
        }
        if (tid < kBM) sel_s[tid] = (row0 + tid < B) ? (int)a.actions[row0 + tid] : 0;
    }
    __syncthreads();

    for (int l = L - 1; l >= 1; --l) {
        const int nred = net.dims[l + 1], K = net.dims[l];       // dA_{l-1} [64][K] = dZ_l [64][nred] . W_l [nred][K]
        const float *W = P + net.w_off[l];
        const int act_prev = net.acts[l - 1];
        const float *a_prev = a.acts[l - 1] + (size_t)pl * B * K;
        float *dz_out = a.dz[l - 1] + (size_t)pl * B * K;
        for (int k0 = 0; k0 < K; k0 += kNC) {
            const int kcols = min(kNC, K - k0), nc8 = (kcols + 31) >> 5;
            float acc[8][8];
#pragma unroll
            for (int r = 0; r < 8; ++r)
#pragma unroll
                for (int c = 0; c < 8; ++c) acc[r][c] = 0.0f;
            cta_gemm_nn<kDense>(acc, cur, lda, nred, W + k0, K, kcols, Ws, l == L - 1, dzc, dsrc, sel_s, D,
                                (size_t)a.n_pol * AD, B - row0);
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const int cc = c * 32 + tx, k = k0 + cc;
                if (c < nc8 && cc < kcols) {
#pragma unroll
                    for (int r = 0; r < 8; ++r) {
                        const int row = ty * 8 + r, b = row0 + row;
                        float v = 0.0f;
                        if (b < B) {
                            v = acc[r][c] * act_grad(a_prev[(size_t)b * K + k], act_prev);
                            dz_out[(size_t)b * K + k] = v;
                        }
                        nxt[row * lda + k] = v;
                    }
                }
            }
        }
        const int K4 = (K + 3) & ~3;
        if (K4 != K)
            for (int e = tid; e < kBM * (K4 - K); e += kThreads) {
                int r = e / (K4 - K), k = K + (e - r * (K4 - K));
                nxt[r * lda + k] = 0.0f;
            }
        __syncthreads();
        float *t = cur; cur = nxt; nxt = t;
    }
}

// ---- (2) wgrad: dW_l [N][K] = dZ_l^T [N][B] . in_l [B][K],  db_l = colsum(dZ_l);  split-K over the batch ----
constexpr int kWgN = 64;                 // dW rows per CTA tile
constexpr int kWgLdz = kWgN + 4;
constexpr int kWgStage = kKC * kWgLdz + kKC * kWsNN;     // floats per pipeline stage

__device__ __forceinline__ int wg_tiles_of_layer(const sfgpi_net_desc &net, int l) {
    return ((net.dims[l + 1] + kWgN - 1) / kWgN) * ((net.dims[l] + kNC - 1) / kNC);
}

template <bool kDense>
__global__ void __launch_bounds__(kThreads, 1) mlp_wgrad_kernel(const __grid_constant__ sfgpi_backward_args a, int tiles_per_split) {
    extern __shared__ __align__(16) float smem[];
    const sfgpi_net_desc &net = a.net;
    const int tid = threadIdx.x, tx = tid & 31, ty = tid >> 5;
    const int L = net.n_layers, D = net.n_features, B = a.B;
    const int pl = blockIdx.y;
    const int split = blockIdx.x / tiles_per_split;
    int t = blockIdx.x - split * tiles_per_split;
    int l = 0;
    for (; l < L; ++l) {
        int nt = wg_tiles_of_layer(net, l);
        if (t < nt) break;
        t -= nt;
    }
    const int N = net.dims[l + 1], K = net.dims[l];
    const int kchunks = (K + kNC - 1) / kNC;
    const int n0 = (t / kchunks) * kWgN, k0 = (t % kchunks) * kNC;
    const int nrows = min(kWgN, N - n0), kcols = min(kNC, K - k0);
    const int nc8 = (kcols + 31) >> 5;
    const bool last = (l == L - 1);

    // batch range of this split, in multiples of 32 rows
    const int chunks_total = (B + kKC - 1) / kKC;
    const int chunks_per_split = (chunks_total + a.n_split - 1) / a.n_split;
    const int ch_lo = split * chunks_per_split, ch_hi = min(chunks_total, ch_lo + chunks_per_split);

    const float *in = (l == 0) ? a.x : a.acts[l - 1] + (size_t)pl * B * K;         // [B][K]
    const float *dz = last ? a.d_out + (size_t)pl * B * D : a.dz[l] + (size_t)pl * B * N;
    const bool in_aligned = ((K & 3) == 0) && ((k0 & 3) == 0) && ((reinterpret_cast<uintptr_t>(in) & 15) == 0);
    const bool dz_aligned = !last && ((N & 3) == 0) && ((reinterpret_cast<uintptr_t>(dz) & 15) == 0);

    float acc[8][8], bsum[8];
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        bsum[r] = 0.0f;
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[r][c] = 0.0f;
    }

    auto stage = [&](int ch, int buf) {
        float *dzs = smem + buf * kWgStage, *ins = dzs + kKC * kWgLdz;
        const int b0 = ch * kKC, blen = min(kKC, B - b0);
        stage_rows(ins, kWsNN, in + (size_t)b0 * K + k0, K, blen, kKC, kcols, nc8 * 32, in_aligned);
        if (!last) {
            stage_rows(dzs, kWgLdz, dz + (size_t)b0 * N + n0, N, blen, kKC, nrows, kWgN, dz_aligned);
        } else if constexpr (kDense) {                   // dense d_out [B][n_pol][A*D]: row b of policy pl is strided
            const int ldd = a.n_pol * N;
            const float *src = a.d_out + ((size_t)b0 * a.n_pol + pl) * N + n0;
            const bool al = ((ldd & 3) == 0) && ((reinterpret_cast<uintptr_t>(src) & 15) == 0);
            stage_rows(dzs, kWgLdz, src, ldd, blen, kKC, nrows, kWgN, al);
        } else {
            for (int e = tid; e < kKC * kWgN; e += kThreads) {
                int r = e / kWgN, nn = e - r * kWgN;
                float v = 0.0f;
                if (r < blen && nn < nrows) {
                    unsigned off = (unsigned)(n0 + nn - (int)a.actions[b0 + r] * D);
                    if (off < (unsigned)D) v = dz[(size_t)(b0 + r) * D + off];
                }
                dzs[r * kWgLdz + nn] = v;
            }
        }
    };

    if (ch_lo < ch_hi) {
        stage(ch_lo, 0);
        cp_async_commit();
    }
    for (int ch = ch_lo; ch < ch_hi; ++ch) {
        const int buf = (ch - ch_lo) & 1;
        if (ch + 1 < ch_hi) {
            stage(ch + 1, buf ^ 1);
            cp_async_commit();
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
        const float *dzs = smem + buf * kWgStage + ty * 8, *ins = smem + buf * kWgStage + kKC * kWgLdz + tx;
#pragma unroll 4
        for (int r32 = 0; r32 < kKC; ++r32) {
            const float4 a0 = *reinterpret_cast<const float4 *>(dzs + r32 * kWgLdz);
            const float4 a1 = *reinterpret_cast<const float4 *>(dzs + r32 * kWgLdz + 4);
            const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
            for (int r = 0; r < 8; ++r) bsum[r] += av[r];
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                if (c < nc8) {
                    const float b = ins[r32 * kWsNN + c * 32];
#pragma unroll
                    for (int r = 0; r < 8; ++r) acc[r][c] = fmaf(av[r], b, acc[r][c]);
                }
            }
        }
        __syncthreads();
    }

    float *gp = a.grad_part + ((size_t)pl * a.n_split + split) * net.row_stride;
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        const int n = n0 + ty * 8 + r;
        if (ty * 8 + r < nrows) {
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const int cc = c * 32 + tx;
                if (c < nc8 && cc < kcols) gp[net.w_off[l] + (size_t)n * K + k0 + cc] = acc[r][c];
            }
            if (k0 == 0 && tx == 0) gp[net.b_off[l] + n] = bsum[r];
        }
    }
}

}  // namespace sfgpi

using namespace sfgpi;

extern "C" int sfgpi_mlp_backward(const sfgpi_backward_args *args, void *stream) {
    const sfgpi_backward_args &a = *args;
    const sfgpi_net_desc &net = a.net;
    if (net.n_layers < 1 || net.n_layers > SFGPI_MAX_LAYERS || a.B < 0 || a.n_pol < 0 || a.n_split < 1 ||
        net.dims[net.n_layers] != net.n_actions * net.n_features || net.acts[net.n_layers - 1] != SFGPI_ACT_NONE) {
        set_error("sfgpi_mlp_backward: invalid arguments (the output layer must be linear)");
        return SFGPI_E_INVALID;
    }
    if (a.B == 0 || a.n_pol == 0) return SFGPI_OK;
    if (!a.d_out) { set_error("sfgpi_mlp_backward: d_out is NULL"); return SFGPI_E_INVALID; }
    const bool dense = a.actions == nullptr;             // d_out [B][n_pol][A*D] instead of [n_pol][B][D]
    cudaStream_t st = (cudaStream_t)stream;
    if (net.n_layers > 1) {
        const BwdSmem lay = bwd_smem_layout(net);
        if (lay.total_bytes > kMaxSmem) { set_error("sfgpi_mlp_backward: needs %d B shared memory", lay.total_bytes); return SFGPI_E_SMEM; }
        static bool cfg = false;
        if (!cfg) {
            cudaFuncSetAttribute(mlp_dgrad_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem);
            cudaFuncSetAttribute(mlp_dgrad_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem);
            cfg = true;
        }
        dim3 grid((a.B + kBM - 1) / kBM, a.n_pol);
        if (dense) mlp_dgrad_kernel<true><<<grid, kThreads, lay.total_bytes, st>>>(a);
        else mlp_dgrad_kernel<false><<<grid, kThreads, lay.total_bytes, st>>>(a);
        int rc = check_launch("sfgpi_mlp_backward(dgrad)");
        if (rc) return rc;
    }
    int tiles = 0;
    for (int l = 0; l < net.n_layers; ++l)
        tiles += ((net.dims[l + 1] + kWgN - 1) / kWgN) * ((net.dims[l] + kNC - 1) / kNC);
    static bool cfg2 = false;
    const int wg_bytes = 2 * kWgStage * (int)sizeof(float);
    if (!cfg2) {
        cudaFuncSetAttribute(mlp_wgrad_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, wg_bytes);
        cudaFuncSetAttribute(mlp_wgrad_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, wg_bytes);
        cfg2 = true;
    }
    dim3 grid(tiles * a.n_split, a.n_pol);
    if (dense) mlp_wgrad_kernel<true><<<grid, kThreads, wg_bytes, st>>>(a, tiles);
    else mlp_wgrad_kernel<false><<<grid, kThreads, wg_bytes, st>>>(a, tiles);
    return check_launch("sfgpi_mlp_backward(wgrad)");
}
