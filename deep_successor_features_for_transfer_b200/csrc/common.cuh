// Shared device helpers for the fp32 (CUDA-core, 1e-5 parity) path of the SF/GPI hot path.  sm_100a only.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/sfgpi.h"

namespace sfgpi {

constexpr int kThreads = 256;      // 8 warps per CTA: warp = 8-row band, lane = column (mod 32)
constexpr int kBM = 64;            // rows (states) per CTA tile
constexpr int kKC = 32;            // reduction chunk staged in shared memory
constexpr int kNC = 256;           // output-column chunk: 8 columns per lane, interleaved by 32
constexpr int kWsNT = kKC + 4;     // row stride of a [n][k] weight chunk: 36 == 4 (mod 32) -> conflict-free LDS.128
constexpr int kWsNN = kNC + 4;     // row stride of a [k_red][n] chunk (lanes read consecutive words)
constexpr int kWsFloats = kNC * kWsNT;   // one weight stage (9216 floats) -- also holds a [32][260] NN chunk (8320)
constexpr int kMaxSmem = 227 * 1024;

void set_error(const char *fmt, ...);
int check_launch(const char *what);

// ---- programmatic dependent launch (PDL): the kernels of one train step are a dependent chain of a dozen small launches, so
// launch latency and per-kernel set-up are a large share of the step.  Every kernel lets its successor be scheduled at once
// (launch_dependents) and itself waits for its predecessor's memory (wait) only after its own data-independent set-up.
// Developer aid (env SFGPI_TRACE=1, sfgpi_trace_dump): %globaltimer window of every step kernel -- first CTA entry, first CTA
// past its dependency wait, last CTA exit -- so that the gaps BETWEEN the kernels of a step can be read, not only their own
// durations.  The buffer pointer is a per-translation-unit device global bound lazily by trace_bind() in the launching host code.
enum { SFGPI_TR_PREP = 0, SFGPI_TR_FWD = 1, SFGPI_TR_TD = 2, SFGPI_TR_DGRAD = 3, SFGPI_TR_WGRAD = 4, SFGPI_TR_ADAM = 5, SFGPI_TR_PEER_X = 6, SFGPI_TR_SLOTS = 8 };
unsigned long long *trace_buffer();          // gpi.cu: device buffer [SFGPI_TR_SLOTS][3], or NULL while tracing is off
int trace_generation();                       // gpi.cu: bumped by sfgpi_trace_enable(); a translation unit re-binds when it changed
static __device__ unsigned long long *g_trace = nullptr;
static inline void trace_bind() {
    static int bound_gen = -1;
    const int gen = trace_generation();
    if (bound_gen == gen) return;
    unsigned long long *p = trace_buffer();
    cudaMemcpyToSymbol(g_trace, &p, sizeof(p));
    bound_gen = gen;
}
__device__ __forceinline__ void trace_mark(int slot, int what) {
    if (slot >= 0 && threadIdx.x == 0 && g_trace != nullptr) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        if (what == 2) atomicMax(g_trace + 3 * slot + 2, t);
        else atomicMin(g_trace + 3 * slot + what, t);
    }
}
__device__ __forceinline__ void pdl_launch_dependents(int trace_slot = -1) {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    trace_mark(trace_slot, 0);
}
__device__ __forceinline__ void pdl_wait(int trace_slot = -1) {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    trace_mark(trace_slot, 1);
}
__device__ __forceinline__ void trace_exit(int trace_slot) { trace_mark(trace_slot, 2); }

bool pdl_enabled();

template <typename... KArgs, typename... Args>
inline void launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args &&...args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    int n = 0;
    if (pdl_enabled()) {
        attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[n].val.programmaticStreamSerializationAllowed = 1;
        ++n;
    }
    cfg.attrs = attr;
    cfg.numAttrs = n;
    cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}

__device__ __forceinline__ float apply_act(float v, int act) {
    if (act == SFGPI_ACT_RELU) return fmaxf(v, 0.0f);
    if (act == SFGPI_ACT_TANH) return tanhf(v);
    return v;
}
// derivative of the activation expressed through its OUTPUT a (torch: threshold_backward / tanh_backward)
__device__ __forceinline__ float act_grad(float a, int act) {
    if (act == SFGPI_ACT_RELU) return a > 0.0f ? 1.0f : 0.0f;
    if (act == SFGPI_ACT_TANH) return 1.0f - a * a;
    return 1.0f;
}

// ---- packed (value, index) keys: signed int64 max == (max value, then smallest index) -------------------------
__device__ __forceinline__ long long pack_key(float v, uint32_t idx) {
    v += 0.0f;                                   // -0 -> +0 so that equal values order equally
    int32_t b = __float_as_int(v);
    b = b >= 0 ? b : (b ^ 0x7FFFFFFF);           // monotone map float -> int32
    return (long long)(((unsigned long long)(uint32_t)b << 32) | (unsigned long long)(0xFFFFFFFFu - idx));
}
__device__ __forceinline__ uint32_t key_index(long long k) { return 0xFFFFFFFFu - (uint32_t)((unsigned long long)k & 0xFFFFFFFFull); }
__device__ __forceinline__ float key_value(long long k) {
    int32_t b = (int32_t)((unsigned long long)k >> 32);
    b = b >= 0 ? b : (b ^ 0x7FFFFFFF);
    return __int_as_float(b);
}

// ---------------------------------------------------------------------------------------------------------------
// CTA-level GEMM building blocks.  Thread (ty = warp, tx = lane) owns rows ty*8+r (r<8) and columns c*32+tx (c<8) of a
// 64 x 256 output chunk; nc8 = ceil(valid_cols/32) bounds the (warp-uniform) column loop.
// ---------------------------------------------------------------------------------------------------------------

// Stage W[n0+n][k0 .. k0+klen) (global, [n][K] row-major) into Ws[n][0..klen4) for n < ncols; zero-fill the rest of the
// touched rectangle (rows up to nc8*32, columns up to klen4).
__device__ __forceinline__ void stage_w_nt(float *Ws, const float *__restrict__ W, int K, int k0, int klen, int klen4,
                                           int ncols, int nc8, bool aligned) {
    const int tid = threadIdx.x;
    const int nrows = nc8 * 32;
    if (aligned) {                                // K % 4 == 0 and 16B-aligned base: 8 lanes cover one 128 B row segment
        const int q = tid & 7, nq = klen4 >> 2;
        for (int n = tid >> 3; n < nrows; n += kThreads / 8) {
            if (q < nq) {
                float *dst = Ws + n * kWsNT + q * 4;
                if (n < ncols) cp_async16(dst, W + (size_t)n * K + k0 + q * 4);
                else *reinterpret_cast<float4 *>(dst) = make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
    } else {
        for (int e = tid; e < nrows * klen4; e += kThreads) {
            int n = e / klen4, k = e - n * klen4;
            Ws[n * kWsNT + k] = (n < ncols && k < klen) ? W[(size_t)n * K + k0 + k] : 0.0f;
        }
    }
}

// acc[r][c] += sum_k As[(ty*8+r)*lda + k] * W[n0 + c*32+tx][k]    (NT: both operands contiguous along k)
__device__ __forceinline__ void cta_gemm_nt(float (&acc)[8][8], const float *As, int lda, const float *__restrict__ W,
                                            int K, int ncols, float *Ws /* 2 stages */) {
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int nc8 = (ncols + 31) >> 5;
    const bool aligned = ((K & 3) == 0) && ((reinterpret_cast<uintptr_t>(W) & 15) == 0);
    const int nchunks = (K + kKC - 1) / kKC;
    {
        int klen = min(kKC, K);
        stage_w_nt(Ws, W, K, 0, klen, (klen + 3) & ~3, ncols, nc8, aligned);
        cp_async_commit();
    }
    for (int ch = 0; ch < nchunks; ++ch) {
        const int k0 = ch * kKC;
        const int klen4 = (min(kKC, K - k0) + 3) & ~3;
        if (ch + 1 < nchunks) {
            int k1 = k0 + kKC, klen1 = min(kKC, K - k1);
            stage_w_nt(Ws + ((ch + 1) & 1) * kWsFloats, W, K, k1, klen1, (klen1 + 3) & ~3, ncols, nc8, aligned);
            cp_async_commit();
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
        const float *Wb = Ws + (ch & 1) * kWsFloats + tx * kWsNT;
        const float *Ab = As + (ty * 8) * lda + k0;
        for (int kk = 0; kk < klen4; kk += 4) {
            float4 a[8];
#pragma unroll
            for (int r = 0; r < 8; ++r) a[r] = *reinterpret_cast<const float4 *>(Ab + r * lda + kk);
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                if (c < nc8) {
                    const float4 b = *reinterpret_cast<const float4 *>(Wb + c * 32 * kWsNT + kk);
#pragma unroll
                    for (int r = 0; r < 8; ++r) {
                        acc[r][c] = fmaf(a[r].x, b.x, acc[r][c]);
                        acc[r][c] = fmaf(a[r].y, b.y, acc[r][c]);
                        acc[r][c] = fmaf(a[r].z, b.z, acc[r][c]);
                        acc[r][c] = fmaf(a[r].w, b.w, acc[r][c]);
                    }
                }
            }
        }
        __syncthreads();
    }
}

// Stage M[r0 + r][c0 .. c0+ncols) (global, row-major with leading dim ld) into Ms[r][0..nc8*32) for r < nrows_valid,
// zero-filling rows up to nrows_pad and columns up to nc8*32.  Used for the NN / TN operands (reduction index = row).
__device__ __forceinline__ void stage_rows(float *Ms, int lds, const float *__restrict__ M, int ld, int nrows_valid,
                                           int nrows_pad, int ncols, int ncols_pad, bool aligned) {
    const int tid = threadIdx.x;
    if (aligned) {
        const int nq = ncols_pad >> 2;
        for (int e = tid; e < nrows_pad * nq; e += kThreads) {
            int r = e / nq, q = e - r * nq;
            float *dst = Ms + r * lds + q * 4;
            if (r < nrows_valid && q * 4 + 3 < ncols) cp_async16(dst, M + (size_t)r * ld + q * 4);
            else {
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (r < nrows_valid) {
                    const float *src = M + (size_t)r * ld + q * 4;
                    if (q * 4 + 0 < ncols) v.x = src[0];
                    if (q * 4 + 1 < ncols) v.y = src[1];
                    if (q * 4 + 2 < ncols) v.z = src[2];
                    if (q * 4 + 3 < ncols) v.w = src[3];
                }
                *reinterpret_cast<float4 *>(dst) = v;
            }
        }
    } else {
        for (int e = tid; e < nrows_pad * ncols_pad; e += kThreads) {
            int r = e / ncols_pad, c = e - r * ncols_pad;
            Ms[r * lds + c] = (r < nrows_valid && c < ncols) ? M[(size_t)r * ld + c] : 0.0f;
        }
    }
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---- TSF expand (csrc/td.cu explains the mathematics) ---------------------------------------------------------------------
__host__ __device__ inline int tsf_flow_len(int S, int K) { return K * (2 * S + 1); }      // K x (weight[S] | bias | scale[S])
__host__ __device__ inline int tsf_red_len(int D, int S, int K = 0) { return D + D * S + D + tsf_flow_len(S, K); }      // [dw | T | t | flow gradients]

// TSF: (dw, T, t) partials [n_pol][nclu][2D + D*S] -> the full reduced gradient row [dw | dWg | dbg | dWh | dbh] of each
// policy (written to partial slot 0 of aux_grad_part; the Adam kernel reads it with n_part = 1).  red: [n_red] shared scratch,
// Wg_s: [G][S] | bg [G], Wh_s: [D][G] already staged in shared memory; nt threads of one CTA take part.
__device__ __forceinline__ void tsf_expand_policy(const sfgpi_td_args &a, int pl, int nclu, float *red, const float *Wg_s,
                                                  const float *Wh_s, int tid, int nt) {
    const int S = a.S, D = a.D, G = a.G, nfl = tsf_flow_len(a.S, a.n_flows);
    const int n_red = tsf_red_len(D, S, a.n_flows);
    const float *part = a.tsf_part + (size_t)pl * nclu * n_red;
    for (int e = tid; e < n_red; e += nt) {                  // fixed order k = 0, 1, ...; 8 loads in flight at a time
        float acc = 0.0f;
        int k = 0;
        for (; k + 8 <= nclu; k += 8) {
            float v[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) v[q] = part[(size_t)(k + q) * n_red + e];
#pragma unroll
            for (int q = 0; q < 8; ++q) acc += v[q];
        }
        for (; k < nclu; ++k) acc += part[(size_t)k * n_red + e];
        red[e] = acc;
    }
    __syncthreads();
    const float *T = red + D, *tv = T + D * S, *bg_s = Wg_s + G * S;
    float *out = a.aux_grad_part + (size_t)pl * nclu * a.aux_len;        // slot 0 of this policy
    float *gW = out + D, *gb = gW + G * S, *gf = gb + G, *hW = gf + nfl, *hb = hW + D * G;
    for (int d = tid; d < D; d += nt) { out[d] = red[d]; hb[d] = 2.0f * tv[d]; }
    for (int e = tid; e < nfl; e += nt) gf[e] = tv[D + e];    // the flows' gradients are complete sums already
    for (int e = tid; e < G * S; e += nt) {                  // dWg[g][s] = sum_d Wh[d][g] T[d][s]
        const int g = e / S, s = e - g * S;
        float acc = 0.0f;
        for (int d = 0; d < D; ++d) acc = fmaf(Wh_s[d * G + g], T[d * S + s], acc);
        gW[e] = acc;
    }
    for (int g = tid; g < G; g += nt) {                      // dbg[g] = 2 sum_d Wh[d][g] t[d]
        float acc = 0.0f;
        for (int d = 0; d < D; ++d) acc = fmaf(Wh_s[d * G + g], tv[d], acc);
        gb[g] = 2.0f * acc;
    }
    for (int e = tid; e < D * G; e += nt) {                  // dWh[d][g] = sum_s T[d][s] Wg[g][s] + 2 bg[g] t[d]
        const int d = e / G, g = e - d * G;
        float acc = 2.0f * bg_s[g] * tv[d];
        for (int s = 0; s < S; ++s) acc = fmaf(T[d * S + s], Wg_s[g * S + s], acc);
        hW[e] = acc;
    }
}

// whole expand of policy pl by one CTA of nt threads; sm: dynamic shared memory of >= tsf_expand_smem_floats() floats
__host__ __device__ inline int tsf_expand_smem_floats(int D, int S, int G, int K = 0) { return tsf_red_len(D, S, K) + G * S + G + D * G; }
__device__ __forceinline__ void tsf_expand_cta(const sfgpi_td_args &a, int pl, int nclu, float *sm, int tid, int nt) {
    const int S = a.S, D = a.D, G = a.G;
    float *red = sm;                              // [dw | T | t]
    float *Wg_s = red + tsf_red_len(D, S, a.n_flows);   // [G][S] | bg [G]
    float *Wh_s = Wg_s + G * S + G;               // [D][G]
    const float *gp = a.g + (size_t)pl * a.g_stride;
    for (int e = tid; e < G * S + G; e += nt) Wg_s[e] = gp[e];
    for (int e = tid; e < D * G; e += nt) Wh_s[e] = a.h[e];
    tsf_expand_policy(a, pl, nclu, red, Wg_s, Wh_s, tid, nt);
}

}  // namespace sfgpi
