// Input gradient of the psi MLP: dx[b][s] = sum_p sum_k dZ0[p][b][k] * W0_p[k][s]  (include/sfgpi.h, sfgpi_mlp_input_grad).
//
// dZ0 is the layer-0 pre-activation gradient every backward entry point already leaves in its scratch (the W_0 weight gradient
// needs it), so the state gradient is one reduction over the policies and the hidden width: K = dims[1] (256 in the tensor-core
// modes), N = S <= 63: a small FFMA reduction on the CUDA cores, not tensor-core work.
//
// One CTA = 32 batch rows x up to SC output columns, 8 warps: lane = row, warp w owns the k slice [32w, 32w + 32) of each
// 256-wide reduction chunk.  Per (policy, chunk) the CTA stages the dZ0 tile [32 rows][256] in its native type (the rows of one
// policy are contiguous: coalesced 16-byte cp.async) and W0[chunk][SC] rounded as the mode's forward rounded it, in a ring of
// up to 4 stages so the next tiles load while this one is reduced.  Every thread keeps SC fp32 accumulators over all policies
// and chunks in a fixed order; the 8 warps' partial sums are added in warp order at the end.  No atomics: two runs give the
// same bits.
#include "stream_tc.cuh"

namespace sfgpi {
namespace ig {

constexpr int kIgRows = 32;               // batch rows per CTA (lane = row)
constexpr int kIgKC = 256;                // reduction chunk per stage; warp w reduces [32w, 32w + 32) of it
constexpr int kIgLd = kIgKC + 4;          // fp32 tile row stride: lanes 260 words apart -> conflict-free LDS.128
constexpr int kIgLd16 = kIgKC + 8;        // bf16 tile row stride: lanes 132 words apart -> conflict-free LDS.128
enum { kDzF32 = 0, kDzF32x2 = 1, kDzBf16 = 2 };      // dZ0 element: fp32, fp32 hi + lo (tf32x3), bf16
enum { kRoundNone = 0, kRoundBf16 = 1, kRoundTf32 = 2 };

template <int kKind>
__host__ __device__ constexpr int tile_bytes() {
    return kKind == kDzBf16 ? kIgRows * kIgLd16 * 2 : (kKind == kDzF32x2 ? 2 : 1) * kIgRows * kIgLd * 4;
}
template <int kKind, int SC>
__host__ __device__ constexpr int stage_bytes() { return tile_bytes<kKind>() + kIgKC * SC * 4; }
// Ring depth: up to 4 stages (3 in flight while one is reduced) within the shared memory of an SM.  A stage costs a CTA a memory
// round trip and little arithmetic, so loading the policies one after another would serialise those round trips.
template <int kKind, int SC>
__host__ __device__ constexpr int ig_stages() {
    return 4 * stage_bytes<kKind, SC>() <= kMaxSmem ? 4 : (3 * stage_bytes<kKind, SC>() <= kMaxSmem ? 3 : 2);
}
template <int kKind, int SC>
__host__ __device__ constexpr int ig_smem_bytes() {
    return ig_stages<kKind, SC>() * stage_bytes<kKind, SC>() > 8 * 32 * (SC + 4) * 4 ? ig_stages<kKind, SC>() * stage_bytes<kKind, SC>()
                                                                                    : 8 * 32 * (SC + 4) * 4;
}

// columns of the chunk at k0 that are staged: whole 32-wide warp slices (the slice holding K's end is zero-padded)
__device__ __forceinline__ int chunk_width(int K, int k0) { return min(kIgKC, (K - k0 + 31) & ~31); }

__device__ __forceinline__ void cp_async4(void *smem, const void *gmem) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(s), "l"(gmem));
}

// Stage policy p's dZ0 rows [row0, row0 + 32) x columns [k0, k0 + kw) and W0_p[k0 .. k0 + kw)[s0 .. s0 + SC) into one stage:
// out-of-range elements are stored as zeros, W0 raw (rounded by round_w once the copies have landed).
template <int kKind, int SC>
__device__ __forceinline__ void issue_stage(unsigned char *st, const sfgpi_input_grad_args &a, int p, int k0, int row0, int s0,
                                            bool vec) {
    const int tid = threadIdx.x, S = a.net.dims[0], K = a.net.dims[1], B = a.B, kw = chunk_width(K, k0);
    const float *W = a.params + (size_t)(a.policy_lo + p) * a.net.row_stride + a.net.w_off[0];
    float *Ws = reinterpret_cast<float *>(st + tile_bytes<kKind>());
    for (int e = tid; e < kw * SC; e += kThreads) {
        const int kk = e / SC, c = e - kk * SC;
        if (k0 + kk < K && s0 + c < S) cp_async4(Ws + e, W + (size_t)(k0 + kk) * S + s0 + c);
        else Ws[e] = 0.0f;
    }
    constexpr int kVec = kKind == kDzBf16 ? 8 : 4;            // elements per 16-byte copy
    const int kPerRow = kw / kVec;
    for (int g = tid; g < kIgRows * kPerRow; g += kThreads) {
        const int r = g / kPerRow, kk = (g - r * kPerRow) * kVec, row = row0 + r, k = k0 + kk;
        const size_t off = ((size_t)p * B + row) * K + k;
        if constexpr (kKind == kDzBf16) {                     // K == 256: whole 16-byte groups
            __nv_bfloat16 *dst = reinterpret_cast<__nv_bfloat16 *>(st) + r * kIgLd16 + kk;
            if (row < B) cp_async16(dst, reinterpret_cast<const __nv_bfloat16 *>(a.dz0) + off);
            else *reinterpret_cast<uint4 *>(dst) = make_uint4(0u, 0u, 0u, 0u);
        } else {
            const float *src = reinterpret_cast<const float *>(a.dz0) + off;
#pragma unroll
            for (int part = 0; part < (kKind == kDzF32x2 ? 2 : 1); ++part) {
                float *dst = reinterpret_cast<float *>(st) + part * kIgRows * kIgLd + r * kIgLd + kk;
                const float *s = src + part * a.dz0_part_stride;
                if (vec && row < B && k < K) {
                    cp_async16(dst, s);
                } else {                                      // ragged hidden width (fp32 mode): element by element
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        if (row < B && k + j < K) cp_async4(dst + j, s + j);
                        else dst[j] = 0.0f;
                    }
                }
            }
        }
    }
}

// W0 as the mode's forward multiplied it: the bf16 shadow's value (sfgpi_pack_bf16) or the tf32 one (sfgpi_pack_f32, hi part).
// Each thread rounds the elements it copied itself, so its own cp.async wait is enough before the CTA barrier.
template <int kKind, int SC>
__device__ __forceinline__ void round_w(unsigned char *st, int kw, int rounding) {
    if (rounding == kRoundNone) return;
    float *Ws = reinterpret_cast<float *>(st + tile_bytes<kKind>());
    for (int e = threadIdx.x; e < kw * SC; e += kThreads)
        Ws[e] = rounding == kRoundBf16 ? __bfloat162float(__float2bfloat16_rn(Ws[e])) : tc::tf32_rna(Ws[e]);
}

template <int SC>
__device__ __forceinline__ void fma_row(float (&acc)[SC], float v, const float *wrow) {
#pragma unroll
    for (int c = 0; c < SC; c += 4) {
        const float4 w = *reinterpret_cast<const float4 *>(wrow + c);       // warp-uniform address: broadcast
        acc[c] = fmaf(v, w.x, acc[c]);
        acc[c + 1] = fmaf(v, w.y, acc[c + 1]);
        acc[c + 2] = fmaf(v, w.z, acc[c + 2]);
        acc[c + 3] = fmaf(v, w.w, acc[c + 3]);
    }
}

template <int kKind, int SC>
__global__ void __launch_bounds__(kThreads, 1) mlp_input_grad_kernel(const __grid_constant__ sfgpi_input_grad_args a, int rounding,
                                                                     int vec) {
    extern __shared__ __align__(16) unsigned char smem_ig[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int S = a.net.dims[0], K = a.net.dims[1];
    const int row0 = blockIdx.x * kIgRows, s0 = blockIdx.y * SC;
    const int n_kc = (K + kIgKC - 1) / kIgKC, n_it = a.n_pol * n_kc;
    pdl_launch_dependents();
    pdl_wait();

    float acc[SC];
#pragma unroll
    for (int c = 0; c < SC; ++c) acc[c] = 0.0f;

    // ring of NS stages: iteration `it` reduces stage it % NS while stages it+1 .. it+NS-1 load.  One commit group per
    // iteration (empty past the end), so waiting for all but the NS-1 newest groups always means "stage it has landed".
    constexpr int NS = ig_stages<kKind, SC>();
    for (int j = 0; j < NS - 1; ++j) {
        if (j < n_it) issue_stage<kKind, SC>(smem_ig + j * stage_bytes<kKind, SC>(), a, j / n_kc, (j % n_kc) * kIgKC, row0, s0, vec);
        cp_async_commit();
    }
    for (int it = 0; it < n_it; ++it) {
        unsigned char *st = smem_ig + (it % NS) * stage_bytes<kKind, SC>();
        const int nx = it + NS - 1;
        if (nx < n_it)
            issue_stage<kKind, SC>(smem_ig + (nx % NS) * stage_bytes<kKind, SC>(), a, nx / n_kc, (nx % n_kc) * kIgKC, row0, s0, vec);
        cp_async_commit();
        cp_async_wait<NS - 1>();
        round_w<kKind, SC>(st, chunk_width(K, (it % n_kc) * kIgKC), rounding);
        __syncthreads();
        const int kb = warp * 32;
        if ((it % n_kc) * kIgKC + kb < K) {                   // warp-uniform: slices past a narrow hidden width hold zeros only
            const float *Ws = reinterpret_cast<const float *>(st + tile_bytes<kKind>()) + kb * SC;
            if constexpr (kKind == kDzBf16) {
                const __nv_bfloat16 *t = reinterpret_cast<const __nv_bfloat16 *>(st) + lane * kIgLd16 + kb;
#pragma unroll
                for (int kk = 0; kk < 32; kk += 8) {
                    const uint4 u = *reinterpret_cast<const uint4 *>(t + kk);
                    const uint32_t w4[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        fma_row<SC>(acc, __uint_as_float(w4[j] << 16), Ws + (kk + 2 * j) * SC);
                        fma_row<SC>(acc, __uint_as_float(w4[j] & 0xFFFF0000u), Ws + (kk + 2 * j + 1) * SC);
                    }
                }
            } else {
                const float *t = reinterpret_cast<const float *>(st) + lane * kIgLd + kb;
#pragma unroll
                for (int kk = 0; kk < 32; kk += 4) {
                    float4 v = *reinterpret_cast<const float4 *>(t + kk);
                    if constexpr (kKind == kDzF32x2) {        // dZ0 = hi + lo
                        const float4 lo = *reinterpret_cast<const float4 *>(t + kIgRows * kIgLd + kk);
                        v.x += lo.x; v.y += lo.y; v.z += lo.z; v.w += lo.w;
                    }
                    fma_row<SC>(acc, v.x, Ws + kk * SC);
                    fma_row<SC>(acc, v.y, Ws + (kk + 1) * SC);
                    fma_row<SC>(acc, v.z, Ws + (kk + 2) * SC);
                    fma_row<SC>(acc, v.w, Ws + (kk + 3) * SC);
                }
            }
        }
        __syncthreads();
    }

    // the 8 k slices' partial sums, added in warp order
    float *red = reinterpret_cast<float *>(smem_ig);           // [warp][lane][SC + 4]
#pragma unroll
    for (int c = 0; c < SC; c += 4)
        *reinterpret_cast<float4 *>(red + (warp * 32 + lane) * (SC + 4) + c) = make_float4(acc[c], acc[c + 1], acc[c + 2], acc[c + 3]);
    __syncthreads();
    for (int e = tid; e < kIgRows * SC; e += kThreads) {
        const int r = e / SC, c = e - r * SC, row = row0 + r, s = s0 + c;
        float v = 0.0f;
#pragma unroll
        for (int w = 0; w < 8; ++w) v += red[(w * 32 + r) * (SC + 4) + c];
        if (row < a.B && s < S) a.dx[(size_t)row * S + s] = v;
    }
}

template <int kKind, int SC>
static int launch_input_grad(const sfgpi_input_grad_args &a, int rounding, int vec, cudaStream_t st) {
    constexpr int smem = ig_smem_bytes<kKind, SC>();
    static_assert(smem <= kMaxSmem, "input-gradient stage does not fit in shared memory");
    static bool cfg = false;
    if (!cfg) {
        cudaFuncSetAttribute(mlp_input_grad_kernel<kKind, SC>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        cfg = true;
    }
    const int S = a.net.dims[0];
    dim3 grid((a.B + kIgRows - 1) / kIgRows, (S + SC - 1) / SC);
    launch_pdl(mlp_input_grad_kernel<kKind, SC>, grid, dim3(kThreads), smem, st, a, rounding, vec);
    return check_launch("sfgpi_mlp_input_grad");
}

template <int kKind>
static int launch_input_grad_sc(const sfgpi_input_grad_args &a, int rounding, int vec, cudaStream_t st) {
    // the broadcast reads of W0 from shared memory bound the reduction (about 4 cycles per 4 columns and k per warp, measured),
    // so the column block follows S closely: padding columns cost as much as real ones
    const int S = a.net.dims[0];
    if (S <= 4) return launch_input_grad<kKind, 4>(a, rounding, vec, st);
    if (S <= 8) return launch_input_grad<kKind, 8>(a, rounding, vec, st);
    if (S <= 12) return launch_input_grad<kKind, 12>(a, rounding, vec, st);
    if (S <= 16) return launch_input_grad<kKind, 16>(a, rounding, vec, st);
    if constexpr (kKind == kDzF32x2) return launch_input_grad<kKind, 32>(a, rounding, vec, st);      // tf32x3: S <= 31
    else {
        if (S <= 32) return launch_input_grad<kKind, 32>(a, rounding, vec, st);
        return launch_input_grad<kKind, 64>(a, rounding, vec, st);        // wider fp32 states: grid.y covers 64 columns each
    }
}

}  // namespace ig
}  // namespace sfgpi

using namespace sfgpi;
using namespace sfgpi::ig;

extern "C" int sfgpi_mlp_input_grad(const sfgpi_input_grad_args *args, void *stream) {
    if (!args) { set_error("sfgpi_mlp_input_grad: args is NULL"); return SFGPI_E_INVALID; }
    const sfgpi_input_grad_args &a = *args;
    const sfgpi_net_desc &net = a.net;
    if (a.precision < SFGPI_PREC_FP32 || a.precision > SFGPI_PREC_TF32X3) {
        set_error("sfgpi_mlp_input_grad: unknown precision %d", a.precision);
        return SFGPI_E_INVALID;
    }
    if (net.n_layers < 2 || net.n_layers > SFGPI_MAX_LAYERS) {
        set_error("sfgpi_mlp_input_grad: needs 2..%d Linear layers (dZ_0 is the first hidden layer's gradient)", SFGPI_MAX_LAYERS);
        return SFGPI_E_INVALID;
    }
    if (a.B < 0 || a.n_pol < 0 || a.policy_lo < 0 || a.dz0_part_stride < 0 || net.dims[0] < 1 || net.dims[1] < 1) {
        set_error("sfgpi_mlp_input_grad: negative or empty sizes");
        return SFGPI_E_INVALID;
    }
    if (net.w_off[0] < 0 || (int64_t)net.w_off[0] + (int64_t)net.dims[1] * net.dims[0] > net.row_stride) {
        set_error("sfgpi_mlp_input_grad: W_0 [%d][%d] at offset %d does not fit a row of %d floats", net.dims[1], net.dims[0],
                  net.w_off[0], net.row_stride);
        return SFGPI_E_INVALID;
    }
    if (!a.params || !a.dz0 || !a.dx) { set_error("sfgpi_mlp_input_grad: params, dz0 and dx must not be NULL"); return SFGPI_E_INVALID; }
    const int S = net.dims[0];
    if (a.precision != SFGPI_PREC_FP32) {
        const int s_max = a.precision == SFGPI_PREC_BF16 ? 63 : 31;
        if (net.dims[1] != 256) {
            set_error("sfgpi_mlp_input_grad: the tensor-core modes need a first hidden width of 256, got %d", net.dims[1]);
            return SFGPI_E_INVALID;
        }
        if (S > s_max) {
            set_error("sfgpi_mlp_input_grad: S = %d exceeds the %s limit of %d", S, a.precision == SFGPI_PREC_BF16 ? "bf16" : "tf32", s_max);
            return SFGPI_E_INVALID;
        }
    }
    if (a.precision == SFGPI_PREC_TF32X3 && a.dz0_part_stride < (int64_t)a.n_pol * a.B * 256) {
        set_error("sfgpi_mlp_input_grad: dz0_part_stride %lld overlaps the hi part [n_pol][B][256]", (long long)a.dz0_part_stride);
        return SFGPI_E_INVALID;
    }
    if (a.B == 0 || a.n_pol == 0) return SFGPI_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const int K = net.dims[1];
    const int vec = (K % 4 == 0) && (reinterpret_cast<uintptr_t>(a.dz0) % 16 == 0) && (a.dz0_part_stride % 4 == 0);
    switch (a.precision) {
    case SFGPI_PREC_BF16: return launch_input_grad_sc<kDzBf16>(a, kRoundBf16, 1, st);
    case SFGPI_PREC_TF32: return launch_input_grad_sc<kDzF32>(a, kRoundTf32, vec, st);
    case SFGPI_PREC_TF32X3: return launch_input_grad_sc<kDzF32x2>(a, kRoundNone, vec, st);
    default: return launch_input_grad_sc<kDzF32>(a, kRoundNone, vec, st);
    }
}
