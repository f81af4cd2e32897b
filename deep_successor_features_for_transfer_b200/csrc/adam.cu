// Fused multi-tensor Adam for n_pol optimizers in ONE launch (replaces torch.optim.Adam's 9-13 per-tensor loops,
// sfdqn.py:282-286 / tsfdqn.py:255-270 + 700).  Arithmetic order follows torch/optim/adam.py::_single_tensor_adam:
//   g += wd*p ; m = lerp(m, g, 1-b1) ; v = b2*v + (1-b2)*g*g ; denom = sqrt(v)/sqrt(1-b2^t) + eps ; p -= (lr/(1-b1^t)) * m/denom
// Gradients arrive as split partials (wgrad split-K, TD per-CTA partials) and are summed here in a fixed order, so the
// whole step is deterministic.  HBM-bound: 16 B read + 12 B written per parameter (+ 4 B * n_part of partials).
#include "common.cuh"

namespace sfgpi {

constexpr int kAdamThreads = 256;

struct AdamConsts { float b2, one_m_b1, one_m_b2, eps; };

__device__ __forceinline__ void adam_elem(float &p, float &m, float &v, float g, float step_size, float sqrt_bc2, float wd,
                                          const AdamConsts &k) {
    // every multiply-add is explicit, so each inlined copy rounds alike: left to the compiler, the v update was contracted
    // differently in the 128-bit and the scalar copy
    if (wd != 0.0f) g = fmaf(wd, p, g);
    m = fmaf(k.one_m_b1, g - m, m);                        // lerp_, weight < 0.5 branch
    v = fmaf(v, k.b2, __fmul_rn(__fmul_rn(k.one_m_b2, g), g));     // mul_ then addcmul_
    const float denom = __fdiv_rn(sqrtf(v), sqrt_bc2) + k.eps;
    p = p - __fdiv_rn(step_size * m, denom);               // addcdiv_(value = -step_size): self + value*t1/t2
}

// bias corrections of optimizer q for this step: {1 - beta1^t, sqrt(1 - beta2^t)} in double, as torch computes them on the
// host.  Read from a.consts, which the previous launch wrote (as its consts_next), so no double-precision pow sits on the
// critical path of the step.
__device__ __forceinline__ void bias_corrections(const sfgpi_adam_args &a, int q, double &bc1, float &sqrt_bc2) {
    if (a.fresh) {                                           // first step of a brand-new optimizer: t = 1
        bc1 = 1.0 - a.beta1;
        sqrt_bc2 = (float)sqrt(1.0 - a.beta2);
    } else {
        bc1 = a.consts[2 * q];
        sqrt_bc2 = (float)a.consts[2 * q + 1];
    }
}

// fixed-order sum of n_part gradient partials, `stride` floats apart; four independent chains keep the loads in flight
__device__ __forceinline__ float sum_partials(const float *__restrict__ gp, int n_part, size_t stride) {
    float g0 = 0.0f, g1 = 0.0f, g2 = 0.0f, g3 = 0.0f;
    int k = 0;
    for (; k + 4 <= n_part; k += 4) {
        const float t0 = __ldg(gp + (size_t)k * stride), t1 = __ldg(gp + (size_t)(k + 1) * stride),
                    t2 = __ldg(gp + (size_t)(k + 2) * stride), t3 = __ldg(gp + (size_t)(k + 3) * stride);
        g0 += t0; g1 += t1; g2 += t2; g3 += t3;
    }
    for (; k < n_part; ++k) g0 += __ldg(gp + (size_t)k * stride);
    return (g0 + g1) + (g2 + g3);
}

__device__ __forceinline__ float4 sum_partials4(const float4 *__restrict__ gp, int n_part, size_t stride4) {
    float4 g0 = make_float4(0.f, 0.f, 0.f, 0.f), g1 = g0, g2 = g0, g3 = g0;
    int k = 0;
    for (; k + 4 <= n_part; k += 4) {
        const float4 t0 = __ldg(gp + (size_t)k * stride4), t1 = __ldg(gp + (size_t)(k + 1) * stride4),
                     t2 = __ldg(gp + (size_t)(k + 2) * stride4), t3 = __ldg(gp + (size_t)(k + 3) * stride4);
        g0.x += t0.x; g0.y += t0.y; g0.z += t0.z; g0.w += t0.w;
        g1.x += t1.x; g1.y += t1.y; g1.z += t1.z; g1.w += t1.w;
        g2.x += t2.x; g2.y += t2.y; g2.z += t2.z; g2.w += t2.w;
        g3.x += t3.x; g3.y += t3.y; g3.z += t3.z; g3.w += t3.w;
    }
    for (; k < n_part; ++k) {
        const float4 t = __ldg(gp + (size_t)k * stride4);
        g0.x += t.x; g0.y += t.y; g0.z += t.z; g0.w += t.w;
    }
    return make_float4((g0.x + g1.x) + (g2.x + g3.x), (g0.y + g1.y) + (g2.y + g3.y), (g0.z + g1.z) + (g2.z + g3.z),
                       (g0.w + g1.w) + (g2.w + g3.w));
}

// N consecutive floats (N = 4: one 128-bit access) <-> registers
template <int N> __device__ __forceinline__ void load_n(float (&r)[N], const float *src) {
    if constexpr (N == 4) {
        const float4 t = *reinterpret_cast<const float4 *>(src);
        r[0] = t.x; r[1] = t.y; r[2] = t.z; r[3] = t.w;
    } else {
        r[0] = *src;
    }
}
template <int N> __device__ __forceinline__ void store_n(float *dst, const float (&r)[N]) {
    if constexpr (N == 4) *reinterpret_cast<float4 *>(dst) = make_float4(r[0], r[1], r[2], r[3]);
    else *dst = r[0];
}

// item i of a per-optimizer segment: parameters [N*i, N*i + N) of optimizer p.  Every load (bias corrections, p, m, v,
// partials) is issued before the first use and the step size (a double division, as on the host) is computed while they are
// in flight.  Per element the arithmetic is the same for N = 4 and N = 1, so the kind of range does not change a bit.
template <int N>
__device__ __forceinline__ void adam_item(const sfgpi_adam_args &a, const sfgpi_adam_segment &sg, int p, int i, const AdamConsts &kc) {
    double bc1;
    float sqrt_bc2;
    bias_corrections(a, p, bc1, sqrt_bc2);
    const size_t e0 = (size_t)i * N;
    const float *gp = sg.grad_part + (size_t)p * sg.grad_pol_stride + e0;
    float *pp = sg.param + (size_t)p * sg.param_stride + e0;
    float *pm = a.fresh ? nullptr : sg.m + (size_t)p * sg.m_stride + e0;       // fresh: moments start at 0 and are not stored
    float *pv = a.fresh ? nullptr : sg.v + (size_t)p * sg.v_stride + e0;
    float w[N], m[N] = {}, v[N] = {}, g[N];
    load_n(w, pp);
    if (!a.fresh) { load_n(m, pm); load_n(v, pv); }
    if constexpr (N == 4) {
        const float4 g4 = sum_partials4(reinterpret_cast<const float4 *>(gp), sg.n_part, (size_t)(sg.grad_part_stride >> 2));
        g[0] = g4.x; g[1] = g4.y; g[2] = g4.z; g[3] = g4.w;
    } else {
        g[0] = sum_partials(gp, sg.n_part, (size_t)sg.grad_part_stride);
    }
    const float step_size = (float)((double)sg.lr / bc1);
#pragma unroll
    for (int e = 0; e < N; ++e) adam_elem(w[e], m[e], v[e], g[e], step_size, sqrt_bc2, sg.weight_decay, kc);
    if (sg.clamp_min < sg.clamp_max) {                       // (the G4 loss coefficient)
#pragma unroll
        for (int e = 0; e < N; ++e) w[e] = fminf(fmaxf(w[e], sg.clamp_min), sg.clamp_max);
    }
    store_n(pp, w);
    if (!a.fresh) { store_n(pm, m); store_n(pv, v); }
}

// Block layout of one launch, per grid row (= optimizer): every per-optimizer segment owns a block range, 128-bit (4
// parameters per thread) or scalar (1 per thread) as its lengths, strides and pointers allow; then the blocks that step the
// shared segments; then one last block.  A segment-by-segment loop behind a one-thread prologue was a chain of 5-6 dependent
// memory round trips (17.0 -> 8.6 us, DESIGN.md).
struct AdamGrid {
    int blk_end[SFGPI_MAX_SEGMENTS];   // exclusive prefix ends of the per-optimizer segments' block ranges (shared segments: empty)
    int vec_mask;                      // bit s: segment s's range is 128-bit
    int n_own;                         // blocks of per-optimizer segments
    int n_shared;                      // blocks (per grid row) that step the shared segments, warp per element
};

// At most 64 registers (4 blocks per SM): with more freedom ptxas spills more, not less, around the slow-path calls of the
// correctly rounded divisions.
__global__ void __launch_bounds__(kAdamThreads, 4) adam_step_kernel(const __grid_constant__ sfgpi_adam_args a, const __grid_constant__ AdamGrid f) {
    pdl_launch_dependents(SFGPI_TR_ADAM);
    pdl_wait(SFGPI_TR_ADAM);
    const int p = blockIdx.y;                               // optimizer (policy slot)
    const int bid = blockIdx.x;
    const AdamConsts kc = {(float)a.beta2, (float)(1.0 - a.beta1), (float)(1.0 - a.beta2), (float)a.eps};
    if (bid < f.n_own) {
        int s = 0;
        while (bid >= f.blk_end[s]) ++s;
        const sfgpi_adam_segment &sg = a.seg[s];
        const int i = (bid - (s ? f.blk_end[s - 1] : 0)) * kAdamThreads + threadIdx.x;
        if ((f.vec_mask >> s) & 1) {
            if (i < (sg.len >> 2)) adam_item<4>(a, sg, p, i, kc);
        } else if (i < sg.len) {
            adam_item<1>(a, sg, p, i, kc);
        }
    } else if (bid < f.n_own + f.n_shared) {
        // shared tensors (TSF's h): every optimizer steps them from the SAME pre-step value, each with its own moments and
        // bias corrections (frozen-snapshot ensemble semantics, DESIGN.md); one warp per element, lane = optimizer, deltas
        // summed by a fixed butterfly
        const int lane = threadIdx.x & 31;
        const int warps_total = f.n_shared * gridDim.y * (kAdamThreads / 32);
        const int wg = (blockIdx.y * f.n_shared + (bid - f.n_own)) * (kAdamThreads / 32) + (threadIdx.x >> 5);
        for (int s = 0; s < a.n_seg; ++s) {
            const sfgpi_adam_segment &sg = a.seg[s];
            if (!(sg.param_stride == 0 && a.n_pol > 1)) continue;
            for (int i = wg; i < sg.len; i += warps_total) {
                const float p0 = sg.param[i];
                float dsum = 0.0f;
                for (int q0 = 0; q0 < a.n_pol; q0 += 32) {
                    const int q = q0 + lane;
                    float delta = 0.0f;
                    if (q < a.n_pol) {
                        double qbc1;
                        float qsb2;
                        bias_corrections(a, q, qbc1, qsb2);
                        float *pm = sg.m + (size_t)q * sg.m_stride + i;
                        float *pv = sg.v + (size_t)q * sg.v_stride + i;
                        float pw = p0, m = *pm, v = *pv;
                        const float g = sum_partials(sg.grad_part + (size_t)q * sg.grad_pol_stride + i, sg.n_part, (size_t)sg.grad_part_stride);
                        adam_elem(pw, m, v, g, (float)((double)sg.lr / qbc1), qsb2, sg.weight_decay, kc);
                        *pm = m; *pv = v;
                        delta = pw - p0;
                    }
                    dsum += warp_sum(delta);
                }
                __syncwarp();
                if (lane == 0) sg.param[i] = p0 + dsum;
            }
        }
    } else {
        // the last block of every grid row: the losses (fixed-order sum of the TD kernel's per-CTA partials) and the step
        // counter / next step's bias corrections (consts_next: nothing in this launch reads it or `step`)
        if (a.loss_part != nullptr && threadIdx.x < 32) {
            float s1 = 0.0f, s2 = 0.0f;
            const float *lp = a.loss_part + (size_t)p * a.n_loss_part * 2;
            for (int i = threadIdx.x; i < a.n_loss_part; i += 32) { s1 += lp[2 * i]; s2 += lp[2 * i + 1]; }
            s1 = warp_sum(s1); s2 = warp_sum(s2);
            if (threadIdx.x == 0) {
                const float l1 = s1 * a.l1_scale, l2 = s2 * a.l2_scale;
                a.losses[p * 3 + 0] = l1 + a.beta_loss * l2;
                a.losses[p * 3 + 1] = l1;
                a.losses[p * 3 + 2] = l2;
                if (a.losses_host != nullptr) {              // the step's result, straight into pinned host memory
                    a.losses_host[p * 3 + 0] = l1 + a.beta_loss * l2;
                    a.losses_host[p * 3 + 1] = l1;
                    a.losses_host[p * 3 + 2] = l2;
                }
            }
        }
        if (!a.fresh && threadIdx.x == 32) {
            const int s_new = a.step[p] + 1;
            a.step[p] = s_new;
            const double t = (double)(s_new + 1);
            a.consts_next[2 * p] = 1.0 - pow(a.beta1, t);
            a.consts_next[2 * p + 1] = sqrt(1.0 - pow(a.beta2, t));
        }
    }
    trace_exit(SFGPI_TR_ADAM);
}

__global__ void adam_refresh_kernel(const int32_t *step, double *ca, double *cb, int n, double beta1, double beta2) {
    pdl_launch_dependents();
    pdl_wait();
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const double t = (double)(step[i] + 1);
        const double c0 = 1.0 - pow(beta1, t), c1 = sqrt(1.0 - pow(beta2, t));
        ca[2 * i] = c0; ca[2 * i + 1] = c1;
        cb[2 * i] = c0; cb[2 * i + 1] = c1;
    }
}

}  // namespace sfgpi

using namespace sfgpi;

extern "C" int sfgpi_adam_step(const sfgpi_adam_args *args, void *stream) {
    sfgpi_adam_args a = *args;
    if (a.n_seg < 1 || a.n_seg > SFGPI_MAX_SEGMENTS || a.n_pol < 1) { set_error("sfgpi_adam_step: invalid arguments"); return SFGPI_E_INVALID; }
    if (!a.fresh) {
        const char *missing = !a.step ? "step" : !a.consts ? "consts" : !a.consts_next ? "consts_next" : nullptr;
        if (missing) { set_error("sfgpi_adam_step: a non-fresh step needs %s", missing); return SFGPI_E_INVALID; }
        if (a.consts_next == a.consts) { set_error("sfgpi_adam_step: consts_next must be a buffer distinct from consts"); return SFGPI_E_INVALID; }
    }
    AdamGrid f = {};
    int nb = 0, shared_len = 0;
    for (int s = 0; s < a.n_seg; ++s) {
        const sfgpi_adam_segment &sg = a.seg[s];
        if (sg.len < 0 || sg.n_part < 1) { set_error("sfgpi_adam_step: bad segment %d", s); return SFGPI_E_INVALID; }
        if (sg.param_stride == 0 && a.n_pol > 1) {
            if (a.fresh) { set_error("sfgpi_adam_step: fresh optimizers cannot share a tensor"); return SFGPI_E_INVALID; }
            shared_len = sg.len > shared_len ? sg.len : shared_len;
        } else {
            const bool vec = ((sg.len | sg.grad_part_stride | sg.grad_pol_stride | sg.param_stride | sg.m_stride | sg.v_stride) & 3) == 0 &&
                             ((reinterpret_cast<uintptr_t>(sg.grad_part) | reinterpret_cast<uintptr_t>(sg.param) |
                               reinterpret_cast<uintptr_t>(sg.m) | reinterpret_cast<uintptr_t>(sg.v)) & 15) == 0;
            const int items = vec ? sg.len >> 2 : sg.len;
            f.vec_mask |= (int)vec << s;
            nb += items / kAdamThreads + (items % kAdamThreads != 0);
        }
        f.blk_end[s] = nb;
    }
    for (int s = a.n_seg; s < SFGPI_MAX_SEGMENTS; ++s) f.blk_end[s] = nb;
    f.n_own = nb;
    const int warps = (shared_len + a.n_pol - 1) / a.n_pol;                  // warps per grid row: one element each
    f.n_shared = shared_len > 0 ? (warps + kAdamThreads / 32 - 1) / (kAdamThreads / 32) : 0;
    if (f.n_shared > 296) f.n_shared = 296;
    if (a.losses_host != nullptr) {                          // the kernel needs the device-visible address of the pinned buffer
        cudaPointerAttributes at;
        if (a.loss_part == nullptr || cudaPointerGetAttributes(&at, a.losses_host) != cudaSuccess || at.type != cudaMemoryTypeHost ||
            !at.devicePointer) {
            cudaGetLastError();
            set_error("sfgpi_adam_step: losses_host must be pinned host memory (and needs loss_part)");
            return SFGPI_E_INVALID;
        }
        a.losses_host = reinterpret_cast<float *>(at.devicePointer);
    }
    trace_bind();
    launch_pdl(adam_step_kernel, dim3(f.n_own + f.n_shared + 1, a.n_pol), dim3(kAdamThreads), 0, (cudaStream_t)stream, a, f);
    return check_launch("sfgpi_adam_step");
}

extern "C" int sfgpi_adam_refresh(const int32_t *step, double *consts_a, double *consts_b, int32_t n, double beta1, double beta2, void *stream) {
    if (n < 0 || !step || !consts_a || !consts_b) { set_error("sfgpi_adam_refresh: invalid arguments"); return SFGPI_E_INVALID; }
    if (n == 0) return SFGPI_OK;
    launch_pdl(adam_refresh_kernel, dim3((n + 127) / 128), dim3(128), 0, (cudaStream_t)stream, step, consts_a, consts_b, (int)n, beta1, beta2);
    return check_launch("sfgpi_adam_refresh");
}
