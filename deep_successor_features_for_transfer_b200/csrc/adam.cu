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
    if (wd != 0.0f) g = fmaf(wd, p, g);
    m = m + k.one_m_b1 * (g - m);                          // lerp_, weight < 0.5 branch
    v = v * k.b2 + k.one_m_b2 * g * g;                     // mul_ then addcmul_
    const float denom = __fdiv_rn(sqrtf(v), sqrt_bc2) + k.eps;
    p = p - __fdiv_rn(step_size * m, denom);               // addcdiv_(value = -step_size): self + value*t1/t2
}

// bias corrections of optimizer q for its NEXT step: {1 - beta1^t, sqrt(1 - beta2^t)} in double, as torch computes them on
// the host.  Read from a.consts when the caller maintains it (adam_finish_kernel refreshes it after every step, so no
// double-precision pow sits on the critical path of the step), else computed here.
__device__ __forceinline__ void bias_corrections(const sfgpi_adam_args &a, int q, double &bc1, float &sqrt_bc2) {
    if (a.fresh) {                                           // first step of a brand-new optimizer: t = 1
        bc1 = 1.0 - a.beta1;
        sqrt_bc2 = (float)sqrt(1.0 - a.beta2);
    } else if (a.consts != nullptr) {
        bc1 = a.consts[2 * q];
        sqrt_bc2 = (float)a.consts[2 * q + 1];
    } else {
        const double t = (double)(a.step[q] + 1);
        bc1 = 1.0 - pow(a.beta1, t);
        sqrt_bc2 = (float)sqrt(1.0 - pow(a.beta2, t));
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

// step += 1 and, when the caller keeps them, the bias corrections of the step after that
__device__ __forceinline__ void adam_finish_one(int32_t *step, double *consts, int i, double beta1, double beta2) {
    const int s = step[i] + 1;
    step[i] = s;
    if (consts != nullptr) {
        const double t = (double)(s + 1);
        consts[2 * i] = 1.0 - pow(beta1, t);
        consts[2 * i + 1] = sqrt(1.0 - pow(beta2, t));
    }
}

__global__ void __launch_bounds__(kAdamThreads) adam_kernel(const __grid_constant__ sfgpi_adam_args a, int blocks_per_pol) {
    __shared__ float sqrt_bc2_s, step_size_s[SFGPI_MAX_SEGMENTS];
    pdl_launch_dependents(SFGPI_TR_ADAM);
    pdl_wait(SFGPI_TR_ADAM);
    const int p = blockIdx.y;                               // optimizer (policy slot)
    // ---- losses (block 0 of each optimizer): fixed-order sum of the TD kernel's per-CTA partials ----
    if (blockIdx.x == 0 && a.loss_part != nullptr && threadIdx.x < 32) {
        float s1 = 0.0f, s2 = 0.0f;
        const float *lp = a.loss_part + (size_t)p * a.n_loss_part * 2;
        for (int i = threadIdx.x; i < a.n_loss_part; i += 32) { s1 += lp[2 * i]; s2 += lp[2 * i + 1]; }
        s1 = warp_sum(s1); s2 = warp_sum(s2);
        if (threadIdx.x == 0) {
            const float l1 = s1 * a.l1_scale, l2 = s2 * a.l2_scale;
            a.losses[p * 3 + 0] = l1 + a.beta_loss * l2;
            a.losses[p * 3 + 1] = l1;
            a.losses[p * 3 + 2] = l2;
            if (a.losses_host != nullptr) {                  // the step's result, straight into pinned host memory
                a.losses_host[p * 3 + 0] = l1 + a.beta_loss * l2;
                a.losses_host[p * 3 + 1] = l1;
                a.losses_host[p * 3 + 2] = l2;
            }
        }
    }
    if (threadIdx.x == 0) {
        double bc1;
        float sb2;
        bias_corrections(a, p, bc1, sb2);
        sqrt_bc2_s = sb2;
        for (int s = 0; s < a.n_seg; ++s) step_size_s[s] = (float)((double)a.seg[s].lr / bc1);
    }
    __syncthreads();
    const float sqrt_bc2 = sqrt_bc2_s;
    const AdamConsts kc = {(float)a.beta2, (float)(1.0 - a.beta1), (float)(1.0 - a.beta2), (float)a.eps};

    for (int s = 0; s < a.n_seg; ++s) {
        const sfgpi_adam_segment &sg = a.seg[s];
        const bool shared = (sg.param_stride == 0 && a.n_pol > 1);
        const float step_size = step_size_s[s];
        if (!shared) {
            const float *gp0 = sg.grad_part + (size_t)p * sg.grad_pol_stride;
            float *pp0 = sg.param + (size_t)p * sg.param_stride;
            float *pm0 = sg.m + (size_t)p * sg.m_stride;
            float *pv0 = sg.v + (size_t)p * sg.v_stride;
            const bool vec = ((sg.len | sg.grad_part_stride) & 3) == 0 &&
                             ((reinterpret_cast<uintptr_t>(gp0) | reinterpret_cast<uintptr_t>(pp0) |
                               reinterpret_cast<uintptr_t>(pm0) | reinterpret_cast<uintptr_t>(pv0)) & 15) == 0;
            const bool clamp = sg.clamp_min < sg.clamp_max;
            if (a.fresh || clamp) {                           // first-step / clamped segments (G4, target-task adaptation): scalar path
                for (int i = blockIdx.x * kAdamThreads + threadIdx.x; i < sg.len; i += blocks_per_pol * kAdamThreads) {
                    const float g = sum_partials(gp0 + i, sg.n_part, (size_t)sg.grad_part_stride);
                    float pw = pp0[i], m = a.fresh ? 0.0f : pm0[i], v = a.fresh ? 0.0f : pv0[i];
                    adam_elem(pw, m, v, g, step_size, sqrt_bc2, sg.weight_decay, kc);
                    if (clamp) pw = fminf(fmaxf(pw, sg.clamp_min), sg.clamp_max);
                    pp0[i] = pw;
                    if (!a.fresh) { pm0[i] = m; pv0[i] = v; }
                }
            } else if (vec) {                                 // 128-bit path: 4 parameters per thread per trip
                const int n4 = sg.len >> 2;
                for (int i = blockIdx.x * kAdamThreads + threadIdx.x; i < n4; i += blocks_per_pol * kAdamThreads) {
                    float4 g = sum_partials4(reinterpret_cast<const float4 *>(gp0) + i, sg.n_part, (size_t)(sg.grad_part_stride >> 2));
                    float4 pw = reinterpret_cast<float4 *>(pp0)[i], m = reinterpret_cast<float4 *>(pm0)[i],
                           v = reinterpret_cast<float4 *>(pv0)[i];
                    adam_elem(pw.x, m.x, v.x, g.x, step_size, sqrt_bc2, sg.weight_decay, kc);
                    adam_elem(pw.y, m.y, v.y, g.y, step_size, sqrt_bc2, sg.weight_decay, kc);
                    adam_elem(pw.z, m.z, v.z, g.z, step_size, sqrt_bc2, sg.weight_decay, kc);
                    adam_elem(pw.w, m.w, v.w, g.w, step_size, sqrt_bc2, sg.weight_decay, kc);
                    reinterpret_cast<float4 *>(pp0)[i] = pw;
                    reinterpret_cast<float4 *>(pm0)[i] = m;
                    reinterpret_cast<float4 *>(pv0)[i] = v;
                }
            } else {
                for (int i = blockIdx.x * kAdamThreads + threadIdx.x; i < sg.len; i += blocks_per_pol * kAdamThreads) {
                    const float g = sum_partials(gp0 + i, sg.n_part, (size_t)sg.grad_part_stride);
                    float pw = pp0[i], m = pm0[i], v = pv0[i];
                    adam_elem(pw, m, v, g, step_size, sqrt_bc2, sg.weight_decay, kc);
                    pp0[i] = pw; pm0[i] = m; pv0[i] = v;
                }
            }
        } else {
            // shared tensor (TSF's h) stepped by every optimizer from the SAME pre-step value (frozen-snapshot ensemble semantics,
            // see DESIGN.md); each optimizer has its own moments and step.  One WARP per element, lane = optimizer: the per-optimizer
            // work (partial sums, moments, delta) runs in parallel and the deltas are summed by a fixed butterfly.  Every block of
            // the grid takes part.
            const int lane = threadIdx.x & 31;
            const int warps_total = gridDim.x * gridDim.y * (kAdamThreads / 32);
            const int wg = (blockIdx.y * gridDim.x + blockIdx.x) * (kAdamThreads / 32) + (threadIdx.x >> 5);
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
                        const float g = sum_partials(sg.grad_part + (size_t)q * sg.grad_pol_stride + i, sg.n_part,
                                                     (size_t)sg.grad_part_stride);
                        float *pm = sg.m + (size_t)q * sg.m_stride + i;
                        float *pv = sg.v + (size_t)q * sg.v_stride + i;
                        float pw = p0, m = *pm, v = *pv;
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
    }
    // fused finish (consts_next given): optimizer p's first CTA advances the step counter and derives the NEXT step's bias
    // corrections into the other buffer.  Nothing in this launch reads `step` or `consts_next`, so there is no ordering to
    // enforce -- unlike a last-CTA tail, this adds no serial work after the update itself.
    if (a.consts_next != nullptr && !a.fresh && blockIdx.x == 0 && threadIdx.x == 0) {
        const int s_new = a.step[p] + 1;
        a.step[p] = s_new;
        const double t = (double)(s_new + 1);
        a.consts_next[2 * p] = 1.0 - pow(a.beta1, t);
        a.consts_next[2 * p + 1] = sqrt(1.0 - pow(a.beta2, t));
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

__global__ void adam_finish_kernel(int32_t *step, double *consts, int n, double beta1, double beta2) {
    pdl_launch_dependents();
    pdl_wait();
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) adam_finish_one(step, consts, i, beta1, beta2);
}

// ---- flattened fast path -----------------------------------------------------------------------------------------------------
// adam_kernel above walks the segments one after the other and starts with a one-thread prologue (bias corrections in double,
// __syncthreads): with ~1 trip per thread that is a chain of 5-6 dependent memory round trips (prologue, psi, w, g, shared h)
// on a kernel that moves 31 MB -- 16.5 us for 4.8 us of HBM time (profiles/r01_step_kernels_full_v2.md).  Here every segment
// has its own block range of ONE grid, every thread owns exactly one 128-bit item and issues all of its loads (bias
// corrections, partials, p, m, v) before the first use, and the step size (lr / (1 - beta1^t), a double division as on the
// host) is computed by each thread while those loads are in flight.  Same arithmetic and summation order per element as
// adam_kernel: bit-identical results.  Taken when every per-optimizer segment is 128-bit aligned and neither fresh nor clamped.
struct AdamFlat {
    int blk_end[SFGPI_MAX_SEGMENTS];   // exclusive prefix ends of the per-optimizer segments' block ranges (shared segments: empty)
    int n_own;                         // blocks of per-optimizer segments
    int n_shared;                      // blocks (per grid row) that step the shared segments, warp per element
};

__global__ void __launch_bounds__(kAdamThreads) adam_flat_kernel(const __grid_constant__ sfgpi_adam_args a, const __grid_constant__ AdamFlat f) {
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
        if (i < (sg.len >> 2)) {
            const double bc1 = a.consts[2 * p];
            const float sqrt_bc2 = (float)a.consts[2 * p + 1];
            const float4 *gp = reinterpret_cast<const float4 *>(sg.grad_part + (size_t)p * sg.grad_pol_stride) + i;
            float4 *pp = reinterpret_cast<float4 *>(sg.param + (size_t)p * sg.param_stride) + i;
            float4 *pm = reinterpret_cast<float4 *>(sg.m + (size_t)p * sg.m_stride) + i;
            float4 *pv = reinterpret_cast<float4 *>(sg.v + (size_t)p * sg.v_stride) + i;
            float4 pw = *pp, m = *pm, v = *pv;
            const float4 g = sum_partials4(gp, sg.n_part, (size_t)(sg.grad_part_stride >> 2));
            const float step_size = (float)((double)sg.lr / bc1);
            adam_elem(pw.x, m.x, v.x, g.x, step_size, sqrt_bc2, sg.weight_decay, kc);
            adam_elem(pw.y, m.y, v.y, g.y, step_size, sqrt_bc2, sg.weight_decay, kc);
            adam_elem(pw.z, m.z, v.z, g.z, step_size, sqrt_bc2, sg.weight_decay, kc);
            adam_elem(pw.w, m.w, v.w, g.w, step_size, sqrt_bc2, sg.weight_decay, kc);
            *pp = pw; *pm = m; *pv = v;
        }
    } else if (bid < f.n_own + f.n_shared) {
        // shared tensors (TSF's h): every optimizer steps them from the SAME pre-step value, each with its own moments; one warp
        // per element, lane = optimizer, deltas summed by a fixed butterfly (as in adam_kernel)
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
                        const double qbc1 = a.consts[2 * q];
                        const float qsb2 = (float)a.consts[2 * q + 1];
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
        if (threadIdx.x == 32) {
            const int s_new = a.step[p] + 1;
            a.step[p] = s_new;
            const double t = (double)(s_new + 1);
            a.consts_next[2 * p] = 1.0 - pow(a.beta1, t);
            a.consts_next[2 * p + 1] = sqrt(1.0 - pow(a.beta2, t));
        }
    }
    trace_exit(SFGPI_TR_ADAM);
}

}  // namespace sfgpi

using namespace sfgpi;

extern "C" int sfgpi_adam_step(const sfgpi_adam_args *args, void *stream) {
    trace_bind();
    sfgpi_adam_args a_host = *args;
    if (a_host.losses_host != nullptr) {                     // the kernel needs the device-visible address of the pinned buffer
        cudaPointerAttributes at;
        if (a_host.loss_part == nullptr || cudaPointerGetAttributes(&at, a_host.losses_host) != cudaSuccess || at.type != cudaMemoryTypeHost ||
            !at.devicePointer) {
            cudaGetLastError();
            set_error("sfgpi_adam_step: losses_host must be pinned host memory (and needs loss_part)");
            return SFGPI_E_INVALID;
        }
        a_host.losses_host = reinterpret_cast<float *>(at.devicePointer);
    }
    const sfgpi_adam_args &a = a_host;
    if (a.n_seg < 1 || a.n_seg > SFGPI_MAX_SEGMENTS || a.n_pol < 1 || (a.step == nullptr && !a.fresh)) {
        set_error("sfgpi_adam_step: invalid arguments");
        return SFGPI_E_INVALID;
    }
    if (a.consts_next != nullptr && (a.consts == nullptr || a.consts_next == a.consts)) {
        set_error("sfgpi_adam_step: consts_next needs a distinct consts buffer to read from");
        return SFGPI_E_INVALID;
    }
    int max_len = 0;
    for (int s = 0; s < a.n_seg; ++s) {
        if (a.fresh && a.seg[s].param_stride == 0 && a.n_pol > 1) { set_error("sfgpi_adam_step: fresh optimizers cannot share a tensor"); return SFGPI_E_INVALID; }
        if (a.seg[s].len < 0 || a.seg[s].n_part < 1) { set_error("sfgpi_adam_step: bad segment %d", s); return SFGPI_E_INVALID; }
        max_len = a.seg[s].len > max_len ? a.seg[s].len : max_len;
    }
    cudaStream_t st = (cudaStream_t)stream;
    // flattened fast path (see adam_flat_kernel): the train steps' shape -- double-buffered corrections, 128-bit aligned segments
    if (!a.fresh && a.consts != nullptr && a.consts_next != nullptr) {
        AdamFlat f;
        bool ok = true;
        int nb = 0, shared_len = 0;
        for (int s = 0; s < SFGPI_MAX_SEGMENTS; ++s) {
            if (s < a.n_seg) {
                const sfgpi_adam_segment &sg = a.seg[s];
                const bool shared = sg.param_stride == 0 && a.n_pol > 1;
                if (shared) shared_len = sg.len > shared_len ? sg.len : shared_len;
                else {
                    const bool vec = ((sg.len | sg.grad_part_stride | sg.grad_pol_stride | sg.param_stride | sg.m_stride | sg.v_stride) & 3) == 0 &&
                                     ((reinterpret_cast<uintptr_t>(sg.grad_part) | reinterpret_cast<uintptr_t>(sg.param) |
                                       reinterpret_cast<uintptr_t>(sg.m) | reinterpret_cast<uintptr_t>(sg.v)) & 15) == 0;
                    if (!vec || sg.clamp_min < sg.clamp_max) { ok = false; break; }
                    nb += ((sg.len >> 2) + kAdamThreads - 1) / kAdamThreads;
                }
            }
            f.blk_end[s] = nb;
        }
        if (ok) {
            f.n_own = nb;
            const int warps = (shared_len + a.n_pol - 1) / a.n_pol;                  // warps per grid row: one element each
            f.n_shared = shared_len > 0 ? (warps + kAdamThreads / 32 - 1) / (kAdamThreads / 32) : 0;
            if (f.n_shared > 296) f.n_shared = 296;
            launch_pdl(adam_flat_kernel, dim3(f.n_own + f.n_shared + 1, a.n_pol), dim3(kAdamThreads), 0, st, a, f);
            return check_launch("sfgpi_adam_step(flat)");
        }
    }
    int blocks = (max_len + kAdamThreads - 1) / kAdamThreads;
    if (blocks < 1) blocks = 1;
    const int cap = (148 * 8 + a.n_pol - 1) / a.n_pol;                 // ~8 CTAs per SM over the whole launch
    if (blocks > cap) blocks = cap < 1 ? 1 : cap;
    dim3 grid(blocks, a.n_pol);
    launch_pdl(adam_kernel, grid, dim3(kAdamThreads), 0, st, a, blocks);
    int rc = check_launch("sfgpi_adam_step");
    if (rc || a.consts_next != nullptr || a.fresh) return rc;
    launch_pdl(adam_finish_kernel, dim3((a.n_pol + 127) / 128), dim3(128), 0, st, a.step, a.consts, a.n_pol, a.beta1, a.beta2);
    return check_launch("sfgpi_adam_step(finish)");
}

extern "C" int sfgpi_adam_refresh(const int32_t *step, double *consts_a, double *consts_b, int32_t n, double beta1, double beta2, void *stream) {
    if (n < 0 || !step || !consts_a || !consts_b) { set_error("sfgpi_adam_refresh: invalid arguments"); return SFGPI_E_INVALID; }
    if (n == 0) return SFGPI_OK;
    launch_pdl(adam_refresh_kernel, dim3((n + 127) / 128), dim3(128), 0, (cudaStream_t)stream, step, consts_a, consts_b, (int)n, beta1, beta2);
    return check_launch("sfgpi_adam_refresh");
}
