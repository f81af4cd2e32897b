// Target-task adaptation of the TSF agent (SURVEY 8f N1; tsfdqn.py:859-997), the part around the two ensemble forwards.
//   sfgpi_target_q      get_test_action's greedy branch (:864-871): q = w(sum_j omega^_j psi_j(s)), argmax_a -- one kernel
//   sfgpi_target_adapt  update_test_reward_mapper (:917-997) + scheduler.step(): omega^ = omega / sum omega, TSF mix of psi(s)[a]
//                       and psi^-(s')[a'], phi~ = phi * (h(sum_j omega^_j g_j(s)) + h(sum_j omega^_j g_j(s'))), the three loss terms,
//                       d/dw and d/domega by hand, Adam on (w, omega) in torch's operation order with the LambdaLR-decayed omega
//                       rate, omega.clamp_(1e-7).  Batch 1, N policies: a few thousand FMAs -- ONE small CTA replaces ~20 eager
//                       launches + torch.optim per environment step (4x more frequent than the train step).
#include "common.cuh"

namespace sfgpi {

constexpr int kTgtThreads = 256;

__device__ __forceinline__ float block_sum(float v, float *red) {
    v = warp_sum(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    float t = 0.0f;
    for (int k = 0; k < kTgtThreads / 32; ++k) t += red[k];
    return t;
}

__global__ void __launch_bounds__(kTgtThreads) target_q_kernel(const float *__restrict__ psi, int N, int A, int D,
                                                               const float *__restrict__ omegas, const float *__restrict__ w,
                                                               float *__restrict__ q_out, long long *__restrict__ action_out) {
    __shared__ float red[kTgtThreads / 32];
    __shared__ float q_s[256];
    pdl_launch_dependents();
    pdl_wait();
    float so = 0.0f;
    for (int j = threadIdx.x; j < N; j += kTgtThreads) so += omegas[j];
    const float S = block_sum(so, red);
    for (int a = threadIdx.x; a < A; a += kTgtThreads) {
        // q[a] = sum_d w[d] * sum_j (omega_j / S) psi[j][a][d]   (sum over j first, as the reference's torch.sum(axis=1) then w())
        float q = 0.0f;
        for (int d = 0; d < D; ++d) {
            float mix = 0.0f;
            for (int j = 0; j < N; ++j) mix = fmaf(psi[((size_t)j * A + a) * D + d], omegas[j] / S, mix);
            q = fmaf(w[d], mix, q);
        }
        q_s[a] = q;
        if (q_out) q_out[a] = q;
    }
    __syncthreads();
    if (threadIdx.x == 0 && action_out) {
        float best_q = -INFINITY;
        int best = 0;
        for (int a = 0; a < A; ++a)                            // first maximal index (torch.argmax); a NaN is never selected,
            if (q_s[a] > best_q) { best_q = q_s[a]; best = a; }     // all NaN / -inf: 0 (the packed GPI keys' rule)
        action_out[0] = best;
    }
}

__global__ void __launch_bounds__(kTgtThreads) target_adapt_kernel(const __grid_constant__ sfgpi_target_args a) {
    extern __shared__ float sm[];
    __shared__ float red[kTgtThreads / 32];
    pdl_launch_dependents();
    pdl_wait();
    const int N = a.N, A = a.A, D = a.D, G = a.G, S_ = a.S, tid = threadIdx.x;
    float *norm = sm;                 // [N]
    float *vj = norm + N;             // [N][G]  g_j(s) + g_j(s')
    float *u = vj + (size_t)N * G;    // [G]     sum_j norm_j vj
    float *aff = u + G;               // [D]
    float *tphi = aff + D;            // [D]
    float *delta = tphi + D;          // [D]     tsf - next_tsf
    float *dtphi = delta + D;         // [D]
    float *qv = dtphi + D;            // [G]     Wh^T (dtphi * phi)
    float *dnorm = qv + G;            // [N]
    float so = 0.0f;
    for (int j = tid; j < N; j += kTgtThreads) so += a.omegas[j];
    const float Ssum = block_sum(so, red);
    for (int j = tid; j < N; j += kTgtThreads) norm[j] = a.omegas[j] / Ssum;
    for (int e = tid; e < N * G; e += kTgtThreads) {          // v_j = Wg_j (s + s') + 2 bg_j
        const int j = e / G, g = e - j * G;
        const float *gp = a.g + (size_t)j * a.g_stride;
        float acc = 2.0f * gp[G * S_ + g];
        for (int s = 0; s < S_; ++s) acc = fmaf(gp[g * S_ + s], a.s[s] + a.s1[s], acc);
        vj[e] = acc;
    }
    __syncthreads();
    for (int g = tid; g < G; g += kTgtThreads) {
        float acc = 0.0f;
        for (int j = 0; j < N; ++j) acc = fmaf(vj[(size_t)j * G + g], norm[j], acc);
        u[g] = acc;
    }
    __syncthreads();
    const float *Wh = a.h, *bh = a.h + (size_t)D * G;
    for (int d = tid; d < D; d += kTgtThreads) {
        float acc = 2.0f * bh[d];                              // h(u_s) + h(u_s') = Wh (u_s + u_s') + 2 bh
        for (int g = 0; g < G; ++g) acc = fmaf(Wh[(size_t)d * G + g], u[g], acc);
        aff[d] = acc;
        tphi[d] = a.phi[d] * acc;
        float tsf = 0.0f, ntsf = 0.0f;
        for (int j = 0; j < N; ++j) {
            tsf = fmaf(a.psi[((size_t)j * A + a.a) * D + d], norm[j], tsf);
            ntsf = fmaf(a.next_psi[((size_t)j * A + a.a1) * D + d], norm[j], ntsf);
        }
        delta[d] = tsf - (tphi[d] + a.gamma * ntsf);
    }
    __syncthreads();
    float e_part = 0.0f, l1_part = 0.0f, l1n_part = 0.0f;
    for (int d = tid; d < D; d += kTgtThreads) { e_part = fmaf(a.w[d], tphi[d], e_part); l1_part = fmaf(delta[d], delta[d], l1_part); }
    for (int j = tid; j < N; j += kTgtThreads) l1n_part += fabsf(a.omegas[j]);
    const float e = block_sum(e_part, red) - a.r;
    const float l1 = block_sum(l1_part, red) / (float)D;
    const float onorm = block_sum(l1n_part, red);
    const float l2 = e * e;
    const float c1 = 2.0f / (float)D, c2 = 2.0f * a.beta * e;
    for (int d = tid; d < D; d += kTgtThreads) dtphi[d] = (c2 * a.w[d] - c1 * delta[d]) * a.phi[d];     // dL/daff
    __syncthreads();
    for (int g = tid; g < G; g += kTgtThreads) {
        float acc = 0.0f;
        for (int d = 0; d < D; ++d) acc = fmaf(Wh[(size_t)d * G + g], dtphi[d], acc);
        qv[g] = acc;
    }
    __syncthreads();
    float dot_part = 0.0f;
    for (int j = tid; j < N; j += kTgtThreads) {
        float acc = 0.0f;
        for (int d = 0; d < D; ++d)
            acc = fmaf(c1 * delta[d], a.psi[((size_t)j * A + a.a) * D + d] - a.gamma * a.next_psi[((size_t)j * A + a.a1) * D + d], acc);
        for (int g = 0; g < G; ++g) acc = fmaf(qv[g], vj[(size_t)j * G + g], acc);
        dnorm[j] = acc;
        dot_part = fmaf(acc, norm[j], dot_part);
    }
    const float dot = block_sum(dot_part, red);
    // ---- Adam (torch/optim/adam.py::_single_tensor_adam order), step t = step + 1 ----
    const double t = (double)(a.step[0] + 1);
    const double bc1 = 1.0 - pow(0.9, t);
    const float sqrt_bc2 = (float)sqrt(1.0 - pow(0.999, t));
    const float lr_o = (float)((double)a.lr_omega * pow(1.0 - (double)a.lr_omega_decay, (double)a.epoch[0]));
    auto adam = [&](float &p, float &m, float &v, float g, float lr, float wd) {
        if (wd != 0.0f) g = fmaf(wd, p, g);
        m = m + 0.1f * (g - m);
        v = v * 0.999f + 0.001f * g * g;
        const float denom = __fdiv_rn(sqrtf(v), sqrt_bc2) + 1e-8f;
        p = p - __fdiv_rn((float)((double)lr / bc1) * m, denom);
    };
    for (int d = tid; d < D; d += kTgtThreads) {
        float p = a.w[d], m = a.w_m[d], v = a.w_v[d];
        adam(p, m, v, c2 * tphi[d], a.lr_w, a.wd_w);
        a.w[d] = p; a.w_m[d] = m; a.w_v[d] = v;
    }
    for (int j = tid; j < N; j += kTgtThreads) {
        const float om = a.omegas[j];
        const float g = (dnorm[j] - dot) / Ssum + a.l1_coef * (om > 0.0f ? 1.0f : (om < 0.0f ? -1.0f : 0.0f));
        float p = om, m = a.o_m[j], v = a.o_v[j];
        adam(p, m, v, g, lr_o, a.wd_omega);
        a.omegas[j] = fmaxf(p, 1e-7f);                         // omegas.clamp_(1e-7), tsfdqn.py:977-979
        a.o_m[j] = m; a.o_v[j] = v;
    }
    __syncthreads();
    if (tid == 0) {
        a.losses[0] = l1 + a.beta * l2 + a.l1_coef * onorm;
        a.losses[1] = l2;
        a.losses[2] = l1;
        a.step[0] += 1;
        a.epoch[0] += 1;                                       // scheduler.step() (tsfdqn.py:895)
    }
}

}  // namespace sfgpi

using namespace sfgpi;

extern "C" int sfgpi_target_q(const float *psi, int32_t N, int32_t A, int32_t D, const float *omegas, const float *w, float *q_out,
                              int64_t *action_out, void *stream) {
    if (!psi || !omegas || !w || N < 1 || A < 1 || A > 256 || D < 1) { set_error("sfgpi_target_q: invalid arguments (1 <= A <= 256)"); return SFGPI_E_INVALID; }
    launch_pdl(target_q_kernel, dim3(1), dim3(kTgtThreads), 0, (cudaStream_t)stream, psi, (int)N, (int)A, (int)D, omegas, w, q_out,
               reinterpret_cast<long long *>(action_out));
    return check_launch("sfgpi_target_q");
}

extern "C" int sfgpi_target_adapt(const sfgpi_target_args *args, void *stream) {
    if (!args) { set_error("sfgpi_target_adapt: null args"); return SFGPI_E_INVALID; }
    const sfgpi_target_args &a = *args;
    if (a.N < 1 || a.A < 1 || a.D < 1 || a.G < 1 || a.S < 1 || a.a < 0 || a.a >= a.A || a.a1 < 0 || a.a1 >= a.A) {
        set_error("sfgpi_target_adapt: invalid sizes / actions");
        return SFGPI_E_INVALID;
    }
    if (!a.psi || !a.next_psi || !a.g || !a.h || !a.s || !a.s1 || !a.phi || !a.w || !a.omegas || !a.w_m || !a.w_v || !a.o_m || !a.o_v ||
        !a.step || !a.epoch || !a.losses) {
        set_error("sfgpi_target_adapt: null buffer");
        return SFGPI_E_INVALID;
    }
    const size_t fl = (size_t)a.N * 2 + (size_t)a.N * a.G + 2 * (size_t)a.G + 4 * (size_t)a.D;
    const size_t bytes = fl * sizeof(float);
    static int adapt_static = -1;
    if (int rc = smem_opt_in(target_adapt_kernel, bytes, &adapt_static, "sfgpi_target_adapt (N * G too large)")) return rc;
    launch_pdl(target_adapt_kernel, dim3(1), dim3(kTgtThreads), bytes, (cudaStream_t)stream, a);
    return check_launch("sfgpi_target_adapt");
}

namespace sfgpi {
__global__ void lms_kernel(float *__restrict__ w, const float *__restrict__ phi, const float *__restrict__ r, int D, float alpha) {
    pdl_launch_dependents();
    pdl_wait();
    float dot = 0.0f;
    for (int d = threadIdx.x; d < D; d += 32) dot = fmaf(phi[d], w[d], dot);
    dot = warp_sum(dot);
    const float err = alpha * (r[0] - dot);
    for (int d = threadIdx.x; d < D; d += 32) w[d] = fmaf(err, phi[d], w[d]);
}
}  // namespace sfgpi

extern "C" int sfgpi_lms_update(float *w, const float *phi, const float *r, int32_t D, float alpha, void *stream) {
    if (!w || !phi || !r || D < 1) { set_error("sfgpi_lms_update: invalid arguments"); return SFGPI_E_INVALID; }
    launch_pdl(sfgpi::lms_kernel, dim3(1), dim3(32), 0, (cudaStream_t)stream, w, phi, r, (int)D, alpha);
    return check_launch("sfgpi_lms_update");
}
