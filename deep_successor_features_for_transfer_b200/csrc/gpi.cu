// GPI helpers: packed-key fill / decode, the unfused GPI epilogue on a materialised psi, error plumbing.
#include <stdarg.h>
#include <limits.h>
#include <stdlib.h>
#include "common.cuh"

namespace sfgpi {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

bool pdl_enabled() {
    static const bool on = getenv("SFGPI_NO_PDL") == nullptr;
    return on;
}

static unsigned long long *g_trace_buf = nullptr;
static int g_trace_on = -1, g_trace_gen = 0;      // -1: not decided yet (env SFGPI_TRACE)

static void trace_reset_buffer() {
    unsigned long long h[SFGPI_TR_SLOTS * 3];
    for (int i = 0; i < SFGPI_TR_SLOTS; ++i) { h[3 * i] = h[3 * i + 1] = ~0ull; h[3 * i + 2] = 0; }
    cudaMemcpy(g_trace_buf, h, sizeof(h), cudaMemcpyHostToDevice);
}
unsigned long long *trace_buffer() {
    if (g_trace_on < 0) g_trace_on = getenv("SFGPI_TRACE") != nullptr ? 1 : 0;
    if (!g_trace_on) return nullptr;
    if (g_trace_buf == nullptr) {
        if (cudaMalloc(&g_trace_buf, SFGPI_TR_SLOTS * 3 * sizeof(unsigned long long)) != cudaSuccess) { g_trace_buf = nullptr; return nullptr; }
        trace_reset_buffer();
    }
    return g_trace_buf;
}
int trace_generation() { return g_trace_gen; }

int check_launch(const char *what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: CUDA error: %s", what, cudaGetErrorString(e));
        return SFGPI_E_CUDA;
    }
    return SFGPI_OK;
}

}  // namespace sfgpi

// Developer aid, see include/sfgpi.h.  sfgpi_trace_enable: switches the kernel-window trace on / off (takes effect at each
// kernel family's next launch); sfgpi_trace_read: synchronises the device, copies out [slots][3] = {first CTA entry, first CTA
// past its dependency wait, last CTA exit} in %globaltimer ns (entry = ~0 for kernels that did not run) and resets the windows;
// sfgpi_trace_dump: the same, printed to stderr.
extern "C" void sfgpi_trace_enable(int32_t on) {
    sfgpi::g_trace_on = on ? 1 : 0;
    ++sfgpi::g_trace_gen;
    if (on && sfgpi::trace_buffer() != nullptr) { cudaDeviceSynchronize(); sfgpi::trace_reset_buffer(); }
}

extern "C" int sfgpi_trace_read(uint64_t *out, int32_t n_slots) {
    unsigned long long *buf = sfgpi::g_trace_on > 0 ? sfgpi::trace_buffer() : nullptr;
    if (buf == nullptr || out == nullptr) return 0;
    cudaDeviceSynchronize();
    unsigned long long h[sfgpi::SFGPI_TR_SLOTS * 3];
    cudaMemcpy(h, buf, sizeof(h), cudaMemcpyDeviceToHost);
    const int n = n_slots < sfgpi::SFGPI_TR_SLOTS ? n_slots : sfgpi::SFGPI_TR_SLOTS;
    for (int i = 0; i < 3 * n; ++i) out[i] = h[i];
    sfgpi::trace_reset_buffer();
    return n;
}

extern "C" void sfgpi_trace_dump(void) {
    uint64_t h[sfgpi::SFGPI_TR_SLOTS * 3], t0 = ~0ull;
    if (sfgpi_trace_read(h, sfgpi::SFGPI_TR_SLOTS) == 0) return;
    static const char *name[sfgpi::SFGPI_TR_SLOTS] = {"prep", "forward", "td", "dgrad", "wgrad", "adam", "peer_x", "-"};
    for (int i = 0; i < sfgpi::SFGPI_TR_SLOTS; ++i) if (h[3 * i] < t0) t0 = h[3 * i];
    fprintf(stderr, "[sfgpi trace] ns since the first kernel entry: entry / past dependency wait / last exit\n");
    for (int i = 0; i < sfgpi::SFGPI_TR_SLOTS; ++i)
        if (h[3 * i + 2] != 0)
            fprintf(stderr, "  %-8s %8lld %8lld %8lld\n", name[i], (long long)(h[3 * i] - t0), (long long)(h[3 * i + 1] - t0), (long long)(h[3 * i + 2] - t0));
}

namespace sfgpi {

__global__ void keys_fill_kernel(long long *keys, long long n) {
    pdl_launch_dependents();
    pdl_wait();
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) keys[i] = LLONG_MIN;
}

__global__ void keys_decode_kernel(const long long *__restrict__ keys, long long n, long long *__restrict__ index_out,
                                   float *__restrict__ value_out) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        const long long k = keys[i];
        if (index_out) index_out[i] = (long long)key_index(k);
        if (value_out) value_out[i] = key_value(k);
    }
}

// One warp per state: lanes stride over the N*A (policy, action) cells, each cell a D-long dot product with w.
// psi [B][N][A][D] is read exactly once (HBM-bound: 4*N*A*D bytes per state), q [B][N][A] optionally written.
__global__ void __launch_bounds__(256) gpi_from_psi_kernel(const float *__restrict__ psi, const float *__restrict__ w, int B,
                                                           int N, int A, int D, int task_base, float *__restrict__ q_out,
                                                           long long *__restrict__ key_action,
                                                           long long *__restrict__ key_task) {
    extern __shared__ float w_s[];
    for (int d = threadIdx.x; d < D; d += blockDim.x) w_s[d] = w[d];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int warps_per_block = blockDim.x >> 5;
    for (int b = blockIdx.x * warps_per_block + (threadIdx.x >> 5); b < B; b += gridDim.x * warps_per_block) {
        const float *pb = psi + (size_t)b * N * A * D;
        long long kA = LLONG_MIN, kT = LLONG_MIN;
        for (int cell = lane; cell < N * A; cell += 32) {
            const float *pv = pb + (size_t)cell * D;
            float q = 0.0f;
            if ((D & 3) == 0) {
                for (int d = 0; d < D; d += 4) {
                    const float4 v = *reinterpret_cast<const float4 *>(pv + d);
                    q = fmaf(v.x, w_s[d], q);
                    q = fmaf(v.y, w_s[d + 1], q);
                    q = fmaf(v.z, w_s[d + 2], q);
                    q = fmaf(v.w, w_s[d + 3], q);
                }
            } else {
                for (int d = 0; d < D; ++d) q = fmaf(pv[d], w_s[d], q);
            }
            if (q_out) q_out[(size_t)b * N * A + cell] = q;
            const int j = cell / A, act = cell - j * A;
            const long long ka = pack_key(q, (uint32_t)act), kt = pack_key(q, (uint32_t)(task_base + j));
            kA = ka > kA ? ka : kA;
            kT = kt > kT ? kt : kT;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const long long oa = __shfl_xor_sync(0xffffffffu, kA, o), ot = __shfl_xor_sync(0xffffffffu, kT, o);
            kA = oa > kA ? oa : kA;
            kT = ot > kT ? ot : kT;
        }
        if (lane == 0) {
            if (key_action) key_action[b] = kA;
            if (key_task) key_task[b] = kT;
        }
    }
}

}  // namespace sfgpi

using namespace sfgpi;

extern "C" const char *sfgpi_last_error(void) { return g_err; }
extern "C" int sfgpi_version(void) { return 103; }

extern "C" int sfgpi_keys_fill(int64_t *keys, int64_t n, void *stream) {
    if (n <= 0) return SFGPI_OK;
    int blocks = (int)((n + 255) / 256);
    if (blocks > 148 * 8) blocks = 148 * 8;
    launch_pdl(keys_fill_kernel, dim3(blocks), dim3(256), 0, (cudaStream_t)stream, reinterpret_cast<long long *>(keys), (long long)n);
    return check_launch("sfgpi_keys_fill");
}

extern "C" int sfgpi_keys_decode(const int64_t *keys, int64_t n, int64_t *index_out, float *value_out, void *stream) {
    if (n <= 0) return SFGPI_OK;
    int blocks = (int)((n + 255) / 256);
    if (blocks > 148 * 8) blocks = 148 * 8;
    keys_decode_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const long long *>(keys), (long long)n,
                                                                  reinterpret_cast<long long *>(index_out), value_out);
    return check_launch("sfgpi_keys_decode");
}

extern "C" int sfgpi_gpi_from_psi(const float *psi, const float *w, int32_t B, int32_t N, int32_t A, int32_t D,
                                  int32_t task_base, float *q_out, int64_t *key_action, int64_t *key_task, void *stream) {
    if (B < 0 || N < 1 || A < 1 || D < 1 || D > 8192) { set_error("sfgpi_gpi_from_psi: invalid sizes"); return SFGPI_E_INVALID; }
    if (B == 0) return SFGPI_OK;
    int blocks = (B + 7) / 8;
    if (blocks > 148 * 8) blocks = 148 * 8;
    gpi_from_psi_kernel<<<blocks, 256, D * sizeof(float), (cudaStream_t)stream>>>(
        psi, w, B, N, A, D, task_base, q_out, reinterpret_cast<long long *>(key_action), reinterpret_cast<long long *>(key_task));
    return check_launch("sfgpi_gpi_from_psi");
}

// ---- policy sharding: ONE all-gather per train step carries everything the ranks exchange besides the GPI keys --------------
// x_local = [ w of the local policies (nw floats) | delta of the shared h applied by the local optimizers (nh floats) ]
namespace sfgpi {
__global__ void shard_pack_kernel(const float *__restrict__ w, int nw, const float *__restrict__ h, const float *__restrict__ h_prev,
                                  int nh, float *__restrict__ x_local) {
    pdl_launch_dependents();
    pdl_wait();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nw) x_local[i] = w[i];
    else if (i < nw + nh) x_local[i] = h[i - nw] - h_prev[i - nw];
}
// x_all [world][nw + nh] -> w_all [world * nw] (reward vectors of ALL policies, rank-major = global policy order),
// h = h_prev + sum_r delta_r (rank order: identical on every rank), h_prev = h
__global__ void shard_unpack_kernel(const float *__restrict__ x_all, int world, int nw, int nh, float *__restrict__ w_all,
                                    float *__restrict__ h, float *__restrict__ h_prev) {
    pdl_launch_dependents();
    pdl_wait();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int stride = nw + nh;
    if (i < world * nw) {
        const int r = i / nw, k = i - r * nw;
        w_all[i] = x_all[(size_t)r * stride + k];
    } else if (i < world * nw + nh) {
        const int k = i - world * nw;
        float acc = h_prev[k];
        for (int r = 0; r < world; ++r) acc += x_all[(size_t)r * stride + nw + k];
        h[k] = acc;
        h_prev[k] = acc;
    }
}
}  // namespace sfgpi

extern "C" int sfgpi_shard_pack(const float *w, int32_t nw, const float *h, const float *h_prev, int32_t nh, float *x_local,
                                void *stream) {
    if (nw < 0 || nh < 0 || (nh > 0 && (!h || !h_prev)) || !x_local) { set_error("sfgpi_shard_pack: invalid arguments"); return SFGPI_E_INVALID; }
    if (nw + nh == 0) return SFGPI_OK;
    launch_pdl(shard_pack_kernel, dim3((nw + nh + 255) / 256), dim3(256), 0, (cudaStream_t)stream, w, (int)nw, h, h_prev, (int)nh, x_local);
    return check_launch("sfgpi_shard_pack");
}

extern "C" int sfgpi_shard_unpack(const float *x_all, int32_t world, int32_t nw, int32_t nh, float *w_all, float *h, float *h_prev,
                                  void *stream) {
    if (world < 1 || nw < 0 || nh < 0 || !x_all) { set_error("sfgpi_shard_unpack: invalid arguments"); return SFGPI_E_INVALID; }
    const int n = world * nw + nh;
    if (n == 0) return SFGPI_OK;
    launch_pdl(shard_unpack_kernel, dim3((n + 255) / 256), dim3(256), 0, (cudaStream_t)stream, x_all, (int)world, (int)nw, (int)nh, w_all,
               h, h_prev);
    return check_launch("sfgpi_shard_unpack");
}
