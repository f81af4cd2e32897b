// Folded-GPI column order, shared by the tensor-core forward kernels (mlp_forward_tc.cu: bf16; mlp_stream_tc.cu: tf32 / tf32x3),
// and the blocked running (max, argmax) scan of the tf32 kernel.
#pragma once
#include "tc_common.cuh"

namespace sfgpi {
namespace tc {

// Column order of the folded GPI output layer.  The epilogue scans the columns with ONE thread per state, so a running
// (max, argmax) per reward vector is a dependent compare/select chain; with the plain order column = wi * A + act a trip of 8
// columns belongs to one or two vectors and runs at the chain's latency (~66 cycles per column measured).  Reward vectors are
// therefore interleaved in blocks of WB = 8 (4 for 4..7 vectors): column = (block * A + act) * WB + w_in_block, so one 8-column
// trip feeds WB INDEPENDENT chains.  Vectors are padded to a multiple of WB (zero columns, never emitted).  WB = 1: plain order.
__host__ __device__ inline int gpi_wblock(int nw) { return nw >= 8 ? 8 : (nw >= 4 ? 4 : 1); }
__host__ __device__ inline int gpi_ncols(int nw, int A) { const int wb = gpi_wblock(nw); return (nw + wb - 1) / wb * wb * A; }
// folded row -> (reward vector, action); wi >= nw: padding
__device__ __forceinline__ void gpi_row_to_wa(int row, int nw, int A, int &wi, int &act) {
    const int wb = gpi_wblock(nw);
    const int blk = row / (wb * A), rem = row - blk * (wb * A);
    act = rem / wb;
    wi = blk * wb + (rem - act * wb);
}

// 8 columns (registers OFF .. OFF+7 of a 32-column TMEM load) of the blocked scan: 8 / WB actions x WB reward vectors
template <int WB, int OFF>
__device__ __forceinline__ void gpi_scan_blocked(const uint32_t (&v)[32], const float (&bv)[8], int col, int ncol, int A_, int nw, float (&bb)[8],
                                                 int (&ba)[8], int &act_i, int &g, long long *&kp, long long *&tp, uint32_t kstep,
                                                 bool k_has, bool t_has, bool row_ok, uint32_t task_id, float *q_row) {
#pragma unroll
    for (int j = 0; j < 8 / WB; ++j) {
        if (col + j * WB < ncol) {                           // (ncol is a multiple of WB)
#pragma unroll
            for (int ws = 0; ws < WB; ++ws) {
                const float q = __uint_as_float(v[OFF + j * WB + ws]) + bv[j * WB + ws];
                if (q > bb[ws]) { bb[ws] = q; ba[ws] = act_i; }
            }
            if (q_row != nullptr && g == 0) q_row[act_i] = __uint_as_float(v[OFF + j * WB]) + bv[j * WB];       // reward vector 0
            if (++act_i == A_) {                             // block complete: WB keys out, state reset
#pragma unroll
                for (int ws = 0; ws < WB; ++ws) {
                    if (row_ok && g * WB + ws < nw) {
                        if (k_has) atomicMax(kp + (size_t)ws * kstep, pack_key(bb[ws], (uint32_t)ba[ws]));
                        if (t_has) atomicMax(tp + (size_t)ws * kstep, pack_key(bb[ws], task_id));
                    }
                    bb[ws] = -INFINITY;
                    ba[ws] = 0;
                }
                kp += (size_t)WB * kstep;
                tp += (size_t)WB * kstep;
                act_i = 0;
                ++g;
            }
        }
    }
}

}  // namespace tc
}  // namespace sfgpi
