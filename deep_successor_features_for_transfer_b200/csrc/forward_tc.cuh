// Definitions shared by the tensor-core forward kernels (mlp_forward_tc.cu: ping-pong pairs;
// mlp_chain_tc.cu: the single-tile layer-pipelined chain): job / launch parameter blocks, the item (layer) table, the hidden-layer epilogue.
#pragma once
#include "tc_common.cuh"
#include "gpi_scan.cuh"

namespace sfgpi {
namespace tc {

constexpr int kNB = 128;                 // weight rows (output columns) per stage
constexpr int kStageBytes = kNB * kKB * 2;          // 16 KB
constexpr int kNStage = 4;
constexpr int kABytes = kTM * kH * 2;               // 64 KB per tile slot
constexpr int kThreadsTc = 416;                      // 4 producer warps + 1 MMA warp + 2 x 4 epilogue warps
constexpr int kMmaWarp = 4, kEpiWarp0 = 5;
constexpr int kBiasFloatsMax = 6144;                // all layers' biases of one policy, fp32 (24 KB)

struct TcParams {
    sfgpi_forward_args a;
    int rows_per_policy;     // rows of the bf16 shadow per policy = (1 + Lh)*256 + n3pad
    int n_final;             // output columns actually computed (padded to 16): n3pad (psi form) or nqpad (GPI form)
    int Lh;                  // number of 256x256 MMA layers (n_layers - 2)
    int n_items;             // 1 + Lh + ceil(n_final / 256)
    int ks0;                 // K=16 steps of the input layer = ceil(S / 16)
    int gpi;                 // 1: GPI form (folded weights, tmap_q / bq)
    int nw;                  // reward vectors scored per policy in GPI form
    int tiles_per_policy, pairs_per_policy, total_pairs, paired;
    const float *bq;         // folded bias [n_pol][n_final] (GPI form)
};

struct ItemInfo { int row_base, n_cols, col0, kind, n_kb, n_k16; };   // kind: 0 input layer, 1 hidden, 2 final

__device__ __forceinline__ ItemInfo item_info(const TcParams &p, int it) {
    ItemInfo r;
    if (it == 0) { r.row_base = 0; r.n_cols = kH; r.col0 = 0; r.kind = 0; r.n_kb = 1; r.n_k16 = p.ks0; }
    else if (it <= p.Lh) { r.row_base = it * kH; r.n_cols = kH; r.col0 = 0; r.kind = 1; r.n_kb = kH / kKB; r.n_k16 = kKB / 16; }
    else {
        const int c = it - 1 - p.Lh;
        r.col0 = c * 256;
        r.n_cols = min(256, p.n_final - r.col0);
        r.row_base = (p.gpi ? 0 : (1 + p.Lh) * kH) + r.col0;
        r.kind = 2; r.n_kb = kH / kKB; r.n_k16 = kKB / 16;
    }
    return r;
}

// (lo, hi) + (blo, bhi) as one packed fp32 instruction (sm_100: add.f32x2; each lane rounds exactly like add.rn.f32)
__device__ __forceinline__ void add_f32x2(float lo, float hi, float blo, float bhi, float &rlo, float &rhi) {
    asm("{\n\t.reg .b64 a, b, c;\n\tmov.b64 a, {%2, %3};\n\tmov.b64 b, {%4, %5};\n\tadd.rn.f32x2 c, a, b;\n\tmov.b64 {%0, %1}, c;\n\t}"
        : "=f"(rlo), "=f"(rhi) : "f"(lo), "f"(hi), "f"(blo), "f"(bhi));
}
// bf16x2(max(lo, 0), max(hi, 0)), round to nearest even: the ReLU rides in the conversion
__device__ __forceinline__ uint32_t pack_bf16x2_relu(float lo, float hi) {
    uint32_t d;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
}

__device__ __forceinline__ float act_apply_fast(float v, int act) {
    return act == SFGPI_ACT_RELU ? fmaxf(v, 0.0f) : (act == SFGPI_ACT_TANH ? tanhf(v) : v);
}

// One hidden-type epilogue for one row: 256 accumulator columns -> bias + activation -> bf16 -> next layer's A operand.
// The TMEM load of the next 32 columns is in flight while the current 32 are processed.
// NCH = 32-column chunks handled by this thread (8: the whole row; 4: one half, when both epilogue groups share a tile),
// starting at column cbase.
template <int ACT, int NCH, bool MASK>
__device__ __forceinline__ void hidden_epilogue(uint32_t t_lane, uint32_t bias, uint32_t Arow, int r, float *save,
                                                uint32_t *mask_out, int cbase) {
    uint32_t v[2][32];
    uint32_t mbits[NCH];                               // bit i of word cb: activation (cbase + 32 cb + i) > 0
    tmem_ld32(t_lane + cbase, v[0]);
#pragma unroll
    for (int cb = 0; cb < NCH; ++cb) {
        const int c0 = cbase + cb * 32;
        tmem_wait_ld();
        if (cb + 1 < NCH) tmem_ld32(t_lane + c0 + 32, v[(cb + 1) & 1]);
        const uint32_t(&u)[32] = v[cb & 1];
        uint32_t pk[16];
        uint32_t mb = 0;
#pragma unroll
        for (int g = 0; g < 8; ++g) {
            const float4 bv = lds128(bias + 4u * (c0 + 4 * g));
            // packed fp32 adds (add.f32x2) and, for ReLU, the clamp fused into the bf16 conversion (cvt.rn.relu.bf16x2.f32):
            // 4 instructions per 4 columns instead of 10 -- the epilogue is issue / latency bound (2 warps per scheduler)
            float h0, h1, h2, h3;
            add_f32x2(__uint_as_float(u[4 * g]), __uint_as_float(u[4 * g + 1]), bv.x, bv.y, h0, h1);
            add_f32x2(__uint_as_float(u[4 * g + 2]), __uint_as_float(u[4 * g + 3]), bv.z, bv.w, h2, h3);
            if (ACT == SFGPI_ACT_RELU) {
                if (MASK)
                    mb |= (h0 > 0.f ? 1u : 0u) << (4 * g) | (h1 > 0.f ? 2u : 0u) << (4 * g) | (h2 > 0.f ? 4u : 0u) << (4 * g) |
                          (h3 > 0.f ? 8u : 0u) << (4 * g);
                pk[2 * g] = pack_bf16x2_relu(h0, h1);
                pk[2 * g + 1] = pack_bf16x2_relu(h2, h3);
            } else {
                if (ACT == SFGPI_ACT_TANH) { h0 = tanhf(h0); h1 = tanhf(h1); h2 = tanhf(h2); h3 = tanhf(h3); }
                pk[2 * g] = pack_bf16x2(h0, h1);
                pk[2 * g + 1] = pack_bf16x2(h2, h3);
            }
        }
#pragma unroll
        for (int g = 0; g < 4; ++g)
            sts128(Arow + a_chunk_off(r, c0 + 8 * g), pk[4 * g], pk[4 * g + 1], pk[4 * g + 2], pk[4 * g + 3]);
        mbits[cb] = mb;
        if (save) {                                    // the bf16-rounded values the next layer really consumed
#pragma unroll
            for (int g = 0; g < 8; ++g)
                *reinterpret_cast<float4 *>(save + c0 + 4 * g) =
                    make_float4(__uint_as_float(pk[2 * g] << 16), __uint_as_float(pk[2 * g] & 0xFFFF0000u),
                                __uint_as_float(pk[2 * g + 1] << 16), __uint_as_float(pk[2 * g + 1] & 0xFFFF0000u));
        }
    }
    if (MASK && ACT == SFGPI_ACT_RELU && mask_out != nullptr) {    // 1 bit per activation: all the backward pass needs of a ReLU layer
        static_assert(NCH == 4 || NCH == 2, "mask row layout: 8 words per row; a call covers 4 (column half) or 2 (quarter) of them");
        if (NCH == 4) *reinterpret_cast<uint4 *>(mask_out + (cbase >> 5)) = make_uint4(mbits[0], mbits[1], mbits[NCH - 2], mbits[NCH - 1]);
        else *reinterpret_cast<uint2 *>(mask_out + (cbase >> 5)) = make_uint2(mbits[0], mbits[1]);
    }
}

// ---- folded-GPI scan of the columns [c_begin, c_end) of one accumulator chunk by one thread (= one state), 8 columns per trip
// of a rolled loop.  Column = (block * A + act) * WB + w_in_block (gpi_scan.cuh), WB | 8.  The range need not start or end at a
// block boundary: a partially seen block is emitted as it is -- every emission is an atomicMax on the (reward vector, state)
// key, so the rest of the block (the other epilogue group's half, or the next chunk) merges.
// one key out (action key and / or task key of one reward vector): out of line, so that the scan below stays a few cache lines
// of code.  The scan runs once per GPI tile, tens of thousands of cycles apart, and by then its code has left the instruction
// cache: its first trip pays an instruction fetch per cache line (measured: a first call of the inlined-emission version, 10 KB
// of code, cost 9-11 k cycles against 2.2 k for a second call right after it -- with or without keys to emit).
static __device__ __noinline__ void gpi_emit1(long long *ka, long long *kt, float best, int best_a, uint32_t task_id) {
    if (ka != nullptr) atomicMax(ka, pack_key(best, (uint32_t)best_a));
    if (kt != nullptr) atomicMax(kt, pack_key(best, task_id));
}

template <int WB>
__device__ __noinline__ void gpi_scan_rolled(uint32_t t_acc, uint32_t bias0, int col0_it, int c_begin, int c_end, int A_, int nw,
                                            long long *ka, long long *kt, uint32_t kstep, bool row_ok, uint32_t task_id, float *q_row) {
    const int per_blk = A_ * WB;
    int blk = c_begin / per_blk;
    int act_i = (c_begin - blk * per_blk) / WB;
    float bb[WB];
    int ba[WB];
#pragma unroll
    for (int i = 0; i < WB; ++i) { bb[i] = -INFINITY; ba[i] = 0; }
    // key of reward vector blk * WB for this thread's state; the pointers advance by one vector per emitted key (NULL stays NULL)
    const size_t sa = ka ? kstep : 0, st = kt ? kstep : 0;
    long long *pa = ka ? ka + (size_t)blk * WB * kstep : nullptr, *pt = kt ? kt + (size_t)blk * WB * kstep : nullptr;
#pragma unroll 1
    for (int c0 = c_begin; c0 < c_end; c0 += 8) {
        uint32_t v[8];
            tmem_ld8(t_acc + (uint32_t)(c0 - col0_it), v);
        const float4 b0 = lds128(bias0 + 4u * (uint32_t)c0), b1 = lds128(bias0 + 4u * (uint32_t)(c0 + 4));
        const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
        tmem_wait_ld();
    #pragma unroll
        for (int j = 0; j < 8 / WB; ++j) {
            const int col = c0 + j * WB;
            if (col < c_end) {                                   // (a range may end inside a trip: c_end is a multiple of WB, not of 8)
#pragma unroll
                for (int ws = 0; ws < WB; ++ws) {
                    const float q = __uint_as_float(v[j * WB + ws]) + bv[j * WB + ws];
                    if (q > bb[ws]) { bb[ws] = q; ba[ws] = act_i; }
                }
                if (q_row != nullptr && blk == 0) q_row[act_i] = __uint_as_float(v[j * WB]) + bv[j * WB];      // reward vector 0
                ++act_i;
                if (act_i == A_ || col + WB >= c_end) {          // block complete, or the range ends inside it
                    // A ROLLED loop over the block's vectors (the running state rotates through slot 0) and one out-of-line
                    // call per key: ~40 instructions of code per emission site instead of ~30 per key.
                    const int n_valid = row_ok ? min(WB, nw - blk * WB) : 0;
#pragma unroll 1
                    for (int ws = 0; ws < WB; ++ws) {
                        if (ws < n_valid) gpi_emit1(pa, pt, bb[0], ba[0], task_id);
                        pa += sa;
                        pt += st;
#pragma unroll
                        for (int i = 0; i + 1 < WB; ++i) { bb[i] = bb[i + 1]; ba[i] = ba[i + 1]; }
                    }
#pragma unroll
                    for (int i = 0; i < WB; ++i) { bb[i] = -INFINITY; ba[i] = 0; }
                    if (act_i == A_) { act_i = 0; ++blk; }
                    else { pa -= WB * sa; pt -= WB * st; }       // (range ended inside the block: the vector pointers stay on it)
                }
            }
        }
    }
}

// ---- psi-form output chunk of one accumulator for one thread (= one state): columns [col0, col0 + n_cols), the 8-column trips
// c_first, c_first + 16, ... (the two epilogue groups alternate).  psi_row: this state's row of the psi output ([A*D] floats, 16-byte
// aligned when A*D % 4 == 0) or NULL; sel_row: its gathered row [D] or NULL with sel_base = a * D (a negative sel_base: no gather).
// Out of line and rolled for the same reason as the GPI scan: it runs once per tile.
static __device__ __noinline__ void psi_out_rolled(uint32_t t_acc, uint32_t bias_chunk, int col0, int n_cols, int c_first, float *psi_row,
                                                  int AD, float *sel_row, int sel_base, int D, bool row_ok) {
#pragma unroll 1
    for (int c0 = c_first; c0 < n_cols; c0 += 16) {
        uint32_t v[8];
        tmem_ld8(t_acc + (uint32_t)c0, v);
        const float4 b0 = lds128(bias_chunk + 4u * (uint32_t)c0), b1 = lds128(bias_chunk + 4u * (uint32_t)(c0 + 4));
        const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
        tmem_wait_ld();
        const int colb = col0 + c0;
        float val[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) val[i] = __uint_as_float(v[i]) + bv[i];
        if (row_ok) {
            if (psi_row != nullptr) {
                float *po = psi_row + colb;
                if ((AD & 3) == 0) {                          // rows are 16-byte aligned: 128-bit stores
                    if (colb < AD) *reinterpret_cast<float4 *>(po) = make_float4(val[0], val[1], val[2], val[3]);
                    if (colb + 4 < AD) *reinterpret_cast<float4 *>(po + 4) = make_float4(val[4], val[5], val[6], val[7]);
                } else {
#pragma unroll
                    for (int i = 0; i < 8; ++i)
                        if (colb + i < AD) po[i] = val[i];
                }
            }
            if (sel_row != nullptr && (unsigned)(colb + 7 - sel_base) < (unsigned)(D + 7)) {         // trip overlaps [sel, sel + D)
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const unsigned off = (unsigned)(colb + i - sel_base);
                    if (off < (unsigned)D) sel_row[off] = val[i];
                }
            }
        }
    }
}

// ---- the same scan for launches with MANY reward vectors (n_w * A of several hundred columns: BASELINE config 4 scores every
// policy under 256 vectors = 2304 columns per tile).  There the scan -- not the MMAs -- paces the kernel (in-kernel timeline:
// 6.4-7 k cycles per 128 columns per epilogue group against ~3.9 k for the chunk's MMAs; ncu: the epilogue warps issue one
// instruction per ~5 cycles in the loop above -- fixed-latency dependencies, the bias loads behind the TMEM wait, instruction
// fetch over four inlined copies of the emission), and the loop runs tens of times per tile, so compact-and-rolled no longer
// matters.  This variant: 16 columns per TMEM load with the next load in flight, the window's biases fetched BEFORE the wait
// on the TMEM load, max by fmaxf beside the compare (no select on the value chain), and the emission out of line
// (gpi_emit8: one call per finished block of 8 reward vectors).
// Requires WB = 8, (c_end - c_begin) % 32 == 0, c_begin % 8 == 0 and no q output; same keys as gpi_scan_rolled<8> bit for bit.
static __device__ __noinline__ void gpi_emit8(char *pa, char *pt, uint32_t pitch, int n_valid, uint32_t task_id,
                                              float b0, float b1, float b2, float b3, float b4, float b5, float b6, float b7,
                                              int a0, int a1, int a2, int a3, int a4, int a5, int a6, int a7) {
    const float bb[8] = {b0, b1, b2, b3, b4, b5, b6, b7};
    const int ba[8] = {a0, a1, a2, a3, a4, a5, a6, a7};
    if (n_valid >= 8) {                                          // all but the last block of a padded vector count: no per-key guards
        if (pa != nullptr) {
#pragma unroll
            for (int ws = 0; ws < 8; ++ws)
                atomicMax(reinterpret_cast<long long *>(pa + (unsigned long long)ws * pitch), pack_key(bb[ws], (uint32_t)ba[ws]));
        }
        if (pt != nullptr) {
#pragma unroll
            for (int ws = 0; ws < 8; ++ws)
                atomicMax(reinterpret_cast<long long *>(pt + (unsigned long long)ws * pitch), pack_key(bb[ws], task_id));
        }
        return;
    }
    if (pa != nullptr) {
#pragma unroll
        for (int ws = 0; ws < 8; ++ws)
            if (ws < n_valid) atomicMax(reinterpret_cast<long long *>(pa + (unsigned long long)ws * pitch), pack_key(bb[ws], (uint32_t)ba[ws]));
    }
    if (pt != nullptr) {
#pragma unroll
        for (int ws = 0; ws < 8; ++ws)
            if (ws < n_valid) atomicMax(reinterpret_cast<long long *>(pt + (unsigned long long)ws * pitch), pack_key(bb[ws], task_id));
    }
}

static __device__ __noinline__ void gpi_scan_wide8(uint32_t t_acc, uint32_t bias0, int col0_it, int c_begin, int c_end, int A_, int nw,
                                                  long long *ka, long long *kt, uint32_t kstep, bool row_ok, uint32_t task_id) {
    const int per_blk = A_ * 8;
    int blk = c_begin / per_blk;
    int act_i = (c_begin - blk * per_blk) >> 3;
    float bb[8];
    int ba[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { bb[i] = -INFINITY; ba[i] = 0; }
    const uint32_t pitch = kstep * 8u;                            // bytes between the key rows of consecutive reward vectors
    // key of reward vector blk * 8 for this thread's state (NULL stays NULL: gpi_emit8 tests it)
    char *pa = ka ? reinterpret_cast<char *>(ka) + (size_t)blk * 8u * pitch : nullptr;
    char *pt = kt ? reinterpret_cast<char *>(kt) + (size_t)blk * 8u * pitch : nullptr;
    auto emit = [&]() {
        if (row_ok)
            gpi_emit8(pa, pt, pitch, nw - blk * 8, task_id, bb[0], bb[1], bb[2], bb[3], bb[4], bb[5], bb[6], bb[7], ba[0], ba[1],
                      ba[2], ba[3], ba[4], ba[5], ba[6], ba[7]);
#pragma unroll
        for (int ws = 0; ws < 8; ++ws) { bb[ws] = -INFINITY; ba[ws] = 0; }
    };
    auto window = [&](const uint32_t (&u)[16], const float4 (&bz)[4]) {
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const float bv[8] = {bz[2 * j].x, bz[2 * j].y, bz[2 * j].z, bz[2 * j].w, bz[2 * j + 1].x, bz[2 * j + 1].y, bz[2 * j + 1].z, bz[2 * j + 1].w};
#pragma unroll
            for (int ws = 0; ws < 8; ++ws) {
                const float q = __uint_as_float(u[8 * j + ws]) + bv[ws];
                if (q > bb[ws]) ba[ws] = act_i;                  // (first index wins ties; a NaN never wins, as in the rolled scan)
                bb[ws] = fmaxf(bb[ws], q);
            }
            if (++act_i == A_) {                                 // block complete: 8 keys out, on to the next block
                emit();
                act_i = 0;
                ++blk;
                if (pa) pa += 8u * (size_t)pitch;
                if (pt) pt += 8u * (size_t)pitch;
            }
        }
    };
    uint32_t v[2][16];
    float4 bz[4];
    tmem_ld16(t_acc + (uint32_t)(c_begin - col0_it), v[0]);
#pragma unroll 1
    for (int c0 = c_begin; c0 < c_end; c0 += 32) {
#pragma unroll
        for (int i = 0; i < 4; ++i) bz[i] = lds128(bias0 + 4u * (uint32_t)(c0 + 4 * i));
        tmem_wait_ld();
        tmem_ld16(t_acc + (uint32_t)(c0 + 16 - col0_it), v[1]);
        window(v[0], bz);
#pragma unroll
        for (int i = 0; i < 4; ++i) bz[i] = lds128(bias0 + 4u * (uint32_t)(c0 + 16 + 4 * i));
        tmem_wait_ld();
        if (c0 + 32 < c_end) tmem_ld16(t_acc + (uint32_t)(c0 + 32 - col0_it), v[0]);
        window(v[1], bz);
    }
    if (act_i != 0) emit();                                      // the range ends inside a block: the rest of it merges by atomicMax
}

// Up to kMaxJobs independent forwards (e.g. online psi(s), GPI on s', target psi(s') of one train step) share ONE launch: the
// persistent tile loop runs over the concatenated pair lists, so the small per-step forwards fill the machine together
// instead of queueing as three single-wave kernels.
constexpr int kMaxJobs = 3;
struct TcMulti {
    long long *timeline;             // developer aid (env SFGPI_TIMELINE=1): clock64() stamps of CTA 0's roles, else NULL
    int n_jobs, total_pairs;
    int sched;                       // 1: work units come from the UnitTable (see below)
    int paired;                      // 1: two tiles ping-pong per CTA; 0: one tile per CTA (small launches), see kernel header
    int wide_min;                    // GPI scans of at least this many folded columns take gpi_scan_wide8
    int pair_start[kMaxJobs + 1];
    TcParams job[kMaxJobs];
};
struct TmapSet { CUtensorMap w[kMaxJobs]; CUtensorMap q[kMaxJobs]; CUtensorMap acts[kMaxJobs]; };

// Balanced schedule for mid-size launches (m.sched = 1): the host lists the work units explicitly -- ping-pong PAIRS of row
// tiles for the full rounds, then SINGLE tiles for the remainder -- so that no CTA is left with a whole extra pair while
// others idle (384 tiles on 148 SMs: pair + single everywhere instead of 2 pairs on 44 CTAs and 1 on 104).
// entry = job << 30 | has_y << 29 | policy << 16 | first tile.
constexpr int kMaxUnits = 1024;
struct UnitTable { uint32_t u[kMaxUnits]; };
struct Unit { int jb, pl, tile0; bool has_y; };


// role 0 = epilogue X (thread 0), 1 = MMA issuer, 2 = producer warp 0, 3 = epilogue Y (thread 0); 64 slots each
#define TL_STAMP(role, cnt) do { if (m.timeline != nullptr && blockIdx.x == 0 && (cnt) < 64) m.timeline[(role) * 64 + (cnt)++] = clock64(); } while (0)

// mlp_chain_tc.cu: the layer-pipelined single-tile kernel (the default for cta_group::1 launches)
bool forward_chain_supported(const TcMulti &m);
int launch_forward_chain(TcMulti &m, const TmapSet &maps, int total_tiles, cudaStream_t st);

}  // namespace tc
}  // namespace sfgpi
