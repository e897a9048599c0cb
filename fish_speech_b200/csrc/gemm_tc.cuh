// Generic multi-tap GEMM on the 5th-gen tensor cores (tcgen05.mma, accumulators in TMEM, operands
// staged by TMA with the 128-byte swizzle).  One kernel serves
//   * the Dual-AR decode step (weights = operand A on the TMEM lanes, the <=32 batch rows = operand B,
//     host-scheduled stream-K work items, fp32 partial sums reduced by the consuming kernel),
//   * LM prefill (same orientation, wide N tiles),
//   * the codec's Conv1d / ConvTranspose1d / Linear layers as implicit-im2col GEMMs: each conv tap is
//     a K-range whose activation tile is fetched by TMA at a shifted time coordinate; out-of-range
//     rows (the causal left pad) are zero-filled by the TMA unit itself.
//
//   D[z][i][j] = sum_tap sum_k  A[zA][i + a_shift[tap]][a_tapk*tap + k] * B[zB][j + b_shift[tap]][b_tapk*tap + k]
//
// i indexes TMEM lanes (128 per tile), j indexes TMEM columns (BN per tile).
#pragma once
#include "common.cuh"

namespace fsb {

enum GemmAct { ACT_NONE = 0, ACT_GELU = 1, ACT_TANH = 2 };

constexpr int kMaxTaps = 8;
constexpr int kMaxStages = 12;

struct GemmParams {
    // ---- K loop ----
    int kb_per_tap;  // 64-element k-blocks per tap
    int num_taps;
    int a_tapk, b_tapk;                        // k offset (elements) per tap
    int a_shift[kMaxTaps], b_shift[kMaxTaps];  // row shift per tap
    int a_batched, b_batched;                  // operand has a batch (z) coordinate
    unsigned long long a_hint, b_hint;         // L2 eviction policy per operand
    int stages;
    int a_static;  // operand A is constant data (weights): prefetch it before griddepcontrol.wait
    // ---- work decomposition ----
    const int4* sched;     // optional items {tile_i | tile_j<<16, kb_begin, kb_end, slot}; else blockIdx
    const int* cta_items;  // [grid.x + 1] item range of each CTA (stream-K)
    int tiled_total, tiled_ti, tiled_tj;  // persistent tiled mode: items = (z, tile_i, tile_j), tile_j fastest
    int rows_i, rows_j;  // valid output extents
    // ---- epilogue: mode 0 = fp32 partials ws[slot][j][i]; mode 1 = direct ----
    int mode;
    float* ws;
    long long ws_slot_stride;
    int ws_ld;
    void* out0;               // raw result (may be null)
    void* out1;               // snake-activated copy for the consuming conv (may be null)
    int out_f32;              // outputs are fp32 instead of bf16
    long long o_zs, o_is, o_js;  // element strides of out0/out1/resid
    int chan_on_i;            // per-channel vectors are indexed by i (else by j)
    const float* bias;        // [C] or null
    const float* gamma;       // [C] or null  (LayerScale / ConvNeXt gamma), applied after act
    const __nv_bfloat16* resid;  // same strides as out, added after gamma
    int act;                  // GemmAct applied to (acc + bias); TANH is applied last
    const float* snake_alpha;      // [C] for out1
    const float* snake_inv_alpha;  // [C] 1/(alpha+1e-9)
};

struct GemmOperand {
    const __nv_bfloat16* ptr;
    long long k;           // inner extent (elements) visible to TMA
    long long rows;        // row extent
    long long batch;       // batch extent (1 if none)
    long long row_stride;  // elements
    long long batch_stride;
};

struct GemmPlan {
    CUtensorMap tmA, tmB;
    GemmParams p;
    dim3 grid;
    int bn;
    size_t smem;
    void* sched_dev;  // owned (cudaMalloc) when stream-K scheduled
    int* cta_items_dev;
    int* nparts_dev;  // owned: partial count per i-tile
    int max_parts;
};

// Build the two tensor maps + launch geometry. `bn` in {32,64,128,256}. The caller fills the
// remaining GemmParams fields (taps, epilogue) in plan->p before/after this call.
int gemm_plan_init(GemmPlan* plan, const GemmOperand& A, const GemmOperand& B, int bn, int stages,
                   int tiles_i, int tiles_j, int batch);
// Host-scheduled stream-K for the skinny (decode) case: `tiles_i` x 1 output tiles, `kblocks`
// k-blocks each, spread evenly over `num_ctas` CTAs. Partials of tile t land in slots
// [0, nparts[t]) of the workspace.
int gemm_plan_streamk(GemmPlan* plan, int tiles_i, int kblocks, int num_ctas, bool keep_empty_ctas = false);
// Persistent tiled schedule (no table): tiles_i x tiles_j x batch full-K tiles spread over <= 2 CTAs per SM.
int gemm_plan_tiled(GemmPlan* plan, int tiles_i, int tiles_j, int batch, int ctas_per_sm = 1);
void gemm_plan_free(GemmPlan* plan);
int gemm_launch(const GemmPlan& plan, cudaStream_t stream);
int gemm_init();  // set kernel attributes (idempotent)
// 3-D {k, rows, batch} bf16 tensor map with the 128-byte swizzle and a {64, box_rows, 1} box.
int gemm_make_tmap(CUtensorMap* tm, const GemmOperand& op, int box_rows);

// csrc/codec_resunit.cu: a whole decoder ResidualUnit (modded_dac.py:599-620) as one kernel. d_a = Snake-activated
// input, d_x = raw residual stream, both bf16 [B][T][C]; w7 = [C][7][pad64(C)], w1 = [C][pad64(C)] bf16; out0 (raw, may
// alias d_x, may be null) and out1 = Snake_next(result) (must not alias d_a).
bool res_unit_supported(int C);
void res_unit_set_trace(unsigned long long* d_trace);  // diagnostics: [64][6] stamps of CTA 0 (null = off)
int res_unit_run(const void* d_a, const void* d_x, int B, int T, int C, int dilation, const void* d_w7,
                 const float* d_b7, const float* d_alpha1, const float* d_inv1, const void* d_w1, const float* d_b1,
                 void* d_out0, void* d_out1, const float* d_alpha_n, const float* d_inv_n, cudaStream_t st);

}  // namespace fsb
