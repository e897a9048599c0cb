// Step GEMM: the weight-streaming matmul of the Dual-AR decode step (llama.py:831-987 one TransformerBlock;
// inference.py:96-181 one frame).
//
//   D[i][j] = sum_k W[i][k] * X[j][k]        i = output feature (128 per tile, on the TMEM lanes)
//                                            j = sequence slot of the batch (<= 32, the UMMA N)
//
// Life of one launch (one CTA = 6 warps + 4 normaliser warps, two CTAs per SM, the whole grid in one wave):
//   1. The TMA producer requests the first ring-full of weight tiles at once -- before griddepcontrol.wait, i.e.
//      while the previous kernels are still finishing: weights do not depend on anything.
//   2. Main loop: weights HBM -> shared memory by TMA (SWIZZLE_128B, EVICT_FIRST), operand X by TMA from L2; where X
//      is the residual stream it is *normalised on load* -- four warps apply the reference's RMSNorm
//      (llama.py:990-1001: round(x * rsqrt(mean(x^2) + eps)) * w, two bf16 roundings) in place in shared memory, with
//      the per-row sum of squares the producer of the residual stream left behind -- and tcgen05.mma accumulates in
//      TMEM.  Work is a host-built stream-K schedule: (tile, k-block) units cut into equal contiguous ranges, one per
//      CTA, so every SM streams the same number of weight bytes whatever the shape.
//   3. Each CTA stores its fp32 partials and exits: no tail holds shared memory, so the next GEMM's CTAs move in and
//      start step 1 while this launch drains and its consumer runs.
// Whoever consumes the result finishes the GEMM: it sums the partials IN SLOT ORDER (deterministic, independent of
// arrival order and of the batch) and applies what the reference does next:
//   step_finalize (this file)  PRO_RESID   bias, residual add, new residual stream + per-128-feature sum of squares
//                                          for the next normalise-on-load                          (llama.py:842-845)
//                              PRO_SWIGLU  silu(w1 x) * w3 x on the row-interleaved w1|w3 result   (llama.py:979-987)
//   attention (lm_kernels.cuh) bias, per-head nn.RMSNorm, RoPE, KV append for the qkv GEMM          (llama.py:891-911)
//   sampler (lm_kernels.cuh)   bf16 logits of the two heads                                        (llama.py:447-457)
// Measured alternatives (profiles/r02_decode_structure.md): finishing a GEMM inside its own kernel (last-arriving CTA
// or all contributors after a per-tile arrival) or inside the consumer GEMM's prologue behind a grid-wide arrival
// were 6.2-7.2 ms per frame against 5.5 ms for this schedule: a tail or a prologue holds the shared memory the next
// GEMM's weight prefetch needs.
#pragma once
#include "gemm_tc.cuh"

namespace fsb {

enum StepPro { PRO_NONE = 0, PRO_RESID = 1, PRO_SWIGLU = 2 };

constexpr int kStepRows = 32;   // batch rows per step = UMMA N
constexpr int kSsqStride = 32;  // floats per row of a sum-of-squares array: one per 128-feature tile (D <= 4096)

// fp32 stream-K partials of one step GEMM:
//   value(row j, feature i) = sum_{q < nparts[i/128]} ws[((q*tiles + i/128)*32 + j)*128 + i%128]
struct StepPartials {
    const float* ws;
    const int* nparts;  // [tiles]
    int tiles;
    int n_out;      // output features (rows of the weight matrix)
    int max_parts;  // max over tiles of nparts: slots [0, max_parts) exist in ws for every tile
};

#ifdef __CUDACC__
// N output elements of one row at once, partials added in slot order: all loads of an 8-slot round are in flight
// together (N * 8 requests).  The loads are bounded by max_parts (a launch constant), not by each tile's count: they
// leave together with the load of the count instead of one round trip behind it; slots >= np hold stale data and are
// not added.
template <int N>
__device__ __forceinline__ void step_partial_sums(const StepPartials& P, int row, const int (&feat)[N], const bool (&ok)[N],
                                                  float (&out)[N]) {
    const size_t ss = static_cast<size_t>(P.tiles) * 32 * 128;
    int np[N];
    const float* p[N];
#pragma unroll
    for (int k = 0; k < N; ++k) {
        const int f = ok[k] ? feat[k] : 0;
        np[k] = ok[k] ? __ldg(P.nparts + (f >> 7)) : 0;
        p[k] = P.ws + (static_cast<size_t>(f >> 7) * 32 + row) * 128 + (f & 127);
        out[k] = 0.f;
    }
    for (int q = 0; q < P.max_parts; q += 8) {
        float a[N][8];
#pragma unroll
        for (int k = 0; k < N; ++k)
#pragma unroll
            for (int u = 0; u < 8; ++u)
                a[k][u] = (ok[k] && q + u < P.max_parts) ? __ldcg(p[k] + static_cast<size_t>(q + u) * ss) : 0.f;
#pragma unroll
        for (int k = 0; k < N; ++k)
#pragma unroll
            for (int u = 0; u < 8; ++u)
                if (q + u < np[k]) out[k] += a[k][u];
    }
}
#endif

struct StepGemmParams {
    // ---- schedule ----
    const int4* sched;      // items {tile, kb_begin, kb_end, slot}
    const int* cta_items;   // [grid + 1]
    int tiles, stages;
    int n_out, K;           // output features, reduction length
    int rows;               // live batch rows (<= 32)
    unsigned long long a_hint, b_hint;
    float* ws;              // out: [slot][tile][32 rows][128 features] fp32 partials
    // ---- step_finalize of the GEMM that produces this one's operand (pro != PRO_NONE) ----
    StepPartials prev;
    int prev_rb;                  // batch rows per finalize unit (power of two)
    const __nv_bfloat16* bias;    // PRO_RESID: [prev.n_out] or null
    const __nv_bfloat16* resid;   // PRO_RESID: [32][prev.n_out]; may alias x_out; null => no add
    __nv_bfloat16* x_out;         // PRO_RESID: [32][prev.n_out] new residual stream
    float* ssq_out;               // PRO_RESID: [32][kSsqStride]
    __nv_bfloat16* h;             // PRO_SWIGLU: [32][I]; prev tile t = features [64t, 64t+64): lanes 32w+l (l < 16) =
    int I;                        //             w1 row, lanes 32w+16+l = w3 row
    // ---- operand X by normalise-on-load (NORM = 1) ----
    const float* x_ssq;           // [32][kSsqStride] per-tile sum of squares of x
    const __nv_bfloat16* norm_w;  // [K]
    int x_nt;                     // tiles per row in x_ssq
    float eps;
    // diagnostics: optional [grid][8] globaltimer stamps {start, previous grid complete, -, -, first accumulator done,
    // end, normalisers ready, first tile normalised}
    unsigned long long* trace;
};

struct StepGemmPlan {
    CUtensorMap tmA, tmB;
    StepGemmParams p;
    dim3 grid;
    size_t smem;
    int pro, norm;
    void* sched_dev;
    int* cta_items_dev;
    int* nparts_dev;
    int max_parts;
    double weight_bytes;
};

// Operand X = act [32][K], fetched by TMA; norm_on_load: act is the un-normalised residual stream (the caller fills
// p.x_ssq / p.norm_w / p.x_nt / p.eps).
int step_plan_init(StepGemmPlan* plan, const __nv_bfloat16* w, int n_out, int K, const __nv_bfloat16* act,
                   bool norm_on_load, int num_ctas, int stages, float* ws, size_t ws_floats);
// the partials `plan` produces, as a consumer sees them
StepPartials step_plan_partials(const StepGemmPlan& plan);
// `plan`'s operand is the output of `prev` finished with `pro` (PRO_RESID / PRO_SWIGLU): records what
// step_finalize_launch(plan) has to do before `plan` runs (the caller fills bias / resid / x_out / ssq_out or h / I)
void step_plan_set_prev(StepGemmPlan* plan, int pro, const StepGemmPlan& prev);
void step_plan_free(StepGemmPlan* plan);
int step_gemm_launch(const StepGemmPlan& plan, cudaStream_t stream);
// finish the GEMM that produces `consumer`'s operand (no-op when consumer.pro == PRO_NONE); launch it before the consumer.
// rb: batch rows per finalize unit (power of two <= 32); 0 = the measured best (8 for SwiGLU, 2 for the residual add)
int step_finalize_launch(const StepGemmPlan& consumer, cudaStream_t stream, int rb = 0);
int step_gemm_init();  // kernel attributes (idempotent)

// Row index of the fused w1|w3 weight for SwiGLU: h feature f -> row of w1[f]; w3[f] sits 16 rows further.
__host__ __device__ inline int w13_gate_row(int f) { return (f >> 6) * 128 + ((f >> 4) & 3) * 32 + (f & 15); }

}  // namespace fsb
