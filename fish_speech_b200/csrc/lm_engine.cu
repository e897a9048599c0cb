// Dual-AR engine: owns the KV caches, workspaces and GEMM plans of one model replica and runs
// prefill / per-frame decode as a fixed kernel sequence (captured into a CUDA graph for decode).
//
// HBM layout (all bf16 unless noted)
//   weights            caller-owned, row-major [out, in] as in the checkpoint (TMA-ready, K-major); the fused
//                      w1|w3 matrix has its rows interleaved per 128-row tile (lm_gemm.cuh, w13_gate_row)
//   slow KV cache      [n_layer][max_batch][Hkv][kv_len][Dh]   x2 (K, V)
//   fast KV cache      [n_fast_layer][max_batch][fHkv][num_codebooks][fDh]  x2
//   decode state       residual streams x_slow / x_fast [32][D] + their per-128-feature sums of squares
//                      (fp32 [32][32]); q / attention / SwiGLU operands [32][*]; logits fp32 [32][n]
//   step_ws            fp32 stream-K partials of the step GEMMs: [slot][tile][32 rows][128 features]
//   prefill workspaces [max_rows][*] operands + ws fp32 [max_rows][N]
//
// One decode frame (inference.py:96-181) = embed, 36 x {qkv GEMM (norm on load), attention (finishes qkv: bias /
// qk-norm / RoPE / KV append), wo GEMM, finalize (residual add), w1|w3 GEMM (norm on load), finalize (SwiGLU), w2 GEMM,
// finalize (residual add)}, head GEMM + sampler, then 10 fast passes of 4 such layers each: ~640 kernels, eight per
// layer; every GEMM only stores fp32 partials, its consumer finishes it (lm_gemm.cuh).
//
// Reference: fish_speech/models/text2semantic/llama.py:390-466 (slow step), :799-817 (fast step),
// fish_speech/models/text2semantic/inference.py:96-181 (one frame), :184-238 (frame loop).
#include <algorithm>
#include <map>
#include <string>
#include <vector>

#include "../../include/fishb200.h"
#include "gemm_tc.cuh"
#include "lm_gemm.cuh"
#include "lm_kernels.cuh"

using namespace fsb;

namespace {

typedef __nv_bfloat16 bf16;
constexpr int kDecRows = kStepRows;  // decode GEMM N tile: up to 32 sequences per step
// step GEMM ring depth and resident CTAs per SM: measured best (profiles/r02_decode_structure.md item 7)
constexpr int kStepStages = 4;
constexpr int kStepCtasPerSm = 2;

struct LayerW {
    const bf16 *attn_norm, *wqkv, *bqkv, *q_norm, *k_norm, *wo, *bo, *ffn_norm, *w13, *w2;
};
struct StepLayer {
    StepGemmPlan qkv, wo, w13, w2;
};
struct PrefillLayer {
    GemmPlan qkv, wo, w13, w2;
    GemmPlan qkv_wide, w13_wide;  // the same GEMMs with 256-row tiles of the token rows (half the weight-tile traffic)
};

struct Stack {
    int D = 0, H = 0, Hkv = 0, Dh = 0, I = 0, nl = 0, S = 0;
    int n13 = 0;  // rows of the interleaved w1|w3 matrix: ceil(I / 64) * 128
    bool qk_norm = false;
    int bf16_math = 0;
    std::vector<LayerW> w;
    std::vector<StepLayer> dec;     // decode: fused step GEMMs
    std::vector<PrefillLayer> pf;   // prefill: BN=128 tiles, fp32 result + consumer kernels (slow only)
    bf16 *kcache = nullptr, *vcache = nullptr;
    const bf16* freqs = nullptr;
    size_t cache_layer_stride = 0;
    bf16* xres = nullptr;  // decode residual stream [32][D]
    float* ssq = nullptr;  // its per-tile sums of squares [32][kSsqStride]
};

}  // namespace

struct fsb_lm {
    // per-slot request control (continuous batching): see SlotCtl in lm_kernels.cuh
    bool slot_control = false;
    int* slot_state = nullptr;
    int* slot_limit = nullptr;
    float* slot_temperature = nullptr;
    float* slot_top_p = nullptr;
    int* slot_top_k = nullptr;
    unsigned long long* slot_seed = nullptr;
    bool graph_slot_control = false;
    fsb_lm_config cfg;
    int num_sms = 148;
    int step_ctas = 0;
    Stack slow, fast;
    const bf16 *emb = nullptr, *cb_emb = nullptr, *norm_w = nullptr, *head_w = nullptr;
    const bf16 *fast_emb = nullptr, *fast_norm_w = nullptr, *fast_out_w = nullptr;
    const bf16 *fast_proj_w = nullptr, *fast_proj_b = nullptr;
    int head_rows = 0;
    StepGemmPlan head_plan, head_plan_direct, fast_out_plan, proj_plan, fast_qkv0_proj;  // *_direct: operand already final
    bool has_proj = false;
    // decode workspaces
    bf16 *q_d = nullptr, *attn_d = nullptr, *h_d = nullptr, *hid_d = nullptr;
    float* step_ws = nullptr;
    size_t step_ws_floats = 0;
    // prefill workspaces
    bf16 *xres_p = nullptr, *xn_p = nullptr, *q_p = nullptr, *attn_p = nullptr, *h_p = nullptr;
    float* ws = nullptr;
    size_t ws_floats = 0;
    // state
    int *cur_tok = nullptr, *out_tokens = nullptr, *n_out = nullptr, *pos = nullptr, *finished = nullptr;
    int *ras_window = nullptr, *iota = nullptr, *fpos = nullptr;
    unsigned long long* step = nullptr;
    // debug / test hooks
    float *slow_logits = nullptr, *fast_logits = nullptr;
    const float* noise_u = nullptr;
    int noise_draws = 0, noise_ld = 0;
    int ctx_lcap = 0;  // score-buffer bound for the slow attention (0 = capacity)
    unsigned long long* trace_base = nullptr;  // fsb_lm_trace_frame: per-CTA stamps of every step GEMM of one frame
    int trace_next = 0, trace_max = 0;
    unsigned long long* attn_trace_base = nullptr;  // 8 stamps of CTA (0, 0) of every decode attention launch
    int attn_trace_next = 0, attn_trace_max = 0;
    int graph_lcap = -1;
    // decode graph cache
    cudaGraphExec_t graph_exec = nullptr;
    int graph_batch = -1;
    int graph_kernels = 0;  // kernels inside one captured frame
    const float* graph_noise = nullptr;
    fsb_sampling graph_sampling{};
    std::vector<void*> owned;
    std::map<std::string, std::pair<void*, size_t>> named;
};

namespace {

template <typename T>
int dalloc(fsb_lm* h, T** p, size_t count, const char* name = nullptr) {
    void* q = nullptr;
    const size_t bytes = std::max<size_t>(count * sizeof(T), 256);
    FSB_CUDA(cudaMalloc(&q, bytes));
    FSB_CUDA(cudaMemset(q, 0, bytes));
    h->owned.push_back(q);
    *p = reinterpret_cast<T*>(q);
    if (name) h->named[name] = {q, count * sizeof(T)};
    return 0;
}

// Prefill plan: A = weight [n_out, k] on the TMEM lanes, B = activations [rows, k], fp32 result ws[row][n_out].
int make_prefill_plan(fsb_lm* h, GemmPlan* plan, const bf16* w, int n_out, int k, const bf16* act, int act_rows,
                      int bn = 128) {
    memset(plan, 0, sizeof(*plan));
    GemmOperand A{w, k, n_out, 1, k, static_cast<long long>(n_out) * k};
    GemmOperand B{act, k, act_rows, 1, k, static_cast<long long>(act_rows) * k};
    GemmParams& p = plan->p;
    p.kb_per_tap = cdiv(k, 64);
    p.num_taps = 1;
    p.a_hint = kEvictNormal;
    p.a_static = 1;
    p.b_hint = kEvictLast;
    p.rows_i = n_out;
    p.mode = 0;
    p.ws = h->ws;
    p.ws_ld = n_out;
    FSB_TRY(gemm_plan_init(plan, A, B, bn, 4, cdiv(n_out, 128), cdiv(act_rows, bn), 1));
    p.rows_j = act_rows;
    p.ws_slot_stride = 0;
    FSB_CHECK(static_cast<size_t>(act_rows) * n_out <= h->ws_floats, "prefill workspace too small");
    return 0;
}

// 256-row tiles once enough token rows exist to fill the SMs with them: per output element the K loop is the same
// sequence of MMAs, so the result does not depend on the tile width (chunked prefill == one pass stays bit-exact)
int launch_rows_of(const GemmPlan& plan, const GemmPlan& wide, int rows, cudaStream_t st);
int launch_rows_of(const GemmPlan& plan, int rows, cudaStream_t st) {
    GemmPlan q = plan;  // restrict the column tiles to the live rows
    q.grid.y = cdiv(rows, plan.bn);
    q.p.rows_j = rows;
    return gemm_launch(q, st);
}

int launch_rows_of(const GemmPlan& plan, const GemmPlan& wide, int rows, cudaStream_t st) {
    const long long tiles_wide = static_cast<long long>(wide.grid.x) * cdiv(rows, 256);
    return (rows >= 512 && tiles_wide >= 296) ? launch_rows_of(wide, rows, st) : launch_rows_of(plan, rows, st);
}

// Step GEMM over the weight `w` [n_out, K]. act != null: operand X = act, used as it is; act == null: operand X = the
// stack's residual stream, normalised on load (bind_norm_on_load supplies the norm).
int make_step_plan(fsb_lm* h, StepGemmPlan* plan, const bf16* w, int n_out, int K, const bf16* act,
                   const Stack* norm_of = nullptr) {
    const bool norm = act == nullptr;
    if (norm) act = norm_of->xres;
    return step_plan_init(plan, w, n_out, K, act, norm, h->step_ctas, kStepStages, h->step_ws, h->step_ws_floats);
}

// Finish the GEMM that produces `plan`'s operand (residual add / SwiGLU), then launch `plan` itself over `rows` batch
// rows; under fsb_lm_trace_frame the step GEMM records its per-CTA stamps.
int launch_step(fsb_lm* h, const StepGemmPlan& plan, int rows, cudaStream_t st) {
    StepGemmPlan q = plan;
    q.p.rows = rows;
    FSB_TRY(step_finalize_launch(q, st));
    if (h->trace_base && h->trace_next < h->trace_max && q.grid.x <= 512)
        q.p.trace = h->trace_base + static_cast<size_t>(h->trace_next++) * 8 * 512;
    return step_gemm_launch(q, st);
}

void bind_norm_on_load(StepGemmPlan* plan, const Stack& s, const bf16* norm_w, float eps) {
    plan->p.x_ssq = s.ssq;
    plan->p.norm_w = norm_w;
    plan->p.x_nt = cdiv(s.D, 128);
    plan->p.eps = eps;
}

// `plan` reads the residual stream of stack s after `prev` (a Linear) has been added to it: PRO_RESID finalize of prev
void bind_resid(StepGemmPlan* plan, const StepGemmPlan& prev, const Stack& s, const bf16* bias, bool add_residual) {
    step_plan_set_prev(plan, PRO_RESID, prev);
    plan->p.bias = bias;
    plan->p.resid = add_residual ? s.xres : nullptr;
    plan->p.x_out = s.xres;
    plan->p.ssq_out = s.ssq;
}

SlotCtl slot_ctl(const fsb_lm* h) {
    SlotCtl c{};
    if (!h->slot_control) return c;
    c.state = h->slot_state;
    c.limit = h->slot_limit;
    c.temperature = h->slot_temperature;
    c.top_p = h->slot_top_p;
    c.top_k = h->slot_top_k;
    c.seed = h->slot_seed;
    c.n_out = h->n_out;
    return c;
}

// ---- decode: one transformer stack over the batch rows, five kernels per layer. `first_qkv`: the plan of layer 0's
// qkv GEMM when its operand is produced by a GEMM (fast_project_in) instead of a row kernel. After the last layer the
// residual stream is complete only once the NEXT step GEMM (head / fast_output) has run its prologue. ----
int run_stack_decode(fsb_lm* h, Stack& s, int rows, const int* row_seq, const int* row_pos, bool stop_after_kv,
                     cudaStream_t st, const StepGemmPlan* first_qkv = nullptr) {
    const float eps = h->cfg.norm_eps;
    for (int l = 0; l < s.nl; ++l) {
        StepLayer& P = s.dec[l];
        const LayerW& w = s.w[l];
        const StepGemmPlan& qkv = (l == 0 && first_qkv) ? *first_qkv : P.qkv;
        FSB_TRY(launch_step(h, qkv, rows, st));
        AttnDecodeArgs aa{};
        aa.qkv = step_plan_partials(qkv);
        aa.bias = w.bqkv;
        aa.q_norm = s.qk_norm ? w.q_norm : nullptr;
        aa.k_norm = s.qk_norm ? w.k_norm : nullptr;
        aa.freqs = s.freqs;
        aa.kcache = s.kcache + l * s.cache_layer_stride;
        aa.vcache = s.vcache + l * s.cache_layer_stride;
        aa.row_seq = row_seq;
        aa.row_pos = row_pos;
        aa.out = h->attn_d;
        aa.rows = rows; aa.H = s.H; aa.Hkv = s.Hkv; aa.Dh = s.Dh; aa.S = s.S;
        aa.lcap = (s.bf16_math == 0) ? h->ctx_lcap : 0;  // slow stack: bounded by the live context, not the capacity
        aa.bf16_math = s.bf16_math;
        aa.kv_only = (stop_after_kv && l == s.nl - 1) ? 1 : 0;  // fast pass 0 only fills the KV cache (inference.py:147)
        aa.eps = eps;
        if (h->attn_trace_base && h->attn_trace_next < h->attn_trace_max)
            aa.trace = h->attn_trace_base + static_cast<size_t>(h->attn_trace_next++) * 8;
        FSB_TRY(launch_attn_decode(aa, st));
        if (aa.kv_only) return 0;
        FSB_TRY(launch_step(h, P.wo, rows, st));
        FSB_TRY(launch_step(h, P.w13, rows, st));
        FSB_TRY(launch_step(h, P.w2, rows, st));
    }
    return 0;
}

// ---- prefill: the same stack over `rows` token rows with wide-N tensor-core GEMMs and consumer kernels.
// On entry xn_p = attention_norm_0(xres_p). ----
int run_stack_prefill(fsb_lm* h, Stack& s, int rows, const int* row_seq, const int* row_pos, cudaStream_t st) {
    const float eps = h->cfg.norm_eps;
    const int Nqkv = (s.H + 2 * s.Hkv) * s.Dh;
    for (int l = 0; l < s.nl; ++l) {
        const LayerW& w = s.w[l];
        PrefillLayer& P = s.pf[l];
        FSB_TRY(launch_rows_of(P.qkv, P.qkv_wide, rows, st));
        QkvPrepArgs qa{};
        qa.y = h->ws; qa.ld = Nqkv;
        qa.bias = w.bqkv;
        qa.q_norm = s.qk_norm ? w.q_norm : nullptr;
        qa.k_norm = s.qk_norm ? w.k_norm : nullptr;
        qa.freqs = s.freqs;
        qa.row_seq = row_seq;
        qa.row_pos = row_pos;
        qa.q = h->q_p;
        qa.kcache = s.kcache + l * s.cache_layer_stride;
        qa.vcache = s.vcache + l * s.cache_layer_stride;
        qa.rows = rows; qa.H = s.H; qa.Hkv = s.Hkv; qa.Dh = s.Dh; qa.S = s.S;
        qa.eps = eps;
        FSB_TRY(launch_qkv_prep(qa, st));
        AttnArgs aa{};
        aa.q = h->q_p;
        aa.kcache = qa.kcache;
        aa.vcache = qa.vcache;
        aa.row_seq = row_seq;
        aa.row_pos = row_pos;
        aa.out = h->attn_p;
        aa.rows = rows; aa.H = s.H; aa.Hkv = s.Hkv; aa.Dh = s.Dh; aa.S = s.S;
        aa.window = 0;
        FSB_TRY(launch_attn(aa, st));
        FSB_TRY(launch_rows_of(P.wo, rows, st));
        ResidNormArgs r1{};
        r1.y = h->ws; r1.ld = s.D;
        r1.bias = w.bo;
        r1.x_in = h->xres_p; r1.x_out = h->xres_p;
        r1.norm_w = w.ffn_norm; r1.n_out = h->xn_p;
        r1.rows = rows; r1.D = s.D; r1.eps = eps;
        FSB_TRY(launch_resid_norm(r1, st));
        FSB_TRY(launch_rows_of(P.w13, P.w13_wide, rows, st));
        SwigluArgs sa{};
        sa.y = h->ws; sa.ld = s.n13;
        sa.h = h->h_p; sa.rows = rows; sa.I = s.I;
        sa.interleaved = 1;
        FSB_TRY(launch_swiglu(sa, st));
        FSB_TRY(launch_rows_of(P.w2, rows, st));
        ResidNormArgs r2{};
        r2.y = h->ws; r2.ld = s.D;
        r2.x_in = h->xres_p; r2.x_out = h->xres_p;
        // the final norm is applied by the head GEMM's normalise-on-load on the last-token rows only
        r2.norm_w = (l + 1 < s.nl) ? s.w[l + 1].attn_norm : nullptr;
        r2.n_out = h->xn_p;
        r2.rows = rows; r2.D = s.D; r2.eps = eps;
        FSB_TRY(launch_resid_norm(r2, st));
    }
    return 0;
}

// Head + sampling + fast passes + bookkeeping for `rows` sequences whose last residual-stream rows (un-normed)
// are in slow.xres[0..rows) with their sums of squares in slow.ssq. inference.py:114-181.
int run_frame_tail(fsb_lm* h, int rows, const int* row_slot, bool use_ras, const int* set_pos_rows,
                   const int* row_pos_src, const fsb_sampling& sp, cudaStream_t st, bool x_is_final = false) {
    const fsb_lm_config& c = h->cfg;
    const int C = c.num_codebooks;
    const int* slots = row_slot ? row_slot : h->iota;
    Stack& s = h->slow;
    Stack& f = h->fast;
    auto sample_args = [&](int n, const StepGemmPlan& head) {
        SampleArgs a{};
        a.ctl = slot_ctl(h);
        a.parts = step_plan_partials(head);
        a.n = n;
        a.rows = rows;
        a.temperature = sp.temperature; a.top_p = sp.top_p; a.top_k = sp.top_k;
        a.seed = sp.seed;
        a.rng_offset = h->step;
        a.cur_tok = h->cur_tok;
        a.num_cb = C;
        a.row_slot = row_slot;
        a.noise_u = h->noise_u;
        a.noise_draws = h->noise_draws;
        a.noise_ld = h->noise_ld;
        return a;
    };
    // ---- slow head over the selectable rows (first the last layer's FFN output is added to the residual stream,
    // unless the rows come from a prefill; the final norm is applied on load) ----
    const StepGemmPlan& head = x_is_final ? h->head_plan_direct : h->head_plan;
    FSB_TRY(launch_step(h, head, rows, st));
    SampleArgs sa = sample_args(h->head_rows, head);
    sa.slow = 1;
    sa.n_sem = h->head_rows - 1;
    sa.sem_begin = c.semantic_begin_id;
    sa.im_end_id = c.im_end_id;
    sa.codebook_size = c.codebook_size;
    sa.use_ras = use_ras ? 1 : 0;
    sa.ras_window = h->ras_window;
    sa.ras_update = use_ras ? 1 : 0;
    sa.draw_id = 0;
    sa.cb_index = 0;
    sa.logits_out = h->slow_logits;
    sa.finished = h->finished;
    FSB_TRY(launch_sample(sa, st));

    // ---- fast pass 0 input: hidden = norm(x) (norm_fastlayer_input) [-> fast_project_in]  (llama.py:459-461, 819-828)
    RowsArgs hr{};
    hr.x = s.xres;
    hr.ssq_in = s.ssq;
    hr.norm_w = c.norm_fastlayer_input ? h->norm_w : nullptr;
    hr.rows = rows; hr.D = s.D; hr.eps = c.norm_eps;
    if (h->has_proj) {
        hr.y = h->hid_d;
        FSB_TRY(launch_rows(hr, st));
        // fast_project_in; the finalize in front of layer 0's qkv GEMM adds the bias
        FSB_TRY(launch_step(h, h->proj_plan, rows, st));
    } else {
        hr.y = f.xres;
        hr.ssq = f.ssq;
        FSB_TRY(launch_rows(hr, st));
    }
    for (int p = 0; p < C; ++p) {
        if (p > 0) {
            // input = fast_embeddings[code_{p-1}] ; codes live in cur_tok[slot][p]
            RowsArgs er{};
            er.x = h->fast_emb;
            er.y = f.xres;
            er.ssq = f.ssq;
            er.gather = h->cur_tok + p;
            er.gather_map = row_slot;
            er.gather_stride = C + 1;
            er.rows = rows; er.D = f.D; er.eps = c.norm_eps;
            FSB_TRY(launch_rows(er, st));
        }
        FSB_TRY(run_stack_decode(h, f, rows, slots, h->fpos + p * kDecRows, p == 0, st,
                                 (p == 0 && h->has_proj) ? &h->fast_qkv0_proj : nullptr));
        if (p == 0) continue;
        FSB_TRY(launch_step(h, h->fast_out_plan, rows, st));
        SampleArgs fa = sample_args(c.codebook_size, h->fast_out_plan);
        fa.slow = 0;
        fa.draw_id = p;
        fa.cb_index = p;
        fa.logits_out = h->fast_logits ? h->fast_logits + static_cast<size_t>(p - 1) * c.max_batch * c.codebook_size
                                       : nullptr;
        FSB_TRY(launch_sample(fa, st));
    }
    FrameEndArgs fe{};
    fe.ctl = slot_ctl(h);
    fe.cur_tok = h->cur_tok;
    fe.out_tokens = h->out_tokens;
    fe.n_out = h->n_out;
    fe.pos = h->pos;
    fe.row_slot = row_slot;
    fe.set_pos_rows = set_pos_rows;
    fe.row_pos_src = row_pos_src;
    fe.step = h->step;
    fe.rows = rows; fe.ncols = C + 1; fe.T_cap = c.max_frames;
    FSB_TRY(launch_frame_end(fe, st));
    return 0;
}

EmbedArgs embed_args(fsb_lm* h, const int* tokens, bf16* x, float* ssq, int rows) {
    const fsb_lm_config& c = h->cfg;
    EmbedArgs ea{};
    ea.tokens = tokens;
    ea.emb = h->emb; ea.cb_emb = h->cb_emb; ea.x = x; ea.ssq = ssq;
    ea.rows = rows; ea.D = h->slow.D; ea.C = c.num_codebooks; ea.cs = c.codebook_size; ea.vocab = c.vocab_size;
    ea.sem_begin = c.semantic_begin_id; ea.sem_end = c.semantic_end_id;
    ea.scale = c.scale_codebook_embeddings;
    return ea;
}

int decode_one_frame(fsb_lm* h, int batch, const fsb_sampling& sp, cudaStream_t st) {
    Stack& s = h->slow;
    FSB_TRY(launch_embed(embed_args(h, h->cur_tok, s.xres, s.ssq, batch), st));
    FSB_TRY(run_stack_decode(h, s, batch, h->iota, h->pos, false, st));
    return run_frame_tail(h, batch, nullptr, true, nullptr, nullptr, sp, st);
}

size_t step_ws_bound(int n_out, int ctas) {
    const int tiles = cdiv(n_out, 128);
    return static_cast<size_t>(tiles) * (cdiv(ctas, tiles) + 2) * 128 * 32;
}

}  // namespace

extern "C" {

int fsb_lm_create(const fsb_lm_config* cfg, const fsb_lm_weights* w, fsb_lm** out) {
    FSB_CHECK(cfg && w && out, "fsb_lm_create: null argument");
    FSB_CHECK(cfg->max_batch >= 1 && cfg->max_batch <= kDecRows, "max_batch must be in [1,32]");
    FSB_CHECK(cfg->dim % 8 == 0 && cfg->fast_dim % 8 == 0 && cfg->intermediate % 16 == 0 &&
                  cfg->fast_intermediate % 16 == 0,
              "dims must be multiples of 8, intermediate sizes of 16 (TMA 16-byte strides, SwiGLU interleave)");
    FSB_CHECK(cfg->dim <= 4096 && cfg->fast_dim <= 4096, "model dim above 4096 is not supported");
    FSB_CHECK((cfg->head_dim == 64 || cfg->head_dim == 128) && (cfg->fast_head_dim == 64 || cfg->fast_head_dim == 128),
              "head_dim must be 64 or 128");
    FSB_CHECK(w->head_rows == cfg->semantic_end_id - cfg->semantic_begin_id + 2, "head_rows mismatch");
    fsb_lm* h = new fsb_lm();
    h->cfg = *cfg;
    int dev = 0;
    cudaDeviceProp prop;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaGetDeviceProperties(&prop, dev) != cudaSuccess) {
        set_error("fsb_lm_create: no CUDA device");
        delete h;
        return 1;
    }
    if (prop.major != 10) {
        set_error("fishb200 kernels are built for sm_100a only (device is sm_%d%d)", prop.major, prop.minor);
        delete h;
        return 1;
    }
    h->num_sms = prop.multiProcessorCount;
    if (gemm_init() != 0 || attn_init() != 0 || step_gemm_init() != 0) {
        delete h;
        return 1;
    }
    h->step_ctas = h->num_sms * kStepCtasPerSm;

    auto B16 = [](const void* p) { return reinterpret_cast<const bf16*>(p); };
    h->emb = B16(w->d_embeddings);
    h->cb_emb = B16(w->d_codebook_embeddings);
    h->norm_w = B16(w->d_norm);
    h->head_w = B16(w->d_head);
    h->head_rows = w->head_rows;
    h->fast_emb = B16(w->d_fast_embeddings);
    h->fast_norm_w = B16(w->d_fast_norm);
    h->fast_out_w = B16(w->d_fast_output);
    h->fast_proj_w = B16(w->d_fast_proj_w);
    h->fast_proj_b = B16(w->d_fast_proj_b);
    h->has_proj = w->d_fast_proj_w != nullptr;

    Stack& s = h->slow;
    s.D = cfg->dim; s.H = cfg->n_head; s.Hkv = cfg->n_kv_head; s.Dh = cfg->head_dim; s.I = cfg->intermediate;
    s.nl = cfg->n_layer; s.S = cfg->kv_len; s.qk_norm = cfg->qk_norm != 0; s.bf16_math = 0;
    s.n13 = cdiv(s.I, 64) * 128;
    s.freqs = B16(w->d_freqs);
    Stack& f = h->fast;
    f.D = cfg->fast_dim; f.H = cfg->fast_n_head; f.Hkv = cfg->fast_n_kv_head; f.Dh = cfg->fast_head_dim;
    f.I = cfg->fast_intermediate; f.nl = cfg->n_fast_layer; f.S = cfg->num_codebooks;
    f.qk_norm = cfg->fast_qk_norm != 0; f.bf16_math = 1;
    f.n13 = cdiv(f.I, 64) * 128;
    f.freqs = B16(w->d_fast_freqs);
    auto copy_layers = [&](Stack& st, const fsb_lm_layer* L) {
        st.w.resize(st.nl);
        for (int l = 0; l < st.nl; ++l) {
            st.w[l] = LayerW{B16(L[l].d_attn_norm), B16(L[l].d_wqkv), B16(L[l].d_bqkv), B16(L[l].d_q_norm),
                            B16(L[l].d_k_norm), B16(L[l].d_wo), B16(L[l].d_bo), B16(L[l].d_ffn_norm),
                            B16(L[l].d_w13), B16(L[l].d_w2)};
        }
    };
    copy_layers(s, w->layers);
    copy_layers(f, w->fast_layers);

    const int C = cfg->num_codebooks;
    const int Dm = std::max(s.D, f.D), Qm = std::max(s.H * s.Dh, f.H * f.Dh), Im = std::max(s.I, f.I);
    const int Nqkv_s = (s.H + 2 * s.Hkv) * s.Dh, Nqkv_f = (f.H + 2 * f.Hkv) * f.Dh;
    const int R = std::max(cfg->max_rows, 128);
    h->ws_floats = static_cast<size_t>(R) * std::max({Nqkv_s, s.n13, s.D});
    h->step_ws_floats = 0;
    for (int n : {Nqkv_s, Nqkv_f, s.n13, f.n13, s.D, f.D, h->head_rows, cfg->codebook_size})
        h->step_ws_floats = std::max(h->step_ws_floats, step_ws_bound(n, h->step_ctas));
#define TRYC(x)                  \
    do {                         \
        if ((x) != 0) {          \
            fsb_lm_destroy(h);   \
            return 1;            \
        }                        \
    } while (0)
    TRYC(dalloc(h, &h->ws, h->ws_floats));
    TRYC(dalloc(h, &h->step_ws, h->step_ws_floats));
    TRYC(dalloc(h, &s.xres, static_cast<size_t>(kDecRows) * s.D));
    TRYC(dalloc(h, &s.ssq, static_cast<size_t>(kDecRows) * kSsqStride));
    TRYC(dalloc(h, &f.xres, static_cast<size_t>(kDecRows) * f.D));
    TRYC(dalloc(h, &f.ssq, static_cast<size_t>(kDecRows) * kSsqStride));
    TRYC(dalloc(h, &h->hid_d, static_cast<size_t>(kDecRows) * Dm));
    TRYC(dalloc(h, &h->q_d, static_cast<size_t>(kDecRows) * Qm));
    TRYC(dalloc(h, &h->attn_d, static_cast<size_t>(kDecRows) * Qm));
    TRYC(dalloc(h, &h->h_d, static_cast<size_t>(kDecRows) * Im));
    TRYC(dalloc(h, &h->xres_p, static_cast<size_t>(R) * s.D));
    TRYC(dalloc(h, &h->xn_p, static_cast<size_t>(R) * s.D));
    TRYC(dalloc(h, &h->q_p, static_cast<size_t>(R) * s.H * s.Dh));
    TRYC(dalloc(h, &h->attn_p, static_cast<size_t>(R) * s.H * s.Dh));
    TRYC(dalloc(h, &h->h_p, static_cast<size_t>(R) * s.I));
    s.cache_layer_stride = static_cast<size_t>(cfg->max_batch) * s.Hkv * s.S * s.Dh;
    f.cache_layer_stride = static_cast<size_t>(cfg->max_batch) * f.Hkv * f.S * f.Dh;
    TRYC(dalloc(h, &s.kcache, s.cache_layer_stride * s.nl));
    TRYC(dalloc(h, &s.vcache, s.cache_layer_stride * s.nl));
    TRYC(dalloc(h, &f.kcache, f.cache_layer_stride * f.nl));
    TRYC(dalloc(h, &f.vcache, f.cache_layer_stride * f.nl));
    TRYC(dalloc(h, &h->cur_tok, static_cast<size_t>(cfg->max_batch) * (C + 1), "cur_tok"));
    TRYC(dalloc(h, &h->out_tokens, static_cast<size_t>(cfg->max_batch) * (C + 1) * cfg->max_frames, "out_tokens"));
    TRYC(dalloc(h, &h->n_out, cfg->max_batch, "n_out"));
    TRYC(dalloc(h, &h->pos, kDecRows, "pos"));
    TRYC(dalloc(h, &h->finished, cfg->max_batch, "finished"));
    TRYC(dalloc(h, &h->ras_window, static_cast<size_t>(cfg->max_batch) * 10, "ras_window"));
    TRYC(dalloc(h, &h->slot_state, cfg->max_batch, "slot_state"));
    TRYC(dalloc(h, &h->slot_limit, cfg->max_batch, "slot_limit"));
    TRYC(dalloc(h, &h->slot_temperature, cfg->max_batch, "slot_temperature"));
    TRYC(dalloc(h, &h->slot_top_p, cfg->max_batch, "slot_top_p"));
    TRYC(dalloc(h, &h->slot_top_k, cfg->max_batch, "slot_top_k"));
    TRYC(dalloc(h, &h->slot_seed, cfg->max_batch, "slot_seed"));
    TRYC(dalloc(h, &h->iota, kDecRows));
    TRYC(dalloc(h, &h->fpos, static_cast<size_t>(C) * kDecRows));
    TRYC(dalloc(h, &h->step, 1));
    if (cfg->debug) {
        TRYC(dalloc(h, &h->slow_logits, static_cast<size_t>(cfg->max_batch) * h->head_rows, "slow_logits"));
        TRYC(dalloc(h, &h->fast_logits, static_cast<size_t>(C) * cfg->max_batch * cfg->codebook_size, "fast_logits"));
    }
    {
        std::vector<int> io(kDecRows), fp(static_cast<size_t>(C) * kDecRows);
        for (int i = 0; i < kDecRows; ++i) io[i] = i;
        for (int p = 0; p < C; ++p)
            for (int i = 0; i < kDecRows; ++i) fp[p * kDecRows + i] = p;
        if (cudaMemcpy(h->iota, io.data(), io.size() * 4, cudaMemcpyHostToDevice) != cudaSuccess ||
            cudaMemcpy(h->fpos, fp.data(), fp.size() * 4, cudaMemcpyHostToDevice) != cudaSuccess) {
            set_error("fsb_lm_create: state upload failed");
            fsb_lm_destroy(h);
            return 1;
        }
    }
    // ---- GEMM plans ----
    const float eps = cfg->norm_eps;
    auto build = [&](Stack& st, bool with_prefill) -> int {
        st.dec.resize(st.nl);
        if (with_prefill) st.pf.resize(st.nl);
        const int Nqkv = (st.H + 2 * st.Hkv) * st.Dh;
        for (int l = 0; l < st.nl; ++l) {
            const LayerW& lw = st.w[l];
            StepLayer& P = st.dec[l];
            // qkv: layer 0 reads a residual stream a row kernel wrote; later layers first add the previous FFN output
            FSB_TRY(make_step_plan(h, &P.qkv, lw.wqkv, Nqkv, st.D, nullptr, &st));
            bind_norm_on_load(&P.qkv, st, lw.attn_norm, eps);
            if (l > 0) bind_resid(&P.qkv, st.dec[l - 1].w2, st, nullptr, true);
            FSB_TRY(make_step_plan(h, &P.wo, lw.wo, st.D, st.H * st.Dh, h->attn_d));
            FSB_TRY(make_step_plan(h, &P.w13, lw.w13, st.n13, st.D, nullptr, &st));
            bind_norm_on_load(&P.w13, st, lw.ffn_norm, eps);
            bind_resid(&P.w13, P.wo, st, lw.bo, true);
            FSB_TRY(make_step_plan(h, &P.w2, lw.w2, st.D, st.I, h->h_d));
            step_plan_set_prev(&P.w2, PRO_SWIGLU, P.w13);
            P.w2.p.h = h->h_d;
            P.w2.p.I = st.I;
            if (with_prefill) {
                FSB_TRY(make_prefill_plan(h, &st.pf[l].qkv, lw.wqkv, Nqkv, st.D, h->xn_p, R));
                FSB_TRY(make_prefill_plan(h, &st.pf[l].wo, lw.wo, st.D, st.H * st.Dh, h->attn_p, R));
                FSB_TRY(make_prefill_plan(h, &st.pf[l].w13, lw.w13, st.n13, st.D, h->xn_p, R));
                FSB_TRY(make_prefill_plan(h, &st.pf[l].qkv_wide, lw.wqkv, Nqkv, st.D, h->xn_p, R, 256));
                FSB_TRY(make_prefill_plan(h, &st.pf[l].w13_wide, lw.w13, st.n13, st.D, h->xn_p, R, 256));
                FSB_TRY(make_prefill_plan(h, &st.pf[l].w2, lw.w2, st.D, st.I, h->h_p, R));
            }
        }
        return 0;
    };
    TRYC(build(s, true));
    TRYC(build(f, false));
    TRYC(make_step_plan(h, &h->head_plan, h->head_w, h->head_rows, s.D, nullptr, &s));
    bind_norm_on_load(&h->head_plan, s, h->norm_w, eps);
    bind_resid(&h->head_plan, s.dec[s.nl - 1].w2, s, nullptr, true);
    TRYC(make_step_plan(h, &h->head_plan_direct, h->head_w, h->head_rows, s.D, nullptr, &s));
    bind_norm_on_load(&h->head_plan_direct, s, h->norm_w, eps);
    TRYC(make_step_plan(h, &h->fast_out_plan, h->fast_out_w, cfg->codebook_size, f.D, nullptr, &f));
    bind_norm_on_load(&h->fast_out_plan, f, h->fast_norm_w, eps);
    bind_resid(&h->fast_out_plan, f.dec[f.nl - 1].w2, f, nullptr, true);
    if (h->has_proj) {
        TRYC(make_step_plan(h, &h->proj_plan, h->fast_proj_w, f.D, s.D, h->hid_d));
        // fast layer 0 of pass 0: its operand = fast_project_in(hidden) + bias, finished in the qkv GEMM's prologue
        const LayerW& l0 = f.w[0];
        TRYC(make_step_plan(h, &h->fast_qkv0_proj, l0.wqkv, (f.H + 2 * f.Hkv) * f.Dh, f.D, nullptr, &f));
        bind_norm_on_load(&h->fast_qkv0_proj, f, l0.attn_norm, eps);
        bind_resid(&h->fast_qkv0_proj, h->proj_plan, f, h->fast_proj_b, false);
    }
#undef TRYC
    *out = h;
    return 0;
}

void fsb_lm_destroy(fsb_lm* h) {
    if (!h) return;
    if (h->graph_exec) cudaGraphExecDestroy(h->graph_exec);
    auto free_plans = [](Stack& st) {
        for (auto& p : st.dec) { step_plan_free(&p.qkv); step_plan_free(&p.wo); step_plan_free(&p.w13); step_plan_free(&p.w2); }
        for (auto& p : st.pf) { gemm_plan_free(&p.qkv); gemm_plan_free(&p.wo); gemm_plan_free(&p.w13); gemm_plan_free(&p.w2); gemm_plan_free(&p.qkv_wide); gemm_plan_free(&p.w13_wide); }
    };
    free_plans(h->slow);
    free_plans(h->fast);
    step_plan_free(&h->head_plan);
    step_plan_free(&h->head_plan_direct);
    step_plan_free(&h->fast_out_plan);
    if (h->has_proj) {
        step_plan_free(&h->proj_plan);
        step_plan_free(&h->fast_qkv0_proj);
    }
    for (void* p : h->owned) cudaFree(p);
    delete h;
}

int fsb_lm_reset(fsb_lm* h, void* stream) {
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const fsb_lm_config& c = h->cfg;
    FSB_CUDA(cudaMemsetAsync(h->n_out, 0, c.max_batch * 4, st));
    FSB_CUDA(cudaMemsetAsync(h->finished, 0, c.max_batch * 4, st));
    FSB_CUDA(cudaMemsetAsync(h->slot_state, 0, c.max_batch * 4, st));
    FSB_CUDA(cudaMemsetAsync(h->ras_window, 0, static_cast<size_t>(c.max_batch) * 10 * 4, st));
    FSB_CUDA(cudaMemsetAsync(h->pos, 0, kDecRows * 4, st));
    FSB_CUDA(cudaMemsetAsync(h->step, 0, 8, st));
    return 0;
}

int fsb_lm_prefill(fsb_lm* h, const int32_t* d_tokens, const int32_t* d_row_slot, const int32_t* d_row_pos,
                   int rows, const int32_t* d_last_rows, const int32_t* d_slots, int nseq, int do_sample,
                   const fsb_sampling* sp, void* stream) {
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const fsb_lm_config& c = h->cfg;
    FSB_CHECK(rows >= 1 && rows <= std::max(c.max_rows, 128), "prefill: rows=%d exceeds max_rows=%d", rows, c.max_rows);
    FSB_CHECK(nseq >= 1 && nseq <= c.max_batch, "prefill: nseq=%d out of range", nseq);
    Stack& s = h->slow;
    FSB_TRY(launch_embed(embed_args(h, d_tokens, h->xres_p, nullptr, rows), st));
    ResidNormArgs r{};
    r.x_in = h->xres_p;
    r.norm_w = s.w[0].attn_norm; r.n_out = h->xn_p;
    r.rows = rows; r.D = s.D; r.eps = c.norm_eps;
    FSB_TRY(launch_resid_norm(r, st));
    FSB_TRY(run_stack_prefill(h, s, rows, d_row_slot, d_row_pos, st));
    if (!do_sample) return 0;
    FSB_CHECK(sp != nullptr || h->slot_control, "prefill: sampling parameters required");
    const fsb_sampling sp_none{1.f, 1.f, 1, 0};
    if (sp == nullptr) sp = &sp_none;
    // last-token rows -> decode residual stream (llama.py:447-448 keeps only the last position)
    RowsArgs g{};
    g.x = h->xres_p;
    g.y = s.xres;
    g.ssq = s.ssq;
    g.gather = d_last_rows;
    g.gather_stride = 1;
    g.rows = nseq; g.D = s.D; g.eps = c.norm_eps;
    FSB_TRY(launch_rows(g, st));
    // the reference resets the RAS window per generate() call and prefill uses no RAS
    return run_frame_tail(h, nseq, d_slots, false, d_last_rows, d_row_pos, *sp, st, /*x_is_final=*/true);
}

int fsb_lm_set_slot_control(fsb_lm* h, int enable) {
    FSB_CHECK(h != nullptr, "set_slot_control: null handle");
    h->slot_control = enable != 0;
    return 0;
}

int fsb_lm_set_sampler_noise(fsb_lm* h, const float* d_u, int draws_per_frame, int ld) {
    FSB_CHECK(h != nullptr, "set_sampler_noise: null handle");
    FSB_CHECK(d_u == nullptr || (draws_per_frame >= 2 * h->cfg.num_codebooks && ld >= h->head_rows && ld >= h->cfg.codebook_size),
              "set_sampler_noise: need >= %d draws per frame and ld >= %d", 2 * h->cfg.num_codebooks,
              std::max(h->head_rows, h->cfg.codebook_size));
    h->noise_u = d_u;
    h->noise_draws = draws_per_frame;
    h->noise_ld = ld;
    return 0;
}

int fsb_lm_decode(fsb_lm* h, int batch, int nframes, const fsb_sampling* sp, int use_graph, void* stream) {
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    FSB_CHECK(batch >= 1 && batch <= h->cfg.max_batch, "decode: batch=%d out of range", batch);
    FSB_CHECK(sp != nullptr || h->slot_control, "decode: sampling parameters required");
    const fsb_sampling sp_none{1.f, 1.f, 1, 0};
    if (sp == nullptr || h->slot_control) sp = &sp_none;  // per-slot parameters: one graph for every mix of requests
    if (!use_graph) {
        for (int i = 0; i < nframes; ++i) FSB_TRY(decode_one_frame(h, batch, *sp, st));
        return 0;
    }
    const bool same = h->graph_exec && h->graph_batch == batch && h->graph_lcap == h->ctx_lcap &&
                      h->graph_slot_control == h->slot_control && h->graph_noise == h->noise_u &&
                      memcmp(&h->graph_sampling, sp, sizeof(fsb_sampling)) == 0;
    if (!same) {
        if (h->graph_exec) {
            cudaGraphExecDestroy(h->graph_exec);
            h->graph_exec = nullptr;
        }
        // capture on a private stream so the caller's stream mode does not matter
        cudaStream_t cs;
        FSB_CUDA(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
        cudaGraph_t g = nullptr;
        cudaError_t e = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
        int rc = 1;
        const int launches_before = g_launch_count;
        if (e == cudaSuccess) {
            rc = decode_one_frame(h, batch, *sp, cs);
            e = cudaStreamEndCapture(cs, &g);
        }
        h->graph_kernels = g_launch_count - launches_before;
        g_launch_count = launches_before;  // captured, not launched
        if (e != cudaSuccess || rc != 0 || g == nullptr) {
            if (rc == 0) set_error("decode: graph capture failed: %s", cudaGetErrorString(e));
            cudaStreamDestroy(cs);
            if (g) cudaGraphDestroy(g);
            return 1;
        }
        cudaGraphExec_t ge = nullptr;
        e = cudaGraphInstantiate(&ge, g, 0);
        cudaGraphDestroy(g);
        cudaStreamDestroy(cs);
        if (e != cudaSuccess) {
            set_error("decode: cudaGraphInstantiate failed: %s", cudaGetErrorString(e));
            return 1;
        }
        h->graph_exec = ge;
        h->graph_batch = batch;
        h->graph_lcap = h->ctx_lcap;
        h->graph_slot_control = h->slot_control;
        h->graph_noise = h->noise_u;
        h->graph_sampling = *sp;
    }
    for (int i = 0; i < nframes; ++i) {
        FSB_CUDA(cudaGraphLaunch(h->graph_exec, st));
        g_launch_count += h->graph_kernels;
    }
    return 0;
}

int fsb_lm_bench_gemms(fsb_lm* h, int reps, double* weight_bytes_per_rep, int* launches_per_rep, void* stream) {
    // Every weight-streaming step GEMM of one decode frame (36 slow layers x 4, head, 10 fast passes x
    // (4 layers x 4 + head)) back to back, without the attention / sampling kernels: the measured stream of the
    // dominant kernel for the roofline line of bench.py. Operands are whatever the workspaces hold; the
    // epilogues run (and overwrite the decode state), so call it after the timed generation only.
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const fsb_lm_config& c = h->cfg;
    double bytes = 0;
    int launches = 0;
    const int rows = c.max_batch;
    auto run = [&](const StepGemmPlan& p) -> int {
        bytes += p.weight_bytes;
        ++launches;
        return launch_step(h, p, rows, st);
    };
    for (int r = 0; r < reps; ++r) {
        bytes = 0;
        launches = 0;
        auto stack = [&](Stack& s, bool skip_tail) -> int {
            for (int l = 0; l < s.nl; ++l) {
                FSB_TRY(run(s.dec[l].qkv));
                if (skip_tail && l == s.nl - 1) break;
                FSB_TRY(run(s.dec[l].wo));
                FSB_TRY(run(s.dec[l].w13));
                FSB_TRY(run(s.dec[l].w2));
            }
            return 0;
        };
        FSB_TRY(stack(h->slow, false));
        FSB_TRY(run(h->head_plan));
        for (int p = 0; p < c.num_codebooks; ++p) {
            FSB_TRY(stack(h->fast, p == 0));
            if (p > 0) FSB_TRY(run(h->fast_out_plan));
        }
    }
    if (weight_bytes_per_rep) *weight_bytes_per_rep = bytes;
    if (launches_per_rep) *launches_per_rep = launches;
    return 0;
}

int fsb_lm_copy_kv(fsb_lm* h, int src_slot, int dst_slot, int n_pos, void* stream) {
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    FSB_CHECK(h != nullptr, "copy_kv: null handle");
    Stack& s = h->slow;
    FSB_CHECK(n_pos >= 0 && n_pos <= s.S, "copy_kv: n_pos=%d outside the KV cache (%d)", n_pos, s.S);
    FSB_TRY(launch_kv_copy(s.kcache, s.nl, h->cfg.max_batch, s.Hkv, s.S, s.Dh, src_slot, dst_slot, n_pos, st));
    FSB_TRY(launch_kv_copy(s.vcache, s.nl, h->cfg.max_batch, s.Hkv, s.S, s.Dh, src_slot, dst_slot, n_pos, st));
    return 0;
}

int fsb_lm_trace_frame(fsb_lm* h, int batch, const fsb_sampling* sp, unsigned long long* d_trace, int max_launches,
                       unsigned long long* d_attn_trace, int max_attn, void* stream) {
    // Diagnostic: ONE decode frame, eager launches (same kernels, same programmatic dependent launch as the graph),
    // every step GEMM recording its per-CTA stamps in launch order: the in-frame timeline at GEMM granularity.
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    FSB_CHECK(h != nullptr && sp != nullptr && d_trace != nullptr, "trace_frame: null argument");
    FSB_CHECK(batch >= 1 && batch <= h->cfg.max_batch, "trace_frame: batch=%d", batch);
    h->trace_base = d_trace;
    h->trace_next = 0;
    h->trace_max = max_launches;
    h->attn_trace_base = d_attn_trace;
    h->attn_trace_next = 0;
    h->attn_trace_max = d_attn_trace ? max_attn : 0;
    const int rc = decode_one_frame(h, batch, *sp, st);
    const int n = h->trace_next;
    h->attn_trace_base = nullptr;
    h->trace_base = nullptr;
    h->trace_next = h->trace_max = 0;
    return rc != 0 ? -1 : n;
}

int fsb_lm_repeat_step_gemm(fsb_lm* h, int layer, int kind, int reps, void* stream) {
    // Diagnostic: the SAME step GEMM of one slow layer `reps` times back to back: from the second launch on its weights
    // come from L2 where they fit (126 MB), which separates "bound by HBM" from "bound by the SM-side pipeline".
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    Stack& s = h->slow;
    FSB_CHECK(layer >= 0 && layer < s.nl && kind >= 0 && kind < 4, "repeat_step_gemm: layer %d kind %d", layer, kind);
    const StepGemmPlan* plans[4] = {&s.dec[layer].qkv, &s.dec[layer].wo, &s.dec[layer].w13, &s.dec[layer].w2};
    StepGemmPlan q = *plans[kind];
    q.p.rows = h->cfg.max_batch;
    for (int i = 0; i < reps; ++i) FSB_TRY(step_gemm_launch(q, st));
    return 0;
}

int fsb_lm_trace_step_gemms(fsb_lm* h, unsigned long long* d_trace, int max_launches, int* grid_out, void* stream) {
    // Diagnostic: the four step GEMMs of the first slow layers, each CTA recording globaltimer stamps
    // (lm_gemm.cuh StepGemmParams::trace): shows where a launch spends its time and which CTAs share an SM.
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    Stack& s = h->slow;
    int id = 0, grid = 0;
    for (int l = 0; l < s.nl && id + 4 <= max_launches; ++l) {
        const StepGemmPlan* plans[4] = {&s.dec[l].qkv, &s.dec[l].wo, &s.dec[l].w13, &s.dec[l].w2};
        for (int k = 0; k < 4; ++k) {
            StepGemmPlan q = *plans[k];
            grid = std::max(grid, static_cast<int>(q.grid.x));
            q.p.rows = h->cfg.max_batch;
            q.p.trace = d_trace + static_cast<size_t>(id++) * 8 * 512;  // 512 CTA records per launch
            FSB_CHECK(q.grid.x <= 512, "trace: grid too large");
            FSB_TRY(step_gemm_launch(q, st));
        }
    }
    if (grid_out) *grid_out = grid;
    return id;
}

int fsb_lm_set_context_bound(fsb_lm* h, int max_positions) {
    // The attention kernel keeps one fp32 score per live position in shared memory; sizing that buffer by
    // the KV capacity would cap max_seq_len at ~12k. The host knows an upper bound of every slot's length
    // (prompt + frames so far): round it up to a 1024 bucket (the decode graph is re-captured per bucket).
    FSB_CHECK(max_positions >= 0, "set_context_bound: negative bound");
    int b = ((max_positions + 1023) / 1024) * 1024;
    if (b > h->cfg.kv_len) b = h->cfg.kv_len;
    h->ctx_lcap = b;
    return 0;
}

int fsb_lm_buffer(fsb_lm* h, const char* name, void** d_ptr, size_t* bytes) {
    auto it = h->named.find(name);
    FSB_CHECK(it != h->named.end(), "fsb_lm_buffer: unknown buffer '%s'", name);
    if (d_ptr) *d_ptr = it->second.first;
    if (bytes) *bytes = it->second.second;
    return 0;
}

}  // extern "C"
