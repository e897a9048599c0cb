// Library-level C-ABI entry points + the unit-test hooks declared in include/fishb200.h.
#include "../../include/fishb200.h"
#include "gemm_tc.cuh"
#include "lm_kernels.cuh"

using namespace fsb;

extern "C" {

const char* fsb_last_error(void) { return get_error(); }
long long fsb_launch_count(void) { return g_launch_count; }

int fsb_device_info(int* sm_count, int* cc_major, int* cc_minor) {
    int dev = 0;
    cudaDeviceProp prop;
    FSB_CUDA(cudaGetDevice(&dev));
    FSB_CUDA(cudaGetDeviceProperties(&prop, dev));
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    return 0;
}

int fsb_memcpy_d2h(void* h_dst, const void* d_src, size_t bytes, void* stream) {
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    FSB_CUDA(cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, st));
    FSB_CUDA(cudaStreamSynchronize(st));
    return 0;
}
int fsb_memcpy_h2d(void* d_dst, const void* h_src, size_t bytes, void* stream) {
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    FSB_CUDA(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, st));
    FSB_CUDA(cudaStreamSynchronize(st));
    return 0;
}

// Reduce stream-K partial sums: out[j][i] = sum_s ws[s][j][i]
static __global__ void reduce_parts_kernel(const float* ws, long long slot_stride, const int* nparts,
                                           float* out, int m, int n) {
    pdl_wait();
    const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
    if (i >= m || j >= n) return;
    const int np = nparts[i >> 7];
    float s = 0.f;
    for (int q = 0; q < np; ++q) s += ws[q * slot_stride + static_cast<long long>(j) * m + i];
    out[static_cast<long long>(j) * m + i] = s;
}

int fsb_op_gemm(const void* d_a, const void* d_b, float* d_out, int m, int n, int k, int bn,
                int streamk_ctas, void* stream) {
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    GemmPlan plan;
    memset(&plan, 0, sizeof(plan));
    GemmOperand A{reinterpret_cast<const __nv_bfloat16*>(d_a), k, m, 1, k, static_cast<long long>(m) * k};
    GemmOperand B{reinterpret_cast<const __nv_bfloat16*>(d_b), k, n, 1, k, static_cast<long long>(n) * k};
    const int kblocks = cdiv(k, 64);
    plan.p.kb_per_tap = kblocks;
    plan.p.num_taps = 1;
    plan.p.rows_i = m;
    plan.p.rows_j = n;
    const int tiles_i = cdiv(m, 128), tiles_j = cdiv(n, bn);
    FSB_TRY(gemm_plan_init(&plan, A, B, bn, 6, tiles_i, tiles_j, 1));
    float* ws = nullptr;
    if (streamk_ctas > 0) {
        FSB_CHECK(tiles_j == 1, "stream-K hook needs n <= bn");
        FSB_TRY(gemm_plan_streamk(&plan, tiles_i, kblocks, streamk_ctas));
        const size_t slot = static_cast<size_t>(n) * m;
        FSB_CUDA(cudaMalloc(&ws, slot * plan.max_parts * sizeof(float)));
        plan.p.mode = 0;
        plan.p.ws = ws;
        plan.p.ws_ld = m;
        plan.p.ws_slot_stride = static_cast<long long>(slot);
        int rc = gemm_launch(plan, st);
        if (rc == 0) {
            reduce_parts_kernel<<<dim3(cdiv(m, 256), n), 256, 0, st>>>(ws, plan.p.ws_slot_stride,
                                                                       plan.nparts_dev, d_out, m, n);
            if (cudaGetLastError() != cudaSuccess) rc = 1;
        }
        cudaError_t e = cudaStreamSynchronize(st);
        cudaFree(ws);
        gemm_plan_free(&plan);
        FSB_CHECK(rc == 0, "%s", get_error());
        FSB_CUDA(e);
        return 0;
    }
    // direct fp32 epilogue: out[j*m + i]
    plan.p.mode = 1;
    plan.p.out0 = d_out;
    plan.p.out_f32 = 1;
    plan.p.o_zs = 0;
    plan.p.o_is = 1;
    plan.p.o_js = m;
    plan.p.chan_on_i = 1;
    int rc = gemm_launch(plan, st);
    cudaError_t e = cudaStreamSynchronize(st);
    gemm_plan_free(&plan);
    if (rc != 0) return rc;
    FSB_CUDA(e);
    return 0;
}

int fsb_op_step_gemm(const void* d_w, int n_out, int K, const void* d_x, int rows, int norm_on_load,
                     const float* d_x_ssq, int x_nt, const void* d_norm_w, float eps, int num_ctas, int stages,
                     float* d_ws, size_t ws_floats, int32_t* h_nparts, int* max_parts, int* grid, int* stages_used,
                     void* stream) {
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    FSB_CHECK(rows >= 1 && rows <= kStepRows, "step GEMM hook: rows=%d", rows);
    FSB_CHECK(!norm_on_load || (x_nt >= 1 && x_nt <= kSsqStride && d_x_ssq && d_norm_w), "step GEMM hook: norm inputs");
    StepGemmPlan plan;
    FSB_TRY(step_plan_init(&plan, reinterpret_cast<const __nv_bfloat16*>(d_w), n_out, K,
                           reinterpret_cast<const __nv_bfloat16*>(d_x), norm_on_load != 0, num_ctas, stages, d_ws,
                           ws_floats));
    plan.p.rows = rows;
    if (norm_on_load) {
        plan.p.x_ssq = d_x_ssq;
        plan.p.norm_w = reinterpret_cast<const __nv_bfloat16*>(d_norm_w);
        plan.p.x_nt = x_nt;
        plan.p.eps = eps;
    }
    int rc = step_gemm_launch(plan, st);
    cudaError_t e = cudaStreamSynchronize(st);
    if (rc == 0 && e == cudaSuccess)
        e = cudaMemcpy(h_nparts, plan.nparts_dev, plan.p.tiles * sizeof(int32_t), cudaMemcpyDeviceToHost);
    *max_parts = plan.max_parts;
    *grid = static_cast<int>(plan.grid.x);
    *stages_used = plan.p.stages;
    step_plan_free(&plan);
    if (rc != 0) return rc;
    FSB_CUDA(e);
    return 0;
}

// The consumer-side plan of a partial set as the hooks below receive it (slot-major layout of StepPartials).
static StepPartials hook_partials(const float* d_ws, const int32_t* d_nparts, int tiles, int n_out, int max_parts) {
    StepPartials P;
    P.ws = d_ws;
    P.nparts = d_nparts;
    P.tiles = tiles;
    P.n_out = n_out;
    P.max_parts = max_parts;
    return P;
}

int fsb_op_step_finalize(int pro, const float* d_ws, const int32_t* d_nparts, int tiles, int n_out, int max_parts,
                         int rows, int rb, const void* d_bias, const void* d_resid, void* d_x_out, float* d_ssq_out,
                         void* d_h, int I, void* stream) {
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    FSB_CHECK(pro == PRO_RESID || pro == PRO_SWIGLU, "finalize hook: pro=%d", pro);
    FSB_CHECK(rows >= 1 && rows <= kStepRows && max_parts >= 1 && tiles == cdiv(n_out, 128), "finalize hook: shape");
    FSB_CHECK(pro != PRO_RESID || (d_x_out && d_ssq_out && tiles <= kSsqStride), "finalize hook: residual outputs");
    FSB_CHECK(pro != PRO_SWIGLU || (d_h && I >= 1 && I <= tiles * 64), "finalize hook: SwiGLU output");
    StepGemmPlan consumer;
    memset(&consumer, 0, sizeof(consumer));
    consumer.pro = pro;
    consumer.p.prev = hook_partials(d_ws, d_nparts, tiles, n_out, max_parts);
    consumer.p.rows = rows;
    consumer.p.bias = reinterpret_cast<const __nv_bfloat16*>(d_bias);
    consumer.p.resid = reinterpret_cast<const __nv_bfloat16*>(d_resid);
    consumer.p.x_out = reinterpret_cast<__nv_bfloat16*>(d_x_out);
    consumer.p.ssq_out = d_ssq_out;
    consumer.p.h = reinterpret_cast<__nv_bfloat16*>(d_h);
    consumer.p.I = I;
    FSB_TRY(step_finalize_launch(consumer, st, rb));
    FSB_CUDA(cudaStreamSynchronize(st));
    return 0;
}

int fsb_op_attn_decode(const float* d_ws, const int32_t* d_nparts, int tiles, int max_parts, const void* d_bias,
                       const void* d_q_norm, const void* d_k_norm, const void* d_freqs, void* d_kcache, void* d_vcache,
                       const int32_t* d_row_seq, const int32_t* d_row_pos, void* d_out, int rows, int H, int Hkv,
                       int Dh, int S, int lcap, int bf16_math, int kv_only, float eps, void* stream) {
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const int n_out = (H + 2 * Hkv) * Dh;
    FSB_CHECK(rows >= 1 && rows <= kStepRows && max_parts >= 1 && tiles == cdiv(n_out, 128), "attention hook: shape");
    FSB_TRY(attn_init());
    AttnDecodeArgs a{};
    a.qkv = hook_partials(d_ws, d_nparts, tiles, n_out, max_parts);
    a.bias = reinterpret_cast<const __nv_bfloat16*>(d_bias);
    a.q_norm = reinterpret_cast<const __nv_bfloat16*>(d_q_norm);
    a.k_norm = reinterpret_cast<const __nv_bfloat16*>(d_k_norm);
    a.freqs = reinterpret_cast<const __nv_bfloat16*>(d_freqs);
    a.kcache = reinterpret_cast<__nv_bfloat16*>(d_kcache);
    a.vcache = reinterpret_cast<__nv_bfloat16*>(d_vcache);
    a.row_seq = d_row_seq;
    a.row_pos = d_row_pos;
    a.out = reinterpret_cast<__nv_bfloat16*>(d_out);
    a.rows = rows; a.H = H; a.Hkv = Hkv; a.Dh = Dh; a.S = S;
    a.lcap = lcap;
    a.bf16_math = bf16_math;
    a.kv_only = kv_only;
    a.eps = eps;
    FSB_TRY(launch_attn_decode(a, st));
    FSB_CUDA(cudaStreamSynchronize(st));
    return 0;
}

static int hook_slot_ctl(const fsb_op_slot_ctl* c, SlotCtl* out) {
    *out = SlotCtl{};
    if (c == nullptr || c->state == nullptr) {
        FSB_CHECK(c == nullptr || (!c->limit && !c->temperature && !c->top_p && !c->top_k && !c->seed && !c->n_out),
                  "slot control without state");
        return 0;
    }
    out->state = c->state;
    out->limit = c->limit;
    out->temperature = c->temperature;
    out->top_p = c->top_p;
    out->top_k = c->top_k;
    out->seed = c->seed;
    out->n_out = c->n_out;
    return 0;
}

int fsb_op_sample(const fsb_op_sample_args* h, void* stream) {
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    FSB_CHECK(h->rows >= 1 && h->rows <= kStepRows && h->max_parts >= 1 && h->tiles == cdiv(h->n, 128),
              "sample hook: shape");
    SampleArgs a{};
    FSB_TRY(hook_slot_ctl(&h->ctl, &a.ctl));
    FSB_CHECK(!a.ctl.state || (a.ctl.limit && a.ctl.temperature && a.ctl.top_p && a.ctl.top_k && a.ctl.seed &&
                               a.ctl.n_out),
              "sample hook: slot control needs all seven arrays");
    a.parts = hook_partials(h->ws, h->nparts, h->tiles, h->n, h->max_parts);
    a.n = h->n;
    a.rows = h->rows;
    a.temperature = h->temperature; a.top_p = h->top_p; a.top_k = h->top_k;
    a.slow = h->slow;
    a.n_sem = h->n_sem; a.sem_begin = h->sem_begin; a.im_end_id = h->im_end_id; a.codebook_size = h->codebook_size;
    a.use_ras = h->use_ras;
    a.ras_window = h->ras_window;
    a.ras_update = h->ras_update;
    a.seed = h->seed;
    a.rng_offset = h->rng_offset;
    a.draw_id = h->draw_id;
    a.cur_tok = h->cur_tok;
    a.cb_index = h->cb_index;
    a.num_cb = h->num_cb;
    a.logits_out = h->logits_out;
    a.finished = h->finished;
    a.row_slot = h->row_slot;
    a.noise_u = h->noise_u;
    a.noise_draws = h->noise_draws;
    a.noise_ld = h->noise_ld;
    FSB_TRY(launch_sample(a, st));
    FSB_CUDA(cudaStreamSynchronize(st));
    return 0;
}

int fsb_op_frame_end(const int32_t* d_cur_tok, int32_t* d_out_tokens, int32_t* d_n_out, int32_t* d_pos,
                     const int32_t* d_row_slot, const int32_t* d_set_pos_rows, const int32_t* d_row_pos_src,
                     unsigned long long* d_step, int rows, int ncols, int T_cap, const fsb_op_slot_ctl* ctl,
                     void* stream) {
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    FSB_CHECK(rows >= 1 && ncols >= 1 && ncols <= 32 && T_cap >= 1 && d_step, "frame_end hook: shape");
    FSB_CHECK(!d_set_pos_rows || d_row_pos_src, "frame_end hook: set_pos_rows needs row_pos_src");
    FrameEndArgs a{};
    FSB_TRY(hook_slot_ctl(ctl, &a.ctl));
    FSB_CHECK(!a.ctl.state || a.ctl.limit, "frame_end hook: slot control needs state and limit");
    a.cur_tok = d_cur_tok;
    a.out_tokens = d_out_tokens;
    a.n_out = d_n_out;
    a.pos = d_pos;
    a.row_slot = d_row_slot;
    a.set_pos_rows = d_set_pos_rows;
    a.row_pos_src = d_row_pos_src;
    a.step = d_step;
    a.rows = rows; a.ncols = ncols; a.T_cap = T_cap;
    FSB_TRY(launch_frame_end(a, st));
    FSB_CUDA(cudaStreamSynchronize(st));
    return 0;
}

}  // extern "C"
