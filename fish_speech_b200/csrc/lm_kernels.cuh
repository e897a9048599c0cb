// Memory-bound kernels of the Dual-AR path that are not part of a step GEMM (lm_gemm.cuh):
//   * decode frame: embed, attention over the KV cache, sampling, frame bookkeeping, row gathers / norms that
//     re-seed the residual stream (each leaves the per-128-feature sum of squares the next step GEMM's
//     normalise-on-load needs);
//   * prefill and the codec's WindowLimitedTransformer: consumers of a plain fp32 GEMM result y[row][ld]
//     (residual + fish RMSNorm, q/k/v post-processing, SwiGLU), rounding to bf16 at exactly the points where the
//     reference's bf16 tensors round (llama.py:990-1001 RMSNorm, :891-908 qk-norm/RoPE, :979-987 SwiGLU,
//     :842-845 residual adds).
#pragma once
#include "common.cuh"
#include "lm_gemm.cuh"

namespace fsb {

constexpr int kSsqTile = 128;     // features per sum-of-squares entry (= step GEMM tile)
constexpr int kSsqRowStride = 32; // floats per row (== kSsqStride in lm_gemm.cuh)

struct EmbedArgs {
    const int* tokens;  // [rows][C+1] (row-major per token row)
    const __nv_bfloat16* emb;     // [V, D]
    const __nv_bfloat16* cb_emb;  // [C*cs, D]
    __nv_bfloat16* x;             // [rows, D]
    float* ssq;                   // optional [rows][kSsqRowStride]: sum of x^2 per 128-feature tile
    int rows, D, C, cs, vocab;
    int sem_begin, sem_end;
    int scale;  // scale_codebook_embeddings
};
int launch_embed(const EmbedArgs& a, cudaStream_t st);

// y_out[r] = norm_w ? rbf(rbf(x[src(r)] * rsqrt(mean(x^2) + eps)) * norm_w) : x[src(r)], plus its per-tile sum of squares.
// src(r) = gather ? gather[map(r) * gather_stride] : r   (embedding lookups, last-token rows of a prefill)
struct RowsArgs {
    const __nv_bfloat16* x;     // [*, D]
    const __nv_bfloat16* norm_w;  // [D] or null (plain copy)
    const float* ssq_in;          // [*][kSsqRowStride] per-tile sum of squares of x (required with norm_w)
    __nv_bfloat16* y;           // [rows, D]
    float* ssq;                 // [rows][kSsqRowStride] of y (may be null)
    const int* gather;
    const int* gather_map;
    int gather_stride;
    int rows, D;
    float eps;
};
int launch_rows(const RowsArgs& a, cudaStream_t st);

// x_out = rbf(x_in + rbf(y + bias) [* scale])   (skip the add when y == null)
// n_out = rbf(rbf(x_out * rsqrt(mean(x_out^2)+eps)) * w)     [fish RMSNorm: round, then * weight]
struct ResidNormArgs {
    const float* y;  // [rows][ld] fp32 GEMM result or null
    int ld;
    const __nv_bfloat16* bias;   // [D] or null (attention_o_bias)
    const __nv_bfloat16* scale;  // [D] or null: y *= scale (codec LayerScale, modded_dac.py:329-341)
    const __nv_bfloat16* x_in;   // [rows, D] residual input (null => 0)
    __nv_bfloat16* x_out;        // [rows, D] (may alias x_in; null => don't store)
    const __nv_bfloat16* norm_w;  // [D] (null => no norm output)
    __nv_bfloat16* n_out;         // [rows, D]
    int rows, D;
    float eps;
};
int launch_resid_norm(const ResidNormArgs& a, cudaStream_t st);

// q,k,v = rbf(y [+bias]); optional per-head nn.RMSNorm (single rounding); interleaved RoPE in
// fp32 with bf16 tables; q -> qbuf[row][H][Dh]; k,v -> cache[b][hkv][pos][Dh].
struct QkvPrepArgs {
    const float* y;  // [rows][ld]
    int ld;
    const __nv_bfloat16* bias;  // [(H+2Hkv)*Dh] or null
    const __nv_bfloat16* q_norm;  // [Dh] or null
    const __nv_bfloat16* k_norm;
    const __nv_bfloat16* freqs;  // [S, Dh/2, 2] bf16 (cos, sin)
    const int* row_seq;          // [rows] cache slot of each row
    const int* row_pos;          // [rows] position of each row
    __nv_bfloat16* q;            // [rows, H, Dh]
    __nv_bfloat16* kcache;       // [Bslots, Hkv, S, Dh]
    __nv_bfloat16* vcache;
    int rows, H, Hkv, Dh, S;
    float eps;
};
int launch_qkv_prep(const QkvPrepArgs& a, cudaStream_t st);

// out[row][h][:] = softmax(q.k^T * scale over cache positions [max(0,pos-window+1), pos]) . v  (fp32 softmax)
struct AttnArgs {
    const __nv_bfloat16* q;  // [rows, H, Dh]
    const __nv_bfloat16* kcache;
    const __nv_bfloat16* vcache;
    const int* row_seq;
    const int* row_pos;
    __nv_bfloat16* out;  // [rows, H*Dh]
    int rows, H, Hkv, Dh, S;
    int window;  // <=0: unlimited
};
// csrc/attn_tile.cu: 64 rows of one head per CTA, K/V tiles staged once, mma.sync tensor cores, online softmax; for any
// number of rows (prefill, codec transformer).  head_dim 64 or 128.
int launch_attn(const AttnArgs& a, cudaStream_t st);
int attn_init();  // set the decode attention's kernel attributes (idempotent)
void attn_set_score_chunk(int positions);  // tests: force the decode attention's score-buffer chunk (0 = automatic)

// Decode-step attention: the consumer of the qkv step GEMM. One CTA per (batch row, KV group) first finishes that
// GEMM for its own (G + 2) heads -- slot-ordered sum of the stream-K partials, bias, per-head nn.RMSNorm, interleaved
// RoPE (llama.py:891-908) -- appends K/V to the cache (KVCache.update, llama.py:196-214), then attends over the cache
// with q still in shared memory. kv_only: stop after the append (fast pass 0 of a frame, inference.py:147).
// A row parked at position -1 (idle slot) is skipped.
struct AttnDecodeArgs {
    StepPartials qkv;
    const __nv_bfloat16* bias;    // [(H+2Hkv)*Dh] or null
    const __nv_bfloat16* q_norm;  // [Dh] or null
    const __nv_bfloat16* k_norm;
    const __nv_bfloat16* freqs;   // [S, Dh/2, 2] bf16 (cos, sin)
    __nv_bfloat16* kcache;        // [slots, Hkv, S, Dh]
    __nv_bfloat16* vcache;
    const int* row_seq;
    const int* row_pos;
    __nv_bfloat16* out;  // [rows, H*Dh]
    int rows, H, Hkv, Dh, S;
    int lcap;       // score-buffer length: an upper bound of (row_pos + 1); 0 = cache capacity S
    int bf16_math;  // the fast stack's all-bf16 attention (llama.py:948-976)
    int kv_only;
    float eps;
    // diagnostics: optional 8 globaltimer stamps of CTA (0, 0): {start, wait returned, partials summed, q/k/v finished,
    // scores done, softmax done, values summed, end}
    unsigned long long* trace;
};
int launch_attn_decode(const AttnDecodeArgs& a, cudaStream_t st);

// h = rbf( rbf(silu(rbf(a))) * rbf(c) ): a = w1 feature i, c = w3 feature i of the fused GEMM result.
// interleaved = 0: a = y[i], c = y[I + i];  1: the step-GEMM row order (w13_gate_row in lm_gemm.cuh)
struct SwigluArgs {
    const float* y;  // [rows][ld]
    int ld;
    __nv_bfloat16* h;  // [rows, I]
    int rows, I;
    int interleaved;
};
int launch_swiglu(const SwigluArgs& a, cudaStream_t st);

// Per-slot request control (continuous batching, SURVEY 8f.1). When `state` is non-null the frame kernels
// take the sampling parameters, the RNG stream and the stop rule from these arrays instead of the per-call
// values, so that every request computes exactly what it would compute alone, whatever shares the batch.
//   state: 0 idle, 1 active, 2 finished (frozen until the host retires it), 3 finishing (set by the slow
//   sampler on <|im_end|>; this frame is still recorded, inference.py:233-234)
struct SlotCtl {
    int* state;
    const int* limit;  // frames this request may produce (the prefill frame included)
    const float* temperature;
    const float* top_p;
    const int* top_k;
    const unsigned long long* seed;
    const int* n_out;  // frames produced so far = RNG counter of the request
};
__device__ __forceinline__ bool slot_live(const SlotCtl& c, int slot) {
    if (c.state == nullptr) return true;
    const int s = c.state[slot];
    return s == 1 || s == 3;
}

struct SampleArgs {
    StepPartials parts;  // stream-K partials of the (restricted) head GEMM: logit = rbf(slot-ordered sum)
    int n;           // number of candidate entries (<= 8192)
    int rows;
    // sampling parameters
    float temperature, top_p;
    int top_k;
    // token mapping for the slow head: entry e -> token id (e < n_sem ? sem_begin + e : im_end_id)
    int slow;  // 1: slow head (RAS + token mapping), 0: fast head (codes)
    int n_sem, sem_begin, im_end_id, codebook_size;
    int use_ras;              // RAS only in decode frames (previous_tokens given)
    int* ras_window;          // [rows][10] ring of previous main tokens (slow only)
    int ras_update;           // push the chosen token into the window
    unsigned long long seed;  // Philox key
    const unsigned long long* rng_offset;  // device counter (frame index) mixed into the stream
    int draw_id;              // distinguishes the samples of one frame
    // outputs
    int* cur_tok;     // [rows][C+1]
    int cb_index;     // slow: writes column 0 (token) and 1 (code a0); fast: writes column cb_index+1
    int num_cb;
    float* logits_out;  // optional [rows][n] fp32 copy of the logits (tests)
    int* finished;      // slow only: set when token == im_end
    const int* row_slot;  // optional: state (cur_tok / window / finished / logits_out) index of a row
    // Test hook (parity with the reference's torch RNG stream): when non-null, draw (frame f, draw d) of
    // slot 0 takes its uniforms U from noise_u[(f * noise_draws + d) * noise_ld + candidate] (the values
    // torch.rand produced in the probs dtype, inference.py:43-46) instead of the Philox stream, and scores
    // are formed in bf16 like the reference's tensors.
    const float* noise_u;
    int noise_draws, noise_ld;
    SlotCtl ctl;
};
int launch_sample(const SampleArgs& a, cudaStream_t st);

// bookkeeping at the end of a frame for each row's slot:
//   out_tokens[slot][c][n_out[slot]] = cur_tok[slot][c]; n_out[slot]++;
//   pos[slot] = set_pos_rows ? row_pos_src[set_pos_rows[row]] + 1 : pos[slot] + 1;   step++
struct FrameEndArgs {
    const int* cur_tok;
    int* out_tokens;  // [slots][C+1][T_cap]
    int* n_out;
    int* pos;
    const int* row_slot;      // optional
    const int* set_pos_rows;  // optional (prefill): last token row of each sequence
    const int* row_pos_src;
    unsigned long long* step;
    int rows, ncols, T_cap;
    SlotCtl ctl;
};
int launch_frame_end(const FrameEndArgs& a, cudaStream_t st);

// Prefix reuse: cache[layer][dst][g][0..n_pos) = cache[layer][src][g][0..n_pos) for every layer and KV head of one
// cache tensor laid out [layers][slots][Hkv][S][Dh].
int launch_kv_copy(__nv_bfloat16* cache, int layers, int slots, int Hkv, int S, int Dh, int src, int dst, int n_pos,
                   cudaStream_t st);

}  // namespace fsb
