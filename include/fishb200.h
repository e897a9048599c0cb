/* fishb200 — C-ABI of the B200-native Fish-Speech inference hot path.
 *
 * The reference (fishaudio/fish-speech @ 3dd1f85c) is pure Python/PyTorch and has no FFI of its own:
 * its boundary for this path is the Python API listed in SURVEY.md §8(b).  This header is what a
 * maintainer's `ctypes` stub binds instead of the eager PyTorch modules; every entry point names the
 * reference symbol (file:line under the reference checkout) whose work it replaces.  See
 * INTEGRATION.md for the reference-side binding.
 *
 * Conventions: plain pointers and sizes only (no torch types).  All `d_` pointers are CUDA device
 * pointers owned by the caller and must stay valid for the lifetime of the handle they are given to;
 * `h_` pointers are host memory.  Every function returns 0 on success, non-zero on failure with the
 * message available from fsb_last_error() (per host thread).  `stream` is a cudaStream_t passed as
 * void*.  Handles are not thread-safe; distinct handles may be driven from different host threads
 * (the reference runs the LM worker thread and the codec caller concurrently:
 * fish_speech/models/text2semantic/inference.py:748-799).
 */
#ifndef FISHB200_H
#define FISHB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

const char* fsb_last_error(void);
/* Number of kernels this host thread has launched through the library (bench.py: gpu_launches). */
long long fsb_launch_count(void);
int fsb_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* cudaMemcpy helpers so Python hosts need no CUDA bindings of their own. */
int fsb_memcpy_d2h(void* h_dst, const void* d_src, size_t bytes, void* stream);
int fsb_memcpy_h2d(void* d_dst, const void* h_src, size_t bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Dual-AR text2semantic transformer
 *   replaces DualARTransformer.forward_generate / forward_generate_fast
 *     (fish_speech/models/text2semantic/llama.py:390-466, 799-828) and
 *   decode_one_token_ar / decode_n_tokens / the prefill call in generate
 *     (fish_speech/models/text2semantic/inference.py:96-181, 184-238, 322-335).
 * ---------------------------------------------------------------------------------------------- */
typedef struct fsb_lm fsb_lm;

typedef struct {
    /* slow (time-axis) stack: BaseModelArgs, llama.py:28-73 */
    int dim, n_layer, n_head, n_kv_head, head_dim, intermediate;
    /* fast (codebook-axis) stack: DualARModelArgs, llama.py:156-193 */
    int fast_dim, n_fast_layer, fast_n_head, fast_n_kv_head, fast_head_dim, fast_intermediate;
    int vocab_size, codebook_size, num_codebooks;
    int semantic_begin_id, semantic_end_id, im_end_id;
    float norm_eps;
    int qk_norm, fast_qk_norm;           /* attention_qk_norm / fast_attention_qk_norm */
    int scale_codebook_embeddings;       /* llama.py:416-420 */
    int norm_fastlayer_input;            /* llama.py:459-461 */
    int max_batch;                       /* resident sequences ("slots"), <= 32 */
    int kv_len;                          /* KV-cache positions per sequence */
    int max_rows;                        /* token rows per prefill pass */
    int max_frames;                      /* generated frames kept per sequence */
    int debug;                           /* keep logits / per-layer activations for tests */
} fsb_lm_config;

/* One TransformerBlock (llama.py:831-987). bf16, row-major [out_features, in_features]. */
typedef struct {
    const void* d_attn_norm;  /* [dim] */
    const void* d_wqkv;       /* [(H+2Hkv)*Dh, dim] */
    const void* d_bqkv;       /* optional */
    const void* d_q_norm;     /* [Dh] optional */
    const void* d_k_norm;     /* [Dh] optional */
    const void* d_wo;         /* [dim, H*Dh] */
    const void* d_bo;         /* optional */
    const void* d_ffn_norm;   /* [dim] */
    const void* d_w13;        /* [ceil(I/64)*128, dim]: w1 and w3 interleaved per 128-row tile so that SwiGLU runs in
                                 the GEMM epilogue: tile t holds hidden features [64t, 64t+64); inside it, row
                                 32w + l (l < 16) = w1[64t + 16w + l] and row 32w + 16 + l = w3[64t + 16w + l];
                                 rows past I are zero (fish_speech_b200.engine.interleave_w13 builds it) */
    const void* d_w2;         /* [dim, I] */
} fsb_lm_layer;

typedef struct {
    const void* d_embeddings;           /* [vocab, dim] */
    const void* d_codebook_embeddings;  /* [num_codebooks*codebook_size, dim] */
    const void* d_norm;                 /* [dim] */
    const void* d_head;                 /* [head_rows, dim]: the rows of the (tied) LM head that the
                                           semantic_logit_bias leaves selectable — semantic ids in
                                           order, then <|im_end|> (inference.py:308-320) */
    int head_rows;                      /* (semantic_end_id - semantic_begin_id + 1) + 1 */
    const void* d_freqs;                /* bf16 [kv_len, head_dim/2, 2] (llama.py:1004-1023) */
    const fsb_lm_layer* layers;         /* host array [n_layer] */
    const void* d_fast_embeddings;      /* [codebook_size, fast_dim] */
    const void* d_fast_norm;            /* [fast_dim] */
    const void* d_fast_output;          /* [codebook_size, fast_dim] */
    const void* d_fast_freqs;           /* bf16 [num_codebooks, fast_head_dim/2, 2] */
    const void* d_fast_proj_w;          /* optional [fast_dim, dim] (llama.py:665-668) */
    const void* d_fast_proj_b;          /* optional [fast_dim] */
    const fsb_lm_layer* fast_layers;    /* host array [n_fast_layer] */
} fsb_lm_weights;

/* sample() parameters (inference.py:54-93).  temperature / top_p must already be rounded to the
 * model dtype the way the reference builds them (torch.tensor(v, dtype=bf16), inference.py:303-304). */
typedef struct {
    float temperature;
    float top_p;
    int top_k;
    unsigned long long seed;
} fsb_sampling;

int fsb_lm_create(const fsb_lm_config* cfg, const fsb_lm_weights* w, fsb_lm** out);
void fsb_lm_destroy(fsb_lm* h);

/* Prefill = decode_one_token_ar on whole prompts (inference.py:322-335), for `nseq` sequences packed
 * as `rows` token rows: d_tokens[row][0] = token id, [1..C] = codes; d_row_slot / d_row_pos give the
 * sequence slot and position of each row.  If do_sample != 0 the first frame of each sequence is
 * sampled from its last row (d_last_rows[k], slot d_slots[k]) and stored as output frame 0. */
int fsb_lm_prefill(fsb_lm* h, const int32_t* d_tokens, const int32_t* d_row_slot,
                   const int32_t* d_row_pos, int rows, const int32_t* d_last_rows,
                   const int32_t* d_slots, int nseq, int do_sample, const fsb_sampling* s,
                   void* stream);

/* decode_n_tokens (inference.py:184-238): `nframes` more frames for slots [0, batch). One frame =
 * slow step + constrained sampling (+RAS) + num_codebooks fast steps; captured as a CUDA graph when
 * use_graph != 0. The per-frame <|im_end|> test is kept on the device (finished flags). */
int fsb_lm_decode(fsb_lm* h, int batch, int nframes, const fsb_sampling* s, int use_graph,
                  void* stream);

/* Prefix KV reuse (SURVEY §8(f).2; the reference re-prefills the whole growing conversation for every chunk,
 * inference.py:611-721). The slow KV cache of a slot stays valid for the positions a prefill wrote until they are
 * overwritten, so a prompt that shares its first p rows with what a slot already holds only needs rows [p, T):
 * call fsb_lm_prefill with d_row_pos starting at p. fsb_lm_copy_kv makes the K/V of positions [0, n_pos) of
 * `src_slot` available in `dst_slot` (every layer, every KV head) for requests that share a system / reference
 * prompt with another slot. Prefill is row-independent, so reused K/V is bit-identical to recomputed K/V. */
int fsb_lm_copy_kv(fsb_lm* h, int src_slot, int dst_slot, int n_pos, void* stream);

/* Upper bound of (position + 1) over all slots for the calls that follow (prompt length + frames decoded so
 * far). Sizes the attention score buffer; must be set before prefill / decode whenever it grows. */
int fsb_lm_set_context_bound(fsb_lm* h, int max_positions);

/* Per-slot request control — continuous batching over the KV slots, i.e. the batched form of the loop
 * in decode_n_tokens / generate (inference.py:184-359) that the reference runs for one request at a
 * time behind launch_thread_safe_queue (inference.py:748-799). When enabled, prefill and decode ignore
 * `s` (may be NULL) and read, per slot, the device arrays
 *   "slot_state" int32 (0 idle, 1 active, 2 finished, 3 finishing), "slot_limit" int32 (frames allowed,
 *   the prefill's frame included), "slot_temperature" f32, "slot_top_p" f32 (both already rounded to
 *   bf16 by the host, as the reference's tensors are), "slot_top_k" int32, "slot_seed" uint64.
 * The host writes them (fsb_lm_buffer) before prefilling a request into a slot; the frame kernels stop
 * a slot on <|im_end|> (from its second frame on) or at its limit, freeze its position and counters,
 * and set state = 2; the host collects "out_tokens"[slot][:, :n_out[slot]] and sets the state to 0.
 * The random stream of a request depends on (seed, own frame index, draw) only: a request produces
 * the same tokens alone or with any neighbours, in any slot. */
int fsb_lm_set_slot_control(fsb_lm* h, int enable);

/* Reset per-slot generation state (frame counters, RAS window, finished flags, slot states). */
int fsb_lm_reset(fsb_lm* h, void* stream);

/* Named device buffers of the handle, for reading results and for tests:
 *   "out_tokens" int32 [max_batch][C+1][max_frames], "n_out" int32 [max_batch], "pos" int32 [max_batch],
 *   "finished" int32 [max_batch], "cur_tok" int32 [max_batch][C+1], "ras_window" int32 [max_batch][10],
 *   the slot-control arrays listed at fsb_lm_set_slot_control,
 *   debug only: "slow_logits" f32 [max_batch][head_rows], "fast_logits" f32 [C][max_batch][codebook_size] */
int fsb_lm_buffer(fsb_lm* h, const char* name, void** d_ptr, size_t* bytes);

/* Measurement hook for bench.py: launch every weight-streaming step GEMM of one decode frame `reps` times
 * (no attention / sampling kernels; the fused epilogues run and overwrite the decode state, so call it after
 * the timed generation); returns the algorithmic weight bytes and launch count of one repetition. */
int fsb_lm_bench_gemms(fsb_lm* h, int reps, double* weight_bytes_per_rep, int* launches_per_rep,
                       void* stream);

/* Diagnostics: per-CTA globaltimer stamps of step GEMM launches, d_trace[launch][512][8] = {start, previous grid
 * complete (griddepcontrol.wait returned), -, -, first accumulator complete, end, normaliser warps ready,
 * first operand tile normalised} (0 = not recorded).
 * fsb_lm_trace_step_gemms: the step GEMMs of the first slow layers (qkv, wo, w1|w3, w2, ...) launched back to back;
 * returns the number of launches traced (0 = failure); overwrites the decode state like fsb_lm_bench_gemms.
 * fsb_lm_repeat_step_gemm: the SAME step GEMM of one slow layer `reps` times back to back (weights from L2 after the
 * first launch, where they fit); overwrites the decode state.
 * fsb_lm_trace_frame: ONE whole decode frame (eager launches, the kernels and launch attributes of the graph), every
 * step GEMM traced in launch order; advances the decode state by one frame; returns the launches traced or -1.
 * d_attn_trace (optional) [max_attn][8]: stamps of CTA (0, 0) of every decode attention launch = {start, wait returned,
 * qkv partials summed, q/k/v finished, scores, softmax, values summed, end}. */
int fsb_lm_repeat_step_gemm(fsb_lm* h, int layer, int kind, int reps, void* stream); /* kind: 0 qkv, 1 wo, 2 w1|w3, 3 w2 */
int fsb_lm_trace_frame(fsb_lm* h, int batch, const fsb_sampling* sampling, unsigned long long* d_trace,
                       int max_launches, unsigned long long* d_attn_trace, int max_attn, void* stream);
int fsb_lm_trace_step_gemms(fsb_lm* h, unsigned long long* d_trace, int max_launches, int* grid_out, void* stream);

/* Test hook for bit-exact parity of the STOCHASTIC sampler with the reference's torch RNG stream
 * (inference.py:43-46 multinomial_sample_one_no_sync, :114-144 RAS): when d_u != NULL, slot 0 takes the uniforms
 * of draw d of frame f from d_u[(f * draws_per_frame + d) * ld + candidate] (f = frames produced since
 * fsb_lm_reset; d = 0 slow token, 1 slow RAS re-draw, 2p fast codebook p; candidate = restricted head row /
 * code) instead of the library's Philox stream, and forms -log(U) and the scores in bf16 like the reference's
 * tensors. Pass NULL to restore the Philox stream. */
int fsb_lm_set_sampler_noise(fsb_lm* h, const float* d_u, int draws_per_frame, int ld);

/* ------------------------------------------------------------------------------------------------
 * Codec ("Firefly VQ-GAN" = modified Descript-DAC) operators
 *   replace DAC.from_indices / DAC.encode and everything under them
 *     (fish_speech/models/dac/modded_dac.py:874-946, fish_speech/models/dac/rvq.py:293-366).
 * Activations are channels-last bf16 [B][T][C]. The host mirror (fish_speech_b200/models/dac/) walks the
 * reference's module tree and issues one call per layer; weight-norm is folded once at load.
 * ---------------------------------------------------------------------------------------------- */
/* Conv1d / ConvTranspose1d / Linear as a tcgen05 multi-tap implicit-im2col GEMM with fused epilogue:
 *   out[b][t][co] = epi( sum_tap sum_ci x[b][t + shifts[tap]][ci] * w[co][tap*kpad + ci] )
 * rows outside [0, T_in) read as zero (= CausalConvNet's left pad, modded_dac.py:546-552).
 * epi: +bias[co]; GELU if act==1; *gamma[co]; +resid[b][t][co]; tanh if act==2; out0 = value,
 * out1 = Snake(value; alpha[co]) (dac.nn.layers.Snake1d) for the consuming layer. */
int fsb_conv_gemm(const void* d_x, int B, int T_in, int C_in, int row_stride, long long batch_stride,
                  const void* d_w, int C_out, int taps, int kpad, const int* shifts, int T_out,
                  const float* d_bias, const float* d_gamma, const void* d_resid, int act,
                  void* d_out0, void* d_out1, const float* d_alpha, const float* d_inv_alpha, int out_f32,
                  void* stream);
/* ws[row][n] (fp32) = sum_k x[row][k] * w[n][k] — feeds the transformer glue below. */
int fsb_linear_f32(const void* d_x, int rows, int K, const void* d_w, int N, float* d_ws, void* stream);
/* z[b][t][:] = tab_0[idx[b][0][t]] + sum_{c>=1} tab_c[idx[b][c][t]]  (rvq.py:352-363; tab_c =
 * out_proj_c(codebook_c), fp32 [size_c][D]); indices are clamped to the table size like the reference. */
int fsb_codebook_sum(const int32_t* d_idx, const float* const* d_tabs, const int32_t* d_sizes, int ncb, int B,
                     int T, int D, void* d_out, void* stream);
/* ConvNeXt front: causal depthwise conv (k taps) + LayerNorm (rvq.py:176-179). w fp32 [C][K]. */
int fsb_dwconv_ln(const void* d_x, const float* d_w, const float* d_bias, const float* d_ln_w, const float* d_ln_b,
                  int B, int T, int C, int K, float eps, void* d_y, void* stream);
/* Decoder tail: conv K taps C->1 on the Snake'd activation + tanh -> fp32 waveform (modded_dac.py:793-797). */
int fsb_final_conv_tanh(const void* d_a, const float* d_w, float bias, int B, int T, int C, int K, float* d_wav,
                        void* stream);
/* Encoder head: conv K taps 1->C on the fp32 waveform (modded_dac.py:683); raw and/or Snake'd output. */
int fsb_first_conv(const float* d_wav, const float* d_w, const float* d_bias, const float* d_alpha,
                   const float* d_inv_alpha, int B, int T, int C, int K, void* d_raw, void* d_act, void* stream);
int fsb_snake(const void* d_x, const float* d_alpha, const float* d_inv_alpha, long long n, int C, void* d_y,
              void* stream);
/* One decoder ResidualUnit -- y = x + conv1(snake_1(conv7_dilated(a))), a = snake_0(x) -- as ONE kernel (dac
 * ResidualUnit, modded_dac.py:599-620 causal variant): the intermediate stays in shared memory. d_a / d_x bf16
 * [B][T][C]; d_w7 [C][7][pad64(C)], d_w1 [C][pad64(C)] bf16 (the packing of fsb_conv_gemm); out0 = y (may alias d_x,
 * may be NULL), out1 = snake_next(y) (must not alias d_a). C in {96, 192, 384} (fsb_res_unit_supported). */
int fsb_res_unit_supported(int C);
int fsb_res_unit(const void* d_a, const void* d_x, int B, int T, int C, int dilation, const void* d_w7,
                 const float* d_b7, const float* d_alpha1, const float* d_inv1, const void* d_w1, const float* d_b1,
                 void* d_out0, void* d_out1, const float* d_alpha_n, const float* d_inv_n, void* stream);
/* 1 semantic + n residual vector-quantiser stages per latent frame (rvq.py:304-317, dac VectorQuantize). */
int fsb_vq_encode(const void* d_z, const float* d_in_w, const float* d_in_b, const float* d_cbn,
                  const int32_t* d_cb_off, const int32_t* d_sizes, const float* const* d_tabs, int S, int cd, int B,
                  int T, int D, int32_t* d_codes, void* stream);
/* WindowLimitedTransformer glue (modded_dac.py:174-346) on fp32 GEMM results. */
int fsb_resid_scale_norm(const float* d_y, int ld, const void* d_scale, const void* d_x_in, void* d_x_out,
                         const void* d_norm_w, void* d_n_out, int rows, int D, float eps, int round_bf16,
                         void* stream);
int fsb_qkv_rope(const float* d_qkv, int rows, int H, int Hkv, int Dh, const void* d_freqs, const int32_t* d_row_seq,
                 const int32_t* d_row_pos, void* d_q, void* d_k, void* d_v, int S, void* stream);
int fsb_window_attn(const void* d_q, const void* d_k, const void* d_v, const int32_t* d_row_seq,
                    const int32_t* d_row_pos, int rows, int H, int Hkv, int Dh, int S, int window, void* d_out,
                    void* stream);
int fsb_swiglu_f32(const float* d_y, int rows, int I, void* d_h, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Unit-test hooks (used by tests/ only)
 * ---------------------------------------------------------------------------------------------- */
/* out[j][i] (fp32, ld = m) = sum_k A[i][k] * B[j][k]; A [m,k], B [n,k] bf16 row-major.
 * bn in {32,64,128,256}; streamk_ctas > 0 uses the decode-style stream-K schedule + partial sums. */
int fsb_op_gemm(const void* d_a, const void* d_b, float* d_out, int m, int n, int k, int bn,
                int streamk_ctas, void* stream);

/* The decode step's kernels one at a time, through the host code the decode frame uses (csrc/lm_gemm.cu,
 * csrc/lm_kernels.cu). Each call synchronises `stream`. A partial set is the stream-K output of one step GEMM:
 *   value(row j, feature i) = sum over slots q < nparts[i/128], in slot order, of
 *                             ws[((q * tiles + i/128) * 32 + j) * 128 + i%128]
 * fsb_op_step_gemm: partials of W [n_out, K] x X [32, K]^T for batch rows [0, rows) into the caller's d_ws
 * (ws_floats floats; slots >= nparts of a tile and rows >= rows are not written). norm_on_load != 0: X is the
 * residual stream, normalised on load with d_x_ssq [32][32] (x_nt per-128-feature sums of squares per row),
 * d_norm_w [K] and eps. Returns nparts [ceil(n_out/128)] in h_nparts, the slot count, the grid and the ring depth. */
int fsb_op_step_gemm(const void* d_w, int n_out, int K, const void* d_x, int rows, int norm_on_load,
                     const float* d_x_ssq, int x_nt, const void* d_norm_w, float eps, int num_ctas, int stages,
                     float* d_ws, size_t ws_floats, int32_t* h_nparts, int* max_parts, int* grid, int* stages_used,
                     void* stream);
/* step_finalize over a partial set (d_nparts on the device) with `rb` batch rows per unit (0 = the default):
 * pro 1 = residual add: x_out = rbf(resid + rbf(sum + bias)), ssq_out [32][32] per-tile sums of squares
 * (d_bias, d_resid optional; d_resid may alias d_x_out); pro 2 = SwiGLU on the interleaved w1|w3 result into d_h [rows][I]. */
int fsb_op_step_finalize(int pro, const float* d_ws, const int32_t* d_nparts, int tiles, int n_out, int max_parts,
                         int rows, int rb, const void* d_bias, const void* d_resid, void* d_x_out, float* d_ssq_out,
                         void* d_h, int I, void* stream);
/* Decode attention over a qkv partial set (n_out = (H + 2*Hkv) * Dh): bias, q/k RMSNorm, RoPE, KV append at
 * [row_seq][g][row_pos], attention into d_out [rows][H*Dh]; the fields of the decode frame's call, all exposed. */
int fsb_op_attn_decode(const float* d_ws, const int32_t* d_nparts, int tiles, int max_parts, const void* d_bias,
                       const void* d_q_norm, const void* d_k_norm, const void* d_freqs, void* d_kcache, void* d_vcache,
                       const int32_t* d_row_seq, const int32_t* d_row_pos, void* d_out, int rows, int H, int Hkv,
                       int Dh, int S, int lcap, int bf16_math, int kv_only, float eps, void* stream);

/* Per-slot request control of the frame kernels (SlotCtl, csrc/lm_kernels.cuh): with `state` set, the sampler takes
 * temperature / top_p / top_k / seed and its RNG counter (n_out) from these [slots] arrays, and idle (0) and
 * finished (2) slots are left untouched. All NULL = no slot control. */
typedef struct {
    int32_t* state;
    const int32_t* limit;
    const float* temperature;
    const float* top_p;
    const int32_t* top_k;
    const unsigned long long* seed;
    const int32_t* n_out;
} fsb_op_slot_ctl;
/* Every field of the sampler's SampleArgs; the logits are the slot-ordered sums of the partial set (ws, nparts,
 * tiles = ceil(n / 128), max_parts) rounded to bf16. Rows index the partial set, `row_slot` (optional) maps a row to
 * the slot whose state it reads and writes. */
typedef struct {
    const float* ws;
    const int32_t* nparts;
    int tiles, max_parts;
    int n, rows;
    float temperature, top_p;
    int top_k;
    int slow, n_sem, sem_begin, im_end_id, codebook_size;
    int use_ras;
    int32_t* ras_window; /* [slots][10] */
    int ras_update;
    unsigned long long seed;
    const unsigned long long* rng_offset; /* device counter, may be NULL (0) */
    int draw_id;
    int32_t* cur_tok; /* [slots][num_cb + 1] */
    int cb_index, num_cb;
    float* logits_out;     /* optional [slots][n] */
    int32_t* finished;     /* optional [slots] */
    const int32_t* row_slot;
    const float* noise_u;  /* optional uniforms of slot 0, see fsb_lm_set_sampler_noise */
    int noise_draws, noise_ld;
    fsb_op_slot_ctl ctl;
} fsb_op_sample_args;
/* sample_kernel (top-k / top-p / temperature / RAS / Philox draw) through launch_sample. */
int fsb_op_sample(const fsb_op_sample_args* a, void* stream);
/* frame_end_kernel + the step counter increment through launch_frame_end: out_tokens [slots][ncols][T_cap] gets
 * cur_tok [slots][ncols] at n_out[slot], n_out and pos advance (pos = row_pos_src[set_pos_rows[row]] + 1 when
 * set_pos_rows is given), and *d_step += 1. ctl (may be NULL) needs state and limit only. */
int fsb_op_frame_end(const int32_t* d_cur_tok, int32_t* d_out_tokens, int32_t* d_n_out, int32_t* d_pos,
                     const int32_t* d_row_slot, const int32_t* d_set_pos_rows, const int32_t* d_row_pos_src,
                     unsigned long long* d_step, int rows, int ncols, int T_cap, const fsb_op_slot_ctl* ctl,
                     void* stream);

/* The decode attention (fsb_op_attn_decode, the decode frame) keeps one fp32 score per position and head in shared
 * memory; contexts longer than the buffer are walked in chunks, bit-identically (csrc/lm_kernels.cu attend()).
 * positions > 0 forces a smaller chunk; 0 = automatic. */
int fsb_op_attn_score_chunk(int positions);
/* Diagnostics of fsb_res_unit: d_trace [64][6] globaltimer stamps of CTA 0's first tiles = {epilogue idle, conv7
 * accumulator ready, h written, conv1 accumulator ready, outputs staged, stores issued}; NULL switches it off. */
int fsb_op_res_unit_trace(unsigned long long* d_trace);

#ifdef __cplusplus
}
#endif
#endif /* FISHB200_H */
