// Codec (modified Descript-DAC) kernels that are not GEMM-shaped, plus the op-level C-ABI of the codec.
//
// Activations are channels-last bf16 [B][T][C]; every Conv1d / ConvTranspose1d / Linear runs on the
// tcgen05 multi-tap GEMM (gemm_tc.cu) with the causal left pad supplied by TMA zero fill; this file
// holds the small memory-bound pieces around it:
//   codebook_sum   rvq.py:361-363 + dac/nn/quantize.py from_codes (tables = out_proj(codebook), folded at load)
//   dwconv_ln      rvq.py:176-179 (ConvNeXt: causal depthwise conv k=7, LayerNorm eps 1e-6)
//   final_conv     modded_dac.py:793-797 (Snake'd input -> conv7 C->1 -> tanh)
//   first_conv     modded_dac.py:683 (conv7 1->C on the raw waveform)
//   vq_encode      rvq.py:304-317 + dac/nn/quantize.py VectorQuantize.forward (10 residual VQ stages)
#include <map>
#include <mutex>
#include <vector>

#include "../../include/fishb200.h"
#include "gemm_tc.cuh"
#include "lm_kernels.cuh"

using namespace fsb;
typedef __nv_bfloat16 bf16;

namespace {

// ------------------------------------------------------------------------------------------------
__global__ void codebook_sum_kernel(const int* __restrict__ idx, const float* const* __restrict__ tabs,
                                    const int* __restrict__ sizes, int ncb, int T, int D,
                                    bf16* __restrict__ out) {
    pdl_launch_dependents();
    pdl_wait();
    const int t = blockIdx.x, b = blockIdx.y;
    for (int d = threadIdx.x; d < D; d += blockDim.x) {
        float first = 0.f, rest = 0.f;
        for (int c = 0; c < ncb; ++c) {
            int code = idx[(static_cast<size_t>(b) * ncb + c) * T + t];
            code = min(max(code, 0), sizes[c] - 1);
            const float v = tabs[c][static_cast<size_t>(code) * D + d];
            if (c == 0) first = v; else rest += v;
        }
        out[(static_cast<size_t>(b) * T + t) * D + d] = f2bf(first + rest);
    }
}

// ------------------------------------------------------------------------------------------------
constexpr int kDwThreads = 256;
__global__ void __launch_bounds__(kDwThreads)
dwconv_ln_kernel(const bf16* __restrict__ x, const float* __restrict__ w /*[C][K]*/, const float* __restrict__ bias,
                 const float* __restrict__ ln_w, const float* __restrict__ ln_b, int T, int C, int K, float eps,
                 bf16* __restrict__ y) {
    __shared__ float red[33];
    pdl_launch_dependents();
    pdl_wait();
    const int t = blockIdx.x, b = blockIdx.y;
    float v[8];
    float s = 0.f;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        const int c = threadIdx.x + e * kDwThreads;
        v[e] = 0.f;
        if (c < C) {
            float acc = bias[c];
            for (int j = 0; j < K; ++j) {
                const int tt = t - (K - 1) + j;
                if (tt >= 0) acc += w[c * K + j] * bf2f(x[(static_cast<size_t>(b) * T + tt) * C + c]);
            }
            v[e] = acc;
            s += acc;
        }
    }
    const float mean = block_sum(s, red) / static_cast<float>(C);
    float q = 0.f;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        const int c = threadIdx.x + e * kDwThreads;
        if (c < C) q += (v[e] - mean) * (v[e] - mean);
    }
    const float var = block_sum(q, red) / static_cast<float>(C);
    const float r = rsqrtf(var + eps);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        const int c = threadIdx.x + e * kDwThreads;
        if (c < C) y[(static_cast<size_t>(b) * T + t) * C + c] = f2bf((v[e] - mean) * r * ln_w[c] + ln_b[c]);
    }
}

// ------------------------------------------------------------------------------------------------
// wav[b][t] = tanh(bias + sum_{j<K} sum_c w[j][c] * a[b][t-(K-1)+j][c])   (a already Snake-activated)
// One CTA = kFcTile consecutive time steps: the activation rows (with the K-1 row halo) are fetched with 16-byte
// loads and kept as bf16 pairs in shared memory (row stride C/2 + 1 words: conflict-free for threads on consecutive
// rows); each thread produces kFcPer outputs kFcThreads rows apart, so one weight read serves kFcPer FMAs.
constexpr int kFcThreads = 128;
constexpr int kFcPer = 2;
constexpr int kFcTile = kFcThreads * kFcPer;
__global__ void __launch_bounds__(kFcThreads)
final_conv_tanh_kernel(const bf16* __restrict__ a, const float* __restrict__ w /*[K][C]*/, float bias, int T, int C,
                       int K, float* __restrict__ wav) {
    extern __shared__ float fsm[];
    float* ws = fsm;                                             // [K*C]
    uint32_t* xs = reinterpret_cast<uint32_t*>(fsm + K * C);     // [kFcTile + K - 1][C/2 + 1] bf16 pairs
    pdl_launch_dependents();
    for (int e = threadIdx.x; e < K * C; e += kFcThreads) ws[e] = w[e];
    pdl_wait();
    const int b = blockIdx.y, t0 = blockIdx.x * kFcTile;
    const int rows = kFcTile + K - 1, ldw = C / 2 + 1, vpr = C / 8;  // 16-byte vectors per row
    if ((C & 7) == 0) {
        for (int e = threadIdx.x; e < rows * vpr; e += kFcThreads) {
            const int r = e / vpr, v = e - r * vpr;
            const int tt = t0 - (K - 1) + r;
            uint4 u = make_uint4(0, 0, 0, 0);
            if (tt >= 0 && tt < T) u = *reinterpret_cast<const uint4*>(a + (static_cast<size_t>(b) * T + tt) * C + v * 8);
            uint32_t* d = xs + r * ldw + v * 4;
            d[0] = u.x; d[1] = u.y; d[2] = u.z; d[3] = u.w;
        }
    } else {  // narrow test geometries: one bf16 pair per load
        for (int e = threadIdx.x; e < rows * (C / 2); e += kFcThreads) {
            const int r = e / (C / 2), v = e - r * (C / 2);
            const int tt = t0 - (K - 1) + r;
            uint32_t u = 0;
            if (tt >= 0 && tt < T) u = *reinterpret_cast<const uint32_t*>(a + (static_cast<size_t>(b) * T + tt) * C + v * 2);
            xs[r * ldw + v] = u;
        }
    }
    __syncthreads();
    float acc[kFcPer];
#pragma unroll
    for (int o = 0; o < kFcPer; ++o) acc[o] = bias;
    for (int j = 0; j < K; ++j) {
        const float2* wr = reinterpret_cast<const float2*>(ws + j * C);
        const uint32_t* xr = xs + (threadIdx.x + j) * ldw;
#pragma unroll 8
        for (int cw = 0; cw < C / 2; ++cw) {
            const float2 wv = wr[cw];
#pragma unroll
            for (int o = 0; o < kFcPer; ++o) {
                const uint32_t x2 = xr[o * kFcThreads * ldw + cw];
                acc[o] = fmaf(wv.x, bf_lo(x2), acc[o]);
                acc[o] = fmaf(wv.y, bf_hi(x2), acc[o]);
            }
        }
    }
#pragma unroll
    for (int o = 0; o < kFcPer; ++o) {
        const int t = t0 + o * kFcThreads + threadIdx.x;
        if (t < T) wav[static_cast<size_t>(b) * T + t] = tanhf(acc[o]);
    }
}

// ------------------------------------------------------------------------------------------------
// y[b][t][co] = bias[co] + sum_j w[co][j] * wav[b][t-(K-1)+j]   (+ optional Snake for the consumer)
__global__ void first_conv_kernel(const float* __restrict__ wav, const float* __restrict__ w /*[C][K]*/,
                                  const float* __restrict__ bias, const float* __restrict__ alpha,
                                  const float* __restrict__ inv_alpha, int T, int C, int K, bf16* __restrict__ raw,
                                  bf16* __restrict__ act) {
    pdl_launch_dependents();
    pdl_wait();
    const int b = blockIdx.y;
    const long long e = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (e >= static_cast<long long>(T) * C) return;
    const int t = static_cast<int>(e / C), c = static_cast<int>(e - static_cast<long long>(t) * C);
    float acc = bias[c];
    for (int j = 0; j < K; ++j) {
        const int tt = t - (K - 1) + j;
        if (tt >= 0) acc += w[c * K + j] * wav[static_cast<size_t>(b) * T + tt];
    }
    const size_t o = (static_cast<size_t>(b) * T + t) * C + c;
    if (raw) raw[o] = f2bf(acc);
    if (act) {
        const float s = sinf(alpha[c] * acc);
        act[o] = f2bf(acc + inv_alpha[c] * s * s);
    }
}

// elementwise Snake (used where no producing GEMM exists to fuse it into)
__global__ void snake_kernel(const bf16* __restrict__ x, const float* __restrict__ alpha,
                             const float* __restrict__ inv_alpha, long long n, int C, bf16* __restrict__ y) {
    pdl_launch_dependents();
    pdl_wait();
    const long long e = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const int c = static_cast<int>(e % C);
    const float v = bf2f(x[e]);
    const float s = sinf(alpha[c] * v);
    y[e] = f2bf(v + inv_alpha[c] * s * s);
}

// ------------------------------------------------------------------------------------------------
// Residual vector quantisation of one latent frame per CTA (10 stages in sequence):
//   e = in_proj_s(res) (8 dims); code = argmax_k cos(e, codebook_s[k]); res -= out_proj_s(codebook_s[code])
// in_w [S][cd][D], in_b [S][cd], cbn [sum sizes][cd] (L2-normalised codebooks), tabs[s] = out_proj(codebook) [size][D]
constexpr int kVqThreads = 256;
constexpr int kVqMaxCd = 16;
__global__ void __launch_bounds__(kVqThreads)
vq_encode_kernel(const bf16* __restrict__ z, const float* __restrict__ in_w, const float* __restrict__ in_b,
                 const float* __restrict__ cbn, const int* __restrict__ cb_off, const int* __restrict__ sizes,
                 const float* const* __restrict__ tabs, int S, int cd, int T, int D, int* __restrict__ codes) {
    extern __shared__ float vsm[];
    float* res = vsm;  // [D]
    __shared__ float e_s[kVqMaxCd];
    __shared__ float redv[kVqThreads / 32];
    __shared__ int redi[kVqThreads / 32];
    __shared__ int s_code;
    pdl_launch_dependents();
    pdl_wait();
    const int t = blockIdx.x, b = blockIdx.y;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int d = threadIdx.x; d < D; d += kVqThreads) res[d] = bf2f(z[(static_cast<size_t>(b) * T + t) * D + d]);
    __syncthreads();
    for (int s = 0; s < S; ++s) {
        // in_proj: cd dot products of length D (warp per output, strided)
        for (int o = warp; o < cd; o += kVqThreads / 32) {
            const float* wr = in_w + (static_cast<size_t>(s) * cd + o) * D;
            float acc = 0.f;
            for (int d = lane; d < D; d += 32) acc += wr[d] * res[d];
            acc = warp_sum(acc);
            if (lane == 0) e_s[o] = acc + in_b[s * cd + o];
        }
        __syncthreads();
        // cosine nearest neighbour: the reference maximises -(|e|^2 - 2 e.c + |c|^2) over L2-normalised
        // e and c, i.e. the largest dot product e.c / |e| (|e| > 0 is a common positive factor)
        float ev[kVqMaxCd];
        float n2 = 0.f;
        for (int o = 0; o < cd; ++o) {
            ev[o] = e_s[o];
            n2 += ev[o] * ev[o];
        }
        const float inv = rsqrtf(fmaxf(n2, 1e-24f));
        float best = -INFINITY;
        int besti = 0x7fffffff;
        const float* cb = cbn + static_cast<size_t>(cb_off[s]) * cd;
        for (int k = threadIdx.x; k < sizes[s]; k += kVqThreads) {
            float dot = 0.f;
            for (int o = 0; o < cd; ++o) dot += ev[o] * inv * cb[static_cast<size_t>(k) * cd + o];
            if (dot > best) {
                best = dot;
                besti = k;
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, besti, o);
            if (ov > best || (ov == best && oi < besti)) {
                best = ov;
                besti = oi;
            }
        }
        if (lane == 0) {
            redv[warp] = best;
            redi[warp] = besti;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            float bv = redv[0];
            int bi = redi[0];
            for (int q = 1; q < kVqThreads / 32; ++q)
                if (redv[q] > bv || (redv[q] == bv && redi[q] < bi)) {
                    bv = redv[q];
                    bi = redi[q];
                }
            s_code = bi;
            codes[(static_cast<size_t>(b) * S + s) * T + t] = bi;
        }
        __syncthreads();
        const float* tab = tabs[s] + static_cast<size_t>(s_code) * D;
        for (int d = threadIdx.x; d < D; d += kVqThreads) res[d] -= tab[d];
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------
// plan cache for the conv GEMMs: keyed by every field that enters a tensor map or the grid
struct ConvKey {
    const void *x, *w;
    int B, T_in, T_out, C_in, row_stride, C_out, taps, kpad, bn;
    long long batch_stride;
    int shifts[kMaxTaps];
    bool operator<(const ConvKey& o) const { return memcmp(this, &o, sizeof(ConvKey)) < 0; }
};
std::map<ConvKey, GemmPlan> g_conv_plans;
// Plans are keyed by operand pointers and shapes; a long-running server that sees many distinct lengths (or whose
// workspaces are re-allocated) would otherwise grow this map without bound. Tiled plans own no device memory.
constexpr size_t kMaxConvPlans = 8192;
std::mutex g_conv_mutex;

}  // namespace

extern "C" {

// Conv1d / ConvTranspose1d / Linear as a multi-tap GEMM with a fused epilogue (see gemm_tc.cuh).
//   out[b][t][co] = epi( sum_tap sum_ci x[b][t + shift[tap]][ci] * w[co][tap*kpad + ci] )
// x: bf16 rows of `row_stride` elements (C_in valid), `T_in` rows per batch item, batches `batch_stride`
// elements apart; rows outside [0, T_in) read as zero (TMA fill) — the causal left pad of
// CausalConvNet.forward (modded_dac.py:546-552). w: bf16 [C_out][taps*kpad], zero padded.
// epi: + bias[co]; GELU (act=1); * gamma[co]; + resid[b][t][co]; tanh (act=2); out0 = value (bf16 or
// fp32), out1 = Snake(value; alpha[co]) for the consuming conv (dac Snake1d). Output rows are C_out apart.
int fsb_conv_gemm(const void* d_x, int B, int T_in, int C_in, int row_stride, long long batch_stride,
                  const void* d_w, int C_out, int taps, int kpad, const int* shifts, int T_out,
                  const float* d_bias, const float* d_gamma, const void* d_resid, int act,
                  void* d_out0, void* d_out1, const float* d_alpha, const float* d_inv_alpha, int out_f32,
                  void* stream) {
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    FSB_CHECK(taps >= 1 && taps <= kMaxTaps, "conv_gemm: taps=%d out of range", taps);
    FSB_CHECK(kpad % 64 == 0, "conv_gemm: kpad must be a multiple of 64");
    FSB_CHECK(d_out0 || d_out1, "conv_gemm: no output");
    // tile width along the output channels: no padding waste for the 192- and 384-channel blocks (UMMA N = 192)
    const int bn = C_out <= 32 ? 32 : (C_out <= 64 ? 64 : (C_out <= 128 ? 128 : ((C_out % 256 != 0 && C_out % 192 == 0) ? 192 : 256)));
    const int two = bn <= 128 ? 2 : 1;  // CTAs per SM (shared memory: 3 x 32 KB stages each; TMEM: 2 x 256 columns)
    ConvKey key;
    memset(&key, 0, sizeof(key));
    key.x = d_x; key.w = d_w; key.B = B; key.T_in = T_in; key.T_out = T_out; key.C_in = C_in;
    key.row_stride = row_stride; key.C_out = C_out; key.taps = taps; key.kpad = kpad; key.bn = bn;
    key.batch_stride = batch_stride;
    for (int i = 0; i < taps; ++i) key.shifts[i] = shifts[i];
    GemmPlan plan;
    {
        std::lock_guard<std::mutex> lk(g_conv_mutex);
        auto it = g_conv_plans.find(key);
        if (it == g_conv_plans.end()) {
            GemmPlan np;
            memset(&np, 0, sizeof(np));
            GemmOperand A{reinterpret_cast<const bf16*>(d_x), C_in, T_in, B, row_stride, batch_stride};
            GemmOperand Bw{reinterpret_cast<const bf16*>(d_w), static_cast<long long>(taps) * kpad, C_out, 1,
                           static_cast<long long>(taps) * kpad, static_cast<long long>(C_out) * taps * kpad};
            np.p.kb_per_tap = kpad / 64;
            np.p.num_taps = taps;
            np.p.a_tapk = 0;
            np.p.b_tapk = kpad;
            for (int i = 0; i < taps; ++i) np.p.a_shift[i] = shifts[i];
            np.p.a_batched = 1;
            np.p.b_batched = 0;
            np.p.a_hint = kEvictNormal;
            np.p.b_hint = kEvictLast;  // the weights are re-read by every time tile
            FSB_TRY(gemm_init());
            FSB_TRY(gemm_plan_init(&np, A, Bw, bn, bn == 128 ? 3 : 4, cdiv(T_out, 128), cdiv(C_out, bn), B));
            FSB_TRY(gemm_plan_tiled(&np, cdiv(T_out, 128), cdiv(C_out, bn), B, two));
            if (g_conv_plans.size() >= kMaxConvPlans) g_conv_plans.clear();
            it = g_conv_plans.emplace(key, np).first;
        }
        plan = it->second;
    }
    GemmParams& p = plan.p;
    p.rows_i = T_out;
    p.rows_j = C_out;
    p.mode = 1;
    p.out0 = d_out0;
    p.out1 = d_out1;
    p.out_f32 = out_f32;
    p.o_zs = static_cast<long long>(T_out) * C_out;
    p.o_is = C_out;
    p.o_js = 1;
    p.chan_on_i = 0;
    p.bias = d_bias;
    p.gamma = d_gamma;
    p.resid = reinterpret_cast<const bf16*>(d_resid);
    p.act = act;
    p.snake_alpha = d_alpha;
    p.snake_inv_alpha = d_inv_alpha;
    FSB_CHECK(!d_out1 || (d_alpha && d_inv_alpha), "conv_gemm: out1 needs snake parameters");
    return gemm_launch(plan, st);
}

// One decoder ResidualUnit (Snake -> dilated conv7 -> Snake -> conv1 -> + x) as one kernel: csrc/codec_resunit.cu.
int fsb_res_unit_supported(int C) { return res_unit_supported(C) ? 1 : 0; }
int fsb_op_res_unit_trace(unsigned long long* d_trace) {
    res_unit_set_trace(d_trace);
    return 0;
}
int fsb_res_unit(const void* d_a, const void* d_x, int B, int T, int C, int dilation, const void* d_w7,
                 const float* d_b7, const float* d_alpha1, const float* d_inv1, const void* d_w1, const float* d_b1,
                 void* d_out0, void* d_out1, const float* d_alpha_n, const float* d_inv_n, void* stream) {
    FSB_TRY(gemm_init());
    return res_unit_run(d_a, d_x, B, T, C, dilation, d_w7, d_b7, d_alpha1, d_inv1, d_w1, d_b1, d_out0, d_out1, d_alpha_n,
                        d_inv_n, reinterpret_cast<cudaStream_t>(stream));
}

// Same GEMM, LM-style: fp32 results (one partial) for the transformer glue kernels below.
//   ws[row][n] = sum_k x[row][k] * w[n][k]      x bf16 [rows, K], w bf16 [N, K]
int fsb_linear_f32(const void* d_x, int rows, int K, const void* d_w, int N, float* d_ws, void* stream) {
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    ConvKey key;
    memset(&key, 0, sizeof(key));
    key.x = d_x; key.w = d_w; key.B = -1; key.T_in = rows; key.C_in = K; key.C_out = N; key.bn = 128;
    GemmPlan plan;
    {
        std::lock_guard<std::mutex> lk(g_conv_mutex);
        auto it = g_conv_plans.find(key);
        if (it == g_conv_plans.end()) {
            GemmPlan np;
            memset(&np, 0, sizeof(np));
            GemmOperand A{reinterpret_cast<const bf16*>(d_w), K, N, 1, K, static_cast<long long>(N) * K};
            GemmOperand Bx{reinterpret_cast<const bf16*>(d_x), K, rows, 1, K, static_cast<long long>(rows) * K};
            np.p.kb_per_tap = cdiv(K, 64);
            np.p.num_taps = 1;
            np.p.a_hint = kEvictNormal;
            np.p.b_hint = kEvictNormal;
            FSB_TRY(gemm_init());
            FSB_TRY(gemm_plan_init(&np, A, Bx, 128, 4, cdiv(N, 128), cdiv(rows, 128), 1));
            if (g_conv_plans.size() >= kMaxConvPlans) g_conv_plans.clear();
            it = g_conv_plans.emplace(key, np).first;
        }
        plan = it->second;
    }
    plan.p.rows_i = N;
    plan.p.rows_j = rows;
    plan.p.mode = 0;
    plan.p.ws = d_ws;
    plan.p.ws_ld = N;
    plan.p.ws_slot_stride = 0;
    return gemm_launch(plan, st);
}

int fsb_codebook_sum(const int32_t* d_idx, const float* const* d_tabs, const int32_t* d_sizes, int ncb, int B,
                     int T, int D, void* d_out, void* stream) {
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    FSB_LAUNCH(codebook_sum_kernel, dim3(T, B), dim3(256), 0, st, d_idx, d_tabs, d_sizes, ncb, T, D,
               reinterpret_cast<bf16*>(d_out));
    return 0;
}

int fsb_dwconv_ln(const void* d_x, const float* d_w, const float* d_bias, const float* d_ln_w, const float* d_ln_b,
                  int B, int T, int C, int K, float eps, void* d_y, void* stream) {
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    FSB_CHECK(C <= 8 * kDwThreads, "dwconv_ln: C=%d too large", C);
    FSB_LAUNCH(dwconv_ln_kernel, dim3(T, B), dim3(kDwThreads), 0, st, reinterpret_cast<const bf16*>(d_x), d_w, d_bias,
               d_ln_w, d_ln_b, T, C, K, eps, reinterpret_cast<bf16*>(d_y));
    return 0;
}

int fsb_final_conv_tanh(const void* d_a, const float* d_w, float bias, int B, int T, int C, int K, float* d_wav,
                        void* stream) {
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const size_t smem = (static_cast<size_t>(K) * C + static_cast<size_t>(kFcTile + K - 1) * (C / 2 + 1)) * sizeof(float);
    FSB_CHECK(smem <= 200 * 1024 && (C & 1) == 0, "final_conv: C=%d not supported", C);
    static bool attr = false;
    if (!attr) {
        FSB_CUDA(cudaFuncSetAttribute(final_conv_tanh_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        attr = true;
    }
    FSB_LAUNCH(final_conv_tanh_kernel, dim3(cdiv(T, kFcTile), B), dim3(kFcThreads), smem, st,
               reinterpret_cast<const bf16*>(d_a), d_w, bias, T, C, K, d_wav);
    return 0;
}

int fsb_first_conv(const float* d_wav, const float* d_w, const float* d_bias, const float* d_alpha,
                   const float* d_inv_alpha, int B, int T, int C, int K, void* d_raw, void* d_act, void* stream) {
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const long long n = static_cast<long long>(T) * C;
    FSB_LAUNCH(first_conv_kernel, dim3(static_cast<unsigned>(cdivll(n, 256)), B), dim3(256), 0, st, d_wav, d_w, d_bias,
               d_alpha, d_inv_alpha, T, C, K, reinterpret_cast<bf16*>(d_raw), reinterpret_cast<bf16*>(d_act));
    return 0;
}

int fsb_snake(const void* d_x, const float* d_alpha, const float* d_inv_alpha, long long n, int C, void* d_y,
              void* stream) {
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    FSB_LAUNCH(snake_kernel, dim3(static_cast<unsigned>(cdivll(n, 256))), dim3(256), 0, st,
               reinterpret_cast<const bf16*>(d_x), d_alpha, d_inv_alpha, n, C, reinterpret_cast<bf16*>(d_y));
    return 0;
}

int fsb_vq_encode(const void* d_z, const float* d_in_w, const float* d_in_b, const float* d_cbn,
                  const int32_t* d_cb_off, const int32_t* d_sizes, const float* const* d_tabs, int S, int cd, int B,
                  int T, int D, int32_t* d_codes, void* stream) {
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    FSB_CHECK(cd <= kVqMaxCd, "vq_encode: codebook_dim %d too large", cd);
    FSB_LAUNCH(vq_encode_kernel, dim3(T, B), dim3(kVqThreads), static_cast<size_t>(D) * sizeof(float), st,
               reinterpret_cast<const bf16*>(d_z), d_in_w, d_in_b, d_cbn, d_cb_off, d_sizes, d_tabs, S, cd, T, D,
               d_codes);
    return 0;
}

// ---- transformer glue of the codec's WindowLimitedTransformer (modded_dac.py:174-346), reusing the
// LM kernels: fp32 GEMM results in, bf16 operands out ----
// x_out = x_in + scale * y ;  n_out = fish RMSNorm(x_out) * norm_w   (LayerScale: scale = gamma)
int fsb_resid_scale_norm(const float* d_y, int ld, const void* d_scale, const void* d_x_in, void* d_x_out,
                         const void* d_norm_w, void* d_n_out, int rows, int D, float eps, int round_bf16,
                         void* stream) {
    ResidNormArgs a{};
    a.y = d_y;
    a.ld = ld;
    a.scale = reinterpret_cast<const bf16*>(d_scale);
    a.x_in = reinterpret_cast<const bf16*>(d_x_in);
    a.x_out = reinterpret_cast<bf16*>(d_x_out);
    a.norm_w = reinterpret_cast<const bf16*>(d_norm_w);
    a.n_out = reinterpret_cast<bf16*>(d_n_out);
    a.rows = rows;
    a.D = D;
    a.eps = eps;
    (void)round_bf16;
    return launch_resid_norm(a, reinterpret_cast<cudaStream_t>(stream));
}

int fsb_qkv_rope(const float* d_qkv, int rows, int H, int Hkv, int Dh, const void* d_freqs, const int32_t* d_row_seq,
                 const int32_t* d_row_pos, void* d_q, void* d_k, void* d_v, int S, void* stream) {
    QkvPrepArgs a{};
    a.y = d_qkv;
    a.ld = (H + 2 * Hkv) * Dh;
    a.freqs = reinterpret_cast<const bf16*>(d_freqs);
    a.row_seq = d_row_seq;
    a.row_pos = d_row_pos;
    a.q = reinterpret_cast<bf16*>(d_q);
    a.kcache = reinterpret_cast<bf16*>(d_k);
    a.vcache = reinterpret_cast<bf16*>(d_v);
    a.rows = rows; a.H = H; a.Hkv = Hkv; a.Dh = Dh; a.S = S;
    a.eps = 1e-6f;
    return launch_qkv_prep(a, reinterpret_cast<cudaStream_t>(stream));
}

int fsb_window_attn(const void* d_q, const void* d_k, const void* d_v, const int32_t* d_row_seq,
                    const int32_t* d_row_pos, int rows, int H, int Hkv, int Dh, int S, int window, void* d_out,
                    void* stream) {
    AttnArgs a{};
    a.q = reinterpret_cast<const bf16*>(d_q);
    a.kcache = reinterpret_cast<const bf16*>(d_k);
    a.vcache = reinterpret_cast<const bf16*>(d_v);
    a.row_seq = d_row_seq;
    a.row_pos = d_row_pos;
    a.out = reinterpret_cast<bf16*>(d_out);
    a.rows = rows; a.H = H; a.Hkv = Hkv; a.Dh = Dh; a.S = S;
    a.window = window;
    return launch_attn(a, reinterpret_cast<cudaStream_t>(stream));
}

int fsb_op_attn_score_chunk(int positions) {
    attn_set_score_chunk(positions);
    return 0;
}

int fsb_swiglu_f32(const float* d_y, int rows, int I, void* d_h, void* stream) {
    SwigluArgs a{};
    a.y = d_y;
    a.ld = 2 * I;
    a.h = reinterpret_cast<bf16*>(d_h);
    a.rows = rows;
    a.I = I;
    return launch_swiglu(a, reinterpret_cast<cudaStream_t>(stream));
}

}  // extern "C"
