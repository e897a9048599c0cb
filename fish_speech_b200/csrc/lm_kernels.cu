// See lm_kernels.cuh.  All kernels here are HBM/L2-bound glue: vectorised, coalesced, warp-shuffle
// reductions, fp32 math with bf16 rounding at the reference's rounding points.
#include "lm_kernels.cuh"

namespace fsb {

namespace {

// Sum of squares of 4 consecutive features per lane over one 128-feature tile -> all lanes.
__device__ __forceinline__ float tile_ssq(const float (&x)[4]) {
    return warp_sum(((x[0] * x[0] + x[1] * x[1]) + x[2] * x[2]) + x[3] * x[3]);
}

// ------------------------------------------------------------------------------------------------
// embed: llama.py:399-420 (+ per-tile sum of squares for the first layer's normalise-on-load)
// ------------------------------------------------------------------------------------------------
constexpr int kRowThreads = 256;

__global__ void __launch_bounds__(kRowThreads) embed_kernel(EmbedArgs a, float inv_div) {
    pdl_launch_dependents();
    pdl_wait();
    const int row = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int* t = a.tokens + static_cast<size_t>(row) * (a.C + 1);
    int tok = t[0];
    const bool sem = tok >= a.sem_begin && tok <= a.sem_end;
    tok = min(max(tok, 0), a.vocab - 1);
    const int nt = (a.D + kSsqTile - 1) / kSsqTile;
    for (int tile = warp; tile < nt; tile += kRowThreads / 32) {
        const int f = tile * kSsqTile + lane * 4;
        float x[4] = {0.f, 0.f, 0.f, 0.f};
        if (f < a.D) {  // D % 4 == 0
            float s[4] = {0.f, 0.f, 0.f, 0.f};
            if (sem) {
                for (int c = 0; c < a.C; ++c) {
                    const int code = min(max(t[c + 1], 0), a.cs - 1);
                    const uint2 u = *reinterpret_cast<const uint2*>(a.cb_emb + (static_cast<size_t>(c) * a.cs + code) * a.D + f);
                    s[0] += bf_lo(u.x); s[1] += bf_hi(u.x); s[2] += bf_lo(u.y); s[3] += bf_hi(u.y);
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) s[q] = rbf(s[q]);  // torch.stack(...).sum(dim=1) -> one bf16 rounding
            }
            const uint2 e = *reinterpret_cast<const uint2*>(a.emb + static_cast<size_t>(tok) * a.D + f);
            const float ev[4] = {bf_lo(e.x), bf_hi(e.x), bf_lo(e.y), bf_hi(e.y)};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                x[q] = rbf(ev[q] + s[q]);
                if (sem && a.scale) x[q] = rbf(x[q] / inv_div);  // x / sqrt(C+1)
            }
            uint2 o;
            o.x = pack_bf2(x[0], x[1]);
            o.y = pack_bf2(x[2], x[3]);
            *reinterpret_cast<uint2*>(a.x + static_cast<size_t>(row) * a.D + f) = o;
        }
        const float ss = tile_ssq(x);
        if (a.ssq != nullptr && lane == 0) a.ssq[row * kSsqRowStride + tile] = ss;
    }
}

// ------------------------------------------------------------------------------------------------
// rows: gather (+ fish RMSNorm) of whole rows into a residual stream, with its per-tile sum of squares
// ------------------------------------------------------------------------------------------------
constexpr int kRowsMaxTilesPerWarp = 4;  // D <= 4096 with 8 warps

__global__ void __launch_bounds__(kRowThreads) rows_kernel(RowsArgs a) {
    pdl_launch_dependents();
    pdl_wait();
    const int row = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m = a.gather_map ? a.gather_map[row] : row;
    const int src = a.gather ? a.gather[static_cast<size_t>(m) * a.gather_stride] : row;
    const int nt = (a.D + kSsqTile - 1) / kSsqTile;
    float x[kRowsMaxTilesPerWarp][4];
#pragma unroll
    for (int e = 0; e < kRowsMaxTilesPerWarp; ++e) {
        const int tile = warp + e * (kRowThreads / 32);
        const int f = tile * kSsqTile + lane * 4;
        x[e][0] = x[e][1] = x[e][2] = x[e][3] = 0.f;
        if (tile < nt && f < a.D) {
            const uint2 u = *reinterpret_cast<const uint2*>(a.x + static_cast<size_t>(src) * a.D + f);
            x[e][0] = bf_lo(u.x); x[e][1] = bf_hi(u.x); x[e][2] = bf_lo(u.y); x[e][3] = bf_hi(u.y);
        }
    }
    float r = 1.f;
    if (a.norm_w != nullptr) {
        // the row's sum of squares as the producing kernel left it, added tile by tile in tile order: exactly
        // what the step GEMM's normalise-on-load computes, so both see the same rsqrt
        const float* q = a.ssq_in + static_cast<size_t>(src) * kSsqRowStride;
        float tot = 0.f;
        for (int t = 0; t < nt; ++t) tot += q[t];
        r = rsqrtf(tot / static_cast<float>(a.D) + a.eps);
    }
#pragma unroll
    for (int e = 0; e < kRowsMaxTilesPerWarp; ++e) {
        const int tile = warp + e * (kRowThreads / 32);
        const int f = tile * kSsqTile + lane * 4;
        const bool live = tile < nt && f < a.D;
        if (live && a.norm_w != nullptr) {
            const uint2 w = *reinterpret_cast<const uint2*>(a.norm_w + f);
            const float wf[4] = {bf_lo(w.x), bf_hi(w.x), bf_lo(w.y), bf_hi(w.y)};
#pragma unroll
            for (int q = 0; q < 4; ++q) x[e][q] = rbf(rbf(x[e][q] * r) * wf[q]);
        }
        if (live) {
            uint2 o;
            o.x = pack_bf2(x[e][0], x[e][1]);
            o.y = pack_bf2(x[e][2], x[e][3]);
            *reinterpret_cast<uint2*>(a.y + static_cast<size_t>(row) * a.D + f) = o;
        }
        if (tile < nt) {
            const float ss = tile_ssq(x[e]);
            if (a.ssq != nullptr && lane == 0) a.ssq[row * kSsqRowStride + tile] = ss;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// residual add + fish RMSNorm on a plain fp32 GEMM result (prefill, codec transformer)
// ------------------------------------------------------------------------------------------------
// 4 consecutive features per thread (D % 4 == 0, ld % 4 == 0): 16-byte loads of y.
constexpr int kRnThreads = 256;
constexpr int kRnMaxPer = 4;  // D <= 4096
__global__ void __launch_bounds__(kRnThreads) resid_norm_kernel(ResidNormArgs a) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ float red[33];
    const int row = blockIdx.x;
    float v[kRnMaxPer][4];
    float ss = 0.f;
#pragma unroll
    for (int e = 0; e < kRnMaxPer; ++e) {
        const int f = (threadIdx.x + e * kRnThreads) * 4;
        v[e][0] = v[e][1] = v[e][2] = v[e][3] = 0.f;
        if (f >= a.D) continue;
        float x[4] = {0.f, 0.f, 0.f, 0.f};
        if (a.x_in) {
            const uint2 u = *reinterpret_cast<const uint2*>(a.x_in + static_cast<size_t>(row) * a.D + f);
            x[0] = bf_lo(u.x); x[1] = bf_hi(u.x); x[2] = bf_lo(u.y); x[3] = bf_hi(u.y);
        }
        if (a.y) {
            const float4 y4 = *reinterpret_cast<const float4*>(a.y + static_cast<size_t>(row) * a.ld + f);
            float yy[4] = {y4.x, y4.y, y4.z, y4.w};
            if (a.bias) {
                const uint2 b = *reinterpret_cast<const uint2*>(a.bias + f);
                yy[0] += bf_lo(b.x); yy[1] += bf_hi(b.x); yy[2] += bf_lo(b.y); yy[3] += bf_hi(b.y);
            }
#pragma unroll
            for (int c = 0; c < 4; ++c) yy[c] = rbf(yy[c]);
            if (a.scale) {
                const uint2 sc = *reinterpret_cast<const uint2*>(a.scale + f);
                yy[0] *= bf_lo(sc.x); yy[1] *= bf_hi(sc.x); yy[2] *= bf_lo(sc.y); yy[3] *= bf_hi(sc.y);
            }
#pragma unroll
            for (int c = 0; c < 4; ++c) x[c] = rbf(x[c] + yy[c]);
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            v[e][c] = x[c];
            ss += x[c] * x[c];
        }
        if (a.x_out) {
            uint2 o;
            o.x = pack_bf2(x[0], x[1]);
            o.y = pack_bf2(x[2], x[3]);
            *reinterpret_cast<uint2*>(a.x_out + static_cast<size_t>(row) * a.D + f) = o;
        }
    }
    if (a.norm_w != nullptr) {
        const float tot = block_sum(ss, red);
        const float r = rsqrtf(tot / static_cast<float>(a.D) + a.eps);
#pragma unroll
        for (int e = 0; e < kRnMaxPer; ++e) {
            const int f = (threadIdx.x + e * kRnThreads) * 4;
            if (f >= a.D) continue;
            const uint2 w = *reinterpret_cast<const uint2*>(a.norm_w + f);
            const float wf[4] = {bf_lo(w.x), bf_hi(w.x), bf_lo(w.y), bf_hi(w.y)};
            float n[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) n[c] = rbf(rbf(v[e][c] * r) * wf[c]);
            uint2 o;
            o.x = pack_bf2(n[0], n[1]);
            o.y = pack_bf2(n[2], n[3]);
            *reinterpret_cast<uint2*>(a.n_out + static_cast<size_t>(row) * a.D + f) = o;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// q/k/v post-processing: llama.py:891-911
// ------------------------------------------------------------------------------------------------
// One CTA per row: a warp takes whole heads (lane = rotary pair, two pairs per lane at head_dim 128), so the per-head
// norm is a warp reduction.
constexpr int kQkvThreads = 256;
template <int DH>
__global__ void __launch_bounds__(kQkvThreads) qkv_prep_kernel(QkvPrepArgs a) {
    pdl_launch_dependents();
    pdl_wait();
    constexpr int PPL = DH / 64;  // rotary pairs per lane
    const int row = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int pos = a.row_pos[row];
    const int b = a.row_seq[row];
    const int NH = a.H + 2 * a.Hkv;
    for (int head = warp; head < NH; head += kQkvThreads / 32) {
        const int kind = head < a.H ? 0 : (head < a.H + a.Hkv ? 1 : 2);  // q, k, v
        const __nv_bfloat16* nw = kind == 0 ? a.q_norm : (kind == 1 ? a.k_norm : nullptr);
        float v0[PPL], v1[PPL];
        float ss = 0.f;
#pragma unroll
        for (int u = 0; u < PPL; ++u) {
            const int t = lane + 32 * u;
            const int f0 = head * DH + 2 * t;
            const float2 y2 = *reinterpret_cast<const float2*>(a.y + static_cast<size_t>(row) * a.ld + f0);
            v0[u] = y2.x;
            v1[u] = y2.y;
            if (a.bias) {
                v0[u] += bf2f(a.bias[f0]);
                v1[u] += bf2f(a.bias[f0 + 1]);
            }
            v0[u] = rbf(v0[u]);
            v1[u] = rbf(v1[u]);
            ss += v0[u] * v0[u] + v1[u] * v1[u];
        }
        if (nw != nullptr) {
            // nn.RMSNorm(head_dim): fp32 math, weight multiply included, ONE rounding
            const float r = rsqrtf(warp_sum(ss) / static_cast<float>(DH) + a.eps);
#pragma unroll
            for (int u = 0; u < PPL; ++u) {
                const int t = lane + 32 * u;
                v0[u] = rbf(v0[u] * r * bf2f(nw[2 * t]));
                v1[u] = rbf(v1[u] * r * bf2f(nw[2 * t + 1]));
            }
        }
#pragma unroll
        for (int u = 0; u < PPL; ++u) {
            const int t = lane + 32 * u;
            if (kind != 2) {
                const uint32_t cs = *reinterpret_cast<const uint32_t*>(a.freqs + (static_cast<size_t>(max(pos, 0)) * (DH / 2) + t) * 2);
                const float c = bf_lo(cs), sn = bf_hi(cs);
                const float o0 = __fsub_rn(__fmul_rn(v0[u], c), __fmul_rn(v1[u], sn));
                const float o1 = __fadd_rn(__fmul_rn(v1[u], c), __fmul_rn(v0[u], sn));
                v0[u] = rbf(o0);
                v1[u] = rbf(o1);
            }
            const uint32_t packed = pack_bf2(v0[u], v1[u]);
            if (kind == 0) {
                reinterpret_cast<uint32_t*>(a.q + (static_cast<size_t>(row) * a.H + head) * DH)[t] = packed;
            } else if (pos >= 0 && pos < a.S) {
                const int g = kind == 1 ? head - a.H : head - a.H - a.Hkv;
                __nv_bfloat16* cache = kind == 1 ? a.kcache : a.vcache;
                reinterpret_cast<uint32_t*>(cache + ((static_cast<size_t>(b) * a.Hkv + g) * a.S + pos) * DH)[t] = packed;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// length-aware GQA attention over the KV cache (one query token per CTA, all G heads of a KV group)
// ------------------------------------------------------------------------------------------------
constexpr int kAttnThreads = 256;
constexpr int kAttnWarps = kAttnThreads / 32;
constexpr int kAttnPrefetchPos = 2048;  // positions of K/V history the decode attention prefetches to L2 (8 lines per thread)

// Softmax(q k^T) v of one query token against positions [0, L) of one KV group: all G query heads of the group at once.
// The score buffer holds `lcap` positions per head (a multiple of 32).  A context that fits is scored once; a longer
// one is walked in chunks of lcap three times -- maximum, sum of exponentials, weighted values -- recomputing the
// scores each time.  Chunk boundaries are multiples of 32, so every lane and every warp accumulates exactly the
// sequence of terms it would in one pass: the result is bit-identical to the unchunked kernel, whatever lcap is.
template <int DH, int G>
__device__ __forceinline__ void attend(const float* qs, float* sc, float* red, const __nv_bfloat16* kc,
                                       const __nv_bfloat16* vc, int L, int lcap, float scale, int bf16_math,
                                       __nv_bfloat16* out, unsigned long long* trace = nullptr) {
    static_assert(G <= kAttnWarps, "one warp per query head in the softmax");
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int LPR = DH / 8;    // lanes per cache row (16-byte loads)
    constexpr int RPW = 32 / LPR;  // rows per warp iteration
    constexpr int UNR = 4;         // independent 16-byte loads in flight per lane
    constexpr int DPL = DH / 32;   // value dims per lane
    const int sub = lane / LPR, li = lane % LPR;
    float qr[G][8];
#pragma unroll
    for (int gg = 0; gg < G; ++gg)
#pragma unroll
        for (int e = 0; e < 8; ++e) qr[gg][e] = qs[gg * DH + li * 8 + e];

    auto scores = [&](int c0, int n) {  // sc[gg][p - c0] for p in [c0, c0 + n)
        const __nv_bfloat16* kcc = kc + static_cast<size_t>(c0) * DH;
        for (int pb = warp * RPW * UNR; pb < n; pb += kAttnWarps * RPW * UNR) {
            uint4 u[UNR];
#pragma unroll
            for (int j = 0; j < UNR; ++j) {
                const int p = pb + j * RPW + sub;
                u[j] = make_uint4(0, 0, 0, 0);
                if (p < n) u[j] = *reinterpret_cast<const uint4*>(kcc + static_cast<size_t>(p) * DH + li * 8);
            }
#pragma unroll
            for (int j = 0; j < UNR; ++j) {
                const int p = pb + j * RPW + sub;
                const bool ok = p < n;
                const float kf[8] = {bf_lo(u[j].x), bf_hi(u[j].x), bf_lo(u[j].y), bf_hi(u[j].y),
                                     bf_lo(u[j].z), bf_hi(u[j].z), bf_lo(u[j].w), bf_hi(u[j].w)};
#pragma unroll
                for (int gg = 0; gg < G; ++gg) {
                    float d = 0.f;
#pragma unroll
                    for (int e = 0; e < 8; ++e) d += qr[gg][e] * kf[e];
#pragma unroll
                    for (int o = LPR / 2; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
                    if (ok && li == 0) sc[gg * lcap + p] = bf16_math ? rbf(rbf(d) * scale) : d * scale;
                }
            }
        }
        __syncthreads();
    };

    const bool one = L <= lcap;
    float m = -INFINITY, z = 0.f;  // of head `warp` (warps < G)
    if (one) {
        scores(0, L);
        if (trace && threadIdx.x == 0) trace[4] = globaltimer_ns();
        if (warp < G) {
            float* s = sc + warp * lcap;
            for (int p = lane; p < L; p += 32) m = fmaxf(m, s[p]);
            m = warp_max(m);
            for (int p = lane; p < L; p += 32) {
                const float e = expf(s[p] - m);
                s[p] = e;
                z += e;
            }
            z = warp_sum(z);
            for (int p = lane; p < L; p += 32) {
                const float pr = s[p] / z;
                s[p] = bf16_math ? rbf(pr) : pr;
            }
        }
        __syncthreads();
        if (trace && threadIdx.x == 0) trace[5] = globaltimer_ns();
    } else {
        for (int c0 = 0; c0 < L; c0 += lcap) {
            const int n = min(lcap, L - c0);
            scores(c0, n);
            if (warp < G)
                for (int p = lane; p < n; p += 32) m = fmaxf(m, sc[warp * lcap + p]);
            __syncthreads();
        }
        m = warp_max(m);
        for (int c0 = 0; c0 < L; c0 += lcap) {
            const int n = min(lcap, L - c0);
            scores(c0, n);
            if (warp < G)
                for (int p = lane; p < n; p += 32) z += expf(sc[warp * lcap + p] - m);
            __syncthreads();
        }
        z = warp_sum(z);
    }

    float acc[G][DPL];
#pragma unroll
    for (int gg = 0; gg < G; ++gg)
#pragma unroll
        for (int e = 0; e < DPL; ++e) acc[gg][e] = 0.f;
    for (int c0 = 0; c0 < L; c0 += lcap) {
        const int n = min(lcap, L - c0);
        if (!one) {
            scores(c0, n);
            if (warp < G) {
                float* s = sc + warp * lcap;
                for (int p = lane; p < n; p += 32) {
                    const float pr = expf(s[p] - m) / z;
                    s[p] = bf16_math ? rbf(pr) : pr;
                }
            }
            __syncthreads();
        }
        const __nv_bfloat16* vcc = vc + static_cast<size_t>(c0) * DH;
        for (int pb = warp; pb < n; pb += kAttnWarps * UNR) {
            float vf[UNR][DPL];
#pragma unroll
            for (int j = 0; j < UNR; ++j) {
                const int p = pb + j * kAttnWarps;
#pragma unroll
                for (int e = 0; e < DPL; ++e) vf[j][e] = 0.f;
                if (p < n) {
                    if (DPL == 4) {
                        const uint2 u2 = *reinterpret_cast<const uint2*>(vcc + static_cast<size_t>(p) * DH + lane * 4);
                        vf[j][0] = bf_lo(u2.x); vf[j][1] = bf_hi(u2.x); vf[j][2 % DPL] = bf_lo(u2.y); vf[j][3 % DPL] = bf_hi(u2.y);
                    } else {
                        const uint32_t u1 = *reinterpret_cast<const uint32_t*>(vcc + static_cast<size_t>(p) * DH + lane * 2);
                        vf[j][0] = bf_lo(u1); vf[j][1] = bf_hi(u1);
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < UNR; ++j) {
                const int p = pb + j * kAttnWarps;
                if (p < n) {
#pragma unroll
                    for (int gg = 0; gg < G; ++gg) {
                        const float w = sc[gg * lcap + p];
#pragma unroll
                        for (int e = 0; e < DPL; ++e) acc[gg][e] += w * vf[j][e];
                    }
                }
            }
        }
        if (!one) __syncthreads();  // the next chunk overwrites the scores
    }
#pragma unroll
    for (int gg = 0; gg < G; ++gg)
#pragma unroll
        for (int e = 0; e < DPL; ++e) red[(warp * G + gg) * DH + lane * DPL + e] = acc[gg][e];
    __syncthreads();
    if (trace && threadIdx.x == 0) trace[6] = globaltimer_ns();
    for (int e = threadIdx.x; e < G * DH; e += kAttnThreads) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < kAttnWarps; ++w) s += red[w * G * DH + e];
        out[e] = f2bf(s);
    }
    if (trace && threadIdx.x == 0) trace[7] = globaltimer_ns();
}


// ------------------------------------------------------------------------------------------------
// decode-step attention with the qkv GEMM's fix-up in front (see lm_kernels.cuh)
// ------------------------------------------------------------------------------------------------
template <int DH, int G>
__global__ void __launch_bounds__(kAttnThreads) attn_decode_kernel(AttnDecodeArgs a, float scale, int lcap) {
    unsigned long long* trace = (a.trace != nullptr && blockIdx.x == 0 && blockIdx.y == 0) ? a.trace : nullptr;
    if (trace && threadIdx.x == 0) trace[0] = globaltimer_ns();
    pdl_launch_dependents();
    const int row = blockIdx.y, g = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // ---- before the qkv GEMM has finished: pull this row's K/V history towards L2.  The cache lines of positions
    // < pos were written frames ago; the position read here may be one frame stale (it only steers prefetch hints,
    // the real one is read after the dependency wait).  The scores / values loops then find L2 hits instead of paying
    // the HBM latency while the next GEMM's weight prefetch keeps the memory queues full. ----
    {
        const int pb = a.row_seq[row];
        const int pp = min(max(a.row_pos[row], 0), a.S - 1);
        const int n = min(pp + 1, kAttnPrefetchPos);
        const size_t base = (static_cast<size_t>(pb) * a.Hkv + g) * a.S * DH;
        const int lines = n * DH * 2 / 128;  // 128-byte lines of K (and as many of V)
        for (int i = threadIdx.x; i < lines; i += kAttnThreads) {
            prefetch_l2(reinterpret_cast<const char*>(a.kcache + base) + static_cast<size_t>(i) * 128);
            prefetch_l2(reinterpret_cast<const char*>(a.vcache + base) + static_cast<size_t>(i) * 128);
        }
    }
    // what the front end needs besides the GEMM result (static data): requested before the wait as well
    constexpr int HPR = kAttnThreads / DH;   // heads per round
    constexpr int WPH = DH / 32;             // warps per head
    constexpr int NH = G + 2;
    constexpr int NR = (NH + HPR - 1) / HPR;  // rounds: this thread's features, one per round
    const int hsub = threadIdx.x / DH, d = threadIdx.x % DH;
    float bias_r[NR], normw_r[NR];
#pragma unroll
    for (int r = 0; r < NR; ++r) {
        const int hh = r * HPR + hsub;
        const int kind = hh < G ? 0 : (hh == G ? 1 : 2);
        const int head = kind == 0 ? g * G + hh : (kind == 1 ? a.H + g : a.H + a.Hkv + g);
        const __nv_bfloat16* nw = kind == 0 ? a.q_norm : (kind == 1 ? a.k_norm : nullptr);
        bias_r[r] = (a.bias != nullptr && hh < NH) ? bf2f(a.bias[head * DH + d]) : 0.f;
        normw_r[r] = (nw != nullptr && hh < NH) ? bf2f(nw[d]) : 0.f;
    }
    pdl_wait();
    if (trace && threadIdx.x == 0) trace[1] = globaltimer_ns();
    extern __shared__ float sm[];
    float* qs = sm;                      // [G][DH]
    float* sc = qs + G * DH;             // [G][lcap]
    float* red = sc + G * lcap;          // [kAttnWarps][G][DH]
    __shared__ float wred[NR][kAttnWarps];
    // ---- finish the qkv GEMM for this row's heads: q heads g*G .. g*G+G-1, then k, then v of KV group g.  The
    // partials are requested before the row's position is looked at (they do not depend on it) ----
    const int b = a.row_seq[row];
    const int rpos = a.row_pos[row];
    float vsum[NR];
    {
        int feat[NR];
        bool ok[NR];
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            const int hh = r * HPR + hsub;
            ok[r] = hh < NH;
            const int kind = hh < G ? 0 : (hh == G ? 1 : 2);
            const int head = kind == 0 ? g * G + hh : (kind == 1 ? a.H + g : a.H + a.Hkv + g);
            feat[r] = head * DH + d;
        }
        step_partial_sums<NR>(a.qkv, row, feat, ok, vsum);  // every partial of every round in flight at once
    }
    if (rpos < 0) {  // idle slot parked at position -1: neither the cache nor the output row is touched
        return;
    }
    const int wpos = min(rpos, a.S - 1);
    // (cos, sin) of this lane's rotary pair at the row's position: the same for q and k
    const uint32_t cs = *reinterpret_cast<const uint32_t*>(a.freqs + (static_cast<size_t>(wpos) * (DH / 2) + (d >> 1)) * 2);
    if (trace && threadIdx.x == 0) trace[2] = globaltimer_ns() + (vsum[0] == 12345.f ? 1 : 0);  // after the sums arrive
    // bias, the GEMM output's bf16 rounding, and per-head nn.RMSNorm (fp32 math, weight multiply included, ONE
    // rounding): the sums of squares of all rounds cross the warps behind one barrier
    const bool any_norm = a.q_norm != nullptr || a.k_norm != nullptr;
    float v[NR];
#pragma unroll
    for (int r = 0; r < NR; ++r) {
        const int hh = r * HPR + hsub;
        v[r] = 0.f;
        if (hh < NH) {
            v[r] = vsum[r];
            if (a.bias) v[r] += bias_r[r];
            v[r] = rbf(v[r]);
        }
        if (any_norm) {
            const float ws = warp_sum(v[r] * v[r]);
            if (lane == 0) wred[r][warp] = ws;
        }
    }
    if (any_norm) __syncthreads();
#pragma unroll
    for (int r = 0; r < NR; ++r) {
        const int hh = r * HPR + hsub;
        const bool live = hh < NH;
        const int kind = hh < G ? 0 : (hh == G ? 1 : 2);
        const bool normed = kind == 0 ? a.q_norm != nullptr : (kind == 1 ? a.k_norm != nullptr : false);
        float x = v[r];
        if (live && normed) {
            const int w0 = (warp / WPH) * WPH;
            float tot = 0.f;
#pragma unroll
            for (int u = 0; u < WPH; ++u) tot += wred[r][w0 + u];
            const float rinv = rsqrtf(tot / static_cast<float>(DH) + a.eps);
            x = rbf(x * rinv * normw_r[r]);
        }
        if (kind != 2) {
            const float c = bf_lo(cs), sn = bf_hi(cs);
            const float partner = __shfl_xor_sync(0xffffffffu, x, 1);
            x = (lane & 1) ? __fadd_rn(__fmul_rn(x, c), __fmul_rn(partner, sn)) : __fsub_rn(__fmul_rn(x, c), __fmul_rn(partner, sn));
            x = rbf(x);
        }
        if (live) {
            if (kind == 0) {
                qs[hh * DH + d] = x;
            } else if (rpos < a.S) {
                __nv_bfloat16* cache = kind == 1 ? a.kcache : a.vcache;
                cache[((static_cast<size_t>(b) * a.Hkv + g) * a.S + rpos) * DH + d] = f2bf(x);
            }
        }
    }
    if (a.kv_only) return;
    __syncthreads();  // q in shared memory, this row's new K/V visible to the whole CTA
    if (trace && threadIdx.x == 0) trace[3] = globaltimer_ns();

    const int pos = wpos;
    const int L = pos + 1;
    const size_t cache_base = (static_cast<size_t>(b) * a.Hkv + g) * a.S * DH;
    const __nv_bfloat16* kc = a.kcache + cache_base;
    const __nv_bfloat16* vc = a.vcache + cache_base;

    attend<DH, G>(qs, sc, red, kc, vc, L, lcap, scale, a.bf16_math,
                  a.out + (static_cast<size_t>(row) * a.H + g * G) * DH, trace);
}

// ------------------------------------------------------------------------------------------------
// SwiGLU on a plain fp32 GEMM result (prefill, codec): 4 consecutive features per thread (I % 4 == 0, ld % 4 == 0)
// ------------------------------------------------------------------------------------------------
__global__ void swiglu_kernel(SwigluArgs a) {
    pdl_launch_dependents();
    pdl_wait();
    const int row = blockIdx.y;
    const int i = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i >= a.I) return;
    const float* y = a.y + static_cast<size_t>(row) * a.ld;
    // 4 consecutive h features never straddle a 16-feature interleave group
    const int gi = a.interleaved ? w13_gate_row(i) : i;
    const int ui = a.interleaved ? gi + 16 : a.I + i;
    const float4 g4 = *reinterpret_cast<const float4*>(y + gi);
    const float4 u4 = *reinterpret_cast<const float4*>(y + ui);
    const float gv[4] = {g4.x, g4.y, g4.z, g4.w}, uv[4] = {u4.x, u4.y, u4.z, u4.w};
    float h[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        const float gg = rbf(gv[c]), cc = rbf(uv[c]);
        const float sl = rbf(gg / (1.f + expf(-gg)));
        h[c] = sl * cc;
    }
    uint2 o;
    o.x = pack_bf2(h[0], h[1]);
    o.y = pack_bf2(h[2], h[3]);
    *reinterpret_cast<uint2*>(a.h + static_cast<size_t>(row) * a.I + i) = o;
}

// ------------------------------------------------------------------------------------------------
// sampling: inference.py:43-93 (logits_to_probs / multinomial_sample_one_no_sync / sample) and the
// slow-token RAS rule inference.py:114-144.
// ------------------------------------------------------------------------------------------------
constexpr int kSampleThreads = 1024;
constexpr int kSampleMaxN = 8192;
constexpr int kSelCap = 256;  // ranks materialised for top-k / top-p

__device__ __forceinline__ void philox4x32(uint32_t k0, uint32_t k1, uint32_t c0, uint32_t c1,
                                           uint32_t c2, uint32_t c3, uint32_t out[4]) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

struct ArgMax {
    float v;
    int i;
};
__device__ __forceinline__ ArgMax better(ArgMax a, ArgMax b) {
    // larger value wins; ties -> smaller index
    if (b.v > a.v || (b.v == a.v && b.i < a.i)) return b;
    return a;
}
__device__ __forceinline__ ArgMax block_argmax(ArgMax x, ArgMax* red) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        ArgMax y;
        y.v = __shfl_xor_sync(0xffffffffu, x.v, o);
        y.i = __shfl_xor_sync(0xffffffffu, x.i, o);
        x = better(x, y);
    }
    __syncthreads();
    if (lane == 0) red[w] = x;
    __syncthreads();
    if (w == 0) {
        ArgMax t = red[lane];  // kSampleThreads/32 == 32 warps
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            ArgMax y;
            y.v = __shfl_xor_sync(0xffffffffu, t.v, o);
            y.i = __shfl_xor_sync(0xffffffffu, t.i, o);
            t = better(t, y);
        }
        if (lane == 0) red[32] = t;
    }
    __syncthreads();
    return red[32];
}

__global__ void __launch_bounds__(kSampleThreads) sample_kernel(SampleArgs a) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ float lg[kSampleMaxN];
    __shared__ ArgMax red[33];
    __shared__ float fred[33];
    __shared__ float sel_v[kSelCap];
    __shared__ int sel_i[kSelCap];
    __shared__ float sel_cum[kSelCap];
    __shared__ int s_nsel;
    __shared__ int s_choice[2];
    const SlotCtl& ctl = a.ctl;
    const int row = blockIdx.x;
    const int slot = a.row_slot ? a.row_slot[row] : row;
    const int n = a.n;
    if (!slot_live(ctl, slot)) return;  // idle / frozen slot: nothing is sampled, its state stays as it is
    const bool per_slot = ctl.state != nullptr;
    const float temperature = per_slot ? ctl.temperature[slot] : a.temperature;
    const float top_p = per_slot ? ctl.top_p[slot] : a.top_p;
    const int top_k = per_slot ? ctl.top_k[slot] : a.top_k;
    const unsigned long long seed = per_slot ? ctl.seed[slot] : a.seed;
    for (int e0 = threadIdx.x; e0 < n; e0 += 4 * kSampleThreads) {
        int feat[4];
        bool ok[4];
        float sum[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            feat[k] = e0 + k * kSampleThreads;
            ok[k] = feat[k] < n;
        }
        step_partial_sums<4>(a.parts, row, feat, ok, sum);  // 32 loads in flight per thread, additions in slot order
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (!ok[k]) continue;
            const float v = rbf(sum[k]);  // F.linear output is a bf16 tensor
            lg[feat[k]] = v;
            if (a.logits_out) a.logits_out[static_cast<size_t>(slot) * n + feat[k]] = v;
        }
    }
    __syncthreads();

    const bool two = a.slow && a.use_ras && top_k != 1;
    if (top_k == 1) {
        ArgMax x{-INFINITY, 0x7fffffff};
        for (int e = threadIdx.x; e < n; e += kSampleThreads) x = better(x, ArgMax{lg[e], e});
        x = block_argmax(x, red);
        if (threadIdx.x == 0) s_choice[0] = s_choice[1] = x.i;
        __syncthreads();
    } else {
        // softmax denominator over every candidate (the -inf-biased vocabulary contributes 0)
        float m = -INFINITY;
        for (int e = threadIdx.x; e < n; e += kSampleThreads) m = fmaxf(m, lg[e]);
        m = block_max(m, fred);
        float z = 0.f;
        for (int e = threadIdx.x; e < n; e += kSampleThreads) z += expf(lg[e] - m);
        z = block_sum(z, fred);
        // descending ranks until neither criterion can keep anything further
        const float p_lim = two ? fmaxf(top_p, 0.9f) : top_p;
        int kcap = top_k < n ? top_k : n;
        if (kcap > kSelCap) kcap = kSelCap;
        float cumf = 0.f;  // torch.cumsum over bf16 accumulates in fp32 and rounds each output
        int nsel = 0;
        for (int r = 0; r < kcap; ++r) {
            ArgMax x{-INFINITY, 0x7fffffff};
            for (int e = threadIdx.x; e < n; e += kSampleThreads) x = better(x, ArgMax{lg[e], e});
            x = block_argmax(x, red);
            const float pr = rbf(expf(x.v - m) / z);
            cumf += pr;
            const float cum = rbf(cumf);
            if (threadIdx.x == 0) {
                sel_v[r] = x.v;
                sel_i[r] = x.i;
                sel_cum[r] = cum;
                lg[x.i] = -INFINITY;
            }
            nsel = r + 1;
            __syncthreads();
            if (cum > p_lim) break;
        }
        if (threadIdx.x == 0) s_nsel = nsel;
        __syncthreads();
        // the two draws (normal, RAS high-temperature); warp 0 / warp 1
        const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
        if (w < (two ? 2 : 1)) {
            const float T = w == 0 ? temperature : 1.0f;
            const float tp = w == 0 ? top_p : 0.9f;
            // torch.clip(temperature, min=1e-5) on the bf16 temperature tensor clamps to bf16(1e-5)
            const float Tc = fmaxf(T, 1.0013580322265625e-05f);
            // survivors: rank 0 always; rank r kept iff cum[r] <= top_p (and r < top_k, implied)
            int ns = 1;
            while (ns < nsel && !(sel_cum[ns] > tp)) ++ns;
            float mx = -INFINITY;
            for (int r = lane; r < ns; r += 32) mx = fmaxf(mx, rbf(sel_v[r] / Tc));
            mx = warp_max(mx);
            float zz = 0.f;
            for (int r = lane; r < ns; r += 32) zz += expf(rbf(sel_v[r] / Tc) - mx);
            zz = warp_sum(zz);
            // RNG stream: per call (seed, global frame counter, slot) or, with slot control, per request
            // (its own seed and frame index, no slot) so that the draw does not depend on the schedule
            const unsigned long long off =
                per_slot ? static_cast<unsigned long long>(ctl.n_out[slot]) : (a.rng_offset ? *a.rng_offset : 0ull);
            const uint32_t lane_id = per_slot ? 0u : static_cast<uint32_t>(slot);
            const int draw = a.draw_id * 2 + w;
            const float* noise = (a.noise_u != nullptr && slot == 0)
                                     ? a.noise_u + (static_cast<size_t>(off) * a.noise_draws + draw) * a.noise_ld
                                     : nullptr;
            ArgMax best{-INFINITY, 0x7fffffff};
            for (int r = lane; r < ns; r += 32) {
                const float pr = rbf(expf(rbf(sel_v[r] / Tc) - mx) / zz);
                const int e = sel_i[r];
                // torch.argmax returns the first maximum in vocabulary order: ties break on the token id
                const int key = a.slow ? (e < a.n_sem ? a.sem_begin + e : a.im_end_id) : e;
                float score;
                if (noise != nullptr) {
                    const float q = rbf(-logf(noise[e]));  // -log(U) as a bf16 tensor (inference.py:43-46)
                    score = rbf(pr / q);
                } else {
                    uint32_t rnd[4];
                    philox4x32(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32),
                               static_cast<uint32_t>(off), static_cast<uint32_t>(off >> 32), lane_id,
                               static_cast<uint32_t>(draw * kSelCap + r), rnd);
                    const float u = (static_cast<float>(rnd[0] >> 8) + 0.5f) * (1.0f / 16777216.0f);
                    score = pr / -logf(u);
                }
                best = better(best, ArgMax{score, key * kSelCap + r});
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                ArgMax y;
                y.v = __shfl_xor_sync(0xffffffffu, best.v, o);
                y.i = __shfl_xor_sync(0xffffffffu, best.i, o);
                best = better(best, y);
            }
            if (lane == 0) s_choice[w] = sel_i[best.i % kSelCap];
        }
        __syncthreads();
        if (!two && threadIdx.x == 0) s_choice[1] = s_choice[0];
        __syncthreads();
    }

    if (threadIdx.x == 0) {
        int* ct = a.cur_tok + static_cast<size_t>(slot) * (a.num_cb + 1);
        if (a.slow) {
            int e = s_choice[0];
            int tok = e < a.n_sem ? a.sem_begin + e : a.im_end_id;
            if (a.use_ras) {
                const int eh = s_choice[1];
                const int tok_h = eh < a.n_sem ? a.sem_begin + eh : a.im_end_id;
                bool in_win = false;
                for (int k = 0; k < 10; ++k) in_win |= (a.ras_window[slot * 10 + k] == tok);
                const bool is_sem = tok >= a.sem_begin && tok <= a.sem_begin + a.n_sem - 1;
                if (in_win && is_sem) tok = tok_h;
            }
            int c0 = tok - a.sem_begin;
            c0 = c0 < 0 ? 0 : (c0 > a.codebook_size - 1 ? a.codebook_size - 1 : c0);
            ct[0] = tok;
            ct[1] = c0;
            if (a.ras_update) {
                for (int k = 0; k < 9; ++k) a.ras_window[slot * 10 + k] = a.ras_window[slot * 10 + k + 1];
                a.ras_window[slot * 10 + 9] = tok;
            }
            if (a.finished && tok == a.im_end_id) a.finished[slot] = 1;
            // the reference's loop tests <|im_end|> from the second frame on (the prefill's token is not
            // tested, inference.py:336-352 then :233)
            if (per_slot && tok == a.im_end_id && ctl.n_out[slot] >= 1) ctl.state[slot] = 3;
        } else {
            ct[a.cb_index + 1] = s_choice[0];
        }
    }
}

__global__ void frame_end_kernel(FrameEndArgs a) {
    pdl_launch_dependents();
    pdl_wait();
    const SlotCtl& ctl = a.ctl;
    const int row = blockIdx.x;
    const int slot = a.row_slot ? a.row_slot[row] : row;
    if (!slot_live(ctl, slot)) return;
    const int f = a.n_out[slot];
    if (threadIdx.x < a.ncols && f < a.T_cap)
        a.out_tokens[(static_cast<size_t>(slot) * a.ncols + threadIdx.x) * a.T_cap + f] =
            a.cur_tok[slot * a.ncols + threadIdx.x];
    __syncthreads();
    if (threadIdx.x == 0) {
        a.n_out[slot] = f + 1;
        bool advance = true;
        if (ctl.state != nullptr && (ctl.state[slot] == 3 || f + 1 >= ctl.limit[slot])) {
            ctl.state[slot] = 2;  // frozen: position and counters stay at the last frame
            advance = false;
        }
        if (a.set_pos_rows)
            a.pos[slot] = a.row_pos_src[a.set_pos_rows[row]] + (advance ? 1 : 0);
        else if (advance)
            a.pos[slot] = a.pos[slot] + 1;
    }
}
// 16-byte copies of one (layer, KV head) run of n_pos positions per CTA column
__global__ void kv_copy_kernel(uint4* cache, size_t slot_stride16, size_t head_stride16, size_t layer_stride16, int src,
                               int dst, int n16) {
    pdl_launch_dependents();
    pdl_wait();
    const size_t base = blockIdx.z * layer_stride16 + blockIdx.y * head_stride16;
    const uint4* s = cache + base + src * slot_stride16;
    uint4* d = cache + base + dst * slot_stride16;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n16; e += gridDim.x * blockDim.x) d[e] = s[e];
}

__global__ void step_inc_kernel(unsigned long long* step) {
    pdl_launch_dependents();
    pdl_wait();
    *step += 1;
}

}  // namespace

int launch_embed(const EmbedArgs& a, cudaStream_t st) {
    if (a.rows <= 0) return 0;
    FSB_CHECK(a.D % 4 == 0 && a.D <= kSsqTile * kSsqRowStride, "embed: D=%d unsupported", a.D);
    FSB_LAUNCH(embed_kernel, dim3(a.rows), dim3(kRowThreads), 0, st, a, sqrtf(static_cast<float>(a.C + 1)));
    return 0;
}

int launch_rows(const RowsArgs& a, cudaStream_t st) {
    if (a.rows <= 0) return 0;
    FSB_CHECK(a.D % 4 == 0 && a.D <= kSsqTile * kSsqRowStride, "rows: D=%d unsupported", a.D);
    FSB_CHECK(a.norm_w == nullptr || a.ssq_in != nullptr, "rows: the norm needs the input's sum of squares");
    FSB_LAUNCH(rows_kernel, dim3(a.rows), dim3(kRowThreads), 0, st, a);
    return 0;
}

int launch_resid_norm(const ResidNormArgs& a, cudaStream_t st) {
    if (a.rows <= 0) return 0;
    FSB_CHECK(a.D % 4 == 0 && a.D <= 4 * kRnThreads * kRnMaxPer, "resid_norm: D=%d unsupported", a.D);
    FSB_CHECK(a.y == nullptr || (a.ld % 4 == 0 && (reinterpret_cast<uintptr_t>(a.y) & 15) == 0),
              "resid_norm: misaligned GEMM result");
    FSB_LAUNCH(resid_norm_kernel, dim3(a.rows), dim3(kRnThreads), 0, st, a);
    return 0;
}

int launch_qkv_prep(const QkvPrepArgs& a, cudaStream_t st) {
    if (a.rows <= 0) return 0;
    FSB_CHECK(a.Dh == 64 || a.Dh == 128, "qkv_prep: head_dim %d unsupported", a.Dh);
    FSB_CHECK((a.ld & 1) == 0 && (reinterpret_cast<uintptr_t>(a.y) & 7) == 0, "qkv_prep: misaligned GEMM result");
    if (a.Dh == 64) FSB_LAUNCH(qkv_prep_kernel<64>, dim3(a.rows), dim3(kQkvThreads), 0, st, a);
    else FSB_LAUNCH(qkv_prep_kernel<128>, dim3(a.rows), dim3(kQkvThreads), 0, st, a);
    return 0;
}

// Score-buffer positions per head for a context bound of `need`: rounded up to a multiple of 32 and cut to what fits
// 200 KB of shared memory (a longer context is walked in chunks, see attend()).  g_attn_chunk (tests) forces a chunk.
static int g_attn_chunk = 0;
void attn_set_score_chunk(int positions) { g_attn_chunk = positions > 0 ? (positions + 31) / 32 * 32 : 0; }
template <int DH, int G>
static size_t attn_smem_bytes(int lcap) {
    return (static_cast<size_t>(G) * DH + static_cast<size_t>(G) * lcap + static_cast<size_t>(kAttnWarps) * G * DH) *
           sizeof(float);
}
template <int DH, int G>
static int attn_score_chunk(int need) {
    int lcap = (need + 31) / 32 * 32;
    const int fit = static_cast<int>((200 * 1024 - attn_smem_bytes<DH, G>(0)) / (sizeof(float) * G)) / 32 * 32;
    if (lcap > fit) lcap = fit;
    if (g_attn_chunk > 0 && g_attn_chunk < lcap) lcap = g_attn_chunk;
    return lcap;
}

int attn_init() {
    static bool done = false;
    if (done) return 0;
#define FSB_ATTN_ATTR(DH_, G_) \
    FSB_CUDA(cudaFuncSetAttribute(attn_decode_kernel<DH_, G_>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    FSB_ATTN_ATTR(128, 1) FSB_ATTN_ATTR(128, 2) FSB_ATTN_ATTR(128, 4) FSB_ATTN_ATTR(128, 8)
    FSB_ATTN_ATTR(64, 1) FSB_ATTN_ATTR(64, 2) FSB_ATTN_ATTR(64, 4) FSB_ATTN_ATTR(64, 8)
#undef FSB_ATTN_ATTR
    done = true;
    return 0;
}

template <int DH, int G>
static int launch_attn_decode_t(const AttnDecodeArgs& a, cudaStream_t st) {
    int lcap = a.S;
    if (a.lcap > 0 && a.lcap < lcap) lcap = a.lcap;
    lcap = attn_score_chunk<DH, G>(lcap);
    const size_t smem = attn_smem_bytes<DH, G>(lcap);
    const float scale = 1.0f / sqrtf(static_cast<float>(DH));
    FSB_LAUNCH((attn_decode_kernel<DH, G>), dim3(a.Hkv, a.rows), dim3(kAttnThreads), smem, st, a, scale, lcap);
    return 0;
}

int launch_attn_decode(const AttnDecodeArgs& a, cudaStream_t st) {
    if (a.rows <= 0) return 0;
    const int G = a.H / a.Hkv;
    FSB_CHECK(a.H % a.Hkv == 0, "attention: H %% Hkv != 0");
#define FSB_ATTN_CASE(DH_, G_) \
    if (a.Dh == DH_ && G == G_) return launch_attn_decode_t<DH_, G_>(a, st);
    FSB_ATTN_CASE(128, 1) FSB_ATTN_CASE(128, 2) FSB_ATTN_CASE(128, 4) FSB_ATTN_CASE(128, 8)
    FSB_ATTN_CASE(64, 1) FSB_ATTN_CASE(64, 2) FSB_ATTN_CASE(64, 4) FSB_ATTN_CASE(64, 8)
#undef FSB_ATTN_CASE
    set_error("attention: unsupported head_dim=%d group=%d", a.Dh, G);
    return 1;
}

int launch_swiglu(const SwigluArgs& a, cudaStream_t st) {
    if (a.rows <= 0) return 0;
    FSB_CHECK(a.I % 4 == 0, "swiglu: I=%d unsupported", a.I);
    FSB_CHECK(a.ld % 4 == 0 && (reinterpret_cast<uintptr_t>(a.y) & 15) == 0, "swiglu: misaligned GEMM result");
    FSB_LAUNCH(swiglu_kernel, dim3(cdiv(a.I, 1024), a.rows), dim3(256), 0, st, a);
    return 0;
}

int launch_sample(const SampleArgs& a, cudaStream_t st) {
    if (a.rows <= 0) return 0;
    FSB_CHECK(a.n > 0 && a.n <= kSampleMaxN, "sample: n=%d out of range", a.n);
    FSB_CHECK(a.ctl.state != nullptr || a.top_k >= 1, "sample: top_k must be >= 1");
    FSB_LAUNCH(sample_kernel, dim3(a.rows), dim3(kSampleThreads), 0, st, a);
    return 0;
}

int launch_kv_copy(__nv_bfloat16* cache, int layers, int slots, int Hkv, int S, int Dh, int src, int dst, int n_pos,
                   cudaStream_t st) {
    if (n_pos <= 0 || src == dst) return 0;
    FSB_CHECK(src >= 0 && src < slots && dst >= 0 && dst < slots && n_pos <= S, "kv_copy: bad slot / length");
    FSB_CHECK(Dh % 8 == 0, "kv_copy: head_dim %d", Dh);
    const size_t head16 = static_cast<size_t>(S) * Dh / 8, slot16 = head16 * Hkv, layer16 = slot16 * slots;
    const int n16 = n_pos * (Dh / 8);
    FSB_LAUNCH(kv_copy_kernel, dim3(cdiv(n16, 256 * 4), Hkv, layers), dim3(256), 0, st,
               reinterpret_cast<uint4*>(cache), slot16, head16, layer16, src, dst, n16);
    return 0;
}

int launch_frame_end(const FrameEndArgs& a, cudaStream_t st) {
    FSB_LAUNCH(frame_end_kernel, dim3(a.rows), dim3(32), 0, st, a);
    FSB_LAUNCH(step_inc_kernel, dim3(1), dim3(1), 0, st, a.step);
    return 0;
}

}  // namespace fsb
