// See lm_gemm.cuh.  CTA = 10 warps (6 when operand X needs no normalisation):
//   warps 0-3  TMEM -> registers -> fp32 partial stores of this GEMM
//   warp  4    TMA producer (weights and operand X)
//   warp  5    TMEM allocator + single-thread tcgen05.mma issuer
//   warps 6-9  operand-X normalisers (NORM == 1): RMSNorm of the TMA-delivered residual rows, in place in the ring
// step_finalize_kernel (the consumer-side finish of a GEMM: residual add / SwiGLU) lives here as well.
#include "lm_gemm.cuh"
#include "umma.cuh"

#include <algorithm>
#include <vector>

namespace fsb {

namespace {

constexpr int kBN = kStepRows;
constexpr int kBTileBytes = kBN * kBlockK * 2;  // 4 KB
constexpr int kStageBytes = kATileBytes + kBTileBytes;
constexpr int kTmemCols = 2 * kBN;  // two accumulators: the stores of item n overlap the MMAs of item n+1
constexpr int kEpiThreads = 128;
constexpr int kLoaderThreads = 128;  // four normaliser warps: two 16-byte cells per thread and k-block
constexpr int kScratchBytes = 1024;  // r_s[32] | red[4][32]
// batch rows per finalize unit (measured best): one load round per unit (<= 4 / <= 16 partials), every unit on its own CTA
constexpr int kSwigluRowBlock = 8;
constexpr int kResidRowBlock = 2;

__device__ __forceinline__ void bar_sync(int id, int n) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory");
}

// ---- step_finalize: one unit = rows [j0, j0 + R) x the 128 features of tile `tile` of the PREVIOUS GEMM's output;
// thread tid owns feature tile*128 + tid.  `red` = shared float[4][32]. ----

// Per-row sum over the 128 features of the tile: result for row r in red[q*32 + r], q = 0..3 (one per warp).
template <int R>
__device__ __forceinline__ void rows_warp_sums(const float (&sq)[R], float* red, int quad, int lane) {
    float keep = 0.f;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const float s = warp_sum(sq[r]);
        if (lane == r) keep = s;
    }
    red[quad * 32 + lane] = keep;
}

// Slot-ordered sums of the previous GEMM's partials; up to 32 independent loads in flight per thread.
template <int R, int UQ>  // UQ = partials fetched per round
__device__ __forceinline__ void prev_sums(const StepGemmParams& p, int tile, int tid, int j0, float (&acc)[R]) {
    const int np = __ldg(p.prev.nparts + tile);
    const int maxp = p.prev.max_parts;  // loads are bounded by the launch constant, see step_partial_sums
#pragma unroll
    for (int r = 0; r < R; ++r) acc[r] = 0.f;
    const float* src = p.prev.ws + (static_cast<size_t>(tile) * 32 + j0) * 128 + tid;
    const size_t sstride = static_cast<size_t>(p.prev.tiles) * 32 * 128;
    for (int q0 = 0; q0 < maxp; q0 += UQ) {
        float t[UQ][R];
#pragma unroll
        for (int u = 0; u < UQ; ++u)
#pragma unroll
            for (int r = 0; r < R; ++r)
                t[u][r] = (q0 + u < maxp && j0 + r < p.rows) ? __ldcg(src + static_cast<size_t>(q0 + u) * sstride + r * 128) : 0.f;
#pragma unroll
        for (int u = 0; u < UQ; ++u) {
            if (q0 + u < np) {
#pragma unroll
                for (int r = 0; r < R; ++r) acc[r] += t[u][r];
            }
        }
    }
}

// llama.py:842-845 / 944-946: y = Linear(...) (bf16), x = x + y (bf16); plus sum_i x^2 of this tile per row
template <int R>
__device__ __forceinline__ void pro_resid(const StepGemmParams& p, int tile, int tid, int j0, float* red) {
    const int quad = tid >> 5, lane = tid & 31;
    const int i = tile * 128 + tid;
    const int n = p.prev.n_out;
    const bool ok = i < n;
    // the loads that do not depend on the partials go first: their round trip overlaps the partial sums
    float xin[R];
#pragma unroll
    for (int r = 0; r < R; ++r)
        xin[r] = (p.resid != nullptr && ok && j0 + r < p.rows) ? bf2f(p.resid[static_cast<size_t>(j0 + r) * n + i]) : 0.f;
    const float b = (p.bias != nullptr && ok) ? bf2f(p.bias[i]) : 0.f;
    float acc[R], sq[R];
    prev_sums<R, 32 / R>(p, tile, tid, j0, acc);
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const float y = p.bias != nullptr ? rbf(acc[r] + b) : rbf(acc[r]);
        const float x = p.resid != nullptr ? rbf(xin[r] + y) : y;
        const bool live = ok && j0 + r < p.rows;
        if (live) p.x_out[static_cast<size_t>(j0 + r) * n + i] = f2bf(x);
        sq[r] = live ? x * x : 0.f;
    }
    rows_warp_sums<R>(sq, red, quad, lane);
    bar_sync(1, kEpiThreads);
    if (quad == 0 && lane < R && j0 + lane < p.rows)
        p.ssq_out[(j0 + lane) * kSsqStride + tile] = ((red[lane] + red[32 + lane]) + red[64 + lane]) + red[96 + lane];
    bar_sync(1, kEpiThreads);
}

// llama.py:979-987: h = silu(w1 x) * w3 x, every intermediate a bf16 tensor
template <int R>
__device__ __forceinline__ void pro_swiglu(const StepGemmParams& p, int tile, int tid, int j0) {
    const int quad = tid >> 5, lane = tid & 31;
    const bool hi = (lane & 16) != 0;  // lanes 16..31 hold the w3 ("up") rows of the features lanes 0..15 gate
    const int f = tile * 64 + quad * 16 + (lane & 15);
    float acc[R];
    prev_sums<R, (R == 32 ? 2 : (R == 16 ? 3 : 32 / R))>(p, tile, tid, j0, acc);
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const float up = __shfl_xor_sync(0xffffffffu, acc[r], 16);
        if (!hi && j0 + r < p.rows && f < p.I) {
            const float g = rbf(acc[r]), u = rbf(up);
            const float s = rbf(g / (1.f + expf(-g)));
            p.h[static_cast<size_t>(j0 + r) * p.I + f] = f2bf(s * u);
        }
    }
}

template <int PRO, int R>
__device__ __forceinline__ void pro_units(const StepGemmParams& p, int tid, float* red) {
    const int rblocks = (p.rows + R - 1) / R;
    const int units = p.prev.tiles * rblocks;
    for (int u = blockIdx.x; u < units; u += gridDim.x) {
        const int tile = u % p.prev.tiles, j0 = (u / p.prev.tiles) * R;
        if (PRO == PRO_RESID) pro_resid<R>(p, tile, tid, j0, red);
        else pro_swiglu<R>(p, tile, tid, j0);
    }
}

// step_finalize: finishes the GEMM that produced the next GEMM's operand (one unit = R batch rows x one 128-feature
// tile per CTA); launched between the two GEMMs, so the consumer GEMM finds its operand complete.
template <int PRO>
__global__ void __launch_bounds__(kEpiThreads) step_finalize_kernel(const __grid_constant__ StepGemmParams p) {
    __shared__ float red[4 * 32];
    pdl_launch_dependents();
    pdl_wait();
    switch (p.prev_rb) {
        case 1: pro_units<PRO, 1>(p, threadIdx.x, red); break;
        case 2: pro_units<PRO, 2>(p, threadIdx.x, red); break;
        case 4: pro_units<PRO, 4>(p, threadIdx.x, red); break;
        case 8: pro_units<PRO, 8>(p, threadIdx.x, red); break;
        case 16: pro_units<PRO, 16>(p, threadIdx.x, red); break;
        default: pro_units<PRO, 32>(p, threadIdx.x, red); break;
    }
}

template <int NORM>
__global__ void __launch_bounds__(NORM ? 192 + kLoaderThreads : 192, 2)
step_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const __grid_constant__ StepGemmParams p) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t tiles = (raw + 1023u) & ~1023u;  // SWIZZLE_128B tiles need 1024 B alignment
    const int stages = p.stages;
    const uint32_t bars = tiles + static_cast<uint32_t>(stages) * kStageBytes;
    // barrier block: full[stages] (tile ready for the MMA), empty[stages], rawx[stages] (un-normalised X landed),
    // tmem_full[2], tmem_empty[2], TMEM base word
    const uint32_t full0 = bars, empty0 = bars + 8u * stages, rawx0 = bars + 16u * stages;
    const uint32_t tfull0 = bars + 24u * stages, tempty0 = tfull0 + 16u;
    const uint32_t tmem_slot = tempty0 + 16u + 8u;
    const int scratch_off = ((24 * stages + 56 + 15) / 16) * 16;
    uint8_t* gen = smem_raw + (tiles - raw);
    uint8_t* bar_gen = gen + static_cast<size_t>(stages) * kStageBytes;
    uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(bar_gen + 24 * stages + 40);
    float* scratch = reinterpret_cast<float*>(bar_gen + scratch_off);
    float* r_s = scratch;       // [32] per-row rsqrt (normalisers)
    float* red = scratch + 32;  // [4][32] spare
    uint4* normw_s = reinterpret_cast<uint4*>(bar_gen + scratch_off + kScratchBytes);  // [kblocks*8] norm weights

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int item_begin = p.cta_items[blockIdx.x], item_end = p.cta_items[blockIdx.x + 1];
    unsigned long long* trace = p.trace ? p.trace + static_cast<size_t>(blockIdx.x) * 8 : nullptr;
    if (trace && threadIdx.x == 0) trace[0] = globaltimer_ns();

    if (warp == 4 && lane == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
        for (int s = 0; s < stages; ++s) {
            mbar_init(full0 + 8u * s, 1 + (NORM ? kLoaderThreads / 32 : 0));
            mbar_init(empty0 + 8u * s, 1);
            mbar_init(rawx0 + 8u * s, 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(tfull0 + 8u * a, 1);
            mbar_init(tempty0 + 8u * a, 4);  // one arrival per epilogue warp
        }
        fence_mbar_init();
    }
    if (warp == 5) tmem_alloc(tmem_slot, kTmemCols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;

    pdl_launch_dependents();
    if (warp == 4) {
        // ===== TMA producer. Weights do not depend on the upstream kernel: the first ring-full of weight
        // tiles is requested BEFORE griddepcontrol.wait, so this GEMM's HBM stream starts while the previous
        // kernel is still in its tail. Operand X follows once it is complete. =====
        if (lane == 0) {
            int pre = 0;
            {
                int n = item_begin, kb = 0;
                int4 w = make_int4(0, 0, 0, 0);
                if (n < item_end) {
                    w = p.sched[n];
                    kb = w.y;
                }
                while (n < item_end && pre < stages) {
                    const int s = pre;
                    mbar_expect_tx(full0 + 8u * s, NORM ? kATileBytes : kStageBytes);
                    tma_load_3d(tiles + static_cast<uint32_t>(s) * kStageBytes, &tmA, full0 + 8u * s, kb * kBlockK,
                                w.x * kBlockM, 0, p.a_hint);
                    ++pre;
                    if (++kb >= w.z) {
                        if (++n < item_end) {
                            w = p.sched[n];
                            kb = w.y;
                        }
                    }
                }
            }
            pdl_wait();
            if (trace) trace[1] = globaltimer_ns();
            int it = 0;
            for (int n = item_begin; n < item_end; ++n) {
                const int4 w = p.sched[n];
                for (int kb = w.y; kb < w.z; ++kb, ++it) {
                    const int s = it % stages;
                    const uint32_t ph = static_cast<uint32_t>(it / stages) & 1u;
                    const uint32_t a_dst = tiles + static_cast<uint32_t>(s) * kStageBytes;
                    if (it >= pre) {
                        mbar_wait(empty0 + 8u * s, ph ^ 1u);
                        mbar_expect_tx(full0 + 8u * s, NORM ? kATileBytes : kStageBytes);
                        tma_load_3d(a_dst, &tmA, full0 + 8u * s, kb * kBlockK, w.x * kBlockM, 0, p.a_hint);
                    }
                    if (NORM) {
                        mbar_expect_tx(rawx0 + 8u * s, kBTileBytes);
                        tma_load_3d(a_dst + kATileBytes, &tmB, rawx0 + 8u * s, kb * kBlockK, 0, 0, p.b_hint);
                    } else {
                        tma_load_3d(a_dst + kATileBytes, &tmB, full0 + 8u * s, kb * kBlockK, 0, 0, p.b_hint);
                    }
                }
            }
        }
    } else if (warp == 5) {
        // ===== MMA issuer (one thread) =====
        if (lane == 0) {
            constexpr uint32_t idesc = make_idesc(kBN);
            int it = 0;
            for (int n = item_begin; n < item_end; ++n) {
                const int4 w = p.sched[n];
                const int a = (n - item_begin) & 1;
                const uint32_t aph = static_cast<uint32_t>((n - item_begin) >> 1) & 1u;
                mbar_wait(tempty0 + 8u * a, aph ^ 1u);  // the stores of this accumulator's previous item are done
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(a * kBN);
                uint32_t acc = 0;
                for (int kb = w.y; kb < w.z; ++kb, ++it) {
                    const int s = it % stages;
                    const uint32_t ph = static_cast<uint32_t>(it / stages) & 1u;
                    mbar_wait(full0 + 8u * s, ph);
                    tc_fence_after();
                    const uint32_t a_src = tiles + static_cast<uint32_t>(s) * kStageBytes;
                    const uint64_t ad = make_sdesc(a_src), bd = make_sdesc(a_src + kATileBytes);
#pragma unroll
                    for (int k = 0; k < kBlockK / 16; ++k) {
                        umma_bf16(d_tmem, ad + 2u * k, bd + 2u * k, idesc, acc);
                        acc = 1;
                    }
                    umma_commit(empty0 + 8u * s);  // frees the ring slot once these MMAs retire
                }
                umma_commit(tfull0 + 8u * a);  // accumulator complete
            }
        }
    } else if (warp >= 6) {
        // ===== operand-X normalisers: rbf(rbf(x * r_row) * w) in place on the swizzled tile TMA delivered =====
        if (NORM) {
            const int t = threadIdx.x - 192;  // 0..127
            // the norm weights are constants: stage them before waiting for the upstream kernel
            const int nchunks = ((p.K + kBlockK - 1) / kBlockK) * 8;
            for (int ch = t; ch < nchunks; ch += kLoaderThreads)
                normw_s[ch] = ch * 8 < p.K ? __ldg(reinterpret_cast<const uint4*>(p.norm_w + ch * 8)) : make_uint4(0, 0, 0, 0);
            pdl_wait();
            if (t < 32) {
                // rsqrt(mean(x^2) + eps) of row t: the producer's per-tile sums, added in tile order (all loads in flight)
                // (16-byte loads: every CTA of the grid reads these same 32 lines right after the grid-wide arrival)
                const float4* q = reinterpret_cast<const float4*>(p.x_ssq + t * kSsqStride);
                float4 a[kSsqStride / 4];
#pragma unroll
                for (int u = 0; u < kSsqStride / 4; ++u) a[u] = 4 * u < p.x_nt ? __ldcg(q + u) : make_float4(0.f, 0.f, 0.f, 0.f);
                float tot = 0.f;
#pragma unroll
                for (int u = 0; u < kSsqStride / 4; ++u) {
                    if (4 * u < p.x_nt) tot += a[u].x;
                    if (4 * u + 1 < p.x_nt) tot += a[u].y;
                    if (4 * u + 2 < p.x_nt) tot += a[u].z;
                    if (4 * u + 3 < p.x_nt) tot += a[u].w;
                }
                r_s[t] = rsqrtf(tot / static_cast<float>(p.K) + p.eps);
            }
            bar_sync(2, kLoaderThreads);
            if (trace && t == 0) trace[6] = globaltimer_ns();
            // 32 rows x 8 sixteen-byte chunks per k-block; thread t owns chunk (t & 7) of rows (t >> 3) + 16e
            constexpr int kCells = 256 / kLoaderThreads;
            const int c = t & 7, rb = t >> 3;
            float rr[kCells];
            uint32_t off[kCells];
#pragma unroll
            for (int e = 0; e < kCells; ++e) {
                const int row = rb + (kLoaderThreads / 8) * e;
                rr[e] = r_s[row];
                off[e] = static_cast<uint32_t>(row * 128 + ((c ^ (row & 7)) << 4));  // SWIZZLE_128B
            }
            int it = 0;
            for (int n = item_begin; n < item_end; ++n) {
                const int4 w = p.sched[n];
                for (int kb = w.y; kb < w.z; ++kb, ++it) {
                    const int s = it % stages;
                    const uint32_t ph = static_cast<uint32_t>(it / stages) & 1u;
                    const uint4 wv = normw_s[kb * 8 + c];
                    const float wf[8] = {bf_lo(wv.x), bf_hi(wv.x), bf_lo(wv.y), bf_hi(wv.y),
                                         bf_lo(wv.z), bf_hi(wv.z), bf_lo(wv.w), bf_hi(wv.w)};
                    uint8_t* btile = gen + static_cast<size_t>(s) * kStageBytes + kATileBytes;
                    mbar_wait(rawx0 + 8u * s, ph);
#pragma unroll
                    for (int e = 0; e < kCells; ++e) {
                        uint4* cell = reinterpret_cast<uint4*>(btile + off[e]);
                        const uint4 xv = *cell;
                        const float xf[8] = {bf_lo(xv.x), bf_hi(xv.x), bf_lo(xv.y), bf_hi(xv.y),
                                             bf_lo(xv.z), bf_hi(xv.z), bf_lo(xv.w), bf_hi(xv.w)};
                        float nf[8];
#pragma unroll
                        for (int q = 0; q < 8; ++q) nf[q] = rbf(rbf(xf[q] * rr[e]) * wf[q]);
                        uint4 o;
                        o.x = pack_bf2(nf[0], nf[1]);
                        o.y = pack_bf2(nf[2], nf[3]);
                        o.z = pack_bf2(nf[4], nf[5]);
                        o.w = pack_bf2(nf[6], nf[7]);
                        *cell = o;
                    }
                    fence_proxy_async();  // generic-proxy stores -> visible to the tensor core's async proxy
                    __syncwarp();
                    if (lane == 0) mbar_arrive(full0 + 8u * s);
                    if (trace && t == 0 && it == 0) trace[7] = globaltimer_ns();
                }
            }
        }
    } else {
        // ===== warps 0-3: TMEM -> registers -> fp32 partial stores =====
        const int tid = threadIdx.x;  // 0..127 = TMEM lane = feature inside the tile
        pdl_wait();
        for (int n = item_begin; n < item_end; ++n) {
            const int4 w = p.sched[n];
            const int tile = w.x, slot = w.w;
            const int a = (n - item_begin) & 1;
            const uint32_t aph = static_cast<uint32_t>((n - item_begin) >> 1) & 1u;
            mbar_wait(tfull0 + 8u * a, aph);
            tc_fence_after();
            if (trace && tid == 0 && n == item_begin) trace[4] = globaltimer_ns();
            uint32_t r[32];
            tmem_ld32(tmem_base + (static_cast<uint32_t>(warp * 32) << 16) + static_cast<uint32_t>(a * kBN), r);
            tmem_ld_wait();
            // the accumulator is in registers: hand it back to the MMA warp right away
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty0 + 8u * a);
            float* dst = p.ws + ((static_cast<size_t>(slot) * p.tiles + tile) * 32) * 128 + tid;
#pragma unroll
            for (int j = 0; j < 32; ++j)
                if (j < p.rows) __stcg(dst + j * 128, __uint_as_float(r[j]));
        }
    }
    tc_fence_before();
    __syncthreads();
    if (trace && threadIdx.x == 0) trace[5] = globaltimer_ns();
    if (warp == 5) {
        tc_fence_after();
        tmem_dealloc(tmem_base, kTmemCols);
    }
}

template <int NORM>
int launch_t(const StepGemmPlan& plan, cudaStream_t st) {
    auto k = step_gemm_kernel<NORM>;
    FSB_LAUNCH(k, plan.grid, dim3(NORM ? 192 + kLoaderThreads : 192), plan.smem, st, plan.tmA, plan.tmB, plan.p);
    return 0;
}

const void* kernel_of(int norm) {
    return norm ? reinterpret_cast<const void*>(step_gemm_kernel<1>) : reinterpret_cast<const void*>(step_gemm_kernel<0>);
}

}  // namespace

int step_gemm_init() {
    static bool done = false;
    if (done) return 0;
#define FSB_STEP_ATTR(B_)                                                                                          \
    FSB_CUDA(cudaFuncSetAttribute(step_gemm_kernel<B_>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)); \
    FSB_CUDA(cudaFuncSetAttribute(step_gemm_kernel<B_>, cudaFuncAttributePreferredSharedMemoryCarveout,            \
                                  cudaSharedmemCarveoutMaxShared));
    FSB_STEP_ATTR(1) FSB_STEP_ATTR(0)
#undef FSB_STEP_ATTR
    done = true;
    return 0;
}

int step_plan_init(StepGemmPlan* plan, const __nv_bfloat16* w, int n_out, int K, const __nv_bfloat16* act,
                   bool norm_on_load, int num_ctas, int stages, float* ws, size_t ws_floats) {
    memset(plan, 0, sizeof(*plan));
    FSB_CHECK(K % 8 == 0, "step GEMM: K=%d must be a multiple of 8", K);
    FSB_CHECK(act != nullptr, "step GEMM: operand X missing");
    FSB_CHECK(!norm_on_load || cdiv(K, 128) <= kSsqStride, "step GEMM: normalise-on-load needs K <= %d (K=%d)",
              kSsqStride * 128, K);
    const int norm = norm_on_load ? 1 : 0;
    const void* kernel = kernel_of(norm);
    FSB_TRY(step_gemm_init());
    GemmOperand A{w, K, n_out, 1, K, static_cast<long long>(n_out) * K};
    FSB_TRY(gemm_make_tmap(&plan->tmA, A, kBlockM));
    GemmOperand B{act, K, kStepRows, 1, K, static_cast<long long>(kStepRows) * K};
    FSB_TRY(gemm_make_tmap(&plan->tmB, B, kBN));
    const int tiles = cdiv(n_out, kBlockM), kblocks = cdiv(K, kBlockK);
    const int normw_bytes = norm ? kblocks * 128 : 0;
    auto smem_of = [&](int st) {
        return static_cast<size_t>(1024) + static_cast<size_t>(st) * kStageBytes + ((24 * st + 56 + 15) / 16) * 16 +
               kScratchBytes + normw_bytes;
    };
    while (stages > 2 && 2 * (smem_of(stages) + 1024) > 228 * 1024) --stages;  // two CTAs per SM
    FSB_CHECK(stages >= 2, "step GEMM: ring too shallow");
    // One wave: the stream-K ranges assume every CTA runs at once. cudaOccupancyMaxActiveBlocksPerMultiprocessor reports
    // 1 for every kernel that allocates tensor memory, although two such CTAs do share an SM (verified with %smid
    // stamps): count registers and shared memory ourselves.
    int dev = 0, sms = 0, smem_sm = 0, regs_sm = 0, resv = 0;
    FSB_CUDA(cudaGetDevice(&dev));
    FSB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    FSB_CUDA(cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev));
    FSB_CUDA(cudaDeviceGetAttribute(&regs_sm, cudaDevAttrMaxRegistersPerMultiprocessor, dev));
    FSB_CUDA(cudaDeviceGetAttribute(&resv, cudaDevAttrReservedSharedMemoryPerBlock, dev));
    cudaFuncAttributes fa;
    FSB_CUDA(cudaFuncGetAttributes(&fa, kernel));
    const int threads = norm ? 192 + kLoaderThreads : 192;
    const int regs_cta = ((fa.numRegs + 7) / 8) * 8 * threads;
    const int per_sm = std::min<int>(regs_sm / regs_cta, smem_sm / static_cast<int>(smem_of(stages) + resv + fa.sharedSizeBytes));
    FSB_CHECK(per_sm >= 1, "step GEMM: kernel does not fit an SM (smem %zu, %d registers)", smem_of(stages), fa.numRegs);
    if (num_ctas > per_sm * sms) num_ctas = per_sm * sms;
    // stream-K: units are (tile, k-block) pairs in tile-major order; CTA c streams units [c*U/n, (c+1)*U/n)
    const long long U = static_cast<long long>(tiles) * kblocks;
    if (num_ctas > U) num_ctas = static_cast<int>(U);
    std::vector<int4> items;
    std::vector<int> cta_items(num_ctas + 1, 0), nparts(tiles, 0);
    for (int c = 0; c < num_ctas; ++c) {
        long long u0 = U * c / num_ctas;
        const long long u1 = U * (c + 1) / num_ctas;
        cta_items[c] = static_cast<int>(items.size());
        while (u0 < u1) {
            const int t = static_cast<int>(u0 / kblocks);
            const long long tend = static_cast<long long>(t + 1) * kblocks;
            const long long e = u1 < tend ? u1 : tend;
            items.push_back(make_int4(t, static_cast<int>(u0 - static_cast<long long>(t) * kblocks),
                                      static_cast<int>(e - static_cast<long long>(t) * kblocks), nparts[t]++));
            u0 = e;
        }
    }
    cta_items[num_ctas] = static_cast<int>(items.size());
    int maxp = 0;
    for (int t = 0; t < tiles; ++t) maxp = std::max(maxp, nparts[t]);
    plan->max_parts = maxp;
    FSB_CHECK(static_cast<size_t>(maxp) * tiles * 128 * 32 <= ws_floats, "step GEMM: partial workspace too small");
    FSB_CUDA(cudaMalloc(&plan->sched_dev, items.size() * sizeof(int4)));
    FSB_CUDA(cudaMemcpy(plan->sched_dev, items.data(), items.size() * sizeof(int4), cudaMemcpyHostToDevice));
    FSB_CUDA(cudaMalloc(&plan->cta_items_dev, cta_items.size() * sizeof(int)));
    FSB_CUDA(cudaMemcpy(plan->cta_items_dev, cta_items.data(), cta_items.size() * sizeof(int), cudaMemcpyHostToDevice));
    FSB_CUDA(cudaMalloc(&plan->nparts_dev, tiles * sizeof(int)));
    FSB_CUDA(cudaMemcpy(plan->nparts_dev, nparts.data(), tiles * sizeof(int), cudaMemcpyHostToDevice));
    StepGemmParams& p = plan->p;
    p.sched = reinterpret_cast<const int4*>(plan->sched_dev);
    p.cta_items = plan->cta_items_dev;
    p.tiles = tiles;
    p.stages = stages;
    p.n_out = n_out;
    p.K = K;
    p.rows = kStepRows;
    p.a_hint = kEvictFirst;  // weights are streamed once per step (>> L2)
    p.b_hint = kEvictLast;   // the activation tile is re-read by every CTA
    p.ws = ws;
    p.prev_rb = 32;
    plan->grid = dim3(static_cast<unsigned>(num_ctas), 1, 1);
    plan->smem = smem_of(stages);
    plan->pro = PRO_NONE;
    plan->norm = norm;
    plan->weight_bytes = static_cast<double>(n_out) * K * 2;
    return 0;
}

StepPartials step_plan_partials(const StepGemmPlan& plan) {
    StepPartials P;
    P.ws = plan.p.ws;
    P.nparts = plan.nparts_dev;
    P.tiles = plan.p.tiles;
    P.n_out = plan.p.n_out;
    P.max_parts = plan.max_parts;
    return P;
}

void step_plan_set_prev(StepGemmPlan* plan, int pro, const StepGemmPlan& prev) {
    plan->p.prev = step_plan_partials(prev);
    plan->pro = pro;
}

void step_plan_free(StepGemmPlan* plan) {
    if (plan->sched_dev) cudaFree(plan->sched_dev);
    if (plan->cta_items_dev) cudaFree(plan->cta_items_dev);
    if (plan->nparts_dev) cudaFree(plan->nparts_dev);
    plan->sched_dev = nullptr;
    plan->cta_items_dev = nullptr;
    plan->nparts_dev = nullptr;
}

int step_finalize_launch(const StepGemmPlan& consumer, cudaStream_t st, int rb) {
    // `consumer`'s finalize fields (prev, bias / resid / x_out / ssq_out or h / I, rows) describe the work; one unit per CTA
    const int pro = consumer.pro;
    if (pro == PRO_NONE) return 0;
    StepGemmParams p = consumer.p;
    if (rb <= 0) rb = pro == PRO_SWIGLU ? kSwigluRowBlock : kResidRowBlock;
    FSB_CHECK(rb >= 1 && rb <= 32 && (rb & (rb - 1)) == 0, "finalize: row block %d is not a power of two <= 32", rb);
    p.prev_rb = rb;
    const int units = p.prev.tiles * cdiv(p.rows, rb);
    if (pro == PRO_RESID) FSB_LAUNCH(step_finalize_kernel<PRO_RESID>, dim3(units), dim3(kEpiThreads), 0, st, p);
    else FSB_LAUNCH(step_finalize_kernel<PRO_SWIGLU>, dim3(units), dim3(kEpiThreads), 0, st, p);
    return 0;
}

int step_gemm_launch(const StepGemmPlan& plan, cudaStream_t st) {
    return plan.norm ? launch_t<1>(plan, st) : launch_t<0>(plan, st);
}

}  // namespace fsb
