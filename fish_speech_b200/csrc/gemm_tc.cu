// tcgen05 / TMEM / TMA multi-tap GEMM — see gemm_tc.cuh for the contract.
//
// CTA = 192 threads: warps 0-3 epilogue (TMEM lane quadrant = warp id), warp 4 TMA producer,
// warp 5 TMEM allocator + single-thread MMA issuer.  smem ring of `stages` x {A 128x64 bf16 (16 KB),
// B BNx64 bf16}, both written by TMA with SWIZZLE_128B and consumed through UMMA shared-memory
// descriptors (K-major, SBO = 1024 B).  A CTA runs one output tile, or a stream-K range of segments
// with two TMEM accumulators so the epilogue of segment n overlaps the MMAs of segment n+1.
#include "gemm_tc.cuh"
#include "umma.cuh"

#include <vector>

namespace fsb {

int gemm_init();

namespace {


__device__ __forceinline__ float gelu_erf(float x) {
    return 0.5f * x * (1.f + erff(x * 0.70710678118654752440f));
}

// Direct epilogue for one 32-column chunk of an accumulator row:
//   bias -> GELU -> gamma -> +residual -> tanh -> store raw (out0) and/or Snake-activated (out1).
// Fast path (channels on the columns, bf16 outputs contiguous along the columns, full chunk): per-column
// parameters come in as float4 broadcast loads, 8 columns are processed at a time to keep the register
// footprint small, sin() is the MUFU approximation (arguments are O(10), outputs are bf16).
__device__ __forceinline__ float snake_fast(float v, float a, float ia) {
    const float s = __sinf(a * v);
    return fmaf(ia * s, s, v);
}

__device__ __forceinline__ bool epilogue_fast(const GemmParams& p, int jbase) {
    return !p.chan_on_i && (p.o_js == 1) && !p.out_f32 && ((p.o_is & 7) == 0) && ((p.o_zs & 7) == 0) &&
           (jbase + 32 <= p.rows_j);
}

// The residual of a chunk (4 x 16 bytes per thread) is requested BEFORE the accumulator is read from TMEM and
// before any store of the chunk: the stores may alias the residual buffer (in-place residual stream), so the
// compiler cannot hoist these loads itself, and one 16-byte load in flight per thread left the 1x1 convs of
// the wide-time blocks latency-bound at ~2 TB/s.
__device__ __forceinline__ void epilogue_preload(const GemmParams& p, int i, int jbase, int z, uint4 (&rr)[4]) {
    if (p.resid == nullptr || !epilogue_fast(p, jbase)) return;
    const size_t rowoff = static_cast<size_t>(z) * p.o_zs + static_cast<size_t>(i) * p.o_is;
#pragma unroll
    for (int q = 0; q < 4; ++q) rr[q] = *reinterpret_cast<const uint4*>(p.resid + rowoff + jbase + q * 8);
}

template <int BN>
__device__ __forceinline__ void epilogue_chunk(const GemmParams& p, const uint32_t* r, const uint4 (&rr)[4], int i,
                                               int jbase, int z) {
    const size_t zoff = static_cast<size_t>(z) * p.o_zs;
    const size_t rowoff = zoff + static_cast<size_t>(i) * p.o_is;
    const bool fast = epilogue_fast(p, jbase);
    if (fast) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int j = jbase + q * 8;
            float v[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) v[e] = __uint_as_float(r[q * 8 + e]);
            if (p.bias) {
                const float4 b0 = __ldg(reinterpret_cast<const float4*>(p.bias + j));
                const float4 b1 = __ldg(reinterpret_cast<const float4*>(p.bias + j + 4));
                v[0] += b0.x; v[1] += b0.y; v[2] += b0.z; v[3] += b0.w;
                v[4] += b1.x; v[5] += b1.y; v[6] += b1.z; v[7] += b1.w;
            }
            if (p.act == ACT_GELU) {
#pragma unroll
                for (int e = 0; e < 8; ++e) v[e] = gelu_erf(v[e]);
            }
            if (p.gamma) {
                const float4 g0 = __ldg(reinterpret_cast<const float4*>(p.gamma + j));
                const float4 g1 = __ldg(reinterpret_cast<const float4*>(p.gamma + j + 4));
                v[0] *= g0.x; v[1] *= g0.y; v[2] *= g0.z; v[3] *= g0.w;
                v[4] *= g1.x; v[5] *= g1.y; v[6] *= g1.z; v[7] *= g1.w;
            }
            if (p.resid) {
                const uint4 u = rr[q];
                v[0] += bf_lo(u.x); v[1] += bf_hi(u.x); v[2] += bf_lo(u.y); v[3] += bf_hi(u.y);
                v[4] += bf_lo(u.z); v[5] += bf_hi(u.z); v[6] += bf_lo(u.w); v[7] += bf_hi(u.w);
            }
            if (p.act == ACT_TANH) {
#pragma unroll
                for (int e = 0; e < 8; ++e) v[e] = tanhf(v[e]);
            }
            if (p.out0) {
                uint4 u;
                u.x = pack_bf2(v[0], v[1]); u.y = pack_bf2(v[2], v[3]);
                u.z = pack_bf2(v[4], v[5]); u.w = pack_bf2(v[6], v[7]);
                *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.out0) + rowoff + j) = u;
            }
            if (p.out1) {
                const float4 a0 = __ldg(reinterpret_cast<const float4*>(p.snake_alpha + j));
                const float4 a1 = __ldg(reinterpret_cast<const float4*>(p.snake_alpha + j + 4));
                const float4 i0 = __ldg(reinterpret_cast<const float4*>(p.snake_inv_alpha + j));
                const float4 i1 = __ldg(reinterpret_cast<const float4*>(p.snake_inv_alpha + j + 4));
                uint4 u;
                u.x = pack_bf2(snake_fast(v[0], a0.x, i0.x), snake_fast(v[1], a0.y, i0.y));
                u.y = pack_bf2(snake_fast(v[2], a0.z, i0.z), snake_fast(v[3], a0.w, i0.w));
                u.z = pack_bf2(snake_fast(v[4], a1.x, i1.x), snake_fast(v[5], a1.y, i1.y));
                u.w = pack_bf2(snake_fast(v[6], a1.z, i1.z), snake_fast(v[7], a1.w, i1.w));
                *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.out1) + rowoff + j) = u;
            }
        }
        return;
    }
    // generic path (ragged chunks, fp32 outputs, channels on the lanes)
#pragma unroll
    for (int jj = 0; jj < 32; ++jj) {
        const int j = jbase + jj;
        if (j >= p.rows_j) continue;
        const int c = p.chan_on_i ? i : j;
        float x = __uint_as_float(r[jj]);
        if (p.bias) x += p.bias[c];
        if (p.act == ACT_GELU) x = gelu_erf(x);
        if (p.gamma) x *= p.gamma[c];
        const size_t idx = rowoff + static_cast<size_t>(j) * p.o_js;
        if (p.resid) x += bf2f(p.resid[idx]);
        if (p.act == ACT_TANH) x = tanhf(x);
        if (p.out0) {
            if (p.out_f32) reinterpret_cast<float*>(p.out0)[idx] = x;
            else reinterpret_cast<__nv_bfloat16*>(p.out0)[idx] = f2bf(x);
        }
        if (p.out1) {
            const float y = snake_fast(x, p.snake_alpha[c], p.snake_inv_alpha[c]);
            if (p.out_f32) reinterpret_cast<float*>(p.out1)[idx] = y;
            else reinterpret_cast<__nv_bfloat16*>(p.out1)[idx] = f2bf(y);
        }
    }
}

// MODE 0: fp32 partial sums to the workspace (decode / prefill of the LM). Lean in registers and shared
//         memory so that TWO CTAs fit on an SM: the CTA of the next GEMM in the stream becomes resident
//         (programmatic dependent launch) and prefetches its weight tiles while this one still runs.
// MODE 1: direct fused epilogue (codec convolutions / linears).
template <int MODE>
struct GemmRoles {
    static constexpr int kEpiWarps = MODE == 0 ? 4 : 8;  // MODE 1: two warps per TMEM lane quadrant
    static constexpr int kThreads = (kEpiWarps + 2) * 32;
};

template <int BN, int MODE>
__global__ void __launch_bounds__(GemmRoles<MODE>::kThreads, (MODE == 0 || BN <= 128) ? 2 : 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ GemmParams p) {
    extern __shared__ uint8_t smem_raw[];
    constexpr int kBTileBytes = BN * kBlockK * 2;
    constexpr int kStageBytes = kATileBytes + kBTileBytes;
    // two accumulators: epilogue of item n overlaps MMA of n+1 (allocation size must be a power of two)
    constexpr int kTmemCols = BN == 192 ? 512 : 2 * BN;
    constexpr int kEpiWarps = GemmRoles<MODE>::kEpiWarps;
    constexpr int kProducerWarp = kEpiWarps, kMmaWarp = kEpiWarps + 1;

    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t tiles = (raw + 1023u) & ~1023u;  // SWIZZLE_128B tiles need 1024 B alignment
    const int stages = p.stages;
    const uint32_t bars = tiles + static_cast<uint32_t>(stages) * kStageBytes;
    // barrier block: full[stages], empty[stages], tmem_full[2], tmem_empty[2], TMEM base word
    const uint32_t full0 = bars, empty0 = bars + 8u * stages, tfull0 = bars + 16u * stages;
    const uint32_t tempty0 = tfull0 + 16u;
    const uint32_t tmem_slot = tempty0 + 16u;
    uint32_t* tmem_slot_ptr =
        reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - raw));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    // Work items of this CTA: a stream-K range (several segments, each of one output tile), a range of
    // the persistent tiled schedule, or the single tile named by blockIdx.
    int item_begin = 0, item_end = 1;
    if (p.sched != nullptr) {
        item_begin = p.cta_items[blockIdx.x];
        item_end = p.cta_items[blockIdx.x + 1];
    } else if (p.tiled_total > 0) {
        item_begin = static_cast<int>(static_cast<long long>(p.tiled_total) * blockIdx.x / gridDim.x);
        item_end = static_cast<int>(static_cast<long long>(p.tiled_total) * (blockIdx.x + 1) / gridDim.x);
    }
    int z = blockIdx.z;
    auto get_item = [&](int n, int& i0, int& j0, int& kb0, int& kb1, int& slot) {
        if (p.sched != nullptr) {
            const int4 w = p.sched[n];
            i0 = (w.x & 0xffff) * kBlockM;
            j0 = ((w.x >> 16) & 0xffff) * BN;
            kb0 = w.y;
            kb1 = w.z;
            slot = w.w;
        } else if (p.tiled_total > 0) {
            const int per_z = p.tiled_ti * p.tiled_tj;
            z = n / per_z;
            const int rem = n - z * per_z;
            const int ti = rem / p.tiled_tj;
            i0 = ti * kBlockM;
            j0 = (rem - ti * p.tiled_tj) * BN;
            kb0 = 0;
            kb1 = p.kb_per_tap * p.num_taps;
            slot = 0;
        } else {
            i0 = blockIdx.x * kBlockM;
            j0 = blockIdx.y * BN;
            kb0 = 0;
            kb1 = p.kb_per_tap * p.num_taps;
            slot = 0;
        }
    };

    if (warp == kProducerWarp && lane == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
        for (int s = 0; s < stages; ++s) {
            mbar_init(full0 + 8u * s, 1);
            mbar_init(empty0 + 8u * s, 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(tfull0 + 8u * a, 1);
            mbar_init(tempty0 + 8u * a, kEpiWarps);  // one arrival per epilogue warp
        }
        fence_mbar_init();
    }
    if (warp == kMmaWarp) tmem_alloc(tmem_slot, kTmemCols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;

    pdl_launch_dependents();  // let the consumer kernel get resident; it blocks in griddepcontrol.wait
    if (warp == kProducerWarp) {
        // ===== TMA producer: the ring keeps flowing across item boundaries =====
        // Operand A (weights when a_static) does not depend on the upstream kernel: its tiles for the
        // whole ring are requested BEFORE griddepcontrol.wait, so the HBM stream of this GEMM starts
        // while the previous kernel (a small consumer kernel) is still running. Operand B (the
        // activations that kernel produces) is only fetched after the wait.
        if (lane == 0) {
            int it = 0;
            int pre = 0;  // ring slots whose A tile was requested early
            if (p.a_static) {
                int n = item_begin, kb = 0, i0 = 0, j0 = 0, kb0 = 0, kb1 = 0, slot = 0;
                if (n < item_end) {
                    get_item(n, i0, j0, kb0, kb1, slot);
                    kb = kb0;
                }
                while (n < item_end && pre < stages) {
                    const int s = pre;
                    mbar_expect_tx(full0 + 8u * s, kStageBytes);
                    const int tap = kb / p.kb_per_tap;
                    const int kc = (kb - tap * p.kb_per_tap) * kBlockK;
                    tma_load_3d(tiles + static_cast<uint32_t>(s) * kStageBytes, &tmA, full0 + 8u * s,
                                p.a_tapk * tap + kc, i0 + p.a_shift[tap], p.a_batched ? z : 0, p.a_hint);
                    ++pre;
                    if (++kb >= kb1) {
                        if (++n < item_end) {
                            get_item(n, i0, j0, kb0, kb1, slot);
                            kb = kb0;
                        }
                    }
                }
            }
            pdl_wait();
            for (int n = item_begin; n < item_end; ++n) {
                int i0, j0, kb0, kb1, slot;
                get_item(n, i0, j0, kb0, kb1, slot);
                for (int kb = kb0; kb < kb1; ++kb, ++it) {
                    const int s = it % stages;
                    const uint32_t ph = static_cast<uint32_t>(it / stages) & 1u;
                    const int tap = kb / p.kb_per_tap;
                    const int kc = (kb - tap * p.kb_per_tap) * kBlockK;
                    const uint32_t a_dst = tiles + static_cast<uint32_t>(s) * kStageBytes;
                    if (it >= pre) {
                        mbar_wait(empty0 + 8u * s, ph ^ 1u);
                        mbar_expect_tx(full0 + 8u * s, kStageBytes);
                        tma_load_3d(a_dst, &tmA, full0 + 8u * s, p.a_tapk * tap + kc,
                                    i0 + p.a_shift[tap], p.a_batched ? z : 0, p.a_hint);
                    }
                    tma_load_3d(a_dst + kATileBytes, &tmB, full0 + 8u * s, p.b_tapk * tap + kc,
                                j0 + p.b_shift[tap], p.b_batched ? z : 0, p.b_hint);
                }
            }
        }
    } else if (warp == kMmaWarp) {
        // ===== MMA issuer (one thread) =====
        if (lane == 0) {
            constexpr uint32_t idesc = make_idesc(BN);
            int it = 0;
            for (int n = item_begin; n < item_end; ++n) {
                int i0, j0, kb0, kb1, slot;
                get_item(n, i0, j0, kb0, kb1, slot);
                const int a = (n - item_begin) & 1;
                const uint32_t aph = static_cast<uint32_t>((n - item_begin) >> 1) & 1u;
                mbar_wait(tempty0 + 8u * a, aph ^ 1u);  // epilogue has drained this accumulator
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(a * BN);
                uint32_t acc = 0;
                for (int kb = kb0; kb < kb1; ++kb, ++it) {
                    const int s = it % stages;
                    const uint32_t ph = static_cast<uint32_t>(it / stages) & 1u;
                    mbar_wait(full0 + 8u * s, ph);
                    tc_fence_after();
                    const uint32_t a_src = tiles + static_cast<uint32_t>(s) * kStageBytes;
                    const uint64_t ad = make_sdesc(a_src), bd = make_sdesc(a_src + kATileBytes);
#pragma unroll
                    for (int k = 0; k < kBlockK / 16; ++k) {
                        // advance 16 elements (32 B) along K inside the swizzle atom: +2 (16 B units)
                        umma_bf16(d_tmem, ad + 2u * k, bd + 2u * k, idesc, acc);
                        acc = 1;
                    }
                    umma_commit(empty0 + 8u * s);  // frees the smem slot once these MMAs retire
                }
                umma_commit(tfull0 + 8u * a);  // accumulator complete
            }
        }
    } else {
        // ===== epilogue: TMEM -> registers -> global =====
        for (int n = item_begin; n < item_end; ++n) {
            int i0, j0, kb0, kb1, slot;
            get_item(n, i0, j0, kb0, kb1, slot);
            const int a = (n - item_begin) & 1;
            const uint32_t aph = static_cast<uint32_t>((n - item_begin) >> 1) & 1u;
            mbar_wait(tfull0 + 8u * a, aph);
            tc_fence_after();
            const int quad = warp & 3, half = warp >> 2;  // TMEM lane quadrant is fixed by warp id % 4
            const int i = i0 + quad * 32 + lane;
            const bool i_ok = i < p.rows_i;
            const uint32_t taddr =
                tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + static_cast<uint32_t>(a * BN);
            if (MODE == 0) {
                float* base = p.ws + static_cast<size_t>(slot) * p.ws_slot_stride;
#pragma unroll 1
                for (int c0 = 0; c0 < BN; c0 += 32) {
                    uint32_t r[32];
                    tmem_ld32(taddr + c0, r);
                    tmem_ld_wait();
                    if (i_ok) {
#pragma unroll
                        for (int jj = 0; jj < 32; ++jj) {
                            const int j = j0 + c0 + jj;
                            if (j < p.rows_j)
                                base[static_cast<size_t>(j) * p.ws_ld + i] = __uint_as_float(r[jj]);
                        }
                    }
                }
            } else {
                // the two warps of a lane quadrant take alternate 32-column chunks
#pragma unroll 1
                for (int c0 = half * 32; c0 < BN; c0 += 32 * (kEpiWarps / 4)) {
                    uint32_t r[32];
                    uint4 rr[4];
                    const bool live = i_ok && j0 + c0 < p.rows_j;
                    if (live) epilogue_preload(p, i, j0 + c0, z, rr);
                    tmem_ld32(taddr + c0, r);
                    tmem_ld_wait();
                    if (live) epilogue_chunk<BN>(p, r, rr, i, j0 + c0, z);
                }
            }
            // release the accumulator to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty0 + 8u * a);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == kMmaWarp) {
        tc_fence_after();
        tmem_dealloc(tmem_base, kTmemCols);
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (fn) return fn;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || p == nullptr) {
        set_error("cudaGetDriverEntryPoint(cuTensorMapEncodeTiled) failed: %s",
                  cudaGetErrorString(e));
        return nullptr;
    }
    fn = reinterpret_cast<EncodeTiledFn>(p);
    return fn;
}

}  // namespace

int gemm_make_tmap(CUtensorMap* tm, const GemmOperand& op, int box_rows) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) return 1;
    FSB_CHECK((reinterpret_cast<uintptr_t>(op.ptr) & 15) == 0, "TMA operand not 16-byte aligned");
    FSB_CHECK((op.row_stride * 2) % 16 == 0 && (op.batch_stride * 2) % 16 == 0,
              "TMA strides must be multiples of 16 bytes (row_stride=%lld batch_stride=%lld)",
              op.row_stride, op.batch_stride);
    FSB_CHECK(op.k > 0 && op.rows > 0 && op.batch > 0, "empty TMA operand");
    cuuint64_t dims[3] = {static_cast<cuuint64_t>(op.k), static_cast<cuuint64_t>(op.rows),
                          static_cast<cuuint64_t>(op.batch)};
    cuuint64_t strides[2] = {static_cast<cuuint64_t>(op.row_stride) * 2,
                             static_cast<cuuint64_t>(op.batch_stride > 0 ? op.batch_stride
                                                                         : op.row_stride * op.rows) *
                                 2};
    cuuint32_t box[3] = {kBlockK, static_cast<cuuint32_t>(box_rows), 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<__nv_bfloat16*>(op.ptr),
                    dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    FSB_CHECK(r == CUDA_SUCCESS,
              "cuTensorMapEncodeTiled failed (%d): k=%lld rows=%lld batch=%lld rs=%lld bs=%lld",
              static_cast<int>(r), op.k, op.rows, op.batch, op.row_stride, op.batch_stride);
    return 0;
}

namespace {

template <int BN, int MODE>
int launch_bn_mode(const GemmPlan& plan, cudaStream_t stream) {
    auto k = gemm_tc_kernel<BN, MODE>;
    FSB_LAUNCH(k, plan.grid, dim3(GemmRoles<MODE>::kThreads), plan.smem, stream, plan.tmA, plan.tmB, plan.p);
    return 0;
}

template <int BN>
int launch_bn(const GemmPlan& plan, cudaStream_t stream) {
    static bool attr_set = false;
    if (!attr_set) {
        FSB_TRY(gemm_init());
        attr_set = true;
    }
    return plan.p.mode == 0 ? launch_bn_mode<BN, 0>(plan, stream) : launch_bn_mode<BN, 1>(plan, stream);
}

}  // namespace

int gemm_plan_init(GemmPlan* plan, const GemmOperand& A, const GemmOperand& B, int bn, int stages,
                   int tiles_i, int tiles_j, int batch) {
    FSB_CHECK(bn == 32 || bn == 64 || bn == 128 || bn == 192 || bn == 256, "unsupported BN %d", bn);
    FSB_TRY(gemm_make_tmap(&plan->tmA, A, kBlockM));
    FSB_TRY(gemm_make_tmap(&plan->tmB, B, bn));
    const int stage_bytes = kATileBytes + bn * kBlockK * 2;
    const int max_stages = (227 * 1024 - 1024 - 256) / stage_bytes;
    if (stages > max_stages) stages = max_stages;
    if (stages > kMaxStages) stages = kMaxStages;
    FSB_CHECK(stages >= 2, "not enough shared memory for 2 stages");
    plan->bn = bn;
    plan->p.stages = stages;
    plan->smem = static_cast<size_t>(stages) * stage_bytes + 1024 + 16 * stages + 64;
    plan->grid = dim3(tiles_i, tiles_j, batch);
    plan->p.sched = nullptr;
    plan->p.cta_items = nullptr;
    plan->cta_items_dev = nullptr;
    plan->sched_dev = nullptr;
    plan->nparts_dev = nullptr;
    plan->max_parts = 1;
    if (plan->p.a_hint == 0) plan->p.a_hint = kEvictNormal;
    if (plan->p.b_hint == 0) plan->p.b_hint = kEvictNormal;
    return 0;
}

int gemm_plan_streamk(GemmPlan* plan, int tiles_i, int kblocks, int num_ctas, bool keep_empty_ctas) {
    // Units are (tile, k-block) pairs in tile-major order; CTA c streams units [c*U/n, (c+1)*U/n).
    // Where that range crosses a tile boundary it becomes several items (one per tile touched); the
    // CTA runs them back to back with the TMA ring never draining, so every SM pulls the same number
    // of weight bytes. Partials of tile t land in workspace slots [0, nparts[t]).
    const long long U = static_cast<long long>(tiles_i) * kblocks;
    if (num_ctas > U && !keep_empty_ctas) num_ctas = static_cast<int>(U);
    std::vector<int4> items;
    std::vector<int> cta_items(num_ctas + 1, 0);
    std::vector<int> nparts(tiles_i, 0);
    for (int c = 0; c < num_ctas; ++c) {
        long long u0 = U * c / num_ctas, u1 = U * (c + 1) / num_ctas;
        cta_items[c] = static_cast<int>(items.size());
        while (u0 < u1) {
            const int t = static_cast<int>(u0 / kblocks);
            const long long tend = static_cast<long long>(t + 1) * kblocks;
            const long long e = u1 < tend ? u1 : tend;
            int4 w;
            w.x = t;  // tile_j = 0
            w.y = static_cast<int>(u0 - static_cast<long long>(t) * kblocks);
            w.z = static_cast<int>(e - static_cast<long long>(t) * kblocks);
            w.w = nparts[t]++;
            items.push_back(w);
            u0 = e;
        }
    }
    cta_items[num_ctas] = static_cast<int>(items.size());
    int maxp = 0;
    for (int t = 0; t < tiles_i; ++t) maxp = nparts[t] > maxp ? nparts[t] : maxp;
    plan->max_parts = maxp;
    FSB_CUDA(cudaMalloc(&plan->sched_dev, items.size() * sizeof(int4)));
    FSB_CUDA(cudaMemcpy(plan->sched_dev, items.data(), items.size() * sizeof(int4),
                        cudaMemcpyHostToDevice));
    FSB_CUDA(cudaMalloc(&plan->cta_items_dev, cta_items.size() * sizeof(int)));
    FSB_CUDA(cudaMemcpy(plan->cta_items_dev, cta_items.data(), cta_items.size() * sizeof(int),
                        cudaMemcpyHostToDevice));
    FSB_CUDA(cudaMalloc(&plan->nparts_dev, tiles_i * sizeof(int)));
    FSB_CUDA(cudaMemcpy(plan->nparts_dev, nparts.data(), tiles_i * sizeof(int),
                        cudaMemcpyHostToDevice));
    plan->p.sched = reinterpret_cast<const int4*>(plan->sched_dev);
    plan->p.cta_items = plan->cta_items_dev;
    plan->grid = dim3(static_cast<unsigned>(num_ctas), 1, 1);
    return 0;
}

int gemm_plan_tiled(GemmPlan* plan, int tiles_i, int tiles_j, int batch, int ctas_per_sm) {
    const long long total = static_cast<long long>(tiles_i) * tiles_j * batch;
    FSB_CHECK(total > 0 && total < (1ll << 31), "gemm_plan_tiled: bad tile count");
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // persistent CTAs: one per SM, or two where shared memory and TMEM allow (narrow tiles: more epilogue
    // warps in flight for the memory-bound layers)
    const long long slots = static_cast<long long>(sms) * (ctas_per_sm > 1 ? 2 : 1);
    const long long ctas = total < slots ? total : slots;
    plan->p.tiled_total = static_cast<int>(total);
    plan->p.tiled_ti = tiles_i;
    plan->p.tiled_tj = tiles_j;
    plan->grid = dim3(static_cast<unsigned>(ctas), 1, 1);
    return 0;
}

void gemm_plan_free(GemmPlan* plan) {
    if (plan->sched_dev) cudaFree(plan->sched_dev);
    if (plan->nparts_dev) cudaFree(plan->nparts_dev);
    if (plan->cta_items_dev) cudaFree(plan->cta_items_dev);
    plan->cta_items_dev = nullptr;
    plan->sched_dev = nullptr;
    plan->nparts_dev = nullptr;
}

int gemm_init() {
    // opt every instantiation into the large dynamic shared-memory carve-out up front, so that no
    // attribute call is needed later (e.g. while a stream is being captured into a CUDA graph)
#define FSB_GEMM_ATTR(BN_, M_)                                                                       \
    FSB_CUDA(cudaFuncSetAttribute(gemm_tc_kernel<BN_, M_>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                  227 * 1024));                                                        \
    FSB_CUDA(cudaFuncSetAttribute(gemm_tc_kernel<BN_, M_>, cudaFuncAttributePreferredSharedMemoryCarveout, \
                                  cudaSharedmemCarveoutMaxShared));
    FSB_GEMM_ATTR(32, 0) FSB_GEMM_ATTR(64, 0) FSB_GEMM_ATTR(128, 0) FSB_GEMM_ATTR(256, 0)
    FSB_GEMM_ATTR(32, 1) FSB_GEMM_ATTR(64, 1) FSB_GEMM_ATTR(128, 1) FSB_GEMM_ATTR(256, 1)
    FSB_GEMM_ATTR(192, 0) FSB_GEMM_ATTR(192, 1)
#undef FSB_GEMM_ATTR
    return 0;
}

int gemm_launch(const GemmPlan& plan, cudaStream_t stream) {
    switch (plan.bn) {
        case 32: return launch_bn<32>(plan, stream);
        case 64: return launch_bn<64>(plan, stream);
        case 128: return launch_bn<128>(plan, stream);
        case 192: return launch_bn<192>(plan, stream);
        case 256: return launch_bn<256>(plan, stream);
    }
    set_error("gemm_launch: bad BN %d", plan.bn);
    return 1;
}

}  // namespace fsb
