// Tiled attention on the tensor cores for MANY query rows per sequence: LM prefill (llama.py:916-934 with S > 1) and the
// codec's window-limited transformer (modded_dac.py:380-398).  A kernel per row would re-read the whole K/V history of
// a row from L2 for every row: O(L^2) bytes and CUDA-core dot products.  Here one CTA takes 64 consecutive rows of one
// query head: K/V tiles of 64 positions are staged once in shared memory (cp.async, double buffered) and shared by the
// 64 rows, S = Q K^T and O += P V run on mma.sync m16n8k16 (bf16 in, fp32 accumulate; the probabilities as a bf16
// hi + lo pair), the softmax is the online (running max / running sum) form in fp32.
//
// Each row has its own (sequence, position).  A tile is split into runs of consecutive positions of one sequence; each
// run is processed against its own K/V range with the other rows masked (a fully masked K tile leaves a row's running
// state untouched).  K tiles are aligned to absolute multiples of 64 positions and a row's result only depends on its
// own positions, so a prompt gives the same bits however it is cut into prefill chunks or grouped into tiles (prefix
// reuse relies on this).
#include "lm_kernels.cuh"

namespace fsb {

namespace {

constexpr int kTQ = 64, kTK = 64, kAtThreads = 128;

__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], uint32_t addr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t (&r)[4], uint32_t addr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void mma_bf16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, bool valid) {
    const int n = valid ? 16 : 0;  // 0 source bytes: the 16 destination bytes are zero-filled
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <int DH>
__global__ void __launch_bounds__(kAtThreads) attn_tile_kernel(AttnArgs a, float scale_log2e) {
    constexpr int CH = DH / 8;        // 16-byte chunks per row
    constexpr int KS = DH / 16;       // k-steps of Q K^T
    constexpr int NT = DH / 8;        // 8-wide output tiles of O
    constexpr int ROWB = DH * 2;      // bytes per row
    constexpr int TILEB = kTK * ROWB;  // bytes per K or V tile
    extern __shared__ __align__(128) uint8_t sm[];
    __shared__ int s_seq[kTQ], s_pos[kTQ];
    const uint32_t sQ = smem_u32(sm), sK = sQ + kTQ * ROWB, sV = sK + 2 * TILEB;
    const int head = blockIdx.y, g = head / (a.H / a.Hkv);
    const int r0 = blockIdx.x * kTQ;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    pdl_launch_dependents();
    pdl_wait();
    if (tid < kTQ) {
        const int r = r0 + tid;
        s_seq[tid] = r < a.rows ? a.row_seq[r] : -1;
        s_pos[tid] = r < a.rows ? a.row_pos[r] : -1;
    }
    // the swizzle: 16-byte chunk c of row i sits at chunk c ^ (i & 7) -- ldmatrix reads 8 rows x 16 bytes conflict-free
    for (int e = tid; e < kTQ * CH; e += kAtThreads) {
        const int i = e / CH, c = e - i * CH;
        uint4 u = make_uint4(0, 0, 0, 0);
        if (r0 + i < a.rows) u = *reinterpret_cast<const uint4*>(a.q + (static_cast<size_t>(r0 + i) * a.H + head) * DH + c * 8);
        *reinterpret_cast<uint4*>(sm + i * ROWB + ((c ^ (i & 7)) << 4)) = u;
    }
    __syncthreads();
    uint32_t qf[KS][4];
    {
        const int row = warp * 16 + (lane & 15);
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) ldsm_x4(qf[ks], sQ + row * ROWB + (((ks * 2 + (lane >> 4)) ^ (row & 7)) << 4));
    }
    const int qi0 = warp * 16 + (lane >> 2), qi1 = qi0 + 8;  // this thread's two rows of the tile
    float m[2] = {-INFINITY, -INFINITY}, l[2] = {0.f, 0.f};
    float o[NT][4];
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) o[nt][e] = 0.f;

    auto load_tile = [&](int buf, const __nv_bfloat16* kbase, const __nv_bfloat16* vbase, int kt, int hi) {
        for (int e = tid; e < kTK * CH; e += kAtThreads) {
            const int i = e / CH, c = e - i * CH;
            const bool ok = kt + i <= hi;
            const size_t off = static_cast<size_t>(ok ? kt + i : 0) * DH + c * 8;
            const uint32_t d = buf * TILEB + i * ROWB + ((c ^ (i & 7)) << 4);
            cp_async16(sK + d, kbase + off, ok);
            cp_async16(sV + d, vbase + off, ok);
        }
        cp_async_commit();
    };

    int start = 0;
    while (start < kTQ) {
        const int seq = s_seq[start], p0 = s_pos[start];
        int end = start + 1;
        while (end < kTQ && s_seq[end] == seq && s_pos[end] == p0 + (end - start)) ++end;
        if (seq >= 0 && p0 >= 0) {
            // ---- one run: rows [start, end) = positions p0 .. p0 + (end - start) - 1 of sequence `seq` ----
            const int hi = min(p0 + (end - start) - 1, a.S - 1);
            const int lo = a.window > 0 ? max(0, p0 - a.window + 1) : 0;
            const size_t cbase = (static_cast<size_t>(seq) * a.Hkv + g) * a.S * DH;
            const __nv_bfloat16* kbase = a.kcache + cbase;
            const __nv_bfloat16* vbase = a.vcache + cbase;
            const bool v0 = qi0 >= start && qi0 < end, v1 = qi1 >= start && qi1 < end;
            const int pq0 = p0 + (qi0 - start), pq1 = p0 + (qi1 - start);
            const int lo0 = a.window > 0 ? pq0 - a.window + 1 : 0, lo1 = a.window > 0 ? pq1 - a.window + 1 : 0;
            const int kt0 = (lo / kTK) * kTK;
            int buf = 0;
            __syncthreads();  // the previous run's last tile has been consumed
            load_tile(0, kbase, vbase, kt0, hi);
            for (int kt = kt0; kt <= hi; kt += kTK) {
                const bool more = kt + kTK <= hi;
                if (more) {
                    load_tile(buf ^ 1, kbase, vbase, kt + kTK, hi);
                    cp_async_wait<1>();
                } else {
                    cp_async_wait<0>();
                }
                __syncthreads();
                // ---- S = Q K^T (16 rows x 64 positions per warp) ----
                float s[8][4];
#pragma unroll
                for (int nt = 0; nt < 8; ++nt)
#pragma unroll
                    for (int e = 0; e < 4; ++e) s[nt][e] = 0.f;
                const uint32_t kb = sK + buf * TILEB, vb = sV + buf * TILEB;
#pragma unroll
                for (int ks = 0; ks < KS; ++ks) {
#pragma unroll
                    for (int n2 = 0; n2 < 4; ++n2) {
                        const int n = n2 * 16 + (lane & 7) + ((lane >> 4) << 3);
                        uint32_t b[4];
                        ldsm_x4(b, kb + n * ROWB + (((ks * 2 + ((lane >> 3) & 1)) ^ (n & 7)) << 4));
                        mma_bf16(s[2 * n2], qf[ks], b[0], b[1]);
                        mma_bf16(s[2 * n2 + 1], qf[ks], b[2], b[3]);
                    }
                }
                // ---- mask, online softmax (exp2 domain) ----
                float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
                for (int nt = 0; nt < 8; ++nt)
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int kpos = kt + nt * 8 + 2 * (lane & 3) + (e & 1);
                        const bool ok = e < 2 ? (v0 && kpos <= pq0 && kpos >= lo0) : (v1 && kpos <= pq1 && kpos >= lo1);
                        s[nt][e] = ok ? s[nt][e] * scale_log2e : -INFINITY;
                        mx[e >> 1] = fmaxf(mx[e >> 1], s[nt][e]);
                    }
                float alpha[2], mnew[2];
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    mx[h] = fmaxf(mx[h], __shfl_xor_sync(0xffffffffu, mx[h], 1));
                    mx[h] = fmaxf(mx[h], __shfl_xor_sync(0xffffffffu, mx[h], 2));
                    mnew[h] = fmaxf(m[h], mx[h]);
                    alpha[h] = mnew[h] == -INFINITY ? 1.f : exp2f(m[h] - mnew[h]);  // nothing seen yet: state unchanged
                    m[h] = mnew[h];
                }
                float rs[2] = {0.f, 0.f};
                // probabilities as TWO bf16 terms (p = hi + lo, 16 bits of mantissa): the tensor core takes bf16
                // operands, and a single rounding of p would cost the fp32-softmax path (llama.py:916-934 runs SDPA
                // with fp32 probabilities on bf16 values) 8 of its bits
                uint32_t pa[4][4], pl[4][4];
#pragma unroll
                for (int nt = 0; nt < 8; ++nt) {
                    float pv[4], lo_[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        pv[e] = mnew[e >> 1] == -INFINITY ? 0.f : exp2f(s[nt][e] - mnew[e >> 1]);
                        rs[e >> 1] += pv[e];
                        lo_[e] = pv[e] - rbf(pv[e]);
                    }
                    pa[nt >> 1][(nt & 1) * 2 + 0] = pack_bf2(pv[0], pv[1]);
                    pa[nt >> 1][(nt & 1) * 2 + 1] = pack_bf2(pv[2], pv[3]);
                    pl[nt >> 1][(nt & 1) * 2 + 0] = pack_bf2(lo_[0], lo_[1]);
                    pl[nt >> 1][(nt & 1) * 2 + 1] = pack_bf2(lo_[2], lo_[3]);
                }
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    rs[h] += __shfl_xor_sync(0xffffffffu, rs[h], 1);
                    rs[h] += __shfl_xor_sync(0xffffffffu, rs[h], 2);
                    l[h] = l[h] * alpha[h] + rs[h];
                }
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    o[nt][0] *= alpha[0]; o[nt][1] *= alpha[0];
                    o[nt][2] *= alpha[1]; o[nt][3] *= alpha[1];
                }
                // ---- O += P V ----
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
#pragma unroll
                    for (int n2 = 0; n2 < NT / 2; ++n2) {
                        const int kr = kk * 16 + (lane & 7) + (((lane >> 3) & 1) << 3);
                        uint32_t b[4];
                        ldsm_x4_t(b, vb + kr * ROWB + (((n2 * 2 + (lane >> 4)) ^ (kr & 7)) << 4));
                        mma_bf16(o[2 * n2], pa[kk], b[0], b[1]);
                        mma_bf16(o[2 * n2 + 1], pa[kk], b[2], b[3]);
                        mma_bf16(o[2 * n2], pl[kk], b[0], b[1]);
                        mma_bf16(o[2 * n2 + 1], pl[kk], b[2], b[3]);
                    }
                }
                __syncthreads();  // this buffer may be refilled
                buf ^= 1;
            }
        }
        start = end;
    }
    // ---- O / l -> bf16; rows without a position (idle slots) read as zero ----
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int qi = h == 0 ? qi0 : qi1;
        const int r = r0 + qi;
        if (r >= a.rows) continue;
        const float inv = l[h] > 0.f ? 1.f / l[h] : 0.f;
        __nv_bfloat16* dst = a.out + (static_cast<size_t>(r) * a.H + head) * DH + 2 * (lane & 3);
#pragma unroll
        for (int nt = 0; nt < NT; ++nt)
            *reinterpret_cast<uint32_t*>(dst + nt * 8) = pack_bf2(o[nt][2 * h] * inv, o[nt][2 * h + 1] * inv);
    }
}

template <int DH>
int launch_t(const AttnArgs& a, cudaStream_t st) {
    static bool attr = false;
    const size_t smem = static_cast<size_t>(kTQ + 4 * kTK) * DH * 2;
    if (!attr) {
        FSB_CUDA(cudaFuncSetAttribute(attn_tile_kernel<DH>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
        attr = true;
    }
    const float scale_log2e = 1.4426950408889634f / sqrtf(static_cast<float>(DH));
    FSB_LAUNCH((attn_tile_kernel<DH>), dim3(cdiv(a.rows, kTQ), a.H), dim3(kAtThreads), smem, st, a, scale_log2e);
    return 0;
}

}  // namespace

int launch_attn(const AttnArgs& a, cudaStream_t st) {
    if (a.rows <= 0) return 0;
    FSB_CHECK((a.Dh == 64 || a.Dh == 128) && a.Hkv > 0 && a.H % a.Hkv == 0,
              "attention: unsupported geometry (head_dim %d, %d heads, %d KV heads)", a.Dh, a.H, a.Hkv);
    return a.Dh == 64 ? launch_t<64>(a, st) : launch_t<128>(a, st);
}

}  // namespace fsb
