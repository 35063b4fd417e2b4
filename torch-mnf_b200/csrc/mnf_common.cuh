// mnf_common.cuh -- building blocks of the MNF layer kernels:
//   * Philox4x32-10 counter RNG + Box-Muller (noise generated in-kernel when the caller does
//     not inject it; the counter is the GLOBAL element index so results do not depend on how
//     rows are sharded over GPUs)
//   * a bounds-checked fp32 SIMT tiled GEMM skeleton  C[M,N] = A'[M,K] * B'[N,K]^T  whose
//     operand loads and epilogue are functors, so the MNF prologues (mask*z, x*z, x^2,
//     exp(W_log_var)) and epilogues (sigmoid gate, mean + sqrt(var)*eps) fuse into it.
//     This is the exact-fp32 path for arbitrary shapes; large aligned shapes take the
//     tcgen05 path (mnf_tc_gemm.cu).
#pragma once
#include "common.cuh"

namespace mnf {

// ---------------------------------------------------------------------------------------
// Philox4x32-10
// ---------------------------------------------------------------------------------------
struct Philox {
    uint32_t key0, key1;
    __device__ __forceinline__ Philox(uint64_t seed) : key0((uint32_t)seed), key1((uint32_t)(seed >> 32)) {}
    __device__ __forceinline__ uint4 operator()(uint64_t counter, uint32_t stream) const {
        uint32_t c0 = (uint32_t)counter, c1 = (uint32_t)(counter >> 32), c2 = stream, c3 = 0x9E3779B9u;
        uint32_t k0 = key0, k1 = key1;
#pragma unroll
        for (int r = 0; r < 10; ++r) {
            const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
            const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
            c0 = hi1 ^ c1 ^ k0;
            c1 = lo1;
            c2 = hi0 ^ c3 ^ k1;
            c3 = lo0;
            k0 += 0x9E3779B9u;
            k1 += 0xBB67AE85u;
        }
        return make_uint4(c0, c1, c2, c3);
    }
};

__device__ __forceinline__ float u32_to_unit(uint32_t u) { return ((float)(u >> 8) + 0.5f) * (1.0f / 16777216.0f); }

// two standard normals from two 32-bit words (Box-Muller).  The uniforms are built in the mantissa ([1, 2) bit pattern,
// 23 random bits: no I2F on the XU pipe), the radius uses one LG2 and one approximate SQRT -- the noise kernels are
// bound by this arithmetic, and only the distribution matters (every kernel draws through this one definition).
__device__ __forceinline__ float2 box_muller(uint32_t a, uint32_t b) {
    const float u1 = 2.f - __uint_as_float((a >> 9) | 0x3f800000u);  // (0, 1]
    const float u2 = __uint_as_float((b >> 9) | 0x3f800000u) - 1.f;  // [0, 1)
    float lg, r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(u1));
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(-1.3862943611198906f * lg));  // sqrt(-2 ln u1)
    float s, c;
    __sincosf(6.283185307179586f * u2, &s, &c);
    return make_float2(r * c, r * s);
}

// division of a non-negative 32-bit index by a run-time constant without the integer-divide sequence
// (n < 2^31; multiplier / shift found on the host): the noise / pool passes decode four indices per element
struct FastDiv {
    uint32_t d, m, s;
    __host__ FastDiv() : d(1), m(0), s(0) {}
    __host__ explicit FastDiv(uint32_t div) : d(div), m(0), s(0) {
        if (div > 1) {
            uint32_t l = 0;
            while ((1ull << l) < div) ++l;  // ceil(log2 div)
            const uint32_t p = 31 + l;
            m = (uint32_t)(((1ull << p) + div - 1) / div);
            s = p - 32;
        }
    }
    __device__ __forceinline__ uint32_t div(uint32_t n) const { return d == 1 ? n : __umulhi(n, m) >> s; }
    __device__ __forceinline__ void divmod(uint32_t n, uint32_t &q, uint32_t &r) const {
        q = div(n);
        r = n - q * d;
    }
};

// standard normal for global element index e of noise stream `stream`
__device__ __forceinline__ float philox_normal(const Philox &g, uint64_t e, uint32_t stream) {
    const uint4 r = g(e >> 2, stream);
    const uint32_t lane = (uint32_t)e & 3u;
    const float2 n = (lane & 2u) ? box_muller(r.z, r.w) : box_muller(r.x, r.y);
    return (lane & 1u) ? n.y : n.x;
}
// Bernoulli(0.5) in {0,1} for global element index e
__device__ __forceinline__ float philox_bernoulli(const Philox &g, uint64_t e, uint32_t stream) {
    const uint4 r = g(e >> 7, stream);
    const uint32_t bit = (uint32_t)e & 127u;
    const uint32_t w = bit < 32 ? r.x : bit < 64 ? r.y : bit < 96 ? r.z : r.w;
    return (float)((w >> (bit & 31u)) & 1u);
}

struct NoiseSrc {
    const float *ptr;  // injected tensor or nullptr -> Philox(seed, stream) indexed by global element
    uint64_t seed;
    uint32_t stream;
    uint64_t row_offset;  // global index of local row 0 (sharded runs draw the same numbers)
};

__device__ __forceinline__ float noise_normal(const NoiseSrc &s, long long local_idx, long long global_idx) {
    return s.ptr ? s.ptr[local_idx] : philox_normal(Philox(s.seed), (uint64_t)global_idx, s.stream);
}
__device__ __forceinline__ float noise_bernoulli(const NoiseSrc &s, long long local_idx, long long global_idx) {
    return s.ptr ? s.ptr[local_idx] : philox_bernoulli(Philox(s.seed), (uint64_t)global_idx, s.stream);
}

// ---------------------------------------------------------------------------------------
// SIMT GEMM skeleton.  NACC accumulator sets share one pass over K (NACC = 2: the MNF
// mean / variance pair shares the x tile).  Problem functor interface:
//   int M, N, K;
//   RowCtx row_ctx(int m)                             -- per-row addressing state, computed ONCE per thread and
//                                                        tile row (keeps div/mod out of the K loop)
//   void load_a(const RowCtx&, int m, int k, float (&a)[NACC]) -- value(s) of A' at (m, k), in range
//   void load_b(int n, int k, float (&b)[NACC])      -- value(s) of B' at (n, k), in range
//   void epilogue4(int m_base, int n, const float (&acc)[NACC][4], float (&rowsum)[4])
//        -- one output column n, four consecutive rows m_base..m_base+3 (bounds on m are the
//           functor's job: rows >= M must be skipped); may add a per-row contribution
//   static constexpr bool kRowReduce; void row_out(int m, float sum)  -- row sums over this
//        block's 64 columns (used for the RNVP log-det)
// ---------------------------------------------------------------------------------------
constexpr int GBM = 64, GBN = 64, GBK = 16, GTHREADS = 256;

template <class Prob, int NACC>
__global__ void __launch_bounds__(GTHREADS) simt_gemm_kernel(const Prob p) {
    __shared__ float As[NACC][GBK][GBM + 4];
    __shared__ float Bs[NACC][GBK][GBN + 4];
    const int tid = threadIdx.x;
    const int m0 = blockIdx.x * GBM, n0 = blockIdx.y * GBN;
    const int tx = tid % 16, ty = tid / 16;  // 16 x 16 threads, 4 x 4 outputs each
    float acc[NACC][4][4];
#pragma unroll
    for (int s = 0; s < NACC; ++s)
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[s][i][j] = 0.f;

    // a thread always loads the same 4 tile rows (idx / GBK is independent of k0): row contexts are hoisted
    typename Prob::RowCtx rctx[(GBM * GBK) / GTHREADS];
#pragma unroll
    for (int e = 0; e < (GBM * GBK) / GTHREADS; ++e) {
        const int mm = (tid + e * GTHREADS) / GBK;
        rctx[e] = p.row_ctx(m0 + mm < p.M ? m0 + mm : 0);
    }
    for (int k0 = 0; k0 < p.K; k0 += GBK) {
        // each thread loads 4 elements of the A tile and 4 of the B tile; k fastest for coalescing
#pragma unroll
        for (int e = 0; e < (GBM * GBK) / GTHREADS; ++e) {
            const int idx = tid + e * GTHREADS;
            const int kk = idx % GBK, mm = idx / GBK;
            float a[NACC], b[NACC];
#pragma unroll
            for (int s = 0; s < NACC; ++s) a[s] = b[s] = 0.f;
            if (m0 + mm < p.M && k0 + kk < p.K) p.load_a(rctx[e], m0 + mm, k0 + kk, a);
            if (n0 + mm < p.N && k0 + kk < p.K) p.load_b(n0 + mm, k0 + kk, b);
#pragma unroll
            for (int s = 0; s < NACC; ++s) {
                As[s][kk][mm] = a[s];
                Bs[s][kk][mm] = b[s];
            }
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < GBK; ++kk) {
#pragma unroll
            for (int s = 0; s < NACC; ++s) {
                const float4 av = *reinterpret_cast<const float4 *>(&As[s][kk][ty * 4]);
                const float4 bv = *reinterpret_cast<const float4 *>(&Bs[s][kk][tx * 4]);
                const float a4[4] = {av.x, av.y, av.z, av.w}, b4[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[s][i][j] = fmaf(a4[i], b4[j], acc[s][i][j]);
            }
        }
        __syncthreads();
    }
    float rowsum[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int n = n0 + tx * 4 + j;
        if (n >= p.N) continue;
        float r[NACC][4];
#pragma unroll
        for (int s = 0; s < NACC; ++s)
#pragma unroll
            for (int i = 0; i < 4; ++i) r[s][i] = acc[s][i][j];
        p.epilogue4(m0 + ty * 4, n, r, rowsum);
    }
    if constexpr (Prob::kRowReduce) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            float v = rowsum[i];
#pragma unroll
            for (int o = 8; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);  // 16 lanes share a row group
            if (tx == 0 && m0 + ty * 4 + i < p.M) p.row_out(m0 + ty * 4 + i, v);
        }
    }
}

// M <= 4 rows (kl_div runs its RNVP stacks with ONE row): a 64-row tile would leave one CTA walking all of K.
// Instead one CTA per output column reduces over K with all its threads (coalesced reads of the weight row).
template <class Prob, int NACC>
__global__ void __launch_bounds__(128) simt_gemv_kernel(const Prob p) {
    __shared__ float red[NACC][4][4];
    const int n = blockIdx.x, tid = threadIdx.x;
    float acc[NACC][4];
#pragma unroll
    for (int s = 0; s < NACC; ++s)
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[s][i] = 0.f;
    typename Prob::RowCtx rctx[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) rctx[i] = p.row_ctx(i < p.M ? i : 0);
    for (int k = tid; k < p.K; k += 128) {
        float b[NACC];
        p.load_b(n, k, b);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (i < p.M) {
                float a[NACC];
                p.load_a(rctx[i], i, k, a);
#pragma unroll
                for (int s = 0; s < NACC; ++s) acc[s][i] = fmaf(a[s], b[s], acc[s][i]);
            }
        }
    }
#pragma unroll
    for (int s = 0; s < NACC; ++s)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float v = warp_sum(acc[s][i]);
            if ((tid & 31) == 0) red[s][i][tid >> 5] = v;
        }
    __syncthreads();
    if (tid == 0) {
        float r[NACC][4], rowsum[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int s = 0; s < NACC; ++s)
#pragma unroll
            for (int i = 0; i < 4; ++i) r[s][i] = (red[s][i][0] + red[s][i][1]) + (red[s][i][2] + red[s][i][3]);
        p.epilogue4(0, n, r, rowsum);
        if constexpr (Prob::kRowReduce) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
                if (i < p.M) p.row_out(i, rowsum[i]);
        }
    }
}

// batches > 1: that many independent problems of the same shape on grid dimension z; the functor tells them apart by
// blockIdx.z (the groups of a grouped convolution).  gemv_ok = false keeps the tiled form for every M, so that a row's
// sum runs in the same order whatever the number of rows in the call.
template <class Prob, int NACC>
int launch_simt_gemm(const Prob &p, cudaStream_t stream, const char *what, int batches = 1, bool gemv_ok = true) {
    if (p.M <= 0 || p.N <= 0) return 0;
    if (gemv_ok && p.M <= 4 && p.K >= 256) {
        simt_gemv_kernel<Prob, NACC><<<dim3((unsigned)p.N, 1, (unsigned)batches), 128, 0, stream>>>(p);
        return launch_status(what);
    }
    dim3 grid((unsigned)((p.M + GBM - 1) / GBM), (unsigned)((p.N + GBN - 1) / GBN), (unsigned)batches);
    if (grid.y > 65535) return fail(MNF_E_SHAPE, "%s: too many column tiles (%u)", what, grid.y);
    simt_gemm_kernel<Prob, NACC><<<grid, GTHREADS, 0, stream>>>(p);
    return launch_status(what);
}

}  // namespace mnf
