// tc_gemm.cu -- Blackwell tensor-core path of the MNF contractions:
//     C[M,N] = A[M,K] * B[N,K]^T  (fp32 in HBM, TF32 on the 5th-gen tensor cores, fp32 accumulate in TMEM)
// with the MNF epilogues fused (bias, sqrt-variance * noise, ReLU).
//
// Structure (one persistent CTA per SM, 256 threads, warp-specialised):
//   warp 0   TMA producer: cp.async.bulk.tensor 2-D tiles of A (128 x 32 fp32) and B (256 x 32 fp32) into a
//            4-stage shared-memory ring, 128-byte swizzle, completion on mbarriers
//   warp 1   MMA issuer: one elected thread issues tcgen05.mma.cta_group::1.kind::tf32 (M128 x N256 x K8),
//            4 per stage, accumulating into one of two 256-column TMEM accumulators; tcgen05.commit
//            releases the smem stage / publishes the accumulator
//   warp 2   TMEM allocator (512 columns)
//   warps 4-7 epilogue: tcgen05.ld 32x32b.x32 -> registers -> fused epilogue -> global; overlaps the next
//            tile's MMAs through the second accumulator
// TF32 keeps a 10-bit mantissa: products carry ~2e-4 relative error, inside the 2e-3 tolerance BASELINE.json
// states for tensor-core GEMM outputs (the exact-fp32 path is simt_gemm_kernel in mnf_common.cuh).
#include "rnvp_fused.cuh"
#include "tc_common.cuh"

namespace mnf {
// fp16 weights of the implicit-GEMM conv (mnf_layers.cu): Bm = fp16(W_mean * z), Bv = fp16(exp(W_log_var) * 2^8), [Np, Kp]
int conv_pack_weights_f16(const float *z, const float *W_mean, const float *W_log_var, const float *b_log_var, void *Bm,
                          void *Bv, float *bvar_p, int K, int c_out, int Np, int Kp, void *stream);
}  // namespace mnf

namespace mnf {
namespace tc {

constexpr uint32_t A_BYTES = BM * BK * 4;
constexpr int THREADS = 384;  // 4 control warps + 2 groups of 4 epilogue warps
// tile width BN in {32, 64, 128, 256}: narrow outputs (RNVP / MADE hidden layers) take narrow tiles so that
// neither the B-tile TMA nor the MMA is spent on padding; narrow tiles afford a deeper smem ring
template <int BN>
struct Cfg {
    static constexpr int STAGES = BN == 256 ? 4 : (BN == 128 ? 6 : 8);  // <= 192 KB of operand ring
    static constexpr uint32_t B_BYTES = BN * BK * 4, STAGE_BYTES = A_BYTES + B_BYTES;
    // TMEM accumulators in flight: narrow tiles finish their MMAs in a few hundred cycles, so more of them are
    // kept in flight to cover the epilogue's memory latency
    static constexpr int ACC_STAGES = BN == 256 ? 2 : (BN == 128 ? 4 : 8);
    static constexpr uint32_t TMEM_COLS = ACC_STAGES * BN;  // power of two in [64, 512]
    static constexpr uint32_t SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align*/ + 512 /*barriers*/;
    // cute::UMMA::InstrDescriptor: c=F32, a=b=TF32, K-major both, N>>3 at bit 17, M>>4 at bit 24
    static constexpr uint32_t kInstrDesc =
        (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
};

struct Epilogue {
    int mode;           // 0: acc + bias   1: acc + bias + sd[m % sd_rows, n] * eps   2: sqrt(acc + exp(bvar_log[n]))
    const float *bias;  // [N] or nullptr
    const float *sd;    // mode 1: [sd_rows, N]
    int sd_rows;
    const float *bvar_log;  // mode 2: [N]
    const float *eps;       // mode 1: [M, N] or nullptr -> Philox
    uint64_t seed;
    uint32_t noise_stream;
    uint64_t row_offset;
    int relu;
    // mode 1: optional per-column affine map after the noise and ReLU, v = col_scale[n] * v + col_shift[n] (an eval-mode
    // BatchNorm1d folded to its inference coefficients); NULL = none.  16-byte aligned.
    const float *col_scale, *col_shift;
    float *out;  // [M, N]  (mode 3: [M, N/2])
    // mode 0 extras
    int round_out;  // store rn_tf32(value): the output feeds another TF32 GEMM
    // mode 3 (MAF.inverse epilogue, maf.py:53-62): columns are interleaved (s_0, t_0, s_1, t_1, ...);
    // z = x * exp(s) + t, dims flipped if parity, log_det (+)= sum s.  Needs N <= BN (one column tile).
    const float *xin;    // [M, N/2] exact fp32 input of the flow
    float *out_rounded;  // optional second copy of z, TF32-rounded, for the next flow's first GEMM
    const float *ld_in;  // optional running log-det
    float *ld_out;
    int parity;
    // mode 5 (MNFConv2d tail on an im2col GEMM whose rows are pool-major): v = acc + sd[m, n] * eps, ReLU, max over
    // the 4 consecutive rows of a 2x2 window (4 adjacent TMEM lanes -> two shuffles), out[r, n, py, px].
    // sd: [M, N] (row stride N); eps indexed like the un-pooled [R, conv_c, conv_oh, conv_ow] tensor.
    int conv_c, conv_oh, conv_ow;
};

template <int BN>
__global__ void __launch_bounds__(THREADS, 1)
tf32_gemm_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, int M, int N,
                 int K, const Epilogue ep) {
    constexpr int STAGES = Cfg<BN>::STAGES, ACC_STAGES = Cfg<BN>::ACC_STAGES;
    constexpr uint32_t STAGE_BYTES = Cfg<BN>::STAGE_BYTES, TMEM_COLS = Cfg<BN>::TMEM_COLS;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;  // SWIZZLE_128B tiles need 1024-byte alignment
    const uint32_t bars = base + STAGES * STAGE_BYTES;
    // barrier slots: full[STAGES], empty[STAGES], acc_full[ACC], acc_empty[ACC], then the TMEM base address
    auto full = [&](int s) { return bars + 8u * s; };
    auto empty = [&](int s) { return bars + 8u * (STAGES + s); };
    auto acc_full = [&](int a) { return bars + 8u * (2 * STAGES + a); };
    auto acc_empty = [&](int a) { return bars + 8u * (2 * STAGES + ACC_STAGES + a); };
    const uint32_t tmem_slot = bars + 8u * (2 * STAGES + 2 * ACC_STAGES);
    uint32_t *tmem_slot_ptr = reinterpret_cast<uint32_t *>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(full(s), 1);
            mbar_init(empty(s), 1);
        }
        for (int a = 0; a < ACC_STAGES; ++a) {
            mbar_init(acc_full(a), 1);
            mbar_init(acc_empty(a), 256);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(TMEM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot_ptr;

    const int n_mblk = (M + BM - 1) / BM, n_nblk = (N + BN - 1) / BN, n_kblk = (K + BK - 1) / BK;
    const long long n_tiles = (long long)n_mblk * n_nblk;

    if (warp == 0 && lane == 0) {
        // ---------------- TMA producer ----------------
        int stage = 0;
        uint32_t phase = 0;
        for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            const int m_blk = (int)(tile / n_nblk), n_blk = (int)(tile % n_nblk);
            for (int kb = 0; kb < n_kblk; ++kb) {
                mbar_wait(empty(stage), phase ^ 1u);
                mbar_expect_tx(full(stage), STAGE_BYTES);
                const uint32_t sa = base + stage * STAGE_BYTES;
                tma_load_2d(sa, &map_a, full(stage), kb * BK, m_blk * BM);
                tma_load_2d(sa + A_BYTES, &map_b, full(stage), kb * BK, n_blk * BN);
                if (++stage == STAGES) {
                    stage = 0;
                    phase ^= 1u;
                }
            }
        }
    } else if (warp == 1 && lane == 0) {
        // ---------------- MMA issuer ----------------
        int stage = 0, acc = 0;
        uint32_t phase = 0, acc_phase = 0;
        for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            mbar_wait(acc_empty(acc), acc_phase ^ 1u);  // epilogue has drained this accumulator
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BN);
            for (int kb = 0; kb < n_kblk; ++kb) {
                mbar_wait(full(stage), phase);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t sa = base + stage * STAGE_BYTES;
                const uint64_t adesc = make_smem_desc(sa), bdesc = make_smem_desc(sa + A_BYTES);
#pragma unroll
                for (int k = 0; k < BK / UMMA_K; ++k) {
                    // advance 32 bytes (8 tf32) along K inside the 128-byte swizzle atom: +2 in the >>4 address field
                    umma_tf32(tmem_d, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), (kb | k) != 0, Cfg<BN>::kInstrDesc);
                }
                umma_commit(empty(stage));  // frees the smem stage once these MMAs have read it
                if (++stage == STAGES) {
                    stage = 0;
                    phase ^= 1u;
                }
            }
            umma_commit(acc_full(acc));  // accumulator complete -> epilogue
            if (++acc == ACC_STAGES) {
                acc = 0;
                acc_phase ^= 1u;
            }
        }
    } else if (warp >= 4) {
        // ---------------- epilogue (128 threads, one TMEM lane = one output row each) ----------------
        const int quarter = warp & 3;  // a warp may only touch TMEM lanes [32*(warp%4), +32)
        const int group = (warp - 4) >> 2;  // two warps per lane quarter share a tile: even / odd 32-column chunks
        int acc = 0;
        uint32_t acc_phase = 0;
        const Philox rng(ep.seed);
        for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            const int m_blk = (int)(tile / n_nblk), n_blk = (int)(tile % n_nblk);
            mbar_wait(acc_full(acc), acc_phase);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const int m = m_blk * BM + quarter * 32 + lane;
            const uint32_t trow = tmem_base + (uint32_t)(acc * BN) + ((uint32_t)(quarter * 32) << 16);
            float s_sum = 0.f;
#pragma unroll 1
            for (int c = group; c < BN / 32 && n_blk * BN + c * 32 < N; c += 2) {
                uint32_t r[32];
                tmem_ld32(trow + (uint32_t)(c * 32), r);
                const int n0 = n_blk * BN + c * 32;
                if (ep.mode == 3) {
                    if (m < M) {
                        // 32 accumulator columns = 16 (s, t) pairs = 16 consecutive dims: 64 contiguous bytes of
                        // x / z per thread, moved as float4 (reversed within the row when parity flips the dims)
                        const int D = N >> 1, i0 = n0 >> 1;
                        const float *xrow = ep.xin + (size_t)m * D;
                        float zv[16];
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const int i = i0 + 4 * q;
                            if (i < D) {
                                const float4 xv = *reinterpret_cast<const float4 *>(xrow + i);
                                const float4 b0 = *reinterpret_cast<const float4 *>(ep.bias + 2 * i);
                                const float4 b1 = *reinterpret_cast<const float4 *>(ep.bias + 2 * i + 4);
                                const float xs[4] = {xv.x, xv.y, xv.z, xv.w};
                                const float bs[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                                for (int u = 0; u < 4; ++u) {
                                    const float sv = __uint_as_float(r[8 * q + 2 * u]) + bs[2 * u];
                                    const float tv = __uint_as_float(r[8 * q + 2 * u + 1]) + bs[2 * u + 1];
                                    zv[4 * q + u] = xs[u] * expf(sv) + tv;  // maf.py:58
                                    s_sum += sv;
                                }
                            }
                        }
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const int i = i0 + 4 * q;
                            if (i < D) {
                                float4 v = make_float4(zv[4 * q], zv[4 * q + 1], zv[4 * q + 2], zv[4 * q + 3]);
                                size_t o = (size_t)m * D + i;
                                if (ep.parity) {  // maf.py:60: z.flip(dims=[1])
                                    v = make_float4(v.w, v.z, v.y, v.x);
                                    o = (size_t)m * D + (D - 4 - i);
                                }
                                *reinterpret_cast<float4 *>(ep.out + o) = v;
                                if (ep.out_rounded)
                                    *reinterpret_cast<float4 *>(ep.out_rounded + o) =
                                        make_float4(rn_tf32(v.x), rn_tf32(v.y), rn_tf32(v.z), rn_tf32(v.w));
                            }
                        }
                    }
                } else if (ep.mode == 5) {
                    // rows of a warp are 32 consecutive pool-major rows = 8 windows; all lanes take part in the shuffles
                    const int OH = ep.conv_oh, OW = ep.conv_ow, PW = OW >> 1, PH = OH >> 1, Cc = ep.conv_c;
                    const int mm = m < M ? m : M - 1;
                    const int q = mm & 3, w = mm >> 2;
                    const int px = w % PW, py = (w / PW) % PH;
                    const long long rr = w / (PW * PH);
                    const int oy = 2 * py + (q >> 1), ox = 2 * px + (q & 1);
                    const float *sdrow = ep.sd + (size_t)mm * N + n0;
                    float sdv[32];
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        const float4 b = *reinterpret_cast<const float4 *>(sdrow + j);
                        sdv[j] = b.x, sdv[j + 1] = b.y, sdv[j + 2] = b.z, sdv[j + 3] = b.w;
                    }
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const int n = n0 + j;
                        float v = 0.f;
                        if (n < Cc) {
                            const long long le = ((rr * Cc + n) * OH + oy) * OW + ox;
                            const float nz = ep.eps ? ep.eps[le]
                                                    : philox_normal(rng, (uint64_t)(le + (long long)ep.row_offset * Cc * OH * OW),
                                                                    ep.noise_stream);
                            v = fmaxf(fmaf(sdv[j], nz, __uint_as_float(r[j])), 0.f);
                        }
                        v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
                        v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
                        if (q == 0 && m < M && n < Cc) ep.out[((rr * Cc + n) * PH + py) * PW + px] = v;
                    }
                } else if (m < M && n0 + 32 <= N && (N & 3) == 0) {
                    // fast path: whole 32-column chunk in range.  All global operands of the chunk are fetched
                    // with independent float4 loads BEFORE any arithmetic, so the epilogue pays one memory
                    // latency per chunk instead of one per element (it must stay shorter than a tile's MMAs).
                    float *orow = ep.out + (size_t)m * N + n0;
                    float add[32], mul[32], nz[32];
                    const bool has_bias = ep.mode != 2 && ep.bias != nullptr;
                    const float *bsrc = ep.mode == 2 ? ep.bvar_log : ep.bias;
                    if (ep.mode == 2 || has_bias) {
#pragma unroll
                        for (int j = 0; j < 32; j += 4) {
                            const float4 b = *reinterpret_cast<const float4 *>(bsrc + n0 + j);
                            add[j] = b.x, add[j + 1] = b.y, add[j + 2] = b.z, add[j + 3] = b.w;
                        }
                    }
                    if (ep.mode == 1) {
                        const float *sdrow = ep.sd + (size_t)(m % ep.sd_rows) * N + n0;
#pragma unroll
                        for (int j = 0; j < 32; j += 4) {
                            const float4 b = *reinterpret_cast<const float4 *>(sdrow + j);
                            mul[j] = b.x, mul[j + 1] = b.y, mul[j + 2] = b.z, mul[j + 3] = b.w;
                        }
                        const long long e0 = (long long)m * N + n0;
                        if (ep.eps) {
#pragma unroll
                            for (int j = 0; j < 32; j += 4) {
                                const float4 b = *reinterpret_cast<const float4 *>(ep.eps + e0 + j);
                                nz[j] = b.x, nz[j + 1] = b.y, nz[j + 2] = b.z, nz[j + 3] = b.w;
                            }
                        } else {
                            // global element index is a multiple of 4 here: one Philox block = 4 normals
                            const uint64_t g0 = (uint64_t)(ep.row_offset * N + e0);
#pragma unroll
                            for (int j = 0; j < 32; j += 4) {
                                const uint4 q = rng((g0 + j) >> 2, ep.noise_stream);
                                const float2 n01 = box_muller(q.x, q.y), n23 = box_muller(q.z, q.w);
                                nz[j] = n01.x, nz[j + 1] = n01.y, nz[j + 2] = n23.x, nz[j + 3] = n23.y;
                            }
                        }
                    }
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        float v[4];
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            float a = __uint_as_float(r[j + u]);
                            if (ep.mode == 2) {
                                a = sqrtf(a + expf(add[j + u]));
                            } else {
                                if (has_bias) a += add[j + u];
                                if (ep.mode == 1) a = fmaf(mul[j + u], nz[j + u], a);
                                if (ep.relu) a = fmaxf(a, 0.f);
                                if (ep.round_out) a = rn_tf32(a);
                            }
                            v[u] = a;
                        }
                        // per-column affine, 4 columns at a time: the 32-wide staging arrays above are at the register
                        // limit, so the two pointers are re-read from the parameter bank here (volatile) instead of being
                        // held in registers across the chunk -- holding them added spill stores to the BN = 32 kernel
                        const float *cs = *reinterpret_cast<const float *const volatile *>(&ep.col_scale);
                        if (cs) {
                            const float *ch = *reinterpret_cast<const float *const volatile *>(&ep.col_shift);
                            const float4 sc = __ldg(reinterpret_cast<const float4 *>(cs + n0 + j));
                            const float4 sh = __ldg(reinterpret_cast<const float4 *>(ch + n0 + j));
                            v[0] = fmaf(sc.x, v[0], sh.x), v[1] = fmaf(sc.y, v[1], sh.y);
                            v[2] = fmaf(sc.z, v[2], sh.z), v[3] = fmaf(sc.w, v[3], sh.w);
                        }
                        *reinterpret_cast<float4 *>(orow + j) = make_float4(v[0], v[1], v[2], v[3]);
                    }
                } else if (m < M && n0 < N) {
                    // ragged edge: element-wise with bounds checks
                    float *orow = ep.out + (size_t)m * N;
                    const float *sdrow = ep.mode == 1 ? ep.sd + (size_t)(m % ep.sd_rows) * N : nullptr;
                    for (int j = 0; j < 32; ++j) {
                        const int n = n0 + j;
                        if (n >= N) break;
                        float a = __uint_as_float(r[j]);
                        if (ep.mode == 2) {
                            a = sqrtf(a + expf(ep.bvar_log[n]));
                        } else {
                            if (ep.bias) a += ep.bias[n];
                            if (ep.mode == 1) {
                                const long long e = (long long)m * N + n;
                                const float z = ep.eps ? ep.eps[e]
                                                       : philox_normal(rng, (uint64_t)(ep.row_offset * N + e),
                                                                       ep.noise_stream);
                                a = fmaf(sdrow[n], z, a);
                            }
                            if (ep.relu) a = fmaxf(a, 0.f);
                            if (ep.col_scale) a = fmaf(ep.col_scale[n], a, ep.col_shift[n]);
                            if (ep.round_out) a = rn_tf32(a);
                        }
                        orow[n] = a;
                    }
                }
            }
            if (ep.mode == 3 && m < M) atomicAdd(&ep.ld_out[m], s_sum);  // maf.py:61 (ld_out pre-initialised by the host)
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            mbar_arrive(acc_empty(acc));
            if (++acc == ACC_STAGES) {
                acc = 0;
                acc_phase ^= 1u;
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 2) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

bool eligible(const float *A, const float *B, int M, int N, int K) {
    return M >= 1 && N >= 8 && K >= BK && (K % 4) == 0 && ((uintptr_t)A % 16) == 0 && ((uintptr_t)B % 16) == 0;
}

template <int BN>
static int launch_bn(const float *A, const float *B, int M, int N, int K, const Epilogue &ep, const DeviceProps *dp,
                     cudaStream_t stream) {
    CUtensorMap ma, mb;
    int rc = make_map(&ma, A, M, K, BM);
    if (rc) return rc;
    rc = make_map(&mb, B, N, K, BN);
    if (rc) return rc;
    static bool attr_set[64] = {false};
    int dev = 0;
    MNF_CUDA(cudaGetDevice(&dev));
    if (!attr_set[dev & 63]) {
        MNF_CUDA(cudaFuncSetAttribute(tf32_gemm_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)Cfg<BN>::SMEM_BYTES));
        attr_set[dev & 63] = true;
    }
    const long long n_tiles = (long long)((M + BM - 1) / BM) * ((N + BN - 1) / BN);
    const unsigned grid = (unsigned)(n_tiles < dp->sm_count ? n_tiles : dp->sm_count);
    tf32_gemm_kernel<BN><<<grid, THREADS, Cfg<BN>::SMEM_BYTES, stream>>>(ma, mb, M, N, K, ep);
    return launch_status("tf32_gemm_kernel");
}

int launch(const float *A, const float *B, int M, int N, int K, const Epilogue &ep, cudaStream_t stream) {
    const DeviceProps *dp = device_props();
    MNF_REQUIRE(dp != nullptr, MNF_E_DEVICE, "no CUDA device");
    MNF_REQUIRE(dp->cc_major == 10, MNF_E_DEVICE, "tcgen05 path needs an sm_100 device, found sm_%d%d", dp->cc_major,
                dp->cc_minor);
    MNF_REQUIRE(eligible(A, B, M, N, K), MNF_E_SHAPE, "shape/alignment not eligible for the tensor-core path");
    if (N <= 32) return launch_bn<32>(A, B, M, N, K, ep, dp, stream);
    if (N <= 64) return launch_bn<64>(A, B, M, N, K, ep, dp, stream);
    if (N <= 128) return launch_bn<128>(A, B, M, N, K, ep, dp, stream);
    return launch_bn<256>(A, B, M, N, K, ep, dp, stream);
}


// =====================================================================================================================
// Implicit-GEMM MNFConv2d (no im2col in HBM): both moments of the local reparameterisation from ONE pass over x.
//   mean[m, n] = sum_k A[m, k] Bm[n, k]          A[m, k]  = fp16(x[img, ci, oy + ky, ox + kx])     (generated in smem)
//   sd[m, n]   = sqrt(sum_k A2[m, k] Bv[n, k] + exp(b_log_var[n]))    A2 = fp16(x^2)
// Operands are fp16 (kind::f16, fp32 accumulation): the 11-bit significand of TF32 -- the 2e-3 tolerance class BASELINE.json
// states for the MNF GEMMs -- at half the bytes.  The kernel is bound by shared memory (operand tiles written by the
// generators and read by the tensor core: r01 ncu, 152 M wavefronts, tensor pipe 20 %); a k-block of 128-byte rows now
// holds 64 taps instead of 32, so the generators' stores, the MMAs' reads and the MMA count per tile all halve.
// exp(W_log_var) (~1e-4 at the prior's -9) is packed times 2^8 to stay in fp16's normal range; the epilogue undoes it.
// rows m are pool-major (4 * window + 2 * (oy & 1) + (ox & 1)), k = (ci * ks + ky) * ks + kx padded to Kp.
// A tile is 128 rows = IMGS whole images (128 % (OH * OW) == 0).  Roles (512 threads): warp 0 = TMA producer of the
// two weight tiles, warp 1 = single-thread tcgen05.mma issuer (two MMAs per k-step into two 64-column TMEM
// accumulators), warp 2 = TMEM allocator, warps 4-11 = A generators (two threads per tile row: they gather the row's
// taps from the images staged in shared memory by cp.async one tile ahead -- tap offsets come from a kernel-parameter
// table through the uniform datapath -- and write the A and A2 tiles in the 128-byte-swizzle K-major layout the UMMA
// descriptor expects, then fence.proxy.async + mbarrier arrive), warps 12-15 = epilogue (tcgen05.ld -> mean, sd rows).  The materialised im2col this replaces wrote and re-read
// 2 x 4 x Kp bytes per output pixel (6.6 GB + 7 GB per 25 600 LeNet samples); this kernel reads x once.
// =====================================================================================================================
constexpr int CONV_STAGES = 3, CONV_ACC = 4, CONV_BN = 64, CONV_MAX_KP = 512, CONV_BK = 64;
// generator threads per tile row (each takes 8 / CONV_PARTS of the k-block's eight 16-byte chunks).  Measured (cfg4, 64 MC
// samples per step): 2 threads per row 11.87 M samples/s, 4 threads per row (16 generator warps) 11.57 M
constexpr int CONV_PARTS = 2, CONV_GEN = 128 * CONV_PARTS, CONV_CPT = 8 / CONV_PARTS, CONV_THREADS = 128 + CONV_GEN + 128;
constexpr float CONV_VAR_SCALE = 256.f;  // must match conv_pack_weights_f16_kernel (mnf_layers.cu)
struct ConvTaps {  // k -> offset of tap (ci, ky, kx) inside an image (0 for the zero padding of K); travels as a
    int off[CONV_MAX_KP];  // kernel parameter so that the generators read it through the uniform datapath
};
constexpr uint32_t CONV_B_BYTES = CONV_BN * CONV_BK * 2, CONV_STAGE_BYTES = 2 * A_BYTES + 2 * CONV_B_BYTES;
static_assert(BM * CONV_BK * 2 == A_BYTES, "an fp16 k-block of 64 taps fills the same 128-byte rows as 32 fp32 values");
// tcgen05 instruction descriptor, kind::f16: D = F32, A = B = F16, both K-major
constexpr uint32_t conv_f16_idesc(int m, int n) { return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24); }
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate, uint32_t idesc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ uint32_t conv_pack_h2(float lo, float hi) {  // `lo` lands at the lower address
    uint32_t r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}

__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}

__global__ void __launch_bounds__(CONV_THREADS, 1)
conv_implicit_kernel(const __grid_constant__ CUtensorMap map_bm, const __grid_constant__ CUtensorMap map_bv,
                     const __grid_constant__ ConvTaps taps, const float *__restrict__ x, const float *__restrict__ bvar_log, float *__restrict__ mean,
                     float *__restrict__ sd, long long n_imgs, int C, int H, int W, int ks, int Kp, int Np) {
    extern __shared__ uint8_t smem_raw[];
    const int OH = H - ks + 1, OW = W - ks + 1, RPI = OH * OW, IMGS = BM / RPI, CHW = C * H * W;
    const int PW = OW >> 1;
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bars = base + CONV_STAGES * CONV_STAGE_BYTES;
    auto full_a = [&](int s) { return bars + 8u * s; };
    auto full_b = [&](int s) { return bars + 8u * (CONV_STAGES + s); };
    auto empty = [&](int s) { return bars + 8u * (2 * CONV_STAGES + s); };
    auto acc_full = [&](int a) { return bars + 8u * (3 * CONV_STAGES + a); };
    auto acc_empty = [&](int a) { return bars + 8u * (3 * CONV_STAGES + CONV_ACC + a); };
    const uint32_t tmem_slot = bars + 8u * (3 * CONV_STAGES + 2 * CONV_ACC);
    uint8_t *gen = smem_raw + (bars + 256u - smem_u32(smem_raw));  // generic pointers past the barrier block
    uint32_t *tmem_slot_ptr = reinterpret_cast<uint32_t *>(smem_raw + (tmem_slot - smem_u32(smem_raw)));
    float *sbv = reinterpret_cast<float *>(gen);  // [CONV_BN] exp(b_log_var)
    float *xs = sbv + CONV_BN;                    // 2 x [IMGS * CHW] staged images (16-byte aligned)
    const uint32_t xs_u32 = smem_u32(xs);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int n = threadIdx.x; n < CONV_BN; n += blockDim.x) sbv[n] = n < Np ? expf(bvar_log[n]) : 0.f;
    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_bm) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_bv) : "memory");
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < CONV_STAGES; ++s) {
            mbar_init(full_a(s), CONV_GEN);
            mbar_init(full_b(s), 1);
            mbar_init(empty(s), 1);
        }
        for (int a = 0; a < CONV_ACC; ++a) {
            mbar_init(acc_full(a), 1);
            mbar_init(acc_empty(a), 128);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot_ptr;

    const long long M = n_imgs * RPI;
    const long long n_tiles = (n_imgs + IMGS - 1) / IMGS;
    const int n_kblk = Kp / CONV_BK;

    if (warp == 0 && lane == 0) {
        // ---------------- TMA producer: the two weight tiles of every k-block ----------------
        int stage = 0;
        uint32_t phase = 0;
        for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            for (int kb = 0; kb < n_kblk; ++kb) {
                mbar_wait(empty(stage), phase ^ 1u);
                mbar_expect_tx(full_b(stage), 2 * CONV_B_BYTES);
                const uint32_t sb = base + stage * CONV_STAGE_BYTES + 2 * A_BYTES;
                tma_load_2d(sb, &map_bm, full_b(stage), kb * CONV_BK, 0);
                tma_load_2d(sb + CONV_B_BYTES, &map_bv, full_b(stage), kb * CONV_BK, 0);
                if (++stage == CONV_STAGES) stage = 0, phase ^= 1u;
            }
        }
    } else if (warp == 1 && lane == 0) {
        // ---------------- MMA issuer ----------------
        int stage = 0, acc = 0;
        uint32_t phase = 0, acc_phase = 0;
        for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            mbar_wait(acc_empty(acc), acc_phase ^ 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t d_mean = tmem_base + (uint32_t)(acc * 2 * CONV_BN), d_var = d_mean + CONV_BN;
            for (int kb = 0; kb < n_kblk; ++kb) {
                mbar_wait(full_a(stage), phase);
                mbar_wait(full_b(stage), phase);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t sa = base + stage * CONV_STAGE_BYTES;
                const uint64_t a1 = make_smem_desc(sa), a2 = make_smem_desc(sa + A_BYTES);
                const uint64_t b1 = make_smem_desc(sa + 2 * A_BYTES), b2 = make_smem_desc(sa + 2 * A_BYTES + CONV_B_BYTES);
#pragma unroll
                for (int k = 0; k < CONV_BK / 16; ++k) {  // 16 fp16 = 32 bytes per MMA inside the 128-byte swizzle atom
                    umma_f16(d_mean, a1 + (uint64_t)(2 * k), b1 + (uint64_t)(2 * k), (kb | k) != 0, conv_f16_idesc(BM, CONV_BN));
                    umma_f16(d_var, a2 + (uint64_t)(2 * k), b2 + (uint64_t)(2 * k), (kb | k) != 0, conv_f16_idesc(BM, CONV_BN));
                }
                umma_commit(empty(stage));
                if (++stage == CONV_STAGES) stage = 0, phase ^= 1u;
            }
            umma_commit(acc_full(acc));
            if (++acc == CONV_ACC) acc = 0, acc_phase ^= 1u;
        }
    } else if (warp >= 4 && warp < 4 + CONV_GEN / 32) {
        // ---------------- A generators: CONV_PARTS threads per tile row (CONV_CPT 16-byte chunks = 8 CONV_CPT taps of the k-block each) ----------------
        const int gt = threadIdx.x - 128, ml = gt & 127, half = gt >> 7;  // half: which part of the row's chunks
        const int img_l = ml / RPI, p = ml % RPI, q = p & 3, w = p >> 2;
        const int row_base = img_l * CHW + (2 * (w / PW) + (q >> 1)) * W + 2 * (w % PW) + (q & 1);
        const uint32_t row_smem = (uint32_t)((ml >> 3) * 1024 + (ml & 7) * 128);
        const int swz = ml & 7;
        const int n16_full = IMGS * CHW / 4;
        auto prefetch = [&](long long tile, int buf) {
            const long long img0 = tile * IMGS;
            long long left = (n_imgs - img0) * (long long)(CHW / 4);
            const int n16 = (int)(left < n16_full ? left : n16_full);
            const float *src = x + (size_t)img0 * CHW;
            const uint32_t dst = xs_u32 + (uint32_t)buf * (uint32_t)(IMGS * CHW * 4);
            for (int i = gt; i < n16; i += CONV_GEN) cp_async16(dst + 16u * i, src + 4 * i);
            asm volatile("cp.async.commit_group;" ::: "memory");
        };
        int stage = 0, buf = 0;
        uint32_t phase = 0;
        if ((long long)blockIdx.x < n_tiles) prefetch(blockIdx.x, 0);
        for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            const long long next = tile + gridDim.x;
            if (next < n_tiles) prefetch(next, buf ^ 1);  // the other buffer was released by the barrier below
            else asm volatile("cp.async.commit_group;" ::: "memory");
            asm volatile("cp.async.wait_group 1;" ::: "memory");
            asm volatile("bar.sync 1, %0;" ::"n"(CONV_GEN) : "memory");  // every generator's copies of this tile have landed
            const float *xt = xs + (size_t)buf * IMGS * CHW;
            // software pipeline: the 32 taps of the NEXT k-block are gathered into registers right after this one is
            // published, so their shared-memory latency overlaps the wait for the stage to come back from the MMAs
            float v[8 * CONV_CPT];
            // no validity checks: the zero padding of K is done by the WEIGHT tiles (their columns >= K are zero and the
            // padded taps point at offset 0, a finite value), and rows past the last image of a half-filled tile read
            // whatever the buffer holds -- their outputs are never stored and rows do not mix in an MMA
            const float *xrow = xt + row_base;
            auto gather = [&](int kb) {
#pragma unroll
                for (int cc = 0; cc < CONV_CPT; ++cc) {
                    const int kk = kb * CONV_BK + 8 * (half * CONV_CPT + cc);
#pragma unroll
                    for (int u = 0; u < 8; ++u) v[8 * cc + u] = xrow[taps.off[kk + u]];
                }
            };
            gather(0);
            for (int kb = 0; kb < n_kblk; ++kb) {
                mbar_wait(empty(stage), phase ^ 1u);
                uint8_t *sa = smem_raw + (base + stage * CONV_STAGE_BYTES - smem_u32(smem_raw)) + row_smem;
#pragma unroll
                for (int cc = 0; cc < CONV_CPT; ++cc) {
                    const int pos = ((half * CONV_CPT + cc) ^ swz) * 16;
                    const float *q = v + 8 * cc;
                    *reinterpret_cast<uint4 *>(sa + pos) =
                        make_uint4(conv_pack_h2(q[0], q[1]), conv_pack_h2(q[2], q[3]), conv_pack_h2(q[4], q[5]), conv_pack_h2(q[6], q[7]));
                    *reinterpret_cast<uint4 *>(sa + A_BYTES + pos) =
                        make_uint4(conv_pack_h2(q[0] * q[0], q[1] * q[1]), conv_pack_h2(q[2] * q[2], q[3] * q[3]),
                                   conv_pack_h2(q[4] * q[4], q[5] * q[5]), conv_pack_h2(q[6] * q[6], q[7] * q[7]));
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> tensor-core reads
                mbar_arrive(full_a(stage));
                if (kb + 1 < n_kblk) gather(kb + 1);
                if (++stage == CONV_STAGES) stage = 0, phase ^= 1u;
            }
            asm volatile("bar.sync 1, %0;" ::"n"(CONV_GEN) : "memory");  // all rows of this tile generated: its image buffer is free
            buf ^= 1;
        }
        asm volatile("cp.async.wait_group 0;" ::: "memory");
    } else if (warp >= 4 + CONV_GEN / 32) {
        // ---------------- epilogue: TMEM -> mean, sd rows ----------------
        const int quarter = warp & 3;
        int acc = 0;
        uint32_t acc_phase = 0;
        for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            mbar_wait(acc_full(acc), acc_phase);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const long long m = tile * BM + quarter * 32 + lane;
            const uint32_t trow = tmem_base + (uint32_t)(acc * 2 * CONV_BN) + ((uint32_t)(quarter * 32) << 16);
#pragma unroll 1
            for (int c = 0; c < CONV_BN / 32 && c * 32 < Np; ++c) {
                uint32_t rm[32], rv[32];
                tmem_ld32(trow + (uint32_t)(c * 32), rm);
                tmem_ld32(trow + (uint32_t)(CONV_BN + c * 32), rv);
                if (m < M) {
                    float *mrow = mean + (size_t)m * Np + c * 32, *srow = sd + (size_t)m * Np + c * 32;
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        *reinterpret_cast<float4 *>(mrow + j) = make_float4(__uint_as_float(rm[j]), __uint_as_float(rm[j + 1]),
                                                                            __uint_as_float(rm[j + 2]), __uint_as_float(rm[j + 3]));
                        const float4 bv = *reinterpret_cast<const float4 *>(sbv + c * 32 + j);
                        *reinterpret_cast<float4 *>(srow + j) =
                            make_float4(sqrtf(fmaf(__uint_as_float(rv[j]), 1.f / CONV_VAR_SCALE, bv.x)),
                                        sqrtf(fmaf(__uint_as_float(rv[j + 1]), 1.f / CONV_VAR_SCALE, bv.y)),
                                        sqrtf(fmaf(__uint_as_float(rv[j + 2]), 1.f / CONV_VAR_SCALE, bv.z)),
                                        sqrtf(fmaf(__uint_as_float(rv[j + 3]), 1.f / CONV_VAR_SCALE, bv.w)));
                    }
                }
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            mbar_arrive(acc_empty(acc));
            if (++acc == CONV_ACC) acc = 0, acc_phase ^= 1u;
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 2) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// ---- conv tail after the two GEMMs: out = maxpool2(relu(mean + sd * eps)) from pool-major GEMM rows ----
// mean / sd: [M, Np] with row m = 4 * window + 2 * (oy & 1) + (ox & 1), window = (img * PH + py) * PW + px.
// A thread owns one channel of a 2 x 4 patch (two pool windows): the four outputs of a Philox call are four
// consecutive ox of one row, so two calls cover the patch (the GEMM-epilogue form of this stage, mode 5, spends a
// whole Philox call per element on 8 warps per SM and took 3x longer than this full-occupancy pass).
// Needs OW % 4 == 0.  Channels are the fastest thread index: loads of mean / sd are contiguous across the warp.
struct RowsPoolDivs {  // run-time divisors of the index decode, as multiply-shift pairs
    FastDiv c, gx, ph;
};
template <bool IDX32>
__global__ void conv_rows_noise_pool_kernel(const float *__restrict__ mean, const float *__restrict__ sd,
                                            const float *__restrict__ eps, uint64_t seed, uint32_t noise_stream,
                                            uint64_t row_offset, float *__restrict__ out, long long n_imgs, int C, int Np,
                                            int OH, int OW, const float *__restrict__ zs, long long rows_per_z,
                                            const RowsPoolDivs dv) {
    const int PH = OH >> 1, PW = OW >> 1, GX = OW >> 2;
    const long long total = n_imgs * PH * GX * C;
    const Philox rng(seed);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        int n, gx, py;
        long long img;
        if constexpr (IDX32) {  // fewer than 2^31 work items: multiply-shift divisions instead of 64-bit divides
            uint32_t t, a, b, cc;
            dv.c.divmod((uint32_t)i, t, a);
            dv.gx.divmod(t, t, b);
            dv.ph.divmod(t, t, cc);
            n = (int)a, gx = (int)b, py = (int)cc, img = (long long)t;
        } else {
            n = (int)(i % C);
            long long t = i / C;
            gx = (int)(t % GX);
            t /= GX;
            py = (int)(t % PH);
            img = t / PH;
        }
        float best0 = 0.f, best1 = 0.f;  // ReLU folded into the max
        const float zc = zs ? zs[(img / rows_per_z) * C + n] : 1.f;  // per-sample conv z (mean was evaluated for z = 1)
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const int oy = 2 * py + r;
            const long long le = ((img * C + n) * OH + oy) * OW + 4 * gx;
            float nz[4];
            if (eps) {
                const float4 e = *reinterpret_cast<const float4 *>(eps + le);
                nz[0] = e.x, nz[1] = e.y, nz[2] = e.z, nz[3] = e.w;
            } else {
                const uint4 rr = rng((uint64_t)(le + (long long)row_offset * C * OH * OW) >> 2, noise_stream);
                const float2 a = box_muller(rr.x, rr.y), b = box_muller(rr.z, rr.w);
                nz[0] = a.x, nz[1] = a.y, nz[2] = b.x, nz[3] = b.y;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const long long w = (img * PH + py) * PW + 2 * gx + (u >> 1);
                const size_t e = (size_t)(4 * w + 2 * r + (u & 1)) * Np + n;
                const float v = fmaf(sd[e], nz[u], zc * mean[e]);
                if (u < 2) best0 = fmaxf(best0, v);
                else best1 = fmaxf(best1, v);
            }
        }
        float *o = out + ((img * C + n) * PH + py) * PW + 2 * gx;
        o[0] = best0, o[1] = best1;
    }
}

static int launch_rows_noise_pool(const float *mean, const float *sd, const float *eps, uint64_t seed, uint32_t noise_stream,
                                  uint64_t row_offset, float *out, long long n_imgs, int C, int Np, int OH, int OW,
                                  const float *zs, long long rows_per_z, long long total, unsigned blocks, cudaStream_t st) {
    RowsPoolDivs dv;
    dv.c = FastDiv((uint32_t)C), dv.gx = FastDiv((uint32_t)(OW / 4)), dv.ph = FastDiv((uint32_t)(OH / 2));
    if (total < 0x7fffffffLL)
        conv_rows_noise_pool_kernel<true><<<blocks, 256, 0, st>>>(mean, sd, eps, seed, noise_stream, row_offset, out, n_imgs, C, Np,
                                                                 OH, OW, zs, rows_per_z, dv);
    else
        conv_rows_noise_pool_kernel<false><<<blocks, 256, 0, st>>>(mean, sd, eps, seed, noise_stream, row_offset, out, n_imgs, C, Np,
                                                                  OH, OW, zs, rows_per_z, dv);
    return launch_status("conv_rows_noise_pool_kernel");
}

// smem of conv_implicit_kernel for this geometry (0 = not eligible)
static size_t conv_implicit_smem(int c_in, int height, int width, int ksize, int Kp, int Np) {
    const int OH = height - ksize + 1, OW = width - ksize + 1, RPI = OH * OW, CHW = c_in * height * width;
    if (RPI <= 0 || BM % RPI != 0 || Np > CONV_BN || Np % 32 != 0 || CHW % 4 != 0 || Kp % CONV_BK != 0) return 0;
    if (Kp > CONV_MAX_KP) return 0;
    const size_t bytes = (size_t)CONV_STAGES * CONV_STAGE_BYTES + 1024 + 256 + sizeof(float) * CONV_BN +
                         sizeof(float) * 2 * (size_t)(BM / RPI) * CHW + 16;
    return bytes <= 227 * 1024 ? bytes : 0;
}

// fp16 weight matrix [rows, cols] (row pitch cols halves) as a TMA map of 64 x box_rows boxes, 128-byte swizzle
static int make_map_f16(CUtensorMap *map, const void *ptr, int rows, int cols, int box_rows) {
    EncodeTiledFn fn = encode_fn();
    MNF_REQUIRE(fn != nullptr, MNF_E_DEVICE, "cuTensorMapEncodeTiled is not available from this driver");
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)cols * 2};
    cuuint32_t box[2] = {(cuuint32_t)CONV_BK, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, (void *)ptr, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    MNF_REQUIRE(r == CUDA_SUCCESS, MNF_E_ARG, "cuTensorMapEncodeTiled (fp16) failed with CUresult %d (rows=%d cols=%d)", (int)r, rows, cols);
    return 0;
}

// Bm / Bv: fp16 [Np, Kp] from conv_pack_weights_f16_kernel
static int launch_conv_implicit(const float *x, const void *Bm, const void *Bv, const float *bvar_log, float *mean, float *sd,
                                long long n_imgs, int c_in, int height, int width, int ksize, int Kp, int Np,
                                cudaStream_t stream) {
    const DeviceProps *dp = device_props();
    MNF_REQUIRE(dp != nullptr && dp->cc_major == 10, MNF_E_DEVICE, "tcgen05 path needs an sm_100 device");
    const size_t smem = conv_implicit_smem(c_in, height, width, ksize, Kp, Np);
    MNF_REQUIRE(smem != 0, MNF_E_SHAPE, "geometry not eligible for the implicit-GEMM conv");
    MNF_REQUIRE(((uintptr_t)x % 16) == 0 && ((uintptr_t)mean % 16) == 0 && ((uintptr_t)sd % 16) == 0, MNF_E_ALIGN,
                "pointers must be 16-byte aligned");
    CUtensorMap mbm, mbv;
    int rc = make_map_f16(&mbm, Bm, Np, Kp, CONV_BN);
    if (rc) return rc;
    rc = make_map_f16(&mbv, Bv, Np, Kp, CONV_BN);
    if (rc) return rc;
    MNF_CUDA(cudaFuncSetAttribute(conv_implicit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int RPI = (height - ksize + 1) * (width - ksize + 1), IMGS = BM / RPI;
    const long long n_tiles = (n_imgs + IMGS - 1) / IMGS;
    const unsigned grid = (unsigned)(n_tiles < dp->sm_count ? n_tiles : dp->sm_count);
    ConvTaps taps;
    const int K = c_in * ksize * ksize;
    for (int k = 0; k < CONV_MAX_KP; ++k) {
        const int kx = k % ksize, ky = (k / ksize) % ksize, ci = k / (ksize * ksize);
        taps.off[k] = k < K ? (ci * height + ky) * width + kx : 0;  // padded taps: any valid address (weights are zero there)
    }
    conv_implicit_kernel<<<grid, CONV_THREADS, smem, stream>>>(mbm, mbv, taps, x, bvar_log, mean, sd, n_imgs, c_in, height,
                                                               width, ksize, Kp, Np);
    return launch_status("conv_implicit_kernel");
}

}  // namespace tc
}  // namespace mnf

namespace mnf {
namespace tc {

// xz[m,k] = x[m % x_rows, k] * z[m,k]   (A operand of the mean GEMM, mnf_linear.py:48)
__global__ void xz_kernel(const float4 *__restrict__ x, const float4 *__restrict__ z, float4 *__restrict__ xz,
                          long long n_rows, int x_rows, int k4) {
    const long long total = n_rows * k4;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total;
         e += (long long)gridDim.x * blockDim.x) {
        const long long m = e / k4;
        const int c = (int)(e - m * k4);
        const float4 a = x[(size_t)(m % x_rows) * k4 + c], b = z[e];
        xz[e] = make_float4(rn_tf32(a.x * b.x), rn_tf32(a.y * b.y), rn_tf32(a.z * b.z), rn_tf32(a.w * b.w));
    }
}
// out = tf32(f(in)): f = identity (0), exp (1: W_var, mnf_linear.py:50) or square (2: x**2, mnf_linear.py:53)
__global__ void unary_kernel(const float *__restrict__ in, float *__restrict__ out, long long n, int op) {
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        const float v = in[e];
        out[e] = rn_tf32(op == 2 ? v * v : (op == 1 ? expf(v) : v));
    }
}

static unsigned blocks_for(long long n) {
    long long b = (n + 255) / 256;
    return (unsigned)(b > 148 * 32 ? 148 * 32 : (b < 1 ? 1 : b));
}

}  // namespace tc
}  // namespace mnf

using namespace mnf;

extern "C" {

int64_t mnf_linear_tc_workspace(int64_t x_rows, int64_t n_rows, int n_in, int n_out) {
    return n_rows * n_in + 2 * (int64_t)n_out * n_in + x_rows * n_in + x_rows * (int64_t)n_out;
}

// MNFLinear.forward (mnf_linear.py:46-56) on the tensor cores:
//   sd  = sqrt(x^2 exp(W_log_var)^T + exp(b_log_var))      [x_rows, n_out]   (TF32 GEMM, epilogue mode 2)
//   out = (x*z) W_mean^T + b_mean + sd[m % x_rows] * eps   [n_rows, n_out]   (TF32 GEMM, epilogue mode 1)
// The variance depends on x only, so under Monte-Carlo replication (x_rows < n_rows) it is evaluated once per
// distinct input row instead of once per sample -- the flops actually executed are reported as such.
int mnf_linear_forward_tc(const float *x, int64_t x_rows, const float *z, const float *W_mean, const float *W_log_var,
                          const float *b_mean, const float *b_log_var, const float *eps, uint64_t seed,
                          uint32_t noise_stream, uint64_t row_offset, float *out, int64_t n_rows, int n_in, int n_out,
                          int relu, float *workspace, void *stream) {
    return mnf_linear_forward_tc_affine(x, x_rows, z, W_mean, W_log_var, b_mean, b_log_var, eps, seed, noise_stream,
                                        row_offset, out, n_rows, n_in, n_out, relu, nullptr, nullptr, workspace, stream);
}

// ... and out = col_scale[n] * out + col_shift[n] after the ReLU (both NULL: the plain layer, bit for bit)
int mnf_linear_forward_tc_affine(const float *x, int64_t x_rows, const float *z, const float *W_mean,
                                 const float *W_log_var, const float *b_mean, const float *b_log_var, const float *eps,
                                 uint64_t seed, uint32_t noise_stream, uint64_t row_offset, float *out, int64_t n_rows,
                                 int n_in, int n_out, int relu, const float *col_scale, const float *col_shift,
                                 float *workspace, void *stream) {
    MNF_REQUIRE(x && W_mean && W_log_var && b_mean && b_log_var && out && workspace, MNF_E_ARG, "NULL pointer");
    MNF_REQUIRE((col_scale == nullptr) == (col_shift == nullptr), MNF_E_ARG,
                "col_scale and col_shift must both be given or both be NULL");
    MNF_REQUIRE(((uintptr_t)col_scale % 16) == 0 && ((uintptr_t)col_shift % 16) == 0, MNF_E_ALIGN,
                "col_scale and col_shift must be 16-byte aligned");
    MNF_REQUIRE(n_rows >= 0 && n_rows <= 0x7fffffff - 256 && x_rows >= 1 && x_rows <= n_rows + (n_rows == 0), MNF_E_ARG,
                "bad row counts");
    MNF_REQUIRE(n_in % 4 == 0, MNF_E_SHAPE, "tensor-core path needs n_in %% 4 == 0 (got %d)", n_in);
    if (n_rows == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    float *xz = workspace, *expW = xz + (size_t)n_rows * n_in, *wm = expW + (size_t)n_out * n_in,
          *x2 = wm + (size_t)n_out * n_in, *sd = x2 + (size_t)x_rows * n_in;
    const int k4 = n_in / 4;
    if (z)  // z == NULL: the caller (mnf_rnvp_forward_tc) already left tf32(x*z) at the start of the workspace
        tc::xz_kernel<<<tc::blocks_for(n_rows * k4), 256, 0, st>>>((const float4 *)x, (const float4 *)z, (float4 *)xz,
                                                                  n_rows, (int)x_rows, k4);
    tc::unary_kernel<<<tc::blocks_for((long long)n_out * n_in), 256, 0, st>>>(W_log_var, expW, (long long)n_out * n_in, 1);
    tc::unary_kernel<<<tc::blocks_for((long long)n_out * n_in), 256, 0, st>>>(W_mean, wm, (long long)n_out * n_in, 0);
    tc::unary_kernel<<<tc::blocks_for(x_rows * n_in), 256, 0, st>>>(x, x2, x_rows * n_in, 2);
    int rc = launch_status("mnf_linear_forward_tc prologue");
    if (rc) return rc;
    tc::Epilogue ev{};
    ev.mode = 2, ev.sd_rows = 1, ev.bvar_log = b_log_var, ev.out = sd;
    rc = tc::launch(x2, expW, (int)x_rows, n_out, n_in, ev, st);
    if (rc) return rc;
    tc::Epilogue em{};
    em.mode = 1, em.bias = b_mean, em.sd = sd, em.sd_rows = (int)x_rows, em.eps = eps, em.seed = seed;
    em.noise_stream = noise_stream, em.row_offset = row_offset, em.relu = relu, em.out = out;
    em.col_scale = col_scale, em.col_shift = col_shift;
    return tc::launch(xz, wm, (int)n_rows, n_out, n_in, em, st);
}

// C = A B^T (+ bias), TF32 tensor cores.  Test / building-block entry point.
int mnf_tc_linear(const float *A, const float *W, const float *bias, float *out, int64_t M, int N, int K, int relu,
                  int round_out, void *stream) {
    MNF_REQUIRE(A && W && out, MNF_E_ARG, "NULL pointer");
    MNF_REQUIRE(M >= 0 && M <= 0x7fffffff - 256 && N >= 1 && K >= 1, MNF_E_ARG, "bad shape");
    if (M == 0) return 0;
    tc::Epilogue ep{};
    ep.bias = bias, ep.sd_rows = 1, ep.relu = relu, ep.out = out, ep.round_out = round_out;
    return tc::launch(A, W, (int)M, N, K, ep, (cudaStream_t)stream);
}

// MAF.inverse (density direction, maf.py:53-62) for a stack of MAF flows on the tensor cores.
//   layers_host[f]: packed, mask-folded, TF32-rounded weights of flow f (see mnf_made_layer)
//   x [n_rows, dim] -> z [n_rows, dim], log_det [n_rows] (sum over the flows)
//   workspace: mnf_made_workspace() floats
int mnf_made_density_tc(const mnf_made_layer *layers_host, int n_flows, const float *x, float *z, float *log_det,
                        float *intermediates, int64_t n_rows, int dim, float *workspace, void *stream) {
    MNF_REQUIRE(layers_host && x && z && log_det && workspace, MNF_E_ARG, "NULL pointer");
    MNF_REQUIRE(n_flows >= 1 && dim >= 4 && dim % 4 == 0 && 2 * dim <= tc::MAX_BN, MNF_E_SHAPE,
                "tensor-core MADE needs dim %% 4 == 0 and dim <= %d (got %d)", tc::MAX_BN / 2, dim);
    MNF_REQUIRE(n_rows >= 0 && n_rows <= 0x7fffffff - 256, MNF_E_ARG, "bad row count");
    if (n_rows == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    int maxh = 4;
    for (int f = 0; f < n_flows; ++f)
        for (int l = 0; l < layers_host[f].n_hidden; ++l) {
            const int h = layers_host[f].hidden[l];
            MNF_REQUIRE(h % 4 == 0 && h >= 8, MNF_E_SHAPE, "hidden width %d must be a multiple of 4 and >= 8", h);
            maxh = h > maxh ? h : maxh;
        }
    // workspace: xr (rounded input) | zbuf[2] (ping-pong exact z) | h[2]
    float *xr = workspace, *za = xr + (size_t)n_rows * dim, *zb = za + (size_t)n_rows * dim,
          *ha = zb + (size_t)n_rows * dim, *hb = ha + (size_t)n_rows * maxh;
    tc::unary_kernel<<<tc::blocks_for(n_rows * dim), 256, 0, st>>>(x, xr, n_rows * dim, 0);
    MNF_CUDA(cudaMemsetAsync(log_det, 0, sizeof(float) * n_rows, st));  // epilogues accumulate into it
    int rc = launch_status("made round input");
    if (rc) return rc;
    const float *cur_exact = x;
    const float *cur_round = xr;
    for (int f = 0; f < n_flows; ++f) {
        const mnf_made_layer &L = layers_host[f];
        MNF_REQUIRE(L.n_hidden >= 1 && L.n_hidden <= MNF_MADE_MAX_HIDDEN, MNF_E_SHAPE, "flow %d: n_hidden=%d", f, L.n_hidden);
        const float *a = cur_round;
        int k = dim;
        float *hout = ha;
        for (int l = 0; l < L.n_hidden; ++l) {
            tc::Epilogue ep{};
            ep.bias = L.b[l], ep.sd_rows = 1, ep.relu = 1, ep.out = hout, ep.round_out = 1;
            rc = tc::launch(a, L.w[l], (int)n_rows, L.hidden[l], k, ep, st);
            if (rc) return rc;
            a = hout;
            k = L.hidden[l];
            hout = (hout == ha) ? hb : ha;
        }
        const bool last = f == n_flows - 1;
        float *zout = intermediates ? intermediates + (size_t)f * n_rows * dim : (last ? z : (cur_exact == za ? zb : za));
        float *zround = last ? nullptr : xr;  // the rounded copy of the previous input is dead by now
        tc::Epilogue ep{};
        ep.mode = 3, ep.bias = L.b_out, ep.sd_rows = 1, ep.out = zout, ep.xin = cur_exact, ep.out_rounded = zround;
        ep.ld_in = f == 0 ? nullptr : log_det, ep.ld_out = log_det, ep.parity = L.parity;
        rc = tc::launch(a, L.w_out, (int)n_rows, 2 * dim, k, ep, st);
        if (rc) return rc;
        cur_exact = zout;
        cur_round = xr;
    }
    if (intermediates)
        MNF_CUDA(cudaMemcpyAsync(z, cur_exact, sizeof(float) * n_rows * dim, cudaMemcpyDeviceToDevice, st));
    return 0;
}

int64_t mnf_made_workspace(int64_t n_rows, int dim, int max_hidden) {
    return n_rows * (3 * (int64_t)dim + 2 * (int64_t)max_hidden);
}

namespace mnf {
namespace tc {

constexpr int RNVP_HP = 64;  // conditioner width padded to one 64-wide tile / two K blocks

// per flow: Wn_p [64, dim] (rows >= h zero), bn_p [64], Wts [2*dim, 64] interleaved (t_n, s_n) rows with K padded,
// bts [2*dim]; everything TF32-rounded
__global__ void rnvp_pack_kernel(const float *__restrict__ Wn, const float *__restrict__ bn,
                                 const float *__restrict__ Wt, const float *__restrict__ bt,
                                 const float *__restrict__ Ws, const float *__restrict__ bsc, int h, int dim,
                                 float *__restrict__ Wn_p, float *__restrict__ bn_p, float *__restrict__ Wts,
                                 float *__restrict__ bts, int bias_column) {
    // bias_column: column 63 of the padded conditioner output is a constant one (its packed bias is 1, its weights 0) and
    // column 63 of Wts holds the shift / scale biases -- the form the fused output-GEMM + gate kernel consumes
    const long long n1 = (long long)RNVP_HP * dim, n2 = 2LL * dim * RNVP_HP;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n1 + n2; e += (long long)gridDim.x * blockDim.x) {
        if (e < n1) {
            const int j = (int)(e / dim), k = (int)(e % dim);
            Wn_p[e] = j < h ? rn_tf32(Wn[(size_t)j * dim + k]) : 0.f;
            if (k == 0) bn_p[j] = j < h ? bn[j] : ((bias_column && j == RNVP_HP - 1) ? 1.f : 0.f);
        } else {
            const long long f = e - n1;
            const int row = (int)(f / RNVP_HP), k = (int)(f % RNVP_HP), n = row >> 1;
            const float *src = (row & 1) ? Ws : Wt;
            const float bias = (row & 1) ? bsc[n] : bt[n];
            Wts[f] = k < h ? rn_tf32(src[(size_t)n * h + k]) : ((bias_column && k == RNVP_HP - 1) ? rn_tf32(bias) : 0.f);
            if (k == 0) bts[row] = bias;
        }
    }
}

// z = q0_mean + sqrt(exp(q0_log_var)) * eps (mnf_linear.py:59-62) and mz = tf32(mask_0 * z) in one pass
__global__ void z0_mask_kernel(const float *__restrict__ q0_mean, const float *__restrict__ q0_log_var,
                               const float *__restrict__ eps, const float *__restrict__ mask, float *__restrict__ z,
                               float *__restrict__ mz, long long n_rows, int dim, uint64_t seed, uint32_t eps_stream,
                               uint32_t mask_stream, uint64_t row_offset) {
    const Philox rng(seed);
    const long long total4 = n_rows * dim / 4;
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < total4; c += (long long)gridDim.x * blockDim.x) {
        const long long e0 = c * 4;
        const int d = (int)(e0 % dim);
        const uint64_t g0 = (uint64_t)row_offset * dim + e0;
        float n4[4], m4[4];
        if (eps) {
            const float4 q = *reinterpret_cast<const float4 *>(eps + e0);
            n4[0] = q.x, n4[1] = q.y, n4[2] = q.z, n4[3] = q.w;
        } else {
            const uint4 q = rng(g0 >> 2, eps_stream);
            const float2 a = box_muller(q.x, q.y), b = box_muller(q.z, q.w);
            n4[0] = a.x, n4[1] = a.y, n4[2] = b.x, n4[3] = b.y;
        }
        if (mask) {
            const float4 q = *reinterpret_cast<const float4 *>(mask + e0);
            m4[0] = q.x, m4[1] = q.y, m4[2] = q.z, m4[3] = q.w;
        } else {
            const uint32_t bits = philox_bits16(rng, g0 & ~15ull, mask_stream) >> (g0 & 15u);
#pragma unroll
            for (int u = 0; u < 4; ++u) m4[u] = (float)((bits >> u) & 1u);
        }
        const float4 mu = *reinterpret_cast<const float4 *>(q0_mean + d);
        const float4 lv = *reinterpret_cast<const float4 *>(q0_log_var + d);
        const float zv[4] = {mu.x + sqrtf(expf(lv.x)) * n4[0], mu.y + sqrtf(expf(lv.y)) * n4[1],
                             mu.z + sqrtf(expf(lv.z)) * n4[2], mu.w + sqrtf(expf(lv.w)) * n4[3]};
        *reinterpret_cast<float4 *>(z + e0) = make_float4(zv[0], zv[1], zv[2], zv[3]);
        *reinterpret_cast<float4 *>(mz + e0) =
            make_float4(rn_tf32(m4[0] * zv[0]), rn_tf32(m4[1] * zv[1]), rn_tf32(m4[2] * zv[2]), rn_tf32(m4[3] * zv[3]));
    }
}

// Philox-only form of z0_mask_kernel for dim % 128 == 0 (BASELINE config 5: 268 M normals per 65 536 rows, ALU-bound).
// A warp owns spans of 4096 consecutive elements: one Philox block yields the Bernoulli bits of 128 elements, so lane L
// draws the mask block of the span's L-th 128-element group once and hands it round by shuffle (the general kernel drew
// one block per float4: 32x the calls); q0_mean and the standard deviation exp(q0_log_var / 2) come from a shared-memory
// table; accesses are 512 contiguous bytes per warp instruction.  Draw numbering identical to the general kernel.
__global__ void __launch_bounds__(256)
z0_mask_philox_kernel(const float *__restrict__ q0_mean, const float *__restrict__ q0_log_var, float *__restrict__ z,
                      float *__restrict__ mz, long long n_rows, int dim, uint64_t seed, uint32_t eps_stream,
                      uint32_t mask_stream, uint64_t row_offset) {
    extern __shared__ float tab[];  // [dim] mean | [dim] std
    for (int i = threadIdx.x; i < dim; i += blockDim.x) tab[i] = q0_mean[i], tab[dim + i] = sqrtf(expf(q0_log_var[i]));
    __syncthreads();
    const Philox rng(seed);
    const long long total = n_rows * dim, n_spans = (total + 4095) >> 12;
    const int lane = threadIdx.x & 31;
    const long long warp_id = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
    const uint64_t gbase = (uint64_t)row_offset * dim;  // a multiple of 128: the groups line up with Philox mask blocks
    for (long long span = warp_id; span < n_spans; span += n_warps) {
        const long long s0 = span << 12;
        const uint4 mb = rng((gbase + (uint64_t)s0 + 128ull * lane) >> 7, mask_stream);  // mask bits of the span's group `lane`
#pragma unroll 4
        for (int i = 0; i < 32; ++i) {
            const uint32_t wx = __shfl_sync(0xffffffffu, mb.x, i), wy = __shfl_sync(0xffffffffu, mb.y, i),
                           wz = __shfl_sync(0xffffffffu, mb.z, i), ww = __shfl_sync(0xffffffffu, mb.w, i);
            const long long e0 = s0 + 128 * i + 4 * lane;
            if (e0 >= total) break;
            const uint32_t word = lane < 8 ? wx : (lane < 16 ? wy : (lane < 24 ? wz : ww));
            const uint32_t bits = (word >> ((4 * lane) & 31)) & 0xFu;
            const uint4 q = rng((gbase + (uint64_t)e0) >> 2, eps_stream);
            const float2 a = box_muller(q.x, q.y), b = box_muller(q.z, q.w);
            const int d = (int)(e0 % dim);
            const float4 mu = *reinterpret_cast<const float4 *>(tab + d), sd = *reinterpret_cast<const float4 *>(tab + dim + d);
            const float z0 = fmaf(sd.x, a.x, mu.x), z1 = fmaf(sd.y, a.y, mu.y), z2 = fmaf(sd.z, b.x, mu.z), z3 = fmaf(sd.w, b.y, mu.w);
            st_stream4(reinterpret_cast<float4 *>(z + e0), make_float4(z0, z1, z2, z3));
            st_stream4(reinterpret_cast<float4 *>(mz + e0),
                       make_float4((bits & 1u) ? rn_tf32(z0) : 0.f, (bits & 2u) ? rn_tf32(z1) : 0.f, (bits & 4u) ? rn_tf32(z2) : 0.f,
                                   (bits & 8u) ? rn_tf32(z3) : 0.f));
        }
    }
}

// mz = tf32(mask * z) for the first flow of the stack
__global__ void mask_mul_kernel(const float *__restrict__ z, const float *__restrict__ mask, float *__restrict__ mz,
                                long long n_rows, int dim, uint64_t seed, uint32_t stream, uint64_t row_offset) {
    const Philox rng(seed);
    const long long total16 = n_rows * dim / 16;
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < total16; c += (long long)gridDim.x * blockDim.x) {
        const long long e0 = c * 16;
        const uint32_t bits = mask ? 0u : philox_bits16(rng, (uint64_t)row_offset * dim + e0, stream);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float4 v = *reinterpret_cast<const float4 *>(z + e0 + 4 * q);
            float m[4];
            if (mask) {
                const float4 mv = *reinterpret_cast<const float4 *>(mask + e0 + 4 * q);
                m[0] = mv.x, m[1] = mv.y, m[2] = mv.z, m[3] = mv.w;
            } else {
#pragma unroll
                for (int u = 0; u < 4; ++u) m[u] = (float)((bits >> (4 * q + u)) & 1u);
            }
            *reinterpret_cast<float4 *>(mz + e0 + 4 * q) =
                make_float4(rn_tf32(m[0] * v.x), rn_tf32(m[1] * v.y), rn_tf32(m[2] * v.z), rn_tf32(m[3] * v.w));
        }
    }
}

// RNVP gate (rnvp.py:32-39) as a full-occupancy streaming pass over ts = [shift_0, scale_0, shift_1, ...] written by
// the GEMM: one CTA per row, float4 over 4 dims, block-reduced log-det (no atomics).  Also stages the next GEMM's
// operand: mz_next = tf32(mask_next * z_new) or xz = tf32(x[m % x_rows] * z_new).
__global__ void __launch_bounds__(256)
rnvp_gate_kernel(const float *__restrict__ ts, float *__restrict__ z, float *__restrict__ log_det,
                 const float *__restrict__ mask, const float *__restrict__ mask_next, float *__restrict__ mz_next,
                 const float *__restrict__ xmul, int xmul_rows, float *__restrict__ xz_out, long long n_rows, int dim,
                 uint64_t seed, uint32_t stream, uint32_t next_stream, uint64_t row_offset) {
    __shared__ float red[8];
    const Philox rng(seed);
    for (long long m = blockIdx.x; m < n_rows; m += gridDim.x) {
        float ld = 0.f;
        for (int j = 4 * threadIdx.x; j < dim; j += 4 * blockDim.x) {
            const size_t e0 = (size_t)m * dim + j;
            const float4 a = *reinterpret_cast<const float4 *>(ts + 2 * e0);      // shift_j, scale_j, shift_j+1, scale_j+1
            const float4 b = *reinterpret_cast<const float4 *>(ts + 2 * e0 + 4);  // ... j+2, j+3
            const float4 zv = *reinterpret_cast<const float4 *>(z + e0);
            const uint64_t g0 = (uint64_t)row_offset * dim + e0;
            float mk[4], mn[4];
            if (mask) {
                const float4 q = *reinterpret_cast<const float4 *>(mask + e0);
                mk[0] = q.x, mk[1] = q.y, mk[2] = q.z, mk[3] = q.w;
            } else {
                const uint32_t bits = philox_bits16(rng, g0 & ~15ull, stream) >> (g0 & 15u);
#pragma unroll
                for (int u = 0; u < 4; ++u) mk[u] = (float)((bits >> u) & 1u);
            }
            const float sh[4] = {a.x, a.z, b.x, b.z}, sc[4] = {a.y, a.w, b.y, b.w}, zi[4] = {zv.x, zv.y, zv.z, zv.w};
            float zn[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const float gate = __fdividef(1.f, 1.f + __expf(-sc[u]));      // torch.sigmoid, rnvp.py:35
                zn[u] = ((1.f - mk[u]) * zi[u] * gate + (1.f - gate) * sh[u]) + mk[u] * zi[u];  // rnvp.py:37
                ld += (1.f - mk[u]) * __logf(gate);                             // rnvp.py:36
            }
            *reinterpret_cast<float4 *>(z + e0) = make_float4(zn[0], zn[1], zn[2], zn[3]);
            if (mz_next) {
                if (mask_next) {
                    const float4 q = *reinterpret_cast<const float4 *>(mask_next + e0);
                    mn[0] = q.x, mn[1] = q.y, mn[2] = q.z, mn[3] = q.w;
                } else {
                    const uint32_t bits = philox_bits16(rng, g0 & ~15ull, next_stream) >> (g0 & 15u);
#pragma unroll
                    for (int u = 0; u < 4; ++u) mn[u] = (float)((bits >> u) & 1u);
                }
                *reinterpret_cast<float4 *>(mz_next + e0) =
                    make_float4(rn_tf32(mn[0] * zn[0]), rn_tf32(mn[1] * zn[1]), rn_tf32(mn[2] * zn[2]), rn_tf32(mn[3] * zn[3]));
            }
            if (xz_out) {
                const float4 xv = *reinterpret_cast<const float4 *>(xmul + (size_t)(m % xmul_rows) * dim + j);
                *reinterpret_cast<float4 *>(xz_out + e0) =
                    make_float4(rn_tf32(xv.x * zn[0]), rn_tf32(xv.y * zn[1]), rn_tf32(xv.z * zn[2]), rn_tf32(xv.w * zn[3]));
            }
        }
        ld = warp_sum(ld);
        __syncthreads();
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ld;
        __syncthreads();
        if (threadIdx.x == 0) {
            float t = 0.f;
            for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
            log_det[m] += t;
        }
    }
}

}  // namespace tc
}  // namespace mnf

int64_t mnf_rnvp_tc_workspace(int n_flows, int64_t n_rows, int dim) {
    const int64_t per_flow = (int64_t)tc::RNVP_HP * dim + tc::RNVP_HP + 2LL * dim * tc::RNVP_HP + 2LL * dim;
    return n_rows * dim + n_rows * tc::RNVP_HP + 2 * n_rows * dim + n_flows * per_flow + 64;
}

// NormalizingFlow([RNVP...]).forward (core.py:17-25 over rnvp.py:25-39) on the tensor cores, in place on z.
// Per flow: y = tf32(mask*z) Wn^T + bn (narrow-tile GEMM), then [shift | scale] = y [Wt; Ws]^T with the gated
// update, the log-det row sum and the staging of the next GEMM's operand fused into the epilogue.
// Needs single-Linear conditioners (h_sizes of length 1, width <= 64) and dim % 16 == 0.
int mnf_rnvp_forward_tc(const mnf_rnvp_flow *flows_host, int n_flows, float *z, float *log_det,
                        const float *const *masks_host, uint64_t seed, uint32_t first_noise_stream, uint64_t row_offset,
                        int64_t n_rows, int dim, const float *x, int64_t x_rows, float *xz_out, float *workspace,
                        const float *q0_mean, const float *q0_log_var, const float *eps_z, uint32_t eps_stream,
                        int z_is_scratch, void *stream) {
    MNF_REQUIRE(flows_host && z && log_det && workspace, MNF_E_ARG, "NULL pointer");
    MNF_REQUIRE(n_flows >= 1 && n_rows >= 0 && n_rows <= 0x7fffffff - 256, MNF_E_ARG, "bad shape");
    MNF_REQUIRE(dim % 16 == 0 && dim >= 32, MNF_E_SHAPE, "tensor-core RNVP needs dim %% 16 == 0 and dim >= 32 (got %d)", dim);
    MNF_REQUIRE(!xz_out || (x && x_rows >= 1), MNF_E_ARG, "xz_out needs x");
    for (int f = 0; f < n_flows; ++f)
        MNF_REQUIRE(flows_host[f].n_net == 1 && flows_host[f].net_sizes[0] <= tc::RNVP_HP, MNF_E_SHAPE,
                    "tensor-core RNVP needs a single-Linear conditioner of width <= %d", tc::RNVP_HP);
    if (n_rows == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    float *mz = workspace, *y = mz + (size_t)n_rows * dim, *ts = y + (size_t)n_rows * tc::RNVP_HP,
          *wbase = ts + 2 * (size_t)n_rows * dim;
    wbase += (16 - ((uintptr_t)wbase / 4) % 16) % 16;  // keep every packed matrix 64-byte aligned
    const size_t per_flow = (size_t)tc::RNVP_HP * dim + tc::RNVP_HP + 2ull * dim * tc::RNVP_HP + 2ull * dim;
    // wide dims take the fused output-GEMM + gate kernel (rnvp_fused.cu): the [R, 2 * dim] shift / scale matrix never exists
    bool fused = true;
    for (int f = 0; f < n_flows; ++f) fused = fused && rnvpf::eligible(dim, flows_host[f].net_sizes[0]);
    if (!fused) MNF_CUDA(cudaMemsetAsync(log_det, 0, sizeof(float) * n_rows, st));
    for (int f = 0; f < n_flows; ++f) {
        const mnf_rnvp_flow &fl = flows_host[f];
        float *Wn_p = wbase + f * per_flow, *bn_p = Wn_p + (size_t)tc::RNVP_HP * dim, *Wts = bn_p + tc::RNVP_HP,
              *bts = Wts + 2ull * dim * tc::RNVP_HP;
        tc::rnvp_pack_kernel<<<tc::blocks_for((long long)tc::RNVP_HP * dim * 3), 256, 0, st>>>(
            fl.net_w[0], fl.net_b[0], fl.t_w, fl.t_b, fl.s_w, fl.s_b, fl.net_sizes[0], dim, Wn_p, bn_p, Wts, bts, fused ? 1 : 0);
    }
    const bool philox_fast = q0_mean && q0_log_var && !eps_z && !masks_host && dim % 128 == 0 && dim <= 8192;
    if (philox_fast) {
        const size_t smem = 2 * sizeof(float) * (size_t)dim;
        if (smem > 48 * 1024)
            MNF_CUDA(cudaFuncSetAttribute(tc::z0_mask_philox_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        tc::z0_mask_philox_kernel<<<148 * 4, 256, smem, st>>>(q0_mean, q0_log_var, z, mz, n_rows, dim, seed, eps_stream,
                                                              first_noise_stream, row_offset);
    } else if (q0_mean && q0_log_var)  // sample z0 here (saves a pass over z): MNFLinear.sample_z, mnf_linear.py:58-62
        tc::z0_mask_kernel<<<tc::blocks_for(n_rows * dim / 4), 256, 0, st>>>(q0_mean, q0_log_var, eps_z,
                                                                           masks_host ? masks_host[0] : nullptr, z, mz,
                                                                           n_rows, dim, seed, eps_stream,
                                                                           first_noise_stream, row_offset);
    else
        tc::mask_mul_kernel<<<tc::blocks_for(n_rows * dim / 16), 256, 0, st>>>(z, masks_host ? masks_host[0] : nullptr,
                                                                             mz, n_rows, dim, seed,
                                                                             first_noise_stream, row_offset);
    int rc = launch_status("rnvp tc prologue");
    if (rc) return rc;
    for (int f = 0; f < n_flows; ++f) {
        float *Wn_p = wbase + f * per_flow, *bn_p = Wn_p + (size_t)tc::RNVP_HP * dim, *Wts = bn_p + tc::RNVP_HP,
              *bts = Wts + 2ull * dim * tc::RNVP_HP;
        tc::Epilogue e1{};
        e1.bias = bn_p, e1.sd_rows = 1, e1.out = y, e1.round_out = 1;
        rc = tc::launch(mz, Wn_p, (int)n_rows, tc::RNVP_HP, dim, e1, st);
        if (rc) return rc;
        const bool last = f == n_flows - 1;
        if (fused) {
            rnvpf::Params gp{};
            gp.z = z, gp.log_det = log_det;
            gp.mask = masks_host ? masks_host[f] : nullptr;
            gp.mask_next = (!last && masks_host) ? masks_host[f + 1] : nullptr;
            gp.mz_next = last ? nullptr : mz;
            gp.xmul = x, gp.xmul_rows = (int)(x_rows > 0 ? x_rows : 1);
            gp.xz_out = (last && xz_out) ? xz_out : nullptr;
            gp.n_rows = n_rows, gp.dim = dim;
            gp.write_z = !(last && z_is_scratch && xz_out);  // a caller that only consumes x * z_final saves the last z store
            gp.accumulate_ld = f != 0;
            gp.seed = seed, gp.row_offset = row_offset;
            gp.stream = first_noise_stream + (uint32_t)f, gp.next_stream = first_noise_stream + (uint32_t)f + 1;
            rc = rnvpf::launch(y, Wts, gp, st);
            if (rc) return rc;
            continue;
        }
        // [shift | scale] = y [Wt; Ws]^T + bias as a plain GEMM, then the gate as a full-occupancy streaming pass
        // (measured: the same arithmetic inside the GEMM epilogue is latency-bound on its 8 warps, 2.6-3.3 ms
        // per 65536 x 4096 flow against ~1.3 ms this way)
        tc::Epilogue e2{};
        e2.bias = bts, e2.sd_rows = 1, e2.out = ts;
        rc = tc::launch(y, Wts, (int)n_rows, 2 * dim, tc::RNVP_HP, e2, st);
        if (rc) return rc;
        const long long blocks = n_rows < 148 * 16 ? n_rows : 148 * 16;
        tc::rnvp_gate_kernel<<<(unsigned)blocks, 256, 0, st>>>(
            ts, z, log_det, masks_host ? masks_host[f] : nullptr, (!last && masks_host) ? masks_host[f + 1] : nullptr,
            last ? nullptr : mz, x, (int)(x_rows > 0 ? x_rows : 1), (last && xz_out) ? xz_out : nullptr, n_rows, dim, seed,
            first_noise_stream + (uint32_t)f, first_noise_stream + (uint32_t)f + 1, row_offset);
        rc = launch_status("rnvp_gate_kernel");
        if (rc) return rc;
    }
    return 0;
}

int mnf_conv_tc_stage(const float *x, const float *z, const float *W_mean, const float *W_log_var,
                      const float *b_log_var, float *a_mean, float *a_var, float *Bm, float *Bv, float *bvar_p,
                      int64_t n_imgs, int c_in, int height, int width, int c_out, int ksize, int Np, int Kp,
                      void *stream);

int64_t mnf_conv_tc_workspace(int64_t n_imgs, int c_in, int height, int width, int c_out, int ksize) {
    const int OH = height - ksize + 1, OW = width - ksize + 1;
    const int64_t Kp = (c_in * ksize * ksize + 31) / 32 * 32, Np = (c_out + 31) / 32 * 32;
    const int64_t M = n_imgs * OH * OW;
    const int64_t Kp64 = (c_in * ksize * ksize + 63) / 64 * 64;
    if (OW % 4 == 0 && tc::conv_implicit_smem(c_in, height, width, ksize, (int)Kp64, (int)Np) != 0)
        return 2 * M * Np + 2 * Np * Kp64 + Np + 64;  // implicit GEMM: mean, sd, packed weights -- no im2col
    return 2 * M * Kp + M * Np + 2 * Np * Kp + Np + 64;
}

// MNFConv2d.forward + ReLU + MaxPool2d(2) (mnf_conv.py:67-78, mnf_lenet.py:16-21) on the tensor cores:
// im2col (pool-major rows, TF32-rounded x and x^2) -> variance GEMM (sd = sqrt(. + exp(b_log_var))) -> mean GEMM whose
// epilogue adds sd * eps, applies ReLU and the 2x2 max-pool.  out: [n_imgs, c_out, OH/2, OW/2].
int mnf_conv2d_forward_tc(const float *x, const float *z, const float *W_mean, const float *W_log_var,
                          const float *b_log_var, const float *eps, uint64_t seed, uint32_t noise_stream,
                          uint64_t row_offset, float *out, int64_t n_imgs, int c_in, int height, int width, int c_out,
                          int ksize, float *workspace, void *stream) {
    MNF_REQUIRE(z, MNF_E_ARG, "NULL pointer");
    return mnf_conv2d_forward_tc_z(x, z, nullptr, 1, W_mean, W_log_var, b_log_var, eps, seed, noise_stream, row_offset, out,
                                   n_imgs, c_in, height, width, c_out, ksize, workspace, stream);
}

// Same with an optional per-sample z: z_rows [ceil(n_imgs / rows_per_z), c_out], image r uses row r / rows_per_z
// (z must then be NULL: the weights are packed with unit scale and the scale is applied in the noise / pool pass).
int mnf_conv2d_forward_tc_z(const float *x, const float *z, const float *z_rows, int64_t rows_per_z, const float *W_mean,
                            const float *W_log_var, const float *b_log_var, const float *eps, uint64_t seed,
                            uint32_t noise_stream, uint64_t row_offset, float *out, int64_t n_imgs, int c_in, int height,
                            int width, int c_out, int ksize, float *workspace, void *stream) {
    MNF_REQUIRE(x && W_mean && W_log_var && b_log_var && out && workspace, MNF_E_ARG, "NULL pointer");
    MNF_REQUIRE((z != nullptr) != (z_rows != nullptr), MNF_E_ARG, "exactly one of z and z_rows must be given");
    MNF_REQUIRE(rows_per_z >= 1, MNF_E_ARG, "rows_per_z must be positive");
    const int OH = height - ksize + 1, OW = width - ksize + 1;
    MNF_REQUIRE(OH >= 2 && OW >= 2 && OH % 2 == 0 && OW % 2 == 0, MNF_E_SHAPE, "output %dx%d must be even for the pool", OH, OW);
    MNF_REQUIRE(c_out <= tc::MAX_BN, MNF_E_SHAPE, "c_out=%d exceeds one column tile", c_out);
    const int Kp = (c_in * ksize * ksize + 31) / 32 * 32, Np = (c_out + 31) / 32 * 32;
    const long long M = (long long)n_imgs * OH * OW;
    MNF_REQUIRE(n_imgs >= 0 && M <= 0x7fffffff - 256, MNF_E_SHAPE, "too many output pixels for one call (%lld)", M);
    if (n_imgs == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const int Kp64 = (c_in * ksize * ksize + 63) / 64 * 64;
    if (OW % 4 == 0 && tc::conv_implicit_smem(c_in, height, width, ksize, Kp64, Np) != 0) {
        // implicit GEMM: x is read once, the fp16 A / A^2 tiles are generated in shared memory
        float *mean = workspace, *sdp = mean + (size_t)M * Np, *Bm = sdp + (size_t)M * Np, *Bv = Bm + (size_t)Np * Kp64,
              *bvar_p = Bv + (size_t)Np * Kp64;
        int rc = mnf::conv_pack_weights_f16(z, W_mean, W_log_var, b_log_var, Bm, Bv, bvar_p, c_in * ksize * ksize, c_out, Np, Kp64, stream);
        if (rc) return rc;
        rc = tc::launch_conv_implicit(x, Bm, Bv, bvar_p, mean, sdp, n_imgs, c_in, height, width, ksize, Kp64, Np, st);
        if (rc) return rc;
        const long long total = n_imgs * (OH / 2) * (OW / 4) * c_out;
        long long blocks = (total + 255) / 256;
        if (blocks > 148 * 32) blocks = 148 * 32;
        return tc::launch_rows_noise_pool(mean, sdp, eps, seed, noise_stream, row_offset, out, n_imgs, c_out, Np, OH, OW, z_rows,
                                          rows_per_z, total, (unsigned)blocks, st);
    }
    float *a_mean = workspace, *a_var = a_mean + (size_t)M * Kp, *sd = a_var + (size_t)M * Kp, *Bm = sd + (size_t)M * Np,
          *Bv = Bm + (size_t)Np * Kp, *bvar_p = Bv + (size_t)Np * Kp;
    int rc = mnf_conv_tc_stage(x, z, W_mean, W_log_var, b_log_var, a_mean, a_var, Bm, Bv, bvar_p, n_imgs, c_in, height,
                               width, c_out, ksize, Np, Kp, stream);
    if (rc) return rc;
    tc::Epilogue ev{};
    ev.mode = 2, ev.sd_rows = 1, ev.bvar_log = bvar_p, ev.out = sd;
    rc = tc::launch(a_var, Bv, (int)M, Np, Kp, ev, st);
    if (rc) return rc;
    tc::Epilogue em{};
    if (OW % 4 == 0) {
        // plain mean GEMM into the (now dead) x^2 operand buffer, then the full-occupancy noise / ReLU / pool pass
        float *mean = a_var;
        em.mode = 0, em.out = mean;
        rc = tc::launch(a_mean, Bm, (int)M, Np, Kp, em, st);
        if (rc) return rc;
        const long long total = n_imgs * (OH / 2) * (OW / 4) * c_out;
        long long blocks = (total + 255) / 256;
        if (blocks > 148 * 32) blocks = 148 * 32;
        return tc::launch_rows_noise_pool(mean, sd, eps, seed, noise_stream, row_offset, out, n_imgs, c_out, Np, OH, OW, z_rows,
                                          rows_per_z, total, (unsigned)blocks, st);
    }
    MNF_REQUIRE(z_rows == nullptr, MNF_E_SHAPE, "per-sample conv z needs an output width that is a multiple of 4");
    em.mode = 5, em.sd = sd, em.sd_rows = 1, em.eps = eps, em.seed = seed, em.noise_stream = noise_stream;
    em.row_offset = row_offset, em.out = out, em.conv_c = c_out, em.conv_oh = OH, em.conv_ow = OW;
    return tc::launch(a_mean, Bm, (int)M, Np, Kp, em, st);
}

int mnf_tc_eligible(const float *A, const float *W, int64_t M, int N, int K) {
    return tc::eligible(A, W, (int)M, N, K) ? 1 : 0;
}

}  // extern "C"
