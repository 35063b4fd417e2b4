// flow_fast.cuh -- register-resident flow-stack kernel for 2-D points (BASELINE configs 1, 2).
//
// Whole stack in one launch: a thread owns TWO points, keeps both points and their log-dets in
// registers across every flow, and evaluates the coupling conditioners (MLP 1 -> H -> H -> H ->
// n_out, LeakyReLU 0.2) fully unrolled with the weights broadcast from shared memory (staged
// once per CTA; the grid is persistent, a multiple of the SM count).  The two points share every
// weight load; the multiplies use Blackwell's packed FFMA2 (fma.rn.f32x2).  HBM traffic is the
// algorithmic minimum: 8 B in, 8 B out, 4 B log-det per point (+4 B for the fused base
// log-density).
//
// Supported ops (all with dim == 2): AffineConstantFlow/ActNormFlow, Glow, AffineHalfFlow with
// h_sizes (H,H,H), NSF_CL with n_h = H and K bins.  Anything else -> flow_generic.cu.
//
// The MLP is mapped onto the packed FMA by output (variant 2 of MNF_RUN_VARIANT): weights stored transposed ([in][out])
// so one LDS.128 delivers two ready (w_j, w_j+1) operands; the activation is duplicated once per input.
#pragma once
#include "flow_math.cuh"

namespace mnf {

#ifndef MNF_SPLINE_FAST
#define MNF_SPLINE_FAST 1
#endif

// shared-memory offsets (in floats) of each op's nets, computed on the host
struct FastLayout {
    int net_slot[MNF_MAX_OPS][2];
    int total_slots;
};

constexpr int round4(int n) { return (n + 3) / 4 * 4; }

// The kernel does not evaluate layers 0 and 1 of a conditioner as layers: its input is ONE scalar c, so
// W1 leaky(w0 c + b0) + b1 is a piecewise-linear function of c with the H breakpoints -b0_j / w0_j; on each of the H + 1
// intervals it is A_i c + B_i.  The staged net holds the sorted breakpoints and the (A_i | B_i) rows: a point finds its
// interval with H compares and forms the layer-1 pre-activations with H FMAs instead of H + H^2 (RNVP, H = 24: 648 instead
// of 1 224 multiply-adds per conditioner -- and a small-batch call is bound by exactly that dependent chain).
//   staged layout: tb[H] | table[H + 1][pl_stride(H)] | Wt2[in][out] b2[H] | last layer
constexpr int pl_stride(int H) { return 2 * H + 4; }  // padded off the 32-bank period: rows of different intervals do not collide
constexpr int pl_hidden_slots(int H) { return H + (H + 1) * pl_stride(H) + H * H + H; }

// floats one staged net occupies in shared memory
constexpr int fast_net_slots(int H, int n_out) {
    return pl_hidden_slots(H) + (n_out == 1 ? H + 4 : H * round4(n_out) + round4(n_out));
}

__device__ __forceinline__ float2 fma2_packed(float2 a, float2 b, float2 c) {
    unsigned long long ra = *reinterpret_cast<unsigned long long *>(&a);
    unsigned long long rb = *reinterpret_cast<unsigned long long *>(&b);
    unsigned long long rc = *reinterpret_cast<unsigned long long *>(&c);
    unsigned long long rd;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
    return *reinterpret_cast<float2 *>(&rd);
}
__device__ __forceinline__ float2 mul2_packed(float2 a, float2 b) {
    unsigned long long ra = *reinterpret_cast<unsigned long long *>(&a);
    unsigned long long rb = *reinterpret_cast<unsigned long long *>(&b);
    unsigned long long rd;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
    return *reinterpret_cast<float2 *>(&rd);
}

__device__ __forceinline__ float2 leaky2(float2 v) {
    const float2 s = mul2_packed(v, make_float2(0.2f, 0.2f));
    return make_float2(fmaxf(v.x, s.x), fmaxf(v.y, s.y));
}

// weight accessor: offsets are in floats from the start of the staged net
struct WShared {
    const float *p;
    __device__ __forceinline__ float4 ld4(int i) const { return reinterpret_cast<const float4 *>(p)[i >> 2]; }
    __device__ __forceinline__ float ld1(int i) const { return p[i]; }
};

// =====================================================================================
// output-packed engine: float2 = (unit j, unit j+1) of ONE point; two points A, B
// smem net layout: w0[H] b0[H] | Wt1[in][out] b1[H] | Wt2[in][out] b2[H] | Wt3[in][NOP] b3[NOP]
// (n_out == 1: w3[H] b3[4])
// =====================================================================================
template <int H, int NOUT2>
__device__ __forceinline__ void op_dense(const WShared W, int wt_off, int bias_off, const float2 (&inA)[H / 2],
                                         const float2 (&inB)[H / 2], float2 (&outA)[NOUT2],
                                         float2 (&outB)[NOUT2]) {
    // out[j] = bias[j] + sum_i Wt[i][j] * in[i]; NOUT2 pairs of outputs, row stride 2*NOUT2
#pragma unroll
    for (int j = 0; j < NOUT2; j += 2) {
        const float4 b = W.ld4(bias_off + 2 * j);
        outA[j] = outB[j] = make_float2(b.x, b.y);
        if (j + 1 < NOUT2) outA[j + 1] = outB[j + 1] = make_float2(b.z, b.w);
    }
#pragma unroll
    for (int i = 0; i < H; ++i) {
        const float a = (i & 1) ? inA[i >> 1].y : inA[i >> 1].x;
        const float b = (i & 1) ? inB[i >> 1].y : inB[i >> 1].x;
        const float2 aa = make_float2(a, a), bb = make_float2(b, b);
#pragma unroll
        for (int j = 0; j < NOUT2; j += 2) {
            const float4 w = W.ld4(wt_off + i * 2 * NOUT2 + 2 * j);
            outA[j] = fma2_packed(make_float2(w.x, w.y), aa, outA[j]);
            outB[j] = fma2_packed(make_float2(w.x, w.y), bb, outB[j]);
            if (j + 1 < NOUT2) {
                outA[j + 1] = fma2_packed(make_float2(w.z, w.w), aa, outA[j + 1]);
                outB[j + 1] = fma2_packed(make_float2(w.z, w.w), bb, outB[j + 1]);
            }
        }
    }
}

template <int H>
__device__ __forceinline__ void op_hidden(const WShared W, float xA, float xB, float2 (&hA)[H / 2],
                                          float2 (&hB)[H / 2]) {
    static_assert(H % 4 == 0, "hidden width must be a multiple of 4");
    constexpr int TS = pl_stride(H), TBL = H, L2 = H + (H + 1) * TS;
    float2 gA[H / 2], gB[H / 2];
    // layers 0 + 1: interval of each point among the sorted breakpoints, then pre1 = A_i c + B_i
    int ia = 0, ib = 0;
#pragma unroll
    for (int j = 0; j < H; j += 4) {
        const float4 t = W.ld4(j);
        ia += (xA > t.x) + (xA > t.y) + (xA > t.z) + (xA > t.w);
        ib += (xB > t.x) + (xB > t.y) + (xB > t.z) + (xB > t.w);
    }
    const float2 xa = make_float2(xA, xA), xb = make_float2(xB, xB);
    const int ra = TBL + ia * TS, rb = TBL + ib * TS;
#pragma unroll
    for (int j = 0; j < H / 2; j += 2) {
        const float4 aA = W.ld4(ra + 2 * j), bA = W.ld4(ra + H + 2 * j);
        const float4 aB = W.ld4(rb + 2 * j), bB = W.ld4(rb + H + 2 * j);
        gA[j] = leaky2(fma2_packed(make_float2(aA.x, aA.y), xa, make_float2(bA.x, bA.y)));
        gA[j + 1] = leaky2(fma2_packed(make_float2(aA.z, aA.w), xa, make_float2(bA.z, bA.w)));
        gB[j] = leaky2(fma2_packed(make_float2(aB.x, aB.y), xb, make_float2(bB.x, bB.y)));
        gB[j + 1] = leaky2(fma2_packed(make_float2(aB.z, aB.w), xb, make_float2(bB.z, bB.w)));
    }
    op_dense<H, H / 2>(W, L2, L2 + H * H, gA, gB, hA, hB);  // layer 2
#pragma unroll
    for (int j = 0; j < H / 2; ++j) {
        hA[j] = leaky2(hA[j]);
        hB[j] = leaky2(hB[j]);
    }
}

// single output (AffineHalfFlow s / t): dot product packed over input pairs
template <int H>
__device__ __forceinline__ void op_last1(const WShared W, const float2 (&hA)[H / 2], const float2 (&hB)[H / 2],
                                         float &oA, float &oB) {
    const int wo = pl_hidden_slots(H);
    float2 accA = make_float2(0.f, 0.f), accB = make_float2(0.f, 0.f);
#pragma unroll
    for (int i = 0; i < H / 2; i += 2) {
        const float4 w = W.ld4(wo + 2 * i);
        accA = fma2_packed(make_float2(w.x, w.y), hA[i], accA);
        accB = fma2_packed(make_float2(w.x, w.y), hB[i], accB);
        accA = fma2_packed(make_float2(w.z, w.w), hA[i + 1], accA);
        accB = fma2_packed(make_float2(w.z, w.w), hB[i + 1], accB);
    }
    const float b = W.ld1(wo + H);
    oA = (accA.x + accA.y) + b;
    oB = (accB.x + accB.y) + b;
}

// =====================================================================================
// conditioner -> spline for both points
// =====================================================================================
template <int H, int K, bool ONE = false>
__device__ __forceinline__ void spline_half(const float *smem, int slot, const mnf_flow_op &op, float2 cond,
                                            float2 &trans, bool rqs_inverse, float2 &ld) {
    constexpr int NB = 3 * K - 1;
    constexpr bool FAST = MNF_SPLINE_FAST != 0;
    constexpr int NP2 = round4(NB) / 2;
    float2 rA[NP2], rB[NP2];
    {
        const WShared W{smem + slot};
        float2 hA[H / 2], hB[H / 2];
        op_hidden<H>(W, cond.x, cond.y, hA, hB);
        const int wo = pl_hidden_slots(H);
        op_dense<H, NP2>(W, wo, wo + H * 2 * NP2, hA, hB, rA, rB);
    }
#pragma unroll 1
    for (int pt = 0; pt < (ONE ? 1 : 2); ++pt) {
        float raw[NB];
#pragma unroll
        for (int o = 0; o < NB; ++o) {
            const float2 q = pt ? rB[o >> 1] : rA[o >> 1];
            raw[o] = (o & 1) ? q.y : q.x;
        }
        float v = pt ? trans.y : trans.x;
        float l = 0.f;
        rq_spline<K, FAST>(raw, K, op.bound, op.edge_deriv, rqs_inverse, v, l);
        if (pt) { trans.y = v; ld.y += l; } else { trans.x = v; ld.x += l; }
    }
}

// scalar-output conditioner (s or t of AffineHalfFlow) for both points
template <int H>
__device__ __forceinline__ float2 affine_net(const float *smem, int slot, float2 cond) {
    const WShared W{smem + slot};
    float2 hA[H / 2], hB[H / 2];
    op_hidden<H>(W, cond.x, cond.y, hA, hB);
    float2 o;
    op_last1<H>(W, hA, hB, o.x, o.y);
    return o;
}

// stage one net from the parameter blob into shared memory: piecewise-linear table of layers 0 + 1, transposed layer 2,
// last layer (see pl_hidden_slots).  Called by every thread of the CTA (block barriers inside).
template <int H>
__device__ __forceinline__ void stage_net_pl(const float *__restrict__ src, float *dst, int n_out) {
    constexpr int TS = pl_stride(H), TBL = H, L2 = H + (H + 1) * TS, B2 = L2 + H * H, LAST = B2 + H;
    // blob: w0[H] b0[H] | W1[H][H] b1[H] | W2[H][H] b2[H] | W3[n_out][H] b3[n_out]
    const float *w0 = src, *b0 = src + H, *W1 = src + 2 * H, *b1 = W1 + H * H, *W2 = b1 + H, *b2 = W2 + H * H, *W3 = b2 + H,
                *b3 = W3 + n_out * H;
    const int tid = threadIdx.x, nt = blockDim.x;
    for (int j = tid; j < H; j += nt) {  // breakpoint j goes to its rank (ties by index); w0 = 0: no breakpoint (+inf, last)
        const float tj = w0[j] != 0.f ? -b0[j] / w0[j] : INFINITY;
        int rank = 0;
        for (int k = 0; k < H; ++k) {
            const float tk = w0[k] != 0.f ? -b0[k] / w0[k] : INFINITY;
            rank += (tk < tj || (tk == tj && k < j)) ? 1 : 0;
        }
        dst[rank] = tj;
    }
    __syncthreads();
    for (int i = tid; i <= H; i += nt) {  // interval i lies between sorted breakpoints i - 1 and i
        const float lo = i > 0 ? dst[i - 1] : -INFINITY, hi = i < H ? dst[i] : INFINITY;
        float c = 0.f;  // a point inside the interval: fixes the sign of every first-layer pre-activation on it
        if (isfinite(lo) && isfinite(hi)) c = 0.5f * lo + 0.5f * hi;
        else if (isfinite(hi)) c = hi - 1.f - fabsf(hi);
        else if (isfinite(lo)) c = lo + 1.f + fabsf(lo);
        float *row = dst + TBL + i * TS;
        for (int k = 0; k < H; ++k) {
            float A = 0.f, B = b1[k];
            for (int j = 0; j < H; ++j) {
                const float slope = fmaf(w0[j], c, b0[j]) > 0.f ? 1.f : 0.2f;  // LeakyReLU(0.2), mlp.py:9
                const float w = W1[k * H + j] * slope;
                A = fmaf(w, w0[j], A);
                B = fmaf(w, b0[j], B);
            }
            row[k] = A, row[H + k] = B;
        }
        for (int k = 2 * H; k < TS; ++k) row[k] = 0.f;
    }
    for (int e = tid; e < H * H; e += nt) dst[L2 + (e % H) * H + e / H] = W2[e];  // [in][out]
    for (int e = tid; e < H; e += nt) dst[B2 + e] = b2[e];
    if (n_out == 1) {  // w3[H] b3[4]
        for (int e = tid; e < H; e += nt) dst[LAST + e] = W3[e];
        for (int e = tid; e < 4; e += nt) dst[LAST + H + e] = e == 0 ? b3[0] : 0.f;
    } else {  // Wt3[in][NOP] b3[NOP], padding lanes zero
        const int nop = round4(n_out);
        for (int e = tid; e < H * nop; e += nt) {
            const int i = e / nop, o = e % nop;
            dst[LAST + e] = o < n_out ? W3[o * H + i] : 0.f;
        }
        for (int e = tid; e < nop; e += nt) dst[LAST + H * nop + e] = e < n_out ? b3[e] : 0.f;
    }
    __syncthreads();
}

// all nets of a program into shared memory, laid out by `lay`
template <int H>
__device__ __forceinline__ void stage_program(const FlowProgram &prog, const FastLayout &lay,
                                              const float *__restrict__ params, float *image) {
    // padding lanes of the last layers must read zeros
    for (int e = threadIdx.x; e < lay.total_slots; e += blockDim.x) image[e] = 0.f;
    __syncthreads();
    for (int k = 0; k < prog.n_ops; ++k) {
        const mnf_flow_op &op = prog.ops[k];
        if (op.type != MNF_OP_AFFINE_HALF && op.type != MNF_OP_NSF_CL) continue;
        for (int which = 0; which < 2; ++which) {
            if (op.type == MNF_OP_AFFINE_HALF && !(op.flags & (which ? MNF_FLAG_SHIFT : MNF_FLAG_SCALE))) continue;
            stage_net_pl<H>(params + op.net_off[which], image + lay.net_slot[k][which], op.sizes[op.n_lin]);
        }
    }
}

// everything that happens to one pair of points: load, all flows, store.
// ONE: small-batch mode -- `pair` is a POINT index, the B lane of every float2 is a dead copy that the compiler removes
// (nothing is stored from it), so a thread walks half the dependent FFMA2 chain and twice as many warps share the work.
template <int H, int K, bool ONE = false>
__device__ __forceinline__ void process_pair(const FlowProgram &prog, const FastLayout &lay,
                                             const float *__restrict__ params, const float *smem,
                                             const float *__restrict__ x, float *__restrict__ y,
                                             float *__restrict__ log_det, float *__restrict__ base_lp,
                                             float *__restrict__ inter, long long n_rows, int inverse, bool sum_lp,
                                             long long pair, bool live) {
    const bool has_b = ONE ? false : 2 * pair + 1 < n_rows;
    const long long first_pt = ONE ? pair : 2 * pair;  // index of point A
    float2 v0, v1;  // v0 = first coordinate of points (A, B), v1 = second coordinate
    if (has_b) {
        const float4 q = ld_stream4(reinterpret_cast<const float4 *>(x) + pair);
        v0 = make_float2(q.x, q.z);
        v1 = make_float2(q.y, q.w);
    } else {
        const float2 q = ld_stream2(reinterpret_cast<const float2 *>(x) + first_pt);
        v0 = make_float2(q.x, q.x);
        v1 = make_float2(q.y, q.y);
    }
    float2 ld = make_float2(0.f, 0.f);

#pragma unroll 1
    for (int kk = 0; kk < prog.n_ops; ++kk) {
        const int k = inverse ? prog.n_ops - 1 - kk : kk;
        const mnf_flow_op &op = prog.ops[k];
        if (op.type == MNF_OP_AFFINE_CONST) {
            const float s0 = params[op.aux_off], s1 = params[op.aux_off + 1];
            const float t0 = params[op.aux_off + 2], t1 = params[op.aux_off + 3];
            if (inverse) {  // affine_constant_flow.py:24
                const float e0 = expf(-s0), e1 = expf(-s1);
                v0 = make_float2((v0.x - t0) * e0, (v0.y - t0) * e0);
                v1 = make_float2((v1.x - t1) * e1, (v1.y - t1) * e1);
                ld.x -= s0 + s1;
                ld.y -= s0 + s1;
            } else {  // affine_constant_flow.py:19
                const float e0 = expf(s0), e1 = expf(s1);
                v0 = make_float2(v0.x * e0 + t0, v0.y * e0 + t0);
                v1 = make_float2(v1.x * e1 + t1, v1.y * e1 + t1);
                ld.x += s0 + s1;
                ld.y += s0 + s1;
            }
        } else if (op.type == MNF_OP_GLOW) {
            const float *W = params + op.aux_off + (inverse ? 4 : 0);  // glow.py:28,36: v @ W
            const float w00 = W[0], w01 = W[1], w10 = W[2], w11 = W[3];
            const float lg = params[op.aux_off + 8];
            const float2 n0 = make_float2(fmaf(v1.x, w10, v0.x * w00), fmaf(v1.y, w10, v0.y * w00));
            const float2 n1 = make_float2(fmaf(v1.x, w11, v0.x * w01), fmaf(v1.y, w11, v0.y * w01));
            v0 = n0;
            v1 = n1;
            ld.x += inverse ? -lg : lg;
            ld.y += inverse ? -lg : lg;
        } else if (op.type == MNF_OP_AFFINE_HALF) {
            const bool parity = op.flags & MNF_FLAG_PARITY;
            const float2 cond = parity ? v1 : v0;  // affine_half_flow.py:46-50
            float2 tr = parity ? v0 : v1;
            float2 st[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
#pragma unroll 1
            for (int which = 0; which < 2; ++which) {
                if (!(op.flags & (which ? MNF_FLAG_SHIFT : MNF_FLAG_SCALE))) continue;
                const float2 o = affine_net<H>(smem, lay.net_slot[k][which], cond);
                if (which) st[1] = o; else st[0] = o;
            }
            const float2 s = st[0], t = st[1];
            if (inverse) {  // affine_half_flow.py:54-56
                tr = make_float2((tr.x - t.x) / expf(s.x), (tr.y - t.y) / expf(s.y));
                ld.x -= s.x;
                ld.y -= s.y;
            } else {  // affine_half_flow.py:58
                tr = make_float2(expf(s.x) * tr.x + t.x, expf(s.y) * tr.y + t.y);
                ld.x += s.x;
                ld.y += s.y;
            }
            if (parity) v0 = tr; else v1 = tr;
        } else if (op.type == MNF_OP_NSF_CL) {
            // forward: f1 on (lower -> upper) then f2 on (upper -> lower) (spline_flow.py:249-266);
            // inverse: f2 first, then f1, both with the spline inverse (spline_flow.py:268-285).
            // One call site, two trips: keeps the unrolled body in the instruction cache.
#pragma unroll 1
            for (int step = 0; step < 2; ++step) {
                const bool use_f1 = (step == 0) != (inverse != 0);
                const float2 cond = use_f1 ? v0 : v1;
                float2 tr = use_f1 ? v1 : v0;
                spline_half<H, K, ONE>(smem, lay.net_slot[k][use_f1 ? 0 : 1], op, cond, tr, inverse != 0, ld);
                if (use_f1) v1 = tr; else v0 = tr;
            }
        }
        if (inter && live) {
            float *dst = inter + ((size_t)kk * n_rows + first_pt) * 2;
            if (has_b)
                st_stream4(reinterpret_cast<float4 *>(dst), make_float4(v0.x, v1.x, v0.y, v1.y));
            else
                st_stream2(reinterpret_cast<float2 *>(dst), make_float2(v0.x, v1.x));
        }
    }

    const float c = -1.8378770664093453f;  // -(D/2) log(2 pi), D = 2
    float2 lp = make_float2(fmaf(-0.5f, fmaf(v0.x, v0.x, v1.x * v1.x), c),
                            fmaf(-0.5f, fmaf(v0.y, v0.y, v1.y * v1.y), c));
    if (sum_lp) lp = make_float2(lp.x + ld.x, lp.y + ld.y);
    if (!live) return;
    if (has_b) {
        if (y) st_stream4(reinterpret_cast<float4 *>(y) + pair, make_float4(v0.x, v1.x, v0.y, v1.y));
        if (log_det) st_stream2(reinterpret_cast<float2 *>(log_det) + pair, ld);
        if (base_lp) st_stream2(reinterpret_cast<float2 *>(base_lp) + pair, lp);
    } else {
        if (y) st_stream2(reinterpret_cast<float2 *>(y) + first_pt, make_float2(v0.x, v1.x));
        if (log_det) log_det[first_pt] = ld.x;
        if (base_lp) base_lp[first_pt] = lp.x;
    }
}

template <int H, int K, bool ONE = false>
__global__ void __launch_bounds__(128, 4)
flow_fast_kernel(const __grid_constant__ FlowProgram prog, const __grid_constant__ FastLayout lay,
                 const float *__restrict__ params, const float *__restrict__ x, float *__restrict__ y,
                 float *__restrict__ log_det, float *__restrict__ base_lp, float *__restrict__ inter,
                 long long n_rows, int dir_flags) {
    extern __shared__ __align__(16) float smem[];
    const int inverse = dir_flags & 1;
    const bool sum_lp = dir_flags & 2;
    stage_program<H>(prog, lay, params, smem);
    __syncthreads();

    const long long n_pairs = ONE ? n_rows : (n_rows + 1) >> 1;
    const long long first = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    // persistent grid-stride loop: the nets are staged once per CTA
    for (long long pair = first; pair < n_pairs; pair += (long long)gridDim.x * blockDim.x)
        process_pair<H, K, ONE>(prog, lay, params, smem, x, y, log_det, base_lp, inter, n_rows, inverse, sum_lp, pair,
                                true);
}

// batches below this many points take the one-point-per-thread form (latency, not throughput, matters)
constexpr long long kOnePointMaxRows = 148LL * 128;

template <int H, int K, bool ONE = false>
int launch_inst(const FlowProgram &prog, const FastLayout &lay, size_t smem_bytes, const float *params,
                const float *x, float *y, float *log_det, float *base_lp, float *inter, int64_t n_rows,
                int inverse, const DeviceProps *dp, cudaStream_t stream) {
    if constexpr (!ONE) {
        if (n_rows <= kOnePointMaxRows)
            return launch_inst<H, K, true>(prog, lay, smem_bytes, params, x, y, log_det, base_lp, inter, n_rows, inverse, dp,
                                           stream);
    }
    auto kern = flow_fast_kernel<H, K, ONE>;
    static thread_local int occ_cache = -1;
    static thread_local size_t occ_smem = 0;
    if (occ_cache < 0 || occ_smem != smem_bytes) {
        if (smem_bytes > 48 * 1024)
            MNF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
        int occ = 0;
        MNF_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, 128, smem_bytes));
        if (occ < 1) return fail(MNF_E_SHAPE, "flow_fast_kernel does not fit on an SM (smem %zu B)", smem_bytes);
        occ_cache = occ;
        occ_smem = smem_bytes;
    }
    const long long n_pairs = ONE ? n_rows : (n_rows + 1) / 2;
    const int threads = 128;  // measured on config 1: CTAs of 32 / 64 threads lose more to the per-CTA staging of the nets
                              // (128 / 80 us per call) than they gain from spreading the points over more SMs (63 us)
    long long blocks = (n_pairs + threads - 1) / threads;
    const long long cap = (long long)dp->sm_count * occ_cache;  // persistent: one wave, a multiple of the SM count
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    kern<<<(unsigned)blocks, threads, smem_bytes, stream>>>(prog, lay, params, x, y, log_det, base_lp, inter, n_rows,
                                                            inverse & 3);
    return launch_status("flow_fast_kernel");
}

#define MNF_FLOW_FAST_ARGS                                                                                            \
    const FlowProgram &prog, const FastLayout &lay, size_t smem_bytes, const float *params, const float *x, float *y, \
        float *log_det, float *base_lp, float *inter, int64_t n_rows, int inverse, const DeviceProps *dp,             \
        cudaStream_t stream

#define MNF_FLOW_FAST_DEFINE(HH, KK)                                                                                  \
    int launch_fast_##HH##_##KK(MNF_FLOW_FAST_ARGS) {                                                                 \
        return launch_inst<HH, KK>(prog, lay, smem_bytes, params, x, y, log_det, base_lp, inter, n_rows, inverse, dp, \
                                   stream);                                                                           \
    }

}  // namespace mnf
