// flow_math.cuh -- per-point device math shared by the generic flow interpreter and the
// D=2 table kernel: LeakyReLU, softplus, and the rational-quadratic spline of
// NSF_CL / NSF_AR with the reference's exact parameterisation quirks
// (spline_flow.py:29-179, SURVEY.md section 8a row a10):
//   * the raw conditioner outputs are softmax'ed and scaled by 2B in NSF_* (:253-256) and
//     softmax'ed AGAIN inside RQS (:95, :106); raw derivatives get softplus twice (:256, :104)
//   * min bin width / height / derivative 1e-3 (:17-19), knots pinned to +-B (:100-101)
//   * bin search = count(v >= knot) - 1 with 1e-6 added to the last knot (:22-24)
//   * outside [-B, B] (inclusive bounds, :40): identity, log-det 0 (:51-52)
#pragma once
#include "common.cuh"

namespace mnf {

// a flow stack as it travels to the kernels: descriptors by value (__grid_constant__), parameters in a device blob
struct FlowProgram {
    int n_ops;
    mnf_flow_op ops[MNF_MAX_OPS];
};

constexpr float kMinBin = 1e-3f;    // spline_flow.py:17-18
constexpr float kMinDeriv = 1e-3f;  // spline_flow.py:19

__device__ __forceinline__ float leaky02(float x) { return fmaxf(x, 0.2f * x); }  // LeakyReLU(0.2), mlp.py:9

// F.softplus(beta=1, threshold=20)
__device__ __forceinline__ float softplus(float x) { return x > 20.f ? x : log1pf(expf(x)); }

// Math flavour.  FAST = false: libdevice expf/logf/log1pf and IEEE division (generic
// interpreter).  FAST = true (table kernel): MUFU-based forms whose error stays
// ~1e-6 relative on the ranges that occur here, an order below the 1e-5 parity tolerance:
//   exp(x)      -> ex2.approx(x*log2e)      x <= 0 after max subtraction, |x| <= 2B where it matters
//   a / b       -> a * rcp.approx(b)        (__fdividef, 2 ulp)
//   log(n)-2log(d) -> lg2.approx(n * rcp(d)^2) * ln2   (one MUFU.LG2 instead of two)
//   softplus(softplus(r)) -> log(2 + exp(r))           (exact identity below the threshold 20)
template <bool FAST>
__device__ __forceinline__ float sm_exp(float x) {
    if constexpr (FAST) {
        float r;
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x * 1.4426950408889634f));
        return r;
    } else {
        return expf(x);
    }
}
template <bool FAST>
__device__ __forceinline__ float fdiv(float a, float b) {
    if constexpr (FAST) return __fdividef(a, b);
    else return a / b;
}
template <bool FAST>
__device__ __forceinline__ float frcp(float a) {
    if constexpr (FAST) {
        float r;
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(a));
        return r;
    } else {
        return 1.f / a;
    }
}
// interior knot derivative: min_d + softplus(softplus(raw)) (spline_flow.py:256,104)
template <bool FAST>
__device__ __forceinline__ float knot_derivative(float r) {
    if constexpr (FAST) return kMinDeriv + (r > 20.f ? r : __logf(2.f + __expf(r)));
    else return kMinDeriv + softplus(softplus(r));
}

// knots[0..K] of one axis from K raw conditioner outputs: both softmaxes, floor, cumsum, pin.
// KC > 0: compile-time K (registers); KC == 0: runtime K (local memory).
template <int KC, bool FAST>
__device__ __forceinline__ void spline_knots(const float *raw, int K, float B, float *knots) {
    constexpr int KA = KC > 0 ? KC : MNF_MAX_BINS;
    const int Kn = KC > 0 ? KC : K;
    float e[KA];
    float m = raw[0];
#pragma unroll
    for (int k = 1; k < Kn; ++k) m = fmaxf(m, raw[k]);
    const float twoB = 2.f * B;
    const float span = 1.f - kMinBin * (float)Kn;
    if constexpr (FAST) {
        // Same formulas with the constant factors folded (the kernels using this path are instruction-issue bound):
        //   first softmax   e_k = 2^((raw_k - m) log2 e)                      one FFMA + MUFU.EX2 per bin
        //   second softmax  f_k = exp(2B e_k / sum)  (its arguments lie in [0, 2B]: no maximum needs subtracting while
        //                   exp(2B) is representable, B <= 40)                one FMUL + MUFU.EX2 per bin
        //   knots           x_{k+1} = x_k + 2B min_bin + (2B span / sum f) f_k   one FFMA + FADD per bin
        constexpr float LOG2E = 1.4426950408889634f;
        const float mneg = -m * LOG2E;
        float sum = 0.f;
#pragma unroll
        for (int k = 0; k < Kn; ++k) {
            asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e[k]) : "f"(fmaf(raw[k], LOG2E, mneg)));
            sum += e[k];
        }
        const float inv = frcp<true>(sum);
        const bool big = twoB > 80.f;           // uniform across the launch
        const float sc = twoB * inv * LOG2E;     // first softmax scaled by 2B (spline_flow.py:254-255), in log2 units
        const float off = big ? -sc : 0.f;       // its maximum element is e = 1
        float sum2 = 0.f;
#pragma unroll
        for (int k = 0; k < Kn; ++k) {
            asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e[k]) : "f"(fmaf(e[k], sc, off)));  // second softmax (spline_flow.py:95)
            sum2 += e[k];
        }
        const float c1 = twoB * span * frcp<true>(sum2), c0 = twoB * kMinBin;  // spline_flow.py:96-99
        float x = -B;
        knots[0] = -B;
#pragma unroll
        for (int k = 0; k < Kn; ++k) {
            x += fmaf(e[k], c1, c0);
            knots[k + 1] = x;
        }
        knots[Kn] = B;  // spline_flow.py:101
        return;
    }
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < Kn; ++k) {
        e[k] = sm_exp<FAST>(raw[k] - m);
        sum += e[k];
    }
    // first softmax scaled by 2B (spline_flow.py:254-255); its maximum element is 2B/sum
    const float inv = frcp<FAST>(sum);
    const float m2 = twoB * inv;  // e == 1 at the arg-max
    float sum2 = 0.f;
#pragma unroll
    for (int k = 0; k < Kn; ++k) {
        const float w = twoB * (e[k] * inv);
        e[k] = sm_exp<FAST>(w - m2);  // second softmax (spline_flow.py:95)
        sum2 += e[k];
    }
    const float inv2 = frcp<FAST>(sum2);
    float cum = 0.f;
    knots[0] = -B;
#pragma unroll
    for (int k = 0; k < Kn; ++k) {
        cum += kMinBin + span * (e[k] * inv2);  // spline_flow.py:96-97
        knots[k + 1] = twoB * cum + (-B);      // spline_flow.py:99
    }
    knots[Kn] = B;  // spline_flow.py:101
}

// One spline evaluation.  raw = [K widths | K heights | K-1 derivatives] as produced by the
// conditioner.  Updates v in place and ADDS the log|det| contribution to ld.
template <int KC, bool FAST = false>
__device__ __forceinline__ void rq_spline(const float *raw, int K, float B, float edge_deriv, bool inverse,
                                          float &v, float &ld) {
    constexpr int KA = KC > 0 ? KC : MNF_MAX_BINS;
    const int Kn = KC > 0 ? KC : K;
    if (!(v >= -B && v <= B)) return;  // identity tails (also NaN), spline_flow.py:40,51-52

    float cw[KA + 1], ch[KA + 1];
    spline_knots<KC, FAST>(raw, Kn, B, cw);
    spline_knots<KC, FAST>(raw + Kn, Kn, B, ch);

    // bin search (spline_flow.py:22-24,115-118)
    const float *sk = inverse ? ch : cw;
    int idx = -1;
#pragma unroll
    for (int k = 0; k < Kn; ++k) idx += (v >= sk[k]) ? 1 : 0;
    idx += (v >= sk[Kn] + 1e-6f) ? 1 : 0;
    idx = min(max(idx, 0), Kn - 1);

    float xk = 0.f, xk1 = 0.f, yk = 0.f, yk1 = 0.f, r0 = 0.f, r1 = 0.f;
#pragma unroll
    for (int k = 0; k < Kn; ++k) {
        if (k == idx) {
            xk = cw[k];
            xk1 = cw[k + 1];
            yk = ch[k];
            yk1 = ch[k + 1];
            r0 = (k > 0) ? raw[2 * Kn + k - 1] : 0.f;
            r1 = (k < Kn - 1) ? raw[2 * Kn + k] : 0.f;
        }
    }
    const float wk = xk1 - xk;  // spline_flow.py:102
    const float hk = yk1 - yk;  // spline_flow.py:113
    // interior derivatives: min_d + softplus(softplus(raw)) (spline_flow.py:256,104); the two
    // boundary derivatives are the padded constant (:46-49)
    const float dk = (idx > 0) ? knot_derivative<FAST>(r0) : edge_deriv;
    const float dk1 = (idx < Kn - 1) ? knot_derivative<FAST>(r1) : edge_deriv;
    const float sk_ = fdiv<FAST>(hk, wk);  // delta, spline_flow.py:123
    const float dsum = dk + dk1 - 2.f * sk_;

    if (inverse) {  // spline_flow.py:133-162
        const float dy = v - yk;
        const float a = dy * dsum + hk * (sk_ - dk);
        const float b = hk * dk - dy * dsum;
        const float c = -sk_ * dy;
        const float disc = fmaxf(b * b - 4.f * a * c, 0.f);
        const float root = fdiv<FAST>(2.f * c, -b - sqrtf(disc));
        v = root * wk + xk;
        const float tt = root * (1.f - root);
        const float den = sk_ + dsum * tt;
        const float omr = 1.f - root;
        const float num = (sk_ * sk_) * (dk1 * (root * root) + 2.f * sk_ * tt + dk * (omr * omr));
        if constexpr (FAST) {
            const float rd = frcp<true>(den);
            ld -= __logf(num * rd * rd);
        } else {
            ld -= logf(num) - 2.f * logf(den);
        }
    } else {  // spline_flow.py:163-179
        const float th = fdiv<FAST>(v - xk, wk);
        const float tt = th * (1.f - th);
        const float numer = hk * (sk_ * (th * th) + dk * tt);
        const float den = sk_ + dsum * tt;
        const float omt = 1.f - th;
        const float num = (sk_ * sk_) * (dk1 * (th * th) + 2.f * sk_ * tt + dk * (omt * omt));
        if constexpr (FAST) {
            const float rd = frcp<true>(den);
            v = fmaf(numer, rd, yk);
            ld += __logf(num * rd * rd);
        } else {
            v = yk + numer / den;
            ld += logf(num) - 2.f * logf(den);
        }
    }
}

}  // namespace mnf
