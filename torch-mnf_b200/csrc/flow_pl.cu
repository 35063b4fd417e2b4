// flow_pl.cu -- dim-2 coupling stacks (BASELINE configs 1 and 2) with every conditioner evaluated as what it is: a
// PIECEWISE-LINEAR function of ONE scalar.
//
// In two dimensions the conditioner of AffineHalfFlow (affine_half_flow.py:46-50) and of NSF_CL (spline_flow.py:249-257)
// sees a single coordinate c, and an MLP of Linear / LeakyReLU layers (mlp.py:4-12) is piecewise linear in its input:
// along the real line it has a finite list of breakpoints (the zero crossings of every hidden pre-activation; about one
// per hidden unit in practice: ~50 for 1-16-16-16-23, ~70 for 1-24-24-24-1) and between two breakpoints EVERY output is
// A c + B.  So the whole net -- not only its first two layers, as earlier dim-2 kernels had it -- is a table:
//
//   flow_pl_build_kernel   one CTA per conditioner (an AffineHalfFlow's s- and t-net share their input and one table): finds
//                          the breakpoints layer by layer in fp64 (on every current piece each pre-activation is affine, so
//                          it has at most one zero there), sorts them, and writes per piece the slope and the value at the
//                          piece's origin of every output.  Exact up to fp64 rounding -- closer to the real-number net than
//                          an fp32 evaluation of its layers.
//   flow_pl_kernel<K, INV[, DRAW]>
//                          one thread per point, the whole stack in one launch: a conditioner is a branch-free binary
//                          search over <= 511 sorted breakpoints in shared memory and one FMA per output
//                          (out = V_i + A_i (c - origin_i)); the spline (flow_math.cuh) then runs on the raw outputs, and only
//                          the two knot derivatives of the bin the point falls into are ever formed.  Tables with a fast form
//                          (written by the builder next to the plain one) are looked up through a bucket index instead, and
//                          their spline outputs come pre-shifted for the softmax.  DRAW (forward direction only): the
//                          point's z is drawn from Philox in place of being loaded, and log q(x) = log N(z) - log-det
//                          comes out of the same pass (mnf_flow_stack_sample).
//
// Per point and conditioner: ~60 instructions instead of 5 376 multiply-adds (or three MMA round trips).  No tensor core
// and no FMA chain is left to feed: what remains is the spline arithmetic and 12 B/pt of HBM traffic.
// A table with more than 511 breakpoints (e.g. a pair of 1-64-64-64-64-64-1 nets; the bound is pieces x width per layer) is flagged by the
// builder and evaluated layer by layer in fp32 by the threads that need it.  The library owns no device memory: the
// tables live in the caller's workspace (built per call) or in the image of mnf_flow_stack_stage (built per parameter
// version).
#include "flow_math.cuh"
#include "mnf_common.cuh"
#include "tc_common.cuh"

namespace mnf {
namespace fpl {
using tc::smem_u32; using tc::mbar_init; using tc::mbar_arrive; using tc::mbar_wait; using tc::bulk_load;

constexpr int PMAX = 511;       // breakpoints per table
constexpr int BP_FLOATS = 512;  // sorted breakpoints, padded with +inf (search array)
constexpr int MAX_GROUPS = 2 * MNF_MAX_OPS;
constexpr int HDR_INTS = 4;     // per table: breakpoints, overflow flag, fast form's offset and size (floats; 0 = none)
constexpr int HDR_FLOATS = MAX_GROUPS * HDR_INTS;
constexpr int MAX_H = 64;       // hidden width the in-kernel fp32 fallback holds
// Fast form of a table (see the builder): spline rows shifted so that every exponent is <= FAST_T (log2 units), a bucket
// index in place of the binary search.  Only for spline bounds up to FAST_B_MAX: the two second-softmax sums of a point,
// each in [e^-B, K e^B], are then inverted by one reciprocal of their product without leaving the normal fp32 range.
constexpr double FAST_T = 32.0;
constexpr float FAST_B_MAX = 32.f;
constexpr int NB_MIN = 64, NB_MAX = 2048;  // buckets (powers of two)
constexpr int SMEM_TABLE_FLOATS = 216 * 1024 / 4;  // shared memory the point kernel gives the tables of a program
constexpr double LOG2E_D = 1.4426950408889634;

__host__ __device__ constexpr int round4i(int n) { return (n + 3) / 4 * 4; }
// NSF_CL row: K float4 (A_2j, A_2j+1, V_2j, V_2j+1) for the 2K width / height outputs | K - 1 float2 (A, V) of the knot
// derivatives | origin.  AffineHalfFlow row: (A_s, A_t, V_s, V_t) | origin.  Strides are an odd number of float4 so that
// rows of different pieces spread over the banks.
__host__ __device__ constexpr int nsf_doff(int K) { return 4 * K; }
__host__ __device__ constexpr int nsf_org(int K) { return 4 * K + round4i(2 * (K - 1)); }
__host__ __device__ constexpr int nsf_stride4(int K) { return (nsf_org(K) / 4 + 1) | 1; }
constexpr int AFF_ORG = 4, AFF_STRIDE4 = 3;
__host__ __device__ constexpr int region_floats(int stride4) { return BP_FLOATS + (PMAX + 1) * 4 * stride4; }

struct GroupList {
    int n;
    int region[MAX_GROUPS];            // float offset of the table in the image
    unsigned char op[MAX_GROUPS];      // flow it belongs to
    unsigned char which[MAX_GROUPS];   // NSF_CL: 0 = f1, 1 = f2
    signed char group_of[MNF_MAX_OPS][2];
};

// Bucket of c in the fast form's grid (lo, inv, NB - 1): clamp((c - lo) inv) rounded down, NaN to bucket 0.  Monotone
// non-decreasing in c, and the builder files every breakpoint with this same function, so the breakpoints below c are
// those of the buckets before c's plus those of c's own bucket that are < c -- whatever the rounding of the grid.  The
// float-to-int conversion is an add in round-to-zero mode (FMA pipe) instead of F2I (XU pipe).
__device__ __forceinline__ int bucket_of(float c, float lo, float inv, float nbm1) {
    const float t = fminf(fmaxf((c - lo) * inv, 0.f), nbm1);
    return __float_as_int(__fadd_rz(t, 8388608.f)) & 0x7fffff;
}

// ---------------------------------------------------------------------------------------------------------
// builder
// ---------------------------------------------------------------------------------------------------------
constexpr int BW = 8;  // warps per builder CTA

// Of the K outputs o0 .. o0 + K - 1 (affine maps A c + B on the piece (lo, hi)), the one that is maximal at the piece's
// midpoint, or on an unbounded piece the one that is maximal far out (extreme slope, then larger value): a supporting
// line of the outputs' upper envelope on the piece.
__device__ int envelope_line(const double *A, const double *B, int o0, int K, double lo, double hi) {
    int l = o0;
    if (lo == -INFINITY || hi == INFINITY) {
        const double sg = lo == -INFINITY ? -1.0 : 1.0;
        for (int k = o0 + 1; k < o0 + K; ++k)
            if (sg * A[k] > sg * A[l] || (A[k] == A[l] && B[k] > B[l])) l = k;
    } else {
        const double m = 0.5 * lo + 0.5 * hi;
        for (int k = o0 + 1; k < o0 + K; ++k)
            if (fma(A[k], m, B[k]) > fma(A[l], m, B[l])) l = k;
    }
    return l;
}

// largest distance at e, over both spline axes, between the envelope of the outputs and the line envelope_line picks on (lo, hi)
__device__ double envelope_gap(const double *A, const double *B, int K, double lo, double hi, double e) {
    double g = 0.0;
    for (int o0 = 0; o0 < 2 * K; o0 += K) {
        const int l = envelope_line(A, B, o0, K, lo, hi);
        const double vl = fma(A[l], e, B[l]);
        for (int k = o0; k < o0 + K; ++k) g = fmax(g, fma(A[k], e, B[k]) - vl);
    }
    return g;
}

// One thread: split points (fp32 values, strictly inside (lo, hi)) that cut the piece into pieces on which the gap of
// envelope_gap stays <= FAST_T / log2(e) at both ends, hence everywhere (the gap is convex).  An unbounded piece first gets
// one cut beyond which its extreme line is within the bound, the bounded rest is halved as often as needed.  false: no
// such cutting within the split budget (the table then gets no fast form).
__device__ bool split_piece(const double *A, const double *B, int K, double lo, double hi, double *out, int *cnt) {
    const double TN = FAST_T / LOG2E_D;
    auto emit = [&](double s) {
        const int p = atomicAdd(cnt, 1);
        if (p < PMAX) out[p] = s;
        return p < PMAX;
    };
    double seg[2][2] = {{lo, hi}, {0.0, 0.0}};
    int nseg = 1;
    if (lo == -INFINITY && hi == INFINITY) {
        if (!emit(0.0)) return false;
        seg[0][1] = 0.0, seg[1][0] = 0.0, seg[1][1] = INFINITY, nseg = 2;
    }
    for (int q = 0; q < nseg; ++q) {
        double a = seg[q][0], b = seg[q][1];
        const bool left = a == -INFINITY, right = b == INFINITY;
        if (left || right) {
            const double e = left ? b : a;
            if (envelope_gap(A, B, K, a, b, e) <= TN) continue;
            double w = fmax(1.0, fabs(e)), s;
            for (;;) {
                s = (double)(float)(left ? e - w : e + w);
                if (fabs(s) > 1.0e38) return false;
                if (envelope_gap(A, B, K, left ? -INFINITY : s, left ? s : INFINITY, s) <= TN) break;
                w *= 2.0;
            }
            if (!emit(s)) return false;
            a = left ? s : e, b = left ? e : s;
        }
        double st[64][2];
        int sp = 0;
        st[sp][0] = a, st[sp][1] = b, ++sp;
        while (sp) {
            --sp;
            const double x0 = st[sp][0], x1 = st[sp][1];
            if (envelope_gap(A, B, K, x0, x1, x0) <= TN && envelope_gap(A, B, K, x0, x1, x1) <= TN) continue;
            const double s = (double)(float)(0.5 * x0 + 0.5 * x1);
            if (!(s > x0 && s < x1) || sp + 2 > 64 || !emit(s)) return false;
            st[sp][0] = s, st[sp][1] = x1, ++sp;
            st[sp][0] = x0, st[sp][1] = s, ++sp;
        }
    }
    return true;
}

// a point strictly inside piece i of the n sorted breakpoints (fixes the sign of every pre-activation on the piece)
__device__ __forceinline__ double piece_point(const double *bp, int n, int i, double &lo, double &hi) {
    lo = i > 0 ? bp[i - 1] : -INFINITY;
    hi = i < n ? bp[i] : INFINITY;
    if (n == 0) return 0.0;
    if (i == 0) return hi - 1.0 - fabs(hi);
    if (i == n) return lo + 1.0 + fabs(lo);
    return 0.5 * lo + 0.5 * hi;
}

// One warp: affine maps (a c + b) of the pre-activations of Linear layer `upto` (0-based) of a net on the piece that
// contains m.  Two ping-pong vectors per warp; returns the index of the one holding the result.
__device__ int net_pre_maps(const float *__restrict__ net, const int *sizes, int upto, double m, double (*va)[MNF_MAX_HIDDEN],
                            double (*vb)[MNF_MAX_HIDDEN], int lane) {
    const double slope_neg = (double)0.2f;  // LeakyReLU(0.2) on fp32 tensors (mlp.py:9)
    int cur = 0;
    if (lane == 0) va[0][0] = 1.0, vb[0][0] = 0.0;  // layer input: c itself
    __syncwarp();
    const float *p = net;
    for (int t = 0; t <= upto; ++t) {
        const int n_in = sizes[t], n_out = sizes[t + 1];
        const float *bias = p + n_in * n_out;
        for (int k = lane; k < n_out; k += 32) {
            double A = 0.0, B = (double)bias[k];
            const float *w = p + (size_t)k * n_in;
            for (int j = 0; j < n_in; ++j) {
                const double wj = (double)w[j];
                A = fma(wj, va[cur][j], A);
                B = fma(wj, vb[cur][j], B);
            }
            if (t < upto) {  // LeakyReLU with the sign the pre-activation has on this piece
                const double s = fma(A, m, B) > 0.0 ? 1.0 : slope_neg;
                A *= s, B *= s;
            }
            va[cur ^ 1][k] = A, vb[cur ^ 1][k] = B;
        }
        __syncwarp();
        cur ^= 1;
        p += n_in * n_out + n_out;
    }
    return cur;
}

__global__ void __launch_bounds__(32 * BW) flow_pl_build_kernel(const __grid_constant__ FlowProgram prog, const __grid_constant__ GroupList gl,
                                                                const float *__restrict__ params, float *__restrict__ image) {
    __shared__ double s_bp[512], s_tmp[512];
    __shared__ double s_va[BW][2][MNF_MAX_HIDDEN], s_vb[BW][2][MNF_MAX_HIDDEN];
    __shared__ int s_bidx[PMAX];
    __shared__ int s_n, s_ncand, s_fail;
    const int g = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nt = blockDim.x;
    auto sort_bp = [&](int tot) {  // s_bp[0 .. tot) in ascending order (rank sort, ties by index)
        for (int e = tid; e < tot; e += nt) {
            const double v = s_bp[e];
            int r = 0;
            for (int u = 0; u < tot; ++u) r += (s_bp[u] < v || (s_bp[u] == v && u < e)) ? 1 : 0;
            s_tmp[r] = v;
        }
        __syncthreads();
        for (int e = tid; e < tot; e += nt) s_bp[e] = s_tmp[e];
        __syncthreads();
    };
    const mnf_flow_op &op = prog.ops[gl.op[g]];
    const bool nsf = op.type == MNF_OP_NSF_CL;
    const int K = op.K, L = op.n_lin, n_out = op.sizes[L];
    int n_nets = 0, net_off[2], net_slot[2];
    if (nsf) {
        net_off[0] = op.net_off[gl.which[g]], net_slot[0] = 0, n_nets = 1;
    } else {  // AffineHalfFlow: s_net and t_net read the same coordinate (affine_half_flow.py:49-50)
        if (op.flags & MNF_FLAG_SCALE) net_off[n_nets] = op.net_off[0], net_slot[n_nets++] = 0;
        if (op.flags & MNF_FLAG_SHIFT) net_off[n_nets] = op.net_off[1], net_slot[n_nets++] = 1;
    }
    if (tid == 0) s_n = 0, s_ncand = 0;
    __syncthreads();

    bool over = false;
    for (int l = 1; l < L; ++l) {  // new breakpoints: zeros of the pre-activations of hidden layer l inside the current pieces
        const int n = s_n;
        for (int i = warp; i <= n; i += BW) {
            double lo, hi;
            const double m = piece_point(s_bp, n, i, lo, hi);
            for (int q = 0; q < n_nets; ++q) {
                const int cur = net_pre_maps(params + net_off[q], op.sizes, l - 1, m, s_va[warp], s_vb[warp], lane);
                for (int k = lane; k < op.sizes[l]; k += 32) {
                    const double a = s_va[warp][cur][k], b = s_vb[warp][cur][k];
                    if (a != 0.0) {
                        const double tz = -b / a;
                        // (a kink beyond the fp32 range -- a first-layer weight of ~1e-39 -- is no kink for any fp32 input,
                        // and would give its piece an infinite origin)
                        if (tz > lo && tz < hi && fabs(tz) < 3.0e38) {
                            const int pos = atomicAdd(&s_ncand, 1);
                            if (pos < 512) s_tmp[pos] = tz;
                        }
                    }
                }
                __syncwarp();
            }
        }
        __syncthreads();
        const int nc = s_ncand, tot = n + nc;
        if (tot > PMAX) {
            over = true;
            break;
        }
        for (int e = tid; e < nc; e += nt) s_bp[n + e] = s_tmp[e];
        __syncthreads();
        sort_bp(tot);
        if (tid == 0) s_n = tot, s_ncand = 0;
        __syncthreads();
    }

    float *region = image + gl.region[g];
    int *hdr = reinterpret_cast<int *>(image) + g * HDR_INTS;
    const int n = over ? 0 : s_n;
    if (tid == 0) hdr[0] = n, hdr[1] = over ? 1 : 0, hdr[2] = 0, hdr[3] = 0;
    for (int e = tid; e < BP_FLOATS; e += nt) region[e] = e < n ? (float)s_bp[e] : INFINITY;
    if (over) return;
    const int stride = 4 * (nsf ? nsf_stride4(K) : AFF_STRIDE4);
    // Rows of the nn + 1 pieces of s_bp.  fast: the spline outputs of each axis minus the axis's envelope_line and, like
    // the knot-derivative outputs, in log2 units (softmax is invariant to the shift; the kernel feeds them to ex2 as they are).
    auto write_rows = [&](int nn, float *rows, bool fast) {
        for (int i = warp; i <= nn; i += BW) {
            double lo, hi;
            const double m = piece_point(s_bp, nn, i, lo, hi);
            // origin: the (fp32) breakpoint the piece starts at -- the kernel forms c - origin exactly there
            const float org = nn == 0 ? 0.f : (float)(i == 0 ? s_bp[0] : s_bp[i - 1]);
            float *row = rows + (size_t)i * stride;
            for (int e = lane; e < stride; e += 32) row[e] = 0.f;
            __syncwarp();
            for (int q = 0; q < n_nets; ++q) {
                const int cur = net_pre_maps(params + net_off[q], op.sizes, L - 1, m, s_va[warp], s_vb[warp], lane);
                const double *va = s_va[warp][cur], *vb = s_vb[warp][cur];
                for (int o = lane; o < n_out; o += 32) {
                    double A = va[o], B = vb[o], sc = 1.0;
                    if (fast && nsf) {
                        sc = LOG2E_D;
                        if (o < 2 * K) {
                            const int l = envelope_line(va, vb, o < K ? 0 : K, K, lo, hi);
                            A -= va[l], B -= vb[l];
                        }
                    }
                    const double V = fma(A, (double)org, B);
                    int ia, iv;
                    if (!nsf) ia = net_slot[q], iv = 2 + net_slot[q];
                    else if (o < 2 * K) ia = 4 * (o >> 1) + (o & 1), iv = ia + 2;
                    else ia = nsf_doff(K) + 2 * (o - 2 * K), iv = ia + 1;
                    row[ia] = (float)(A * sc), row[iv] = (float)(V * sc);
                }
                __syncwarp();
            }
            if (lane == 0) row[nsf ? nsf_org(K) : AFF_ORG] = org;
        }
    };
    write_rows(n, region + BP_FLOATS, false);

    // Fast form, in rows n + 1 .. PMAX of the region (never read otherwise): [lo, inv, NB - 1, offset of the rows]
    // [NB bucket records (number of breakpoints in the buckets before, the <= 3 breakpoints of the bucket padded with +inf)]
    // [rows of the fast pieces].  The fast pieces are the pieces cut further (split_piece) where a spline axis's outputs
    // would reach more than FAST_T above the line they are stored relative to.
    __syncthreads();  // the rows read s_bp, which becomes the list of fast breakpoints
    if (tid == 0) s_ncand = 0, s_fail = nsf && !(op.bound <= FAST_B_MAX);
    __syncthreads();
    if (nsf && !s_fail) {
        for (int i = warp; i <= n; i += BW) {
            double lo, hi;
            const double m = piece_point(s_bp, n, i, lo, hi);
            const int cur = net_pre_maps(params + net_off[0], op.sizes, L - 1, m, s_va[warp], s_vb[warp], lane);
            if (lane == 0 && !split_piece(s_va[warp][cur], s_vb[warp][cur], K, lo, hi, s_tmp, &s_ncand)) s_fail = 1;
            __syncwarp();
        }
    }
    __syncthreads();
    const int nf = n + s_ncand;
    if (s_fail || nf > PMAX) return;
    for (int e = tid; e < nf - n; e += nt) s_bp[n + e] = s_tmp[e];
    __syncthreads();
    sort_bp(nf);
    const int fast_off = BP_FLOATS + (n + 1) * stride, rows_floats = (nf + 1) * stride;
    // Grid: the fewest buckets NB with <= 3 breakpoints in each, spanning the fast breakpoints from the a-th lowest to the
    // b-th highest (a, b <= 2: kinks lie dense around the origin with a few far out, which the two clamped end buckets
    // take).  Bounded so that the fast forms of all tables of the program fit in shared memory together.
    const int budget = min((PMAX - n) * stride, SMEM_TABLE_FLOATS / gl.n);
    int nb = NB_MIN;
    float lo32 = 0.f, inv = 0.f;
    for (bool found = false; !found; nb *= 2) {
        if (nb > NB_MAX || 4 + 4 * nb + rows_floats > budget) return;
        for (int ab = 0; ab < 9 && !found; ++ab) {
            const int a = ab / 3, b = ab % 3;
            if (nf && a + b >= nf) continue;
            lo32 = nf ? (float)s_bp[a] : 0.f;
            const float hi32 = nf ? (float)s_bp[nf - 1 - b] : 0.f;
            inv = hi32 > lo32 ? (float)((double)nb / ((double)hi32 - (double)lo32)) : 0.f;
            for (int e = tid; e < nf; e += nt) s_bidx[e] = bucket_of((float)s_bp[e], lo32, inv, (float)(nb - 1));
            __syncthreads();
            int bad = 0;
            for (int e = tid; e + 3 < nf; e += nt) bad |= s_bidx[e] == s_bidx[e + 3];
            found = !__syncthreads_or(bad);
        }
        if (found) break;
    }
    float *fast = region + fast_off;
    for (int j = tid; j < nb; j += nt) {
        int a = 0, b = nf;  // first breakpoint of bucket >= j
        while (a < b) {
            const int mid = (a + b) >> 1;
            if (s_bidx[mid] < j) a = mid + 1; else b = mid;
        }
        float4 r;
        r.x = __int_as_float(a);
        r.y = a < nf && s_bidx[a] == j ? (float)s_bp[a] : INFINITY;
        r.z = a + 1 < nf && s_bidx[a + 1] == j ? (float)s_bp[a + 1] : INFINITY;
        r.w = a + 2 < nf && s_bidx[a + 2] == j ? (float)s_bp[a + 2] : INFINITY;
        reinterpret_cast<float4 *>(fast)[1 + j] = r;
    }
    if (tid == 0) {
        fast[0] = lo32, fast[1] = inv, fast[2] = (float)(nb - 1), fast[3] = __int_as_float(4 + 4 * nb);
        hdr[2] = fast_off, hdr[3] = 4 + 4 * nb + rows_floats;
    }
    write_rows(nf, fast + 4 + 4 * nb, true);
}

// ---------------------------------------------------------------------------------------------------------
// evaluation
// ---------------------------------------------------------------------------------------------------------
struct Params {
    FlowProgram prog;  // module order
    GroupList gl;
    const float *params, *x, *image;
    float *y, *log_det, *base_lp, *inter;
    long long n_rows;
    int dir_flags, smem_floats;
    mnf_gather_out gather;
    // DRAW only (after the fields above, so that the other instantiations see the same layout)
    unsigned long long seed, row_offset;  // Philox key; global index of local row 0
    float *z;                             // optional output: the drawn base point
    unsigned noise_stream;
};

__device__ __forceinline__ float2 f2_fma(float2 a, float2 b, float2 c) {
    unsigned long long ra = *reinterpret_cast<unsigned long long *>(&a), rb = *reinterpret_cast<unsigned long long *>(&b),
                       rc = *reinterpret_cast<unsigned long long *>(&c), rd;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
    return *reinterpret_cast<float2 *>(&rd);
}
__device__ __forceinline__ float2 f2_add(float2 a, float2 b) {
    unsigned long long ra = *reinterpret_cast<unsigned long long *>(&a), rb = *reinterpret_cast<unsigned long long *>(&b), rd;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
    return *reinterpret_cast<float2 *>(&rd);
}
__device__ __forceinline__ float2 f2_splat(float a) { return make_float2(a, a); }

// exact-fp32 evaluation of a net layer by layer (tables that overflowed): parameter blob, per Linear weight[out][in], bias[out]
__device__ __noinline__ void mlp_fp32(const float *__restrict__ net, int n_lin, const int *sizes, float c, float *out) {
    float h[2][MAX_H];
    h[0][0] = c;
    int cur = 0;
    const float *p = net;
    for (int t = 0; t < n_lin; ++t) {
        const int n_in = sizes[t], n_o = sizes[t + 1];
        for (int k = 0; k < n_o; ++k) {
            float acc = p[n_in * n_o + k];
            for (int j = 0; j < n_in; ++j) acc = fmaf(p[k * n_in + j], h[cur][j], acc);
            if (t + 1 < n_lin) h[cur ^ 1][k] = leaky02(acc);
            else out[k] = acc;
        }
        cur ^= 1;
        p += n_in * n_o + n_o;
    }
}

// (values in and out by value: a reference parameter of a non-inlined function would pin the caller's accumulators to
// local memory on the table path as well)
template <int K>
__device__ __noinline__ float2 nsf_fallback(const float *__restrict__ net, int n_lin, const int *sizes, float B, float edge_deriv, float c,
                                            bool inverse, float tr) {
    float raw[3 * K - 1], ld = 0.f;
    mlp_fp32(net, n_lin, sizes, c, raw);
    rq_spline<K, true>(raw, K, B, edge_deriv, inverse, tr, ld);
    return make_float2(tr, ld);
}
__device__ __noinline__ float mlp_fp32_scalar(const float *__restrict__ net, int n_lin, const int *sizes, float c) {
    float out[1];
    mlp_fp32(net, n_lin, sizes, c, out);
    return out[0];
}

template <int S>
__device__ __forceinline__ void search_steps(uint32_t &a, float c) {
    float t;
    asm("ld.shared.f32 %0, [%1+%2];" : "=f"(t) : "r"(a), "n"(4 * (S - 1)));
    if (c > t) a += 4u * S;
    if constexpr (S > 1) search_steps<S / 2>(a, c);
}

// piece of c: count of breakpoints below it, branch-free over the +inf padded array.  SM: the table is in shared memory and
// the search walks a byte address (load, compare, predicated add per step).
template <bool SM>
__device__ __forceinline__ int find_piece(const float *tb, float c) {
    if constexpr (SM) {
        const uint32_t base = smem_u32(tb);
        uint32_t a = base;
        search_steps<(PMAX + 1) / 2>(a, c);
        return (int)((a - base) >> 2);
    } else {
        int pos = 0;
#pragma unroll
        for (int s = (PMAX + 1) / 2; s >= 1; s >>= 1) pos += (c > tb[pos + s - 1]) ? s : 0;
        return pos;
    }
}

enum { KIND_PLAIN = 0, KIND_FAST = 1, KIND_OVER = 2 };  // table evaluated by binary search / by its fast form / layer by layer

// row of the piece of c.  fast: tb is the table's fast form -- one grid load (the same address for the whole warp), one
// bucket record, three compares; otherwise the binary search over the padded breakpoints.
template <bool SM>
__device__ __forceinline__ const float4 *piece_row(const float *tb, bool fast, float c, int stride4) {
    if (fast) {
        const float4 gr = *reinterpret_cast<const float4 *>(tb);
        const float4 bk = reinterpret_cast<const float4 *>(tb)[1 + bucket_of(c, gr.x, gr.y, gr.z)];
        const int piece = __float_as_int(bk.x) + (c > bk.y) + (c > bk.z) + (c > bk.w);
        return reinterpret_cast<const float4 *>(tb + __float_as_int(gr.w)) + piece * stride4;
    }
    return reinterpret_cast<const float4 *>(tb + BP_FLOATS) + find_piece<SM>(tb, c) * stride4;
}

// MNF_FPL_ABLATE selects a timing ablation of the spline conditioner (tools/bench_flow_pl_pipes.py; its outputs are
// wrong by construction): 1 every ex2 becomes a multiply (no XU work for the exponentials), 2 the bin selection is
// short-circuited to a fixed bin, 3 the knot derivatives are constant.  0, the only value the library is built with,
// leaves the kernel as it is.
#ifndef MNF_FPL_ABLATE
#define MNF_FPL_ABLATE 0
#endif

__device__ __forceinline__ float ex2_approx(float x) {
    float r;
#if MNF_FPL_ABLATE == 1
    asm("mul.f32 %0, %1, 0f3F7FFFFE;" : "=f"(r) : "f"(x));
#else
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
#endif
    return r;
}
__device__ __forceinline__ float sqrt_approx(float x) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float lg2_approx(float x) {
    float r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

constexpr float LOG2E = 1.4426950408889634f, LN2 = 0.6931471805599453f;

// constant part of knot k in units of B: -1 + 2 k min_bin
__device__ __forceinline__ float knot_const(float k) { return fmaf(2.f * kMinBin, k, -1.f); }

// The two spline axes of a conditioner in units of B, as prefix sums S[k < K - 1] = (f_0 + .. + f_k) of the second softmax's
// terms (x = width, y = height axis) and their scales c1 = 2 span / sum f: knot k + 1 is knot_const(k + 1) + c1 S[k], one
// FMA (t[0] = -1, t[K] = 1 pinned) -- the formulas of flow_math.cuh::spline_knots (both softmaxes of
// spline_flow.py:253-255 and :95, floor :96-97, cumsum :99, pinned ends :100-101).
// FAST: raw holds the outputs of a fast table (log2 units, largest in [0, FAST_T]): no max to subtract, every first-softmax
// sum lies in [1, K 2^FAST_T] and, with the second softmax's arguments centred on 0, every second-softmax sum in
// [e^-B, K e^B], so each pair of sums is inverted by one reciprocal of its product.  Otherwise (natural units) the
// largest output of each axis is subtracted first.
// X[k]: the second softmax's (width, height) terms, S[k] = X[0] + .. + X[k] summed in that order.
template <int K, bool FAST>
__device__ __forceinline__ void unit_knots(const float *raw, float twoB, float2 *X, float2 *S, float2 &c1) {
    constexpr float span = 1.f - kMinBin * (float)K;
    float2 e[K], sc, off;
    if constexpr (FAST) {
        float2 s1;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            e[k] = make_float2(ex2_approx(raw[k]), ex2_approx(raw[K + k]));
            s1 = k ? f2_add(s1, e[k]) : e[k];
        }
        const float r = frcp<true>(s1.x * s1.y), s = twoB * LOG2E;  // first softmax scaled by 2B, in log2 units
        sc = make_float2(s * (r * s1.y), s * (r * s1.x));
        off = f2_splat(-0.5f * s);
    } else {
        float mw = raw[0], mh = raw[K], sw = 0.f, sh = 0.f;
#pragma unroll
        for (int k = 1; k < K; ++k) mw = fmaxf(mw, raw[k]), mh = fmaxf(mh, raw[K + k]);
        const float mwn = -mw * LOG2E, mhn = -mh * LOG2E;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            e[k] = make_float2(ex2_approx(fmaf(raw[k], LOG2E, mwn)), ex2_approx(fmaf(raw[K + k], LOG2E, mhn)));
            sw += e[k].x, sh += e[k].y;
        }
        sc = make_float2(twoB * frcp<true>(sw) * LOG2E, twoB * frcp<true>(sh) * LOG2E);
        off = make_float2(twoB > 80.f ? -sc.x : 0.f, twoB > 80.f ? -sc.y : 0.f);  // arguments of the second softmax lie in [0, 2B]
    }
    float2 p;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const float2 a = f2_fma(e[k], sc, off);
        X[k] = make_float2(ex2_approx(a.x), ex2_approx(a.y));
        p = k ? f2_add(p, X[k]) : X[k];
        if (k + 1 < K) S[k] = p;
    }
    if constexpr (FAST) {
        const float r = frcp<true>(p.x * p.y);
        c1 = make_float2(2.f * span * (r * p.y), 2.f * span * (r * p.x));
    } else {
        c1 = make_float2(2.f * span * frcp<true>(p.x), 2.f * span * frcp<true>(p.y));
    }
}

// flow_math.cuh::knot_derivative (FAST flavour) of a raw output given in log2 units, without a branch: lg2(2 + 2^r) is r to
// fp32 precision above 20 log2(e), where the clamp keeps ex2 finite and the max returns r itself.
__device__ __forceinline__ float knot_derivative_log2(float r) {
    return fmaf(LN2, fmaxf(r, lg2_approx(2.f + ex2_approx(fminf(r, 20.f * LOG2E)))), kMinDeriv);
}

// Log-det of the spline conditioners of a point as a running product P in [1, 2) times 2^E: one lg2 per point at the end
// instead of one log per conditioner.  Renormalising multiplies by 2^(127 - exponent field), so 0 and NaN stay what they
// are.
__device__ __forceinline__ void ld_mul(float &P, int &E, float q) {
    P *= q;
    const int eb = __float_as_int(P) & 0x7f800000;
    E += (eb >> 23) - 127;
    P *= __int_as_float(0x7f000000 - eb);
}
// ld += (log P + E log 2) negated for INV, and the product reset.  (Also before the calls of the layer-by-layer fallbacks:
// P and E are then not live across them, which keeps the point loop's state in registers.)
template <bool INV>
__device__ __forceinline__ void ld_flush(float &ld, float &P, int &E) {
    ld = fmaf(INV ? -LN2 : LN2, lg2_approx(P) + (float)E, ld);  // P in [1, 2) (or 0, NaN): no denormal operand
    P = 1.f, E = 0;
}

// The rational-quadratic spline of flow_math.cuh::rq_spline (FAST flavour) for a point already known to lie in [-B, B],
// evaluated in units of B (the bin ratios, the knot derivatives and the log-det do not depend on the unit).  The raw
// derivatives of the two knots around the point's bin are fetched through `deriv(j)` once the bin is known -- the
// conditioner's other K - 3 derivative outputs are never formed.  FAST: raw outputs of a fast table (log2 units).  The
// forward spline's derivative at the point goes into the log-det product (P, E) of ld_mul; INV subtracts its log.
template <int K, bool FAST, bool INV, class DerivFn>
__device__ __forceinline__ void rq_spline_lazy(const float *raw, float B, float inv_B, float edge_deriv, float &v, float &P, int &E,
                                               DerivFn deriv) {
    float2 X[K], S[K - 1], c1;
    unit_knots<K, FAST>(raw, 2.f * B, X, S, c1);
    const float u = v * inv_B;
    // bin = number of interior knots <= u (spline_flow.py:22-24,115-118; u lies inside [t_0, t_K], so the count needs no
    // clamp).  Only the searched axis's knots are formed.  Each compare gives a mask m_k in {0, 1}, non-increasing in k, so
    // the prefix sums at both ends of the bin are masked sums of the terms X in the order S was summed: lo = S[idx - 1]
    // (0 for idx = 0) and hi = S[idx] bit for bit, one FFMA2 per knot and end for both axes.  The knots are made from them
    // afterwards.
    float fidx = 0.f;
    float2 lo = f2_splat(0.f), hi = X[0];
#if MNF_FPL_ABLATE == 2
    fidx = (float)(K / 2), lo = S[K / 2 - 1], hi = S[K / 2];
#else
#pragma unroll
    for (int k = 1; k < K; ++k) {
        const float m = u >= fmaf(INV ? S[k - 1].y : S[k - 1].x, INV ? c1.y : c1.x, knot_const((float)k)) ? 1.f : 0.f;
        fidx += m;
        lo = f2_fma(f2_splat(m), X[k - 1], lo);
        if (k + 1 < K) hi = f2_fma(f2_splat(m), X[k], hi);  // (the last bin's upper knots are pinned)
    }
#endif
    const int idx = __float_as_int(fidx + 8388608.f) - 0x4b000000;  // (int)fidx without the XU pipe
    const float k0 = knot_const(fidx), k1 = knot_const(fidx + 1.f);
    const float2 lk = f2_fma(lo, c1, f2_splat(k0)), hk2 = f2_fma(hi, c1, f2_splat(k1));
    const float xk = lk.x, yk = lk.y;
    const bool last = idx == K - 1;
    const float xk1 = last ? 1.f : hk2.x, yk1 = last ? 1.f : hk2.y;
    const float wk = xk1 - xk, hk = yk1 - yk;  // spline_flow.py:102,113
    // interior knot derivatives (spline_flow.py:256,104), the padded constant at the two ends (:46-49); the loads are
    // unconditional on a clamped index so that lanes in different bins do not diverge
    const float r0 = deriv(max(idx - 1, 0)), r1 = deriv(min(idx, K - 2));
    float dk, dk1;
    if constexpr (FAST) {  // both formed, then selected: no branch around the MUFU work
        const float d0 = knot_derivative_log2(r0), d1 = knot_derivative_log2(r1);
        dk = idx > 0 ? d0 : edge_deriv;
        dk1 = idx < K - 1 ? d1 : edge_deriv;
    } else {
        dk = (idx > 0) ? knot_derivative<true>(r0) : edge_deriv;
        dk1 = (idx < K - 1) ? knot_derivative<true>(r1) : edge_deriv;
    }
#if MNF_FPL_ABLATE == 3
    dk = dk1 = edge_deriv;
#endif
    // Reciprocals are rcp.approx.ftz, which differs from __fdividef only where the operand is not a normal number; every
    // operand below is a product or sum of bin widths and heights (>= 2 min_bin), knot derivatives (>= min_deriv) and
    // terms in [0, 1], so it is not below the normal range.  (-b - sqrt(disc) is -2 hk dk wk at dy = 0 and grows in
    // magnitude with dy.)  Above 2^126 (a knot derivative near the fp32 limit) both forms return 0.
    if constexpr (INV) {  // spline_flow.py:133-162 with the quadratic's coefficients and the log-det's terms multiplied by powers
                          // of wk, which leaves the root and the ratio unchanged and needs no hk / wk
        const float dkw = dk * wk, dk1w = dk1 * wk;
        const float dsw = dkw + dk1w - 2.f * hk;  // dsum wk
        const float dy = u - yk;
        const float a = dy * dsw + hk * (hk - dkw);
        const float b = hk * dkw - dy * dsw;
        const float c = -hk * dy;
        const float disc = fmaxf(b * b - 4.f * a * c, 0.f);
        const float root = 2.f * c * frcp<true>(-b - sqrt_approx(disc));
        v = (root * wk + xk) * B;
        const float tt = root * (1.f - root);
        const float omr = 1.f - root;
        const float den = wk * (hk + dsw * tt);                                                   // den wk^2
        const float num = (hk * hk) * wk * (dk1w * (root * root) + 2.f * hk * tt + dkw * (omr * omr));  // num wk^4
        const float rd = frcp<true>(den);
        ld_mul(P, E, num * rd * rd);
    } else {  // spline_flow.py:163-179
        const float rw = frcp<true>(wk);
        const float sk_ = hk * rw;  // spline_flow.py:123
        const float dsum = dk + dk1 - 2.f * sk_;
        const float th = (u - xk) * rw;
        const float tt = th * (1.f - th);
        const float numer = hk * (sk_ * (th * th) + dk * tt);
        const float den = sk_ + dsum * tt;
        const float omt = 1.f - th;
        const float num = (sk_ * sk_) * (dk1 * (th * th) + 2.f * sk_ * tt + dk * (omt * omt));
        const float rd = frcp<true>(den);
        v = fmaf(numer, rd, yk) * B;
        ld_mul(P, E, num * rd * rd);
    }
}

constexpr int THREADS = 1024;

// The stack as the point loop walks it (execution order, built once per CTA): runs of AffineConstantFlow / ActNormFlow / Glow
// are composed into ONE affine map v -> v M + b with a constant log-det (fp64; not when per-flow outputs are requested),
// the coupling flows carry their constants and table indices -- the loop never touches the descriptors again.
struct Exec {
    int type;   // 0 affine map, 1 AffineHalfFlow, 2 NSF_CL
    int k;      // flow index (parameters of the fp32 fallback)
    int g0, g1; // tables: AffineHalfFlow g0; NSF_CL g0 = first step's, g1 = second step's
    int flag;   // AffineHalfFlow: parity; NSF_CL: the first step is f1 (forward direction)
    int pad[3];
    float c[8]; // affine: m00 m01 m10 m11 | b0 b1 dld - ; NSF_CL: B 1/B edge_deriv - ; AffineHalfFlow: -
};
static_assert(sizeof(Exec) == 64, "two 16-byte rows of ints, two of floats");

__device__ __forceinline__ void build_exec(const Params &p, Exec *ex, int *n_exec, int lane) {
    const int n = p.prog.n_ops, inverse = p.dir_flags & 1;
    if (lane < n) {
        const int k = inverse ? n - 1 - lane : lane;
        const mnf_flow_op &op = p.prog.ops[k];
        Exec e{};
        e.k = k;
        if (op.type == MNF_OP_AFFINE_CONST) {
            const double s0 = p.params[op.aux_off], s1 = p.params[op.aux_off + 1];
            const double t0 = p.params[op.aux_off + 2], t1 = p.params[op.aux_off + 3];
            if (inverse) {  // (v - t) exp(-s), affine_constant_flow.py:24
                const double e0 = exp(-s0), e1 = exp(-s1);
                e.c[0] = (float)e0, e.c[3] = (float)e1, e.c[4] = (float)(-t0 * e0), e.c[5] = (float)(-t1 * e1), e.c[6] = (float)(-(s0 + s1));
            } else {  // v exp(s) + t, affine_constant_flow.py:19
                e.c[0] = (float)exp(s0), e.c[3] = (float)exp(s1), e.c[4] = (float)t0, e.c[5] = (float)t1, e.c[6] = (float)(s0 + s1);
            }
        } else if (op.type == MNF_OP_GLOW) {  // v @ W (glow.py:28) or v @ W^-1 (glow.py:36)
            const float *W = p.params + op.aux_off + (inverse ? 4 : 0);
            e.c[0] = W[0], e.c[1] = W[1], e.c[2] = W[2], e.c[3] = W[3];
            e.c[6] = inverse ? -p.params[op.aux_off + 8] : p.params[op.aux_off + 8];
        } else if (op.type == MNF_OP_AFFINE_HALF) {
            e.type = 1, e.g0 = p.gl.group_of[k][0], e.flag = (op.flags & MNF_FLAG_PARITY) ? 1 : 0;
        } else {  // forward: f1 then f2 (spline_flow.py:249-266); inverse: f2 then f1 (:268-285)
            e.type = 2, e.flag = inverse ? 0 : 1;
            e.g0 = p.gl.group_of[k][inverse ? 1 : 0], e.g1 = p.gl.group_of[k][inverse ? 0 : 1];
            e.c[0] = op.bound, e.c[1] = 1.f / op.bound, e.c[2] = op.edge_deriv;
        }
        ex[lane] = e;
    }
    __syncwarp();
    if (lane == 0) {
        int j = 0;
        bool open = false;  // ex[j - 1] is an affine map that may still absorb the next one
        double M[4], b[2], ld;
        for (int i = 0; i < n; ++i) {
            const Exec e = ex[i];
            if (e.type != 0 || p.inter) {
                ex[j++] = e, open = false;
                continue;
            }
            if (!open) {
                for (int q = 0; q < 4; ++q) M[q] = e.c[q];
                b[0] = e.c[4], b[1] = e.c[5], ld = e.c[6];
                ++j, open = true;
            } else {  // (v M + b) W + t = v (M W) + (b W + t)
                const double W0 = e.c[0], W1 = e.c[1], W2 = e.c[2], W3 = e.c[3];
                const double n00 = M[0] * W0 + M[1] * W2, n01 = M[0] * W1 + M[1] * W3;
                const double n10 = M[2] * W0 + M[3] * W2, n11 = M[2] * W1 + M[3] * W3;
                const double nb0 = b[0] * W0 + b[1] * W2 + e.c[4], nb1 = b[0] * W1 + b[1] * W3 + e.c[5];
                M[0] = n00, M[1] = n01, M[2] = n10, M[3] = n11, b[0] = nb0, b[1] = nb1, ld += e.c[6];
            }
            Exec f{};
            for (int q = 0; q < 4; ++q) f.c[q] = (float)M[q];
            f.c[4] = (float)b[0], f.c[5] = (float)b[1], f.c[6] = (float)ld;
            ex[j - 1] = f;
        }
        *n_exec = j;
    }
}

// SM: every table of the program sits in shared memory (plain LDS); otherwise a table is read through a generic pointer
// (shared memory if it fitted, the image in global memory if not).
template <int K, bool SM, bool INV, bool DRAW>
__device__ __forceinline__ void run_points(const Params &p, const float *smem, const int *s_off, const int *s_goff, const int *s_kind,
                                           const Exec *ex, int n_exec) {
    const bool sum_lp = p.dir_flags & 2;
    auto table = [&](int g) -> const float * {
        if constexpr (SM) return smem + s_off[g];
        const int o = s_off[g];
        return o >= 0 ? smem + o : p.image + s_goff[g];
    };
    const long long stride = (long long)gridDim.x * blockDim.x;
#pragma unroll 1
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < p.n_rows; r += stride) {
        float v0, v1, ld = 0.f, P = 1.f;  // log-det: ld + (log P + E log 2) of the spline conditioners (ld_mul), negated for INV
        int E = 0;
        if constexpr (DRAW) {
            // philox_normal's mapping of global element e = 2 (row_offset + r) + col: counter e >> 2, words (x, y) for even
            // global rows and (z, w) for odd ones -- the numbers every Philox draw of the library gives for these indices.
            // The running log-det starts at -log N(z), so that -ld is log q(x) at the end.
            const unsigned long long gr = p.row_offset + (unsigned long long)r;
            const uint4 w = Philox(p.seed)(gr >> 1, p.noise_stream);
            const bool odd = gr & 1ull;
            const float2 zn = box_muller(odd ? w.z : w.x, odd ? w.w : w.y);
            v0 = zn.x, v1 = zn.y;
            if (p.z) st_stream2(reinterpret_cast<float2 *>(p.z) + r, zn);
            ld = fmaf(0.5f, fmaf(v0, v0, v1 * v1), 1.8378770664093453f);
        } else {
            const float2 xin = ld_stream2(reinterpret_cast<const float2 *>(p.x) + r);
            v0 = xin.x, v1 = xin.y;
        }
#pragma unroll 1
        for (int kk = 0; kk < n_exec; ++kk) {
            const int4 ei = *reinterpret_cast<const int4 *>(&ex[kk]);  // type, k, g0, g1
            if (ei.x == 0) {
                const float4 m = *reinterpret_cast<const float4 *>(ex[kk].c), b = *reinterpret_cast<const float4 *>(ex[kk].c + 4);
                const float n0 = fmaf(v1, m.z, fmaf(v0, m.x, b.x)), n1 = fmaf(v1, m.w, fmaf(v0, m.y, b.y));
                v0 = n0, v1 = n1, ld += b.z;
            } else if (ei.x == 1) {
                const mnf_flow_op &op = p.prog.ops[ei.y];
                const bool parity = ex[kk].flag != 0;
                const float c = parity ? v1 : v0;  // affine_half_flow.py:46-50
                float tr = parity ? v0 : v1;
                const int g = ei.z;
                float s = 0.f, t = 0.f;
                if (g < 0) {  // neither net: s = t = 0
                } else if (s_kind[g] != KIND_OVER) {
                    const float4 *row = piece_row<SM>(table(g), s_kind[g] == KIND_FAST, c, AFF_STRIDE4);
                    const float4 q = row[0];
                    const float d = c - row[1].x;
                    s = fmaf(q.x, d, q.z), t = fmaf(q.y, d, q.w);
                } else {
                    ld_flush<INV>(ld, P, E);
                    if (op.flags & MNF_FLAG_SCALE) s = mlp_fp32_scalar(p.params + op.net_off[0], op.n_lin, op.sizes, c);
                    if (op.flags & MNF_FLAG_SHIFT) t = mlp_fp32_scalar(p.params + op.net_off[1], op.n_lin, op.sizes, c);
                }
                if constexpr (INV) {  // affine_half_flow.py:54-56
                    tr = (tr - t) / expf(s), ld -= s;
                } else {  // affine_half_flow.py:58
                    tr = expf(s) * tr + t, ld += s;
                }
                if (parity) v0 = tr; else v1 = tr;
            } else {
                const float4 cs = *reinterpret_cast<const float4 *>(ex[kk].c);  // B, 1/B, edge_deriv
                const bool first_f1 = ex[kk].flag != 0;
#pragma unroll 1
                for (int step = 0; step < 2; ++step) {
                    const bool use_f1 = (step == 0) == first_f1;
                    const float c = use_f1 ? v0 : v1;
                    float tr = use_f1 ? v1 : v0;
                    const float B = cs.x;
                    if (tr >= -B && tr <= B) {  // identity tails (also NaN), spline_flow.py:40,51-52: the conditioner is not needed
                        const int g = step ? ei.w : ei.z;
                        const int kind = s_kind[g];
                        if (kind != KIND_OVER) {
                            const float4 *row = piece_row<SM>(table(g), kind == KIND_FAST, c, nsf_stride4(K));
                            const float d = c - row[nsf_org(K) / 4].x;
                            const float2 dd = make_float2(d, d);
                            float raw[2 * K];
#pragma unroll
                            for (int j = 0; j < K; ++j) {
                                const float4 q = row[j];
                                const float2 o = f2_fma(make_float2(q.x, q.y), dd, make_float2(q.z, q.w));
                                raw[2 * j] = o.x, raw[2 * j + 1] = o.y;
                            }
                            const float2 *dv = reinterpret_cast<const float2 *>(row) + nsf_doff(K) / 2;
                            const auto deriv = [&](int j) {
                                const float2 q = dv[j];
                                return fmaf(q.x, d, q.y);
                            };
                            if (kind == KIND_FAST) rq_spline_lazy<K, true, INV>(raw, B, cs.y, cs.z, tr, P, E, deriv);
                            else rq_spline_lazy<K, false, INV>(raw, B, cs.y, cs.z, tr, P, E, deriv);
                        } else {
                            const mnf_flow_op &op = p.prog.ops[ei.y];
                            ld_flush<INV>(ld, P, E);
                            const float2 o = nsf_fallback<K>(p.params + op.net_off[use_f1 ? 0 : 1], op.n_lin, op.sizes, B, cs.z, c,
                                                             INV, tr);
                            tr = o.x, ld += o.y;
                        }
                        if (use_f1) v1 = tr; else v0 = tr;
                    }
                }
            }
            if (p.inter) st_stream2(reinterpret_cast<float2 *>(p.inter + ((size_t)kk * p.n_rows + r) * 2), make_float2(v0, v1));
        }
        ld_flush<INV>(ld, P, E);
        float lp = fmaf(-0.5f, fmaf(v0, v0, v1 * v1), -1.8378770664093453f);  // -(D/2) log(2 pi), D = 2
        if (sum_lp) lp += ld;
        if constexpr (DRAW) lp = -ld;  // log N(z) - log_det
        if (p.y) st_stream2(reinterpret_cast<float2 *>(p.y) + r, make_float2(v0, v1));
        if (p.log_det) p.log_det[r] = ld;
        if (p.base_lp) p.base_lp[r] = lp;
        // fused gather: the result also goes straight to the other ranks over NVLink
        if constexpr (DRAW) continue;
        if (p.gather.multicast_ptr) {
            asm volatile("multimem.st.relaxed.sys.global.f32 [%0], %1;" ::"l"(p.gather.multicast_ptr + p.gather.row_offset + r), "f"(lp)
                         : "memory");
        } else {
            for (int g = 0; g < p.gather.n_peers; ++g) p.gather.peer_ptrs[g][p.gather.row_offset + r] = lp;
        }
    }
}

template <int K, bool INV, bool DRAW = false>
__global__ void __launch_bounds__(THREADS, 1) flow_pl_kernel(const __grid_constant__ Params p) {
    extern __shared__ __align__(16) float smem[];
    __shared__ __align__(16) Exec s_exec[MNF_MAX_OPS];
    __shared__ int s_off[MAX_GROUPS], s_goff[MAX_GROUPS], s_kind[MAX_GROUPS];
    __shared__ int s_allfit, s_nexec;
    __shared__ __align__(8) unsigned long long s_bar;
    const int lane = threadIdx.x & 31, ng = p.gl.n;
    const uint32_t bar = smem_u32(&s_bar);
    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x >= 32 && threadIdx.x < 64) build_exec(p, s_exec, &s_nexec, lane);
    if (threadIdx.x < 32) {
        // table sizes from the builder's header -> shared-memory offsets, one bulk copy per table of what its path reads:
        // the fast form if it has one, else the breakpoints and rows
        const int *hdr = reinterpret_cast<const int *>(p.image);
        int total = 0, fit = 1;
        for (int base = 0; base < ng; base += 32) {
            const int g = base + lane;
            int sz = 0, ov = 0, src = 0;
            if (g < ng) {
                const int4 h = *reinterpret_cast<const int4 *>(hdr + g * HDR_INTS);
                const int s4 = p.prog.ops[p.gl.op[g]].type == MNF_OP_NSF_CL ? nsf_stride4(K) : AFF_STRIDE4;
                ov = h.y;
                src = p.gl.region[g] + h.z;
                sz = ov ? 0 : h.z ? h.w : BP_FLOATS + (h.x + 1) * 4 * s4;
                s_kind[g] = ov ? KIND_OVER : h.z ? KIND_FAST : KIND_PLAIN;
                s_goff[g] = src;
            }
            int inc = sz;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= o) inc += t;
            }
            const int off = total + inc - sz;
            const bool ok = off + sz <= p.smem_floats;
            if (g < ng) {
                s_off[g] = (ov || !ok) ? -1 : off;
                if (!ov && ok) {
                    asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"((uint32_t)sz * 4u) : "memory");
                    bulk_load(smem_u32(smem + off), p.image + src, (uint32_t)sz * 4u, bar);
                }
            }
            fit &= __all_sync(0xffffffffu, g >= ng || ov || ok) ? 1 : 0;
            total += __shfl_sync(0xffffffffu, inc, 31);
        }
        __syncwarp();
        if (lane == 0) {
            s_allfit = fit;
            mbar_arrive(bar);
        }
    }
    __syncthreads();
    mbar_wait(bar, 0);
    if (s_allfit) run_points<K, true, INV, DRAW>(p, smem, s_off, s_goff, s_kind, s_exec, s_nexec);
    else run_points<K, false, INV, DRAW>(p, smem, s_off, s_goff, s_kind, s_exec, s_nexec);
}

// ---------------------------------------------------------------------------------------------------------
// host
// ---------------------------------------------------------------------------------------------------------
// bins K the point kernel is instantiated for (the spline lives in registers: K is a template parameter)
#define MNF_PL_BINS(X) X(4) X(5) X(6) X(8) X(10) X(12) X(16)
constexpr int K_MAX = 16;
static bool k_instantiated(int K) {
#define MNF_PL_HAVE(KK) if (K == KK) return true;
    MNF_PL_BINS(MNF_PL_HAVE)
#undef MNF_PL_HAVE
    return false;
}

struct Plan {
    bool ok = false;
    int K = 8;
    GroupList gl;
    int64_t image_floats = 0;
};

static Plan make_plan(const mnf_flow_op *ops, int n_ops, int dim) {
    Plan pl;
    if (dim != 2 || n_ops < 1 || n_ops > MNF_MAX_OPS) return pl;
    int K = 0, n = 0;
    int64_t off = HDR_FLOATS;
    for (int k = 0; k < n_ops; ++k) {
        const mnf_flow_op &op = ops[k];
        pl.gl.group_of[k][0] = pl.gl.group_of[k][1] = -1;
        if (op.type == MNF_OP_AFFINE_CONST || op.type == MNF_OP_GLOW) continue;
        if (op.type != MNF_OP_AFFINE_HALF && op.type != MNF_OP_NSF_CL) return pl;
        if (op.n_lin < 2 || op.n_lin > MNF_MAX_LIN || op.sizes[0] != 1) return pl;
        for (int l = 1; l < op.n_lin; ++l)
            if (op.sizes[l] < 1 || op.sizes[l] > MAX_H) return pl;
        if (op.type == MNF_OP_NSF_CL) {
            if (!k_instantiated(op.K)) return pl;
            if (K && op.K != K) return pl;
            K = op.K;
            if (op.sizes[op.n_lin] != 3 * K - 1) return pl;
            for (int which = 0; which < 2; ++which) {
                pl.gl.group_of[k][which] = (signed char)n;
                pl.gl.op[n] = (unsigned char)k, pl.gl.which[n] = (unsigned char)which, pl.gl.region[n] = (int)off;
                off += region_floats(nsf_stride4(K));
                ++n;
            }
        } else {
            if (op.sizes[op.n_lin] != 1) return pl;
            if (!(op.flags & (MNF_FLAG_SCALE | MNF_FLAG_SHIFT))) continue;  // no net at all: s = t = 0 ... handled as identity below
            pl.gl.group_of[k][0] = (signed char)n;
            pl.gl.op[n] = (unsigned char)k, pl.gl.which[n] = 0, pl.gl.region[n] = (int)off;
            off += region_floats(AFF_STRIDE4);
            ++n;
        }
    }
    pl.gl.n = n;  // 0: a stack without conditioner nets, run without tables
    pl.K = K ? K : 8;
    pl.image_floats = off;
    pl.ok = true;
    return pl;
}

template <int K, bool INV, bool DRAW = false>
static int launch_k(const Params &p, const DeviceProps *dp, size_t smem_bytes, cudaStream_t st) {
    static thread_local size_t attr_set[64] = {};  // per device: the attribute belongs to the device's copy of the function
    int dev = 0;
    MNF_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || attr_set[dev] < smem_bytes) {
        MNF_CUDA(cudaFuncSetAttribute(flow_pl_kernel<K, INV, DRAW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
        if (dev >= 0 && dev < 64) attr_set[dev] = smem_bytes;
    }
    // small batches are bound by the latency of one point's chain: spread the points over the SMs
    const int threads = p.n_rows <= (long long)dp->sm_count * 64 ? 64 : p.n_rows <= (long long)dp->sm_count * 256 ? 256 : THREADS;
    long long blocks = (p.n_rows + threads - 1) / threads;
    if (blocks > dp->sm_count) blocks = dp->sm_count;
    flow_pl_kernel<K, INV, DRAW><<<(unsigned)blocks, threads, smem_bytes, st>>>(p);
    return launch_status("flow_pl_kernel");
}

// The part of a point kernel's launch that does not depend on the direction: the tables (built into `workspace` unless
// it is staged), the program, the row count and the shared memory the kernel asks for (`want` bytes).
static int setup_params(const Plan &pl, const mnf_flow_op *ops, int n_ops, const float *params, float *workspace, int64_t n_rows,
                        bool staged, const DeviceProps *dp, cudaStream_t stream, Params &p, size_t &want);

}  // namespace fpl

// floats of workspace / staged image the piecewise-linear kernel needs for a program of n_ops flows (upper bound)
int64_t flow_pl_workspace_floats(int n_ops) {
    if (n_ops < 1) n_ops = 1;
    if (n_ops > MNF_MAX_OPS) n_ops = MNF_MAX_OPS;
    return fpl::HDR_FLOATS + (int64_t)2 * n_ops * fpl::region_floats(fpl::nsf_stride4(fpl::K_MAX));
}

// floats of the table image of this program, 0 if it has no tables to stage
int64_t flow_pl_image_floats(const mnf_flow_op *ops, int n_ops, int dim) {
    const fpl::Plan pl = fpl::make_plan(ops, n_ops, dim);
    return pl.ok && pl.gl.n > 0 ? pl.image_floats : 0;
}

// whether launch_flow_pl runs this program (given a workspace when it has conditioner nets)
bool flow_pl_accepts(const mnf_flow_op *ops, int n_ops, int dim) { return fpl::make_plan(ops, n_ops, dim).ok; }

int flow_pl_build(const mnf_flow_op *ops, int n_ops, const float *params, int dim, float *image, cudaStream_t stream) {
    using namespace fpl;
    const Plan pl = make_plan(ops, n_ops, dim);
    MNF_REQUIRE(pl.ok && pl.gl.n > 0, MNF_E_SHAPE, "program has no piecewise-linear form");
    MNF_REQUIRE(params && image && ((uintptr_t)image % 16) == 0, MNF_E_ARG, "NULL or misaligned pointer");
    FlowProgram prog;
    prog.n_ops = n_ops;
    for (int k = 0; k < n_ops; ++k) prog.ops[k] = ops[k];
    flow_pl_build_kernel<<<pl.gl.n, 32 * BW, 0, stream>>>(prog, pl.gl, params, image);
    return launch_status("flow_pl_build_kernel");
}

int fpl::setup_params(const Plan &pl, const mnf_flow_op *ops, int n_ops, const float *params, float *workspace, int64_t n_rows,
                      bool staged, const DeviceProps *dp, cudaStream_t stream, Params &p, size_t &want) {
    if (!staged && pl.gl.n > 0) {
        const int rc = flow_pl_build(ops, n_ops, params, 2, workspace, stream);
        if (rc) return rc;
    }
    p.prog.n_ops = n_ops;
    for (int k = 0; k < n_ops; ++k) p.prog.ops[k] = ops[k];
    p.gl = pl.gl;
    p.params = params, p.image = workspace, p.n_rows = n_rows;
    // shared memory: every table at its largest, capped by what a CTA can have
    want = (size_t)(pl.image_floats - HDR_FLOATS) * sizeof(float);
    const size_t cap = (size_t)dp->smem_optin - 4096;  // static shared memory of the kernel: execution list, offsets, barrier
    if (want > cap) want = cap;
    want &= ~(size_t)15;
    p.smem_floats = (int)(want / sizeof(float));
    return 0;
}

// returns 1 if the program is not eligible (caller falls back to the interpreter).  dir_flags: bit0 inverse, bit1 log-det
// summed into base_lp, bit2 `workspace` already holds the image of flow_pl_build for these parameters.  A program without
// conditioner nets has no tables and needs no workspace.
int launch_flow_pl(const mnf_flow_op *ops, int n_ops, const float *params, const float *x, float *y, float *log_det,
                   float *base_lp, float *inter, int64_t n_rows, int dim, int dir_flags, float *workspace,
                   const mnf_gather_out *gather, cudaStream_t stream) {
    using namespace fpl;
    const Plan pl = make_plan(ops, n_ops, dim);
    if (!pl.ok) return 1;
    MNF_REQUIRE(workspace || pl.gl.n == 0, MNF_E_ARG,
                "dim-2 programs with conditioner nets need a workspace of mnf_flow_stack_workspace() floats (or a staged image)");
    const DeviceProps *dp = device_props();
    MNF_REQUIRE(dp != nullptr, MNF_E_DEVICE, "no CUDA device");
    MNF_REQUIRE(((uintptr_t)workspace % 16) == 0, MNF_E_ALIGN, "workspace must be 16-byte aligned");
    MNF_REQUIRE(((uintptr_t)x % 8) == 0 && (!y || ((uintptr_t)y % 8) == 0) && (!inter || ((uintptr_t)inter % 8) == 0), MNF_E_ALIGN,
                "x, y and intermediates must be 8-byte aligned");
    MNF_REQUIRE(n_rows > 0, MNF_E_ARG, "bad row count");
    Params p{};
    size_t want = 0;
    int rc = setup_params(pl, ops, n_ops, params, workspace, n_rows, (dir_flags & 4) != 0, dp, stream, p, want);
    if (rc) return rc;
    p.x = x, p.y = y, p.log_det = log_det, p.base_lp = base_lp, p.inter = inter;
    p.dir_flags = dir_flags & 3;
    if (gather) {
        MNF_REQUIRE(gather->n_peers >= 0 && gather->n_peers <= MNF_MAX_PEERS, MNF_E_ARG, "bad n_peers");
        p.gather = *gather;
    }
#define MNF_PL_LAUNCH(KK) \
    if (pl.K == KK) return (dir_flags & 1) ? launch_k<KK, true>(p, dp, want, stream) : launch_k<KK, false>(p, dp, want, stream);
    MNF_PL_BINS(MNF_PL_LAUNCH)
#undef MNF_PL_LAUNCH
    return 1;
}

// Forward pass of base points drawn in the kernel (flow_pl_kernel<K, false, true>): x [n_rows, 2], log q(x) and the drawn
// z, each optional.  Returns 1 if the program is not eligible or no workspace was given (the caller takes the
// draw-then-forward path).  staged: `workspace` already holds the image of flow_pl_build for these parameters.
int launch_flow_pl_sample(const mnf_flow_op *ops, int n_ops, const float *params, uint64_t seed, uint32_t noise_stream,
                          uint64_t row_offset, float *x, float *log_prob, float *z, int64_t n_rows, int dim, bool staged,
                          float *workspace, cudaStream_t stream) {
    using namespace fpl;
    const Plan pl = make_plan(ops, n_ops, dim);
    if (!pl.ok || pl.gl.n == 0 || !workspace) return 1;
    const DeviceProps *dp = device_props();
    MNF_REQUIRE(dp != nullptr, MNF_E_DEVICE, "no CUDA device");
    MNF_REQUIRE(((uintptr_t)workspace % 16) == 0, MNF_E_ALIGN, "workspace must be 16-byte aligned");
    MNF_REQUIRE((!x || ((uintptr_t)x % 8) == 0) && (!z || ((uintptr_t)z % 8) == 0), MNF_E_ALIGN, "x and z must be 8-byte aligned");
    MNF_REQUIRE(n_rows > 0, MNF_E_ARG, "bad row count");
    Params p{};
    size_t want = 0;
    int rc = setup_params(pl, ops, n_ops, params, workspace, n_rows, staged, dp, stream, p, want);
    if (rc) return rc;
    p.y = x, p.base_lp = log_prob, p.z = z;
    p.seed = seed, p.row_offset = row_offset, p.noise_stream = noise_stream;
#define MNF_PL_LAUNCH(KK) \
    if (pl.K == KK) return launch_k<KK, false, true>(p, dp, want, stream);
    MNF_PL_BINS(MNF_PL_LAUNCH)
#undef MNF_PL_LAUNCH
    return 1;
}

}  // namespace mnf
