// DB (differentiable binarization) text detector: the probability maps of SegDetector and L1BalanceCELoss
// (decoders/seg_detector.py:117-147, decoders/seg_detector_loss.py:157-185 of the reference).
//
// Maps:  b = sigmoid(x_b), t = sigmoid(x_t), tb = 1 / (1 + exp(-k (b - t))); one element-wise pass each way.  Both use
// the accurate expf: the loss selects by the exact values of b.
//
// Loss.  gt g is (N,1,H,W) and mask m is (N,H,W), so the reference's `gt * mask` broadcasts to (N,N,H,W): entry
// [i,j,q] = g_i(q) m_j(q).  With l_j(q) = BCE(b_j(q), g_j(q)) (ATen's formula, logs clamped at -100):
//   P_j(q) = sum_i u8(g_i m_j),  C_j(q) = sum_i u8((1 - g_i) m_j),   pos = sum P,  k = min(sum C, floor(3 pos))
//   topk   = sum of the k largest of {l_j(q) with multiplicity C_j(q)}
//   bce    = (sum P l + topk) / (pos + k + 1e-6),  dice = 1 - 2 I / U,  l1 = sum |t - z| w / sum w
// Nothing of size N^2 H W is formed.  Forward, with no host synchronisation (9 launches):
//   1. stats:     a thread owns a pixel q for every j; it stages g_i(q) for all i in shared memory, so P and C are the
//                 reference's counts for any gt / mask values in [0, 1], and writes a record {l, C, P} per (j, q) plus per-block partial sums.
//   2. select:    weighted radix select on the bit pattern of l (l >= 0, so the bits are monotone), 11/11/10-bit digits:
//                 a histogram pass of 64-bit multiplicity sums and a one-CTA narrowing kernel per digit.  It finds
//                 tau (cumulative weight from the top reaches k there), above = W(l > tau), T = W(l = tau).
//   3. sel-sum:   per-block partial sums of C l over l > tau.
//   4. finalise:  one CTA adds every partial in a fixed order in fp64 (repeated calls are bit-identical), writes
//                 (loss, bce, dice, l1) and the record the backward reads.
// Backward, one element-wise pass: grad_b from ATen's BCE backward with weight (P + S) / denominator, S = C where
// l > tau, C r / T where l = tau > 0 (r = k - above: the tied remainder split evenly), 0 otherwise; grad_tb from the
// dice quotient; grad_t = sign(t - z) w / sum w.  The upstream gradients of all four outputs are read from device memory.
#include "common.cuh"
#include <math.h>

namespace {
using namespace mr;

constexpr int kPix = 128;             // pixels (threads) per block of the statistics kernel
constexpr int kThreads = 256;         // element-wise / histogram kernels
constexpr int kMaxBlocks = 1024;      // grid cap of the statistics and histogram kernels (= partial rows)
constexpr int kMaxN = 256;            // g staged in shared memory: N * kPix floats
constexpr int kBins = 2048;

struct Rec { float l; unsigned short c, p; };                 // one per (sample j, pixel q): 8 bytes
struct StatPart { double pl, inter, tbm, gm, l1, w; unsigned long long pos, negc; };
struct Select {
    unsigned long long k, krem, above, tie, pos, negc;
    unsigned int prefix, pmask, tau_bits, active;
};
struct BwdRec { double denom, inter, uni, sum_w, tie_frac; unsigned int tau_bits, pad; };

struct Layout {
    size_t rec, stat, hist, sel, state, bwd, total;
};
inline size_t al(size_t x) { return (x + 255) & ~(size_t)255; }
inline Layout layout(int64_t N, int64_t HW) {
    Layout L;
    size_t o = 0;
    L.rec = o;   o += al(sizeof(Rec) * (size_t)N * (size_t)HW);
    L.stat = o;  o += al(sizeof(StatPart) * kMaxBlocks);
    L.hist = o;  o += al(sizeof(unsigned long long) * 3 * kBins);
    L.sel = o;   o += al(sizeof(double) * kMaxBlocks);
    L.state = o; o += al(sizeof(Select));
    L.bwd = o;   o += al(sizeof(BwdRec));
    L.total = o;
    return L;
}

__device__ __forceinline__ float bce_elem(float b, float g) {
    // ATen binary_cross_entropy (reduction='none'), CUDA and CPU kernels alike
    const float lb = fmaxf(logf(b), -100.f);
    const float l1b = fmaxf(log1pf(-b), -100.f);
    return (g - 1.f) * l1b - g * lb;
}
// .byte() of a product of two values in [0, 1]: 1 exactly where the product is >= 1
__device__ __forceinline__ unsigned u8(float x) { return x >= 1.f ? 1u : 0u; }
__device__ __forceinline__ unsigned key_of(float l) { return __float_as_uint(l) & 0x7fffffffu; }   // l >= 0 (-0 -> +0)

// Fixed-order block sums (shuffle tree inside a warp, then warps in order).
template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    return v;
}
template <typename T>
__device__ T block_sum(T v, T *red) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) red[w] = v;
    __syncthreads();
    T t = 0;
    if (threadIdx.x == 0)
        for (int i = 0; i < nw; ++i) t += red[i];
    return t;                                                  // valid in thread 0
}

__global__ void __launch_bounds__(kThreads)
db_maps_fwd_kernel(const float *__restrict__ xb, const float *__restrict__ xt, int64_t n, float k,
                   float *__restrict__ b, float *__restrict__ t, float *__restrict__ tb) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const float bv = 1.f / (1.f + expf(-xb[e]));
        const float tv = 1.f / (1.f + expf(-xt[e]));
        b[e] = bv;
        t[e] = tv;
        tb[e] = 1.f / (1.f + expf(-k * (bv - tv)));
    }
}

__global__ void __launch_bounds__(kThreads)
db_maps_bwd_kernel(const float *__restrict__ gb, const float *__restrict__ gt, const float *__restrict__ gtb,
                   const float *__restrict__ b, const float *__restrict__ t, const float *__restrict__ tb, int64_t n,
                   float k, float *__restrict__ gxb, float *__restrict__ gxt) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const float bv = b[e], tv = t[e], y = tb[e];
        // d tb / d(b - t) = k tb^2 exp(-k (b - t)) = k tb (1 - tb), written with exp so that it keeps its precision as tb -> 1
        const float ex = expf(-k * (bv - tv));
        const float gd = (gtb ? gtb[e] : 0.f) * k * y * (ex * y);
        const float g1 = (gb ? gb[e] : 0.f) + gd, g2 = (gt ? gt[e] : 0.f) - gd;
        gxb[e] = g1 * (1.f - bv) * bv;                         // ATen sigmoid_backward
        gxt[e] = g2 * (1.f - tv) * tv;
    }
}

// 1. Statistics.  Block = kPix pixels; dynamic shared memory = N * kPix floats of g (a thread reads only its own column).
__global__ void __launch_bounds__(kPix)
db_stats_kernel(const float *__restrict__ b, const float *__restrict__ t, const float *__restrict__ tb,
                const float *__restrict__ g, const float *__restrict__ m, const float *__restrict__ z,
                const float *__restrict__ w, int N, int64_t HW, Rec *__restrict__ rec, StatPart *__restrict__ part,
                unsigned long long *__restrict__ hist) {
    extern __shared__ float sg[];
    __shared__ double redd[kPix / 32];
    __shared__ unsigned long long redu[kPix / 32];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 3 * kBins; i += gridDim.x * blockDim.x) hist[i] = 0ull;
    double s_pl = 0, s_i = 0, s_tbm = 0, s_gm = 0, s_l1 = 0, s_w = 0;
    unsigned long long s_pos = 0, s_neg = 0;
    const int tid = threadIdx.x;
    for (int64_t q = (int64_t)blockIdx.x * kPix + tid; q < HW; q += (int64_t)gridDim.x * kPix) {
        for (int i = 0; i < N; ++i) sg[i * kPix + tid] = g[(int64_t)i * HW + q];
        for (int j = 0; j < N; ++j) {
            const int64_t e = (int64_t)j * HW + q;
            const float mj = m[e];
            unsigned P = 0, C = 0;
            for (int i = 0; i < N; ++i) {
                const float gi = sg[i * kPix + tid];
                P += u8(gi * mj);
                C += u8((1.f - gi) * mj);
            }
            const float gj = sg[j * kPix + tid];
            const float l = bce_elem(b[e], gj);
            Rec r; r.l = l; r.c = (unsigned short)C; r.p = (unsigned short)P;
            rec[e] = r;
            s_pl += (double)P * (double)l;
            s_pos += P;
            s_neg += C;
            const float tbj = tb[e];
            s_i += (double)(tbj * gj * mj);
            s_tbm += (double)(tbj * mj);
            s_gm += (double)(gj * mj);
            const float wj = w[e];
            s_l1 += (double)(fabsf(t[e] - z[e]) * wj);
            s_w += (double)wj;
        }
    }
    StatPart p;
    p.pl = block_sum(s_pl, redd);
    p.inter = block_sum(s_i, redd);
    p.tbm = block_sum(s_tbm, redd);
    p.gm = block_sum(s_gm, redd);
    p.l1 = block_sum(s_l1, redd);
    p.w = block_sum(s_w, redd);
    p.pos = block_sum(s_pos, redu);
    p.negc = block_sum(s_neg, redu);
    if (tid == 0) part[blockIdx.x] = p;
}

__device__ __forceinline__ void digit_of(int pass, int &shift, int &bits) {
    shift = pass == 0 ? 21 : (pass == 1 ? 10 : 0);
    bits = pass == 2 ? 10 : 11;
}

// 2a. Weighted histogram of the current digit over the records whose higher digits equal the prefix.
__global__ void __launch_bounds__(kThreads)
db_hist_kernel(const Rec *__restrict__ rec, int64_t n, int pass, const Select *__restrict__ st,
               unsigned long long *__restrict__ hist) {
    __shared__ unsigned long long h[kBins];
    unsigned prefix = 0, pmask = 0;                         // pass 0 runs before k is known and takes every record
    if (pass > 0) {
        if (!st->active) return;
        prefix = st->prefix;
        pmask = st->pmask;
    }
    int shift, bits;
    digit_of(pass, shift, bits);
    const unsigned nb = 1u << bits;
    for (int i = threadIdx.x; i < (int)nb; i += blockDim.x) h[i] = 0ull;
    __syncthreads();
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const Rec r = rec[e];
        if (r.c == 0) continue;
        const unsigned key = key_of(r.l);
        if ((key & pmask) != prefix) continue;
        atomicAdd(&h[(key >> shift) & (nb - 1)], (unsigned long long)r.c);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < (int)nb; i += blockDim.x)
        if (h[i]) atomicAdd(&hist[pass * kBins + i], h[i]);
}

// 2b. One CTA of 1024 threads: pick the digit at which the cumulative weight from the top reaches the remaining rank.
//     Pass 0 first reduces pos and sum C (integers: exact in any order) and sets k.
__global__ void __launch_bounds__(1024)
db_narrow_kernel(const StatPart *__restrict__ part, int nparts, float neg_ratio, int pass,
                 const unsigned long long *__restrict__ hist, Select *__restrict__ st) {
    __shared__ unsigned long long red[32];
    __shared__ unsigned long long wsum[32];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (pass == 0) {
        unsigned long long a = 0, c = 0;
        for (int i = tid; i < nparts; i += blockDim.x) { a += part[i].pos; c += part[i].negc; }
        a = block_sum(a, red);
        c = block_sum(c, red);
        if (tid == 0) {
            // int(positive_count * negative_ratio) in Python: a double product, truncated
            const unsigned long long cap = (unsigned long long)floor((double)a * (double)neg_ratio);
            const unsigned long long k = c < cap ? c : cap;
            Select s;
            s.k = k; s.krem = k; s.above = 0; s.tie = 0; s.pos = a; s.negc = c;
            s.prefix = 0; s.pmask = 0; s.tau_bits = 0xffffffffu; s.active = k > 0;
            *st = s;
        }
        __syncthreads();
    }
    if (!st->active) return;
    int shift, bits;
    digit_of(pass, shift, bits);
    const int nb = 1 << bits, per = nb / 1024;
    const unsigned long long *hp = hist + pass * kBins;
    unsigned long long s = 0;
    for (int e = 0; e < per; ++e) s += hp[nb - 1 - tid * per - e];
    // exclusive scan over threads (thread 0 owns the highest bins)
    unsigned long long incl = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) wsum[wid] = incl;
    __syncthreads();
    if (wid == 0) {
        unsigned long long v = wsum[lane], iv = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long u = __shfl_up_sync(0xffffffffu, iv, o);
            if (lane >= o) iv += u;
        }
        wsum[lane] = iv - v;
    }
    __syncthreads();
    const unsigned long long excl = wsum[wid] + incl - s;
    const unsigned long long krem = st->krem;
    __syncthreads();
    if (krem > excl && krem <= excl + s) {
        unsigned long long c = excl;
        for (int e = 0; e < per; ++e) {
            const int bin = nb - 1 - tid * per - e;
            const unsigned long long hcount = hp[bin];
            if (krem <= c + hcount) {
                Select n = *st;
                n.above += c;
                n.krem = krem - c;
                n.tie = hcount;
                n.prefix |= (unsigned)bin << shift;
                n.pmask |= (unsigned)(nb - 1) << shift;
                if (pass == 2) n.tau_bits = n.prefix;
                *st = n;
                break;
            }
            c += hcount;
        }
    }
}

// 3. Per-block sums of C l over the records strictly above tau.
__global__ void __launch_bounds__(kThreads)
db_selsum_kernel(const Rec *__restrict__ rec, int64_t n, const Select *__restrict__ st, double *__restrict__ part) {
    __shared__ double red[kThreads / 32];
    const unsigned tau = st->tau_bits;
    double s = 0;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const Rec r = rec[e];
        if (r.c != 0 && key_of(r.l) > tau) s += (double)r.c * (double)r.l;
    }
    s = block_sum(s, red);
    if (threadIdx.x == 0) part[blockIdx.x] = s;
}

// 4. One CTA: fixed-order fp64 reduction of every partial, the four outputs and the backward's record.
__global__ void __launch_bounds__(kThreads)
db_finalize_kernel(const StatPart *__restrict__ part, int nparts, const double *__restrict__ sel, int nsel,
                   const Select *__restrict__ st, float eps, float bce_eps, float l1_scale, float bce_scale,
                   float *__restrict__ out, BwdRec *__restrict__ bw) {
    __shared__ double red[kThreads / 32];
    double a0 = 0, a1 = 0, a2 = 0, a3 = 0, a4 = 0, a5 = 0, a6 = 0;
    for (int i = threadIdx.x; i < nparts; i += blockDim.x) {
        a0 += part[i].pl; a1 += part[i].inter; a2 += part[i].tbm; a3 += part[i].gm; a4 += part[i].l1; a5 += part[i].w;
    }
    for (int i = threadIdx.x; i < nsel; i += blockDim.x) a6 += sel[i];
    const double pl = block_sum(a0, red), inter = block_sum(a1, red), tbm = block_sum(a2, red), gm = block_sum(a3, red);
    const double l1s = block_sum(a4, red), sw = block_sum(a5, red), above_sum = block_sum(a6, red);
    if (threadIdx.x != 0) return;
    const Select s = *st;
    double topk = above_sum, tie_frac = 0.0;
    if (s.active) {
        const double tau = (double)__uint_as_float(s.tau_bits);
        topk += (double)s.krem * tau;
        tie_frac = (double)s.krem / (double)s.tie;
    }
    const double denom = (double)s.pos + (double)s.k + (double)bce_eps;
    const double bce = (pl + topk) / denom;
    const double uni = tbm + gm + (double)eps;
    const double dice = 1.0 - 2.0 * inter / uni;
    const double l1 = l1s / sw;                              // NaN when sum w = 0, as in the reference
    out[0] = (float)(dice + (double)l1_scale * l1 + (double)bce_scale * bce);
    out[1] = (float)bce;
    out[2] = (float)dice;
    out[3] = (float)l1;
    bw->denom = denom; bw->inter = inter; bw->uni = uni; bw->sum_w = sw; bw->tie_frac = tie_frac;
    bw->tau_bits = s.active ? s.tau_bits : 0xffffffffu;
}

__global__ void __launch_bounds__(kThreads)
db_loss_bwd_kernel(const float *__restrict__ gout, const float *__restrict__ b, const float *__restrict__ t,
                   const float *__restrict__ g, const float *__restrict__ m, const float *__restrict__ z,
                   const float *__restrict__ w, const Rec *__restrict__ rec, const BwdRec *__restrict__ bwp, int64_t n,
                   float l1_scale, float bce_scale, float *__restrict__ gb, float *__restrict__ gt,
                   float *__restrict__ gtb) {
    const BwdRec bw = *bwp;
    const double go0 = gout[0];
    const double cb = go0 * (double)bce_scale + (double)gout[1];
    const double cd = go0 + (double)gout[2];
    const double cl = go0 * (double)l1_scale + (double)gout[3];
    const float fb = (float)(cb / bw.denom);
    const double fd = -2.0 * cd / (bw.uni * bw.uni);
    const float fl = (float)(cl / bw.sum_w);
    const float tie = (float)bw.tie_frac;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const Rec r = rec[e];
        const unsigned key = key_of(r.l);
        float S = 0.f;
        if (r.c != 0) {
            if (key > bw.tau_bits) S = (float)r.c;
            else if (key == bw.tau_bits && key != 0u) S = (float)r.c * tie;
        }
        const float bv = b[e], gv = g[e], mv = m[e];
        gb[e] = (((float)r.p + S) * fb) * (bv - gv) / fmaxf((1.f - bv) * bv, 1e-12f);      // ATen BCE backward
        gtb[e] = (float)(fd * (double)mv * ((double)gv * bw.uni - bw.inter));          // g U - I cancels: fp64
        const float d = t[e] - z[e];
        gt[e] = fl * (float)((d > 0.f) - (d < 0.f)) * w[e];
    }
}

inline int grid_for(int64_t n, int threads, int cap) {
    int64_t g = ceil_div(n, threads);
    if (g > cap) g = cap;
    return (int)(g < 1 ? 1 : g);
}

}  // namespace

extern "C" {

int mr_db_maps_fwd_f32(const float *x_b, const float *x_t, int64_t n, float k, float *b, float *t, float *tb, void *stream) {
    if (n < 0) return MR_ERR_BAD_SHAPE;
    if (n == 0) return MR_OK;
    if (!x_b || !x_t || !b || !t || !tb) return MR_ERR_NULL_POINTER;
    db_maps_fwd_kernel<<<grid_for(n, kThreads, 148 * 16), kThreads, 0, (cudaStream_t)stream>>>(x_b, x_t, n, k, b, t, tb);
    return check_launch("db_maps_fwd_kernel");
}

int mr_db_maps_bwd_f32(const float *grad_b, const float *grad_t, const float *grad_tb, const float *b, const float *t,
                       const float *tb, int64_t n, float k, float *grad_xb, float *grad_xt, void *stream) {
    if (n < 0) return MR_ERR_BAD_SHAPE;
    if (n == 0) return MR_OK;
    if (!b || !t || !tb || !grad_xb || !grad_xt) return MR_ERR_NULL_POINTER;
    db_maps_bwd_kernel<<<grid_for(n, kThreads, 148 * 16), kThreads, 0, (cudaStream_t)stream>>>(
        grad_b, grad_t, grad_tb, b, t, tb, n, k, grad_xb, grad_xt);
    return check_launch("db_maps_bwd_kernel");
}

int64_t mr_db_loss_workspace_bytes(int64_t N, int64_t HW) {
    if (N <= 0 || HW <= 0) return 0;
    return (int64_t)layout(N, HW).total;
}

int mr_db_loss_fwd_f32(const float *b, const float *t, const float *tb, const float *gt, const float *mask,
                       const float *thresh_map, const float *thresh_mask, int64_t N, int64_t HW, float eps,
                       float l1_scale, float bce_scale, float negative_ratio, float bce_eps, void *workspace,
                       int64_t workspace_bytes, float *out, void *stream) {
    if (N <= 0 || HW <= 0) return MR_ERR_BAD_SHAPE;
    if (N > kMaxN) return MR_ERR_UNSUPPORTED;
    if (!b || !t || !tb || !gt || !mask || !thresh_map || !thresh_mask || !workspace || !out) return MR_ERR_NULL_POINTER;
    const Layout L = layout(N, HW);
    if (workspace_bytes < (int64_t)L.total) return MR_ERR_BAD_SHAPE;
    char *ws = (char *)workspace;
    Rec *rec = (Rec *)(ws + L.rec);
    StatPart *part = (StatPart *)(ws + L.stat);
    unsigned long long *hist = (unsigned long long *)(ws + L.hist);
    double *sel = (double *)(ws + L.sel);
    Select *st = (Select *)(ws + L.state);
    BwdRec *bw = (BwdRec *)(ws + L.bwd);
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t n = N * HW;
    const size_t smem = sizeof(float) * (size_t)N * kPix;
    int rc = ensure_dyn_smem((const void *)db_stats_kernel, smem, "db_stats_kernel smem");
    if (rc) return rc;
    const int gs = grid_for(HW, kPix, kMaxBlocks);
    db_stats_kernel<<<gs, kPix, smem, s>>>(b, t, tb, gt, mask, thresh_map, thresh_mask, (int)N, HW, rec, part, hist);
    if ((rc = check_launch("db_stats_kernel"))) return rc;
    const int gh = grid_for(n, kThreads * 8, kMaxBlocks);
    for (int pass = 0; pass < 3; ++pass) {                 // pass 0's narrowing also sets k from the partial counts
        db_hist_kernel<<<gh, kThreads, 0, s>>>(rec, n, pass, st, hist);
        if ((rc = check_launch("db_hist_kernel"))) return rc;
        db_narrow_kernel<<<1, 1024, 0, s>>>(part, gs, negative_ratio, pass, hist, st);
        if ((rc = check_launch("db_narrow_kernel"))) return rc;
    }
    db_selsum_kernel<<<gh, kThreads, 0, s>>>(rec, n, st, sel);
    if ((rc = check_launch("db_selsum_kernel"))) return rc;
    db_finalize_kernel<<<1, kThreads, 0, s>>>(part, gs, sel, gh, st, eps, bce_eps, l1_scale, bce_scale, out, bw);
    return check_launch("db_finalize_kernel");
}

int mr_db_loss_bwd_f32(const float *grad_out, const float *b, const float *t, const float *gt, const float *mask,
                       const float *thresh_map, const float *thresh_mask, int64_t N, int64_t HW, float l1_scale,
                       float bce_scale, const void *workspace, int64_t workspace_bytes, float *grad_b, float *grad_t,
                       float *grad_tb, void *stream) {
    if (N <= 0 || HW <= 0) return MR_ERR_BAD_SHAPE;
    if (!grad_out || !b || !t || !gt || !mask || !thresh_map || !thresh_mask || !workspace || !grad_b || !grad_t || !grad_tb)
        return MR_ERR_NULL_POINTER;
    const Layout L = layout(N, HW);
    if (workspace_bytes < (int64_t)L.total) return MR_ERR_BAD_SHAPE;
    const char *ws = (const char *)workspace;
    const int64_t n = N * HW;
    db_loss_bwd_kernel<<<grid_for(n, kThreads, 148 * 16), kThreads, 0, (cudaStream_t)stream>>>(
        grad_out, b, t, gt, mask, thresh_map, thresh_mask, (const Rec *)(ws + L.rec), (const BwdRec *)(ws + L.bwd), n,
        l1_scale, bce_scale, grad_b, grad_t, grad_tb);
    return check_launch("db_loss_bwd_kernel");
}

}  // extern "C"
