// K2: bilinear upsample + softmax cross-entropy, forward AND backward in one pass.
//
// Replaces reference model/loss.py:19-20 (AuxiliaryLoss: F.interpolate(bilinear, size=H) +
// CrossEntropyLoss) / model/final.py:44 + engine.py:94, and their autograd backward
// (engine.py:100).  The upsampled [B,C,H,W] tensor (2.5 GB at B=16, C=150, 512^2) never
// exists: each CTA stages the low-resolution logits of a pixel tile in shared memory,
// evaluates the softmax of every upsampled pixel in registers and scatters
// (softmax - onehot) * g back through the four bilinear taps into a shared-memory gradient
// tile that is flushed once.
//
// Fast path (scale 4; 8 / 16 take the strip kernels): one thread owns a 4x4 pixel block whose 16 pixels
// share the same 2x2 taps (common.cuh: BlockGeom).  Inside the block the upsampled logit is a
// bilinear polynomial  l(i,j) = l00 + i*P + j*Q + i*j*T, so
//     exp(l(i,j) - M) = E00 * p^i * q^j * t^(i*j)        (4 ex2 per class per 16 pixels,
// the rest are multiplies), with M = max over classes of the block's four taps (an upper
// bound of every pixel's max - a valid softmax shift).  If a pixel's sum under/overflows
// with that shared shift (logits spanning > ~80 within one cell) the thread falls back to
// the exact per-pixel path.  The scatter uses the moments sum(g), sum(i g), sum(j g),
// sum(ij g) instead of 64 weighted adds.
//
// Generic path (any size): one pixel per thread, taps from global, global atomics.
#include "common.cuh"
#include "k2_strip.cuh"
#include <type_traits>
#include <stdlib.h>

namespace lc2is {

// ---------------------------------------------------------------------------------------------
// count valid labels (the 'mean' denominator)
__global__ void k2_count_valid_kernel(const long long* __restrict__ labels, long long n, long long C, long long ignore,
                                      unsigned long long* __restrict__ out) {
    auto counted = [&](long long v) { return (unsigned long long)v < (unsigned long long)C && v != ignore; };
    long long cnt = 0;
    const long long stride = (long long)gridDim.x * blockDim.x;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    // 2 labels (16 B) per load when aligned
    const long long n2 = n / 2;
    const longlong2* l2 = reinterpret_cast<const longlong2*>(labels);
    for (long long k = i; k < n2; k += stride) {
        longlong2 v = __ldg(l2 + k);
        cnt += (int)counted(v.x) + (int)counted(v.y);
    }
    if (i == 0 && (n & 1)) cnt += counted(labels[n - 1]);
    int c = (int)cnt;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    __shared__ int ws[32];
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x < 32) {
        int v = threadIdx.x < (blockDim.x >> 5) ? ws[threadIdx.x] : 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (threadIdx.x == 0 && v) atomicAdd(out, (unsigned long long)v);
    }
}

// sum of the class weights of the counted labels (the 'mean' denominator of the weighted cross-entropy); weight = null
// counts them.  Accumulated in double.
__global__ void k2_weight_sum_kernel(const long long* __restrict__ labels, long long n, long long C, long long ignore,
                                     const float* __restrict__ weight, double* __restrict__ out) {
    auto wl = [&](long long v) {
        return (unsigned long long)v < (unsigned long long)C && v != ignore ? (double)k2_class_weight(weight, (int)v) : 0.0;
    };
    double acc = 0.0;
    const long long stride = (long long)gridDim.x * blockDim.x;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long n2 = n / 2;
    const longlong2* l2 = reinterpret_cast<const longlong2*>(labels);
    for (long long k = i; k < n2; k += stride) {
        longlong2 v = __ldg(l2 + k);
        acc += wl(v.x) + wl(v.y);
    }
    if (i == 0 && (n & 1)) acc += wl(labels[n - 1]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    __shared__ double ws[32];
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x < 32) {
        double v = threadIdx.x < (blockDim.x >> 5) ? ws[threadIdx.x] : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (threadIdx.x == 0 && v != 0.0) atomicAdd(out, v);
    }
}

// ---------------------------------------------------------------------------------------------
// Geometry of the fast path (scale 4).  Thread (ty,tx) of a CTA owns the 4x4-pixel block that interpolates between
// the source cells (ky,kx) = (GY0+ty-1, GX0+tx-1) .. (ky+1, kx+1), index-clamped to the image; there are (h+1) x (w+1)
// blocks per image.  The CTA stages the (tgy+1) x (tgx+1) source cells its tgy x tgx blocks read, and each thread
// sends its four tap gradients to L2 as four float reductions per class.
struct K2Params {
    const float* low;            // [B,C,h,w]
    const long long* labels;     // [B,H,W]
    float* grad_low;             // [B,C,h,w] (pre-zeroed; accumulated with global reductions) or null
    double* loss_sum;
    const float* grad_scale;     // device scalar or null
    long long ignore_index;
    int B, C, h, w, H, W;
    int s, off, q;                // scale, pixel offset of the block grid, offset of block 0
    int tgy, tgx;                 // blocks per CTA
    float rs;
    const float* weight;          // WT: class weights [C] (null = all 1); 1 - eps, eps / C (k2_strip.cuh: k2_class_weight)
    float one_m_eps, eps_c;
};

// exp-polynomial of one class inside a 4x4 block: exp(l(i,j) - M) = E * p^i * q^j * t^(i*j)
struct Poly { float E, p, q, t; };
__device__ __forceinline__ Poly k2_poly(float a, float b, float cc, float d, float ly0, float lx0, float k1,
                                        float k2, float Mk) {
    const float da = cc - a, db = d - b, dd = db - da;
    const float L0 = fmaf(ly0, da, a), R0 = fmaf(ly0, db, b);
    const float rl = R0 - L0;
    const float l00 = fmaf(lx0, rl, L0);
    Poly P;
    P.q = ex2f(rl * k1);
    P.p = ex2f(fmaf(lx0, dd, da) * k1);
    P.t = ex2f(dd * k2);
    P.E = ex2f(fmaf(l00, LOG2E, -Mk));
    return P;
}

// WT: the weighted / label-smoothed form (k2_strip.cuh: k2_class_weight): U = g*a / S, a*lse, a (1-eps) w_t scale on the
// -onehot runs, and the smoothing terms through V = the thread's summed tap weights (loss: V.Q with Q = sum_c w_c * taps
// from the max-tap sweep; gradient: -g (eps/C) w_c V per tap and class).
template <bool WT = false>
__global__ void __launch_bounds__(128)
k2_fast_kernel(const K2Params P) {
    extern __shared__ float smem[];
    const int C = P.C;
    const int ncx = P.tgx + 1, ncy = P.tgy + 1;
    const int cs = ncy * ncx;                               // class stride (floats) in the tile
    const int nthr = blockDim.x;
    float* st = smem;

    const int n = blockIdx.z;
    const int GY0 = blockIdx.y * P.tgy, GX0 = blockIdx.x * P.tgx;
    const int cy0 = GY0 - 1, cx0 = GX0 - 1;                 // first cell of the tile (may be -1)
    const float* lowb = P.low + (size_t)n * C * P.h * P.w;

    // ---- stage the source tile st[c][ncy][ncx]; cells outside the image hold 0 ---------------------
    // (a thread owns tile cells r, r + nthr, ... and walks the classes: no integer division per copied element - the
    // staging loop was a third of this kernel's instructions)
    {
        const size_t plane = (size_t)P.h * P.w;
        for (int r = threadIdx.x; r < cs; r += nthr) {
            const int i = r / ncx, j = r - i * ncx;
            const int gy = cy0 + i, gx = cx0 + j;
            float* dst = st + r;
            if (gy >= 0 && gy < P.h && gx >= 0 && gx < P.w) {
                const float* src = lowb + (size_t)gy * P.w + gx;
#pragma unroll 4
                for (int c = 0; c < C; ++c) cp_async4(dst + (size_t)c * cs, src + (size_t)c * plane);
            } else {
                for (int c = 0; c < C; ++c) dst[(size_t)c * cs] = 0.f;
            }
        }
    }
    cp_async_wait_all();
    __syncthreads();

    // ---- per-thread block setup ---------------------------------------------------------------------
    const int g = threadIdx.x;
    const int tgy = g / P.tgx, tgx = g - tgy * P.tgx;
    const int ky = GY0 + tgy - 1, kx = GX0 + tgx - 1;       // top-left tap of the block (-1 .. h-1)
    const int by = ky + P.q, bx = kx + P.q;
    const int y0 = 4 * by - P.off, x0 = 4 * bx - P.off;
    const float gs = P.grad_scale ? __ldg(P.grad_scale) : 1.f;
    const float rs = P.rs;
    const bool group_in = ky < P.h && kx < P.w;             // block exists in this image
    int lab[16];
    bool any = false;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            int y = y0 + i, x = x0 + j;
            int l = -1;
            if (group_in && y >= 0 && y < P.H && x >= 0 && x < P.W) {
                long long t = __ldg(P.labels + ((size_t)n * P.H + y) * P.W + x);
                if (t != P.ignore_index && t >= 0 && t < C) l = (int)t;
            }
            lab[i * 4 + j] = l;
            any |= l >= 0;
        }
    // clamped tap cells (global)
    const int Ya = clampi(ky, 0, P.h - 1), Yb = clampi(ky + 1, 0, P.h - 1);
    const int Xa = clampi(kx, 0, P.w - 1), Xb = clampi(kx + 1, 0, P.w - 1);
    // tile offsets of the four taps
    int oa = (Ya - cy0) * ncx + (Xa - cx0), ob = (Ya - cy0) * ncx + (Xb - cx0);
    int oc = (Yb - cy0) * ncx + (Xa - cx0), od = (Yb - cy0) * ncx + (Xb - cx0);
    if (!group_in) oa = ob = oc = od = 0;
    auto taps = [&](int c, float& a, float& b, float& cc, float& d) {
        const float* p = st + (size_t)c * cs;
        a = p[oa]; b = p[ob]; cc = p[oc]; d = p[od];
    };
    // lambda of the block's first row / column ((y0+0.5)*rs-0.5-ky is exact for power-of-2 s)
    const float ly0 = ((float)y0 + 0.5f) * rs - 0.5f - (float)ky;
    const float lx0 = ((float)x0 + 0.5f) * rs - 0.5f - (float)kx;

    // ---- softmax shift: M = max over classes of the block's taps (>= every pixel's max) -----------
    float mx = -INFINITY, mn = INFINITY;
    float4 wq = make_float4(0.f, 0.f, 0.f, 0.f);            // WT: sum_c w_c * taps
    float wsum = 0.f;                                       // WT: W = sum_c w_c
    for (int c = 0; c < C; ++c) {
        float a, b, cc, d;
        taps(c, a, b, cc, d);
        mx = fmaxf(mx, fmaxf(fmaxf(a, b), fmaxf(cc, d)));
        mn = fminf(mn, fminf(fminf(a, b), fminf(cc, d)));
        if constexpr (WT) {
            const float wc = k2_class_weight(P.weight, c);
            wq.x = fmaf(wc, a, wq.x); wq.y = fmaf(wc, b, wq.y); wq.z = fmaf(wc, cc, wq.z); wq.w = fmaf(wc, d, wq.w);
            wsum += wc;
        }
    }
    const float M = mx;
    // fast path needs a bounded logit range inside the block (no under/overflow of the shared-shift
    // polynomial); otherwise - or on inf/NaN - the whole warp takes the exact per-pixel path.
    bool slow = any && !((mx - mn) < K2_FAST_RANGE);
    slow = __any_sync(0xffffffffu, slow);
    const bool warp_any = __any_sync(0xffffffffu, any);
    const float Mk = M * LOG2E;
    const float k1 = rs * LOG2E, k2 = rs * rs * LOG2E;

    float U[16];                      // pass A: S(i,j) = sum_c exp(l_c - shift); then U = g / S
    float Mp[16];                     // per-pixel shift (== M on the fast path)
    float loss = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) { U[i] = 0.f; Mp[i] = M; }

    if (warp_any && !slow) {
        // ---- pass A (fast): rows (0,1) and (2,3) packed; S(i,j) += e_i * q_i^j -------------------------
        float2 S01[4], S23[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) { S01[j] = make_float2(0.f, 0.f); S23[j] = make_float2(0.f, 0.f); }
#pragma unroll 4
        for (int c = 0; c < C; ++c) {
            float a, b, cc, d;
            taps(c, a, b, cc, d);
            const Poly y = k2_poly(a, b, cc, d, ly0, lx0, k1, k2, Mk);
            const float2 e01 = make_float2(y.E, y.E * y.p), q01 = make_float2(y.q, y.q * y.t);
            const float2 e23 = fmul2(e01, bc2(y.p * y.p)), q23 = fmul2(q01, bc2(y.t * y.t));
            const float2 qq01 = fmul2(q01, q01), qq23 = fmul2(q23, q23);
            const float2 q301 = fmul2(qq01, q01), q323 = fmul2(qq23, q23);
            S01[0] = fadd2(S01[0], e01);           S23[0] = fadd2(S23[0], e23);
            S01[1] = ffma2(e01, q01, S01[1]);      S23[1] = ffma2(e23, q23, S23[1]);
            S01[2] = ffma2(e01, qq01, S01[2]);     S23[2] = ffma2(e23, qq23, S23[2]);
            S01[3] = ffma2(e01, q301, S01[3]);     S23[3] = ffma2(e23, q323, S23[3]);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            U[0 * 4 + j] = S01[j].x; U[1 * 4 + j] = S01[j].y;
            U[2 * 4 + j] = S23[j].x; U[3 * 4 + j] = S23[j].y;
        }
        bool bad = false;
#pragma unroll
        for (int i = 0; i < 16; ++i)
            if (lab[i] >= 0) bad |= !((U[i] >= S_MIN) && (U[i] <= 3.0e38f));
        slow = __any_sync(0xffffffffu, bad);
    }
    if (warp_any && slow) {
        // ---- pass A (exact): per-pixel max and sum -----------------------------------------------------
#pragma unroll 1
        for (int pix = 0; pix < 16; ++pix) {
            const float ly = ly0 + (float)(pix >> 2) * rs, lx = lx0 + (float)(pix & 3) * rs;
            float m = -INFINITY;
            for (int c = 0; c < C; ++c) {
                float a, b, cc, d;
                taps(c, a, b, cc, d);
                const float L = fmaf(ly, cc - a, a), R = fmaf(ly, d - b, b);
                m = fmaxf(m, fmaf(lx, R - L, L));
            }
            float sum = 0.f;
            for (int c = 0; c < C; ++c) {
                float a, b, cc, d;
                taps(c, a, b, cc, d);
                const float L = fmaf(ly, cc - a, a), R = fmaf(ly, d - b, b);
                sum += ex2f((fmaf(lx, R - L, L) - m) * LOG2E);
            }
#pragma unroll
            for (int i = 0; i < 16; ++i)
                if (i == pix) { Mp[i] = m; U[i] = sum; }
        }
    }
    // ---- loss and per-pixel gradient scale U = g / S ----------------------------------------------------
    const int S2 = 2 * P.s;
    const int lyi0 = 2 * y0 + 1 - P.s - S2 * ky, lxi0 = 2 * x0 + 1 - P.s - S2 * kx;   // lambda * 2s of pixel (0,0)
    float4 kv = make_float4(0.f, 0.f, 0.f, 0.f);            // WT: -g (eps/C) V of the four taps
    if (any) {
        int va = 0, vb = 0, vc = 0, vd = 0;                 // WT: V in units of 1 / (2s)^2
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int t = lab[i * 4 + j];
                float uu = 0.f;
                if (t >= 0) {
                    const float ly = ly0 + (float)i * rs, lx = lx0 + (float)j * rs;
                    float a, b, cc, d;
                    taps(t, a, b, cc, d);
                    const float L = fmaf(ly, cc - a, a), R = fmaf(ly, d - b, b);
                    if constexpr (WT) {
                        const float wt = P.one_m_eps * k2_class_weight(P.weight, t);
                        const float aw = fmaf(P.eps_c, wsum, wt);
                        loss += aw * (logf(U[i * 4 + j]) + Mp[i * 4 + j]) - wt * fmaf(lx, R - L, L);
                        uu = gs * aw / U[i * 4 + j];
                        const int lyi = lyi0 + 2 * i, lxi = lxi0 + 2 * j;
                        va += (S2 - lyi) * (S2 - lxi); vb += (S2 - lyi) * lxi;
                        vc += lyi * (S2 - lxi);        vd += lyi * lxi;
                    } else {
                        loss += logf(U[i * 4 + j]) + Mp[i * 4 + j] - fmaf(lx, R - L, L);
                        uu = gs / U[i * 4 + j];
                    }
                }
                U[i * 4 + j] = uu;
            }
        if constexpr (WT) {
            // smoothing: -(eps/C) sum over the counted pixels of the interpolated sum_c w_c x_c
            const float rn = 1.f / (float)(S2 * S2);
            loss = fmaf(-P.eps_c * rn, (float)va * wq.x + (float)vb * wq.y + (float)vc * wq.z + (float)vd * wq.w, loss);
            const float k = -gs * P.eps_c * rn;
            kv = make_float4(va ? k * (float)va : 0.f, vb ? k * (float)vb : 0.f, vc ? k * (float)vc : 0.f,
                             vd ? k * (float)vd : 0.f);
        }
    } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) U[i] = 0.f;
    }

    // ---- pass B: scatter softmax * U through the taps (warp-collective) ---------------------------------
    float* gb = P.grad_low ? P.grad_low + (size_t)n * C * P.h * P.w : nullptr;
    if (gb && warp_any) {
        const size_t plane = (size_t)P.h * P.w;
        float* gA = gb + (size_t)Ya * P.w + Xa; float* gB = gb + (size_t)Ya * P.w + Xb;
        float* gC = gb + (size_t)Yb * P.w + Xa; float* gD = gb + (size_t)Yb * P.w + Xb;
        auto emit = [&](int c, float G, float Gx, float Gy, float Gxy) {
            const float X = fmaf(rs, Gx, lx0 * G);                        // sum lambda_x g
            const float Y = fmaf(rs, Gy, ly0 * G);                        // sum lambda_y g
            const float XY = fmaf(ly0, X, rs * fmaf(rs, Gxy, lx0 * Gy));  // sum lambda_x lambda_y g
            float A = (G - X) - (Y - XY), Bv = X - XY, Cv = Y - XY, Dv = XY;
            if constexpr (WT) {
                const float wc = k2_class_weight(P.weight, c);
                A = fmaf(kv.x, wc, A); Bv = fmaf(kv.y, wc, Bv); Cv = fmaf(kv.z, wc, Cv); Dv = fmaf(kv.w, wc, Dv);
            }
            if (any) {
                atomicAdd(gA + (size_t)c * plane, A);  atomicAdd(gB + (size_t)c * plane, Bv);
                atomicAdd(gC + (size_t)c * plane, Cv); atomicAdd(gD + (size_t)c * plane, Dv);
            }
        };
        if (!slow) {
            // Horner form.  With e(i,j) = E p^i q_i^j (q_i = q t^i) and weights U(i,j):
            //   h_i  = sum_j q_i^j U(i,j)        hx_i = sum_j j q_i^j U(i,j)
            //   G = E sum_i p^i h_i,  Gy = E sum_i i p^i h_i,  Gx / Gxy the same with hx.
            // (h_i, hx_i) are evaluated together as one packed fp32x2 Horner chain per row.
            float2 K3[4], K2v[4], K1v[4], K0[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                K3[i] = make_float2(U[i * 4 + 3], 3.f * U[i * 4 + 3]);
                K2v[i] = make_float2(U[i * 4 + 2], 2.f * U[i * 4 + 2]);
                K1v[i] = make_float2(U[i * 4 + 1], U[i * 4 + 1]);
                K0[i] = make_float2(U[i * 4 + 0], 0.f);
            }
#pragma unroll 4
            for (int c = 0; c < C; ++c) {
                float a, b, cc, d;
                taps(c, a, b, cc, d);
                const Poly y = k2_poly(a, b, cc, d, ly0, lx0, k1, k2, Mk);
                float2 hh[4];
                float2 qi = bc2(y.q);
                const float2 tt = bc2(y.t);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    float2 v = ffma2(qi, K3[i], K2v[i]);
                    v = ffma2(qi, v, K1v[i]);
                    hh[i] = ffma2(qi, v, K0[i]);                 // (h_i, hx_i)
                    if (i < 3) qi = fmul2(qi, tt);
                }
                const float2 pp = bc2(y.p);
                float2 v0 = ffma2(pp, hh[3], hh[2]);
                v0 = ffma2(pp, v0, hh[1]);
                v0 = ffma2(pp, v0, hh[0]);
                const float2 GG = fmul2(v0, bc2(y.E));              // (G, Gx)
                float2 v1 = ffma2(hh[2], bc2(2.f), fmul2(hh[3], bc2(3.f * y.p)));
                v1 = ffma2(pp, v1, hh[1]);
                const float2 GY = fmul2(v1, bc2(y.E * y.p));        // (Gy, Gxy)
                emit(c, GG.x, GG.y, GY.x, GY.y);
            }
        } else {
#pragma unroll 1
            for (int c = 0; c < C; ++c) {
                float a, b, cc, d;
                taps(c, a, b, cc, d);
                float G = 0.f, Gx = 0.f, Gy = 0.f, Gxy = 0.f;
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float ly = ly0 + (float)i * rs, lx = lx0 + (float)j * rs;
                        const float L = fmaf(ly, cc - a, a), R = fmaf(ly, d - b, b);
                        const float gg = ex2f((fmaf(lx, R - L, L) - Mp[i * 4 + j]) * LOG2E) * U[i * 4 + j];
                        G += gg; Gx += (float)j * gg; Gy += (float)i * gg; Gxy += (float)(i * j) * gg;
                    }
                emit(c, G, Gx, Gy, Gxy);
            }
        }
        // ---- - g * onehot: exact integer tap weights (lambda * 2s are odd integers), aggregated per
        //      distinct label of this thread's 16 pixels (blocky label maps: usually one), 4 reductions each
        const float wscale = -gs / (float)(S2 * S2);
        int cur = 0x7fffffff;
#pragma unroll
        for (int i = 0; i < 16; ++i)
            if (lab[i] >= 0) cur = min(cur, lab[i]);
        while (cur != 0x7fffffff) {
            int wa = 0, wb = 0, wc = 0, wd = 0, nxt = 0x7fffffff;
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int t = lab[i * 4 + j];
                    if (t == cur) {
                        const int lyi = lyi0 + 2 * i, lxi = lxi0 + 2 * j;
                        wa += (S2 - lyi) * (S2 - lxi); wb += (S2 - lyi) * lxi;
                        wc += lyi * (S2 - lxi);        wd += lyi * lxi;
                    } else if (t > cur) {
                        nxt = min(nxt, t);
                    }
                }
            const float ws = WT ? wscale * (P.one_m_eps * k2_class_weight(P.weight, cur)) : wscale;
            atomicAdd(gA + (size_t)cur * plane, ws * (float)wa);
            atomicAdd(gB + (size_t)cur * plane, ws * (float)wb);
            atomicAdd(gC + (size_t)cur * plane, ws * (float)wc);
            atomicAdd(gD + (size_t)cur * plane, ws * (float)wd);
            cur = nxt;
        }
    }
    // ---- loss reduction: one double reduction per warp ---------------------------------------------------
    loss = warp_sum(loss);
    if ((threadIdx.x & 31) == 0 && loss != 0.f) atomicAdd(P.loss_sum, (double)loss);
}

// ---------------------------------------------------------------------------------------------
// Strip path kernel (scale 8 / 16); the device code lives in k2_strip.cuh
// SPLIT = false: the one-call path (int64 labels; loss, -g*onehot and g*softmax all here).
// SPLIT = true : the label-only work (valid count, packing, -onehot term) was done by k2_labels_prepass_kernel;
//                this kernel adds sum(log-sum-exp - target logit) and the softmax term only.
// WT: the weighted / label-smoothed form (SPLIT = false only).
template <int S, bool SPLIT, bool WT = false>
__global__ void __launch_bounds__(128)
k2_strip_kernel(const K2SP<WT> P) {
    constexpr int TPG = S / 2, GPW = 32 / TPG, WGX = GPW / 2, CS = GPW * 4;
    extern __shared__ float smem[];
    const int C = P.C;
    const int lane = threadIdx.x & 31;
    const long long wt = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int tiles_per_img = P.nty * P.ntx;
    if (wt >= (long long)P.B * tiles_per_img) return;       // whole warp; there is no CTA barrier below
    const int n = (int)(wt / tiles_per_img);
    const int trem = (int)(wt - (long long)n * tiles_per_img);
    const int tyi = trem / P.ntx, txi = trem - tyi * P.ntx;
    const int GY0 = tyi * 2, GX0 = txi * WGX;
    float* st = smem + (size_t)(threadIdx.x >> 5) * (C + 2) * CS;   // st[c][group][4 taps] + 2 padding class slots
    const size_t plane = (size_t)P.h * P.w;
    const float* lowb = P.low + (size_t)n * C * plane;
    // ---- stage the warp's taps: lane -> fixed (group, tap), strided over classes -------------------------------
    {
        constexpr int CSTEP = 32 / CS > 0 ? 32 / CS : 1;    // 2 (S=16) / 1 (S=8)
        const int r = lane % CS;
        const int gq = r >> 2, tap = r & 3;
        const int kyy = GY0 + gq / WGX - 1, kxx = GX0 + gq % WGX - 1;
        const bool ok = kyy < P.h && kxx < P.w;
        const int yy = clampi(kyy + (tap >> 1), 0, P.h - 1), xx = clampi(kxx + (tap & 1), 0, P.w - 1);
        const float* src = lowb + (size_t)yy * P.w + xx;
        float* dst = st + r;
        for (int c = lane / CS; c < C; c += CSTEP) {
            if (ok) cp_async4(dst + c * CS, src + (size_t)c * plane);
            else dst[c * CS] = 0.f;
        }
    }
    k2_strip_warp<S, SPLIT, CS, false, WT>(P, st, n, GY0, GX0, lane);
}

// The same strips with the taps read from the class-plane-major map itself (no staged tile): for class counts whose
// tile would not leave enough warps per SM (BASELINE config 5: C = 847 -> 54 KB per warp, four warps per SM).
template <int S, bool SPLIT, bool WT = false>
__global__ void __launch_bounds__(128)
k2_strip_gtaps_kernel(const K2SP<WT> P) {
    constexpr int TPG = S / 2, GPW = 32 / TPG, WGX = GPW / 2, CS = GPW * 4;
    const int lane = threadIdx.x & 31;
    const long long wt = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int tiles_per_img = P.nty * P.ntx;
    if (wt >= (long long)P.B * tiles_per_img) return;       // whole warp; there is no CTA barrier below
    const int n = (int)(wt / tiles_per_img);
    const int trem = (int)(wt - (long long)n * tiles_per_img);
    const int tyi = trem / P.ntx, txi = trem - tyi * P.ntx;
    k2_strip_warp<S, SPLIT, CS, true, WT>(P, nullptr, n, tyi * 2, txi * WGX, lane);
}

// ---------------------------------------------------------------------------------------------
// n_valid += the CTA's sum of cnt (nwarps <= 8 warps): one 64-bit reduction per CTA, none when n_valid is null.
__device__ __forceinline__ void k2_block_count(int cnt, int nwarps, unsigned long long* n_valid) {
    __shared__ int red_c[8];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if ((threadIdx.x & 31) == 0) red_c[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        long long tc = 0;
        for (int i = 0; i < nwarps; ++i) tc += red_c[i];
        if (tc && n_valid) atomicAdd(n_valid, (unsigned long long)tc);
    }
}

// ---------------------------------------------------------------------------------------------
// Label prepass of the split path (power-of-two scale S): everything of the cross-entropy that depends on
// the labels only, in one pass over the int64 label map:
//   * n_valid += #{label != ignore_index and in [0,C)}                         (the 'mean' denominator)
//   * packed[b,y,x] = (uint16) label; bit 15 set where the label is ignore_index (a class id that the
//     cross-entropy does not count, but the confusion matrix does); 0xFFFF where it is no class id at all
//   * grad_low[b,t,tap] -= w_tap(pixel)   for the four bilinear taps of every counted pixel (the -onehot
//     term of dL/dlogits, unscaled; exact integer weights lambda*2S, run-length aggregated along the row)
// One thread owns the S pixels of one row of one group (same group geometry as the strip kernel).
// LT = long long: the reference's int64 label map (packs it); LT = unsigned short: labels already packed on
// the host (lc2is_pack_labels_host, same encoding): only the count and the -onehot term remain.
template <int S, typename LT>
__global__ void __launch_bounds__(256)
k2_labels_prepass_kernel(const LT* __restrict__ labels,
                         int B, int C, int h, int w, int H, int W, long long ignore,
                         unsigned short* __restrict__ packed, unsigned long long* __restrict__ n_valid,
                         float* __restrict__ grad_low) {
    const long long total = (long long)B * H * (w + 1);
    const size_t plane = (size_t)h * w;
    constexpr float WSC = 1.f / (float)(4 * S * S);
    int cnt = 0;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const int gx = (int)(idx % (w + 1));
        const long long t1 = idx / (w + 1);
        const int y = (int)(t1 % H), n = (int)(t1 / H);
        const int kx = gx - 1, x0 = S * kx + S / 2;
        const int ky = (y + S / 2) / S - 1;
        const int lyi = 2 * (y - (S * ky + S / 2)) + 1;                  // lambda_y * 2S
        const int Ya = clampi(ky, 0, h - 1), Yb = clampi(ky + 1, 0, h - 1);
        const int Xa = clampi(kx, 0, w - 1), Xb = clampi(kx + 1, 0, w - 1);
        const size_t oA = (size_t)Ya * w + Xa, oB = (size_t)Ya * w + Xb, oC = (size_t)Yb * w + Xa, oD = (size_t)Yb * w + Xb;
        const LT* row = labels + ((size_t)n * H + y) * W;
        unsigned short* prow = packed ? packed + ((size_t)n * H + y) * W : nullptr;
        const size_t ibase = (size_t)n * C * plane;
        int cur = -1, sw0 = 0, sw1 = 0;
        auto flush = [&]() {
            if (cur < 0 || !grad_low) return;
            const float fa = (float)((2 * S - lyi) * sw0) * WSC, fb = (float)((2 * S - lyi) * sw1) * WSC;
            const float fc = (float)(lyi * sw0) * WSC, fd = (float)(lyi * sw1) * WSC;
            float* gp = grad_low + ibase + (size_t)cur * plane;
            atomicAdd(gp + oA, -fa); atomicAdd(gp + oB, -fb);
            atomicAdd(gp + oC, -fc); atomicAdd(gp + oD, -fd);
        };
        const bool in0 = x0 >= 0, in1 = x0 + S / 2 < W;                  // left / right half inside the row
        if constexpr (sizeof(LT) == 2) {
            // packed input: S/2 labels (S bytes) per load
            using V = typename std::conditional<S == 16, uint4, typename std::conditional<S == 8, uint2, unsigned>::type>::type;
            V hv[2];
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
                if (hh ? in1 : in0) hv[hh] = __ldg(reinterpret_cast<const V*>(row + x0 + hh * (S / 2)));
            }
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
                if (!(hh ? in1 : in0)) continue;
                const unsigned* wv = reinterpret_cast<const unsigned*>(&hv[hh]);
#pragma unroll
                for (int k = 0; k < S / 4; ++k)
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int lab = (int)((wv[k] >> (16 * e)) & 0xffffu);
                        if (lab < C) {                                       // counted: a class id without the flag
                            ++cnt;
                            const int j = hh * (S / 2) + 2 * k + e;
                            if (lab != cur) { flush(); cur = lab; sw0 = 0; sw1 = 0; }
                            sw0 += 2 * S - (2 * j + 1);
                            sw1 += 2 * j + 1;
                        }
                    }
            }
            flush();
            continue;
        }
        // all loads of the segment first (the run-length code below has atomics the loads cannot cross)
        longlong2 tv[S / 2];
#pragma unroll
        for (int k = 0; k < S / 2; ++k) {
            const bool in = k < S / 4 ? in0 : in1;
            tv[k] = in ? __ldg(reinterpret_cast<const longlong2*>(row + x0 + 2 * k)) : make_longlong2(-1, -1);
        }
        unsigned pk[S / 2];
#pragma unroll
        for (int k = 0; k < S / 2; ++k) {
            unsigned word = 0;
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const unsigned long long tl = (unsigned long long)(e ? tv[k].y : tv[k].x);
                const bool inr = tl < (unsigned long long)C;                // a class id
                const bool ok = inr && tl != (unsigned long long)ignore;     // counted by the cross-entropy
                const int lab = (int)tl;
                word |= (unsigned)(inr ? (ok ? lab : (lab | 0x8000)) : 0xffff) << (16 * e);
                if (ok) {
                    ++cnt;
                    const int j = 2 * k + e;
                    if (lab != cur) { flush(); cur = lab; sw0 = 0; sw1 = 0; }
                    sw0 += 2 * S - (2 * j + 1);
                    sw1 += 2 * j + 1;
                }
            }
            pk[k] = word;
        }
        if (prow) {
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
                if (!(hh ? in1 : in0)) continue;
                unsigned short* d = prow + x0 + hh * (S / 2);
                const unsigned* q = pk + hh * (S / 4);
                if constexpr (S == 16) *reinterpret_cast<uint4*>(d) = make_uint4(q[0], q[1], q[2], q[3]);
                else if constexpr (S == 8) *reinterpret_cast<uint2*>(d) = make_uint2(q[0], q[1]);
                else *reinterpret_cast<unsigned*>(d) = q[0];
            }
        }
        flush();
    }
    k2_block_count(cnt, (int)(blockDim.x >> 5), n_valid);
}

// ---------------------------------------------------------------------------------------------
// Pack + count only (what the fused K2+K3 path needs from the labels ahead of time): int64 -> packed uint16 (same
// encoding as k2_labels_prepass_kernel) and n_valid += #counted.  A pure stream: 8 labels (64 B in, 16 B out) per thread.
__global__ void __launch_bounds__(256)
k2_pack_labels_kernel(const long long* __restrict__ labels, long long n8, int C, long long ignore,
                      unsigned short* __restrict__ packed, unsigned long long* __restrict__ n_valid) {
    int cnt = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
        const longlong2* src = reinterpret_cast<const longlong2*>(labels) + 4 * i;
        longlong2 v[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) v[k] = __ldcs(src + k);
        unsigned w[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            unsigned word = 0;
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const unsigned long long tl = (unsigned long long)(e ? v[k].y : v[k].x);
                const bool inr = tl < (unsigned long long)C, ok = inr && tl != (unsigned long long)ignore;
                cnt += ok;
                word |= (unsigned)(inr ? (ok ? (unsigned)tl : ((unsigned)tl | 0x8000u)) : 0xffffu) << (16 * e);
            }
            w[k] = word;
        }
        reinterpret_cast<uint4*>(packed)[i] = make_uint4(w[0], w[1], w[2], w[3]);
    }
    k2_block_count(cnt, (int)(blockDim.x >> 5), n_valid);
}

// ---------------------------------------------------------------------------------------------
// generic path: any (h,w)->(H,W); one pixel per thread; exact 3-pass softmax; global atomics.
// WT: the weighted / label-smoothed form (k2_strip.cuh: k2_class_weight), every term per pixel and class.
template <bool WT = false>
__global__ void __launch_bounds__(256)
k2_generic_kernel(const float* __restrict__ low, const long long* __restrict__ labels,
                  float* __restrict__ grad_low, double* __restrict__ loss_sum,
                  const float* __restrict__ grad_scale, long long ignore_index,
                  int B, int C, int h, int w, int H, int W, float scale_y, float scale_x,
                  const float* __restrict__ weight, float one_m_eps, float eps_c) {
    const long long HW = (long long)H * W;
    const long long total = (long long)B * HW;
    const float gs = grad_scale ? __ldg(grad_scale) : 1.f;
    float loss = 0.f;
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < total;
         p += (long long)gridDim.x * blockDim.x) {
        const int n = (int)(p / HW);
        const long long r = p - (long long)n * HW;
        const int y = (int)(r / W), x = (int)(r - (long long)y * W);
        const long long tl = labels[p];
        if (tl == ignore_index || tl < 0 || tl >= C) continue;
        const int t = (int)tl;
        float sy = scale_y * ((float)y + 0.5f) - 0.5f; if (sy < 0.f) sy = 0.f;
        float sx = scale_x * ((float)x + 0.5f) - 0.5f; if (sx < 0.f) sx = 0.f;
        int ky = (int)sy; if (ky > h - 1) ky = h - 1;
        int kx = (int)sx; if (kx > w - 1) kx = w - 1;
        float ly = fminf(fmaxf(sy - (float)ky, 0.f), 1.f), lx = fminf(fmaxf(sx - (float)kx, 0.f), 1.f);
        const int ky1 = ky + 1 < h ? ky + 1 : h - 1, kx1 = kx + 1 < w ? kx + 1 : w - 1;
        const int oa = ky * w + kx, ob = ky * w + kx1, oc = ky1 * w + kx, od = ky1 * w + kx1;
        const float wa = (1.f - ly) * (1.f - lx), wb = (1.f - ly) * lx, wc = ly * (1.f - lx), wd = ly * lx;
        const float* base = low + (size_t)n * C * h * w;
        float m = -INFINITY;
        for (int c = 0; c < C; ++c) {
            const float* q = base + (size_t)c * h * w;
            float l = (1.f - ly) * ((1.f - lx) * __ldg(q + oa) + lx * __ldg(q + ob)) +
                      ly * ((1.f - lx) * __ldg(q + oc) + lx * __ldg(q + od));
            m = fmaxf(m, l);
        }
        float S = 0.f, lt = 0.f;
        float wl = 0.f, wsum = 0.f;                         // WT: sum_c w_c x_c, sum_c w_c
        for (int c = 0; c < C; ++c) {
            const float* q = base + (size_t)c * h * w;
            float l = (1.f - ly) * ((1.f - lx) * __ldg(q + oa) + lx * __ldg(q + ob)) +
                      ly * ((1.f - lx) * __ldg(q + oc) + lx * __ldg(q + od));
            S += ex2f((l - m) * LOG2E);
            if (c == t) lt = l;
            if constexpr (WT) {
                const float wc = k2_class_weight(weight, c);
                wl = fmaf(wc, l, wl);
                wsum += wc;
            }
        }
        float a = 1.f, wt = 1.f;
        if constexpr (WT) {
            wt = one_m_eps * k2_class_weight(weight, t);
            a = fmaf(eps_c, wsum, wt);
            loss += a * (lg2f(S) * LN2 + m) - wt * lt - eps_c * wl;
        } else {
            loss += lg2f(S) * LN2 + m - lt;
        }
        if (grad_low) {
            const float u = WT ? gs * a / S : gs / S;
            float* gb = grad_low + (size_t)n * C * h * w;
            for (int c = 0; c < C; ++c) {
                const float* q = base + (size_t)c * h * w;
                float l = (1.f - ly) * ((1.f - lx) * __ldg(q + oa) + lx * __ldg(q + ob)) +
                          ly * ((1.f - lx) * __ldg(q + oc) + lx * __ldg(q + od));
                float g = ex2f((l - m) * LOG2E) * u - (c == t ? (WT ? gs * wt : gs) : 0.f);
                if constexpr (WT) g -= gs * eps_c * k2_class_weight(weight, c);
                float* gp = gb + (size_t)c * h * w;
                atomicAdd(gp + oa, g * wa); atomicAdd(gp + ob, g * wb);
                atomicAdd(gp + oc, g * wc); atomicAdd(gp + od, g * wd);
            }
        }
    }
    loss = warp_sum(loss);
    __shared__ float red[8];
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = loss;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += red[i];
        if (t != 0.f) atomicAdd(loss_sum, (double)t);
    }
}

// fp32 [B,C,hw] -> bf16 [B,C_pad,hw], zero pad rows
__global__ void k2_grad_to_bf16_kernel(const float* __restrict__ g, int C, int C_pad, long long hw,
                                       __nv_bfloat16* __restrict__ out, long long total) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        long long p = i % hw;
        long long bc = i / hw;
        int c = (int)(bc % C_pad);
        long long b = bc / C_pad;
        float v = c < C ? g[((size_t)b * C + c) * hw + p] : 0.f;
        out[i] = __float2bfloat16(v);
    }
}

}  // namespace lc2is

using namespace lc2is;

extern "C" int lc2is_count_valid(const int64_t* d_labels, int64_t n, int C, int64_t ignore_index,
                                 int64_t* d_n_valid, lc2is_stream_t stream) {
    if (int e = ensure_device()) return e;
    if (n < 0) return fail(LC2IS_ERR_SHAPE, "negative n%s");
    if (n == 0) return 0;
    if (!d_labels || !d_n_valid) return fail(LC2IS_ERR_ARG, "null pointer%s");
    if ((uintptr_t)d_labels % 16) return fail(LC2IS_ERR_ARG, "labels must be 16-byte aligned%s");
    long long blocks = (n / 2 + 255) / 256;
    long long cap = (long long)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    k2_count_valid_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        (const long long*)d_labels, n, (long long)C, ignore_index, (unsigned long long*)d_n_valid);
    LC2IS_CHECK_LAUNCH("k2_count_valid_kernel");
    return 0;
}

extern "C" int lc2is_ce_weight_sum(const int64_t* d_labels, int64_t n, int C, int64_t ignore_index,
                                   const float* d_weight, double* d_wsum, lc2is_stream_t stream) {
    if (int e = ensure_device()) return e;
    if (n < 0) return fail(LC2IS_ERR_SHAPE, "negative n%s");
    if (n == 0) return 0;
    if (!d_labels || !d_wsum) return fail(LC2IS_ERR_ARG, "null pointer%s");
    if ((uintptr_t)d_labels % 16) return fail(LC2IS_ERR_ARG, "labels must be 16-byte aligned%s");
    long long blocks = (n / 2 + 255) / 256;
    long long cap = (long long)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    k2_weight_sum_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        (const long long*)d_labels, n, (long long)C, ignore_index, d_weight, d_wsum);
    LC2IS_CHECK_LAUNCH("k2_weight_sum_kernel");
    return 0;
}

extern "C" int lc2is_grad_to_bf16(const float* d_grad, int B, int C, int hw, void* d_grad_bf16,
                                  lc2is_stream_t stream) {
    if (int e = ensure_device()) return e;
    if (!d_grad || !d_grad_bf16) return fail(LC2IS_ERR_ARG, "null pointer%s");
    const int C_pad = class_pad(C);
    long long total = (long long)B * C_pad * hw;
    if (total == 0) return 0;
    long long blocks = (total + 255) / 256;
    long long cap = (long long)sm_count() * 16;
    if (blocks > cap) blocks = cap;
    k2_grad_to_bf16_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        d_grad, C, C_pad, hw, (__nv_bfloat16*)d_grad_bf16, total);
    LC2IS_CHECK_LAUNCH("k2_grad_to_bf16_kernel");
    return 0;
}

extern "C" int lc2is_upsample_ce_fwd_bwd(const float* d_low, const int64_t* d_labels,
                                         int B, int C, int h, int w, int H, int W,
                                         int64_t ignore_index, const float* d_grad_scale,
                                         double* d_loss_sum, float* d_grad_low, void* d_grad_low_bf16,
                                         lc2is_stream_t stream) {
    return lc2is_upsample_ce_fwd_bwd_ex(d_low, d_labels, B, C, h, w, H, W, ignore_index, nullptr, 0.f, d_grad_scale,
                                        d_loss_sum, d_grad_low, d_grad_low_bf16, stream);
}

namespace lc2is {
// The strip kernels (scale s = 8 / 16) over P.B images; sets P.nty / P.ntx.  Warps are independent; a warp's staged
// tile of taps takes (C + 2) * (32 / (s/2)) * 16 bytes of shared memory, and above K2_GTAPS_SMEM the taps are read from
// the map itself instead.
template <bool SPLIT, bool WT>
static int launch_k2_strip(K2SP<WT> P, int s, cudaStream_t st) {
    const size_t smem_warp = (size_t)(P.C + 2) * (64 / s) * 16;
    int wpc = 4;
    while (wpc > 1 && smem_warp * wpc > 56 * 1024) wpc /= 2;
    const size_t smem = smem_warp * wpc;
    const bool gtaps = smem_warp > K2_GTAPS_SMEM;               // staged tile too large for a decent occupancy
    const int wgx = (64 / s) / 2;
    P.nty = (P.h + 1 + 1) / 2;
    P.ntx = (P.w + 1 + wgx - 1) / wgx;
    const long long tiles = (long long)P.B * P.nty * P.ntx;
    auto launch = [&](auto kernel, auto kernel_gtaps) -> int {
        if (gtaps) {
            kernel_gtaps<<<(unsigned)((tiles + 3) / 4), 128, 0, st>>>(P);
        } else {
            LC2IS_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            kernel<<<(unsigned)((tiles + wpc - 1) / wpc), wpc * 32, smem, st>>>(P);
        }
        LC2IS_CHECK_LAUNCH(SPLIT ? "k2_strip_kernel(split)" : "k2_strip_kernel");
        return 0;
    };
    return s == 8 ? launch(k2_strip_kernel<8, SPLIT, WT>, k2_strip_gtaps_kernel<8, SPLIT, WT>)
                  : launch(k2_strip_kernel<16, SPLIT, WT>, k2_strip_gtaps_kernel<16, SPLIT, WT>);
}
}  // namespace lc2is

extern "C" int lc2is_upsample_ce_fwd_bwd_ex(const float* d_low, const int64_t* d_labels,
                                            int B, int C, int h, int w, int H, int W,
                                            int64_t ignore_index, const float* d_weight, float label_smoothing,
                                            const float* d_grad_scale, double* d_loss_sum, float* d_grad_low,
                                            void* d_grad_low_bf16, lc2is_stream_t stream) {
    if (int e = ensure_device()) return e;
    if (B < 0 || C <= 0 || h <= 0 || w <= 0 || H <= 0 || W <= 0) return fail(LC2IS_ERR_SHAPE, "bad shape%s");
    if (!(label_smoothing >= 0.f && label_smoothing <= 1.f))
        return fail(LC2IS_ERR_ARG, "label_smoothing must be in [0, 1]%s");
    // the unweighted instantiations unless a weight or a smoothing is asked for
    const bool wt = d_weight != nullptr || label_smoothing != 0.f;
    const float one_m_eps = 1.f - label_smoothing, eps_c = label_smoothing / (float)C;
    if (B == 0) return 0;
    if (!d_low || !d_labels || !d_loss_sum) return fail(LC2IS_ERR_ARG, "null pointer%s");
    if (d_grad_low_bf16 && !d_grad_low)
        return fail(LC2IS_ERR_ARG, "grad_low_bf16 needs the fp32 grad_low buffer as well%s");
    cudaStream_t st = (cudaStream_t)stream;
    if (d_grad_low) LC2IS_CUDA(cudaMemsetAsync(d_grad_low, 0, (size_t)B * C * h * w * sizeof(float), st));

    int s = 0;
    bool fast = fast_scale(h, w, H, W, &s) && s <= 16;
    if (fast && s >= 8 && ((uintptr_t)d_labels % 16) == 0) {
        // ---- strip path: s = 8 / 16 -----------------------------------------------------------------------
        K2SParamsW PW;
        K2SParams& P = PW;
        P.low = d_low; P.labels = (const long long*)d_labels; P.labels16 = nullptr; P.grad_low = d_grad_low;
        P.loss_sum = d_loss_sum; P.grad_scale = d_grad_scale; P.ignore_index = ignore_index;
        P.B = B; P.C = C; P.h = h; P.w = w; P.H = H; P.W = W;
        PW.weight = d_weight; PW.one_m_eps = one_m_eps; PW.eps_c = eps_c;
        if (int e = wt ? launch_k2_strip<false, true>(PW, s, st) : launch_k2_strip<false, false>(P, s, st)) return e;
        if (d_grad_low_bf16) return lc2is_grad_to_bf16(d_grad_low, B, C, h * w, d_grad_low_bf16, stream);
        return 0;
    }
    fast = fast && s == 4;
    K2Params P;
    size_t smem = 0;
    if (fast) {
        BlockGeom g = make_geom(H, W, s);
        P.low = d_low; P.labels = (const long long*)d_labels; P.grad_low = d_grad_low;
        P.loss_sum = d_loss_sum; P.grad_scale = d_grad_scale; P.ignore_index = ignore_index;
        P.B = B; P.C = C; P.h = h; P.w = w; P.H = H; P.W = W;
        P.s = s; P.off = g.off; P.rs = g.rs;
        P.weight = d_weight; P.one_m_eps = one_m_eps; P.eps_c = eps_c;
        P.q = (g.off + s / 2) / 4;
        // 128 threads = 8 x 16 blocks of 4 x 4 pixels; the tile holds the 9 x 17 source cells they read
        P.tgy = 8; P.tgx = 16;
        smem = (size_t)C * (P.tgy + 1) * (P.tgx + 1) * sizeof(float);
        if (smem > 110 * 1024) fast = false;
    }
    if (fast) {
        dim3 grid((w + 1 + P.tgx - 1) / P.tgx, (h + 1 + P.tgy - 1) / P.tgy, B);
        auto launch = [&](auto kernel) -> int {
            LC2IS_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            kernel<<<grid, 128, smem, st>>>(P);
            return 0;
        };
        int e = wt ? launch(k2_fast_kernel<true>) : launch(k2_fast_kernel<false>);
        if (e) return e;
        LC2IS_CHECK_LAUNCH("k2_fast_kernel");
    } else {
        const float sy = (float)h / (float)H, sx = (float)w / (float)W;
        long long total = (long long)B * H * W;
        long long blocks = (total + 255) / 256;
        long long cap = (long long)sm_count() * 8;
        if (blocks > cap) blocks = cap;
        auto kernel = wt ? k2_generic_kernel<true> : k2_generic_kernel<false>;
        kernel<<<(unsigned)blocks, 256, 0, st>>>(d_low, (const long long*)d_labels, d_grad_low, d_loss_sum, d_grad_scale,
                                                 ignore_index, B, C, h, w, H, W, sy, sx, d_weight, one_m_eps, eps_c);
        LC2IS_CHECK_LAUNCH("k2_generic_kernel");
    }
    if (d_grad_low_bf16) return lc2is_grad_to_bf16(d_grad_low, B, C, h * w, d_grad_low_bf16, stream);
    return 0;
}

// ---------------------------------------------------------------------------------------------
// Split path (used by the whole-step entries): label prepass + packed-label strip kernel.
extern "C" int lc2is_ce_split_supported(int h, int w, int H, int W) {
    int s = 0;
    return fast_scale(h, w, H, W, &s) && (s == 8 || s == 16) ? 1 : 0;
}

namespace lc2is {
// Both prepass entries after their argument checks: k2_labels_prepass_kernel<s, LT> for the scale s = 4 / 8 / 16.
template <typename LT>
static int launch_labels_prepass(const LT* labels, int B, int C, int h, int w, int H, int W, long long ignore,
                                 uint16_t* packed, int64_t* n_valid, float* grad_low, cudaStream_t st) {
    int s = 0;
    if (!fast_scale(h, w, H, W, &s) || s > 16)
        return fail(LC2IS_ERR_UNSUPPORTED, "label prepass needs a power-of-two scale 4 / 8 / 16%s");
    if (((uintptr_t)labels % 16) || ((uintptr_t)packed % 16)) return fail(LC2IS_ERR_ARG, "labels must be 16-byte aligned%s");
    const long long total = (long long)B * H * (w + 1);
    long long blocks = (total + 255) / 256;
    const long long cap = (long long)sm_count() * 16;
    if (blocks > cap) blocks = cap;
    auto launch = [&](auto kernel) {
        kernel<<<(unsigned)blocks, 256, 0, st>>>(labels, B, C, h, w, H, W, ignore, (unsigned short*)packed,
                                                 (unsigned long long*)n_valid, grad_low);
    };
    if (s == 4) launch(k2_labels_prepass_kernel<4, LT>);
    else if (s == 8) launch(k2_labels_prepass_kernel<8, LT>);
    else launch(k2_labels_prepass_kernel<16, LT>);
    LC2IS_CHECK_LAUNCH(sizeof(LT) == 2 ? "k2_labels_prepass_kernel(packed)" : "k2_labels_prepass_kernel");
    return 0;
}
}  // namespace lc2is

extern "C" int lc2is_ce_labels_prepass(const int64_t* d_labels,
                                       int B, int C, int h, int w, int H, int W, int64_t ignore_index,
                                       uint16_t* d_labels_packed, int64_t* d_n_valid,
                                       float* d_grad_low, lc2is_stream_t stream) {
    if (int e = ensure_device()) return e;
    if (B < 0 || C <= 0 || h <= 0 || w <= 0 || H <= 0 || W <= 0) return fail(LC2IS_ERR_SHAPE, "bad shape%s");
    if (C >= 0x7fff) return fail(LC2IS_ERR_UNSUPPORTED, "packed labels hold class ids < 32767%s");
    if (B == 0) return 0;
    if (!d_labels) return fail(LC2IS_ERR_ARG, "null pointer%s");
    return launch_labels_prepass((const long long*)d_labels, B, C, h, w, H, W, (long long)ignore_index, d_labels_packed,
                                 d_n_valid, d_grad_low, (cudaStream_t)stream);
}

extern "C" int lc2is_pack_labels(const int64_t* d_labels, int64_t n, int C, int64_t ignore_index,
                                 uint16_t* d_labels_packed, int64_t* d_n_valid, lc2is_stream_t stream) {
    if (int e = ensure_device()) return e;
    if (n < 0 || C <= 0) return fail(LC2IS_ERR_SHAPE, "bad n / C%s");
    if (C >= 0x7fff) return fail(LC2IS_ERR_UNSUPPORTED, "packed labels hold class ids < 32767%s");
    if (n == 0) return 0;
    if (!d_labels || !d_labels_packed) return fail(LC2IS_ERR_ARG, "null pointer%s");
    if (n % 8) return fail(LC2IS_ERR_SHAPE, "lc2is_pack_labels: n must be a multiple of 8%s");
    if (((uintptr_t)d_labels % 16) || ((uintptr_t)d_labels_packed % 16))
        return fail(LC2IS_ERR_ARG, "labels must be 16-byte aligned%s");
    const long long n8 = n / 8;
    long long blocks = (n8 + 255) / 256;
    const long long cap = (long long)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    k2_pack_labels_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        (const long long*)d_labels, n8, C, (long long)ignore_index, (unsigned short*)d_labels_packed,
        (unsigned long long*)d_n_valid);
    LC2IS_CHECK_LAUNCH("k2_pack_labels_kernel");
    return 0;
}

namespace lc2is {
// one-byte host form (C <= 254: class id; 0xFE = label == ignore_index; 0xFF = not a class id) -> packed uint16
__global__ void __launch_bounds__(256)
k2_expand_labels_kernel(const uint4* __restrict__ in, long long n16, unsigned ign16, uint4* __restrict__ out,
                        unsigned long long* __restrict__ n_valid) {
    int cnt = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (long long)gridDim.x * blockDim.x) {
        const uint4 q = __ldcs(in + i);
        const unsigned wds[4] = {q.x, q.y, q.z, q.w};
        unsigned o[8];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const unsigned a = (wds[k] >> (16 * j)) & 0xFFu, b = (wds[k] >> (16 * j + 8)) & 0xFFu;
                cnt += (a < 0xFEu) + (b < 0xFEu);
                const unsigned ea = a < 0xFEu ? a : (a == 0xFEu ? ign16 : 0xFFFFu);
                const unsigned eb = b < 0xFEu ? b : (b == 0xFEu ? ign16 : 0xFFFFu);
                o[2 * k + j] = ea | (eb << 16);
            }
        }
        out[2 * i] = make_uint4(o[0], o[1], o[2], o[3]);
        out[2 * i + 1] = make_uint4(o[4], o[5], o[6], o[7]);
    }
    if (n_valid) {
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, s);
        if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(n_valid, (unsigned long long)cnt);
    }
}
}  // namespace lc2is

extern "C" int lc2is_expand_labels(const uint8_t* d_labels8, int64_t n, int C, int64_t ignore_index,
                                   uint16_t* d_labels_packed, int64_t* d_n_valid, lc2is_stream_t stream) {
    if (int e = ensure_device()) return e;
    if (n < 0 || C <= 0) return fail(LC2IS_ERR_SHAPE, "bad n / C%s");
    if (C > 254) return fail(LC2IS_ERR_UNSUPPORTED, "one-byte labels hold class ids < 254%s");
    if (n == 0) return 0;
    if (!d_labels8 || !d_labels_packed) return fail(LC2IS_ERR_ARG, "null pointer%s");
    if (n % 16) return fail(LC2IS_ERR_SHAPE, "lc2is_expand_labels: n must be a multiple of 16%s");
    if (((uintptr_t)d_labels8 % 16) || ((uintptr_t)d_labels_packed % 16))
        return fail(LC2IS_ERR_ARG, "labels must be 16-byte aligned%s");
    const long long n16 = n / 16;
    long long blocks = (n16 + 255) / 256;
    const long long cap = (long long)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    const unsigned ign16 = (ignore_index >= 0 && ignore_index < C) ? ((unsigned)ignore_index | 0x8000u) : 0xFFFFu;
    k2_expand_labels_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        (const uint4*)d_labels8, n16, ign16, (uint4*)d_labels_packed, (unsigned long long*)d_n_valid);
    LC2IS_CHECK_LAUNCH("k2_expand_labels_kernel");
    return 0;
}

extern "C" int lc2is_ce_labels_prepass_packed(const uint16_t* d_labels_packed, int B, int C, int h, int w, int H,
                                              int W, int64_t* d_n_valid, float* d_grad_low,
                                              lc2is_stream_t stream) {
    if (int e = ensure_device()) return e;
    if (B < 0 || C <= 0 || h <= 0 || w <= 0 || H <= 0 || W <= 0) return fail(LC2IS_ERR_SHAPE, "bad shape%s");
    if (B == 0) return 0;
    if (!d_labels_packed) return fail(LC2IS_ERR_ARG, "null pointer%s");
    return launch_labels_prepass((const unsigned short*)d_labels_packed, B, C, h, w, H, W, 0LL, nullptr, d_n_valid,
                                 d_grad_low, (cudaStream_t)stream);
}

extern "C" int lc2is_upsample_ce_packed(const float* d_low, const uint16_t* d_labels_packed,
                                        int B, int C, int h, int w, int H, int W,
                                        double* d_loss_sum, float* d_grad_low, lc2is_stream_t stream) {
    if (int e = ensure_device()) return e;
    if (B < 0 || C <= 0 || h <= 0 || w <= 0 || H <= 0 || W <= 0) return fail(LC2IS_ERR_SHAPE, "bad shape%s");
    if (B == 0) return 0;
    if (!d_low || !d_labels_packed || !d_loss_sum) return fail(LC2IS_ERR_ARG, "null pointer%s");
    if ((uintptr_t)d_labels_packed % 16) return fail(LC2IS_ERR_ARG, "packed labels must be 16-byte aligned%s");
    int s = 0;
    if (!fast_scale(h, w, H, W, &s) || (s != 8 && s != 16))
        return fail(LC2IS_ERR_UNSUPPORTED, "split path needs scale 8 or 16 (see lc2is_ce_split_supported)%s");
    K2SParams P;
    P.low = d_low; P.labels = nullptr; P.labels16 = d_labels_packed; P.grad_low = d_grad_low;
    P.loss_sum = d_loss_sum; P.grad_scale = nullptr; P.ignore_index = 0;
    P.B = B; P.C = C; P.h = h; P.w = w; P.H = H; P.W = W;
    return launch_k2_strip<true, false>(P, s, (cudaStream_t)stream);
}
