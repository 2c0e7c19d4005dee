// K2 strip path (scale 8 / 16): device code of k2_strip_kernel / k2_strip_gtaps_kernel (k2_upsample_ce.cu); its helpers
// (cp.async, packed fp32x2 arithmetic) serve K3 and k23_rc as well.  See the comment block above k2_strip_warp.
#pragma once
#include "common.cuh"
#include <type_traits>

namespace lc2is {

constexpr float LOG2E = 1.4426950408889634f;
constexpr float LN2 = 0.6931471805599453f;
constexpr float S_MIN = 1e-30f;       // below this the shared shift lost precision -> slow path

__device__ __forceinline__ void cp_async4(void* smem, const void* gmem) {
    unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(sa), "l"(gmem));
}
__device__ __forceinline__ void cp_async_wait_all() {
    asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory");
}

constexpr float K2_FAST_RANGE = 40.f;   // max logit range inside a group for the shared-shift fast path

// ---- packed fp32x2 arithmetic (sm_100: FADD2 / FMUL2 / FFMA2 - two fp32 ops per issue slot) ------
__device__ __forceinline__ unsigned long long pk2(float2 a) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a.x), "f"(a.y));
    return r;
}
__device__ __forceinline__ float2 up2(unsigned long long r) {
    float2 d;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(r));
    return d;
}
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
    unsigned long long d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(pk2(a)), "l"(pk2(b)));
    return up2(d);
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) {
    unsigned long long d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(pk2(a)), "l"(pk2(b)));
    return up2(d);
}
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
    unsigned long long d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(pk2(a)), "l"(pk2(b)), "l"(pk2(c)));
    return up2(d);
}
__device__ __forceinline__ float2 bc2(float x) { return make_float2(x, x); }

// Sum (a,b,c,d) over the LPG consecutive lanes of a group.  After the call lane u of the group
// holds in `a` the total of value number (u * 4 / LPG), i.e. the first quarter of the
// lanes hold sum(a), the second sum(b), ...
template <int LPG>
__device__ __forceinline__ void group_reduce4(float& a, float& b, float& c, float& d, int u) {
    static_assert(LPG >= 4, "a group spans at least four lanes");
    const bool up = u & (LPG / 2);
    float s0 = up ? a : c, s1 = up ? b : d;          // what this lane gives away
    float k0 = up ? c : a, k1 = up ? d : b;          // what it keeps
    k0 += __shfl_xor_sync(0xffffffffu, s0, LPG / 2);
    k1 += __shfl_xor_sync(0xffffffffu, s1, LPG / 2);
    const bool up2 = u & (LPG / 4);
    float g = up2 ? k0 : k1;
    float k = up2 ? k1 : k0;
    k += __shfl_xor_sync(0xffffffffu, g, LPG / 4);
#pragma unroll
    for (int o = LPG / 8; o > 0; o >>= 1) k += __shfl_xor_sync(0xffffffffu, k, o);
    a = k;
}

// ---------------------------------------------------------------------------------------------
// Strip path (scale S = 8 or 16): the dominant kernel at the aux-head geometry (32^2 -> 512^2).
//
// A GROUP (gy,gx) is the S x S pixel region that interpolates between source cells (ky,kx) = (gy-1,gx-1)
// .. (ky+1,kx+1) (index-clamped; (h+1) x (w+1) groups per image, border groups are half empty).  One
// thread owns a STRIP of the group: 2 rows x S columns, the two rows packed as fp32x2.  Along a row the
// upsampled logit is linear in the column, so per (class, row)
//       exp2(k*l(j) - k*M) = E * rho^j ,   E = exp2(k*(L + lx0*(R-L)) - k*M),  rho = exp2(k*(R-L)/S)
// (L / R = the row's left / right source values): 4 ex2 per class per 2*S pixels, then
//   pass A  S(j) += e ; e *= rho                      one FADD2 + one FMUL2 per pixel PAIR and class
//   pass B  with U(j) = g / S(j):  h = sum_j U(j) rho^j and d = dh/drho by one Horner sweep
//           (d = d*rho + h ; h = h*rho + U(j): two FFMA2 per pixel pair), which give the row's
//           sum_j softmax*U = E*h and sum_j j*softmax*U = E*rho*d, i.e. the four tap gradients.
// Warps are independent (no CTA barrier): a warp owns a 2 x (GPW/2) tile of groups, stages their taps
// as per-group quads st[c][group][4] with cp.async, and in pass B the S/2 lanes of a group add their tap
// gradients with a shuffle butterfly and store them IN PLACE over the group's staged taps.  Finally the
// warp sums the quads of its tile per source cell in a fixed order: one L2 reduction per (class, cell),
// 9 instead of 16 per 2x2-group tile.  The class loops are software pipelined by hand (the taps of class
// c+1 are loaded and exponentiated before the chain of class c; the in-place store would otherwise pin
// every shared-memory load behind it).
// M = max tap of the group (a valid softmax shift); groups whose taps span more than K2_FAST_RANGE or are
// not finite take the exact per-pixel path (k2_strip_slow, warp-uniform).
struct K2SParams {
    const float* low;
    const long long* labels;      // int64 labels (one-call path) ...
    const unsigned short* labels16;   // ... or packed labels from the prepass (split path), 0xFFFF = not counted
    float* grad_low;
    double* loss_sum;
    const float* grad_scale;
    long long ignore_index;
    int B, C, h, w, H, W;
    int nty, ntx;                 // warp tiles per image
};
// The weighted form's parameters (a separate type: K2SParams is copied to the stack for k2_strip_slow, and the unweighted
// kernels keep their frame): class weights w[C] (null = all 1), 1 - eps and eps / C of the label smoothing eps.
struct K2SParamsW : K2SParams {
    const float* weight;
    float one_m_eps, eps_c;
};
template <bool WT>
using K2SP = typename std::conditional<WT, K2SParamsW, K2SParams>::type;

// Weighted / label-smoothed cross-entropy (nn.CrossEntropyLoss(weight=w, label_smoothing=eps)); with W = sum_c w_c and
// a = (1-eps) w_t + (eps/C) W, a counted pixel adds  a*lse - (1-eps) w_t x_t - (eps/C) sum_c w_c x_c  to the loss and
//   g * (a * softmax_c - (1-eps) w_t [c == t] - (eps/C) w_c)  to d/dx_c.
__device__ __forceinline__ float k2_class_weight(const float* w, int c) { return w ? __ldg(w + c) : 1.f; }

// Where a group's four taps (a b / c d) of class c come from.  TapsSmem: the staged tile, one LDS.128.  TapsGlobal: the
// class-plane-major map itself (L1 / L2) - for class counts whose staged tile would leave a handful of warps per SM
// (C = 847: 54 KB per warp); look-aheads past the last class re-read it.
constexpr size_t K2_GTAPS_SMEM = 28 * 1024;              // staged bytes per warp above which the taps stay in global memory
struct TapsSmem {
    const float4* p;                                        // quad of class 0
    int cs4;                                                // float4 per class
    __device__ __forceinline__ float4 get(int c) const { return p[(size_t)c * cs4]; }
};
struct TapsGlobal {
    const float* b;                                         // class 0 of the image
    size_t plane;
    int oA, oB, oC, oD, C;
    __device__ __forceinline__ float4 get(int c) const {
        const float* q = b + (size_t)(c < C ? c : C - 1) * plane;
        return make_float4(__ldg(q + oA), __ldg(q + oB), __ldg(q + oC), __ldg(q + oD));
    }
};

template <int S, bool SPLIT, class TQ, bool WT = false>
__device__ __noinline__ float k2_strip_slow(const TQ tq, unsigned vm, int n, int y0, int x0,
                                            int u, const K2SP<WT>& P, float gs, float* gA, float* gB,
                                            float* gC, float* gD) {
    const int C = P.C;
    const size_t plane = (size_t)P.h * P.w;
    float loss = 0.f;
    for (int r = 0; r < 2; ++r)
        for (int j = 0; j < S; ++j) {
            if (!((vm >> (r * 16 + j)) & 1u)) continue;
            // SPLIT: the prepass owns the -onehot term; the caller has already subtracted the target logits
            const int t = SPLIT ? -1 : (int)__ldg(P.labels + ((size_t)n * P.H + (y0 + r)) * P.W + (x0 + j));
            const float ly = ((float)(2 * u + r) + 0.5f) * (1.f / S), lx = ((float)j + 0.5f) * (1.f / S);
            float m = -INFINITY;
            for (int c = 0; c < C; ++c) {
                const float4 q = tq.get(c);
                const float L = fmaf(ly, q.z - q.x, q.x), R = fmaf(ly, q.w - q.y, q.y);
                m = fmaxf(m, fmaf(lx, R - L, L));
            }
            float sum = 0.f, lt = 0.f;
            float wl = 0.f, wsum = 0.f;                     // WT: sum_c w_c x_c, sum_c w_c
            for (int c = 0; c < C; ++c) {
                const float4 q = tq.get(c);
                const float L = fmaf(ly, q.z - q.x, q.x), R = fmaf(ly, q.w - q.y, q.y);
                const float l = fmaf(lx, R - L, L);
                sum += ex2f((l - m) * LOG2E);
                if (c == t) lt = l;
                if constexpr (WT) {
                    const float wc = k2_class_weight(P.weight, c);
                    wl = fmaf(wc, l, wl);
                    wsum += wc;
                }
            }
            float a = 1.f, wt = 1.f;
            if constexpr (WT) {
                wt = P.one_m_eps * k2_class_weight(P.weight, t);
                a = fmaf(P.eps_c, wsum, wt);
                loss += a * (logf(sum) + m) - wt * lt - P.eps_c * wl;
            } else {
                loss += logf(sum) + m - lt;
            }
            if (gA) {
                const float uu = WT ? gs * a / sum : gs / sum;
                const float wa = (1.f - ly) * (1.f - lx), wb = (1.f - ly) * lx, wc = ly * (1.f - lx), wd = ly * lx;
                for (int c = 0; c < C; ++c) {
                    const float4 q = tq.get(c);
                    const float L = fmaf(ly, q.z - q.x, q.x), R = fmaf(ly, q.w - q.y, q.y);
                    float gg = ex2f((fmaf(lx, R - L, L) - m) * LOG2E) * uu - (c == t ? (WT ? gs * wt : gs) : 0.f);
                    if constexpr (WT) gg -= gs * P.eps_c * k2_class_weight(P.weight, c);
                    atomicAdd(gA + (size_t)c * plane, gg * wa); atomicAdd(gB + (size_t)c * plane, gg * wb);
                    atomicAdd(gC + (size_t)c * plane, gg * wc); atomicAdd(gD + (size_t)c * plane, gg * wd);
                }
            }
        }
    return loss;
}

// CSF = floats per class of the warp's tile of quads; st = the warp's first tap quad of class 0.
// WT: the weighted / label-smoothed form (one-call path only).  Besides a*lse and the (1-eps) w_t scale of the -onehot
// runs, the smoothing terms are linear in the logits: the loss takes (eps/C) V.Q per thread, with Q = sum_c w_c * taps
// (accumulated in the max-tap sweep) and V = the thread's summed bilinear tap weights of its counted pixels; the
// gradient takes -g (eps/C) w_c V_cell on the lane that issues the cell's reduction (V merged like the gradients).
template <int S, bool SPLIT, int CSF, bool GTAPS = false, bool WT = false>
__device__ __forceinline__ void k2_strip_warp(const K2SP<WT>& P, float* st, int n, int GY0, int GX0, int lane) {
    static_assert(!(WT && SPLIT), "the weighted form is one-call only");
    constexpr int TPG = S / 2;                              // threads (lanes) per group
    constexpr int GPW = 32 / TPG;                           // groups per warp: 4 (S=16) / 8 (S=8)
    constexpr int WGX = GPW / 2;                            // warp tile = 2 x WGX groups
    constexpr int CS = CSF;                                 // floats per class in the tile
    constexpr int CS4 = CSF / 4;
    constexpr float RS = 1.f / S;
    constexpr float LX0 = 0.5f / S;                         // lambda_x of the group's first column
    const int C = P.C;
    const size_t plane = (size_t)P.h * P.w;

    // ---- this thread's strip ------------------------------------------------------------------------------
    const int gl = lane / TPG, u = lane % TPG;
    const int ky = GY0 + gl / WGX - 1, kx = GX0 + gl % WGX - 1;   // top-left tap of the group (-1 .. h-1)
    const bool group_in = ky < P.h && kx < P.w;
    const int y0 = S * ky + S / 2 + 2 * u, x0 = S * kx + S / 2;
    const float gs = P.grad_scale ? __ldg(P.grad_scale) : 1.f;

    // valid-label mask of the 2 x S pixels (bit r*16 + j); labels are re-read where their value is needed
    unsigned vm = 0;
    unsigned lw[SPLIT ? S : 1];                             // SPLIT: the strip's packed labels (2 per word)
    if constexpr (SPLIT) {
#pragma unroll
        for (int k = 0; k < S; ++k) lw[k] = 0xffffffffu;
    }
    if (group_in) {
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const int y = y0 + r;
            if (y < 0 || y >= P.H) continue;
            if constexpr (SPLIT) {
                // packed labels: S/2 pixels (S bytes) per load
                using V = typename std::conditional<S == 16, uint4, uint2>::type;
                const unsigned short* row = P.labels16 + ((size_t)n * P.H + y) * P.W;
#pragma unroll
                for (int hh = 0; hh < 2; ++hh) {
                    const int x = x0 + hh * (S / 2);
                    if (x < 0 || x >= P.W) continue;
                    const V t = __ldg(reinterpret_cast<const V*>(row + x));
                    const unsigned* wv = reinterpret_cast<const unsigned*>(&t);
#pragma unroll
                    for (int k = 0; k < S / 4; ++k) lw[r * (S / 2) + hh * (S / 4) + k] = wv[k];
                }
            } else {
                const long long* row = P.labels + ((size_t)n * P.H + y) * P.W;
#pragma unroll
                for (int jj = 0; jj < S / 2; ++jj) {
                    const int x = x0 + 2 * jj;
                    if (x < 0 || x >= P.W) continue;
                    const longlong2 t = __ldg(reinterpret_cast<const longlong2*>(row + x));
                    if (t.x != P.ignore_index && t.x >= 0 && t.x < C) vm |= 1u << (r * 16 + 2 * jj);
                    if (t.y != P.ignore_index && t.y >= 0 && t.y < C) vm |= 1u << (r * 16 + 2 * jj + 1);
                }
            }
        }
    }
    if constexpr (SPLIT) {
#pragma unroll
        for (int r = 0; r < 2; ++r)
#pragma unroll
            for (int k = 0; k < S / 2; ++k) {
                const unsigned wd = lw[r * (S / 2) + k];
                if ((wd & 0xffffu) < (unsigned)C) vm |= 1u << (r * 16 + 2 * k);
                if ((wd >> 16) < (unsigned)C) vm |= 1u << (r * 16 + 2 * k + 1);
            }
    }
    cp_async_wait_all();
    __syncwarp();

    const int Ya = clampi(ky, 0, P.h - 1), Yb = clampi(ky + 1, 0, P.h - 1);
    const int Xa = clampi(kx, 0, P.w - 1), Xb = clampi(kx + 1, 0, P.w - 1);
    float* gb = P.grad_low ? P.grad_low + (size_t)n * C * plane : nullptr;
    float* gA = gb ? gb + (size_t)Ya * P.w + Xa : nullptr; float* gB = gb ? gb + (size_t)Ya * P.w + Xb : nullptr;
    float* gC = gb ? gb + (size_t)Yb * P.w + Xa : nullptr; float* gD = gb ? gb + (size_t)Yb * P.w + Xb : nullptr;
    using TQ = typename std::conditional<GTAPS, TapsGlobal, TapsSmem>::type;
    TQ tq;
    if constexpr (GTAPS) {
        tq.b = P.low + (size_t)n * C * plane; tq.plane = plane; tq.C = C;
        tq.oA = Ya * P.w + Xa; tq.oB = Ya * P.w + Xb; tq.oC = Yb * P.w + Xa; tq.oD = Yb * P.w + Xb;
    } else {
        tq.p = reinterpret_cast<const float4*>(st) + gl; tq.cs4 = CS4;
    }

    // ---- softmax shift: M = max over classes of the group's taps --------------------------------------------
    float mx = -INFINITY, mn = INFINITY;
    float4 wq = make_float4(0.f, 0.f, 0.f, 0.f);            // WT: sum_c w_c * taps
    float wsum = 0.f;                                       // WT: W = sum_c w_c
    for (int c = u; c < C; c += TPG) {
        const float4 q = tq.get(c);
        mx = fmaxf(mx, fmaxf(fmaxf(q.x, q.y), fmaxf(q.z, q.w)));
        mn = fminf(mn, fminf(fminf(q.x, q.y), fminf(q.z, q.w)));
        if constexpr (WT) {
            const float wc = k2_class_weight(P.weight, c);
            wq.x = fmaf(wc, q.x, wq.x); wq.y = fmaf(wc, q.y, wq.y);
            wq.z = fmaf(wc, q.z, wq.z); wq.w = fmaf(wc, q.w, wq.w);
            wsum += wc;
        }
    }
#pragma unroll
    for (int o = TPG / 2; o > 0; o >>= 1) {
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        if constexpr (WT) {
            wq.x += __shfl_xor_sync(0xffffffffu, wq.x, o); wq.y += __shfl_xor_sync(0xffffffffu, wq.y, o);
            wq.z += __shfl_xor_sync(0xffffffffu, wq.z, o); wq.w += __shfl_xor_sync(0xffffffffu, wq.w, o);
            wsum += __shfl_xor_sync(0xffffffffu, wsum, o);
        }
    }
    const float M = mx;
    const unsigned bal = __ballot_sync(0xffffffffu, vm != 0);
    const bool warp_any = bal != 0;
    const bool grp_any = ((bal >> (lane & ~(TPG - 1))) & ((1u << TPG) - 1u)) != 0;
    const bool slow = __any_sync(0xffffffffu, vm != 0 && !((mx - mn) < K2_FAST_RANGE));
    const float Mk = M * LOG2E;
    const float2 ly2 = make_float2(((float)(2 * u) + 0.5f) * RS, ((float)(2 * u) + 1.5f) * RS);

    // per class: (E, rho) of the thread's two rows from the group's taps q = (a, b, c, d)
    auto row_exp = [&](const float4 q, float2& e2, float2& r2) {
        const float2 dv = ffma2(make_float2(q.x, q.y), bc2(-1.f), make_float2(q.z, q.w));   // (c-a, d-b)
        const float2 L2 = ffma2(ly2, bc2(dv.x), bc2(q.x));
        const float2 R2 = ffma2(ly2, bc2(dv.y), bc2(q.y));
        const float2 rl2 = ffma2(L2, bc2(-1.f), R2);
        const float2 aE = ffma2(rl2, bc2(LX0 * LOG2E), ffma2(L2, bc2(LOG2E), bc2(-Mk)));
        const float2 aR = fmul2(rl2, bc2(RS * LOG2E));
        e2 = make_float2(ex2f(aE.x), ex2f(aE.y));
        r2 = make_float2(ex2f(aR.x), ex2f(aR.y));
    };

    float loss = 0.f;
    if constexpr (SPLIT) {
        // -sum of the target logits of the strip (the -onehot gradient came from the label prepass)
        if (vm) {
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const float lyr = r ? ly2.y : ly2.x;
#pragma unroll
                for (int j = 0; j < S; ++j) {
                    if (!((vm >> (r * 16 + j)) & 1u)) continue;
                    const unsigned t = (lw[r * (S / 2) + (j >> 1)] >> (16 * (j & 1))) & 0xffffu;
                    const float4 q = tq.get(t);
                    const float L = fmaf(lyr, q.z - q.x, q.x), R = fmaf(lyr, q.w - q.y, q.y);
                    loss -= fmaf(((float)j + 0.5f) * RS, R - L, L);
                }
            }
        }
    }
    if (warp_any && !slow) {
        // ---- pass A ---------------------------------------------------------------------------------------------
        float2 U2[S];                                       // S(j) of rows (0,1); then U(j) = g / S(j)
#pragma unroll
        for (int j = 0; j < S; ++j) U2[j] = make_float2(0.f, 0.f);
        {
            // software pipeline: taps two classes ahead, exponentials one class ahead (the tile has two
            // padding class slots, so the look-ahead needs no bounds check)
            float2 eN, rN;
            row_exp(tq.get(0), eN, rN);
            float4 qn = tq.get(1);
#pragma unroll 2
            for (int c = 0; c < C; ++c) {
                float2 e2 = eN;
                const float2 r2 = rN;
                row_exp(qn, eN, rN);
                qn = tq.get(c + 2);
#pragma unroll
                for (int j = 0; j < S; ++j) {
                    U2[j] = fadd2(U2[j], e2);
                    if (j < S - 1) e2 = fmul2(e2, r2);
                }
            }
        }
        // ---- loss: log-sum-exp part, and U = g / S --------------------------------------------------------------
        // (lg2.approx / rcp.approx: 2^-22 relative; S is in [exp(-K2_FAST_RANGE), C], never denormal)
        int va4[4] = {0, 0, 0, 0};                          // WT: V of the four taps, in units of 1 / (4 S^2)
        if constexpr (WT) {
            // per counted pixel: a*(M + ln S), U = g*a / S, the target logit and the -(1-eps) w_t onehot runs
#pragma unroll
            for (int j = 0; j < S; ++j) {
                if (!((vm >> j) & 1u)) U2[j].x = 0.f;
                if (!((vm >> (16 + j)) & 1u)) U2[j].y = 0.f;
            }
            if (vm) {
                const float wscale = -gs / (float)(4 * S * S);
#pragma unroll
                for (int r = 0; r < 2; ++r) {
                    if (!((vm >> (r * 16)) & 0xffffu)) continue;
                    const long long* row = P.labels + ((size_t)n * P.H + (y0 + r)) * P.W + x0;
                    const float lyr = r ? ly2.y : ly2.x;
                    const int lyi = 2 * (2 * u + r) + 1;    // lambda_y * 2S
                    int cur = -1, sw0 = 0, sw1 = 0, tw0 = 0, tw1 = 0;
                    float wcur = 0.f;
                    auto flush = [&]() {
                        if (cur >= 0 && gb) {
                            const float ws = wscale * wcur;
                            atomicAdd(gA + (size_t)cur * plane, ws * (float)((2 * S - lyi) * sw0));
                            atomicAdd(gB + (size_t)cur * plane, ws * (float)((2 * S - lyi) * sw1));
                            atomicAdd(gC + (size_t)cur * plane, ws * (float)(lyi * sw0));
                            atomicAdd(gD + (size_t)cur * plane, ws * (float)(lyi * sw1));
                        }
                    };
#pragma unroll
                    for (int jj = 0; jj < S / 2; ++jj) {
                        if (!((vm >> (r * 16 + 2 * jj)) & 3u)) continue;
                        const longlong2 t2 = __ldg(reinterpret_cast<const longlong2*>(row + 2 * jj));
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const int j = 2 * jj + e;
                            if (!((vm >> (r * 16 + j)) & 1u)) continue;
                            const int t = (int)(e ? t2.y : t2.x);
                            const float wt = P.one_m_eps * k2_class_weight(P.weight, t);
                            const float a = fmaf(P.eps_c, wsum, wt);
                            float& sv = r ? U2[j].y : U2[j].x;
                            loss = fmaf(a, fmaf(lg2f(sv), LN2, M), loss);
                            sv = gs * a * rcpf(sv);
                            const float4 q = tq.get(t);
                            const float L = fmaf(lyr, q.z - q.x, q.x), R = fmaf(lyr, q.w - q.y, q.y);
                            loss = fmaf(-wt, fmaf(((float)j + 0.5f) * RS, R - L, L), loss);
                            if (t != cur) { flush(); cur = t; wcur = wt; sw0 = 0; sw1 = 0; }
                            sw0 += 2 * S - (2 * j + 1);
                            sw1 += 2 * j + 1;
                            tw0 += 2 * S - (2 * j + 1);
                            tw1 += 2 * j + 1;
                        }
                    }
                    flush();
                    va4[0] += (2 * S - lyi) * tw0; va4[1] += (2 * S - lyi) * tw1;
                    va4[2] += lyi * tw0;           va4[3] += lyi * tw1;
                }
                // smoothing: -(eps/C) sum over the counted pixels of the interpolated sum_c w_c x_c
                const float vq = (float)va4[0] * wq.x + (float)va4[1] * wq.y + (float)va4[2] * wq.z + (float)va4[3] * wq.w;
                loss = fmaf(-P.eps_c * (1.f / (float)(4 * S * S)), vq, loss);
            }
        } else {
            float lg = 0.f;
#pragma unroll
            for (int j = 0; j < S; ++j) {
                const bool va = (vm >> j) & 1u, vb = (vm >> (16 + j)) & 1u;
                const float sa = va ? U2[j].x : 1.f, sb = vb ? U2[j].y : 1.f;
                lg += lg2f(sa) + lg2f(sb);
                U2[j] = make_float2(va ? gs * rcpf(sa) : 0.f, vb ? gs * rcpf(sb) : 0.f);
            }
            loss += fmaf((float)__popc(vm), M, lg * LN2);
        }
        // ---- target logits and the -g*onehot term (exact integer tap weights, run-length per row) ---------------
        if (!SPLIT && !WT && vm) {
            const float wscale = -gs / (float)(4 * S * S);
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                if (!((vm >> (r * 16)) & 0xffffu)) continue;
                const long long* row = P.labels + ((size_t)n * P.H + (y0 + r)) * P.W + x0;
                const float lyr = r ? ly2.y : ly2.x;
                const int lyi = 2 * (2 * u + r) + 1;        // lambda_y * 2S
                int cur = -1, sw0 = 0, sw1 = 0;
                auto flush = [&]() {
                    if (cur >= 0 && gb) {
                        atomicAdd(gA + (size_t)cur * plane, wscale * (float)((2 * S - lyi) * sw0));
                        atomicAdd(gB + (size_t)cur * plane, wscale * (float)((2 * S - lyi) * sw1));
                        atomicAdd(gC + (size_t)cur * plane, wscale * (float)(lyi * sw0));
                        atomicAdd(gD + (size_t)cur * plane, wscale * (float)(lyi * sw1));
                    }
                };
#pragma unroll
                for (int jj = 0; jj < S / 2; ++jj) {
                    if (!((vm >> (r * 16 + 2 * jj)) & 3u)) continue;
                    const longlong2 t2 = __ldg(reinterpret_cast<const longlong2*>(row + 2 * jj));
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int j = 2 * jj + e;
                        if (!((vm >> (r * 16 + j)) & 1u)) continue;
                        const int t = (int)(e ? t2.y : t2.x);
                        const float4 q = tq.get(t);
                        const float L = fmaf(lyr, q.z - q.x, q.x), R = fmaf(lyr, q.w - q.y, q.y);
                        loss -= fmaf(((float)j + 0.5f) * RS, R - L, L);
                        if (t != cur) { flush(); cur = t; sw0 = 0; sw1 = 0; }
                        sw0 += 2 * S - (2 * j + 1);
                        sw1 += 2 * j + 1;
                    }
                }
                flush();
            }
        }
        // ---- pass B: tap gradients of every class -----------------------------------------------------------------
        // The TPG lanes of a group add their four tap gradients with a shuffle butterfly (lane role*(TPG/4) of the
        // group ends up with tap `role`); two more shuffles merge the taps that neighbouring groups of the warp tile
        // share (horizontally, then vertically), and the (2+1) x (WGX+1) lanes that then hold one source cell each
        // send it to L2 as ONE float reduction per (class, cell) - 9 instead of 16 per 2x2 tile, no shared-memory
        // round trip.
        if (gb) {
            const int role = (u * 4) / TPG;
            const bool writer = (u % (TPG / 4)) == 0;
            const int gy_ = gl / WGX, gx_ = gl % WGX, ry = role >> 1, rx = role & 1;
            // horizontal: (gx_, rx = 0) with gx_ >= 1 takes (gx_ - 1, rx = 1); vertical: (gy_ = 1, ry = 0) takes (gy_ = 0, ry = 1)
            const bool h_dst = writer && rx == 0 && gx_ >= 1;
            const int h_src = ((gy_ * WGX + (gx_ >= 1 ? gx_ - 1 : 0)) * TPG) + (ry * 2 + 1) * (TPG / 4);
            const bool holder_x = writer && (rx == 0 || gx_ == WGX - 1);          // holds a complete column cell
            const bool v_dst = holder_x && gy_ == 1 && ry == 0;
            const int v_src = ((0 * WGX + gx_) * TPG) + (2 + rx) * (TPG / 4);
            const bool holder = holder_x && ((gy_ == 0 && ry == 0) || gy_ == 1);   // one lane per source cell
            const int cy = gy_ + ry, cx = gx_ + rx;                                // cell of the warp tile
            const int uy = GY0 - 1 + cy, ux = GX0 - 1 + cx;                        // unclamped source cell
            float* dst = (holder && uy <= P.h && ux <= P.w)
                             ? gb + (size_t)clampi(uy, 0, P.h - 1) * P.w + clampi(ux, 0, P.w - 1) : nullptr;
            const float2 omy = make_float2(1.f - ly2.x, 1.f - ly2.y);
            float kv = 0.f;                                  // WT: -g (eps/C) V of this lane's source cell
            if constexpr (WT) {
                float V0 = (float)va4[0], V1 = (float)va4[1], V2 = (float)va4[2], V3 = (float)va4[3];
                group_reduce4<TPG>(V0, V1, V2, V3, u);
                const float hv = __shfl_sync(0xffffffffu, V0, h_src);
                if (h_dst) V0 += hv;
                const float vv = __shfl_sync(0xffffffffu, V0, v_src);
                if (v_dst) V0 += vv;
                kv = V0 != 0.f ? -gs * P.eps_c * (1.f / (float)(4 * S * S)) * V0 : 0.f;
            }
            float2 eN, rN;
            row_exp(tq.get(0), eN, rN);
            float4 qn = tq.get(1);
#pragma unroll 2
            for (int c = 0; c < C; ++c) {
                const float2 e2 = eN, r2 = rN;
                row_exp(qn, eN, rN);                         // class c+1
                qn = tq.get(c + 2);                          // class c+2
                float2 h2 = U2[S - 1], d2 = h2;
                h2 = ffma2(h2, r2, U2[S - 2]);
#pragma unroll
                for (int j = S - 3; j >= 0; --j) {
                    d2 = ffma2(d2, r2, h2);
                    h2 = ffma2(h2, r2, U2[j]);
                }
                const float2 rd2 = fmul2(r2, d2);                              // sum_j j U rho^j
                const float2 G2 = fmul2(e2, h2);                               // sum_j g
                const float2 X2 = ffma2(fmul2(e2, rd2), bc2(RS), fmul2(G2, bc2(LX0)));   // sum_j lambda_x g
                const float2 N2 = ffma2(X2, bc2(-1.f), G2);                    // sum_j (1 - lambda_x) g
                const float2 a2 = fmul2(omy, N2), b2 = fmul2(omy, X2), c2 = fmul2(ly2, N2), d2y = fmul2(ly2, X2);
                float A = a2.x + a2.y, Bv = b2.x + b2.y, Cv = c2.x + c2.y, Dv = d2y.x + d2y.y;
                group_reduce4<TPG>(A, Bv, Cv, Dv, u);
                A = grp_any ? A : 0.f;                       // no valid pixel -> exactly zero (taps may be NaN)
                const float hx = __shfl_sync(0xffffffffu, A, h_src);
                if (h_dst) A += hx;
                const float vx = __shfl_sync(0xffffffffu, A, v_src);
                if (v_dst) A += vx;
                if constexpr (WT) A = fmaf(kv, k2_class_weight(P.weight, c), A);
                if (dst) atomicAdd(dst + (size_t)c * plane, A);
            }
        }
    } else if (warp_any) {
        loss += k2_strip_slow<S, SPLIT, TQ, WT>(tq, vm, n, y0, x0, u, P, gs, gA, gB, gC, gD);
    }
    loss = warp_sum(loss);
    if (lane == 0 && loss != 0.f) atomicAdd(P.loss_sum, (double)loss);
}

}  // namespace lc2is
