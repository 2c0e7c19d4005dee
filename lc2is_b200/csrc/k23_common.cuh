// Device code shared by the fused upsample + cross-entropy + argmax kernels (k23_rowclass.cu: x16 row / class phases;
// k23_block.cu: x4, one 4 x 4 pixel group per lane): float reductions, the tap "quad" form and the exact per-pixel paths
// for groups whose taps are not finite or span too wide a range.
#pragma once
#include "common.cuh"
#include "k2_strip.cuh"

namespace lc2is {

struct SlowCtx {
    const float* low;                // [B,C,h,w]
    float* grad;                     // [B,C,h,w] or null
    int C, h, w;
};

// float reduction to GLOBAL memory (atomicAdd on a pointer of unknown state space expands to a generic-address sequence)
__device__ __forceinline__ void red_add_f32(float* p, float v) {
    asm volatile("red.global.add.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}

// exact per-pixel argmax of one row with ATen's taps on the global map (non-finite logits; rare)
// (results go through the warp's idle U tile: out[j] - a pointer to registers would put the caller's array on the stack)
template <int S>
__device__ __noinline__ void slow_argmax_row(const SlowCtx P, int n, int ky, int kx, int i, bool row_in, int* out) {
    const float ly = ((float)i + 0.5f) * (1.f / S);
    const int ya = ky < 0 ? 0 : ky, xa = kx < 0 ? 0 : kx;
    const int yb = min(ya + 1, P.h - 1), xb = min(xa + 1, P.w - 1);
    const float tyy = ky < 0 ? 0.f : ly;
    const float* base = P.low + (size_t)n * P.C * P.h * P.w;
#pragma unroll 1
    for (int j = 0; j < S; ++j) {
        const float tx = kx < 0 ? 0.f : ((float)j + 0.5f) * (1.f / S);
        float best = -INFINITY;
        int idx = 0;
        bool bad = false;
        for (int c = 0; c < P.C && row_in; ++c) {
            const float* pc = base + (size_t)c * P.h * P.w;
            const float qx = __ldg(pc + ya * P.w + xa), qy = __ldg(pc + ya * P.w + xb);
            const float qz = __ldg(pc + yb * P.w + xa), qw = __ldg(pc + yb * P.w + xb);
            const float r0 = fmaf(qy, tx, qx * (1.f - tx)), r1 = fmaf(qw, tx, qz * (1.f - tx));
            const float v = fmaf(r1, tyy, r0 * (1.f - tyy));
            bad |= !(v < INFINITY);
            if (v > best) { best = v; idx = c; }
        }
        out[j] = bad ? 0 : idx;
    }
}

// exact per-pixel cross-entropy of one row (index-clamped taps on the global map): returns sum(lse) of the valid pixels
// and adds the softmax term of the gradient with float reductions
template <int S>
__device__ __noinline__ float slow_ce_row(const SlowCtx P, int n, int ky, int kx, int i, unsigned vm) {
    const int C = P.C;
    const size_t plane = (size_t)P.h * P.w;
    const int Ya = clampi(ky, 0, P.h - 1), Yb = clampi(ky + 1, 0, P.h - 1);
    const int Xa = clampi(kx, 0, P.w - 1), Xb = clampi(kx + 1, 0, P.w - 1);
    const float* b = P.low + (size_t)n * C * plane;
    const int oA = Ya * P.w + Xa, oB = Ya * P.w + Xb, oC = Yb * P.w + Xa, oD = Yb * P.w + Xb;
    float* gb = P.grad ? P.grad + (size_t)n * C * plane : nullptr;
    const float ly = ((float)i + 0.5f) * (1.f / S);
    float loss = 0.f;
    for (int j = 0; j < S; ++j) {
        if (!((vm >> j) & 1u)) continue;
        const float lx = ((float)j + 0.5f) * (1.f / S);
        float m = -INFINITY;
        for (int c = 0; c < C; ++c) {
            const float* q = b + (size_t)c * plane;
            const float qa = __ldg(q + oA), qb = __ldg(q + oB), qc = __ldg(q + oC), qd = __ldg(q + oD);
            const float L = fmaf(ly, qc - qa, qa), R = fmaf(ly, qd - qb, qb);
            m = fmaxf(m, fmaf(lx, R - L, L));
        }
        float sum = 0.f;
        for (int c = 0; c < C; ++c) {
            const float* q = b + (size_t)c * plane;
            const float qa = __ldg(q + oA), qb = __ldg(q + oB), qc = __ldg(q + oC), qd = __ldg(q + oD);
            const float L = fmaf(ly, qc - qa, qa), R = fmaf(ly, qd - qb, qb);
            sum += ex2f((fmaf(lx, R - L, L) - m) * LOG2E);
        }
        loss += logf(sum) + m;
        if (gb) {
            const float uu = 1.f / sum;
            const float wa = (1.f - ly) * (1.f - lx), wb = (1.f - ly) * lx, wc = ly * (1.f - lx), wd = ly * lx;
            for (int c = 0; c < C; ++c) {
                const float* q = b + (size_t)c * plane;
                const float qa = __ldg(q + oA), qb = __ldg(q + oB), qc = __ldg(q + oC), qd = __ldg(q + oD);
                const float L = fmaf(ly, qc - qa, qa), R = fmaf(ly, qd - qb, qb);
                const float gg = ex2f((fmaf(lx, R - L, L) - m) * LOG2E) * uu;
                float* g = gb + (size_t)c * plane;
                red_add_f32(g + oA, gg * wa); red_add_f32(g + oB, gg * wb);
                red_add_f32(g + oC, gg * wc); red_add_f32(g + oD, gg * wd);
            }
        }
    }
    return loss;
}

__device__ __forceinline__ float fmax3f(float a, float b, float c) { return fmaxf(fmaxf(a, b), c); }

// The group's taps (a b / c d) as two linear forms in lambda_y: the logit of pixel column j of the row at lambda_y is
//   v(j) = v0 + j * delta,   v0 = p0 + lambda_y * p1 (column 0),   delta = q0 + lambda_y * q1 (column step)
// (exact in fp32 on the dyadic exactness set).
template <int S>
__device__ __forceinline__ float4 rc_quad(float a, float b, float c, float d) {
    constexpr float RS = 1.f / S, LX0 = 0.5f / S;
    const float ba = b - a, ca = c - a, gm = (d - b) - ca;
    return make_float4(fmaf(ba, LX0, a), fmaf(gm, LX0, ca), ba * RS, gm * RS);
}


}  // namespace lc2is
