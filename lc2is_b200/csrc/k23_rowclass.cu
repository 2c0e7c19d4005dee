// k23_rc: bilinear x16 upsample + softmax cross-entropy (forward + backward) + argmax / confusion matrix in ONE
// persistent kernel of independent warps - the dominant kernel of the head step at the aux-head geometry.
//
// Replaces  F.interpolate(bilinear, size=H) + CrossEntropyLoss fwd/bwd   (reference model/loss.py:17-21, engine.py:94-100)
//      and  F.interpolate + Softmax2d + JaccardIndex's argmax / bincount (reference metrics.py:84-92, :127-134)
// on the same low-resolution class-plane-major logits [B,C,h,w]; the upsampled [B,C,H,W] tensor never exists.
//
// Geometry (as in k2_strip.cuh): a GROUP (ky,kx), ky = -1..h-1, kx = -1..w-1, is the 16 x 16 pixel region that interpolates
// between source cells (ky,kx)..(ky+1,kx+1) (index-clamped).  A JOB is two horizontally adjacent groups; a warp owns a
// job from start to end (no CTA barrier anywhere), jobs are dealt round-robin to the warps of a persistent grid.
//
//   stage     the job's source cells of every class land in the warp's private shared-memory tile by ONE TMA box
//             (4-D tensor map [B][C][h][w], box 1 x C x 2 x 8 starting on a 16-byte boundary; out-of-bounds cells are
//             zero-filled and never used).  The landing zone doubles as the U tile of the job, so the box of the warp's
//             NEXT job is issued at the end of the job; its latency is covered by the other 15 warps of the SM.
//   convert   lane = class: the cells become per-group quads (a, b, c-a, d-b), and the same sweep finds the softmax shift
//             M = max tap of the group, the tap range and non-finite taps.
//   row phase lane = one pixel row of one group (2 groups x 16 rows), one sweep over the classes does BOTH
//             pass A of the cross-entropy - S(j) = sum_c E_c rho_c^j: the upsampled logit is linear along the row, so the
//               16 exponentials of a (class,row) are a geometric progression: 2 ex2, then FADD2 / FMUL2 over column pairs
//             and the running maximum of the argmax - v(j) = fma(j, delta, v0) as 8 FFMA2, one FMNMX3 per pixel and class
//               PAIR, chunks of 6 classes: "if (cm > best) { best = cm; chunk = k }", then the winning chunk is rescanned
//               per pixel for the FIRST class that reaches the maximum (torch.argmax's tie rule).
//             The row then has its log-sum-exp, U(j) = valid / S(j) (to shared memory), target logits, the exact integer
//             -onehot tap weights and its confusion-matrix counts, by a sweep over the pixel columns (match.any over rows).
//   class phase lane = CLASS: for a (class, group) the 16 x 16 terms are E(y) rho(y)^j with E(y+1) = E(y) sigma and
//             rho(y+1) = rho(y) tau - four ex2 per (class, group) - and  h = sum_j U(j) rho^j,  d = dh/drho  by one Horner
//             sweep per row pair (two FFMA2 per pixel pair, U broadcast from shared memory) give the four tap gradients
//             in registers: no cross-lane reduction; the six source cells of the job leave as one float reduction each.
// Jobs whose taps are not finite or span more than K2_FAST_RANGE take exact per-pixel paths (warp-uniform; ATen's taps, so
// 0 * inf poisons the same pixels as argmax(softmax(interpolate(x)))).
#include "common.cuh"
#include "k2_strip.cuh"
#include "tc_common.cuh"
#include "k23_common.cuh"
#include <mutex>
#include <unordered_map>

namespace lc2is {

constexpr int RC_S = 16;                 // scale
constexpr int RC_CH = 8;                 // classes per argmax chunk (even)
constexpr int RC_USTRIDE = 16 * 16 + 16; // floats per group in the U tile (+16: the two groups land in different banks)
constexpr int RC_CTR_SLOTS = 64;         // job-counter pairs (see launch_k23_rc)
constexpr float RC_PAD = -1.0e30f;       // padding classes: exp -> 0, never the argmax
// column indices of a pixel pair, (2k, 2k+1): constant-bank operands of the packed fma that evaluates the row
__constant__ float2 RC_J2[RC_S / 2] = {{0.f, 1.f}, {2.f, 3.f}, {4.f, 5.f}, {6.f, 7.f}, {8.f, 9.f}, {10.f, 11.f}, {12.f, 13.f}, {14.f, 15.f}};

struct RCParams {
    const float* low;                // [B,C,h,w]
    const unsigned short* labels;    // packed [B,H,W]: class id, bit 15 = ignore flag, 0xFFFF = not a class id
    float* grad;                     // [B,C,h,w] accumulates the un-scaled gradient (or null: forward only)
    double* loss_sum;
    unsigned long long* n_valid;     // += counted pixels (or null)
    unsigned long long* confmat;     // [C,C]
    unsigned long long* per_image;   // [B,3,C] or null
    long long* pred;                 // [B,H,W] or null
    int onehot;                      // add the -onehot term to grad
    int B, C, h, w, H, W;
    int CP;                          // classes incl. padding (multiple of RC_CH)
    int jpr;                         // jobs per group row = ceil((w + 1) / 2)
    int use_tma;
    long long njobs;
    unsigned* ctr;                   // {next job of the dynamic rounds, finished warps}: zero at launch, reset by the last warp
    unsigned cells_bytes;            // shared memory per warp: TMA landing zone (later the U tile), multiple of 128
    unsigned quads_bytes;            // shared memory per warp: quads + mbarrier
    unsigned stagger_ns;             // start delay unit: warp w of a CTA starts ((w >> 2) & 3) units late (0 = off)
};

__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int x, int y, int z,
                                            int u) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(tc::smem_u32(smem_dst)), "l"(m), "r"(tc::smem_u32(bar)), "r"(x), "r"(y), "r"(z), "r"(u)
        : "memory");
}

#ifdef RC_STAMPS
__device__ unsigned long long rc_stamps[148 * 16 * 16];
__device__ __forceinline__ unsigned long long rc_now() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#endif
struct RCJob {
    int n, ky, kx0;                  // image, group row (-1..h-1), first group column (2*jx - 1)
};
__device__ __noinline__ RCJob rc_decode(const RCParams& P, long long job) {
    RCJob J;
    const int per_img = (P.h + 1) * P.jpr;
    J.n = (int)(job / per_img);
    const int rem = (int)(job - (long long)J.n * per_img);
    const int gy = rem / P.jpr;
    J.ky = gy - 1;
    J.kx0 = 2 * (rem - gy * P.jpr) - 1;
    return J;
}

// The cell tile of a job: rows ys, ys+1 and columns xs..xs+7 of every class, [c][2][8], out of bounds = 0 (never used).
// The box starts on a 16-byte boundary (the TMA unit rejects other start addresses: xs is a multiple of 4 cells) at the
// first cell the job's index-clamped taps touch, so no coordinate is negative.
__device__ __forceinline__ int rc_xs(const RCJob& J) { return max(J.kx0, 0) & ~3; }
__device__ __forceinline__ int rc_ys(const RCJob& J) { return max(J.ky, 0); }
__device__ __forceinline__ void rc_stage(const RCParams& P, const CUtensorMap* tm, float* cells, uint64_t* bar,
                                         const RCJob& J, int lane) {
    const int xs = rc_xs(J), ys = rc_ys(J);
    if (P.use_tma) {
        if (lane == 0) {
            tc::mbar_arrive_expect_tx(bar, (uint32_t)P.C * 64u);
            tma_load_4d(cells, tm, bar, xs, ys, 0, J.n);
        }
    } else {
        const float* base = P.low + (size_t)J.n * P.C * P.h * P.w;
#pragma unroll 1
        for (int idx = lane; idx < P.C * 16; idx += 32) {
            const int c = idx >> 4, r = (idx >> 3) & 1, cx = idx & 7;
            const int y = ys + r, x = xs + cx;
            float v = 0.f;
            if (y < P.h && x < P.w) v = __ldg(base + ((size_t)c * P.h + y) * P.w + x);
            cells[idx] = v;
        }
    }
}

template <int S>
__global__ void __launch_bounds__(512, 1)
k23_rc_kernel(const __grid_constant__ CUtensorMap tm, const __grid_constant__ RCParams P) {
    static_assert(S == 16, "x16 geometry");
    constexpr float RS = 1.f / S, LX0 = 0.5f / S;
    constexpr int CH = RC_CH;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nwarps = blockDim.x >> 5;
    // The first job of every warp is dealt statically, SM-first (consecutive jobs go to different SMs); every further job
    // is taken from a global counter when the warp STARTS its current job (the box of the next job is issued at its end):
    // a CTA that starts late - an NCCL kernel of the data-parallel step holding its SM - or runs slowly just takes fewer
    // jobs instead of stretching the kernel's tail (static dealing cost 33 us per step at 2 GPUs).  The last warp to
    // finish resets the counter pair for the next launch.
    const int gw = warp * (int)gridDim.x + (int)blockIdx.x;                   // (njobs < 2^31: checked at launch)
    const int gstride = (int)gridDim.x * nwarps;
    auto retire = [&]() {
        if (lane == 0 && atomicAdd(P.ctr + 1, 1u) == (unsigned)gstride - 1u) {
            P.ctr[0] = 0u;
            P.ctr[1] = 0u;
        }
    };
    if (gw >= (int)P.njobs) { retire(); return; }                // whole warp; there is no CTA barrier below

    const int C = P.C, CP = P.CP;
    // all landing zones first (each a multiple of 128 bytes, the alignment TMA wants), then the per-warp rest
    float* cells = reinterpret_cast<float*>(smem_raw + (size_t)warp * P.cells_bytes);   // [C][2][8] TMA landing zone
    float* quads = reinterpret_cast<float*>(smem_raw + (size_t)nwarps * P.cells_bytes + (size_t)warp * P.quads_bytes);
    //                                                                     [CP][2 groups][4] = (p0, p1, q0, q1): rc_quad
    // The U tile [2][RC_USTRIDE] (U[g][j][row], and the row records before it) lives in the landing zone: the cells are
    // dead once they are converted, and the box of the NEXT job is only issued when this job's class phase has read U.
    float* Usm = cells;
    uint64_t* bar = reinterpret_cast<uint64_t*>(quads + (size_t)CP * 8);
    const size_t plane = (size_t)P.h * P.w;

    if (lane == 0) {
        tc::mbar_init(bar, 1);
        tc::fence_barrier_init();
        tc::prefetch_tmap(&tm);
    }
    __syncwarp();
    unsigned parity = 0;
    {
        const RCJob J0 = rc_decode(P, gw);
        rc_stage(P, &tm, cells, bar, J0, lane);
    }

#ifdef RC_STAMPS
    unsigned long long* stp = rc_stamps + (size_t)(blockIdx.x * 16 + warp) * 16;
    int sti = 1;
    if (lane == 0) stp[0] = rc_now();
#endif
    // De-phasing: all warps start in step and stay nearly in step (equal jobs), so the SM's 16 warps are in the FMA-bound row
    // phase together and in the LDS-bound class phase together - the first job takes 73 us against 56 us once the warps have
    // drifted apart (tools/k23_timeline.py).  A staggered start trades a few us of idle warps for mixed phases from the start.
    if (P.stagger_ns) __nanosleep((unsigned)((warp >> 2) & 3) * P.stagger_ns);
    // row-phase lane mapping
    const int gi = lane >> 4, i = lane & 15;
    const float ly = ((float)i + 0.5f) * RS;

    const int njobs = (int)P.njobs;
    int next_job = 0;
#pragma unroll 1
    for (int job = gw; job < njobs; job = next_job) {
        {
            unsigned t = 0;
            if (lane == 0) t = atomicAdd(P.ctr, 1u);
            next_job = gstride + (int)__shfl_sync(0xffffffffu, t, 0);
        }
        const RCJob J = rc_decode(P, job);
        const int n = J.n, ky = J.ky, kx0 = J.kx0;
        // ---- wait for the taps -----------------------------------------------------------------------------
        if (P.use_tma) { tc::mbar_wait(bar, parity); parity ^= 1u; }
        else __syncwarp();

        // ---- convert (lane = class): quads, shift, range, non-finite ----------------------------------------
        const bool gin0 = ky < P.h && kx0 < P.w;            // kx0 <= w-1 always; ky <= h-1 always
        const bool gin1 = ky < P.h && kx0 + 1 < P.w;
        float mx0 = -INFINITY, mn0 = INFINITY, mx1 = -INFINITY, mn1 = INFINITY;
        bool bad = false;
        {
            const int xs = rc_xs(J), ys = rc_ys(J);
            const int ya = (clampi2(ky, 0, P.h - 1) - ys) * 8, yb = (clampi2(ky + 1, 0, P.h - 1) - ys) * 8;
            int xa[2], xb[2];
#pragma unroll
            for (int g = 0; g < 2; ++g) {
                const int kx = kx0 + g;
                xa[g] = clampi2(kx, 0, P.w - 1) - xs;                 // 0..6 (phantom group: column w-1)
                xb[g] = clampi2(kx + 1, 0, P.w - 1) - xs;
            }
            for (int k = lane; k < CP; k += 32) {
                const float* cp = cells + k * 16;
                float4 q0, q1;
                if (k < C) {
                    const float a0 = cp[ya + xa[0]], b0 = cp[ya + xb[0]], c0 = cp[yb + xa[0]], d0 = cp[yb + xb[0]];
                    const float a1 = cp[ya + xa[1]], b1 = cp[ya + xb[1]], c1 = cp[yb + xa[1]], d1 = cp[yb + xb[1]];
                    mx0 = fmaxf(mx0, fmaxf(fmaxf(a0, b0), fmaxf(c0, d0)));
                    mn0 = fminf(mn0, fminf(fminf(a0, b0), fminf(c0, d0)));
                    mx1 = fmaxf(mx1, fmaxf(fmaxf(a1, b1), fmaxf(c1, d1)));
                    mn1 = fminf(mn1, fminf(fminf(a1, b1), fminf(c1, d1)));
                    bad |= !(fabsf(a0) < INFINITY) | !(fabsf(b0) < INFINITY) | !(fabsf(c0) < INFINITY) | !(fabsf(d0) < INFINITY);
                    if (gin1)
                        bad |= !(fabsf(a1) < INFINITY) | !(fabsf(b1) < INFINITY) | !(fabsf(c1) < INFINITY) | !(fabsf(d1) < INFINITY);
                    q0 = rc_quad<RC_S>(a0, b0, c0, d0);
                    q1 = rc_quad<RC_S>(a1, b1, c1, d1);
                } else {
                    q0 = make_float4(RC_PAD, RC_PAD, 0.f, 0.f);
                    q1 = q0;
                }
                reinterpret_cast<float4*>(quads)[k * 2] = q0;
                reinterpret_cast<float4*>(quads)[k * 2 + 1] = q1;
            }
            // clamped staging hides ATen's second tap of the top / left border groups (row / column 1, weight 0):
            // 0 * inf = NaN poisons those pixels in the reference - look at it on the global map
            if (ky < 0 || kx0 < 0) {
                const float* base = P.low + (size_t)n * C * plane;
#pragma unroll 1
                for (int g = 0; g < 2; ++g) {
                    const int kx = kx0 + g;
                    if (!(ky < 0 || kx < 0) || kx >= P.w) continue;
                    const int Ya = ky < 0 ? 0 : ky, Xa = kx < 0 ? 0 : kx;
                    const int Yb = min(Ya + 1, P.h - 1), Xb = min(Xa + 1, P.w - 1);
#pragma unroll 1
                    for (int k = lane; k < C; k += 32) {
                        const float* pc = base + (size_t)k * plane;
                        const float t1 = __ldg(pc + Ya * P.w + Xb), t2 = __ldg(pc + Yb * P.w + Xa), t3 = __ldg(pc + Yb * P.w + Xb);
                        bad |= !(fabsf(t1) < INFINITY) | !(fabsf(t2) < INFINITY) | !(fabsf(t3) < INFINITY);
                    }
                }
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, o));
            mn0 = fminf(mn0, __shfl_xor_sync(0xffffffffu, mn0, o));
            mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, o));
            mn1 = fminf(mn1, __shfl_xor_sync(0xffffffffu, mn1, o));
        }
        const bool nonfinite = __any_sync(0xffffffffu, bad);
        __syncwarp();                                       // quads complete, cells free (they become the U tile)

        // ---- this lane's row: labels ---------------------------------------------------------------------------
        const int kx = kx0 + gi;
        const bool group_in = gi ? gin1 : gin0;
        const int y = S * ky + S / 2 + i, x0 = S * kx + S / 2;
        const bool row_in = group_in && y >= 0 && y < P.H;
        unsigned lw16[S / 2];
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
            const int x = x0 + hh * (S / 2);
            const bool in = row_in && x >= 0 && x < P.W;
            uint4 t = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
            if (in) t = __ldg(reinterpret_cast<const uint4*>(P.labels + ((size_t)n * P.H + y) * P.W + x));
            lw16[hh * 4 + 0] = t.x; lw16[hh * 4 + 1] = t.y; lw16[hh * 4 + 2] = t.z; lw16[hh * 4 + 3] = t.w;
        }
        unsigned vm = 0;                                    // pixels counted by the CE (class id without the ignore flag)
#pragma unroll
        for (int k = 0; k < S / 2; ++k) {
            if ((lw16[k] & 0xffffu) < (unsigned)C) vm |= 1u << (2 * k);
            if ((lw16[k] >> 16) < (unsigned)C) vm |= 1u << (2 * k + 1);
        }
        const unsigned bal = __ballot_sync(0xffffffffu, vm != 0);
        const bool any0 = (bal & 0xffffu) != 0, any1 = (bal >> 16) != 0;
        const float M = gi ? mx1 : mx0;
        const bool wide = (any0 && !((mx0 - mn0) < K2_FAST_RANGE)) || (any1 && !((mx1 - mn1) < K2_FAST_RANGE));
        const bool slow = nonfinite || wide;
        const float4* Q = reinterpret_cast<const float4*>(quads) + gi;
        float loss = 0.f;
        int bidx[S];
        float2 S2[S / 2];                                   // fast path: S(j) of the row, column pairs

        if (!slow) {
            // ================= row phase: pass A + running maximum, one sweep over the classes ======================
            const float Mk = M * LOG2E;
            // The loops of this kernel are kept ROLLED on purpose: the warps of an SM are at different places of the job
            // at any time, and with the loop bodies unrolled the kernel ran out of instruction cache (ncu: no_instruction was
            // the top stall reason of the 148 KB version).
            float best[S], snap[S];                         // running maximum; its value at the last chunk boundary
            unsigned bchw[S / 4];                           // chunk of the maximum, one byte per pixel
#pragma unroll
            for (int k = 0; k < S / 2; ++k) S2[k] = make_float2(0.f, 0.f);
#pragma unroll
            for (int j = 0; j < S; ++j) { best[j] = -INFINITY; snap[j] = -INFINITY; }
#pragma unroll
            for (int j = 0; j < S / 4; ++j) bchw[j] = 0u;
            const int nch = CP / CH;
            const float4* qp = Q;
            // software pipeline over the class pairs: the exponentials of pair p+1 and the quads of pair p+2 are in
            // flight while the chains of pair p run (a warp issues in order: without this every pair starts with the
            // full LDS -> FFMA -> MUFU latency)
            struct PairSt { float v0a, da, v0b, db, Ea, ra, Eb, rb; };
            auto setup = [&](const float4 qa, const float4 qb, PairSt& t) {
                t.v0a = fmaf(ly, qa.y, qa.x); t.da = fmaf(ly, qa.w, qa.z);
                t.v0b = fmaf(ly, qb.y, qb.x); t.db = fmaf(ly, qb.w, qb.z);
                t.Ea = ex2f(fmaf(t.v0a, LOG2E, -Mk)); t.ra = ex2f(t.da * LOG2E);
                t.Eb = ex2f(fmaf(t.v0b, LOG2E, -Mk)); t.rb = ex2f(t.db * LOG2E);
            };
            auto chains = [&](const PairSt& t) {
                float2 e2a = make_float2(t.Ea, t.Ea * t.ra), e2b = make_float2(t.Eb, t.Eb * t.rb);
                const float2 r2a = bc2(t.ra * t.ra), r2b = bc2(t.rb * t.rb);
                const float2 da2 = bc2(t.da), db2 = bc2(t.db), va0 = bc2(t.v0a), vb0 = bc2(t.v0b);
#pragma unroll
                for (int jj = 0; jj < S / 2; ++jj) {
                    S2[jj] = fadd2(S2[jj], fadd2(e2a, e2b));
                    if (jj < S / 2 - 1) { e2a = fmul2(e2a, r2a); e2b = fmul2(e2b, r2b); }
                    const float2 va = ffma2(RC_J2[jj], da2, va0), vb = ffma2(RC_J2[jj], db2, vb0);
                    best[2 * jj] = fmax3f(va.x, vb.x, best[2 * jj]);
                    best[2 * jj + 1] = fmax3f(va.y, vb.y, best[2 * jj + 1]);
                }
            };
            // two pairs per iteration (ping-pong states A / B: no register rotation)
            PairSt A, Bq;
            setup(qp[0], qp[2], A);
            const float4* const qlast = Q + (CP - 2) * 2;   // the look-ahead stops at the last pair (CP >= 8)
            float4 na = qp[4], nb = qp[6];
            qp += 8;
#pragma unroll 1
            for (int k = 0; k < nch; ++k) {
#pragma unroll 1
              for (int p = 0; p < CH / 4; ++p) {
                setup(na, nb, Bq);                                     // pair 2p+1
                qp = qp < qlast ? qp : qlast;
                na = qp[0]; nb = qp[2];                                // pair 2p+2
                qp += 4;
                chains(A);
                setup(na, nb, A);                                      // pair 2p+2
                qp = qp < qlast ? qp : qlast;
                na = qp[0]; nb = qp[2];                                // pair 2p+3
                qp += 4;
                chains(Bq);
              }
              // chunk boundary: pixels whose maximum moved inside this chunk (strictly up) remember the chunk
              const unsigned kk = (unsigned)k;
#pragma unroll
              for (int j = 0; j < S; ++j) {
                  // if (best != snap) { snap = best; byte (j & 3) of bchw[j / 4] = k; }  - three instructions
                  if ((j & 3) == 0)
                      asm("{\n.reg .pred p;\nsetp.neu.f32 p, %2, %0;\n@p mov.f32 %0, %2;\n@p prmt.b32 %1, %1, %3, 0x3214;\n}"
                          : "+f"(snap[j]), "+r"(bchw[j >> 2]) : "f"(best[j]), "r"(kk));
                  else if ((j & 3) == 1)
                      asm("{\n.reg .pred p;\nsetp.neu.f32 p, %2, %0;\n@p mov.f32 %0, %2;\n@p prmt.b32 %1, %1, %3, 0x3240;\n}"
                          : "+f"(snap[j]), "+r"(bchw[j >> 2]) : "f"(best[j]), "r"(kk));
                  else if ((j & 3) == 2)
                      asm("{\n.reg .pred p;\nsetp.neu.f32 p, %2, %0;\n@p mov.f32 %0, %2;\n@p prmt.b32 %1, %1, %3, 0x3410;\n}"
                          : "+f"(snap[j]), "+r"(bchw[j >> 2]) : "f"(best[j]), "r"(kk));
                  else
                      asm("{\n.reg .pred p;\nsetp.neu.f32 p, %2, %0;\n@p mov.f32 %0, %2;\n@p prmt.b32 %1, %1, %3, 0x4210;\n}"
                          : "+f"(snap[j]), "+r"(bchw[j >> 2]) : "f"(best[j]), "r"(kk));
              }
            }
            int bch[S];
#pragma unroll
            for (int j = 0; j < S; ++j) bch[j] = (int)((bchw[j >> 2] >> (8 * (j & 3))) & 0xffu);
            // ---- argmax phase 2: the FIRST class of the winning chunk that reaches the maximum ----------------------
#pragma unroll
            for (int j = 0; j < S; ++j) { bch[j] *= CH; bidx[j] = bch[j]; }
#pragma unroll 1
            for (int cc = CH - 1; cc >= 0; --cc) {          // (downwards: the last match written is the first class)
                const float4* qc = Q + cc * 2;
#pragma unroll
                for (int j = 0; j < S; ++j) {
                    const float4 q = qc[bch[j] * 2];
                    const float v = fmaf((float)j, fmaf(ly, q.w, q.z), fmaf(ly, q.y, q.x));
                    if (v == best[j]) bidx[j] = bch[j] + cc;
                }
            }
        } else {
            int* tmp = reinterpret_cast<int*>(Usm) + lane * S;
            slow_argmax_row<RC_S>(SlowCtx{P.low, P.grad, P.C, P.h, P.w}, n, ky, kx, i, row_in, tmp);
#pragma unroll
            for (int j = 0; j < S; ++j) bidx[j] = tmp[j];
            __syncwarp();
            if (vm) loss = slow_ce_row<RC_S>(SlowCtx{P.low, P.grad, P.C, P.h, P.w}, n, ky, kx, i, vm);
        }

        // ---- the row's labels and predictions: a sweep over the 16 pixel COLUMNS (column j of all 32 rows at once) --
        //   confusion matrix: one 64-bit reduction per distinct (target, prediction) pair of the column
        //   cross-entropy   : the pixel's target logit; the -onehot term as exact integer tap weights summed over the
        //                     rows of the same group that carry the same label (their row-weight sums follow from
        //                     the match mask alone), four float reductions per distinct (label, group)
        // The sweep reads the row's (label, prediction) records back from the still idle U tile.
        {
            const unsigned inmask = !row_in ? 0u : (x0 < 0 ? 0xff00u : (x0 + S > P.W ? 0x00ffu : 0xffffu));
            unsigned* rec = reinterpret_cast<unsigned*>(Usm) + lane;
#pragma unroll
            for (int j = 0; j < S; ++j) {
                const unsigned lab = (lw16[j >> 1] >> (16 * (j & 1))) & 0xffffu;
                rec[j * 32] = lab | ((unsigned)bidx[j] << 16);
            }
            if (P.pred != nullptr && inmask) {
                long long* prow = P.pred + ((size_t)n * P.H + y) * P.W + x0;
#pragma unroll
                for (int j = 0; j < S; ++j)
                    if ((inmask >> j) & 1u) prow[j] = bidx[j];
            }
            const int Ya = clampi2(ky, 0, P.h - 1), Yb = clampi2(ky + 1, 0, P.h - 1);
            const int Xa = clampi2(kx, 0, P.w - 1), Xb = clampi2(kx + 1, 0, P.w - 1);
            const int oA = Ya * P.w + Xa, oB = Ya * P.w + Xb, oC = Yb * P.w + Xa, oD = Yb * P.w + Xb;
            const float* lbase = P.low + (size_t)n * C * plane;
            float* gbase = (P.grad && P.onehot) ? P.grad + (size_t)n * C * plane : nullptr;
            unsigned long long* pimg = P.per_image ? P.per_image + (size_t)n * 3 * C : nullptr;
            constexpr float WSC = 1.f / (float)(4 * S * S);
            float tsub = 0.f;
#pragma unroll 2
            for (int j = 0; j < S; ++j) {
                const unsigned r = rec[j * 32];
                const unsigned lab = r & 0xffffu;
                const int t = (int)(lab & 0x7fffu), pr = (int)(r >> 16);      // bit 15: ignore flag of the CE
                const bool c = (vm >> j) & 1u, v = ((inmask >> j) & 1u) && t < C;
                const unsigned actv = __ballot_sync(0xffffffffu, v);
                if (v) {
                    const int key = t * C + pr;
                    const unsigned m = __match_any_sync(actv, key);
                    if (lane == __ffs(m) - 1) {
                        const unsigned long long cnt = (unsigned long long)__popc(m);
                        atomicAdd(&P.confmat[key], cnt);
                        if (pimg) {
                            if (t == pr) atomicAdd(&pimg[t], cnt);
                            atomicAdd(&pimg[C + t], cnt);
                            atomicAdd(&pimg[2 * C + pr], cnt);
                        }
                    }
                }
                const unsigned actc = __ballot_sync(0xffffffffu, c);
                if (c) {
                    float4 q;
                    if (!slow) q = Q[lab * 2];
                    else {
                        const float* t4 = lbase + (size_t)lab * plane;
                        q = rc_quad<RC_S>(__ldg(t4 + oA), __ldg(t4 + oB), __ldg(t4 + oC), __ldg(t4 + oD));
                    }
                    tsub += fmaf((float)j, fmaf(ly, q.w, q.z), fmaf(ly, q.y, q.x));
                    if (gbase) {
                        const unsigned m = __match_any_sync(actc, lab | ((unsigned)gi << 16));
                        if (lane == __ffs(m) - 1) {
                            const unsigned mm = (m >> (16 * gi)) & 0xffffu;          // bit i = row i of this group
                            const int cnt = __popc(mm);
                            const int si = __popc(mm & 0xAAAAu) + 2 * __popc(mm & 0xCCCCu) + 4 * __popc(mm & 0xF0F0u) +
                                           8 * __popc(mm & 0xFF00u);                // sum of the row indices
                            const int sb = 2 * si + cnt, st = 2 * S * cnt - sb;      // sums of (2i+1), 2S - (2i+1)
                            const float c1 = -WSC * (float)(2 * j + 1), c0 = -WSC * (float)(2 * S - (2 * j + 1));
                            float* gp = gbase + (size_t)lab * plane;
                            red_add_f32(gp + oA, c0 * (float)st); red_add_f32(gp + oB, c1 * (float)st);
                            red_add_f32(gp + oC, c0 * (float)sb); red_add_f32(gp + oD, c1 * (float)sb);
                        }
                    }
                }
            }
            loss -= tsub;
            __syncwarp();
        }
        // ---- log-sum-exp of the row, U = valid / S -> shared memory (class phase) ---------------------------------
        if (!slow) {
            float lg = 0.f;
            float* up = Usm + gi * RC_USTRIDE + i;
#pragma unroll
            for (int jj = 0; jj < S / 2; ++jj) {
                const bool va = (vm >> (2 * jj)) & 1u, vb = (vm >> (2 * jj + 1)) & 1u;
                const float sa = va ? S2[jj].x : 1.f, sb = vb ? S2[jj].y : 1.f;
                lg += lg2f(sa) + lg2f(sb);
                up[(2 * jj) * 16] = va ? rcpf(sa) : 0.f;
                up[(2 * jj + 1) * 16] = vb ? rcpf(sb) : 0.f;
            }
            loss += fmaf((float)__popc(vm), M, lg * LN2);
        }

        {
            int cnt = __popc(vm);
            loss = warp_sum(loss);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
            if (lane == 0) {
                if (loss != 0.f) atomicAdd(P.loss_sum, (double)loss);
                if (P.n_valid && cnt) atomicAdd(P.n_valid, (unsigned long long)cnt);
            }
        }
        __syncwarp();                                       // U tile complete

#ifdef RC_STAMPS
        if (lane == 0 && sti < 15) stp[sti++] = rc_now();
#endif
        // ================= class phase (lane = class): tap gradients by Horner sweeps ==============================
        if (!slow && P.grad != nullptr && (any0 || any1)) {
            float* gimg = P.grad + (size_t)n * C * plane;
            const int cy0 = clampi2(ky, 0, P.h - 1), cy1 = clampi2(ky + 1, 0, P.h - 1);
            int cxs[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) cxs[c] = clampi2(kx0 + c, 0, P.w - 1);
            const float Mk0 = mx0 * LOG2E, Mk1 = mx1 * LOG2E;
            // NB blocks of 32 classes per sweep: one broadcast LDS.128 of U then feeds 4 * NB packed fma (with one block
            // the class phase leaned on the shared-memory pipe: 16 LDS.128 per 62 FFMA2, ncu mio_throttle / short
            // scoreboard); an odd last block goes through the NB = 1 instance.  (Scalar FFMA instead of FFMA2 measured the
            // same here: ~3 cycles per FFMA2 with three register-pair operands = 2 x ~1.5 per scalar FFMA with three
            // register operands - tools/micro/loops23.cu.)
            auto sweep = [&](auto nb_tag, int kb) {
                constexpr int NB = decltype(nb_tag)::value;
                int kq[NB];
                float cell[NB][6];
#pragma unroll
                for (int b = 0; b < NB; ++b) {
                    const int k = kb + 32 * b + lane;
                    kq[b] = (k < CP ? k : CP - 1) * 2;
#pragma unroll
                    for (int c = 0; c < 6; ++c) cell[b][c] = 0.f;
                }
#pragma unroll
                for (int g = 0; g < 2; ++g) {
                    if (!(g ? any1 : any0)) continue;
                    float2 e2a[NB], e2b[NB], r2a[NB], r2b[NB], aG[NB], aX[NB], aYG[NB], aYX[NB];
                    float sg4[NB], ta4[NB];
#pragma unroll
                    for (int b = 0; b < NB; ++b) {
                        const float4 q = reinterpret_cast<const float4*>(quads)[kq[b] + g];      // p0, p1, q0, q1
                        // row y: v0 = p0 + ly p1, delta = q0 + ly q1, ly = (y + 0.5) / 16
                        const float aE0 = fmaf(fmaf(0.5f * RS, q.y, q.x), LOG2E, -(g ? Mk1 : Mk0));
                        const float E0 = ex2f(aE0), sg = ex2f(q.y * (RS * LOG2E));
                        const float r0 = ex2f(fmaf(0.5f * RS, q.w, q.z) * LOG2E), ta = ex2f(q.w * (RS * LOG2E));
                        const float sg2 = sg * sg, ta2 = ta * ta;
                        e2a[b] = make_float2(E0, E0 * sg); r2a[b] = make_float2(r0, r0 * ta);
                        e2b[b] = fmul2(e2a[b], bc2(sg2)); r2b[b] = fmul2(r2a[b], bc2(ta2));
                        sg4[b] = sg2 * sg2; ta4[b] = ta2 * ta2;
                        aG[b] = make_float2(0.f, 0.f); aX[b] = aG[b]; aYG[b] = aG[b]; aYX[b] = aG[b];
                    }
                    const float4* U4 = reinterpret_cast<const float4*>(Usm + g * RC_USTRIDE);
                    float2 lya = make_float2(0.5f * RS, 1.5f * RS), lyb = make_float2(2.5f * RS, 3.5f * RS);
#pragma unroll 1
                    for (int up = 0; up < 4; ++up) {
                        // rows 4up..4up+3: chain a = rows (4up, 4up+1), chain b = rows (4up+2, 4up+3)
                        float2 ha[NB], hb[NB], dA[NB], dB[NB];
                        float4 u = U4[(S - 1) * 4];
#pragma unroll
                        for (int b = 0; b < NB; ++b) {
                            ha[b] = make_float2(u.x, u.y); hb[b] = make_float2(u.z, u.w);
                            dA[b] = ha[b]; dB[b] = hb[b];
                        }
                        u = U4[(S - 2) * 4];
#pragma unroll
                        for (int b = 0; b < NB; ++b) {
                            ha[b] = ffma2(ha[b], r2a[b], make_float2(u.x, u.y));
                            hb[b] = ffma2(hb[b], r2b[b], make_float2(u.z, u.w));
                        }
#pragma unroll
                        for (int j = S - 3; j >= 0; --j) {
                            u = U4[j * 4];
#pragma unroll
                            for (int b = 0; b < NB; ++b) {
                                dA[b] = ffma2(dA[b], r2a[b], ha[b]);
                                dB[b] = ffma2(dB[b], r2b[b], hb[b]);
                                ha[b] = ffma2(ha[b], r2a[b], make_float2(u.x, u.y));
                                hb[b] = ffma2(hb[b], r2b[b], make_float2(u.z, u.w));
                            }
                        }
#pragma unroll
                        for (int b = 0; b < NB; ++b) {
                            const float2 Ga = fmul2(e2a[b], ha[b]), Gb = fmul2(e2b[b], hb[b]);                // sum_j g
                            const float2 Xa = fmul2(fmul2(e2a[b], r2a[b]), dA[b]);                            // sum_j j g
                            const float2 Xb = fmul2(fmul2(e2b[b], r2b[b]), dB[b]);
                            aG[b] = fadd2(aG[b], fadd2(Ga, Gb));
                            aX[b] = fadd2(aX[b], fadd2(Xa, Xb));
                            aYG[b] = ffma2(lya, Ga, ffma2(lyb, Gb, aYG[b]));
                            aYX[b] = ffma2(lya, Xa, ffma2(lyb, Xb, aYX[b]));
                            e2a[b] = fmul2(e2a[b], bc2(sg4[b])); e2b[b] = fmul2(e2b[b], bc2(sg4[b]));
                            r2a[b] = fmul2(r2a[b], bc2(ta4[b])); r2b[b] = fmul2(r2b[b], bc2(ta4[b]));
                        }
                        ++U4;
                        lya = fadd2(lya, bc2(4.f * RS)); lyb = fadd2(lyb, bc2(4.f * RS));
                    }
#pragma unroll
                    for (int b = 0; b < NB; ++b) {
                        const float G = aG[b].x + aG[b].y, X = aX[b].x + aX[b].y;
                        const float YG = aYG[b].x + aYG[b].y, YX = aYX[b].x + aYX[b].y;
                        const float SX = fmaf(X, RS, G * LX0);              // sum lambda_x g
                        const float SYX = fmaf(YX, RS, YG * LX0);           // sum lambda_y lambda_x g
                        const float gD = SYX, gB = SX - SYX, gC = YG - SYX, gA = (G - SX) - gC;
                        cell[b][g] += gA; cell[b][g + 1] += gB; cell[b][3 + g] += gC; cell[b][3 + g + 1] += gD;
                    }
                }
#pragma unroll
                for (int b = 0; b < NB; ++b) {
                    const int k = kb + 32 * b + lane;
                    if (k < C) {
                        float* gk = gimg + (size_t)k * plane;
#pragma unroll
                        for (int c = 0; c < 3; ++c) {
                            if (cell[b][c] != 0.f) red_add_f32(gk + (size_t)cy0 * P.w + cxs[c], cell[b][c]);
                            if (cell[b][3 + c] != 0.f) red_add_f32(gk + (size_t)cy1 * P.w + cxs[c], cell[b][3 + c]);
                        }
                    }
                }
            };
            int kb = 0;
#pragma unroll 1
            for (; kb + 32 < C; kb += 64) sweep(std::integral_constant<int, 2>{}, kb);
            if (kb < C) sweep(std::integral_constant<int, 1>{}, kb);
        }
        __syncwarp();                                       // quads / U free for the next job
#ifdef RC_STAMPS
        if (lane == 0 && sti < 15) stp[sti++] = rc_now();
#endif
        // ---- the box of the warp's next job (its latency is covered by the SM's other warps) -----------------------
        if (next_job < njobs) {
            const RCJob Jn = rc_decode(P, next_job);
            rc_stage(P, &tm, cells, bar, Jn, lane);
        }
    }
#ifdef RC_STAMPS
    if (lane == 0) stp[15] = (unsigned long long)sti;
#endif
    retire();
}

// ---- host: 4-D fp32 tensor map of the low-resolution logits, cached per (pointer, shape) ---------------------------
struct RCMapKey {
    const void* p; int B, C, h, w;
    bool operator==(const RCMapKey& o) const { return p == o.p && B == o.B && C == o.C && h == o.h && w == o.w; }
};
struct RCMapHash {
    size_t operator()(const RCMapKey& k) const {
        size_t x = (size_t)k.p;
        x ^= ((size_t)k.B * 1000003u) ^ ((size_t)k.C << 20) ^ ((size_t)k.h << 40) ^ ((size_t)k.w << 52);
        return x * 0x9E3779B97F4A7C15ull;
    }
};
static int rc_tensor_map(const float* low, int B, int C, int h, int w, CUtensorMap* out) {
    static std::mutex mu;
    static std::unordered_map<RCMapKey, CUtensorMap, RCMapHash> cache;
    const RCMapKey key{low, B, C, h, w};
    std::lock_guard<std::mutex> lk(mu);
    auto it = cache.find(key);
    if (it != cache.end()) { *out = it->second; return 0; }
    PFN_encodeTiled enc = get_encode_tiled();
    if (!enc) return fail(LC2IS_ERR_ARG, "cuTensorMapEncodeTiled entry point not found%s");
    cuuint64_t dims[4] = {(cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)C, (cuuint64_t)B};
    cuuint64_t strides[3] = {(cuuint64_t)w * 4, (cuuint64_t)w * h * 4, (cuuint64_t)w * h * C * 4};
    cuuint32_t box[4] = {8, 2, (cuuint32_t)C, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (void*)low, dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(LC2IS_ERR_ARG, "cuTensorMapEncodeTiled(low) failed (%s%lld)", "", (long long)r);
    if (cache.size() >= 256) cache.clear();
    cache.emplace(key, *out);
    return 0;
}

static size_t rc_cells_bytes(int C) {
    size_t b = (size_t)C * 16 * 4;                                       // [C][2][8] floats
    if (b < (size_t)2 * RC_USTRIDE * 4) b = (size_t)2 * RC_USTRIDE * 4;  // ... or the U tile / row records
    return (b + 127) / 128 * 128;
}
static size_t rc_quads_bytes(int C) {
    const int CP = (C + RC_CH - 1) / RC_CH * RC_CH;
    return (size_t)CP * 8 * 4 + 16;
}

// warps per CTA (one CTA per SM) for C classes; 0 = does not fit
int rc_warps_for(int C) {
    const size_t wb = rc_cells_bytes(C) + rc_quads_bytes(C);
    int nw = (int)((size_t)227 * 1024 / wb);
    if (nw > 16) nw = 16;
    return nw >= 8 ? nw : 0;
}

int launch_k23_rc(const float* d_low, const uint16_t* d_labels_packed, int B, int C, int h, int w, int H, int W,
                  double* d_loss_sum, float* d_grad_low, int onehot, int64_t* d_n_valid, int64_t* d_confmat,
                  int64_t* d_per_image, int64_t* d_pred, cudaStream_t st) {
    const int nw = rc_warps_for(C);
    if (!nw) return LC2IS_ERR_UNSUPPORTED;
    RCParams P;
    P.low = d_low; P.labels = d_labels_packed; P.grad = d_grad_low; P.loss_sum = d_loss_sum;
    P.n_valid = (unsigned long long*)d_n_valid; P.confmat = (unsigned long long*)d_confmat;
    P.per_image = (unsigned long long*)d_per_image; P.pred = (long long*)d_pred; P.onehot = onehot;
    P.B = B; P.C = C; P.h = h; P.w = w; P.H = H; P.W = W;
    P.CP = (C + RC_CH - 1) / RC_CH * RC_CH;
    P.jpr = (w + 1 + 1) / 2;
    P.njobs = (long long)B * (h + 1) * P.jpr;
    if (P.njobs > 0x3fffffffLL) return fail(LC2IS_ERR_SHAPE, "too many groups for one launch%s");
    P.cells_bytes = (unsigned)rc_cells_bytes(C);
    P.quads_bytes = (unsigned)rc_quads_bytes(C);
    // staggered start (see the kernel): on when a warp gets three jobs or more - with fewer the idle time is not won back
    P.stagger_ns = P.njobs >= 3LL * sm_count() * nw ? 8000u : 0u;
    P.use_tma = (C <= 256 && w % 4 == 0 && ((uintptr_t)d_low % 16) == 0) ? 1 : 0;
    CUtensorMap tm;
    memset(&tm, 0, sizeof(tm));
    if (P.use_tma)
        if (int e = rc_tensor_map(d_low, B, C, h, w, &tm)) return e;
    const size_t smem = ((size_t)P.cells_bytes + P.quads_bytes) * nw;
    static std::once_flag once;
    static cudaError_t attr_err = cudaSuccess;
    static unsigned* ctr_pool = nullptr;                    // RC_CTR_SLOTS self-resetting counter pairs, used round-robin
    std::call_once(once, [] {
        attr_err = cudaFuncSetAttribute(k23_rc_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (attr_err == cudaSuccess) attr_err = cudaMalloc(&ctr_pool, RC_CTR_SLOTS * 2 * sizeof(unsigned));
        if (attr_err == cudaSuccess) attr_err = cudaMemset(ctr_pool, 0, RC_CTR_SLOTS * 2 * sizeof(unsigned));
    });
    if (attr_err != cudaSuccess) return cuda_fail(attr_err, "k23_rc_kernel set-up (shared-memory attribute / job counters)");
    // launches in flight at the same time (different streams) must not share a pair: 64 pairs in rotation
    static std::atomic<unsigned> seq{0};
    P.ctr = ctr_pool + 2 * (seq.fetch_add(1, std::memory_order_relaxed) % RC_CTR_SLOTS);
    long long ctas = (P.njobs + nw - 1) / nw;
    if (ctas > sm_count()) ctas = sm_count();
    k23_rc_kernel<16><<<(unsigned)ctas, nw * 32, smem, st>>>(tm, P);
    LC2IS_CHECK_LAUNCH("k23_rc_kernel");
    return 0;
}

#ifdef RC_STAMPS
extern "C" int lc2is_debug_stamps(unsigned long long* h_out) {
    return (int)cudaMemcpyFromSymbol(h_out, rc_stamps, sizeof(unsigned long long) * 148 * 16 * 16);
}
#endif
}  // namespace lc2is
