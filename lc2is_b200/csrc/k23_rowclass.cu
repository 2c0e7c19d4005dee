// k23_rc: bilinear x16 upsample + softmax cross-entropy (forward + backward) + argmax / confusion matrix in ONE
// persistent kernel of independent warps - the dominant kernel of the head step at the aux-head geometry.
//
// Replaces  F.interpolate(bilinear, size=H) + CrossEntropyLoss fwd/bwd   (reference model/loss.py:17-21, engine.py:94-100)
//      and  F.interpolate + Softmax2d + JaccardIndex's argmax / bincount (reference metrics.py:84-92, :127-134)
// on the same low-resolution class-plane-major logits [B,C,h,w]; the upsampled [B,C,H,W] tensor never exists.
//
// Geometry (as in k2_strip.cuh): a GROUP (ky,kx), ky = -1..h-1, kx = -1..w-1, is the 16 x 16 pixel region that interpolates
// between source cells (ky,kx)..(ky+1,kx+1) (index-clamped).  A JOB is one group; a warp owns a job from start to end (no
// CTA barrier anywhere), jobs are dealt to the warps of a persistent grid.  Jobs are short (~30 us) so that the warps'
// last jobs end close together: the kernel's tail is a fraction of one job time.
//
//   stage     the group's source cells of every class land in the warp's private shared-memory tile by ONE TMA box
//             (4-D tensor map [B][C][h][w], box 1 x C x 2 x 8 starting on a 16-byte boundary - the group's two clamped
//             columns can straddle a 4-cell boundary; out-of-bounds cells are zero-filled and never used).  The landing
//             zone doubles as the U tile of the job, so the box of the warp's NEXT job is issued at the end of the job; its
//             latency is covered by the other 15 warps of the SM.
//   convert   lane = class: the cells become one quad (a, b, c-a, d-b) per class, and the same sweep finds the softmax
//             shift M = max tap of the group, the tap range and non-finite taps.
//   row phase lane = (half hw, pixel row i): both halves own the 16 rows of the group, half hw sweeps the classes
//             [hw CP/2, (hw+1) CP/2).  One sweep over its classes does BOTH
//             pass A of the cross-entropy - S(j) = sum_c E_c rho_c^j: the upsampled logit is linear along the row, so the
//               16 exponentials of a (class,row) are a geometric progression: 2 ex2, then FADD2 / FMUL2 over column pairs
//             and the running maximum of the argmax - v(j) = fma(j, delta, v0) as 8 FFMA2, one FMNMX3 per pixel and class
//               PAIR, chunks of 8 classes: "if (cm > best) { best = cm; chunk = k }".
//             The halves meet by shuffles (lane ^ 16): half hw keeps pixel columns 8 hw .. 8 hw + 7, adds the other half's
//             partial S(j) and takes its (maximum, chunk) where that is larger - the upper half's only when STRICTLY
//             larger, so the first class still wins a tie - then rescans the winning chunk of each of its pixels for the
//             FIRST class that reaches the maximum (torch.argmax's tie rule).
//             Half hw then handles the labels of its 8 columns: log-sum-exp, U(j) = valid / S(j) (to shared memory),
//             target logits, the exact integer -onehot tap weights and the confusion-matrix counts, by a sweep over its
//             pixel columns (match.any over the rows).
//   class phase lane = CLASS: for a class the 16 x 16 terms are E(y) rho(y)^j with E(y+1) = E(y) sigma and
//             rho(y+1) = rho(y) tau - four ex2 per class - and  h = sum_j U(j) rho^j,  d = dh/drho  by one Horner sweep
//             per row pair (two FFMA2 per pixel pair, U broadcast from shared memory) give the four tap gradients in
//             registers: no cross-lane reduction; the four source cells of the group leave as one float reduction each.
// Border jobs (top / bottom row or left / right column of groups, 2 (h + w) of the (h + 1)(w + 1) per image) are 1-D:
//             their two taps of one axis are the same clamped cell, so the logit is constant along that axis.  Row phase:
//             lane (hw, i) evaluates the diagonal pixel (i, i) - row i's value (left / right) or column i's (top / bottom),
//             with the 2-D expression, so the argmax is bit-identical - one direct ex2 per class, a running (maximum,
//             first class) instead of chunks and rescan; shuffles then give the shared code its per-lane state.  Class
//             phase: U summed along the constant axis gives 16 weights, and per class 16 terms give the two distinct
//             cells' gradients (one at a corner).  Jobs are numbered interior first, so the short border jobs fill the tail.
// Jobs whose taps are not finite or span more than K2_FAST_RANGE take exact per-pixel paths (warp-uniform, one row per
// lane of the lower half; ATen's taps, so 0 * inf poisons the same pixels as argmax(softmax(interpolate(x)))).
#include "common.cuh"
#include "k2_strip.cuh"
#include "tc_common.cuh"
#include "k23_common.cuh"
#include <mutex>
#include <unordered_map>

namespace lc2is {

constexpr int RC_S = 16;                 // scale
constexpr int RC_CH = 8;                 // classes per argmax chunk (even)
constexpr int RC_CTR_SLOTS = 64;         // job-counter pairs (see launch_k23_rc)
constexpr float RC_PAD = -1.0e30f;       // padding classes: exp -> 0, never the argmax
// staggered start (launch_k23_rc): delay unit and the jobs per warp from which it is on (tuned at cfg2, B = 16 and 8)
constexpr unsigned RC_STAGGER_NS = 8000u;
constexpr int RC_STAGGER_MIN_JOBS = 3;
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
    int CP;                          // classes incl. padding, a multiple of 8: each half-warp sweeps CP / 2 classes, whole
                                     // chunks of RC_CH and at most one last chunk of 4; the quads tile has CP + 4 entries
    int use_tma;
    long long njobs;                 // = groups = B (h+1) (w+1)
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
// per warp: [0] start, then two stamps per job (class phase starts, job ends), [RC_STAMP_SLOTS - 1] = stamps taken
constexpr int RC_STAMP_SLOTS = 32;
__device__ unsigned long long rc_stamps[148 * 16 * RC_STAMP_SLOTS];
__device__ __forceinline__ unsigned long long rc_now() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#endif
struct RCJob {
    int n, ky, kx;                   // image, group row (-1..h-1), group column (-1..w-1)
};
// Job order: the (h-1)(w-1) interior groups of every image first (image-major, row-major), then the 2(h+w) border groups
// of every image (per image: top row, bottom row, left column, right column).  Border jobs are the short ones (1-D row
// and class phases), so they fill the kernel's tail.
__device__ __noinline__ RCJob rc_decode(const RCParams& P, long long job) {
    RCJob J;
    const int iw = P.w - 1;                                   // interior groups per group row
    const long long ninner = (long long)P.B * (P.h - 1) * iw;
    if (job < ninner) {
        const int per_img = (P.h - 1) * iw;
        J.n = (int)(job / per_img);
        const int rem = (int)(job - (long long)J.n * per_img);
        J.ky = rem / iw;
        J.kx = rem - J.ky * iw;
    } else {
        job -= ninner;
        const int per_img = 2 * (P.h + P.w);
        J.n = (int)(job / per_img);
        int rem = (int)(job - (long long)J.n * per_img);
        if (rem < 2 * (P.w + 1)) {                            // top / bottom row, corners included
            const bool bot = rem > P.w;
            J.ky = bot ? P.h - 1 : -1;
            J.kx = rem - (bot ? P.w + 1 : 0) - 1;
        } else {                                              // left / right column without the corners
            rem -= 2 * (P.w + 1);
            const bool right = rem >= P.h - 1;
            J.kx = right ? P.w - 1 : -1;
            J.ky = rem - (right ? P.h - 1 : 0);
        }
    }
    return J;
}

// The cell tile of a job: rows ys, ys+1 and columns xs..xs+7 of every class, [c][2][8], out of bounds = 0 (never used).
// The box starts on a 16-byte boundary (the TMA unit rejects other start addresses: xs is a multiple of 4 cells) at the
// first cell the group's index-clamped taps touch, so no coordinate is negative.
__device__ __forceinline__ int rc_xs(const RCJob& J) { return max(J.kx, 0) & ~3; }
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
    constexpr unsigned FULL = 0xffffffffu;
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

    const int C = P.C, CP = P.CP, CPH = CP / 2;
    // all landing zones first (each a multiple of 128 bytes, the alignment TMA wants), then the per-warp rest
    float* cells = reinterpret_cast<float*>(smem_raw + (size_t)warp * P.cells_bytes);   // [C][2][8] TMA landing zone
    float* quads = reinterpret_cast<float*>(smem_raw + (size_t)nwarps * P.cells_bytes + (size_t)warp * P.quads_bytes);
    //                                                                     [CP][4] = (p0, p1, q0, q1): rc_quad
    const float4* const Q4 = reinterpret_cast<const float4*>(quads);
    // The U tile [16 columns][16 rows] (and the row records before it) lives in the landing zone: the cells are dead once
    // they are converted, and the box of the NEXT job is only issued when this job's class phase has read U.
    float* Usm = cells;
    uint64_t* bar = reinterpret_cast<uint64_t*>(quads + (size_t)(CP + 4) * 4);
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
    unsigned long long* stp = rc_stamps + (size_t)(blockIdx.x * 16 + warp) * RC_STAMP_SLOTS;
    int sti = 1;
    if (lane == 0) stp[0] = rc_now();
#endif
    // De-phasing: all warps start in step and stay nearly in step (equal jobs), so the SM's 16 warps are in the FMA-bound row
    // phase together and in the LDS-bound class phase together (tools/k23_timeline.py).  A staggered start trades a few us
    // of idle warps for mixed phases from the start.
    if (P.stagger_ns) __nanosleep((unsigned)((warp >> 2) & 3) * P.stagger_ns);
    // row-phase lane mapping: half hw of the warp, pixel row i of the group (both halves own all 16 rows)
    const int hw = lane >> 4, i = lane & 15;
    const float ly = ((float)i + 0.5f) * RS;

    const int njobs = (int)P.njobs;
    int next_job = 0;
#pragma unroll 1
    for (int job = gw; job < njobs; job = next_job) {
        {
            unsigned t = 0;
            if (lane == 0) t = atomicAdd(P.ctr, 1u);
            next_job = gstride + (int)__shfl_sync(FULL, t, 0);
        }
        const RCJob J = rc_decode(P, job);
        const int n = J.n, ky = J.ky, kx = J.kx;
        // ---- wait for the taps -----------------------------------------------------------------------------
        if (P.use_tma) { tc::mbar_wait(bar, parity); parity ^= 1u; }
        else __syncwarp();

        // ---- convert (lane = class): quads, shift, range, non-finite ----------------------------------------
        float mx = -INFINITY, mn = INFINITY;
        bool bad = false;
        {
            const int xs = rc_xs(J), ys = rc_ys(J);
            const int ya = (clampi(ky, 0, P.h - 1) - ys) * 8, yb = (clampi(ky + 1, 0, P.h - 1) - ys) * 8;
            const int xa = clampi(kx, 0, P.w - 1) - xs, xb = clampi(kx + 1, 0, P.w - 1) - xs;   // 0..4
            for (int k = lane; k < CP + 4; k += 32) {     // (+4: the rescan of a 4-class last chunk reads 8 classes)
                const float* cp = cells + k * 16;
                float4 q;
                if (k < C) {
                    const float a = cp[ya + xa], b = cp[ya + xb], c = cp[yb + xa], d = cp[yb + xb];
                    mx = fmaxf(mx, fmaxf(fmaxf(a, b), fmaxf(c, d)));
                    mn = fminf(mn, fminf(fminf(a, b), fminf(c, d)));
                    bad |= !(fabsf(a) < INFINITY) | !(fabsf(b) < INFINITY) | !(fabsf(c) < INFINITY) | !(fabsf(d) < INFINITY);
                    q = rc_quad<RC_S>(a, b, c, d);
                } else {
                    q = make_float4(RC_PAD, RC_PAD, 0.f, 0.f);
                }
                reinterpret_cast<float4*>(quads)[k] = q;
            }
            // clamped staging hides ATen's second tap of the top / left border groups (row / column 1, weight 0):
            // 0 * inf = NaN poisons those pixels in the reference - look at it on the global map
            if (ky < 0 || kx < 0) {
                const float* base = P.low + (size_t)n * C * plane;
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
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            mx = fmaxf(mx, __shfl_xor_sync(FULL, mx, o));
            mn = fminf(mn, __shfl_xor_sync(FULL, mn, o));
        }
        const bool nonfinite = __any_sync(FULL, bad);
        __syncwarp();                                       // quads complete, cells free (they become the U tile)

        // ---- this lane's pixels: row i, columns 8 hw .. 8 hw + 7 - labels ---------------------------------------------
        const int y = S * ky + S / 2 + i, xh = S * kx + S / 2 + 8 * hw;
        const bool row_in = y >= 0 && y < P.H;
        const bool in = row_in && xh >= 0 && xh < P.W;      // W = 16 w: the 8 columns are all inside or all outside
        unsigned lw[4];
        {
            uint4 t = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
            if (in) t = __ldg(reinterpret_cast<const uint4*>(P.labels + ((size_t)n * P.H + y) * P.W + xh));
            lw[0] = t.x; lw[1] = t.y; lw[2] = t.z; lw[3] = t.w;
        }
        unsigned vm = 0;                                    // pixels counted by the CE (class id without the ignore flag)
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if ((lw[k] & 0xffffu) < (unsigned)C) vm |= 1u << (2 * k);
            if ((lw[k] >> 16) < (unsigned)C) vm |= 1u << (2 * k + 1);
        }
        const bool any = __any_sync(FULL, vm != 0);
        const bool slow = nonfinite || (any && !((mx - mn) < K2_FAST_RANGE));
        // Border groups: both taps of one axis are the same clamped cell, so the quads have p1 = q1 = 0 (top / bottom row
        // of groups) or q0 = q1 = 0 (left / right column): the logit is constant along that axis (over the whole group at
        // a corner), and the 2-D path's expression gives the same value at every pixel of a row (edge_x) or column (edge_y)
        const bool edge_y = ky < 0 || ky == P.h - 1, edge_x = kx < 0 || kx == P.w - 1;
        const bool border = edge_y || edge_x;
        float loss = 0.f;
        int bidx[8];                                        // predictions of the lane's 8 pixels
        float2 S2[4];                                       // fast path: S(j) of the lane's 8 pixels, column pairs

        if (!slow && border) {
            // ================= 1-D row phase: lane (hw, i) evaluates pixel (i, i), which carries the value of row i
            // (edge_x) or of column i (edge_y), for the half's classes: no recurrence, no chunks, no rescan ============
            const float Mk = mx * LOG2E, fi = (float)i;
            const float4* const Q = Q4 + hw * CPH;
            float s = 0.f, bv = -INFINITY;
            int bk = 0;
#pragma unroll 1
            for (int k = 0; k < CPH; k += 4) {              // (CPH is a multiple of 4)
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const float4 q = Q[k + u];
                    const float v = fmaf(fi, fmaf(ly, q.w, q.z), fmaf(ly, q.y, q.x));
                    s += ex2f(fmaf(v, LOG2E, -Mk));
                    if (v > bv) { bv = v; bk = k + u; }     // strictly larger: the first class of a tie stays
                }
            }
            // the halves meet: both hold the same sum (fp addition commutes); the upper half's maximum wins only when
            // strictly larger
            bk += hw * CPH;
            s += __shfl_xor_sync(FULL, s, 16);
            const float ov = __shfl_xor_sync(FULL, bv, 16);
            const int ok = __shfl_xor_sync(FULL, bk, 16);
            if (hw ? !(bv > ov) : (ov > bv)) bk = ok;
            // the shared code's per-lane state: row i, columns 8 hw .. 8 hw + 7 (edge_y: column j's value is on lane j,
            // edge_x: row i's on lane i; a corner is constant)
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {
                const int la = edge_y ? 8 * hw + 2 * jj : i, lb = edge_y ? 8 * hw + 2 * jj + 1 : i;
                S2[jj] = make_float2(__shfl_sync(FULL, s, la), __shfl_sync(FULL, s, lb));
                bidx[2 * jj] = __shfl_sync(FULL, bk, la);
                bidx[2 * jj + 1] = __shfl_sync(FULL, bk, lb);
            }
        } else if (!slow) {
            // ================= row phase: pass A + running maximum, one sweep over the half's classes ===============
            const float Mk = mx * LOG2E;
            // The loops of this kernel are kept ROLLED on purpose: the warps of an SM are at different places of the job
            // at any time, and with the loop bodies unrolled the kernel ran out of instruction cache (ncu: no_instruction was
            // the top stall reason of the 148 KB version).
            float best[S], snap[S];                         // running maximum; its value at the last chunk boundary
            unsigned bchw[S / 4];                           // chunk of the maximum, one byte per pixel
            float2 P2[S / 2];                               // this half's part of S(j), all 16 columns
#pragma unroll
            for (int k = 0; k < S / 2; ++k) P2[k] = make_float2(0.f, 0.f);
#pragma unroll
            for (int j = 0; j < S; ++j) { best[j] = -INFINITY; snap[j] = -INFINITY; }
#pragma unroll
            for (int j = 0; j < S / 4; ++j) bchw[j] = 0u;
            const int nch = (CPH + CH - 1) / CH;            // the last one has 4 classes when CPH is not a multiple of 8
            const float4* const Q = Q4 + hw * CPH;          // the half's classes
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
                    P2[jj] = fadd2(P2[jj], fadd2(e2a, e2b));
                    if (jj < S / 2 - 1) { e2a = fmul2(e2a, r2a); e2b = fmul2(e2b, r2b); }
                    const float2 va = ffma2(RC_J2[jj], da2, va0), vb = ffma2(RC_J2[jj], db2, vb0);
                    best[2 * jj] = fmax3f(va.x, vb.x, best[2 * jj]);
                    best[2 * jj + 1] = fmax3f(va.y, vb.y, best[2 * jj + 1]);
                }
            };
            // two pairs per iteration (ping-pong states A / B: no register rotation)
            PairSt A, Bq;
            setup(qp[0], qp[1], A);
            const float4* const qlast = Q + CPH - 2;        // the look-ahead stops at the half's last pair (CPH >= 4)
            float4 na = qp[2], nb = qp[3];
            qp += 4;
#pragma unroll 1
            for (int k = 0; k < nch; ++k) {
              const int npp = min(CH / 4, (CPH - k * CH) / 4);
#pragma unroll 1
              for (int p = 0; p < npp; ++p) {
                setup(na, nb, Bq);                                     // pair 2p+1
                qp = qp < qlast ? qp : qlast;
                na = qp[0]; nb = qp[1];                                // pair 2p+2
                qp += 2;
                chains(A);
                setup(na, nb, A);                                      // pair 2p+2
                qp = qp < qlast ? qp : qlast;
                na = qp[0]; nb = qp[1];                                // pair 2p+3
                qp += 2;
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
            // ---- the halves meet: half hw keeps columns 8 hw .. 8 hw + 7 and receives the other half's values of them --
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {
                const float2 keep = hw ? P2[4 + jj] : P2[jj], send = hw ? P2[jj] : P2[4 + jj];
                S2[jj] = make_float2(keep.x + __shfl_xor_sync(FULL, send.x, 16), keep.y + __shfl_xor_sync(FULL, send.y, 16));
            }
            // chunk indices of the whole class range (the upper half's chunks follow the lower half's; < 256)
            const unsigned coff = (unsigned)(hw * nch) * 0x01010101u;
            unsigned kw[2], ow[2];
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                kw[q] = (hw ? bchw[2 + q] : bchw[q]) + coff;
                ow[q] = __shfl_xor_sync(FULL, (hw ? bchw[q] : bchw[2 + q]) + coff, 16);
            }
            float bst[8];
            int bch[8];
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
                const float kb = hw ? best[8 + jj] : best[jj];
                const float ob = __shfl_xor_sync(FULL, hw ? best[jj] : best[8 + jj], 16);
                // the lower half's classes come first: the upper half's maximum wins only when strictly larger
                const bool other = hw ? !(kb > ob) : (ob > kb);
                const unsigned kc = (kw[jj >> 2] >> (8 * (jj & 3))) & 0xffu, oc = (ow[jj >> 2] >> (8 * (jj & 3))) & 0xffu;
                bst[jj] = other ? ob : kb;
                const int g = (int)(other ? oc : kc);
                bch[jj] = g * CH + (g >= nch ? CPH - nch * CH : 0);  // first class of the chunk (upper half: from CPH)
                bidx[jj] = bch[jj];
            }
            // ---- argmax phase 2: the FIRST class of the winning chunk that reaches the maximum ----------------------
            const float jh = (float)(8 * hw);
#pragma unroll 1
            for (int cc = CH - 1; cc >= 0; --cc) {          // (downwards: the last match written is the first class)
                const float4* qc = Q4 + cc;
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) {
                    const float4 q = qc[bch[jj]];
                    const float v = fmaf(jh + (float)jj, fmaf(ly, q.w, q.z), fmaf(ly, q.y, q.x));
                    if (v == bst[jj]) bidx[jj] = bch[jj] + cc;
                }
            }
        } else {
            // exact per-pixel paths, one row per lane of the lower half (nothing is counted twice)
            int* tmp = reinterpret_cast<int*>(Usm) + i * S;
            const unsigned vrow = vm | (__shfl_xor_sync(FULL, vm, 16) << 8);           // the row's 16 pixels (lower half)
            if (hw == 0) slow_argmax_row<RC_S>(SlowCtx{P.low, P.grad, P.C, P.h, P.w}, n, ky, kx, i, row_in, tmp);
            __syncwarp();
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) bidx[jj] = tmp[8 * hw + jj];
            __syncwarp();
            if (hw == 0 && vrow) loss = slow_ce_row<RC_S>(SlowCtx{P.low, P.grad, P.C, P.h, P.w}, n, ky, kx, i, vrow);
        }

        // ---- the lane's labels and predictions: a sweep over its 8 pixel COLUMNS (one column of all 16 rows per half) --
        //   confusion matrix: one 64-bit reduction per distinct (target, prediction) pair of the two columns
        //   cross-entropy   : the pixel's target logit; the -onehot term as exact integer tap weights summed over the
        //                     rows of the same column that carry the same label (their row-weight sums follow from the
        //                     match mask alone), four float reductions per distinct (label, half)
        // The sweep reads the lane's (label, prediction) records back from the still idle U tile.
        {
            unsigned* rec = reinterpret_cast<unsigned*>(Usm) + lane;
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
                const unsigned lab = (lw[jj >> 1] >> (16 * (jj & 1))) & 0xffffu;
                rec[jj * 32] = lab | ((unsigned)bidx[jj] << 16);
            }
            if (P.pred != nullptr && in) {
                long long* prow = P.pred + ((size_t)n * P.H + y) * P.W + xh;
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) prow[jj] = bidx[jj];
            }
            const int Ya = clampi(ky, 0, P.h - 1), Yb = clampi(ky + 1, 0, P.h - 1);
            const int Xa = clampi(kx, 0, P.w - 1), Xb = clampi(kx + 1, 0, P.w - 1);
            const int oA = Ya * P.w + Xa, oB = Ya * P.w + Xb, oC = Yb * P.w + Xa, oD = Yb * P.w + Xb;
            const float* lbase = P.low + (size_t)n * C * plane;
            float* gbase = (P.grad && P.onehot) ? P.grad + (size_t)n * C * plane : nullptr;
            unsigned long long* pimg = P.per_image ? P.per_image + (size_t)n * 3 * C : nullptr;
            constexpr float WSC = 1.f / (float)(4 * S * S);
            float tsub = 0.f;
#pragma unroll 2
            for (int jj = 0; jj < 8; ++jj) {
                const int j = 8 * hw + jj;                                     // pixel column in the group
                const unsigned r = rec[jj * 32];
                const unsigned lab = r & 0xffffu;
                const int t = (int)(lab & 0x7fffu), pr = (int)(r >> 16);      // bit 15: ignore flag of the CE
                const bool c = (vm >> jj) & 1u, v = in && t < C;
                const unsigned actv = __ballot_sync(FULL, v);
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
                const unsigned actc = __ballot_sync(FULL, c);
                if (c) {
                    float4 q;
                    if (!slow) q = Q4[lab];
                    else {
                        const float* t4 = lbase + (size_t)lab * plane;
                        q = rc_quad<RC_S>(__ldg(t4 + oA), __ldg(t4 + oB), __ldg(t4 + oC), __ldg(t4 + oD));
                    }
                    tsub += fmaf((float)j, fmaf(ly, q.w, q.z), fmaf(ly, q.y, q.x));
                    if (gbase) {
                        // the two halves are different columns (different tap weights): the half is part of the key
                        const unsigned m = __match_any_sync(actc, lab | ((unsigned)hw << 16));
                        if (lane == __ffs(m) - 1) {
                            const unsigned mm = (m >> (16 * hw)) & 0xffffu;          // bit i = row i
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
        // ---- log-sum-exp of the lane's pixels, U = valid / S -> shared memory (class phase) -----------------------
        if (!slow) {
            float lg = 0.f;
            float* up = Usm + (8 * hw) * 16 + i;            // U[j][row]
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {
                const bool va = (vm >> (2 * jj)) & 1u, vb = (vm >> (2 * jj + 1)) & 1u;
                const float sa = va ? S2[jj].x : 1.f, sb = vb ? S2[jj].y : 1.f;
                lg += lg2f(sa) + lg2f(sb);
                up[(2 * jj) * 16] = va ? rcpf(sa) : 0.f;
                up[(2 * jj + 1) * 16] = vb ? rcpf(sb) : 0.f;
            }
            loss += fmaf((float)__popc(vm), mx, lg * LN2);
        }

        {
            int cnt = __popc(vm);
            loss = warp_sum(loss);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(FULL, cnt, o);
            if (lane == 0) {
                if (loss != 0.f) atomicAdd(P.loss_sum, (double)loss);
                if (P.n_valid && cnt) atomicAdd(P.n_valid, (unsigned long long)cnt);
            }
        }
        __syncwarp();                                       // U tile complete

#ifdef RC_STAMPS
        if (lane == 0 && sti < RC_STAMP_SLOTS - 1) stp[sti++] = rc_now();
#endif
        // ================= class phase (lane = class): tap gradients ======================================================
        if (!slow && P.grad != nullptr && any && border) {
            float* gimg = P.grad + (size_t)n * C * plane;
            const int oA = clampi(ky, 0, P.h - 1) * P.w, oC = clampi(ky + 1, 0, P.h - 1) * P.w;
            const int cxa = clampi(kx, 0, P.w - 1), cxb = clampi(kx + 1, 0, P.w - 1);
            const float Mk = mx * LOG2E;
            // ---- 1-D: U summed along the constant axis gives 16 weights Ub(p) (p = column for edge_y, row for
            // edge_x); per class G = sum_p e(p) Ub(p) and L = sum_p lambda(p) e(p) Ub(p) are the two distinct cells'
            // gradients (G - L, L), one cell (G) at a corner.  Lane (hw, p) adds 8 of the 16 terms of Ub(p), in an
            // order that keeps both read patterns free of bank conflicts.
            {
                const int p = i;
                float t = 0.f;
#pragma unroll
                for (int r = 0; r < 8; ++r) {
                    const int rr = 8 * hw + ((r + (p >> 1) + hw) & 7);
                    t += edge_y ? Usm[p * 16 + rr] : Usm[rr * 16 + p];
                }
                t += __shfl_xor_sync(FULL, t, 16);
                __syncwarp();
                if (hw == 0) Usm[p] = t;
                __syncwarp();
            }
            const float4* const Ub4 = reinterpret_cast<const float4*>(Usm);
            const int o0 = oA + cxa, o1 = edge_y ? oA + cxb : oC + cxa;   // the same cell at a corner
#pragma unroll 1
            for (int k = lane; k < C; k += 32) {
                const float4 q = Q4[k];
                float G = 0.f, L = 0.f;
#pragma unroll 1
                for (int p4 = 0; p4 < 4; ++p4) {
                    const float4 ub = Ub4[p4];
                    const float ubv[4] = {ub.x, ub.y, ub.z, ub.w};
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const float fp = (float)(4 * p4 + u), lp = (fp + 0.5f) * RS;
                        const float v = fmaf(fp, fmaf(lp, q.w, q.z), fmaf(lp, q.y, q.x));
                        const float g = ex2f(fmaf(v, LOG2E, -Mk)) * ubv[u];
                        G += g;
                        L = fmaf(lp, g, L);
                    }
                }
                float* gk = gimg + (size_t)k * plane;
                if (o0 == o1) {
                    if (G != 0.f) red_add_f32(gk + o0, G);
                } else {
                    const float g0 = G - L;
                    if (g0 != 0.f) red_add_f32(gk + o0, g0);
                    if (L != 0.f) red_add_f32(gk + o1, L);
                }
            }
        } else if (!slow && P.grad != nullptr && any) {
            // ---- 2-D: Horner sweeps
            float* gimg = P.grad + (size_t)n * C * plane;
            const int oA = clampi(ky, 0, P.h - 1) * P.w, oC = clampi(ky + 1, 0, P.h - 1) * P.w;
            const int cxa = clampi(kx, 0, P.w - 1), cxb = clampi(kx + 1, 0, P.w - 1);
            const float Mk = mx * LOG2E;
            // NB blocks of 32 classes per sweep: one broadcast LDS.128 of U then feeds 4 * NB packed fma (with one block
            // the class phase leaned on the shared-memory pipe: 16 LDS.128 per 62 FFMA2, ncu mio_throttle / short
            // scoreboard); an odd last block goes through the NB = 1 instance.  (Scalar FFMA instead of FFMA2 measured the
            // same here: ~3 cycles per FFMA2 with three register-pair operands = 2 x ~1.5 per scalar FFMA with three
            // register operands - tools/micro/loops23.cu.)
            auto sweep = [&](auto nb_tag, int kb) {
                constexpr int NB = decltype(nb_tag)::value;
                float2 e2a[NB], e2b[NB], r2a[NB], r2b[NB], aG[NB], aX[NB], aYG[NB], aYX[NB];
                float sg4[NB], ta4[NB];
#pragma unroll
                for (int b = 0; b < NB; ++b) {
                    const int k = kb + 32 * b + lane;
                    const float4 q = Q4[k < CP ? k : CP - 1];                                  // p0, p1, q0, q1
                    // row y: v0 = p0 + ly p1, delta = q0 + ly q1, ly = (y + 0.5) / 16
                    const float aE0 = fmaf(fmaf(0.5f * RS, q.y, q.x), LOG2E, -Mk);
                    const float E0 = ex2f(aE0), sg = ex2f(q.y * (RS * LOG2E));
                    const float r0 = ex2f(fmaf(0.5f * RS, q.w, q.z) * LOG2E), ta = ex2f(q.w * (RS * LOG2E));
                    const float sg2 = sg * sg, ta2 = ta * ta;
                    e2a[b] = make_float2(E0, E0 * sg); r2a[b] = make_float2(r0, r0 * ta);
                    e2b[b] = fmul2(e2a[b], bc2(sg2)); r2b[b] = fmul2(r2a[b], bc2(ta2));
                    sg4[b] = sg2 * sg2; ta4[b] = ta2 * ta2;
                    aG[b] = make_float2(0.f, 0.f); aX[b] = aG[b]; aYG[b] = aG[b]; aYX[b] = aG[b];
                }
                const float4* U4 = reinterpret_cast<const float4*>(Usm);
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
                    const int k = kb + 32 * b + lane;
                    if (k < C) {
                        const float G = aG[b].x + aG[b].y, X = aX[b].x + aX[b].y;
                        const float YG = aYG[b].x + aYG[b].y, YX = aYX[b].x + aYX[b].y;
                        const float SX = fmaf(X, RS, G * LX0);              // sum lambda_x g
                        const float SYX = fmaf(YX, RS, YG * LX0);           // sum lambda_y lambda_x g
                        const float gD = SYX, gB = SX - SYX, gC = YG - SYX, gA = (G - SX) - gC;
                        float* gk = gimg + (size_t)k * plane;
                        if (gA != 0.f) red_add_f32(gk + oA + cxa, gA);
                        if (gB != 0.f) red_add_f32(gk + oA + cxb, gB);
                        if (gC != 0.f) red_add_f32(gk + oC + cxa, gC);
                        if (gD != 0.f) red_add_f32(gk + oC + cxb, gD);
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
        if (lane == 0 && sti < RC_STAMP_SLOTS - 1) stp[sti++] = rc_now();
#endif
        // ---- the box of the warp's next job (its latency is covered by the SM's other warps) -----------------------
        if (next_job < njobs) {
            const RCJob Jn = rc_decode(P, next_job);
            rc_stage(P, &tm, cells, bar, Jn, lane);
        }
    }
#ifdef RC_STAMPS
    if (lane == 0) stp[RC_STAMP_SLOTS - 1] = (unsigned long long)sti;
#endif
    // the next kernel of the step (the gradient scale, then the logits backward) may be scheduled once the warp has no
    // job left; it reads the gradient only after griddep_wait(), i.e. after this grid's last reduction has landed
    griddep_launch_dependents();
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

// classes incl. padding: each half-warp sweeps CP / 2 classes, a multiple of the 4 classes of one pipeline step
static int rc_cp(int C) { return (C + 7) / 8 * 8; }
static size_t rc_cells_bytes(int C) {
    size_t b = (size_t)C * 16 * 4;                                       // [C][2][8] floats
    if (b < (size_t)16 * 16 * 4) b = (size_t)16 * 16 * 4;                // ... or the U tile / row records (16 x 16 words)
    return (b + 127) / 128 * 128;
}
static size_t rc_quads_bytes(int C) { return (size_t)(rc_cp(C) + 4) * 4 * 4 + 16; }   // [CP + 4][4] floats + mbarrier

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
    P.CP = rc_cp(C);
    P.njobs = (long long)B * (h + 1) * (w + 1);
    if (P.njobs > 0x3fffffffLL) return fail(LC2IS_ERR_SHAPE, "too many groups for one launch%s");
    P.cells_bytes = (unsigned)rc_cells_bytes(C);
    P.quads_bytes = (unsigned)rc_quads_bytes(C);
    // staggered start (see the kernel): on when a warp gets RC_STAGGER_MIN_JOBS jobs or more - with fewer the idle time is
    // not won back
    P.stagger_ns = P.njobs >= (long long)RC_STAGGER_MIN_JOBS * sm_count() * nw ? RC_STAGGER_NS : 0u;
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
    return (int)cudaMemcpyFromSymbol(h_out, rc_stamps, sizeof(unsigned long long) * 148 * 16 * RC_STAMP_SLOTS);
}
#endif
}  // namespace lc2is
