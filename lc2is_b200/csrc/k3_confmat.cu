// K3: per-pixel argmax + confusion matrix (int64, rows = target, cols = prediction).
//
// Replaces reference metrics.py:84-92 / :63-69 / :127-134 and utils.py:15-22:
//   F.interpolate(bicubic|bilinear) -> Softmax2d -> JaccardIndex (argmax + bincount).
// The argmax is taken on the logits (first index wins ties, like torch.argmax).  The reference takes it on
// softmax(logits) (metrics.py:92): in exact arithmetic the same pixel, in fp32 softmax can round a near-tie (top-2 gap
// below ~2^-23 relative to the row sum's scale) onto one value and then the FIRST of the merged classes wins; the
// parity tests bound that set (tests/test_gpu_k3.py::test_argmax_rule_vs_reference_softmax).  NaN / +inf anywhere in a
// pixel's class vector gives class 0, which is what argmax(softmax(x)) returns for an all-NaN row.
//
// Three kernels:
//   k3_full    - logits materialised at mask resolution.  HBM-bound stream: 128-bit loads,
//                8 classes in flight per thread, C x C int32 histogram privatised in shared
//                memory (warp-aggregated with match.any), flushed with int64 global atomics.
//   k3_low_fast- logits at low resolution, power-of-two scale >= 4: each thread owns a 4x4
//                pixel block that shares one set of bilinear (2x2) / bicubic (4x4) taps.
//   k3_low_gen - any output size (compute_gt_mIOU's per-image original sizes): 1 pixel/thread.
#include "common.cuh"
#include "k2_strip.cuh"
#include <type_traits>

namespace lc2is {

constexpr int K3_THREADS = 256;
constexpr int K3_SMEM_HIST_MAX_C = 300;   // 16-bit counters, two per word: 300*300*2 = 180,000 B
constexpr int K3_FLUSH_PIXELS = 60 * 1024; // flush before a 16-bit counter can overflow (< 65536 pixels between flushes)

struct ArgmaxState {
    float best;
    int idx;
    bool bad;
};
__device__ __forceinline__ void am_init(ArgmaxState& s) { s.best = -INFINITY; s.idx = 0; s.bad = false; }
__device__ __forceinline__ void am_update(ArgmaxState& s, float v, int c) {
    s.bad |= !(v < INFINITY);                 // NaN or +inf
    if (v > s.best) { s.best = v; s.idx = c; }
}
__device__ __forceinline__ int am_result(const ArgmaxState& s) { return s.bad ? 0 : s.idx; }

// Add one (target, pred) observation.  Shared histogram when hist != nullptr, else global.
__device__ __forceinline__ void hist_add(int* hist, unsigned long long* confmat,
                                         unsigned long long* per_img, int C, bool valid, int t, int p) {
    unsigned act = __ballot_sync(0xffffffffu, valid);
    if (!valid) return;
    int key = t * C + p;
    unsigned m = __match_any_sync(act, key);
    int leader = __ffs(m) - 1;
    if ((int)(threadIdx.x & 31) == leader) {
        int cnt = __popc(m);
        if (hist) {
            atomicAdd(&hist[key >> 1], cnt << ((key & 1) * 16));     // two 16-bit counters per word
        } else {
            atomicAdd(&confmat[key], (unsigned long long)cnt);
            if (per_img) {
                if (t == p) atomicAdd(&per_img[t], (unsigned long long)cnt);
                atomicAdd(&per_img[C + t], (unsigned long long)cnt);
                atomicAdd(&per_img[2 * C + p], (unsigned long long)cnt);
            }
        }
    }
}

// Flush the shared histogram of ONE image into the global matrix / per-image stats and zero it.
__device__ __forceinline__ void hist_flush(int* hist, unsigned long long* confmat,
                                           unsigned long long* per_img, int C) {
    __syncthreads();
    const int nw = (C * C + 1) >> 1;
    for (int wi = threadIdx.x; wi < nw; wi += blockDim.x) {
        const unsigned word = (unsigned)hist[wi];
        if (word) {
            hist[wi] = 0;
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const unsigned v = (word >> (16 * k)) & 0xffffu;
                const int i = wi * 2 + k;
                if (v) {
                    atomicAdd(&confmat[i], (unsigned long long)v);
                    if (per_img) {
                        int t = i / C, p = i - t * C;
                        if (t == p) atomicAdd(&per_img[t], (unsigned long long)v);
                        atomicAdd(&per_img[C + t], (unsigned long long)v);
                        atomicAdd(&per_img[2 * C + p], (unsigned long long)v);
                    }
                }
            }
        }
    }
    __syncthreads();
}

template <typename T> struct Vec;
template <> struct Vec<float> {
    static constexpr int PIX = 4;
    using V = float4;
    __device__ static __forceinline__ void load(const float* p, float (&o)[4]) {
        float4 v = __ldcs(reinterpret_cast<const float4*>(p));
        o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w;
    }
    __device__ static __forceinline__ float load1(const float* p) { return __ldcs(p); }
};
template <> struct Vec<__nv_bfloat16> {
    static constexpr int PIX = 8;
    __device__ static __forceinline__ void load(const __nv_bfloat16* p, float (&o)[8]) {
        uint4 v = __ldcs(reinterpret_cast<const uint4*>(p));
        unsigned w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            o[2 * i] = __uint_as_float(w[i] << 16);
            o[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
        }
    }
    __device__ static __forceinline__ float load1(const __nv_bfloat16* p) {
        return __bfloat162float(*p);
    }
};

// ---------------------------------------------------------------------------------------------
// k3_full: grid-stride over (image, chunk) items, contiguous range per CTA.
// VEC: vector path (HW % PIX == 0) or scalar path.
template <typename T, bool VEC>
__global__ void __launch_bounds__(K3_THREADS)
k3_full_kernel(const T* __restrict__ logits, int N, int C, int H, int W,
               const long long* __restrict__ labels, int lh, int lw,
               unsigned long long* __restrict__ confmat, unsigned long long* __restrict__ per_image,
               long long* __restrict__ pred_out, int use_smem_hist) {
    extern __shared__ int hist_smem[];
    int* hist = use_smem_hist ? hist_smem : nullptr;
    constexpr int PIX = VEC ? Vec<T>::PIX : 1;
    constexpr int U = VEC ? 16 : 8;     // independent 128-bit loads in flight per thread
    const long long HW = (long long)H * W;
    const int chunk = K3_THREADS * PIX;
    const int chunks_per_img = (int)((HW + chunk - 1) / chunk);
    const long long items = (long long)N * chunks_per_img;
    const long long per_cta = (items + gridDim.x - 1) / gridDim.x;
    const long long it0 = (long long)blockIdx.x * per_cta;
    const long long it1 = it0 + per_cta < items ? it0 + per_cta : items;
    const int ry = H / lh, rx = W / lw;

    if (hist) {
        for (int i = threadIdx.x; i < (C * C + 1) / 2; i += blockDim.x) hist[i] = 0;
        __syncthreads();
    }
    int cur_img = -1;
    int since_flush = 0;
    for (long long it = it0; it < it1; ++it) {
        const int n = (int)(it / chunks_per_img);
        const int k = (int)(it - (long long)n * chunks_per_img);
        if (n != cur_img || since_flush >= K3_FLUSH_PIXELS / chunk) {   // an item is `chunk` pixels (1024 fp32 / 2048 bf16)
            if (hist && cur_img >= 0)
                hist_flush(hist, confmat, per_image ? per_image + (size_t)cur_img * 3 * C : nullptr, C);
            cur_img = n;
            since_flush = 0;
        }
        ++since_flush;
        const long long p0 = (long long)k * chunk + (long long)threadIdx.x * PIX;
        const bool in = p0 < HW;
        ArgmaxState st[PIX];
#pragma unroll
        for (int j = 0; j < PIX; ++j) am_init(st[j]);
        if (in) {
            const T* base = logits + (size_t)n * C * HW + p0;
            int c0 = 0;
            for (; c0 + U <= C; c0 += U) {
                float v[U][PIX];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    if constexpr (VEC) Vec<T>::load(base + (size_t)(c0 + u) * HW, v[u]);
                    else v[u][0] = Vec<T>::load1(base + (size_t)(c0 + u) * HW);
                }
#pragma unroll
                for (int u = 0; u < U; ++u)
#pragma unroll
                    for (int j = 0; j < PIX; ++j) am_update(st[j], v[u][j], c0 + u);
            }
            for (; c0 < C; ++c0) {
                float v[PIX];
                if constexpr (VEC) Vec<T>::load(base + (size_t)c0 * HW, v);
                else v[0] = Vec<T>::load1(base + (size_t)c0 * HW);
#pragma unroll
                for (int j = 0; j < PIX; ++j) am_update(st[j], v[j], c0);
            }
        }
        unsigned long long* pimg = per_image ? per_image + (size_t)n * 3 * C : nullptr;
#pragma unroll
        for (int j = 0; j < PIX; ++j) {
            const long long p = p0 + j;
            bool valid = in && p < HW;
            int t = 0, pr = am_result(st[j]);
            if (valid) {
                int y = (int)(p / W), x = (int)(p - (long long)y * W);
                long long tl = labels[((size_t)n * lh + y / ry) * lw + x / rx];
                if (pred_out) pred_out[(size_t)n * HW + p] = pr;
                valid = tl >= 0 && tl < C;
                t = (int)tl;
            }
            hist_add(hist, confmat, pimg, C, valid, t, pr);
        }
    }
    if (hist && cur_img >= 0)
        hist_flush(hist, confmat, per_image ? per_image + (size_t)cur_img * 3 * C : nullptr, C);
}

// ---------------------------------------------------------------------------------------------
// k3_low_fast: power-of-two scale s in {4, 8, 16}.  Same geometry as K2 (k2_upsample_ce.cu): a GROUP is
// the bps x bps (bps = s/4) 4x4-pixel blocks that share one set of taps; one thread owns one block.
// The CTA stages the index-clamped source cells of its 32 x 64 pixel tile in shared memory once
// (cp.async), then every thread walks the classes:
//   bilinear: the 16 values of a block are l00 + i*P + j*Q + i*j*T -> evaluated incrementally with
//             packed fp32x2 adds (exact for the dyadic exactness set; fp32-order noise otherwise)
//   bicubic : ATen's evaluation order is kept (horizontal 4-tap fmaf chain, then vertical), packed
//             as fp32x2 over output-column pairs - bit-identical to the scalar chain.
// Non-finite taps (inf / NaN) send the warp down the per-pixel path that reproduces
// argmax(softmax(x)) = 0 for poisoned pixels.  Counts go to global memory with warp-aggregated
// (match.any) 64-bit atomics: a 32 x 64 tile holds few distinct (target, prediction) pairs.
struct K3LowParams {
    const float* low;
    const long long* labels;
    unsigned long long* confmat;
    unsigned long long* per_image;
    long long* pred_out;
    int C, h, w, H, W, lh, lw;
    int s, off, q, tgy, tgx;
    float rs;
};

// fast argmax update (values known finite)
__device__ __forceinline__ void am_upd(float& best, int& idx, float v, int c) {
    if (v > best) { best = v; idx = c; }
}

template <int MODE, int BPS>   // MODE 0 bilinear / 1 bicubic
__global__ void __launch_bounds__(128)
k3_low_fast_kernel(const K3LowParams P) {
    constexpr int LPG = BPS * BPS;
    constexpr int NT = MODE == 0 ? 2 : 4;                   // taps per dimension
    constexpr int HALO = MODE == 0 ? 0 : 1;                 // extra cells before the first tap
    extern __shared__ float st[];                           // [C][ncy][ncx] source cells (index-clamped)
    const int C = P.C;
    const int ncy = P.tgy + NT - 1, ncx = P.tgx + NT - 1;
    const int cs = ncy * ncx;
    const int n = blockIdx.z;
    const int GY0 = blockIdx.y * P.tgy, GX0 = blockIdx.x * P.tgx;
    const int cy0 = GY0 - 1 - HALO, cx0 = GX0 - 1 - HALO;   // first (unclamped) cell of the tile
    const float* lowb = P.low + (size_t)n * C * P.h * P.w;

    // ---- stage: cell (i,j) of the tile holds source pixel (clamp(cy0+i), clamp(cx0+j)) -------------
    // (a thread owns tile cells r, r + 128, ... and walks the classes: the cell's coordinates are computed once, not with
    // two integer divisions per copied element - the staging loop was 42 % of this kernel's instructions)
    {
        const size_t plane = (size_t)P.h * P.w;
        for (int r = threadIdx.x; r < cs; r += 128) {
            const int i = r / ncx, j = r - i * ncx;
            const int gy = clampi(cy0 + i, 0, P.h - 1), gx = clampi(cx0 + j, 0, P.w - 1);
            const float* src = lowb + (size_t)gy * P.w + gx;
            float* dst = st + r;
#pragma unroll 4
            for (int c = 0; c < C; ++c) cp_async4(dst + (size_t)c * cs, src + (size_t)c * plane);
        }
    }
    asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory");
    __syncthreads();

    const int g = threadIdx.x / LPG, u = threadIdx.x % LPG;
    const int tgy = g / P.tgx, tgx = g - tgy * P.tgx;
    const int uy = u / BPS, ux = u % BPS;
    const int ky = GY0 + tgy - 1, kx = GX0 + tgx - 1;       // floor(src) of the group, -1 .. h-1
    const int by = ky * BPS + P.q + uy, bx = kx * BPS + P.q + ux;
    const int y0 = 4 * by - P.off, x0 = 4 * bx - P.off;
    const bool group_in = ky < P.h && kx < P.w;
    // offset of tap (0,0) of this group in the tile: cell (ky - HALO, kx - HALO)
    const int o00 = (ky - HALO - cy0) * ncx + (kx - HALO - cx0);
    const float rs = P.rs;
    const float ty0 = ((float)y0 + 0.5f) * rs - 0.5f - (float)ky;     // fractional source position of row 0
    const float tx0 = ((float)x0 + 0.5f) * rs - 0.5f - (float)kx;

    // ---- non-finite taps are detected inside the class loops (a value that involves all taps of the group is folded into
    // `poison`: 0 * inf = NaN); a separate sweep over the taps was 11 % of the x4 kernel's instructions.  A warp that saw
    // one re-evaluates its groups with the exact per-pixel path below.
    bool exotic = false;

    float best[16];
    int bidx[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) { best[i] = -INFINITY; bidx[i] = 0; }

    float poison = 0.f;                                     // becomes NaN when a tap of the group is not finite
    if (group_in && !exotic) {
        if constexpr (MODE == 0) {
            // bilinear; at the clamped borders both taps are the same cell, so any lambda is exact
#pragma unroll 8
            for (int c = 0; c < C; ++c) {
                const float* p = st + (size_t)c * cs + o00;
                const float a = p[0], b = p[1], cc = p[ncx], d = p[ncx + 1];
                const float da = cc - a, db = d - b, dd = db - da;
                poison = fmaf(0.f, dd, poison);                  // dd involves all four taps: inf / NaN -> NaN
                const float L0 = fmaf(ty0, da, a), R0 = fmaf(ty0, db, b);
                const float rl = R0 - L0;
                const float l00 = fmaf(tx0, rl, L0);
                const float Pv = fmaf(tx0, dd, da) * rs;        // row step of column 0
                const float Q0 = rl * rs;                       // column step in row 0
                const float Tv = dd * rs * rs;                  // growth of the column step per row
                float2 v01 = make_float2(l00, l00 + Pv), s01 = make_float2(Q0, Q0 + Tv);
                const float2 P2 = make_float2(Pv + Pv, Pv + Pv), T2 = make_float2(Tv + Tv, Tv + Tv);
                float2 v23 = fadd2(v01, P2), s23 = fadd2(s01, T2);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    am_upd(best[0 * 4 + j], bidx[0 * 4 + j], v01.x, c);
                    am_upd(best[1 * 4 + j], bidx[1 * 4 + j], v01.y, c);
                    am_upd(best[2 * 4 + j], bidx[2 * 4 + j], v23.x, c);
                    am_upd(best[3 * 4 + j], bidx[3 * 4 + j], v23.y, c);
                    if (j < 3) { v01 = fadd2(v01, s01); v23 = fadd2(v23, s23); }
                }
            }
        } else {
            // bicubic: ATen order  out = sum_a wy[a] * (sum_b wx[b] * tap[a][b]), fmaf chains
            float2 wxp[2][4];      // (wx[j][b], wx[j+1][b]) for column pairs j = 0, 2
            float wy[4][4];
#pragma unroll
            for (int i = 0; i < 4; ++i) cubic_coeffs(ty0 + (float)i * rs, wy[i]);
            {
                float wx[4][4];
#pragma unroll
                for (int j = 0; j < 4; ++j) cubic_coeffs(tx0 + (float)j * rs, wx[j]);
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    wxp[0][b] = make_float2(wx[0][b], wx[1][b]);
                    wxp[1][b] = make_float2(wx[2][b], wx[3][b]);
                }
            }
#pragma unroll 4
            for (int c = 0; c < C; ++c) {
                const float* p = st + (size_t)c * cs + o00;
                float2 hr[4][2];                                 // horizontal result of tap row a, column pairs
#pragma unroll
                for (int a = 0; a < 4; ++a) {
                    const float t0 = p[a * ncx], t1 = p[a * ncx + 1], t2 = p[a * ncx + 2], t3 = p[a * ncx + 3];
#pragma unroll
                    for (int jp = 0; jp < 2; ++jp) {
                        float2 acc = fmul2(make_float2(t0, t0), wxp[jp][0]);
                        acc = ffma2(make_float2(t1, t1), wxp[jp][1], acc);
                        acc = ffma2(make_float2(t2, t2), wxp[jp][2], acc);
                        hr[a][jp] = ffma2(make_float2(t3, t3), wxp[jp][3], acc);
                    }
                }
                // (the cubic weights are never 0 at half-pixel offsets: every tap of the group reaches this sum)
                poison = fmaf(0.f, (hr[0][0].x + hr[1][0].x) + (hr[2][0].x + hr[3][0].x), poison);
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int jp = 0; jp < 2; ++jp) {
                        float2 acc = fmul2(hr[0][jp], make_float2(wy[i][0], wy[i][0]));
                        acc = ffma2(hr[1][jp], make_float2(wy[i][1], wy[i][1]), acc);
                        acc = ffma2(hr[2][jp], make_float2(wy[i][2], wy[i][2]), acc);
                        acc = ffma2(hr[3][jp], make_float2(wy[i][3], wy[i][3]), acc);
                        am_upd(best[i * 4 + jp * 2], bidx[i * 4 + jp * 2], acc.x, c);
                        am_upd(best[i * 4 + jp * 2 + 1], bidx[i * 4 + jp * 2 + 1], acc.y, c);
                    }
            }
        }
    }
    exotic = __any_sync(0xffffffffu, poison != poison);
    if (group_in && exotic) {
        // exact per-pixel path with the NaN / +inf rule (rare; it replaces the results above)
        ArgmaxState stt[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) am_init(stt[i]);
        for (int c = 0; c < C; ++c) {
            const float* p = st + (size_t)c * cs + o00;
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float wyv[NT], wxv[NT];
                    const float ty = ty0 + (float)i * rs, tx = tx0 + (float)j * rs;
                    if (MODE == 0) { wyv[0] = 1.f - ty; wyv[1] = ty; wxv[0] = 1.f - tx; wxv[1] = tx; }
                    else {
                        float cy[4], cx[4];
                        cubic_coeffs(ty, cy); cubic_coeffs(tx, cx);
#pragma unroll
                        for (int a = 0; a < NT; ++a) { wyv[a] = cy[a]; wxv[a] = cx[a]; }
                    }
                    float acc = 0.f;
#pragma unroll
                    for (int a = 0; a < NT; ++a) {
                        float r = p[a * ncx] * wxv[0];
#pragma unroll
                        for (int b = 1; b < NT; ++b) r = fmaf(p[a * ncx + b], wxv[b], r);
                        acc = a == 0 ? r * wyv[0] : fmaf(r, wyv[a], acc);
                    }
                    am_update(stt[i * 4 + j], acc, c);
                }
        }
#pragma unroll
        for (int i = 0; i < 16; ++i) bidx[i] = am_result(stt[i]);
    }

    // ---- labels, predictions, counts ------------------------------------------------------------------
    const int ry = P.H / P.lh, rx = P.W / P.lw;
    unsigned long long* pimg = P.per_image ? P.per_image + (size_t)n * 3 * C : nullptr;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int y = y0 + i, x = x0 + j;
            bool valid = group_in && y >= 0 && y < P.H && x >= 0 && x < P.W;
            int t = 0;
            const int pr = bidx[i * 4 + j];
            if (valid) {
                const long long tl = __ldg(P.labels + ((size_t)n * P.lh + y / ry) * P.lw + x / rx);
                if (P.pred_out) P.pred_out[((size_t)n * P.H + y) * P.W + x] = pr;
                valid = tl >= 0 && tl < C;
                t = (int)tl;
            }
            hist_add(nullptr, P.confmat, pimg, C, valid, t, pr);
        }
}

// ---------------------------------------------------------------------------------------------
// k3_strip: bilinear, scale S = 8 / 16 (the x16 aux-head geometry of the whole-step path).
// Same group geometry as the K2 strip kernel: a GROUP is the S x S pixel region between source cells
// (ky,kx)..(ky+1,kx+1); one thread owns ONE ROW of a group (S pixels), so the S lanes of a group are
// consecutive lanes and a warp owns 32/S groups whose four taps it stages as quads st[c][group][4].
// Along the row the upsampled logit is linear:  v(j) = fma(j, delta, v0)  - evaluated for all S columns
// as S/2 packed FFMA2 per class (exact on the dyadic exactness set).
// The argmax is taken in two phases so that the inner loop is one FMNMX3 per pixel per class PAIR:
//   phase 1: chunks of 8 classes; cm(j) = max over the chunk (FMNMX3), and at the end of the chunk
//            "if (cm > best) { best = cm; chunk = k }" (strict: the FIRST chunk reaching the maximum)
//   phase 2: per pixel, the 8 classes of its winning chunk are re-evaluated with the identical
//            arithmetic and scanned with a strict '>' (the FIRST class reaching the maximum).
// Non-finite taps send the warp down the exact per-pixel path (argmax(softmax(x)) = 0 for poisoned pixels).
struct K3SParams {
    const float* low;
    const void* labels;           // int64 [N,lh,lw] (nearest-upsampled) or packed uint16 [N,H,W]
    unsigned long long* confmat;
    unsigned long long* per_image;
    long long* pred_out;
    int N, C, h, w, H, W, lh, lw;
};

__device__ __forceinline__ float k3_strip_value(const float4 q, float ly, float lx0, float rsx, int j) {
    const float L = fmaf(ly, q.z - q.x, q.x), R = fmaf(ly, q.w - q.y, q.y);
    const float rl = R - L;
    return fmaf((float)j, rl * rsx, fmaf(rl, lx0, L));
}

// One row (S pixels) of one group per lane.  st4 = the group's tap quad of class 0, CS4 = float4 stride between
// classes; (ly, lx0, rsx): lambda_y of the row and lambda_x(j) = lx0 + j * rsx.  The lane's cp.async copies of the taps
// are waited for here, after the label loads have been issued.
template <int S, bool PACKED, int CS4>
__device__ __forceinline__ void k3_strip_rows(const K3SParams& P, const float4* st4, int n, int ky, int kx, int i,
                                              bool group_in, float ly, float lx0, float rsx) {
    constexpr int CH = 8;                                   // classes per chunk
    const int C = P.C;
    const int y = S * ky + S / 2 + i, x0 = S * kx + S / 2;
    const bool row_in = group_in && y >= 0 && y < P.H;
    // the row's labels (issued before the taps are waited for)
    unsigned lw16[PACKED ? S / 2 : 1];
    long long lab64[PACKED ? 1 : S];
    if constexpr (PACKED) {
        using V = typename std::conditional<S == 16, uint4, uint2>::type;
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
            const int x = x0 + hh * (S / 2);
            const bool in = row_in && x >= 0 && x < P.W;
            V t = {};
            if (in) t = __ldg(reinterpret_cast<const V*>((const unsigned short*)P.labels + ((size_t)n * P.H + y) * P.W + x));
            const unsigned* wv = reinterpret_cast<const unsigned*>(&t);
#pragma unroll
            for (int k = 0; k < S / 4; ++k) lw16[hh * (S / 4) + k] = in ? wv[k] : 0xffffffffu;
        }
    } else {
        const int ryl = P.H / P.lh, rxl = P.W / P.lw;
#pragma unroll
        for (int j = 0; j < S; ++j) {
            const int x = x0 + j;
            lab64[j] = (row_in && x >= 0 && x < P.W)
                           ? __ldg((const long long*)P.labels + ((size_t)n * P.lh + y / ryl) * P.lw + x / rxl) : -1;
        }
    }
    asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory");
    __syncwarp();

    // ---- non-finite taps? ------------------------------------------------------------------------------------
    bool exotic = false;
    for (int c = i; c < C; c += S) {
        const float4 q = st4[c * CS4];
        exotic |= !(fabsf(q.x) < INFINITY) | !(fabsf(q.y) < INFINITY) | !(fabsf(q.z) < INFINITY) | !(fabsf(q.w) < INFINITY);
    }
    exotic = __any_sync(0xffffffffu, exotic);

    int bidx[S];
    if (!exotic) {
        // ---- phase 1: running maximum per pixel, chunk of the first maximum -------------------------------
        float best[S];
        int bch[S];
#pragma unroll
        for (int j = 0; j < S; ++j) { best[j] = -INFINITY; bch[j] = 0; }
        float2 J2[S / 2];
#pragma unroll
        for (int k = 0; k < S / 2; ++k) J2[k] = make_float2((float)(2 * k), (float)(2 * k + 1));
        const int nch = (C + CH - 1) / CH;
        const float4* qp = st4;
#pragma unroll 1
        for (int k = 0; k < nch; ++k) {
            float cm[S];
#pragma unroll
            for (int j = 0; j < S; ++j) cm[j] = -INFINITY;
#pragma unroll
            for (int cc = 0; cc < CH; cc += 2) {
                const float4 qa = qp[0], qb = qp[CS4];
                qp += 2 * CS4;
                const float La = fmaf(ly, qa.z - qa.x, qa.x), Ra = fmaf(ly, qa.w - qa.y, qa.y);
                const float Lb = fmaf(ly, qb.z - qb.x, qb.x), Rb = fmaf(ly, qb.w - qb.y, qb.y);
                const float rla = Ra - La, rlb = Rb - Lb;
                const float2 va0 = make_float2(fmaf(rla, lx0, La), fmaf(rla, lx0, La)), da = make_float2(rla * rsx, rla * rsx);
                const float2 vb0 = make_float2(fmaf(rlb, lx0, Lb), fmaf(rlb, lx0, Lb)), db = make_float2(rlb * rsx, rlb * rsx);
#pragma unroll
                for (int jj = 0; jj < S / 2; ++jj) {
                    const float2 va = ffma2(J2[jj], da, va0), vb = ffma2(J2[jj], db, vb0);
                    cm[2 * jj] = fmaxf(fmaxf(va.x, vb.x), cm[2 * jj]);
                    cm[2 * jj + 1] = fmaxf(fmaxf(va.y, vb.y), cm[2 * jj + 1]);
                }
            }
#pragma unroll
            for (int j = 0; j < S; ++j)
                if (cm[j] > best[j]) { best[j] = cm[j]; bch[j] = k; }
        }
        // ---- phase 2: first class of the winning chunk that reaches the maximum ---------------------------
#pragma unroll
        for (int j = 0; j < S; ++j) {
            const int c0 = bch[j] * CH;
            float bv = -INFINITY;
            int bi = c0;
#pragma unroll
            for (int cc = 0; cc < CH; ++cc) {
                const float v = k3_strip_value(st4[(c0 + cc) * CS4], ly, lx0, rsx, j);
                if (v > bv) { bv = v; bi = c0 + cc; }
            }
            bidx[j] = bi;
        }
    } else {
        // exact per-pixel path with the NaN / +inf rule (rare)
#pragma unroll 1
        for (int j = 0; j < S; ++j) {
            ArgmaxState a;
            am_init(a);
            const float tx = lx0 + (float)j * rsx;
            for (int c = 0; c < C; ++c) {
                const float4 q = st4[c * CS4];
                const float r0 = fmaf(q.y, tx, q.x * (1.f - tx)), r1 = fmaf(q.w, tx, q.z * (1.f - tx));
                am_update(a, fmaf(r1, ly, r0 * (1.f - ly)), c);
            }
#pragma unroll
            for (int jj = 0; jj < S; ++jj)
                if (jj == j) bidx[jj] = am_result(a);
        }
    }

    // ---- labels, predictions, counts ---------------------------------------------------------------------------
    // one warp-aggregated (match.any) 64-bit reduction per distinct (target, prediction) pair of a pixel column.
    // (Per-thread run-length reductions without the warp aggregation measured faster under ncu's isolated,
    // cache-flushed launch but 20 us slower inside the step.)
    unsigned long long* pimg = P.per_image ? P.per_image + (size_t)n * 3 * C : nullptr;
#pragma unroll
    for (int j = 0; j < S; ++j) {
        const int x = x0 + j;
        bool valid = row_in && x >= 0 && x < P.W;
        int t = 0;
        const int pr = bidx[j];
        if (valid) {
            if (P.pred_out) P.pred_out[((size_t)n * P.H + y) * P.W + x] = pr;
            if constexpr (PACKED) t = (int)((lw16[j >> 1] >> (16 * (j & 1))) & 0x7fffu);   // bit 15: ignore flag of the CE
            else { const long long tl = lab64[j]; t = (tl >= 0 && tl < C) ? (int)tl : C; }
            valid = t < C;
        }
        hist_add(nullptr, P.confmat, pimg, C, valid, t, pr);
    }
}

template <int S, bool PACKED>
__global__ void __launch_bounds__(128)
k3_strip_kernel(const K3SParams P) {
    constexpr int GPW = 32 / S;                             // groups per warp
    constexpr int CS = GPW * 4;                             // floats per class in the warp's tile
    constexpr int CH = 8;                                   // classes per chunk
    constexpr float RS = 1.f / S, LX0 = 0.5f / S;
    extern __shared__ float smem[];
    const int C = P.C;
    const int lane = threadIdx.x & 31;
    const long long wg = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int gpi = (P.h + 1) * (P.w + 1);                  // groups per image
    const long long ngroups = (long long)P.N * gpi;
    if (wg * GPW >= ngroups) return;                        // whole warp; no CTA barrier below
    float* st = smem + (size_t)(threadIdx.x >> 5) * (C + CH) * CS;   // + padding: the last chunk may overrun C
    const size_t plane = (size_t)P.h * P.w;

    // ---- stage: lane -> fixed (group, tap), strided over classes -----------------------------------------
    {
        constexpr int CSTEP = 32 / CS;                      // 4 (S=16) / 2 (S=8)
        const int r = lane % CS;
        const long long gq = wg * GPW + (r >> 2);
        const int tap = r & 3;
        const bool ok = gq < ngroups;
        const int n = ok ? (int)(gq / gpi) : 0;
        const int rem = ok ? (int)(gq - (long long)n * gpi) : 0;
        const int ky = rem / (P.w + 1) - 1, kx = rem % (P.w + 1) - 1;
        // ATen's taps (UpSample.h:289-312): index0 = max(k, 0), index1 = min(index0 + 1, size - 1); at the
        // top / left border (k = -1) lambda is 0 but the second tap is still row / column 1 (matters only
        // for non-finite logits: 0 * inf = NaN)
        const int ya = ky < 0 ? 0 : ky, xa = kx < 0 ? 0 : kx;
        const int yy = (tap >> 1) ? min(ya + 1, P.h - 1) : ya, xx = (tap & 1) ? min(xa + 1, P.w - 1) : xa;
        const float* src = P.low + (size_t)n * C * plane + (size_t)yy * P.w + xx;
        float* dst = st + r;
        for (int c = lane / CS; c < C; c += CSTEP) {
            if (ok) cp_async4(dst + c * CS, src + (size_t)c * plane);
            else dst[c * CS] = 0.f;
        }
        for (int c = C + lane / CS; c < C + CH; c += CSTEP) dst[c * CS] = -3.0e38f;    // padding never wins
    }
    const int gl = lane / S, i = lane % S;
    const long long gid = wg * GPW + gl;
    const bool group_in = gid < ngroups;
    const int n = group_in ? (int)(gid / gpi) : 0;
    const int rem = group_in ? (int)(gid - (long long)n * gpi) : 0;
    const int ky = rem / (P.w + 1) - 1, kx = rem % (P.w + 1) - 1;
    const float ly = ky < 0 ? 0.f : ((float)i + 0.5f) * RS;
    const float lx0 = kx < 0 ? 0.f : LX0, rsx = kx < 0 ? 0.f : RS;      // lambda_x(j) = lx0 + j * rsx
    k3_strip_rows<S, PACKED, GPW>(P, reinterpret_cast<const float4*>(st) + gl, n, ky, kx, i, group_in, ly, lx0, rsx);
}

// ---------------------------------------------------------------------------------------------
// k3_low_gen: arbitrary output size, one pixel per thread, taps from global (L1/L2 cached).
// scale_y/scale_x = the ATen source scale (in/out as float, or 1/scale_factor).
template <int MODE>
__global__ void __launch_bounds__(K3_THREADS)
k3_low_gen_kernel(const float* __restrict__ low, int C, int h, int w, int H, int W,
                  float scale_y, float scale_x,
                  const long long* __restrict__ labels, int lh, int lw,
                  unsigned long long* __restrict__ confmat, unsigned long long* __restrict__ per_image,
                  long long* __restrict__ pred_out, int use_smem_hist) {
    extern __shared__ int hist_smem[];
    int* hist = use_smem_hist ? hist_smem : nullptr;
    const int n = blockIdx.y;
    if (hist) {
        for (int i = threadIdx.x; i < (C * C + 1) / 2; i += blockDim.x) hist[i] = 0;
        __syncthreads();
    }
    constexpr int NT = MODE == 0 ? 2 : 4;
    const long long HW = (long long)H * W;
    const int ry = H / lh, rx = W / lw;
    unsigned long long* pimg = per_image ? per_image + (size_t)n * 3 * C : nullptr;
    int since_flush = 0;
    for (long long p0 = (long long)blockIdx.x * K3_THREADS; p0 < HW; p0 += (long long)gridDim.x * K3_THREADS) {
        if (hist && ++since_flush > 200) { hist_flush(hist, confmat, pimg, C); since_flush = 0; }   // 16-bit counters
        const long long p = p0 + threadIdx.x;
        bool valid = p < HW;
        int pr = 0, t = 0;
        if (valid) {
            const int y = (int)(p / W), x = (int)(p - (long long)y * W);
            float sy = scale_y * ((float)y + 0.5f) - 0.5f;
            float sx = scale_x * ((float)x + 0.5f) - 0.5f;
            int iy[NT], ix[NT];
            float wy[NT], wx[NT];
            if (MODE == 0) {
                if (sy < 0.f) sy = 0.f;
                if (sx < 0.f) sx = 0.f;
                int ky = (int)sy, kx = (int)sx;
                ky = ky > h - 1 ? h - 1 : ky;
                kx = kx > w - 1 ? w - 1 : kx;
                float ty = sy - (float)ky, tx = sx - (float)kx;
                ty = ty < 0.f ? 0.f : (ty > 1.f ? 1.f : ty);
                tx = tx < 0.f ? 0.f : (tx > 1.f ? 1.f : tx);
                iy[0] = ky; iy[1] = ky + 1 < h ? ky + 1 : h - 1;
                ix[0] = kx; ix[1] = kx + 1 < w ? kx + 1 : w - 1;
                wy[0] = 1.f - ty; wy[1] = ty;
                wx[0] = 1.f - tx; wx[1] = tx;
            } else {
                int ky = (int)floorf(sy), kx = (int)floorf(sx);
                float cy[4], cx[4];
                cubic_coeffs(sy - (float)ky, cy);
                cubic_coeffs(sx - (float)kx, cx);
#pragma unroll
                for (int a = 0; a < NT; ++a) {
                    iy[a] = clampi(ky - 1 + a, 0, h - 1);
                    ix[a] = clampi(kx - 1 + a, 0, w - 1);
                    wy[a] = cy[a]; wx[a] = cx[a];
                }
            }
            ArgmaxState st;
            am_init(st);
            const float* base = low + (size_t)n * C * h * w;
            for (int c = 0; c < C; ++c) {
                const float* pc = base + (size_t)c * h * w;
                float acc = 0.f;
#pragma unroll
                for (int a = 0; a < NT; ++a) {
                    float r = __ldg(pc + iy[a] * w + ix[0]) * wx[0];
#pragma unroll
                    for (int b = 1; b < NT; ++b) r = fmaf(__ldg(pc + iy[a] * w + ix[b]), wx[b], r);
                    acc = a == 0 ? r * wy[0] : fmaf(r, wy[a], acc);
                }
                am_update(st, acc, c);
            }
            pr = am_result(st);
            long long tl = labels[((size_t)n * lh + y / ry) * lw + x / rx];
            if (pred_out) pred_out[(size_t)n * HW + p] = pr;
            valid = tl >= 0 && tl < C;
            t = (int)tl;
        }
        hist_add(hist, confmat, pimg, C, valid, t, pr);
    }
    if (hist) hist_flush(hist, confmat, pimg, C);
}

// ---------------------------------------------------------------------------------------------
template <typename K>
static int set_smem(K kernel, size_t bytes) {
    if (bytes > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(smem)");
    }
    return 0;
}

static int check_labels_ratio(int H, int W, int lh, int lw) {
    if (lh <= 0 || lw <= 0 || H % lh || W % lw)
        return fail(LC2IS_ERR_SHAPE, "labels [%s] must divide the mask size (%lld x %lld)", "lh,lw", H, W);
    return 0;
}

static int launch_k3_strip(const float* d_low, int N, int C, int h, int w, int H, int W, int s, const void* labels,
                           bool packed, int lh, int lw, int64_t* d_confmat, int64_t* d_per_image, int64_t* d_pred,
                           cudaStream_t st) {
    const size_t smem_warp = (size_t)(C + 8) * (32 / s) * 16;
    int wpc = 4;
    while (wpc > 1 && smem_warp * wpc > 56 * 1024) wpc /= 2;
    const size_t smem = smem_warp * wpc;
    if (smem > 200 * 1024) return LC2IS_ERR_UNSUPPORTED;
    K3SParams P;
    P.low = d_low; P.labels = labels; P.confmat = (unsigned long long*)d_confmat;
    P.per_image = (unsigned long long*)d_per_image; P.pred_out = (long long*)d_pred;
    P.N = N; P.C = C; P.h = h; P.w = w; P.H = H; P.W = W; P.lh = lh; P.lw = lw;
    const long long ngroups = (long long)N * (h + 1) * (w + 1);
    const long long warps = (ngroups + (32 / s) - 1) / (32 / s);
    const unsigned grid = (unsigned)((warps + wpc - 1) / wpc);
    auto launch = [&](auto kernel) -> int {
        if (int e = set_smem(kernel, smem)) return e;
        kernel<<<grid, wpc * 32, smem, st>>>(P);
        return 0;
    };
    int e;
    if (s == 16) e = packed ? launch(k3_strip_kernel<16, true>) : launch(k3_strip_kernel<16, false>);
    else e = packed ? launch(k3_strip_kernel<8, true>) : launch(k3_strip_kernel<8, false>);
    if (e) return e;
    LC2IS_CHECK_LAUNCH("k3_strip_kernel");
    return 0;
}

}  // namespace lc2is

using namespace lc2is;

// K2 (split form) + K3 fused for the x16 geometry: d_loss_sum += sum(lse - target logit); d_grad_low ACCUMULATES the
// un-scaled softmax term (or NULL) - and, with onehot != 0, the -onehot term as well (then the labels only need
// lc2is_pack_labels, not the label prepass); d_n_valid (optional) += #counted pixels, for labels that were packed without
// counting; d_confmat / d_per_image ACCUMULATE; d_pred optional.
namespace lc2is {
int rc_warps_for(int C);                                    // k23_rowclass.cu
int launch_k23_rc(const float* d_low, const uint16_t* d_labels_packed, int B, int C, int h, int w, int H, int W,
                  double* d_loss_sum, float* d_grad_low, int onehot, int64_t* d_n_valid, int64_t* d_confmat,
                  int64_t* d_per_image, int64_t* d_pred, cudaStream_t st);
}
extern "C" int lc2is_ce_argmax_fused_supported(int C, int h, int w, int H, int W) {
    int s = 0;
    if (!fast_scale(h, w, H, W, &s) || s != 16) return 0;
    return rc_warps_for(C) > 0 ? 1 : 0;                     // the job tiles of >= 8 warps fit one SM
}

extern "C" int lc2is_ce_argmax_fused_packed(const float* d_low, const uint16_t* d_labels_packed,
                                            int B, int C, int h, int w, int H, int W,
                                            double* d_loss_sum, float* d_grad_low, int onehot, int64_t* d_n_valid,
                                            int64_t* d_confmat, int64_t* d_per_image, int64_t* d_pred,
                                            lc2is_stream_t stream) {
    if (int e = ensure_device()) return e;
    if (B < 0 || C <= 0 || h <= 0 || w <= 0 || H <= 0 || W <= 0) return fail(LC2IS_ERR_SHAPE, "bad shape%s");
    if (B == 0) return 0;
    if (!d_low || !d_labels_packed || !d_loss_sum || !d_confmat) return fail(LC2IS_ERR_ARG, "null pointer%s");
    if ((uintptr_t)d_labels_packed % 16) return fail(LC2IS_ERR_ARG, "packed labels must be 16-byte aligned%s");
    if (!lc2is_ce_argmax_fused_supported(C, h, w, H, W))
        return fail(LC2IS_ERR_UNSUPPORTED, "fused K2+K3 needs scale 16 and a class count whose job tiles fit one SM%s");
    return launch_k23_rc(d_low, d_labels_packed, B, C, h, w, H, W, d_loss_sum, d_grad_low, onehot, d_n_valid,
                         d_confmat, d_per_image, d_pred, (cudaStream_t)stream);
}

extern "C" int lc2is_argmax_confmat_lowres_packed(const float* d_low, int N, int C, int h, int w, int H, int W,
                                                  const uint16_t* d_labels_packed,
                                                  int64_t* d_confmat, int64_t* d_per_image, int64_t* d_pred,
                                                  lc2is_stream_t stream) {
    if (int e = ensure_device()) return e;
    if (N < 0 || C <= 0 || h <= 0 || w <= 0 || H <= 0 || W <= 0) return fail(LC2IS_ERR_SHAPE, "bad shape%s");
    if (N == 0) return 0;
    if (!d_low || !d_labels_packed || !d_confmat) return fail(LC2IS_ERR_ARG, "null pointer%s");
    if ((uintptr_t)d_labels_packed % 16) return fail(LC2IS_ERR_ARG, "packed labels must be 16-byte aligned%s");
    int s = 0;
    if (!fast_scale(h, w, H, W, &s) || (s != 8 && s != 16))
        return fail(LC2IS_ERR_UNSUPPORTED, "packed-label argmax needs scale 8 or 16%s");
    int e = launch_k3_strip(d_low, N, C, h, w, H, W, s, d_labels_packed, true, H, W, d_confmat, d_per_image, d_pred,
                            (cudaStream_t)stream);
    if (e == LC2IS_ERR_UNSUPPORTED) return fail(e, "too many classes for the strip kernel%s");
    return e;
}

extern "C" int lc2is_argmax_confmat(const void* d_logits, int dtype, int N, int C, int H, int W,
                                    const int64_t* d_labels, int lh, int lw,
                                    int64_t* d_confmat, int64_t* d_per_image, int64_t* d_pred,
                                    lc2is_stream_t stream) {
    if (int e = ensure_device()) return e;
    if (N < 0 || C <= 0 || H <= 0 || W <= 0) return fail(LC2IS_ERR_SHAPE, "bad shape%s");
    if (N == 0) return 0;
    if (!d_logits || !d_labels || !d_confmat) return fail(LC2IS_ERR_ARG, "null pointer%s");
    if (int e = check_labels_ratio(H, W, lh, lw)) return e;
    cudaStream_t st = (cudaStream_t)stream;
    const int use_hist = C <= K3_SMEM_HIST_MAX_C;
    const size_t smem = use_hist ? ((size_t)C * C + 1) / 2 * sizeof(int) : 0;
    const long long HW = (long long)H * W;
    const int ctas_per_sm = smem > 100 * 1024 ? 1 : (smem > 50 * 1024 ? 2 : 4);
    auto launch = [&](auto kernel, int pix, auto ptr) -> int {
        if (int e = set_smem(kernel, smem)) return e;
        long long chunk = (long long)K3_THREADS * pix;
        long long items = (long long)N * ((HW + chunk - 1) / chunk);
        long long grid = (long long)sm_count() * ctas_per_sm;
        if (grid > items) grid = items;
        kernel<<<(unsigned)grid, K3_THREADS, smem, st>>>(ptr, N, C, H, W, (const long long*)d_labels, lh, lw,
                                                         (unsigned long long*)d_confmat,
                                                         (unsigned long long*)d_per_image,
                                                         (long long*)d_pred, use_hist);
        return 0;
    };
    int e = 0;
    if (dtype == LC2IS_F32) {
        const float* p = (const float*)d_logits;
        bool vec = HW % 4 == 0 && ((uintptr_t)p % 16 == 0);
        e = vec ? launch(k3_full_kernel<float, true>, 4, p) : launch(k3_full_kernel<float, false>, 1, p);
    } else if (dtype == LC2IS_BF16) {
        const __nv_bfloat16* p = (const __nv_bfloat16*)d_logits;
        bool vec = HW % 8 == 0 && ((uintptr_t)p % 16 == 0);
        e = vec ? launch(k3_full_kernel<__nv_bfloat16, true>, 8, p)
                : launch(k3_full_kernel<__nv_bfloat16, false>, 1, p);
    } else {
        return fail(LC2IS_ERR_ARG, "dtype must be LC2IS_F32 or LC2IS_BF16%s");
    }
    if (e) return e;
    LC2IS_CHECK_LAUNCH("k3_full_kernel");
    return 0;
}

extern "C" int lc2is_argmax_confmat_lowres(const float* d_low, int N, int C, int h, int w, int H, int W,
                                           int mode, const int64_t* d_labels, int lh, int lw,
                                           int64_t* d_confmat, int64_t* d_per_image, int64_t* d_pred,
                                           lc2is_stream_t stream) {
    if (int e = ensure_device()) return e;
    if (N < 0 || C <= 0 || h <= 0 || w <= 0 || H <= 0 || W <= 0) return fail(LC2IS_ERR_SHAPE, "bad shape%s");
    if (mode != LC2IS_BILINEAR && mode != LC2IS_BICUBIC) return fail(LC2IS_ERR_ARG, "bad mode%s");
    if (N == 0) return 0;
    if (!d_low || !d_labels || !d_confmat) return fail(LC2IS_ERR_ARG, "null pointer%s");
    if (int e = check_labels_ratio(H, W, lh, lw)) return e;
    cudaStream_t st = (cudaStream_t)stream;
    const int use_hist = C <= K3_SMEM_HIST_MAX_C;
    const size_t smem = use_hist ? ((size_t)C * C + 1) / 2 * sizeof(int) : 0;
    int s = 0;
    if (mode == LC2IS_BILINEAR && fast_scale(h, w, H, W, &s) && (s == 8 || s == 16)) {
        int e = launch_k3_strip(d_low, N, C, h, w, H, W, s, d_labels, false, lh, lw, d_confmat, d_per_image, d_pred, st);
        if (e != LC2IS_ERR_UNSUPPORTED) return e;
    }
    if (fast_scale(h, w, H, W, &s) && s <= 16) {
        BlockGeom g = make_geom(H, W, s);
        K3LowParams P;
        P.low = d_low; P.labels = (const long long*)d_labels; P.confmat = (unsigned long long*)d_confmat;
        P.per_image = (unsigned long long*)d_per_image; P.pred_out = (long long*)d_pred;
        P.C = C; P.h = h; P.w = w; P.H = H; P.W = W; P.lh = lh; P.lw = lw;
        P.s = s; P.off = g.off; P.rs = g.rs;
        const int bps = s / 4;
        P.q = (g.off + s / 2) / 4;
        P.tgy = 8 / bps; P.tgx = 16 / bps;
        const int nt = mode == LC2IS_BILINEAR ? 2 : 4;
        const size_t tile = (size_t)C * (P.tgy + nt - 1) * (P.tgx + nt - 1) * sizeof(float);
        if (tile <= 200 * 1024) {
            dim3 grid((w + 1 + P.tgx - 1) / P.tgx, (h + 1 + P.tgy - 1) / P.tgy, N);
            auto launch = [&](auto kernel) -> int {
                if (int e = set_smem(kernel, tile)) return e;
                kernel<<<grid, 128, tile, st>>>(P);
                return 0;
            };
            int e;
            if (mode == LC2IS_BILINEAR)
                e = s == 4 ? launch(k3_low_fast_kernel<0, 1>) : s == 8 ? launch(k3_low_fast_kernel<0, 2>)
                                                                       : launch(k3_low_fast_kernel<0, 4>);
            else
                e = s == 4 ? launch(k3_low_fast_kernel<1, 1>) : s == 8 ? launch(k3_low_fast_kernel<1, 2>)
                                                                       : launch(k3_low_fast_kernel<1, 4>);
            if (e) return e;
            LC2IS_CHECK_LAUNCH("k3_low_fast_kernel");
            return 0;
        }
    }
    // generic: ATen scale for size= mode is (float)in / out
    const float sy = (float)h / (float)H, sx = (float)w / (float)W;
    long long HW = (long long)H * W;
    long long gx = (HW + K3_THREADS - 1) / K3_THREADS;
    long long cap = (long long)sm_count() * 2;
    if (N > 0 && gx > (cap + N - 1) / N) gx = (cap + N - 1) / N;
    if (gx < 1) gx = 1;
    dim3 grid((unsigned)gx, N);
    if (mode == LC2IS_BILINEAR) {
        if (int e = set_smem(k3_low_gen_kernel<0>, smem)) return e;
        k3_low_gen_kernel<0><<<grid, K3_THREADS, smem, st>>>(
            d_low, C, h, w, H, W, sy, sx, (const long long*)d_labels, lh, lw,
            (unsigned long long*)d_confmat, (unsigned long long*)d_per_image, (long long*)d_pred, use_hist);
    } else {
        if (int e = set_smem(k3_low_gen_kernel<1>, smem)) return e;
        k3_low_gen_kernel<1><<<grid, K3_THREADS, smem, st>>>(
            d_low, C, h, w, H, W, sy, sx, (const long long*)d_labels, lh, lw,
            (unsigned long long*)d_confmat, (unsigned long long*)d_per_image, (long long*)d_pred, use_hist);
    }
    LC2IS_CHECK_LAUNCH("k3_low_gen_kernel");
    return 0;
}
