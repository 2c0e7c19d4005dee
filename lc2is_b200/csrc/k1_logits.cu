// K0 proto_normalize, K1a patch-row normalise, K1 cosine-logits GEMM (tcgen05 + TMEM + TMA).
//
// Replaces reference model/final.py:41-43:
//     v = F.normalize(v, dim=1, p=2); t = F.normalize(t, dim=2, p=2)
//     score_map = torch.einsum('bchw,bkc->bkhw', v, t)
// (and the un-normalised matmul of model/model.py:50,53).
//
// GEMM view: logits[b, c, p] = scale * sum_d Vhat[b*hw + p, d] * That[c, d]
//   A = Vhat  [B*hw, D]   bf16, K-major, 128-row tiles          (TMA, 128B swizzle)
//   B = That  [C_pad, D]  bf16, K-major, NB <= 256 row tiles    (TMA, 128B swizzle)
//   D = 128 x NB fp32 accumulator in TMEM, two buffers (2 x 256 columns) so the epilogue of
//       tile i overlaps the loads + MMAs of tile i+1.
// Persistent CTAs (one per SM), 6 warps: warp 0 = TMA producer, warp 1 = MMA issuer (one
// elected thread) + TMEM owner, warps 2..5 = epilogue.  The epilogue writes class-plane major
// [B, C, hw]: TMEM lane = pixel, so for a fixed class the 32 lanes of a warp store 128
// contiguous bytes.
#include "common.cuh"
#include "tc_common.cuh"

namespace lc2is {

// ---------------------------------------------------------------------------------------------
// One warp per row: out = bf16(x / max(||x||, 1e-12)) (or bf16(x)), inv_norm = 1/max(||x||,eps).
// rows_out >= rows_in: extra rows (class padding) are zero-filled.  pad_group: rows_in rows are
// grouped as [n_sets][rows_per_set] and written to [n_sets][rows_per_set_pad].
template <typename T>
__global__ void __launch_bounds__(256)
rownorm_kernel(const T* __restrict__ x, long long n_sets, int rows_per_set, int rows_per_set_pad, int D,
               int normalize, __nv_bfloat16* __restrict__ out, float* __restrict__ inv_norm) {
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const long long total = n_sets * rows_per_set_pad;
    for (long long r = warp; r < total; r += nwarps) {
        const long long set = r / rows_per_set_pad;
        const int row = (int)(r - set * rows_per_set_pad);
        __nv_bfloat16* o = out + (size_t)r * D;
        if (row >= rows_per_set) {
            for (int d = lane * 8; d < D; d += 256) *reinterpret_cast<uint4*>(o + d) = make_uint4(0, 0, 0, 0);
            continue;
        }
        const T* xi = x + ((size_t)set * rows_per_set + row) * D;
        auto load8 = [&](int d, float (&v)[8]) {
            if constexpr (sizeof(T) == 4) {
                float4 a = __ldg(reinterpret_cast<const float4*>(xi + d));
                float4 b = __ldg(reinterpret_cast<const float4*>(xi + d) + 1);
                v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
            } else {
                uint4 a = __ldg(reinterpret_cast<const uint4*>(xi + d));
                unsigned w[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    v[2 * i] = __uint_as_float(w[i] << 16);
                    v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
                }
            }
        };
        // x * (1 / denom) with a correctly rounded reciprocal: against F.normalize's x / denom the fp32 product can be
        // one ulp off, which survives the rounding to bf16 for about one element in 2^15 (by one bf16 ulp) - and a
        // true division per element is ten instructions where this is one (the kernel is issue-bound: 64 KB rows/us)
        auto store8 = [&](int d, const float (&v)[8], float rden) {
            __nv_bfloat162 p[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) p[i] = __floats2bfloat162_rn(v[2 * i] * rden, v[2 * i + 1] * rden);
            *reinterpret_cast<uint4*>(o + d) = *reinterpret_cast<uint4*>(p);
        };
        float ss = 0.f;
        // 8 elements per lane per step (D % 8 == 0); rows of up to 1024 elements stay in registers between the
        // norm and the scaling (one pass over memory)
        if (D <= 1024) {
            float v[4][8];
#pragma unroll
            for (int it = 0; it < 4; ++it) {
                const int d = lane * 8 + it * 256;
                if (d < D) {
                    load8(d, v[it]);
#pragma unroll
                    for (int i = 0; i < 8; ++i) ss = fmaf(v[it][i], v[it][i], ss);
                }
            }
            ss = warp_sum(ss);
            const float denom = normalize ? fmaxf(sqrtf(ss), 1e-12f) : 1.f;
            const float rden = __frcp_rn(denom);
            if (lane == 0 && inv_norm) inv_norm[(size_t)set * rows_per_set + row] = rden;
#pragma unroll
            for (int it = 0; it < 4; ++it) {
                const int d = lane * 8 + it * 256;
                if (d < D) store8(d, v[it], rden);
            }
            continue;
        }
        for (int d = lane * 8; d < D; d += 256) {
            float v[8];
            load8(d, v);
#pragma unroll
            for (int i = 0; i < 8; ++i) ss = fmaf(v[i], v[i], ss);
        }
        ss = warp_sum(ss);
        const float denom = normalize ? fmaxf(sqrtf(ss), 1e-12f) : 1.f;
        const float rden = __frcp_rn(denom);
        if (lane == 0 && inv_norm) inv_norm[(size_t)set * rows_per_set + row] = rden;
        for (int d = lane * 8; d < D; d += 256) {
            float v[8];
            load8(d, v);
            store8(d, v, rden);
        }
    }
}

// ---------------------------------------------------------------------------------------------
constexpr int K1_THREADS = 192;
constexpr int K1_BM = 128;
constexpr int K1_BK = 64;                 // 64 bf16 = 128 B = one swizzle row
constexpr int K1_A_BYTES = K1_BM * K1_BK * 2;
constexpr int K1_MAX_STAGES = 8;

struct K1Params {
    float* out;            // EPI 0: [B, C, hw] fp32 (class-plane major)
    void* out_rm;          // EPI 1: [M, C] row major, bf16 or fp32
    const float* bias;     // EPI 1: [C] or null
    int out_f32;           // EPI 1
    int B, hw, C, C_pad, n_sets;
    int NB, n_ntiles, tiles_per_img, num_kb, stages;
    float scale;
    // EPI 0 with fuse_norm: A is the RAW bf16 V; warps 6-9 sum the squares of each row from the staged A tiles while
    // the MMAs run and the epilogue scales the row by 1 / max(||v||, 1e-12) (F.normalize) - no v_hat round trip
    int fuse_norm;
    float* inv_v;          // [B*hw] out (fuse_norm): the row factors, for the backward
};

// Row-major epilogue staging.  In TMEM a thread owns a ROW, so storing straight from registers makes every warp store
// touch 32 rows (32 half-written sectors: the projection GEMM spent 8.9 us per tile in its epilogue against 3.3 us of
// MMA).  Instead each warp passes 128 bytes per row (64 bf16 / 32 fp32 channels) through a swizzled 4 KB scratch and
// writes them back as 8 stores of 4 rows x 128 contiguous bytes; two warps per TMEM lane quarter share the columns.
constexpr int K1_EPI_WARPS_RM = 8;                 // row-major epilogue: two warps per TMEM lane quarter
constexpr int K1_EPI_SCRATCH = K1_EPI_WARPS_RM * 4096;
// one warp: rows [m0, m0 + 32) x columns [n0, n0 + ncols) of the row-major output from TMEM address `taddr`
__device__ __forceinline__ void epi_rowmajor(const K1Params& P, uint8_t* scr, int lane, uint32_t taddr, size_t m0,
                                             int rows_valid, int n0, int ncols);

__device__ __forceinline__ void epi_rowmajor(const K1Params& P, uint8_t* scr, int lane, uint32_t taddr, size_t m0,
                                             int rows_valid, int n0, int ncols) {
    const int esize = P.out_f32 ? 4 : 2;
    const int G = 128 / esize;                                  // channels per 128-byte group
    uint8_t* out = reinterpret_cast<uint8_t*>(P.out_rm);
    for (int cg = 0; cg < ncols; cg += G) {
        for (int sub = 0; sub < G && cg + sub < ncols; sub += 32) {
            uint32_t r[32];
            if (cg + sub + 32 <= ncols) {
                tc::tmem_ld32(taddr + cg + sub, r);
            } else {                                            // ragged tail: 16 columns
                uint32_t r16[16];
                tc::tmem_ld16(taddr + cg + sub, r16);
#pragma unroll
                for (int j = 0; j < 16; ++j) { r[j] = r16[j]; r[16 + j] = 0u; }
            }
            tc::tmem_ld_wait();
#pragma unroll
            for (int hq = 0; hq < 2; ++hq) {
                if (cg + sub + 16 * hq >= ncols) break;
                float o[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) o[j] = __uint_as_float(r[16 * hq + j]) * P.scale;
                if (P.bias) {
                    const float4* bp = reinterpret_cast<const float4*>(P.bias + n0 + cg + sub + 16 * hq);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float4 bv = __ldg(bp + j);
                        o[4 * j] += bv.x; o[4 * j + 1] += bv.y; o[4 * j + 2] += bv.z; o[4 * j + 3] += bv.w;
                    }
                }
                const int c16 = sub + 16 * hq;                  // channel offset inside the group
                if (P.out_f32) {
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        epi_put(scr, lane, (c16 >> 2) + j,
                                make_uint4(__float_as_uint(o[4 * j]), __float_as_uint(o[4 * j + 1]),
                                           __float_as_uint(o[4 * j + 2]), __float_as_uint(o[4 * j + 3])));
                } else {
                    __nv_bfloat162 pk[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) pk[j] = __floats2bfloat162_rn(o[2 * j], o[2 * j + 1]);
                    epi_put(scr, lane, (c16 >> 3), *reinterpret_cast<uint4*>(&pk[0]));
                    epi_put(scr, lane, (c16 >> 3) + 1, *reinterpret_cast<uint4*>(&pk[4]));
                }
            }
        }
        __syncwarp();
        const int cols_here = ncols - cg < G ? ncols - cg : G;
        epi_flush(scr, lane, out + (m0 * (size_t)P.C + n0 + cg) * esize, (size_t)P.C * esize, rows_valid,
                  cols_here * esize / 16);
        __syncwarp();
    }
}
// how the epilogue warps of one TMEM lane quarter split the tile's columns (whole 128-byte groups each)
__device__ __forceinline__ void epi_split(int ncols, int esize, int part, int nparts, int* c0, int* c1) {
    const int G = 128 / esize, groups = (ncols + G - 1) / G;
    const int g0 = groups * part / nparts, g1 = groups * (part + 1) / nparts;
    *c0 = g0 * G;
    *c1 = g1 * G < ncols ? g1 * G : ncols;
}

// EPI 0: the cosine-logits epilogue (class-plane major fp32).  EPI 1: the linear-projection epilogue of
// TextToPatch.visual (model/text_patch.py:12,17): row-major out[m, n] = acc + bias[n], bf16 or fp32.
template <int EPI>
__global__ void __launch_bounds__(64 + 32 * K1_EPI_WARPS_RM, 1)
k1_logits_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const K1Params P) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base_u32 = (tc::smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem = smem_raw + (base_u32 - tc::smem_u32(smem_raw));
    const int stage_bytes = K1_A_BYTES + P.NB * 128;
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)P.stages * stage_bytes);
    uint64_t* empty = full + K1_MAX_STAGES;
    uint64_t* tfull = empty + K1_MAX_STAGES;
    uint64_t* tempty = tfull + 2;
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tempty + 2);
    uint64_t* nfull = tempty + 3;                                // fuse_norm: row factors of accumulator buffer i ready
    uint8_t* epi_scr = reinterpret_cast<uint8_t*>(full) + 256;   // EPI 1 only: 4 warps x 4 KB (16-byte aligned)
    float* inv_s = reinterpret_cast<float*>(epi_scr);            // EPI 0 + fuse_norm: [2][128] row factors
    const bool fuse_norm = EPI == 0 && P.fuse_norm;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int total_tiles = P.B * P.tiles_per_img * P.n_ntiles;

    if (warp == 0 && lane == 0) {
        tc::prefetch_tmap(&tmA);
        tc::prefetch_tmap(&tmB);
        // a stage is free when its MMAs have retired AND (fuse_norm) the four norm warps have read it
        for (int i = 0; i < P.stages; ++i) { tc::mbar_init(full + i, 1); tc::mbar_init(empty + i, fuse_norm ? 5 : 1); }
        for (int i = 0; i < 2; ++i) {
            tc::mbar_init(tfull + i, 1); tc::mbar_init(tempty + i, EPI == 0 ? 4 : K1_EPI_WARPS_RM);
            tc::mbar_init(nfull + i, 4);
        }
        tc::fence_barrier_init();
    }
    if (warp == 1) tc::tmem_alloc(tmem_ptr, 512);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    if (EPI == 0 && warp >= 6) {
        // ===== norm warps (fuse_norm): lane = one row of the 128-row A tile =====
        if (fuse_norm) {
            const int row = (warp - 6) * 32 + lane;
            int stage = 0; uint32_t phase = 0;
            int it = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
                const int buf = it & 1;
                const uint32_t bphase = (it >> 1) & 1;
                const int mt = tile / P.n_ntiles;
                const int b = mt / P.tiles_per_img, ti = mt - b * P.tiles_per_img;
                tc::mbar_wait(tempty + buf, bphase ^ 1);       // the epilogue of tile it-2 has read inv_s[buf]
                float ss = 0.f, ss1 = 0.f;                     // two chains: the 64 dependent fma per k-block were the norm warps' pace
                for (int kb = 0; kb < P.num_kb; ++kb) {
                    tc::mbar_wait(full + stage, phase);
                    const uint8_t* ar = smem + (size_t)stage * stage_bytes + row * 128;
                    // the row's eight 16-byte chunks in any order (a sum); lane-rotated so that the eight rows of a
                    // swizzle atom read eight different chunk positions (no bank conflict)
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const uint4 v = *reinterpret_cast<const uint4*>(ar + (((i + lane) & 7) << 4));
                        const unsigned w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            const float lo = __uint_as_float(w[k] << 16), hi = __uint_as_float(w[k] & 0xffff0000u);
                            ss = fmaf(lo, lo, ss); ss1 = fmaf(hi, hi, ss1);
                        }
                    }
                    __syncwarp();
                    if (lane == 0) tc::mbar_arrive(empty + stage);
                    if (++stage == P.stages) { stage = 0; phase ^= 1; }
                }
                const float inv = __frcp_rn(fmaxf(sqrtf(ss + ss1), 1e-12f));
                inv_s[buf * 128 + row] = inv;
                const int p = ti * K1_BM + row;
                if (p < P.hw && P.inv_v) P.inv_v[(size_t)b * P.hw + p] = inv;
                __syncwarp();
                if (lane == 0) tc::mbar_arrive(nfull + buf);
            }
        }
    } else if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                const int nt = tile % P.n_ntiles, mt = tile / P.n_ntiles;
                const int b = mt / P.tiles_per_img, ti = mt - b * P.tiles_per_img;
                const int arow = b * P.hw + ti * K1_BM;
                const int brow = (P.n_sets > 1 ? b : 0) * P.C_pad + nt * P.NB;
                for (int kb = 0; kb < P.num_kb; ++kb) {
                    tc::mbar_wait(empty + stage, phase ^ 1);
                    uint8_t* sa = smem + (size_t)stage * stage_bytes;
                    tc::mbar_arrive_expect_tx(full + stage, (uint32_t)stage_bytes);
                    tc::tma_load_2d(sa, &tmA, full + stage, kb * K1_BK, arow);
                    tc::tma_load_2d(sa + K1_A_BYTES, &tmB, full + stage, kb * K1_BK, brow);
                    if (++stage == P.stages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (lane == 0) {
            const uint32_t idesc = tc::make_idesc_bf16(K1_BM, P.NB, 0, 0);
            int stage = 0; uint32_t phase = 0;
            int it = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
                const int buf = it & 1;
                const uint32_t bphase = (it >> 1) & 1;
                tc::mbar_wait(tempty + buf, bphase ^ 1);       // epilogue drained this buffer
                tc::tc_fence_after();
                const uint32_t d_tmem = tmem_base + buf * 256;
                for (int kb = 0; kb < P.num_kb; ++kb) {
                    tc::mbar_wait(full + stage, phase);
                    tc::tc_fence_after();
                    const uint32_t sa = base_u32 + stage * stage_bytes;
                    const uint64_t adesc = tc::make_smem_desc(sa, 16, 1024);
                    const uint64_t bdesc = tc::make_smem_desc(sa + K1_A_BYTES, 16, 1024);
#pragma unroll
                    for (int k = 0; k < K1_BK / 16; ++k)
                        tc::umma_bf16(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0);
                    tc::umma_commit(empty + stage);             // frees the smem slot when the MMAs retire
                    if (++stage == P.stages) { stage = 0; phase ^= 1; }
                }
                tc::umma_commit(tfull + buf);                   // accumulator ready
            }
        }
    } else if (EPI != 0 || warp < 6) {
        // ===== epilogue: TMEM -> registers -> global (class-plane major) =====
        const int q = warp & 3;                                 // TMEM lane quarter this warp may read
        int it = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
            const int buf = it & 1;
            const uint32_t bphase = (it >> 1) & 1;
            const int nt = tile % P.n_ntiles, mt = tile / P.n_ntiles;
            const int b = mt / P.tiles_per_img, ti = mt - b * P.tiles_per_img;
            const int p = ti * K1_BM + q * 32 + lane;
            const bool rvalid = p < P.hw;
            float* orow = P.out + (size_t)b * P.C * P.hw + p;
            tc::mbar_wait(tfull + buf, bphase);
            tc::tc_fence_after();
            const uint32_t taddr = tmem_base + buf * 256 + ((uint32_t)(q * 32) << 16);
            const int n0 = nt * P.NB;
            if constexpr (EPI == 0) {
                float sc = P.scale;
                if (fuse_norm) {
                    tc::mbar_wait(nfull + buf, bphase);
                    sc *= inv_s[buf * 128 + q * 32 + lane];
                }
                // A thread owns a pixel ROW in TMEM and the class planes are hw floats apart: a warp store writes 128
                // contiguous bytes of one class plane.  Per class: one FMUL, one IMAD.WIDE (plane offset = constant x hw)
                // and the store - the first version (class index, bound check and a 64-bit address product per store,
                // one tcgen05.wait per 16 columns) spent 20 instructions per class and made this epilogue, not HBM, the
                // bound of the kernel at 128 x 128 patches (profiles/r02_gb_k1_ncu.md).
                const int ncols = P.C - n0 < P.NB ? P.C - n0 : P.NB;       // classes of this N tile (warp-uniform)
                const unsigned hwu = (unsigned)P.hw;
                float* pc = orow + (size_t)n0 * P.hw;
                int col = 0;
                for (; col + 32 <= ncols; col += 32) {
                    uint32_t r[32];
                    tc::tmem_ld32(taddr + col, r);
                    tc::tmem_ld_wait();
                    if (rvalid) {
#pragma unroll
                        for (int j = 0; j < 32; ++j)
                            __stcs(pc + (unsigned long long)hwu * (unsigned)j, __uint_as_float(r[j]) * sc);
                    }
                    pc += 32ull * hwu;
                }
                for (; col < ncols; col += 16) {
                    uint32_t r[16];
                    tc::tmem_ld16(taddr + col, r);
                    tc::tmem_ld_wait();
                    const int nv = ncols - col;                             // 1..16 or more (warp-uniform)
                    if (rvalid) {
                        if (nv >= 16) {
#pragma unroll
                            for (int j = 0; j < 16; ++j)
                                __stcs(pc + (unsigned long long)hwu * (unsigned)j, __uint_as_float(r[j]) * sc);
                        } else {
#pragma unroll
                            for (int j = 0; j < 16; ++j)
                                if (j < nv) __stcs(pc + (unsigned long long)hwu * (unsigned)j, __uint_as_float(r[j]) * sc);
                        }
                    }
                    pc += 16ull * hwu;
                }
            } else {
                // row-major (C % 16 == 0 for this epilogue): this warp's 32 rows, staged for coalesced stores
                const int pw = ti * K1_BM + q * 32;             // first row of the warp inside the image
                const int ncols = P.C - n0 < P.NB ? P.C - n0 : P.NB;
                int c0 = 0, c1 = 0;
                epi_split(ncols > 0 ? ncols : 0, P.out_f32 ? 4 : 2, (warp - 2) >> 2, K1_EPI_WARPS_RM / 4, &c0, &c1);
                if (pw < P.hw && c1 > c0)
                    epi_rowmajor(P, epi_scr + (warp - 2) * 4096, lane, taddr + c0, (size_t)b * P.hw + pw,
                                 P.hw - pw < 32 ? P.hw - pw : 32, n0 + c0, c1 - c0);
            }
            tc::tc_fence_before();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(tempty + buf);
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc::tc_fence_after();
        tc::tmem_dealloc(tmem_base, 512);
    }
}

// ---------------------------------------------------------------------------------------------
// 2-SM form of the projection GEMM (cta_group::2): a CTA pair owns a 256 x 256 output tile.  Each CTA stages its own
// 128 rows of x and HALF of the W tile (128 of the 256 output channels) - 32 KB per k-block instead of 48 KB, so six
// stages fit where the 1-SM kernel has four and the pipeline tolerates ~1.4 us of load latency instead of ~0.8 us (the
// 1-SM kernel is latency-bound at 43 % tensor-pipe activity, profiles/r01_linear_gemm.md).  Only the leader CTA
// (cluster rank 0) issues tcgen05.mma; both CTAs' TMA loads complete on the LEADER's full barrier; tcgen05.commit
// multicasts the "slot free" / "accumulator ready" arrivals to both CTAs; each CTA's epilogue drains its own 128 TMEM
// lanes and the peer's epilogue warps arrive remotely on the leader's "accumulator drained" barrier.
constexpr int K2SM_NB = 256;                                   // output channels per tile (128 staged per CTA)
constexpr int K2SM_STAGE = K1_A_BYTES + (K2SM_NB / 2) * 128;   // 32 KB
constexpr int K2SM_STAGES = 6;

namespace tc2 {
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `p` (a shared::cta pointer) in the CTA of rank `rank`
__device__ __forceinline__ uint32_t mapa(const void* p, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(tc::smem_u32(p)), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    // default semantics (release at CTA scope): the arrival orders this thread's TMEM reads, which tcgen05.wait::ld +
    // tcgen05.fence::before_thread_sync have already completed; a cluster-scope release would also wait for the
    // epilogue's global stores (measured as membar stalls)
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tma_load_2d_2sm(void* smem_dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int x,
                                                int y) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(tc::smem_u32(smem_dst)), "l"(m), "r"(bar_cluster_addr), "r"(x), "r"(y)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t* smem_result, uint32_t ncols) {   // one full warp in EACH CTA
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc::smem_u32(smem_result)),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_bf16_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                              uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive on the barrier at this offset in BOTH CTAs when the MMAs issued so far have completed
__device__ __forceinline__ void umma_commit_2sm(uint64_t* bar) {
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
            tc::smem_u32(bar)),
        "h"((uint16_t)3)
        : "memory");
}
}  // namespace tc2

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(64 + 32 * K1_EPI_WARPS_RM, 1)
k1_linear_2sm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                     const K1Params P) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base_u32 = (tc::smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem = smem_raw + (base_u32 - tc::smem_u32(smem_raw));
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)K2SM_STAGES * K2SM_STAGE);
    uint64_t* empty = full + K1_MAX_STAGES;
    uint64_t* tfull = empty + K1_MAX_STAGES;
    uint64_t* tempty = tfull + 2;
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tempty + 2);
    uint8_t* epi_scr = reinterpret_cast<uint8_t*>(full) + 256;   // 4 warps x 4 KB

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = tc2::cluster_ctarank();
    const int n_clusters = gridDim.x >> 1, cluster_id = blockIdx.x >> 1;
    // pair tiles: 256 rows x 256 channels; the N tile runs fastest so that the two channel halves of the same rows
    // are in flight together (x is read from HBM once)
    const int n_ntiles = P.C / K2SM_NB;
    const int total_tiles = (P.hw / (2 * K1_BM)) * n_ntiles;

    if (warp == 0 && lane == 0) {
        tc::prefetch_tmap(&tmA);
        tc::prefetch_tmap(&tmB);
        for (int i = 0; i < K2SM_STAGES; ++i) { tc::mbar_init(full + i, 1); tc::mbar_init(empty + i, 1); }
        for (int i = 0; i < 2; ++i) { tc::mbar_init(tfull + i, 1); tc::mbar_init(tempty + i, 2 * K1_EPI_WARPS_RM); }   // both CTAs' warps
        tc::fence_barrier_init();
    }
    tc2::cluster_sync();                                        // the peer's barriers exist before anything remote
    if (warp == 1) tc2::tmem_alloc2(tmem_ptr, 512);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    if (warp == 0) {
        // ===== TMA producer (both CTAs): own 128 rows of x, own half of the W tile; bytes land on the leader's barrier
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int tile = cluster_id; tile < total_tiles; tile += n_clusters) {
                const int nt = tile % n_ntiles, mt = tile / n_ntiles;
                const int arow = mt * 2 * K1_BM + (int)rank * K1_BM;
                const int brow = nt * K2SM_NB + (int)rank * (K2SM_NB / 2);
                for (int kb = 0; kb < P.num_kb; ++kb) {
                    tc::mbar_wait(empty + stage, phase ^ 1);
                    uint8_t* sa = smem + (size_t)stage * K2SM_STAGE;
                    if (rank == 0) tc::mbar_arrive_expect_tx(full + stage, 2u * K2SM_STAGE);
                    const uint32_t bar = tc2::mapa(full + stage, 0);
                    tc2::tma_load_2d_2sm(sa, &tmA, bar, kb * K1_BK, arow);
                    tc2::tma_load_2d_2sm(sa + K1_A_BYTES, &tmB, bar, kb * K1_BK, brow);
                    if (++stage == K2SM_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: the leader CTA only =====
        if (lane == 0 && rank == 0) {
            const uint32_t idesc = tc::make_idesc_bf16(2 * K1_BM, K2SM_NB, 0, 0);
            int stage = 0; uint32_t phase = 0;
            int it = 0;
            for (int tile = cluster_id; tile < total_tiles; tile += n_clusters, ++it) {
                const int buf = it & 1;
                const uint32_t bphase = (it >> 1) & 1;
                tc::mbar_wait(tempty + buf, bphase ^ 1);       // both CTAs' epilogues drained this buffer
                tc::tc_fence_after();
                const uint32_t d_tmem = tmem_base + buf * 256;
                for (int kb = 0; kb < P.num_kb; ++kb) {
                    tc::mbar_wait(full + stage, phase);
                    tc::tc_fence_after();
                    const uint32_t sa = base_u32 + stage * K2SM_STAGE;
                    const uint64_t adesc = tc::make_smem_desc(sa, 16, 1024);
                    const uint64_t bdesc = tc::make_smem_desc(sa + K1_A_BYTES, 16, 1024);
#pragma unroll
                    for (int k = 0; k < K1_BK / 16; ++k)
                        tc2::umma_bf16_2sm(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0);
                    tc2::umma_commit_2sm(empty + stage);        // frees the slot in both CTAs
                    if (++stage == K2SM_STAGES) { stage = 0; phase ^= 1; }
                }
                tc2::umma_commit_2sm(tfull + buf);              // accumulator ready in both CTAs
            }
        }
    } else {
        // ===== epilogue (both CTAs): own 128 TMEM lanes -> registers -> row-major global =====
        const int q = warp & 3;
        const uint32_t tempty_leader0 = tc2::mapa(tempty, 0), tempty_leader1 = tc2::mapa(tempty + 1, 0);
        int it = 0;
        for (int tile = cluster_id; tile < total_tiles; tile += n_clusters, ++it) {
            const int buf = it & 1;
            const uint32_t bphase = (it >> 1) & 1;
            const int nt = tile % n_ntiles, mt = tile / n_ntiles;
            const size_t m0w = (size_t)mt * 2 * K1_BM + rank * K1_BM + q * 32;       // first row of this warp
            tc::mbar_wait(tfull + buf, bphase);
            tc::tc_fence_after();
            const uint32_t taddr = tmem_base + buf * 256 + ((uint32_t)(q * 32) << 16);
            const int n0 = nt * K2SM_NB;
            int c0 = 0, c1 = 0;
            epi_split(K2SM_NB, P.out_f32 ? 4 : 2, (warp - 2) >> 2, K1_EPI_WARPS_RM / 4, &c0, &c1);
            epi_rowmajor(P, epi_scr + (warp - 2) * 4096, lane, taddr + c0, m0w, 32, n0 + c0, c1 - c0);
            tc::tc_fence_before();
            __syncwarp();
            if (lane == 0) tc2::mbar_arrive_cluster(buf ? tempty_leader1 : tempty_leader0);
        }
    }
    tc::tc_fence_before();
    tc2::cluster_sync();                                        // nobody leaves while the peer may still touch it
    if (warp == 1) {
        tc::tc_fence_after();
        tc2::tmem_dealloc2(tmem_base, 512);
    }
}

// ---------------------------------------------------------------------------------------------
PFN_encodeTiled get_encode_tiled() {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (PFN_encodeTiled)p;
    }
    return fn;
}

int make_tmap_2d_bf16(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows,
                      uint32_t box_cols) {
    PFN_encodeTiled enc = get_encode_tiled();
    if (!enc) return fail(LC2IS_ERR_NODEVICE, "cuTensorMapEncodeTiled entry point unavailable%s");
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {cols * 2};
    cuuint32_t box[2] = {box_cols, box_rows};
    cuuint32_t es[2] = {1, 1};
    CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(LC2IS_ERR_ARG, "cuTensorMapEncodeTiled(2d) failed: %s%lld", "CUresult ", (long long)r);
    return 0;
}

int make_tmap_3d_bf16(CUtensorMap* out, const void* base, uint64_t d2, uint64_t d1, uint64_t d0, uint32_t box1,
                      uint32_t box0) {
    PFN_encodeTiled enc = get_encode_tiled();
    if (!enc) return fail(LC2IS_ERR_NODEVICE, "cuTensorMapEncodeTiled entry point unavailable%s");
    cuuint64_t dims[3] = {d0, d1, d2};
    cuuint64_t strides[2] = {d0 * 2, d0 * d1 * 2};
    cuuint32_t box[3] = {box0, box1, 1};
    cuuint32_t es[3] = {1, 1, 1};
    CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(LC2IS_ERR_ARG, "cuTensorMapEncodeTiled(3d) failed: %s%lld", "CUresult ", (long long)r);
    return 0;
}

template <typename T>
static int launch_rownorm(const T* x, long long n_sets, int rows, int rows_pad, int D, int normalize,
                          __nv_bfloat16* out, float* inv, cudaStream_t st) {
    long long total = n_sets * rows_pad;
    long long blocks = (total + 7) / 8;
    long long cap = (long long)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    rownorm_kernel<T><<<(unsigned)blocks, 256, 0, st>>>(x, n_sets, rows, rows_pad, D, normalize, out, inv);
    return 0;
}

}  // namespace lc2is

using namespace lc2is;

extern "C" int lc2is_class_pad(int C) { return class_pad(C); }

extern "C" int lc2is_proto_normalize(const float* d_t, int n_sets, int C, int D, int normalize,
                                     void* d_t_hat, float* d_inv_norm, lc2is_stream_t stream) {
    if (int e = ensure_device()) return e;
    if (!d_t || !d_t_hat) return fail(LC2IS_ERR_ARG, "null pointer%s");
    if (n_sets <= 0 || C <= 0 || D <= 0 || D % 8) return fail(LC2IS_ERR_SHAPE, "need n_sets,C > 0 and D %% 8 == 0%s");
    launch_rownorm<float>(d_t, n_sets, C, class_pad(C), D, normalize, (__nv_bfloat16*)d_t_hat, d_inv_norm,
                          (cudaStream_t)stream);
    LC2IS_CHECK_LAUNCH("rownorm_kernel(t)");
    return 0;
}

extern "C" int lc2is_cosine_logits_fwd(const void* d_v, int v_dtype, int B, int hw, int D,
                                       const void* d_t_hat, int n_sets, int C,
                                       int normalize, float logit_scale,
                                       void* d_v_hat, float* d_inv_norm_v, float* d_logits,
                                       lc2is_stream_t stream) {
    if (int e = ensure_device()) return e;
    if (!d_v || !d_t_hat || !d_logits) return fail(LC2IS_ERR_ARG, "null pointer%s");
    // d_v_hat == NULL: the normalisation runs inside the GEMM on the raw bf16 V (no v_hat is written; the backward then
    // takes V itself with LC2IS_BWD_RAW_V)
    const bool fuse = d_v_hat == nullptr;
    if (fuse && (v_dtype != LC2IS_BF16 || !normalize || !d_inv_norm_v))
        return fail(LC2IS_ERR_ARG, "d_v_hat may only be NULL for bf16 V with normalize = 1 and d_inv_norm_v given%s");
    if (B < 0 || hw <= 0 || C <= 0 || D <= 0) return fail(LC2IS_ERR_SHAPE, "bad shape%s");
    if (D % K1_BK) return fail(LC2IS_ERR_SHAPE, "D must be a multiple of 64 (got %s%lld)", "", D);
    if (n_sets != 1 && n_sets != B) return fail(LC2IS_ERR_SHAPE, "n_sets must be 1 or B%s");
    if (((uintptr_t)d_v_hat | (uintptr_t)d_t_hat | (uintptr_t)d_v) % 16) return fail(LC2IS_ERR_ARG, "pointers must be 16-byte aligned%s");
    if (B == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const long long M = (long long)B * hw;
    // ---- K1a: normalise rows, round to bf16 -------------------------------------------------------
    if (fuse) {
        // (inside the GEMM)
    } else if (v_dtype == LC2IS_F32)
        launch_rownorm<float>((const float*)d_v, 1, (int)M, (int)M, D, normalize, (__nv_bfloat16*)d_v_hat, d_inv_norm_v, st);
    else if (v_dtype == LC2IS_BF16)
        launch_rownorm<__nv_bfloat16>((const __nv_bfloat16*)d_v, 1, (int)M, (int)M, D, normalize, (__nv_bfloat16*)d_v_hat, d_inv_norm_v, st);
    else
        return fail(LC2IS_ERR_ARG, "v_dtype must be LC2IS_F32 or LC2IS_BF16%s");
    if (!fuse) LC2IS_CHECK_LAUNCH("rownorm_kernel(v)");

    // ---- K1: GEMM ------------------------------------------------------------------------------------
    K1Params P;
    P.out = d_logits; P.out_rm = nullptr; P.bias = nullptr; P.out_f32 = 0;
    P.B = B; P.hw = hw; P.C = C; P.C_pad = class_pad(C); P.n_sets = n_sets;
    const int n_ntiles0 = (P.C_pad + 255) / 256;
    P.NB = ((P.C_pad + n_ntiles0 - 1) / n_ntiles0 + 15) / 16 * 16;
    P.n_ntiles = (P.C_pad + P.NB - 1) / P.NB;
    P.tiles_per_img = (hw + K1_BM - 1) / K1_BM;
    P.num_kb = D / K1_BK;
    P.scale = logit_scale;
    P.fuse_norm = fuse ? 1 : 0;
    P.inv_v = fuse ? d_inv_norm_v : nullptr;
    const int stage_bytes = K1_A_BYTES + P.NB * 128;
    int stages = (200 * 1024) / stage_bytes;
    if (stages > K1_MAX_STAGES) stages = K1_MAX_STAGES;
    if (stages > P.num_kb * 2) stages = P.num_kb * 2;
    if (stages < 2) stages = 2;
    P.stages = stages;
    size_t smem = (size_t)stages * stage_bytes + 1024 /*align*/ + 256 /*barriers*/ + 1024 /*row factors*/;
    if (smem < 120 * 1024) smem = 120 * 1024;      // one CTA per SM: it owns all 512 TMEM columns
    CUtensorMap tmA, tmB;
    if (int e = make_tmap_2d_bf16(&tmA, fuse ? d_v : d_v_hat, (uint64_t)M, (uint64_t)D, K1_BM, K1_BK)) return e;
    if (int e = make_tmap_2d_bf16(&tmB, d_t_hat, (uint64_t)n_sets * P.C_pad, (uint64_t)D, P.NB, K1_BK)) return e;
    LC2IS_CUDA(cudaFuncSetAttribute(k1_logits_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int total_tiles = B * P.tiles_per_img * P.n_ntiles;
    int grid = sm_count();
    if (grid > total_tiles) grid = total_tiles;
    k1_logits_kernel<0><<<grid, fuse ? K1_THREADS + 128 : K1_THREADS, smem, st>>>(tmA, tmB, P);
    LC2IS_CHECK_LAUNCH("k1_logits_kernel");
    return 0;
}

// ---------------------------------------------------------------------------------------------
// TextToPatch.visual / .textual forward (model/text_patch.py:11-12,16-17): y = x W^T + b on the same tcgen05 / TMEM /
// TMA pipeline as the logits GEMM (A = x [M,K] bf16 K-major, B = W [N,K] bf16 K-major - nn.Linear's own layout).
extern "C" int lc2is_linear_fwd(const void* d_x_bf16, const void* d_w_bf16, const float* d_bias,
                                long long M, int N, int K, void* d_y, int y_dtype, lc2is_stream_t stream) {
    if (int e = ensure_device()) return e;
    if (!d_x_bf16 || !d_w_bf16 || !d_y) return fail(LC2IS_ERR_ARG, "null pointer%s");
    if (M < 0 || N <= 0 || K <= 0) return fail(LC2IS_ERR_SHAPE, "bad shape%s");
    if (K % K1_BK) return fail(LC2IS_ERR_SHAPE, "K must be a multiple of 64 (got %s%lld)", "", K);
    if (N % 16) return fail(LC2IS_ERR_SHAPE, "N must be a multiple of 16 (got %s%lld)", "", N);
    if (M > 0x7fffffffLL / 2) return fail(LC2IS_ERR_SHAPE, "M too large%s");
    if (y_dtype != LC2IS_F32 && y_dtype != LC2IS_BF16) return fail(LC2IS_ERR_ARG, "y_dtype%s");
    // x and W are TMA bases, y is written and the bias read with 16-byte vectors by the epilogue
    if (((uintptr_t)d_x_bf16 | (uintptr_t)d_w_bf16 | (uintptr_t)d_y | (uintptr_t)d_bias) % 16)
        return fail(LC2IS_ERR_ARG, "x, W, y and the bias must be 16-byte aligned%s");
    if (M == 0) return 0;
    K1Params P;
    P.out = nullptr; P.out_rm = d_y; P.bias = d_bias; P.out_f32 = y_dtype == LC2IS_F32;
    P.fuse_norm = 0; P.inv_v = nullptr;
    P.B = 1; P.hw = (int)M; P.C = N; P.C_pad = N; P.n_sets = 1;
    // 2-SM form (CTA pairs, 256 x 256 tiles) for shapes it tiles exactly and that fill the GPU more than once
    const bool fits_2sm = M % (2 * K1_BM) == 0 && N % K2SM_NB == 0;
    const long long pair_tiles = (M / (2 * K1_BM)) * (N / K2SM_NB);
    if (fits_2sm && pair_tiles >= 2LL * (sm_count() / 2)) {
        P.num_kb = K / K1_BK; P.scale = 1.f; P.NB = K2SM_NB; P.n_ntiles = N / K2SM_NB; P.tiles_per_img = 0; P.stages = K2SM_STAGES;
        const size_t smem2 = (size_t)K2SM_STAGES * K2SM_STAGE + 1024 + 256 + K1_EPI_SCRATCH;
        CUtensorMap tmA2, tmB2;
        if (int e = make_tmap_2d_bf16(&tmA2, d_x_bf16, (uint64_t)M, (uint64_t)K, K1_BM, K1_BK)) return e;
        if (int e = make_tmap_2d_bf16(&tmB2, d_w_bf16, (uint64_t)N, (uint64_t)K, K2SM_NB / 2, K1_BK)) return e;
        LC2IS_CUDA(cudaFuncSetAttribute(k1_linear_2sm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2));
        long long grid2 = 2 * (long long)(sm_count() / 2);
        if (grid2 > 2 * pair_tiles) grid2 = 2 * pair_tiles;
        k1_linear_2sm_kernel<<<(unsigned)grid2, 64 + 32 * K1_EPI_WARPS_RM, smem2, (cudaStream_t)stream>>>(tmA2, tmB2, P);
        LC2IS_CHECK_LAUNCH("k1_linear_2sm_kernel");
        return 0;
    }
    const int n_ntiles0 = (N + 255) / 256;
    P.NB = ((N + n_ntiles0 - 1) / n_ntiles0 + 15) / 16 * 16;
    P.n_ntiles = (N + P.NB - 1) / P.NB;
    P.tiles_per_img = (int)((M + K1_BM - 1) / K1_BM);
    P.num_kb = K / K1_BK;
    P.scale = 1.f;
    const int stage_bytes = K1_A_BYTES + P.NB * 128;
    int stages = (232448 - 1024 - 256 - K1_EPI_SCRATCH) / stage_bytes;   // 227 KB of dynamic shared memory
    if (stages > K1_MAX_STAGES) stages = K1_MAX_STAGES;
    if (stages > P.num_kb * 2) stages = P.num_kb * 2;
    if (stages < 2) stages = 2;
    P.stages = stages;
    size_t smem = (size_t)stages * stage_bytes + 1024 + 256 + K1_EPI_SCRATCH;
    if (smem < 120 * 1024) smem = 120 * 1024;
    CUtensorMap tmA, tmB;
    if (int e = make_tmap_2d_bf16(&tmA, d_x_bf16, (uint64_t)M, (uint64_t)K, K1_BM, K1_BK)) return e;
    if (int e = make_tmap_2d_bf16(&tmB, d_w_bf16, (uint64_t)N, (uint64_t)K, P.NB, K1_BK)) return e;
    LC2IS_CUDA(cudaFuncSetAttribute(k1_logits_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int total_tiles = P.tiles_per_img * P.n_ntiles;
    int grid = sm_count();
    if (grid > total_tiles) grid = total_tiles;
    k1_logits_kernel<1><<<grid, 64 + 32 * K1_EPI_WARPS_RM, smem, (cudaStream_t)stream>>>(tmA, tmB, P);
    LC2IS_CHECK_LAUNCH("k1_logits_kernel<linear>");
    return 0;
}
