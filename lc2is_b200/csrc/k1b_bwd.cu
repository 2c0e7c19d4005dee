// K1b: backward of the cosine-logits GEMM (autograd of model/final.py:41-43; engine.py:100).
//
// With  logits[m,c] = s * <vhat_m, that_c>,  G = dL/dlogits  and  g = upstream scalar:
//   dVhat = s*g * G  That         [M,C] x [C,D]     (K = classes)
//   dThat = s*g * G^T Vhat        [C,M] x [M,D]     (K = pixels, split-K over CTAs)
// and the normalise-backward  dx = (dxhat - xhat <xhat, dxhat>) / ||x||  needs only
//   <vhat_m, dVhat_m> = g * sum_c G[m,c] logits[m,c] =: g * r[m]
//   <that_c, dThat_c> = g * sum_m G[m,c] logits[m,c] =: g * rt[c]
// i.e. row / column sums of G (.) logits (k1b_prep_kernel) - no second pass over D.
//
// Both GEMMs run on tcgen05 straight from the forward's layouts - no transposes in memory:
//   dV : A = G  [b][c][p] (p contiguous)  -> MN-major A,   B = That [c][d] -> MN-major B
//   dT : A = Vhat [m][d] (d contiguous)   -> MN-major A,   B = G [b][c][p]  -> K-major B
// MN-major 128B-swizzled operand tiles are [K rows][64 elements] boxes written by TMA: 8 K-rows
// form one 1024-B swizzle atom (stride-byte-offset 1024 between atoms along K), 64-element
// groups along M/N are `box bytes` apart (leading-byte-offset).
#include "common.cuh"
#include "tc_common.cuh"

namespace lc2is {

constexpr int KB_THREADS = 192;

// ---------------------------------------------------------------------------------------------
// r[m] = sum_c G[m,c]*L[m,c]   ;   rt[set][c] += sum_m G[m,c]*L[m,c]
// CTA = 64 pixels x 4 class quarters (256 threads): thread (quarter q, pixel) walks the classes of its
// quarter (coalesced along pixels); class sums are reduced with warp shuffles (one warp = 32 pixels of one
// quarter) and added to rt with one reduction per (warp, class); pixel sums meet in shared memory.
constexpr int PREP_PX = 64, PREP_Q = 4;
__global__ void __launch_bounds__(PREP_PX * PREP_Q)
k1b_prep_kernel(const __nv_bfloat16* __restrict__ G, const float* __restrict__ L, int B, int C, int C_pad, int hw,
                int n_sets, float* __restrict__ r, float* __restrict__ rt) {
    __shared__ float racc[PREP_Q][PREP_PX];
    const int b = blockIdx.y;
    const int px = threadIdx.x % PREP_PX, q = threadIdx.x / PREP_PX;
    const int p = blockIdx.x * PREP_PX + px;
    const bool in = p < hw;
    const int lane = threadIdx.x & 31;
    const int cq = (C + PREP_Q - 1) / PREP_Q;
    const int c_lo = q * cq, c_hi = min(C, c_lo + cq);
    const __nv_bfloat16* g = G + (size_t)b * C_pad * hw + p;
    const float* l = L + (size_t)b * C * hw + p;
    float* rts = rt + (size_t)(n_sets > 1 ? b : 0) * C;
    float acc = 0.f;
    for (int c0 = c_lo; c0 < c_hi; c0 += 8) {
        float v[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int c = c0 + k;
            v[k] = (c < c_hi && in) ? __bfloat162float(g[(size_t)c * hw]) * __ldg(l + (size_t)c * hw) : 0.f;
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            acc += v[k];
            const float w = warp_sum(v[k]);
            if (lane == 0 && c0 + k < c_hi && w != 0.f) atomicAdd(rts + c0 + k, w);
        }
    }
    racc[q][px] = acc;
    __syncthreads();
    if (q == 0 && in) r[(size_t)b * hw + p] = (racc[0][px] + racc[1][px]) + (racc[2][px] + racc[3][px]);
}

// Same projections from the fp32 gradient [B,C,hw] (what K2 produces), fused with its conversion to the
// bf16 [B,C_pad,hw] operand of the two GEMMs (pad rows zeroed): one pass over G and the logits.
// CTA = 128 pixels x one class slice (blockIdx.z of PREPF_CS slices): warp w walks classes w, w+8, ... of the slice with
// one float4 of G and of the logits per lane; class sums leave with one reduction per (class, CTA), pixel sums meet in
// shared memory and leave with one reduction per (pixel, slice) (r is zeroed by the caller).
constexpr int PREPF_PX = 128, PREPF_W = 8, PREPF_CS = 4;
constexpr int PREPF_CPW = 8;                  // classes per warp and class round
__global__ void __launch_bounds__(PREPF_W * 32)
k1b_prep_f32_kernel(const float* __restrict__ G, const float* __restrict__ L, int B, int C, int C_pad, int hw,
                    int n_sets, int want_proj, int px_blocks, __nv_bfloat16* __restrict__ Gb, float* __restrict__ r,
                    float* __restrict__ rt, const float* __restrict__ row_scale) {
    // row_scale (LC2IS_BWD_RAW_V): the bf16 operand is G[m,c] * inv||v_m||, so that both GEMMs can run on the RAW V:
    //   dThat = (G inv)^T V = G^T Vhat,   dV = s (G inv) That - V inv^2 r   (the projections r, rt use the unscaled G)
    // px_blocks consecutive 128-pixel blocks per CTA: the class sums of a warp stay in registers across them, so rt
    // receives one reduction per (class, CTA) - with one block per CTA the 128^2 grid would hammer 150 addresses
    // with 300 K reductions
    __shared__ float racc_s[PREPF_W][PREPF_PX];
    griddep_wait();                               // G (and the gradient scale) come from the kernels before
    griddep_launch_dependents();                  // the GEMMs set up while this pass runs
    const int b = blockIdx.y;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int cper = ((C_pad + PREPF_CS - 1) / PREPF_CS + PREPF_W - 1) / PREPF_W * PREPF_W;
    const int c_lo = blockIdx.z * cper, c_hi = min(C_pad, c_lo + cper);
    float* rts = rt + (size_t)(n_sets > 1 ? b : 0) * C;
    // class rounds of PREPF_W * PREPF_CPW classes (one round up to C_pad = 256)
    for (int cr = c_lo; cr < c_hi; cr += PREPF_W * PREPF_CPW) {
        float csum[PREPF_CPW];
#pragma unroll
        for (int k = 0; k < PREPF_CPW; ++k) csum[k] = 0.f;
        for (int pb = 0; pb < px_blocks; ++pb) {
            const int p0 = (blockIdx.x * px_blocks + pb) * PREPF_PX;
            if (p0 >= hw) break;
            const int p = p0 + lane * 4;
            const bool in = p < hw;                              // hw % 4 == 0
            const float* g = G + (size_t)b * C * hw + p;
            const float* l = L + (size_t)b * C * hw + p;
            __nv_bfloat16* gb = Gb + (size_t)b * C_pad * hw + p;
            float4 racc = make_float4(0.f, 0.f, 0.f, 0.f);
            float4 rs = make_float4(1.f, 1.f, 1.f, 1.f);
            if (row_scale && in) rs = __ldg(reinterpret_cast<const float4*>(row_scale + (size_t)b * hw + p));
            // every load of the warp's classes is issued before the first value is used (one class at a time left two 16-byte
            // loads in flight per lane and the kernel at 4.3 TB/s: 68 % of its samples waited on the first use of gv)
            float4 gv[PREPF_CPW], lv[PREPF_CPW];
#pragma unroll
            for (int k = 0; k < PREPF_CPW; ++k) {
                const int c = cr + warp + k * PREPF_W;
                gv[k] = make_float4(0.f, 0.f, 0.f, 0.f);
                lv[k] = gv[k];
                if (c < c_hi && c < C && in) {
                    gv[k] = __ldcs(reinterpret_cast<const float4*>(g + (size_t)c * hw));
                    if (want_proj) lv[k] = __ldg(reinterpret_cast<const float4*>(l + (size_t)c * hw));
                }
            }
#pragma unroll
            for (int k = 0; k < PREPF_CPW; ++k) {
                const int c = cr + warp + k * PREPF_W;
                if (c < c_hi && in) {
                    __nv_bfloat162 lo = __floats2bfloat162_rn(gv[k].x * rs.x, gv[k].y * rs.y), hi = __floats2bfloat162_rn(gv[k].z * rs.z, gv[k].w * rs.w);
                    uint2 pk;
                    pk.x = *reinterpret_cast<unsigned*>(&lo); pk.y = *reinterpret_cast<unsigned*>(&hi);
                    *reinterpret_cast<uint2*>(gb + (size_t)c * hw) = pk;
                }
                if (want_proj && c < c_hi && c < C) {
                    const float4 pr = make_float4(gv[k].x * lv[k].x, gv[k].y * lv[k].y, gv[k].z * lv[k].z, gv[k].w * lv[k].w);
                    racc.x += pr.x; racc.y += pr.y; racc.z += pr.z; racc.w += pr.w;
                    csum[k] += (pr.x + pr.y) + (pr.z + pr.w);
                }
            }
            if (want_proj) {
                *reinterpret_cast<float4*>(&racc_s[warp][lane * 4]) = racc;
                __syncthreads();
                if (threadIdx.x < PREPF_PX) {
                    const int pp = p0 + threadIdx.x;
                    float t = 0.f;
#pragma unroll
                    for (int w = 0; w < PREPF_W; ++w) t += racc_s[w][threadIdx.x];
                    if (pp < hw) atomicAdd(r + (size_t)b * hw + pp, t);
                }
                __syncthreads();
            }
        }
        if (want_proj) {
#pragma unroll
            for (int k = 0; k < PREPF_CPW; ++k) {
                const int c = cr + warp + k * PREPF_W;
                const float s = warp_sum(csum[k]);
                if (lane == 0 && c < c_hi && c < C && s != 0.f) atomicAdd(rts + c, s);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// dV GEMM.  Tile = 128 pixels x 256 channels (2 n-tiles of D=512 ...), K = C_pad in steps of 16.
struct DvParams {
    void* grad_v;               // [M, D] bf16 or fp32
    const __nv_bfloat16* v_hat; // [M, D]
    const float* inv_v;         // [M]
    const float* r;             // [M]
    const float* grad_scale;    // device scalar or null
    int B, hw, D, C_pad, n_sets;
    int tiles_per_img, n_ntiles, num_kb, stages;
    int normalize, out_f32;
    int raw_v;                  // v_hat points at the RAW bf16 V and G was scaled by inv||v|| (LC2IS_BWD_RAW_V)
    float scale;
};
constexpr int DV_BM = 128, DV_BN = 256, DV_KB = 16;
constexpr int DV_A_BYTES = 2 * DV_KB * 128;            // 2 boxes [16 k][64 p]
constexpr int DV_B_BYTES = (DV_BN / 64) * DV_KB * 128; // 4 boxes [16 k][64 d]
constexpr int DV_STAGE = DV_A_BYTES + DV_B_BYTES;      // 12 KB
constexpr int DV_MAX_STAGES = 12;

constexpr int DV_EPI_WARPS = 8;                        // two epilogue warps per TMEM lane quarter
constexpr int DV_THREADS = 64 + 32 * DV_EPI_WARPS;
__global__ void __launch_bounds__(DV_THREADS, 1)
k1b_dv_kernel(const __grid_constant__ CUtensorMap tmG, const __grid_constant__ CUtensorMap tmT, const DvParams P) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base_u32 = (tc::smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem = smem_raw + (base_u32 - tc::smem_u32(smem_raw));
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)P.stages * DV_STAGE);
    uint64_t* empty = full + DV_MAX_STAGES;
    uint64_t* tfull = empty + DV_MAX_STAGES;
    uint64_t* tempty = tfull + 2;
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tempty + 2);
    uint8_t* epi_scr = reinterpret_cast<uint8_t*>(full) + 512;  // 8 warps x (4 KB v_hat in + 4 KB gradient out)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int total_tiles = P.B * P.tiles_per_img * P.n_ntiles;

    if (warp == 0 && lane == 0) {
        tc::prefetch_tmap(&tmG);
        tc::prefetch_tmap(&tmT);
        for (int i = 0; i < P.stages; ++i) { tc::mbar_init(full + i, 1); tc::mbar_init(empty + i, 1); }
        for (int i = 0; i < 2; ++i) { tc::mbar_init(tfull + i, 1); tc::mbar_init(tempty + i, DV_EPI_WARPS); }
        tc::fence_barrier_init();
    }
    if (warp == 1) tc::tmem_alloc(tmem_ptr, 512);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    griddep_wait();                                      // the bf16 operand and r come from the prep kernel
    griddep_launch_dependents();

    if (warp == 0) {
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                const int nt = tile % P.n_ntiles, mt = tile / P.n_ntiles;
                const int b = mt / P.tiles_per_img, ti = mt - b * P.tiles_per_img;
                const int trow0 = (P.n_sets > 1 ? b : 0) * P.C_pad;
                for (int kb = 0; kb < P.num_kb; ++kb) {
                    tc::mbar_wait(empty + stage, phase ^ 1);
                    uint8_t* sa = smem + (size_t)stage * DV_STAGE;
                    tc::mbar_arrive_expect_tx(full + stage, DV_STAGE);
#pragma unroll
                    for (int j = 0; j < 2; ++j)     // A: G[b][kb*16 .. +16][ti*128 + j*64 .. +64]
                        tc::tma_load_3d(sa + j * DV_KB * 128, &tmG, full + stage, ti * DV_BM + j * 64, kb * DV_KB, b);
#pragma unroll
                    for (int j = 0; j < DV_BN / 64; ++j)   // B: That[trow0 + kb*16 .. +16][nt*256 + j*64 .. +64]
                        tc::tma_load_2d(sa + DV_A_BYTES + j * DV_KB * 128, &tmT, full + stage,
                                        nt * DV_BN + j * 64, trow0 + kb * DV_KB);
                    if (++stage == P.stages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc = tc::make_idesc_bf16(DV_BM, DV_BN, 1, 1);
            int stage = 0; uint32_t phase = 0;
            int it = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
                const int buf = it & 1;
                const uint32_t bphase = (it >> 1) & 1;
                tc::mbar_wait(tempty + buf, bphase ^ 1);
                tc::tc_fence_after();
                const uint32_t d_tmem = tmem_base + buf * 256;
                for (int kb = 0; kb < P.num_kb; ++kb) {
                    tc::mbar_wait(full + stage, phase);
                    tc::tc_fence_after();
                    const uint32_t sa = base_u32 + stage * DV_STAGE;
                    // MN-major: LBO = bytes between 64-element M/N groups, SBO = 1024 (8 K-rows)
                    const uint64_t adesc = tc::make_smem_desc(sa, DV_KB * 128, 1024);
                    const uint64_t bdesc = tc::make_smem_desc(sa + DV_A_BYTES, DV_KB * 128, 1024);
                    tc::umma_bf16(d_tmem, adesc, bdesc, idesc, kb != 0);
                    tc::umma_commit(empty + stage);
                    if (++stage == P.stages) { stage = 0; phase ^= 1; }
                }
                tc::umma_commit(tfull + buf);
            }
        }
    } else {
        const int q = warp & 3;
        const float gs = P.grad_scale ? __ldg(P.grad_scale) : 1.f;
        const float sg = P.scale * gs;
        int it = 0;
        // the row's factors (1 / ||v||, r) are fetched one TILE ahead: read at the top of the tile they were an exposed
        // global-load latency per tile (19 % of the kernel's samples with 28 tiles per CTA at 128 x 128 patches)
        float inv_n = 0.f, r_n = 0.f;
        auto fetch_row = [&](int tile) {
            const int mt = tile / P.n_ntiles;
            const int b = mt / P.tiles_per_img, ti = mt - b * P.tiles_per_img;
            const int p = ti * DV_BM + q * 32 + lane;
            const bool rv = p < P.hw;
            const size_t m = (size_t)b * P.hw + (rv ? p : 0);
            inv_n = rv ? __ldg(P.inv_v + m) : 0.f;
            r_n = (rv && P.normalize) ? __ldg(P.r + m) : 0.f;
        };
        if ((int)blockIdx.x < total_tiles) fetch_row(blockIdx.x);
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
            const int buf = it & 1;
            const uint32_t bphase = (it >> 1) & 1;
            const int nt = tile % P.n_ntiles, mt = tile / P.n_ntiles;
            const int b = mt / P.tiles_per_img, ti = mt - b * P.tiles_per_img;
            const float inv = inv_n;
            float rr = r_n * gs;
            if (tile + (int)gridDim.x < total_tiles) fetch_row(tile + (int)gridDim.x);
            // raw V: acc already carries inv (G was scaled by it): dV = s acc - v (inv^2 r)
            const float oinv = P.raw_v ? 1.f : inv;
            if (P.raw_v) rr *= inv * inv;
            // 64 channels = 128 bytes of v_hat per row at a time.  The two warps of a lane quarter take alternate groups.
            // v_hat is fetched coalesced (4 rows x 128 bytes per load) one group AHEAD into registers - the first group
            // before the accumulator is even ready - parked in the warp's swizzled scratch and read back by the thread that
            // owns the row; the gradient leaves the same way (a thread owns a ROW in TMEM: direct accesses touch 32 rows).
            const int part = (warp - 2) >> 2;
            uint8_t* scr_in = epi_scr + (warp - 2) * 8192;
            uint8_t* scr_out = scr_in + 4096;
            const int pw = ti * DV_BM + q * 32;
            const int rows_valid = P.hw - pw < 0 ? 0 : (P.hw - pw < 32 ? P.hw - pw : 32);
            const size_t m0 = (size_t)b * P.hw + pw;
            const int d0 = nt * DV_BN;
            const int n_groups = (P.D - d0 < DV_BN ? P.D - d0 : DV_BN) / 64;      // D % 64 == 0
            uint4 pf[8];
            auto ldg_group = [&](int g) {
                const uint8_t* src = reinterpret_cast<const uint8_t*>(P.v_hat + m0 * P.D + d0 + g * 64);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int row = i * 4 + (lane >> 3);
                    pf[i] = row < rows_valid
                                ? __ldg(reinterpret_cast<const uint4*>(src + (size_t)row * P.D * 2 + ((lane & 7) << 4)))
                                : make_uint4(0u, 0u, 0u, 0u);
                }
            };
            if (P.normalize && part < n_groups) ldg_group(part);
            tc::mbar_wait(tfull + buf, bphase);
            tc::tc_fence_after();
            const uint32_t taddr = tmem_base + buf * 256 + ((uint32_t)(q * 32) << 16);
            for (int g = part; g < n_groups; g += DV_EPI_WARPS / 4) {
                const int col0 = g * 64;
                if (P.normalize) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int row = i * 4 + (lane >> 3);
                        *reinterpret_cast<uint4*>(scr_in + row * 128 + (((lane & 7) ^ (row & 7)) << 4)) = pf[i];
                    }
                    __syncwarp();
                    if (g + DV_EPI_WARPS / 4 < n_groups) ldg_group(g + DV_EPI_WARPS / 4);
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int col = col0 + 16 * k;
                    uint32_t acc[16];
                    tc::tmem_ld16(taddr + col, acc);
                    tc::tmem_ld_wait();
                    float o[16];
                    if (P.normalize) {
                        const uint4 v0 = epi_get(scr_in, lane, 2 * k), v1 = epi_get(scr_in, lane, 2 * k + 1);
                        unsigned w[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const float va = __uint_as_float(w[j] << 16), vb = __uint_as_float(w[j] & 0xffff0000u);
                            o[2 * j] = (__uint_as_float(acc[2 * j]) * sg - va * rr) * oinv;
                            o[2 * j + 1] = (__uint_as_float(acc[2 * j + 1]) * sg - vb * rr) * oinv;
                        }
                    } else {
#pragma unroll
                        for (int j = 0; j < 16; ++j) o[j] = __uint_as_float(acc[j]) * sg;
                    }
                    if (P.out_f32) {                            // 32 fp32 channels per 128-byte group: flush after two chunks
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            epi_put(scr_out, lane, (k & 1) * 4 + j,
                                    make_uint4(__float_as_uint(o[4 * j]), __float_as_uint(o[4 * j + 1]),
                                               __float_as_uint(o[4 * j + 2]), __float_as_uint(o[4 * j + 3])));
                        if (k & 1) {
                            __syncwarp();
                            epi_flush(scr_out, lane,
                                      reinterpret_cast<uint8_t*>(P.grad_v) + (m0 * P.D + d0 + col - 16) * 4,
                                      (size_t)P.D * 4, rows_valid, 8);
                            __syncwarp();
                        }
                    } else {
                        __nv_bfloat162 pk[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) pk[j] = __floats2bfloat162_rn(o[2 * j], o[2 * j + 1]);
                        epi_put(scr_out, lane, 2 * k, *reinterpret_cast<uint4*>(&pk[0]));
                        epi_put(scr_out, lane, 2 * k + 1, *reinterpret_cast<uint4*>(&pk[4]));
                    }
                }
                if (!P.out_f32) {
                    __syncwarp();
                    epi_flush(scr_out, lane, reinterpret_cast<uint8_t*>(P.grad_v) + (m0 * P.D + d0 + col0) * 2,
                              (size_t)P.D * 2, rows_valid, 8);
                }
                __syncwarp();                                   // scr_in / scr_out are rewritten by the next group
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
// dT GEMM (split-K).  Work item = (set, d-tile of 128, class tile of NB, K range of 64-pixel blocks);
// the partial [128 x NB] accumulator is added to dT_raw[set][c][d] with fp32 L2 reductions.
struct DtParams {
    float* dt_raw;              // [n_sets, C, D] fp32, pre-zeroed
    int B, hw, D, C, C_pad, n_sets;
    int NB, n_ntiles, n_dtiles, ksplit, kb_per_img, stages;
};
constexpr int DT_BM = 128, DT_KB = 64;
constexpr int DT_A_BYTES = 2 * DT_KB * 128;           // 2 boxes [64 p][64 d] = 16 KB
constexpr int DT_MAX_STAGES = 8;

// B_MN = false: B = G [b][class][pixel], K-major (the prototype gradient).  B_MN = true: B = a row-major [rows][N] matrix,
// i.e. MN-major like A (the weight gradient of TextToPatch.visual: dW^T tile = X^T . Gy, lc2is_linear_bwd).
// MT = number of 128-row M tiles per CTA (accumulators side by side in TMEM; MT = 2 halves the L2 traffic of B per flop -
// the split-K weight gradient is L2-bound).  STORE: the partial tile is written with plain stores to slice `ks` of a
// [ksplit][C][D] workspace (summed by reduce_partials_kernel) instead of fp32 reductions into dt_raw.
template <bool B_MN, int MT, bool STORE>
__global__ void __launch_bounds__(KB_THREADS, 1)
k1b_dt_kernel(const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmG, const DtParams P) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base_u32 = (tc::smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem = smem_raw + (base_u32 - tc::smem_u32(smem_raw));
    const int stage_bytes = MT * DT_A_BYTES + P.NB * 128;
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)P.stages * stage_bytes);
    uint64_t* empty = full + DT_MAX_STAGES;
    uint64_t* tfull = empty + DT_MAX_STAGES;
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tfull + 1);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    // decode the work item of this CTA
    int w = blockIdx.x;
    const int ks = w % P.ksplit; w /= P.ksplit;
    const int nt = w % P.n_ntiles; w /= P.n_ntiles;
    const int dt = w % P.n_dtiles; w /= P.n_dtiles;
    const int set = w;                                   // 0 when the prototypes are shared
    // K blocks: shared prototypes -> all images concatenated; per-image prompts -> image `set` only
    const int total_kb = (P.n_sets > 1 ? 1 : P.B) * P.kb_per_img;
    const int kb_lo = (int)((long long)total_kb * ks / P.ksplit);
    const int kb_hi = (int)((long long)total_kb * (ks + 1) / P.ksplit);
    const int nkb = kb_hi - kb_lo;

    if (warp == 0 && lane == 0) {
        tc::prefetch_tmap(&tmV);
        tc::prefetch_tmap(&tmG);
        for (int i = 0; i < P.stages; ++i) { tc::mbar_init(full + i, 1); tc::mbar_init(empty + i, 1); }
        tc::mbar_init(tfull, 1);
        tc::fence_barrier_init();
    }
    if (warp == 1) tc::tmem_alloc(tmem_ptr, MT * 256);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    griddep_wait();                                      // B (and A) may come from the kernel before
    griddep_launch_dependents();

    if (nkb > 0) {
        if (warp == 0) {
            if (lane == 0) {
                int stage = 0; uint32_t phase = 0;
                for (int kb = kb_lo; kb < kb_hi; ++kb) {
                    const int b = P.n_sets > 1 ? set : kb / P.kb_per_img;
                    const int kl = P.n_sets > 1 ? kb : kb - b * P.kb_per_img;
                    tc::mbar_wait(empty + stage, phase ^ 1);
                    uint8_t* sa = smem + (size_t)stage * stage_bytes;
                    tc::mbar_arrive_expect_tx(full + stage, (uint32_t)stage_bytes);
#pragma unroll
                    for (int j = 0; j < 2 * MT; ++j)   // A: Vhat[b*hw + kl*64 .. +64][dt*128*MT + j*64 .. +64]
                        tc::tma_load_2d(sa + j * DT_KB * 128, &tmV, full + stage, dt * DT_BM * MT + j * 64,
                                        b * P.hw + kl * DT_KB);
                    if (B_MN) {                   // B: Gy[b*hw + kl*64 .. +64][nt*NB + j*64 .. +64], boxes [64 k][64 n]
                        for (int j = 0; j < P.NB / 64; ++j)
                            tc::tma_load_2d(sa + MT * DT_A_BYTES + j * DT_KB * 128, &tmG, full + stage, nt * P.NB + j * 64,
                                            b * P.hw + kl * DT_KB);
                    } else {
                        // B: G[b][nt*NB .. +NB][kl*64 .. +64]   (K-major; OOB pixels / classes read as 0)
                        tc::tma_load_3d(sa + MT * DT_A_BYTES, &tmG, full + stage, kl * DT_KB, nt * P.NB, b);
                    }
                    if (++stage == P.stages) { stage = 0; phase ^= 1; }
                }
            }
        } else if (warp == 1) {
            if (lane == 0) {
                const uint32_t idesc = tc::make_idesc_bf16(DT_BM, P.NB, 1, B_MN ? 1 : 0);
                int stage = 0; uint32_t phase = 0;
                for (int kb = kb_lo; kb < kb_hi; ++kb) {
                    tc::mbar_wait(full + stage, phase);
                    tc::tc_fence_after();
                    const uint32_t sa = base_u32 + stage * stage_bytes;
                    const uint64_t bdesc = B_MN ? tc::make_smem_desc(sa + MT * DT_A_BYTES, DT_KB * 128, 1024)   // MN-major B
                                                : tc::make_smem_desc(sa + MT * DT_A_BYTES, 16, 1024);           // K-major B
#pragma unroll
                    for (int mt = 0; mt < MT; ++mt) {
                        const uint64_t adesc = tc::make_smem_desc(sa + mt * DT_A_BYTES, DT_KB * 128, 1024);   // MN-major A
#pragma unroll
                        for (int k = 0; k < DT_KB / 16; ++k)   // MN-major: +16 K-rows = 2 atoms = 2048 B; K-major B: +32 B
                            tc::umma_bf16(tmem_base + (uint32_t)(mt * P.NB), adesc + (uint64_t)(k * 128),
                                          bdesc + (uint64_t)(B_MN ? k * 128 : 2 * k), idesc, (kb != kb_lo) || (k != 0));
                    }
                    tc::umma_commit(empty + stage);
                    if (++stage == P.stages) { stage = 0; phase ^= 1; }
                }
                tc::umma_commit(tfull);
            }
        } else {
            const int q = warp & 3;
            tc::mbar_wait(tfull, 0);
            tc::tc_fence_after();
            const int c0 = nt * P.NB;
#pragma unroll 1
            for (int mt = 0; mt < MT; ++mt) {
                const int d = (dt * MT + mt) * DT_BM + q * 32 + lane;
                const uint32_t taddr = tmem_base + (uint32_t)(mt * P.NB) + ((uint32_t)(q * 32) << 16);
                float* out = P.dt_raw + (size_t)(STORE ? ks : set) * P.C * P.D + d;
                for (int col = 0; col < P.NB; col += 16) {
                    if (c0 + col >= P.C) break;
                    uint32_t acc[16];
                    tc::tmem_ld16(taddr + col, acc);
                    tc::tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const int c = c0 + col + j;
                        if (c < P.C && d < P.D) {
                            if (STORE) out[(size_t)c * P.D] = __uint_as_float(acc[j]);     // lanes: consecutive d
                            else atomicAdd(out + (size_t)c * P.D, __uint_as_float(acc[j]));
                        }
                    }
                }
            }
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc::tc_fence_after();
        tc::tmem_dealloc(tmem_base, MT * 256);
    }
}

// out[i] += sum_s part[s][i]   (the split-K slices of the weight gradient)
__global__ void __launch_bounds__(256)
reduce_partials_kernel(const float4* __restrict__ part, int nslices, long long n4, float4* __restrict__ out) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
        float4 a = out[i];
        for (int s = 0; s < nslices; ++s) {
            const float4 v = __ldcs(part + (size_t)s * n4 + i);
            a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
        }
        out[i] = a;
    }
}

// dT[set][c][:] += inv_t * g * (s * dT_raw - that * rt)      (normalise-backward of the prototypes)
__global__ void __launch_bounds__(256)
k1b_dt_finish_kernel(const float* __restrict__ dt_raw, const float* __restrict__ rt,
                     const __nv_bfloat16* __restrict__ t_hat, const float* __restrict__ inv_t,
                     const float* __restrict__ grad_scale, int n_sets, int C, int C_pad, int D, int normalize,
                     float scale, float* __restrict__ grad_t) {
    griddep_wait();
    const float gs = grad_scale ? __ldg(grad_scale) : 1.f;
    const long long total = (long long)n_sets * C * D;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const int d = (int)(i % D);
        const long long sc = i / D;
        const int c = (int)(sc % C);
        const int set = (int)(sc / C);
        float v = scale * dt_raw[i];
        if (normalize) {
            const float th = __bfloat162float(t_hat[((size_t)set * C_pad + c) * D + d]);
            v = (v - th * rt[(size_t)set * C + c]) * inv_t[(size_t)set * C + c];
        }
        grad_t[i] += gs * v;
    }
}

// ---- TextToPatch.visual backward helpers ---------------------------------------------------------------------------
// W [N][K] -> Wt [K][N] (bf16): the weight in the layout lc2is_linear_fwd wants for gx = gy . W
__global__ void __launch_bounds__(256)
transpose_bf16_kernel(const __nv_bfloat16* __restrict__ in, int N, int K, __nv_bfloat16* __restrict__ out) {
    __shared__ __nv_bfloat16 tile[32][33];
    const int k0 = blockIdx.x * 32, n0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int r = ty; r < 32; r += 8)
        if (n0 + r < N && k0 + tx < K) tile[r][tx] = in[(size_t)(n0 + r) * K + k0 + tx];
    __syncthreads();
    for (int r = ty; r < 32; r += 8)
        if (k0 + r < K && n0 + tx < N) out[(size_t)(k0 + r) * N + n0 + tx] = tile[tx][r];
}
// part[cta][n] = sum over the CTA's rows of gy[m][n]: a pure HBM stream (16-byte loads, eight columns per thread, eight
// loads in flight); colsum_finish_kernel adds the CTAs' partial sums to gb (same-address reductions from ~600 CTAs
// serialise in L2: 107 us for 268 MB with atomics)
constexpr int CS_THREADS = 1024;                           // 2 CTAs per SM: latency is hidden by warps, not by unrolling
__global__ void __launch_bounds__(CS_THREADS)
colsum_bf16_kernel(const __nv_bfloat16* __restrict__ gy, long long M, int N, float* __restrict__ part) {
    const int nvec = N / 8;                                   // N % 8 == 0
    const int tpr = nvec < CS_THREADS ? nvec : CS_THREADS;                  // threads that own a column group in this CTA's pass
    const int rows_per_pass = CS_THREADS / tpr;
    const int cg = threadIdx.x % tpr, rsub = threadIdx.x / tpr;
    for (int v0 = 0; v0 < nvec; v0 += tpr) {
        const int vcol = v0 + cg;
        float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        if (vcol < nvec && rsub < rows_per_pass)
        {
            const long long stride = (long long)gridDim.x * rows_per_pass;
            const uint4* src = reinterpret_cast<const uint4*>(gy) + vcol;
            const size_t rowv = (size_t)N / 8;                 // 16-byte vectors per row
            auto add = [&](const uint4 q) {
                const unsigned wd[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    acc[2 * i] += __uint_as_float(wd[i] << 16);
                    acc[2 * i + 1] += __uint_as_float(wd[i] & 0xffff0000u);
                }
            };
            long long m0 = (long long)blockIdx.x * rows_per_pass + rsub;
            for (; m0 + 7 * stride < M; m0 += 8 * stride) {   // eight unconditional 16-byte loads in flight per thread
                uint4 q[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) q[u] = __ldcs(src + (size_t)(m0 + u * stride) * rowv);
#pragma unroll
                for (int u = 0; u < 8; ++u) add(q[u]);
            }
            for (; m0 < M; m0 += stride) add(__ldcs(src + (size_t)m0 * rowv));
        }
        // the CTA's row groups are summed in shared memory first: one reduction per column and CTA
        __shared__ float red[CS_THREADS][8];
#pragma unroll
        for (int i = 0; i < 8; ++i) red[threadIdx.x][i] = acc[i];
        __syncthreads();
        if (vcol < nvec && rsub == 0) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                float t = 0.f;
                for (int r = 0; r < rows_per_pass; ++r) t += red[r * tpr + cg][i];
                part[(size_t)blockIdx.x * N + vcol * 8 + i] = t;
            }
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256)
colsum_finish_kernel(const float* __restrict__ part, int nparts, int N, float* __restrict__ gb) {
    // 32 columns per CTA, the partial sums split eight ways (a thread that walked all of them alone was latency-bound)
    __shared__ float red[8][32];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int n = blockIdx.x * 32 + tx;
    float t = 0.f;
    if (n < N)
        for (int b = ty; b < nparts; b += 8) t += part[(size_t)b * N + n];
    red[ty][tx] = t;
    __syncthreads();
    if (ty == 0 && n < N) {
#pragma unroll
        for (int r = 1; r < 8; ++r) t += red[r][tx];
        gb[n] += t;
    }
}

struct BwdWs { size_t r, rt, dt_raw, gbf, total; };
static BwdWs bwd_layout(int B, int hw, int D, int n_sets, int C) {
    auto al = [](size_t x) { return (x + 255) / 256 * 256; };
    BwdWs w; size_t o = 0;
    w.r = o; o += al((size_t)B * hw * 4);
    w.rt = o; o += al((size_t)n_sets * C * 4);
    w.dt_raw = o; o += al((size_t)n_sets * C * D * 4);
    w.gbf = o; o += al((size_t)B * class_pad(C) * hw * 2);     // bf16 copy of an fp32 gradient
    w.total = o;
    return w;
}

}  // namespace lc2is

using namespace lc2is;

extern "C" int64_t lc2is_cosine_logits_bwd_workspace(int B, int hw, int D, int n_sets, int C) {
    return (int64_t)bwd_layout(B, hw, D, n_sets, C).total;
}

// r, rt and dt_raw: the head of the workspace that LC2IS_BWD_WS_ZEROED says is zero
extern "C" int64_t lc2is_cosine_logits_bwd_workspace_zeroed(int B, int hw, int D, int n_sets, int C) {
    return (int64_t)bwd_layout(B, hw, D, n_sets, C).gbf;
}

extern "C" int lc2is_cosine_logits_bwd_ex(const void* d_grad_logits, int g_dtype, const float* d_logits,
                                       const void* d_v_hat, const float* d_inv_norm_v,
                                       const void* d_t_hat, const float* d_inv_norm_t,
                                       int B, int hw, int D, int n_sets, int C,
                                       int normalize, float logit_scale, const float* d_grad_scale,
                                       void* d_grad_v, int gv_dtype, float* d_grad_t,
                                       void* d_ws, lc2is_stream_t stream, int flags) {
    if (int e = ensure_device()) return e;
    if (B < 0 || hw <= 0 || C <= 0 || D <= 0) return fail(LC2IS_ERR_SHAPE, "bad shape%s");
    if (B == 0) return 0;
    if (!d_grad_logits || !d_logits || !d_v_hat || !d_inv_norm_v || !d_t_hat || !d_ws)
        return fail(LC2IS_ERR_ARG, "null pointer%s");
    if (g_dtype != LC2IS_F32 && g_dtype != LC2IS_BF16) return fail(LC2IS_ERR_ARG, "g_dtype%s");
    if (normalize && !d_inv_norm_t) return fail(LC2IS_ERR_ARG, "inv_norm_t required when normalize%s");
    if (D % 64) return fail(LC2IS_ERR_SHAPE, "D must be a multiple of 64%s");
    if (hw % 8) return fail(LC2IS_ERR_SHAPE, "hw must be a multiple of 8 for the backward (TMA 16-byte strides); got %s%lld", "", hw);
    if (n_sets != 1 && n_sets != B) return fail(LC2IS_ERR_SHAPE, "n_sets must be 1 or B%s");
    if (gv_dtype != LC2IS_F32 && gv_dtype != LC2IS_BF16) return fail(LC2IS_ERR_ARG, "gv_dtype%s");
    cudaStream_t st = (cudaStream_t)stream;
    const int C_pad = class_pad(C);
    const BwdWs L = bwd_layout(B, hw, D, n_sets, C);
    uint8_t* ws = (uint8_t*)d_ws;
    float* d_r = (float*)(ws + L.r);
    float* d_rt = (float*)(ws + L.rt);
    float* d_dtraw = (float*)(ws + L.dt_raw);
    const bool reuse = (flags & LC2IS_BWD_REUSE_PREP) != 0;
    const bool raw_v = (flags & LC2IS_BWD_RAW_V) != 0;
    if (raw_v && (!normalize || g_dtype != LC2IS_F32))
        return fail(LC2IS_ERR_ARG, "LC2IS_BWD_RAW_V needs normalize = 1 and an fp32 gradient (its bf16 operand is scaled by inv||v||)%s");
    if (reuse && d_grad_t) return fail(LC2IS_ERR_ARG, "LC2IS_BWD_REUSE_PREP is for a dV-only call (d_grad_t must be NULL)%s");
    // r, rt and dt_raw.  The kernels below are launched with launch_pdl: a memset between two of them would break the
    // chain, so a step that zero-fills them at its start passes LC2IS_BWD_WS_ZEROED
    if (!reuse && !(flags & LC2IS_BWD_WS_ZEROED)) LC2IS_CUDA(cudaMemsetAsync(ws + L.r, 0, L.gbf - L.r, st));

    // ---- projections r, rt (and the bf16 operand copy of an fp32 gradient) -------------------------
    const void* d_grad_logits_bf16 = g_dtype == LC2IS_F32 ? (const void*)(ws + L.gbf) : d_grad_logits;
    if (reuse) {
        // projections / bf16 operand are in the workspace already
    } else if (g_dtype == LC2IS_F32) {
        const int nblk = (hw + PREPF_PX - 1) / PREPF_PX;
        int px_blocks = nblk / 16;                           // >= 16 CTAs per image and class slice
        if (px_blocks < 1) px_blocks = 1;
        if (px_blocks > 16) px_blocks = 16;
        dim3 grid((nblk + px_blocks - 1) / px_blocks, B, PREPF_CS);
        LC2IS_CUDA(launch_pdl(k1b_prep_f32_kernel, grid, PREPF_W * 32, 0, st, (const float*)d_grad_logits, d_logits, B,
                              C, C_pad, hw, n_sets, normalize, px_blocks, (__nv_bfloat16*)(ws + L.gbf), d_r, d_rt,
                              raw_v ? d_inv_norm_v : nullptr));
        LC2IS_CHECK_LAUNCH("k1b_prep_f32_kernel");
    } else if (normalize) {
        dim3 grid((hw + PREP_PX - 1) / PREP_PX, B);
        k1b_prep_kernel<<<grid, PREP_PX * PREP_Q, 0, st>>>((const __nv_bfloat16*)d_grad_logits_bf16, d_logits, B, C,
                                                           C_pad, hw, n_sets, d_r, d_rt);
        LC2IS_CHECK_LAUNCH("k1b_prep_kernel");
    }
    // ---- dV ----------------------------------------------------------------------------------------
    if (d_grad_v) {
        DvParams P;
        P.grad_v = d_grad_v; P.v_hat = (const __nv_bfloat16*)d_v_hat; P.inv_v = d_inv_norm_v; P.r = d_r;
        P.grad_scale = d_grad_scale; P.B = B; P.hw = hw; P.D = D; P.C_pad = C_pad; P.n_sets = n_sets;
        P.tiles_per_img = (hw + DV_BM - 1) / DV_BM;
        P.n_ntiles = (D + DV_BN - 1) / DV_BN;
        P.num_kb = C_pad / DV_KB;
        P.stages = P.num_kb * 2 < 8 ? P.num_kb * 2 : 8;       // the K loop is short: 8 x 12 KB leaves room for the epilogue scratch
        if (P.stages < 2) P.stages = 2;
        P.normalize = normalize; P.out_f32 = gv_dtype == LC2IS_F32; P.scale = logit_scale; P.raw_v = raw_v ? 1 : 0;
        CUtensorMap tmG, tmT;
        if (int e = make_tmap_3d_bf16(&tmG, d_grad_logits_bf16, B, C_pad, hw, DV_KB, 64)) return e;
        if (int e = make_tmap_2d_bf16(&tmT, d_t_hat, (uint64_t)n_sets * C_pad, D, DV_KB, 64)) return e;
        size_t smem = (size_t)P.stages * DV_STAGE + 1024 + 512 + DV_EPI_WARPS * 8192;
        if (smem < 120 * 1024) smem = 120 * 1024;
        LC2IS_CUDA(cudaFuncSetAttribute(k1b_dv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const int total_tiles = B * P.tiles_per_img * P.n_ntiles;
        int grid = sm_count() < total_tiles ? sm_count() : total_tiles;
        LC2IS_CUDA(launch_pdl(k1b_dv_kernel, grid, DV_THREADS, smem, st, tmG, tmT, P));
        LC2IS_CHECK_LAUNCH("k1b_dv_kernel");
    }
    // ---- dT ----------------------------------------------------------------------------------------
    if (d_grad_t) {
        DtParams P;
        P.dt_raw = d_dtraw; P.B = B; P.hw = hw; P.D = D; P.C = C; P.C_pad = C_pad; P.n_sets = n_sets;
        const int n0 = (C_pad + 255) / 256;
        P.NB = ((C_pad + n0 - 1) / n0 + 15) / 16 * 16;
        P.n_ntiles = (C_pad + P.NB - 1) / P.NB;
        P.n_dtiles = (D + DT_BM - 1) / DT_BM;
        P.kb_per_img = (hw + DT_KB - 1) / DT_KB;
        const int base_items = n_sets * P.n_dtiles * P.n_ntiles;
        const int total_kb = (n_sets > 1 ? 1 : B) * P.kb_per_img;
        int ksplit = sm_count() / base_items;
        if (ksplit < 1) ksplit = 1;
        if (ksplit > total_kb) ksplit = total_kb;
        P.ksplit = ksplit;
        const int stage_bytes = DT_A_BYTES + P.NB * 128;
        int stages = (200 * 1024) / stage_bytes;
        if (stages > DT_MAX_STAGES) stages = DT_MAX_STAGES;
        P.stages = stages;
        CUtensorMap tmV, tmG;
        if (int e = make_tmap_2d_bf16(&tmV, d_v_hat, (uint64_t)B * hw, D, DT_KB, 64)) return e;
        if (int e = make_tmap_3d_bf16(&tmG, d_grad_logits_bf16, B, C_pad, hw, P.NB, 64)) return e;
        size_t smem = (size_t)stages * stage_bytes + 1024 + 256;
        if (smem < 120 * 1024) smem = 120 * 1024;
        LC2IS_CUDA(cudaFuncSetAttribute(k1b_dt_kernel<false, 1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        LC2IS_CUDA(launch_pdl(k1b_dt_kernel<false, 1, false>, base_items * ksplit, KB_THREADS, smem, st, tmV, tmG, P));
        LC2IS_CHECK_LAUNCH("k1b_dt_kernel");
        long long total = (long long)n_sets * C * D;
        long long blocks = (total + 255) / 256;
        if (blocks > sm_count() * 8) blocks = sm_count() * 8;
        LC2IS_CUDA(launch_pdl(k1b_dt_finish_kernel, (unsigned)blocks, 256, 0, st, d_dtraw, d_rt,
                              (const __nv_bfloat16*)d_t_hat, d_inv_norm_t, d_grad_scale, n_sets, C, C_pad, D, normalize,
                              logit_scale, d_grad_t));
        LC2IS_CHECK_LAUNCH("k1b_dt_finish_kernel");
    }
    return 0;
}

extern "C" int lc2is_cosine_logits_bwd(const void* d_grad_logits, int g_dtype, const float* d_logits,
                                       const void* d_v_hat, const float* d_inv_norm_v,
                                       const void* d_t_hat, const float* d_inv_norm_t,
                                       int B, int hw, int D, int n_sets, int C,
                                       int normalize, float logit_scale, const float* d_grad_scale,
                                       void* d_grad_v, int gv_dtype, float* d_grad_t,
                                       void* d_ws, lc2is_stream_t stream) {
    return lc2is_cosine_logits_bwd_ex(d_grad_logits, g_dtype, d_logits, d_v_hat, d_inv_norm_v, d_t_hat, d_inv_norm_t, B, hw,
                                      D, n_sets, C, normalize, logit_scale, d_grad_scale, d_grad_v, gv_dtype, d_grad_t,
                                      d_ws, stream, 0);
}

// ---------------------------------------------------------------------------------------------
// TextToPatch.visual backward (autograd of model/text_patch.py:12,17; y = x W^T + b):
//   gx [M,K]  = gy [M,N] . W [N,K]       lc2is_linear_fwd's tcgen05 pipeline on the transposed weight (workspace)
//   gw [N,K] += gy^T . x                  tcgen05 split-K over the rows, both operands MN-major; each slice stored to the
//                                         workspace, reduce_partials_kernel adds the slices to gw
//   gb [N]   += column sums of gy
constexpr int LINEAR_BWD_MAX_COLSUM_CTAS = 1024;            // per-CTA partial column sums of gy (workspace bound)
constexpr int LINEAR_BWD_MAX_SLICES = 32;                  // split-K slices of the weight gradient (workspace bound)
extern "C" int64_t lc2is_linear_bwd_workspace(int N, int K) {
    // the transposed bf16 weight (gx) + LINEAR_BWD_MAX_SLICES fp32 partial weight gradients (gw)
    return ((int64_t)N * K * 2 + 255) / 256 * 256 + (int64_t)LINEAR_BWD_MAX_SLICES * N * K * 4 +
           (int64_t)LINEAR_BWD_MAX_COLSUM_CTAS * N * 4;
}

extern "C" int lc2is_linear_bwd(const void* d_gy_bf16, const void* d_x_bf16, const void* d_w_bf16, long long M, int N,
                                int K, void* d_gx, int gx_dtype, float* d_gw, float* d_gb, void* d_ws,
                                lc2is_stream_t stream) {
    if (int e = ensure_device()) return e;
    if (M < 0 || N <= 0 || K <= 0) return fail(LC2IS_ERR_SHAPE, "bad shape%s");
    if (N % 64 || K % 64) return fail(LC2IS_ERR_SHAPE, "N and K must be multiples of 64%s");
    if (M > 0x7fffffffLL / 2) return fail(LC2IS_ERR_SHAPE, "M too large%s");
    if (!d_gy_bf16) return fail(LC2IS_ERR_ARG, "null pointer%s");
    // every argument is checked before the first launch, so that a rejected call leaves all outputs untouched
    if (d_gx && (!d_w_bf16 || !d_ws)) return fail(LC2IS_ERR_ARG, "gx needs the weight and the workspace%s");
    if (d_gx && gx_dtype != LC2IS_F32 && gx_dtype != LC2IS_BF16) return fail(LC2IS_ERR_ARG, "gx_dtype%s");
    if (d_gw && (!d_x_bf16 || !d_ws)) return fail(LC2IS_ERR_ARG, "gw needs x and the workspace%s");
    if (d_gb && !d_ws) return fail(LC2IS_ERR_ARG, "gb needs the workspace%s");
    // gy, x and the workspace are TMA bases and read with 16-byte vectors (colsum_bf16_kernel, reduce_partials_kernel),
    // gx is written by lc2is_linear_fwd's vector epilogue and gw read and written as float4; gb is accessed per element
    if (((uintptr_t)d_gy_bf16 | (uintptr_t)d_x_bf16 | (uintptr_t)d_gx | (uintptr_t)d_gw | (uintptr_t)d_ws) % 16)
        return fail(LC2IS_ERR_ARG, "gy, x, gx, gw and the workspace must be 16-byte aligned%s");
    if (M == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    if (d_gx) {
        dim3 grid((K + 31) / 32, (N + 31) / 32);
        transpose_bf16_kernel<<<grid, 256, 0, st>>>((const __nv_bfloat16*)d_w_bf16, N, K, (__nv_bfloat16*)d_ws);
        LC2IS_CHECK_LAUNCH("transpose_bf16_kernel");
        // gx[m][k] = sum_n gy[m][n] Wt[k][n]: "x" = gy (inner size N), "W" = Wt [K out][N in]
        if (int e = lc2is_linear_fwd(d_gy_bf16, d_ws, nullptr, M, K, N, d_gx, gx_dtype, stream)) return e;
    }
    if (d_gw) {
        // out[n][k] += sum_m gy[m][n] x[m][k]: A = x (M side = the K input features, 256 per CTA), B = gy (N side);
        // every CTA stores its partial tile into slice ks of the workspace, reduce_partials_kernel adds the slices to gw
        DtParams P;
        float* part = reinterpret_cast<float*>(static_cast<uint8_t*>(d_ws) + ((size_t)N * K * 2 + 255) / 256 * 256);
        P.dt_raw = part; P.B = 1; P.hw = (int)M; P.D = K; P.C = N; P.C_pad = N; P.n_sets = 1;
        P.NB = N % 256 == 0 ? 256 : (N % 128 == 0 ? 128 : 64);
        P.n_ntiles = N / P.NB;
        P.n_dtiles = (K + 2 * DT_BM - 1) / (2 * DT_BM);
        P.kb_per_img = (int)((M + DT_KB - 1) / DT_KB);
        const int base_items = P.n_dtiles * P.n_ntiles;
        int ksplit = sm_count() / base_items;
        if (ksplit < 1) ksplit = 1;
        if (ksplit > P.kb_per_img) ksplit = P.kb_per_img;
        if (ksplit > LINEAR_BWD_MAX_SLICES) ksplit = LINEAR_BWD_MAX_SLICES;
        P.ksplit = ksplit;
        const int stage_bytes = 2 * DT_A_BYTES + P.NB * 128;
        int stages = (200 * 1024) / stage_bytes;
        if (stages > DT_MAX_STAGES) stages = DT_MAX_STAGES;
        P.stages = stages;
        CUtensorMap tmX, tmGy;
        if (int e = make_tmap_2d_bf16(&tmX, d_x_bf16, (uint64_t)M, K, DT_KB, 64)) return e;
        if (int e = make_tmap_2d_bf16(&tmGy, d_gy_bf16, (uint64_t)M, N, DT_KB, 64)) return e;
        size_t smem = (size_t)stages * stage_bytes + 1024 + 256;
        if (smem < 120 * 1024) smem = 120 * 1024;
        LC2IS_CUDA(cudaFuncSetAttribute(k1b_dt_kernel<true, 2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k1b_dt_kernel<true, 2, true><<<base_items * ksplit, KB_THREADS, smem, st>>>(tmX, tmGy, P);
        LC2IS_CHECK_LAUNCH("k1b_dt_kernel<linear dW>");
        const long long n4 = (long long)N * K / 4;
        long long blocks = (n4 + 255) / 256;
        if (blocks > sm_count() * 8) blocks = sm_count() * 8;
        reduce_partials_kernel<<<(unsigned)blocks, 256, 0, st>>>(reinterpret_cast<const float4*>(part), ksplit, n4,
                                                                 reinterpret_cast<float4*>(d_gw));
        LC2IS_CHECK_LAUNCH("reduce_partials_kernel");
    }
    if (d_gb) {
        float* cpart = reinterpret_cast<float*>(static_cast<uint8_t*>(d_ws) + ((size_t)N * K * 2 + 255) / 256 * 256 +
                                                (size_t)LINEAR_BWD_MAX_SLICES * N * K * 4);
        long long blocks = (M + 255) / 256;
        if (blocks > sm_count() * 2) blocks = sm_count() * 2;
        if (blocks > LINEAR_BWD_MAX_COLSUM_CTAS) blocks = LINEAR_BWD_MAX_COLSUM_CTAS;
        colsum_bf16_kernel<<<(unsigned)blocks, CS_THREADS, 0, st>>>((const __nv_bfloat16*)d_gy_bf16, M, N, cpart);
        LC2IS_CHECK_LAUNCH("colsum_bf16_kernel");
        colsum_finish_kernel<<<(N + 31) / 32, 256, 0, st>>>(cpart, (int)blocks, N, d_gb);
        LC2IS_CHECK_LAUNCH("colsum_finish_kernel");
    }
    return 0;
}
