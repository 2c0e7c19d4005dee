// C-ABI glue: error text, device probing, scalar helpers and the whole-step-from-host entry.
#include "common.cuh"
#include <immintrin.h>
#include <condition_variable>
#include <deque>
#include <mutex>
#include <thread>
#include <vector>

namespace lc2is {

thread_local char g_err[512] = "";
std::atomic<long long> g_launches{0};

static int g_sm_count = 0;

int ensure_device() {
    static int state = 0;   // 0 unknown, 1 ok, -1 none
    if (state == 1) return 0;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        cudaGetLastError();
        state = -1;
        return fail(LC2IS_ERR_NODEVICE, "no CUDA device available: lc2is_b200 has no CPU fallback%s");
    }
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceProp p;
    e = cudaGetDeviceProperties(&p, dev);
    if (e != cudaSuccess) return cuda_fail(e, "cudaGetDeviceProperties");
    if (p.major != 10) {
        snprintf(g_err, sizeof(g_err), "device '%s' is sm_%d%d; this library is built for sm_100a (B200) only",
                 p.name, p.major, p.minor);
        return LC2IS_ERR_NODEVICE;
    }
    g_sm_count = p.multiProcessorCount;
    state = 1;
    return 0;
}
int sm_count() { return g_sm_count > 0 ? g_sm_count : 148; }

// scale = mult / max(n_valid, 1)   (n_valid == 0 -> scale = 0: no valid pixel, no gradient)
__global__ void mean_scale_kernel(const long long* n_valid, float mult, float* out) {
    long long n = *n_valid;
    *out = n > 0 ? mult / (float)n : 0.f;
}
// loss = loss_sum / n_valid   (0/0 -> NaN, as torch's CrossEntropyLoss('mean') with no valid target)
__global__ void finalize_loss_kernel(const double* loss_sum, const long long* n_valid, float* out) {
    *out = (float)(*loss_sum / (double)(*n_valid));
}

// both scalars of a 'mean' step in one launch (the loss sum is complete once K2 has run, the gradient scale is needed by K1b)
// Launched with launch_pdl after the CE kernel.  It lets the logits backward be scheduled at once: that kernel only runs
// its prologue before griddep_wait(), which returns after this one-thread grid has completed.
__global__ void mean_scale_finalize_kernel(const long long* n_valid, float mult, float* scale, const double* loss_sum,
                                           float* loss) {
    griddep_launch_dependents();
    griddep_wait();
    const long long n = *n_valid;
    *scale = n > 0 ? mult / (float)n : 0.f;
    *loss = (float)(*loss_sum / (double)n);
}

}  // namespace lc2is

using namespace lc2is;

extern "C" const char* lc2is_last_error(void) { return g_err; }
extern "C" int lc2is_abi_version(void) { return 5; }
extern "C" int64_t lc2is_launch_count(void) { return g_launches.load(); }

extern "C" int lc2is_mean_scale(const int64_t* d_n_valid, float mult, float* d_scale, lc2is_stream_t stream) {
    if (int e = ensure_device()) return e;
    if (!d_n_valid || !d_scale) return fail(LC2IS_ERR_ARG, "null pointer%s");
    mean_scale_kernel<<<1, 1, 0, (cudaStream_t)stream>>>((const long long*)d_n_valid, mult, d_scale);
    LC2IS_CHECK_LAUNCH("mean_scale_kernel");
    return 0;
}

extern "C" int lc2is_mean_scale_finalize(const int64_t* d_n_valid, float mult, float* d_scale, const double* d_loss_sum,
                                         float* d_loss, lc2is_stream_t stream) {
    if (int e = ensure_device()) return e;
    if (!d_n_valid || !d_scale || !d_loss_sum || !d_loss) return fail(LC2IS_ERR_ARG, "null pointer%s");
    LC2IS_CUDA(launch_pdl(mean_scale_finalize_kernel, 1, 1, 0, (cudaStream_t)stream, (const long long*)d_n_valid, mult,
                          d_scale, d_loss_sum, d_loss));
    LC2IS_CHECK_LAUNCH("mean_scale_finalize_kernel");
    return 0;
}

extern "C" int lc2is_finalize_loss(const double* d_loss_sum, const int64_t* d_n_valid, float* d_loss,
                                   lc2is_stream_t stream) {
    if (int e = ensure_device()) return e;
    if (!d_loss_sum || !d_n_valid || !d_loss) return fail(LC2IS_ERR_ARG, "null pointer%s");
    finalize_loss_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(d_loss_sum, (const long long*)d_n_valid, d_loss);
    LC2IS_CHECK_LAUNCH("finalize_loss_kernel");
    return 0;
}

// ---------------------------------------------------------------------------------------------
// Host-side label packing (the reference hands int64 label maps over in host memory: data/collator.py:91;
// 8 bytes per pixel would make the PCIe copy of the labels the longest stage of the step).  Same encoding as
// k2_labels_prepass_kernel: class id; bit 15 = label == ignore_index; 0xFFFF = outside [0,C) - or, for C <= 254, one
// byte per label (below).
namespace {
// (every variant returns the number of COUNTED labels: a class id other than ignore_index)
long long pack_labels_scalar(const int64_t* src, uint16_t* dst, size_t n, int C, int64_t ign) {
    long long cnt = 0;
    for (size_t i = 0; i < n; ++i) {
        const uint64_t v = (uint64_t)src[i];
        const bool inr = v < (uint64_t)C;
        uint16_t o = inr ? (uint16_t)v : (uint16_t)0xFFFF;
        if (inr && src[i] == ign) o |= 0x8000;
        cnt += inr && src[i] != ign;
        dst[i] = o;
    }
    return cnt;
}
__attribute__((target("avx2,popcnt")))
long long pack_labels_avx2(const int64_t* src, uint16_t* dst, size_t n, int C, int64_t ign) {
    long long cnt = 0;
    const __m256i vC = _mm256_set1_epi64x((long long)C - 1), vign = _mm256_set1_epi64x(ign);
    const __m256i zero = _mm256_setzero_si256(), ffff = _mm256_set1_epi64x(0xFFFF), flag = _mm256_set1_epi64x(0x8000);
    const __m256i idx = _mm256_setr_epi32(0, 2, 4, 6, 0, 2, 4, 6);
    const bool aligned = ((uintptr_t)dst % 16) == 0;
    size_t i = 0;
    for (; i + 16 <= n; i += 16) {
        __m128i q[4];
        for (int k = 0; k < 4; ++k) {
            const __m256i v = _mm256_loadu_si256((const __m256i*)(src + i + 4 * k));
            const __m256i bad = _mm256_or_si256(_mm256_cmpgt_epi64(zero, v), _mm256_cmpgt_epi64(v, vC));
            const __m256i isign = _mm256_cmpeq_epi64(v, vign);
            cnt += 4 - __builtin_popcount((unsigned)_mm256_movemask_pd(_mm256_castsi256_pd(_mm256_or_si256(bad, isign))));
            __m256i r = _mm256_or_si256(v, _mm256_and_si256(isign, flag));
            r = _mm256_blendv_epi8(r, ffff, bad);
            q[k] = _mm256_castsi256_si128(_mm256_permutevar8x32_epi32(r, idx));   // low 32 bits of the 4 lanes
        }
        // non-temporal stores: the buffer is read next by the GPU's copy engine, not by this core
        if (aligned) {
            _mm_stream_si128((__m128i*)(dst + i), _mm_packus_epi32(q[0], q[1]));
            _mm_stream_si128((__m128i*)(dst + i + 8), _mm_packus_epi32(q[2], q[3]));
        } else {
            _mm_storeu_si128((__m128i*)(dst + i), _mm_packus_epi32(q[0], q[1]));
            _mm_storeu_si128((__m128i*)(dst + i + 8), _mm_packus_epi32(q[2], q[3]));
        }
    }
    _mm_sfence();
    return cnt + pack_labels_scalar(src + i, dst + i, n - i, C, ign);
}
// One-byte host form for C <= 254 (half the PCIe bytes again; expanded to the 2-byte form on the device by
// lc2is_expand_labels): class id; 0xFE = label == ignore_index (a class id); 0xFF = outside [0,C).
long long pack_labels8_scalar(const int64_t* src, uint8_t* dst, size_t n, int C, int64_t ign) {
    long long cnt = 0;
    for (size_t i = 0; i < n; ++i) {
        const uint64_t v = (uint64_t)src[i];
        const bool inr = v < (uint64_t)C;
        dst[i] = !inr ? (uint8_t)0xFF : (src[i] == ign ? (uint8_t)0xFE : (uint8_t)v);
        cnt += inr && src[i] != ign;
    }
    return cnt;
}
__attribute__((target("avx2,popcnt")))
long long pack_labels8_avx2(const int64_t* src, uint8_t* dst, size_t n, int C, int64_t ign) {
    long long cnt = 0;
    const __m256i vC = _mm256_set1_epi64x((long long)C - 1), vign = _mm256_set1_epi64x(ign);
    const __m256i zero = _mm256_setzero_si256(), ff = _mm256_set1_epi64x(0xFF), fe = _mm256_set1_epi64x(0xFE);
    const __m256i idx = _mm256_setr_epi32(0, 2, 4, 6, 0, 2, 4, 6);
    const bool aligned = ((uintptr_t)dst % 16) == 0;
    size_t i = 0;
    for (; i + 16 <= n; i += 16) {
        __m128i q[4];
        for (int k = 0; k < 4; ++k) {
            const __m256i v = _mm256_loadu_si256((const __m256i*)(src + i + 4 * k));
            const __m256i bad = _mm256_or_si256(_mm256_cmpgt_epi64(zero, v), _mm256_cmpgt_epi64(v, vC));
            const __m256i isign = _mm256_cmpeq_epi64(v, vign);
            cnt += 4 - __builtin_popcount((unsigned)_mm256_movemask_pd(_mm256_castsi256_pd(_mm256_or_si256(bad, isign))));
            __m256i r = _mm256_blendv_epi8(v, fe, isign);
            r = _mm256_blendv_epi8(r, ff, bad);
            q[k] = _mm256_castsi256_si128(_mm256_permutevar8x32_epi32(r, idx));   // low 32 bits of the 4 lanes
        }
        const __m128i o = _mm_packus_epi16(_mm_packus_epi32(q[0], q[1]), _mm_packus_epi32(q[2], q[3]));
        if (aligned) _mm_stream_si128((__m128i*)(dst + i), o);       // read next by the copy engine, not by this core
        else _mm_storeu_si128((__m128i*)(dst + i), o);
    }
    _mm_sfence();
    return cnt + pack_labels8_scalar(src + i, dst + i, n - i, C, ign);
}
// AVX-512 forms: vpmovqb / vpmovqw narrow eight labels per instruction and the range / ignore tests are mask
// compares - about one instruction per label instead of three, which is what bounds a core on this path.
__attribute__((target("avx512f,avx512bw,avx512vl,popcnt")))
long long pack_labels8_avx512(const int64_t* src, uint8_t* dst, size_t n, int C, int64_t ign) {
    long long cnt = 0;
    const __m512i vC = _mm512_set1_epi64((long long)C), vign = _mm512_set1_epi64(ign);
    const __m128i fe = _mm_set1_epi8((char)0xFE), ff = _mm_set1_epi8((char)0xFF);
    const bool aligned = ((uintptr_t)dst % 16) == 0;
    size_t i = 0;
    for (; i + 16 <= n; i += 16) {
        const __m512i a = _mm512_loadu_si512((const void*)(src + i)), b = _mm512_loadu_si512((const void*)(src + i + 8));
        // unsigned v >= C: outside [0,C), negatives included
        const unsigned bad = (unsigned)_mm512_cmpge_epu64_mask(a, vC) | ((unsigned)_mm512_cmpge_epu64_mask(b, vC) << 8);
        const unsigned ig = (unsigned)_mm512_cmpeq_epi64_mask(a, vign) | ((unsigned)_mm512_cmpeq_epi64_mask(b, vign) << 8);
        __m128i o = _mm_unpacklo_epi64(_mm512_cvtepi64_epi8(a), _mm512_cvtepi64_epi8(b));
        o = _mm_mask_blend_epi8((__mmask16)ig, o, fe);
        o = _mm_mask_blend_epi8((__mmask16)bad, o, ff);
        cnt += 16 - __builtin_popcount(bad | ig);
        if (aligned) _mm_stream_si128((__m128i*)(dst + i), o);
        else _mm_storeu_si128((__m128i*)(dst + i), o);
    }
    _mm_sfence();
    return cnt + pack_labels8_scalar(src + i, dst + i, n - i, C, ign);
}
__attribute__((target("avx512f,avx512bw,avx512vl,popcnt")))
long long pack_labels_avx512(const int64_t* src, uint16_t* dst, size_t n, int C, int64_t ign) {
    long long cnt = 0;
    const __m512i vC = _mm512_set1_epi64((long long)C), vign = _mm512_set1_epi64(ign);
    const __m128i flag = _mm_set1_epi16((short)0x8000), ffff = _mm_set1_epi16((short)0xFFFF);
    const bool aligned = ((uintptr_t)dst % 16) == 0;
    size_t i = 0;
    for (; i + 8 <= n; i += 8) {
        const __m512i a = _mm512_loadu_si512((const void*)(src + i));
        const unsigned bad = (unsigned)_mm512_cmpge_epu64_mask(a, vC);
        const unsigned ig = (unsigned)_mm512_cmpeq_epi64_mask(a, vign);
        __m128i o = _mm512_cvtepi64_epi16(a);
        o = _mm_mask_blend_epi16((__mmask8)ig, o, _mm_or_si128(o, flag));
        o = _mm_mask_blend_epi16((__mmask8)bad, o, ffff);
        cnt += 8 - __builtin_popcount(bad | ig);
        if (aligned) _mm_stream_si128((__m128i*)(dst + i), o);
        else _mm_storeu_si128((__m128i*)(dst + i), o);
    }
    _mm_sfence();
    return cnt + pack_labels_scalar(src + i, dst + i, n - i, C, ign);
}
// bytes = 2: the packed uint16 form; bytes = 1: the one-byte host form
long long pack_labels_range(const int64_t* src, void* dst, size_t n, int C, int64_t ign, int bytes) {
    static const bool have_avx2 = __builtin_cpu_supports("avx2") && __builtin_cpu_supports("popcnt");
    static const bool have_avx512 = have_avx2 && __builtin_cpu_supports("avx512f") && __builtin_cpu_supports("avx512bw") &&
                                    __builtin_cpu_supports("avx512vl") && !getenv("LC2IS_NO_AVX512");
    if (have_avx512)
        return bytes == 1 ? pack_labels8_avx512(src, (uint8_t*)dst, n, C, ign)
                          : pack_labels_avx512(src, (uint16_t*)dst, n, C, ign);
    if (bytes == 1)
        return have_avx2 ? pack_labels8_avx2(src, (uint8_t*)dst, n, C, ign) : pack_labels8_scalar(src, (uint8_t*)dst, n, C, ign);
    return have_avx2 ? pack_labels_avx2(src, (uint16_t*)dst, n, C, ign) : pack_labels_scalar(src, (uint16_t*)dst, n, C, ign);
}
int host_label_bytes(int C) { return C <= 254 ? 1 : 2; }

// A small persistent worker pool (created on first use, joined at process exit).
class PackPool {
public:
    struct Task { const int64_t* src; void* dst; size_t n; int C; int64_t ign; int bytes; std::atomic<int>* pending;
                  std::atomic<long long>* counted; };
    explicit PackPool(int nthreads) {
        for (int i = 0; i < nthreads; ++i) workers_.emplace_back([this] { run(); });
    }
    ~PackPool() {
        { std::lock_guard<std::mutex> g(m_); stop_ = true; }
        cv_.notify_all();
        for (auto& t : workers_) t.join();
    }
    int size() const { return (int)workers_.size(); }
    void submit(const Task& t) {
        { std::lock_guard<std::mutex> g(m_); q_.push_back(t); }
        cv_.notify_one();
    }
private:
    void run() {
        for (;;) {
            Task t;
            {
                std::unique_lock<std::mutex> lk(m_);
                cv_.wait(lk, [this] { return stop_ || !q_.empty(); });
                if (q_.empty()) return;
                t = q_.front(); q_.pop_front();
            }
            const long long c = pack_labels_range(t.src, t.dst, t.n, t.C, t.ign, t.bytes);
            if (t.counted) t.counted->fetch_add(c, std::memory_order_relaxed);
            t.pending->fetch_sub(1, std::memory_order_release);
        }
    }
    std::vector<std::thread> workers_;
    std::mutex m_;
    std::condition_variable cv_;
    std::deque<Task> q_;
    bool stop_ = false;
};
int pack_threads_default() {
    // hardware threads shared by the ranks of this node (torchrun sets LOCAL_WORLD_SIZE), minus the
    // caller's thread and one spare; LC2IS_PACK_THREADS overrides
    int n = (int)std::thread::hardware_concurrency();
    const char* lws = getenv("LOCAL_WORLD_SIZE");
    const int ranks = lws ? atoi(lws) : 1;
    n = n / (ranks > 1 ? ranks : 1) - 2;
    n = n < 1 ? 1 : (n > 12 ? 12 : n);
    const char* e = getenv("LC2IS_PACK_THREADS");
    if (e && atoi(e) > 0) n = atoi(e) > 64 ? 64 : atoi(e);
    return n;
}
PackPool& pack_pool() {
    static PackPool pool(pack_threads_default());
    return pool;
}
// split [0,n) into pieces for the pool; *pending counts the pieces still running
void pack_submit(const int64_t* src, void* dst, size_t n, int C, int64_t ign, int bytes, std::atomic<int>* pending,
                 std::atomic<long long>* counted = nullptr) {
    PackPool& p = pack_pool();
    const int pieces = p.size();
    const size_t per = ((n + pieces - 1) / pieces + 63) / 64 * 64;
    int cnt = 0;
    for (size_t o = 0; o < n; o += per) ++cnt;
    pending->store(cnt, std::memory_order_relaxed);
    for (size_t o = 0; o < n; o += per)
        p.submit({src + o, (char*)dst + o * bytes, per < n - o ? per : n - o, C, ign, bytes, pending, counted});
}
inline void pack_wait(std::atomic<int>* pending) {
    while (pending->load(std::memory_order_acquire) > 0) _mm_pause();
}
}  // namespace

extern "C" int lc2is_pack_threads(void) { return pack_threads_default(); }
extern "C" int lc2is_host_label_bytes(int C) { return host_label_bytes(C); }

// Asynchronous form: begin returns at once (the pool packs in the background), end blocks until done.
extern "C" int lc2is_pack_labels_host_begin(const int64_t* h_labels, int64_t n, int C, int64_t ignore_index,
                                            void* h_out, void** handle) {
    if (!handle) return fail(LC2IS_ERR_ARG, "handle is NULL%s");
    if (n < 0 || C <= 0 || C >= 0x7fff) return fail(LC2IS_ERR_SHAPE, "bad n / C%s");
    if (!h_labels || !h_out) return fail(LC2IS_ERR_ARG, "null pointer%s");
    std::atomic<int>* pending = new std::atomic<int>(0);
    if (n > 0) pack_submit(h_labels, h_out, (size_t)n, C, ignore_index, host_label_bytes(C), pending);
    *handle = (void*)pending;
    return 0;
}
extern "C" int lc2is_pack_labels_host_end(void* handle) {
    if (!handle) return fail(LC2IS_ERR_ARG, "handle is NULL%s");
    std::atomic<int>* pending = (std::atomic<int>*)handle;
    pack_wait(pending);
    delete pending;
    return 0;
}

extern "C" int lc2is_pack_labels_host(const int64_t* h_labels, int64_t n, int C, int64_t ignore_index,
                                      void* h_out) {
    if (n < 0 || C <= 0 || C >= 0x7fff) return fail(LC2IS_ERR_SHAPE, "bad n / C%s");
    if (n == 0) return 0;
    if (!h_labels || !h_out) return fail(LC2IS_ERR_ARG, "null pointer%s");
    std::atomic<int> pending{0};
    pack_submit(h_labels, h_out, (size_t)n, C, ignore_index, host_label_bytes(C), &pending);
    pack_wait(&pending);
    return 0;
}

// ---------------------------------------------------------------------------------------------
// whole step from host buffers
namespace {
struct StepWs {
    size_t v_in, labels, packed, t_in, t_hat, inv_t, v_hat, inv_v, logits, grad_low, grad_v, grad_t,
        bwd_ws, confmat, scalars, total;
};
inline size_t al(size_t x) { return (x + 255) / 256 * 256; }
StepWs step_layout(int B, int hw, int D, int C, int H, int W) {
    StepWs w;
    const size_t M = (size_t)B * hw, Cp = class_pad(C);
    size_t o = 0;
    w.v_in = o;     o += al(M * D * 2);
    w.labels = o;   o += al((size_t)B * H * W * 8);
    w.packed = o;   o += al((size_t)B * H * W * 2);
    w.t_in = o;     o += al((size_t)C * D * 4);
    w.t_hat = o;    o += al(Cp * D * 2);
    w.inv_t = o;    o += al((size_t)C * 4);
    w.v_hat = o;    o += al(M * D * 2);
    w.inv_v = o;    o += al(M * 4);
    w.logits = o;   o += al(M * C * 4);
    w.grad_low = o; o += al(M * C * 4);
    w.grad_v = o;   o += al(M * D * 2);
    w.grad_t = o;   o += al((size_t)C * D * 4);
    w.bwd_ws = o;   o += al((size_t)lc2is_cosine_logits_bwd_workspace(B, hw, D, 1, C));
    w.confmat = o;  o += al((size_t)C * C * 8);
    w.scalars = o;  o += 256;     // [0] double loss_sum, [8] int64 n_valid, [16] float gscale, [20] float loss
    w.total = o;
    return w;
}
}  // namespace

extern "C" int64_t lc2is_head_step_workspace(int B, int hw, int D, int C, int H, int W) {
    return (int64_t)step_layout(B, hw, D, C, H, W).total;
}

// ---------------------------------------------------------------------------------------------
// The cross-entropy stages of a whole step (HeadStep through the lc2is_step_* entries, and head_step_enqueue).  The
// route follows from the geometry: power-of-two scales 8 / 16 run the split form of K2 (labels packed ahead, packed-label
// K2 / K3), x16 with a class count that fits it runs K2 and K3 as one kernel, other geometries the one-call K2 and the
// int64-label K3.  The split and fused routes accumulate into a zeroed d_grad_low; the one-call K2 overwrites it.
namespace {
enum CeRoute { CE_ONE_CALL, CE_SPLIT, CE_FUSED };
CeRoute ce_route(int C, int h, int w, int H, int W) {
    if (!lc2is_ce_split_supported(h, w, H, W)) return CE_ONE_CALL;
    return lc2is_ce_argmax_fused_supported(C, h, w, H, W) ? CE_FUSED : CE_SPLIT;
}

// Labels of nb images.  lb = 0: all of them int64 at d_labels.  lb = 1 / 2 (the host step's host-form labels, split
// routes only): the first np are on the device in the host form - one byte per label at d_lab8 (lb = 1) or already
// packed in d_packed (lb = 2) - and the other nb - np are int64 at d_labels + np * H * W.  n_valid += the counted
// labels, except for two-byte host labels on the fused route (the CE stage counts those: ce_stage's d_count).
int ce_labels_stage(CeRoute r, const int64_t* d_labels, const uint8_t* d_lab8, int lb, int np, int nb, int C, int h,
                    int w, int H, int W, int64_t ign, uint16_t* d_packed, int64_t* d_nvalid, float* d_glow,
                    lc2is_stream_t stream) {
    const size_t HW = (size_t)H * W;
    if (lb == 0) {
        // the fused kernel only needs the labels packed and counted (it adds the -onehot term itself); the separate
        // kernels need the label prepass (count, packing, -onehot)
        if (r == CE_FUSED) return lc2is_pack_labels(d_labels, (int64_t)nb * HW, C, ign, d_packed, d_nvalid, stream);
        if (r == CE_SPLIT)
            return lc2is_ce_labels_prepass(d_labels, nb, C, h, w, H, W, ign, d_packed, d_nvalid, d_glow, stream);
        return lc2is_count_valid(d_labels, (int64_t)nb * HW, C, ign, d_nvalid, stream);
    }
    // one-byte host labels are widened to the packed form, int64 ones packed; both count the valid pixels when nothing
    // downstream does (the fused kernel counts for two-byte host labels, the prepass otherwise)
    int64_t* cnt = (r == CE_FUSED && lb == 1) ? d_nvalid : nullptr;
    if (lb == 1 && np > 0)
        if (int e = lc2is_expand_labels(d_lab8, (int64_t)np * HW, C, ign, d_packed, cnt, stream)) return e;
    if (np < nb)
        if (int e = lc2is_pack_labels(d_labels + np * HW, (int64_t)(nb - np) * HW, C, ign, d_packed + np * HW, cnt,
                                      stream))
            return e;
    if (r == CE_SPLIT) return lc2is_ce_labels_prepass_packed(d_packed, nb, C, h, w, H, W, d_nvalid, d_glow, stream);
    return 0;
}

// K2 (+ K3 on the fused route).  d_count: n_valid for the fused kernel to add to (labels that arrived un-counted), or NULL.
int ce_stage(CeRoute r, const float* d_low, const int64_t* d_labels, const uint16_t* d_packed, int B, int C, int h,
             int w, int H, int W, int64_t ign, double* d_loss_sum, float* d_glow, int64_t* d_cm, int64_t* d_count,
             lc2is_stream_t stream) {
    if (r == CE_FUSED)
        return lc2is_ce_argmax_fused_packed(d_low, d_packed, B, C, h, w, H, W, d_loss_sum, d_glow, 1, d_count, d_cm,
                                            nullptr, nullptr, stream);
    if (r == CE_SPLIT) return lc2is_upsample_ce_packed(d_low, d_packed, B, C, h, w, H, W, d_loss_sum, d_glow, stream);
    return lc2is_upsample_ce_fwd_bwd(d_low, d_labels, B, C, h, w, H, W, ign, nullptr, d_loss_sum, d_glow, nullptr, stream);
}

// K3 where it is a kernel of its own
int argmax_stage(CeRoute r, const float* d_low, const int64_t* d_labels, const uint16_t* d_packed, int B, int C, int h,
                 int w, int H, int W, int64_t* d_cm, lc2is_stream_t stream) {
    if (r == CE_FUSED) return 0;
    if (r == CE_SPLIT)
        return lc2is_argmax_confmat_lowres_packed(d_low, B, C, h, w, H, W, d_packed, d_cm, nullptr, nullptr, stream);
    return lc2is_argmax_confmat_lowres(d_low, B, C, h, w, H, W, LC2IS_BILINEAR, d_labels, H, W, d_cm, nullptr, nullptr,
                                       stream);
}

int step_route(int C, int h, int w, int H, int W, const uint16_t* d_labels_packed, CeRoute* r) {
    if (int e = ensure_device()) return e;
    *r = ce_route(C, h, w, H, W);
    if (*r != CE_ONE_CALL && !d_labels_packed)
        return fail(LC2IS_ERR_ARG, "d_labels_packed is NULL on a split geometry (scale 8 / 16)%s");
    return 0;
}
}  // namespace

extern "C" int lc2is_step_ce_labels(const int64_t* d_labels, int B, int C, int h, int w, int H, int W,
                                    int64_t ignore_index, uint16_t* d_labels_packed, int64_t* d_n_valid,
                                    float* d_grad_low, lc2is_stream_t stream) {
    CeRoute r;
    if (int e = step_route(C, h, w, H, W, d_labels_packed, &r)) return e;
    return ce_labels_stage(r, d_labels, nullptr, 0, 0, B, C, h, w, H, W, ignore_index, d_labels_packed, d_n_valid,
                           d_grad_low, stream);
}

extern "C" int lc2is_step_ce(const float* d_low, const int64_t* d_labels, const uint16_t* d_labels_packed,
                             int B, int C, int h, int w, int H, int W, int64_t ignore_index,
                             double* d_loss_sum, float* d_grad_low, int64_t* d_confmat, lc2is_stream_t stream) {
    CeRoute r;
    if (int e = step_route(C, h, w, H, W, d_labels_packed, &r)) return e;
    return ce_stage(r, d_low, d_labels, d_labels_packed, B, C, h, w, H, W, ignore_index, d_loss_sum, d_grad_low,
                    d_confmat, nullptr, stream);
}

extern "C" int lc2is_step_argmax(const float* d_low, const int64_t* d_labels, const uint16_t* d_labels_packed,
                                 int B, int C, int h, int w, int H, int W, int64_t* d_confmat, lc2is_stream_t stream) {
    CeRoute r;
    if (int e = step_route(C, h, w, H, W, d_labels_packed, &r)) return e;
    return argmax_stage(r, d_low, d_labels, d_labels_packed, B, C, h, w, H, W, d_confmat, stream);
}

static int head_step_enqueue(const void* h_v, const float* h_t, const int64_t* h_labels,
                             int B, int h, int w, int D, int C, int H, int W,
                             int64_t ignore_index, float logit_scale, int do_backward,
                             float* h_out_loss, int64_t* h_out_n_valid, int64_t* h_out_confmat,
                             void* d_ws, lc2is_stream_t stream, lc2is_stream_t copy_stream,
                             void* h_scratch, int n_raw, int flags, bool async) {
    if (int e = ensure_device()) return e;
    if (!h_v || !h_t || (!h_labels && !h_scratch) || !h_out_loss || !h_out_n_valid || !h_out_confmat || !d_ws)
        return fail(LC2IS_ERR_ARG, "null pointer%s");
    if (B <= 0) return fail(LC2IS_ERR_SHAPE, "B must be positive%s");
    cudaStream_t st = (cudaStream_t)stream;
    cudaStream_t cst = copy_stream ? (cudaStream_t)copy_stream : st;
    const bool piped = copy_stream && copy_stream != stream;
    const int hw = h * w;
    const StepWs L = step_layout(B, hw, D, C, H, W);
    uint8_t* ws = (uint8_t*)d_ws;
    const size_t M = (size_t)B * hw;
    uint8_t* d_v = ws + L.v_in;
    int64_t* d_labels = (int64_t*)(ws + L.labels);
    float* d_t = (float*)(ws + L.t_in);
    void* d_that = ws + L.t_hat;
    float* d_invt = (float*)(ws + L.inv_t);
    uint8_t* d_vhat = ws + L.v_hat;
    float* d_invv = (float*)(ws + L.inv_v);
    float* d_logits = (float*)(ws + L.logits);
    float* d_glow = (float*)(ws + L.grad_low);
    uint16_t* d_packed = (uint16_t*)(ws + L.packed);
    double* d_loss_sum = (double*)(ws + L.scalars);
    int64_t* d_nvalid = (int64_t*)(ws + L.scalars + 8);
    float* d_gscale = (float*)(ws + L.scalars + 16);
    float* d_loss = (float*)(ws + L.scalars + 20);
    int64_t* d_cm = (int64_t*)(ws + L.confmat);
    const CeRoute route = ce_route(C, h, w, H, W);
    const bool split = route != CE_ONE_CALL;

    // The batch is cut into chunks: chunk i+1 is copied host->device on `copy_stream` while the
    // kernels of chunk i run on `stream` (engine.py:75 / :145 copy the whole batch up front).
    // Gradients are produced un-normalised (g = 1) per chunk; the 1/N_valid of the 'mean' reduction is
    // only known after the last chunk and is applied by K1b through its device-side grad_scale.
    // With a pinned scratch buffer the int64 labels are narrowed on the host (worker pool), chunk by chunk ahead of
    // the copies: 1 byte per pixel (2 for C > 254) crosses PCIe instead of 8.
    const bool hpack = split && h_scratch != nullptr && C < 0x7fff;
    // h_scratch already holds the packed labels (of the first B - n_raw images)
    const bool prepacked = h_labels == nullptr || (flags & LC2IS_STEP_LABELS_PREPACKED);
    // The LAST n_raw images' labels cross as int64 and are packed on the device while the host threads narrow the
    // others: on a host whose cores are slower at reading 8 bytes per label than PCIe is at moving them, the two
    // routes share the work (HostStep calibrates the split).
    if (n_raw < 0 || n_raw > B) return fail(LC2IS_ERR_ARG, "n_raw outside [0, B]%s");
    if (n_raw > 0 && !h_labels) return fail(LC2IS_ERR_ARG, "n_raw > 0 needs h_labels%s");
    const int Bp = hpack ? B - n_raw : 0;                   // images whose labels are packed on the host
    // host form of the packed labels: one byte per label for C <= 254 (expanded to uint16 on the device, next to the
    // copy: lc2is_expand_labels), else the uint16 form itself; 0 = no host form, every label crosses as int64
    const int lb = hpack ? host_label_bytes(C) : 0;
    uint8_t* d_lab8 = (uint8_t*)d_labels;                   // the int64 area of the workspace is free when hpack
    if (prepacked && !hpack) return fail(LC2IS_ERR_UNSUPPORTED, "pre-packed labels need a split-path geometry (scale 8 / 16)%s");
    constexpr int MAXCH = 8;
    // chunks: a blocking call overlaps copy and compute inside the step (2 chunks with packed labels, 4 with
    // int64 labels: the copy is the longest stage there); a submitted step overlaps with its neighbours and
    // runs whole-batch kernels (1 chunk)
    const int want_chunks = async ? 1 : (hpack ? 2 : 4);
    const int nchunk = piped ? (B < want_chunks ? B : want_chunks) : 1;
    const int bc = (B + nchunk - 1) / nchunk;
    std::atomic<int> pack_pending[MAXCH];
    for (int i = 0; i < MAXCH; ++i) pack_pending[i].store(0);
    if (hpack && !prepacked)
        for (int i = 0; i < nchunk; ++i) {
            const int b0 = i * bc, nb = (b0 + bc <= B ? bc : B - b0);
            const int np = nb <= 0 ? 0 : (Bp - b0 < 0 ? 0 : (Bp - b0 > nb ? nb : Bp - b0));
            if (np > 0)
                pack_submit(h_labels + (size_t)b0 * H * W, (char*)h_scratch + (size_t)b0 * H * W * lb,
                            (size_t)np * H * W, C, ignore_index, lb, &pack_pending[i]);
        }
    cudaEvent_t ev_start = nullptr, ev_copy[MAXCH] = {};
    auto cleanup = [&]() {
        if (hpack) for (int i = 0; i < nchunk; ++i) pack_wait(&pack_pending[i]);   // workers still read h_labels
        if (ev_start) cudaEventDestroy(ev_start);
        for (auto& e : ev_copy) if (e) cudaEventDestroy(e);
    };
#define STEP_CUDA(call)                                                  \
    do {                                                                 \
        cudaError_t e__ = (call);                                        \
        if (e__ != cudaSuccess) { cleanup(); return lc2is::cuda_fail(e__, #call); } \
    } while (0)
#define STEP_RC(call)                                                    \
    do {                                                                 \
        int rc__ = (call);                                               \
        if (rc__) { cleanup(); return rc__; }                            \
    } while (0)
    if (piped) {
        STEP_CUDA(cudaEventCreateWithFlags(&ev_start, cudaEventDisableTiming));
        for (int i = 0; i < nchunk; ++i) STEP_CUDA(cudaEventCreateWithFlags(&ev_copy[i], cudaEventDisableTiming));
        if (!async) {
            STEP_CUDA(cudaEventRecord(ev_start, st));           // the workspace is free once earlier work on
            STEP_CUDA(cudaStreamWaitEvent(cst, ev_start, 0));   // `stream` has drained
        }   // (a submitted step owns its workspace: the caller waited for the slot's previous step)
    }
    STEP_CUDA(cudaMemsetAsync(ws + L.scalars, 0, 256, st));
    STEP_CUDA(cudaMemsetAsync(d_cm, 0, (size_t)C * C * 8, st));
    if (split && do_backward) STEP_CUDA(cudaMemsetAsync(d_glow, 0, M * C * 4, st));
    STEP_CUDA(cudaMemcpyAsync(d_t, h_t, (size_t)C * D * 4, cudaMemcpyHostToDevice, cst));
    for (int i = 0; i < nchunk; ++i) {
        const int b0 = i * bc, nb = (b0 + bc <= B ? bc : B - b0);
        if (nb <= 0) break;
        const size_t lab_off = (size_t)b0 * H * W, v_off = (size_t)b0 * hw * D * 2;
        STEP_CUDA(cudaMemcpyAsync(d_v + v_off, (const uint8_t*)h_v + v_off, (size_t)nb * hw * D * 2,
                                  cudaMemcpyHostToDevice, cst));
        // images [b0, b0 + np) of the chunk arrive packed from the host, the other nr as int64
        const int np = hpack ? (Bp - b0 < 0 ? 0 : (Bp - b0 > nb ? nb : Bp - b0)) : 0, nr = nb - np;
        const size_t raw_off = lab_off + (size_t)np * H * W;
        if (nr > 0)                                          // (does not wait for the host threads: enqueued first)
            STEP_CUDA(cudaMemcpyAsync(d_labels + raw_off, h_labels + raw_off, (size_t)nr * H * W * 8,
                                      cudaMemcpyHostToDevice, cst));
        if (np > 0) {
            pack_wait(&pack_pending[i]);
            if (lb == 1)                                     // staged in the head of the int64 area: byte b*HW < b*HW*8
                STEP_CUDA(cudaMemcpyAsync(d_lab8 + lab_off, (const uint8_t*)h_scratch + lab_off, (size_t)np * H * W,
                                          cudaMemcpyHostToDevice, cst));
            else
                STEP_CUDA(cudaMemcpyAsync(d_packed + lab_off, (const uint16_t*)h_scratch + lab_off,
                                          (size_t)np * H * W * 2, cudaMemcpyHostToDevice, cst));
        }
        if (piped) {
            STEP_CUDA(cudaEventRecord(ev_copy[i], cst));
            STEP_CUDA(cudaStreamWaitEvent(st, ev_copy[i], 0));
        }
        float* lg = d_logits + (size_t)b0 * C * hw;
        float* gl = do_backward ? d_glow + (size_t)b0 * C * hw : nullptr;
        STEP_RC(ce_labels_stage(route, d_labels + lab_off, d_lab8 + lab_off, lb, np, nb, C, h, w, H, W, ignore_index,
                                d_packed + lab_off, d_nvalid, gl, stream));
        if (i == 0) STEP_RC(lc2is_proto_normalize(d_t, 1, C, D, 1, d_that, d_invt, stream));
        // (row normalisation inside the GEMM: no v_hat; the backward takes the raw V)
        STEP_RC(lc2is_cosine_logits_fwd(d_v + v_off, LC2IS_BF16, nb, hw, D, d_that, 1, C, 1, logit_scale,
                                        nullptr, d_invv + (size_t)b0 * hw, lg, stream));
        // (two-byte labels packed on the host arrive un-counted: the fused kernel counts them)
        STEP_RC(ce_stage(route, lg, d_labels + lab_off, d_packed + lab_off, nb, C, h, w, H, W, ignore_index, d_loss_sum,
                         gl, d_cm, lb == 2 ? d_nvalid : nullptr, stream));
        STEP_RC(argmax_stage(route, lg, d_labels + lab_off, d_packed + lab_off, nb, C, h, w, H, W, d_cm, stream));
    }
    STEP_RC(lc2is_mean_scale(d_nvalid, 1.0f, d_gscale, stream));
    if (do_backward) {
        STEP_CUDA(cudaMemsetAsync(ws + L.grad_t, 0, (size_t)C * D * 4, st));
        STEP_RC(lc2is_cosine_logits_bwd_ex(d_glow, LC2IS_F32, d_logits, d_v, d_invv, d_that, d_invt, B, hw, D, 1, C,
                                           1, logit_scale, d_gscale, ws + L.grad_v, LC2IS_BF16,
                                           (float*)(ws + L.grad_t), ws + L.bwd_ws, stream, LC2IS_BWD_RAW_V));
    }
    STEP_RC(lc2is_finalize_loss(d_loss_sum, d_nvalid, d_loss, stream));
    // D2H of the step's results (engine.py:108 .item(); :162-163)
    STEP_CUDA(cudaMemcpyAsync(h_out_loss, d_loss, 4, cudaMemcpyDeviceToHost, st));
    STEP_CUDA(cudaMemcpyAsync(h_out_n_valid, d_nvalid, 8, cudaMemcpyDeviceToHost, st));
    STEP_CUDA(cudaMemcpyAsync(h_out_confmat, d_cm, (size_t)C * C * 8, cudaMemcpyDeviceToHost, st));
    if (!async) STEP_CUDA(cudaStreamSynchronize(st));
    cleanup();
#undef STEP_CUDA
#undef STEP_RC
    return 0;
}

extern "C" int lc2is_head_step_host(const void* h_v, const float* h_t, const int64_t* h_labels,
                                    int B, int h, int w, int D, int C, int H, int W,
                                    int64_t ignore_index, float logit_scale, int do_backward,
                                    float* h_out_loss, int64_t* h_out_n_valid, int64_t* h_out_confmat,
                                    void* d_ws, lc2is_stream_t stream, lc2is_stream_t copy_stream,
                                    void* h_scratch, int n_raw, int flags) {
    return head_step_enqueue(h_v, h_t, h_labels, B, h, w, D, C, H, W, ignore_index, logit_scale, do_backward,
                             h_out_loss, h_out_n_valid, h_out_confmat, d_ws, stream, copy_stream, h_scratch, n_raw,
                             flags, false);
}

extern "C" int lc2is_head_step_host_submit(const void* h_v, const float* h_t, const int64_t* h_labels,
                                           int B, int h, int w, int D, int C, int H, int W,
                                           int64_t ignore_index, float logit_scale, int do_backward,
                                           float* h_out_loss, int64_t* h_out_n_valid, int64_t* h_out_confmat,
                                           void* d_ws, lc2is_stream_t stream, lc2is_stream_t copy_stream,
                                           void* h_scratch, int n_raw, int flags, void** done_event) {
    if (!done_event) return fail(LC2IS_ERR_ARG, "done_event is NULL%s");
    if (!copy_stream || copy_stream == stream) return fail(LC2IS_ERR_ARG, "submit needs a separate copy stream%s");
    int e = head_step_enqueue(h_v, h_t, h_labels, B, h, w, D, C, H, W, ignore_index, logit_scale, do_backward,
                              h_out_loss, h_out_n_valid, h_out_confmat, d_ws, stream, copy_stream, h_scratch, n_raw, flags, true);
    if (e) return e;
    cudaEvent_t ev;
    LC2IS_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    LC2IS_CUDA(cudaEventRecord(ev, (cudaStream_t)stream));
    *done_event = (void*)ev;
    return 0;
}

extern "C" int lc2is_head_step_host_wait(void* done_event) {
    if (!done_event) return fail(LC2IS_ERR_ARG, "done_event is NULL%s");
    cudaEvent_t ev = (cudaEvent_t)done_event;
    cudaError_t e = cudaEventSynchronize(ev);
    cudaEventDestroy(ev);
    if (e != cudaSuccess) return cuda_fail(e, "cudaEventSynchronize");
    return 0;
}
