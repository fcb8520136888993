// noc_api.cu — C ABI (include/noc_b200.h) over the rollout kernels.
//
// Host-side work per rollout call: validate the inputs into one RolloutCall (noc_launch.cuh), pick the kernel family
// (choose_path: tensor-core, small-batch or FMA tile kernel) and hand the call to its launcher, which packs the
// value-network weights for its kernel (a tiny kernel, stream-ordered) and launches ONE rollout kernel + a 1-block
// finishing reduction.  All scratch is stream-ordered (ScratchBuf), so calls on different streams do not interfere.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "noc_launch.cuh"
#include "noc_tc_rollout.cuh"
#include "noc_ts_rollout.cuh"

namespace noc {

static thread_local std::string g_err;
static std::atomic<long long> g_launches{0};
static thread_local int g_last_path = -1;      // NOC_PATH_* of the calling thread's last rollout

int fail(int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
void count_launch() { g_launches++; }

// out[q] = sum over CTAs of partials[cta][q], fixed order (deterministic); out[7] = sample count
static __global__ void finish_costs_kernel(const double* __restrict__ partials, int nblocks, double* __restrict__ out) {
    int q = threadIdx.x;
    if (q < 8) {
        double s = 0.0;
        for (int b = 0; b < nblocks; ++b) s += partials[b * 8 + q];
        out[q] = s;
    }
}

int launch_finish(const double* partials, int nblocks, double* out, cudaStream_t st) {
    finish_costs_kernel<<<1, 32, 0, st>>>(partials, nblocks, out);
    count_launch();
    NOC_CUDA(cudaGetLastError());
    return NOC_OK;
}

// ------------------------------------------------------------------------------------------------
// FMA peak micro-benchmark (roofline denominator, SURVEY.md H10)
// ------------------------------------------------------------------------------------------------
template <typename real>
static __global__ void __launch_bounds__(256) fma_peak_kernel(real* out, int iters, real a, real b) {
    real acc[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = real(threadIdx.x + i);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int rep = 0; rep < 8; ++rep)
#pragma unroll
            for (int i = 0; i < 16; ++i) acc[i] = r_fma(acc[i], a, b);
    }
    real s = real(0);
#pragma unroll
    for (int i = 0; i < 16; ++i) s += acc[i];
    if (s == real(123456789)) out[blockIdx.x * blockDim.x + threadIdx.x] = s;   // keeps the loop alive
}

// Inner-loop ceiling: the register-tiled outer product of the rollout's contractions (8x8 tile per thread, both
// operand vectors re-read from shared memory every k-step, no barriers, no epilogue) at a given residency.
// It separates "what the FMA pipe + register file sustain for this instruction pattern" from pipeline losses.
template <int WARPS>
static __global__ void __launch_bounds__(32 * WARPS) fma_tile_peak_kernel(float* out, int ksteps) {
    extern __shared__ __align__(16) unsigned char peak_smem[];
    float* sm = reinterpret_cast<float*>(peak_smem);
    const int tid = threadIdx.x, lane = tid & 31;
    for (int i = tid; i < 64 * 64 * 2; i += 32 * WARPS) sm[i] = 1.0f + 1e-6f * (i & 63);
    __syncthreads();
    const float* W = sm + (lane & 7) * 4;             // 8 lanes x 16-byte chunks, like ld_wrow
    const float* Ain = sm + 64 * 64 + (lane >> 3) * 8;
    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    float w[2][8], a[2][8];
    auto ldw = [&](int k, float (&v)[8]) {
        float4 t0 = *reinterpret_cast<const float4*>(W + (k & 63) * 64);
        float4 t1 = *reinterpret_cast<const float4*>(W + (k & 63) * 64 + 32);
        v[0] = t0.x; v[1] = t0.y; v[2] = t0.z; v[3] = t0.w; v[4] = t1.x; v[5] = t1.y; v[6] = t1.z; v[7] = t1.w;
    };
    auto lda = [&](int k, float (&v)[8]) {
        float4 t0 = *reinterpret_cast<const float4*>(Ain + (k & 63) * 64);
        float4 t1 = *reinterpret_cast<const float4*>(Ain + (k & 63) * 64 + 4);
        v[0] = t0.x; v[1] = t0.y; v[2] = t0.z; v[3] = t0.w; v[4] = t1.x; v[5] = t1.y; v[6] = t1.z; v[7] = t1.w;
    };
    ldw(0, w[0]); lda(0, a[0]);
    for (int k = 0; k < ksteps; k += 2) {
        ldw(k + 1, w[1]); lda(k + 1, a[1]);
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(w[0][i], a[0][j], acc[i][j]);
        ldw(k + 2, w[0]); lda(k + 2, a[0]);
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(w[1][i], a[1][j], acc[i][j]);
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) s += acc[i][j];
    if (s == 123456789.f) out[blockIdx.x * blockDim.x + tid] = s;
}

// Blackwell packed FP32: one FFMA2 instruction performs two FMAs per lane (fma.rn.f32x2, sm_100+), and accepts a scalar
// operand broadcast to both halves.  The two kernels below measure what it buys: the dependent-chain peak and the 8x8
// register-tile inner loop with sample pairs packed.
static __global__ void __launch_bounds__(256) ffma2_peak_kernel(float* out, int iters, float a, float b) {
    float2 acc[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = make_float2(float(threadIdx.x + i), float(i));
    const float2 a2 = make_float2(a, a * 1.0000001f), b2 = make_float2(b, b);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int rep = 0; rep < 8; ++rep)
#pragma unroll
            for (int i = 0; i < 16; ++i) acc[i] = __ffma2_rn(acc[i], a2, b2);
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += acc[i].x + acc[i].y;
    if (s == 123456789.f) out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

template <int WARPS>
static __global__ void __launch_bounds__(32 * WARPS) ffma2_tile_peak_kernel(float* out, int ksteps) {
    extern __shared__ __align__(16) unsigned char peak_smem[];
    float* sm = reinterpret_cast<float*>(peak_smem);
    const int tid = threadIdx.x, lane = tid & 31;
    for (int i = tid; i < 64 * 64 * 2; i += 32 * WARPS) sm[i] = 1.0f + 1e-6f * (i & 63);
    __syncthreads();
    const float* W = sm + (lane & 7) * 4;
    const float* Ain = sm + 64 * 64 + (lane >> 3) * 8;
    float2 acc[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = make_float2(0.f, 0.f);
    float w[2][8];
    float2 a[2][4];
    auto ldw = [&](int k, float (&v)[8]) {
        float4 t0 = *reinterpret_cast<const float4*>(W + (k & 63) * 64);
        float4 t1 = *reinterpret_cast<const float4*>(W + (k & 63) * 64 + 32);
        v[0] = t0.x; v[1] = t0.y; v[2] = t0.z; v[3] = t0.w; v[4] = t1.x; v[5] = t1.y; v[6] = t1.z; v[7] = t1.w;
    };
    auto lda = [&](int k, float2 (&v)[4]) {
        float4 t0 = *reinterpret_cast<const float4*>(Ain + (k & 63) * 64);
        float4 t1 = *reinterpret_cast<const float4*>(Ain + (k & 63) * 64 + 4);
        v[0] = make_float2(t0.x, t0.y); v[1] = make_float2(t0.z, t0.w); v[2] = make_float2(t1.x, t1.y); v[3] = make_float2(t1.z, t1.w);
    };
    ldw(0, w[0]); lda(0, a[0]);
    for (int k = 0; k < ksteps; k += 2) {
        ldw(k + 1, w[1]); lda(k + 1, a[1]);
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = __ffma2_rn(make_float2(w[0][i], w[0][i]), a[0][j], acc[i][j]);
        ldw(k + 2, w[0]); lda(k + 2, a[0]);
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = __ffma2_rn(make_float2(w[1][i], w[1][i]), a[1][j], acc[i][j]);
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) s += acc[i][j].x + acc[i][j].y;
    if (s == 123456789.f) out[blockIdx.x * blockDim.x + tid] = s;
}

struct CfgInfo {
    int id, PB, WB, NWO, TS, TSP, NT, TPS, GRP;
    bool wsmem, zglobal;
    size_t elt;
    const char* name;
};
template <class C>
static CfgInfo info_of(int id, const char* name) {
    return CfgInfo{id, C::PB, C::WB, C::NWO, C::TS, C::TSP, C::NT, C::TPS, C::GRP, C::WSMEM, C::ZGLOBAL, sizeof(typename C::real), name};
}
static const CfgInfo kCfgs[] = {
    info_of<CfgF_S4>(0, "f32/small4"), info_of<CfgF_S8>(1, "f32/small8"), info_of<CfgF_M>(2, "f32/mid"),
    info_of<CfgF_L>(3, "f32/large"),   info_of<CfgD_S8>(4, "f64/small8"), info_of<CfgD_M>(5, "f64/mid"),
    info_of<CfgD_L>(6, "f64/large"),   info_of<CfgF_S8Z>(7, "f32/small8z"), info_of<CfgF_S4Z>(8, "f32/small4z"),
};
static const int kNumCfgs = 9;
static inline bool cfg_is_f64(int id) { return id >= 4 && id <= 6; }

// blob layout + padded widths for configuration `ci`.  The matrices are laid out in the order one grad-Phi
// evaluation consumes them (the streamed configurations prefetch along that order).  Returns false when the
// configuration cannot hold the net (streamed configurations are single-pass: m <= PB, ceil(D/WB) <= NWO).
template <typename real>
static bool plan_blob(PhiPack<real>& P, const CfgInfo& ci) {
    if (ci.wsmem) {
        P.Npm = align_up(P.m, ci.PB);
        P.Npd = align_up(P.D, ci.PB);
        P.ntile_d = 1; P.ksplit = 1;
    } else {
        if (P.m > ci.PB) return false;
        P.Npm = ci.PB;
        P.ntile_d = ceil_div(P.D, ci.WB);
        if (P.ntile_d > ci.NWO) return false;
        P.Npd = P.ntile_d * ci.WB;
        // spare warps (NWO > ntile_d) take K-slices of the D-wide contractions
        P.ksplit = ceil_div(ci.NWO, P.ntile_d);                 // most K-slices any output tile gets
    }
    int off = 0, q = 0;
    auto take = [&](int n) { int o = off; off += align_up(n, 8); return o; };
    auto seq = [&](int o, int N, int K) { P.seq_off[q] = o; P.seq_N[q] = N; P.seq_K[q] = K; ++q; };
    for (int l = 0; l < MAXL; ++l) { P.off_Kf[l] = 0; P.off_Kr[l] = 0; P.off_b[l] = 0; }
    P.off_W1 = take(P.D * P.Npm);                  seq(P.off_W1, P.Npm, P.D);
    for (int l = 1; l < P.nTh; ++l) { P.off_Kf[l] = take(P.m * P.Npm); seq(P.off_Kf[l], P.Npm, P.m); }
    for (int l = P.nTh - 1; l >= 1; --l) { P.off_Kr[l] = take(P.m * P.Npm); seq(P.off_Kr[l], P.Npm, P.m); }
    P.off_sym = take(P.D * P.Npd);                 seq(P.off_sym, P.Npd, P.D);
    P.off_W4 = take(P.m * P.Npd);                  seq(P.off_W4, P.Npd, P.m);
    P.nseq = q;
    for (int l = 0; l < P.nTh; ++l) P.off_b[l] = take(P.m);
    P.off_w = take(P.m);
    P.off_cw = take(P.D);
    P.off_cb = take(1);
    P.blob_len = off;
    return true;
}

// shared-memory panel rows for configuration `ci`; returns bytes of dynamic shared memory (0 = does not fit)
template <typename real>
static size_t plan_smem(SmemPlan& sp, const CfgInfo& ci, const PhiPack<real>& P, int kind, int nAgents, size_t limit) {
    const int d = P.d, D = P.D, m = P.m, nTh = P.nTh;
    const int npm = P.Npm / ci.PB, npd = P.Npd / ci.PB;
    const bool inplace = ci.wsmem ? (npm == 1) : true;
    const bool aliasG = ci.wsmem ? (inplace && npd == 1) : true;
    SmemPlan best{};
    size_t best_bytes = 0;
    long best_score = -1;
    for (int zg = ci.zglobal ? 1 : 0; zg < 2; ++zg) { // zg = 1: augmented state in a global scratch (frees shared memory)
        if (zg == 1 && ci.wsmem && !ci.zglobal) break;
        int row = 0;
        auto take = [&](int n) { int o = row; row += n; return o; };
        sp.U = take(std::max(m, D));
        sp.U2 = inplace ? sp.U : take(m);
        for (int i = 0; i < MAXL; ++i) sp.T[i] = 0;
        sp.T[0] = take(std::max(m, D));
        for (int i = 1; i <= nTh - 2; ++i) sp.T[i] = take(m);
        sp.Zb = (nTh > 2) ? take(m) : 0;
        sp.S = take(D);
        sp.G = aliasG ? sp.U : take(D);
        sp.Qs = sp.T[0];
        sp.z_global = zg;
        sp.Z0 = zg ? 0 : take(d + 4);
        sp.ZA = zg ? 0 : take(d + 4);
        sp.SC = take(SC_ROWS);
        sp.RED = (ci.TPS > 1) ? take(3 * ci.TPS) : 0;
        sp.PN = take(ci.NWO);
        sp.QX = (kind == NOC_PROB_QUADCOPTER) ? take(5 * nAgents) : 0;
        // K-split partial sums: inside T[0] above the rows Qs uses when there is room (T[0] is dead by GEMM-4)
        {
            const int gp_rows = (!ci.wsmem && P.ksplit > 1) ? P.Npd : 0;      // one K-slice is exchanged per round
            if (gp_rows == 0) sp.GP = 0;
            else if (D + gp_rows <= std::max(m, D)) sp.GP = sp.T[0] + D;
            else sp.GP = take(gp_rows);
        }
        sp.rows = row;
        sp.wsm_off = align_up(row * ci.TSP, 8);
        sp.ring_slab = 0; sp.ring_ns = 0;
        size_t panel_bytes = (size_t)sp.wsm_off * ci.elt;
        if (ci.wsmem) {
            size_t bytes = panel_bytes + (size_t)P.blob_len * ci.elt;
            return bytes <= limit ? bytes : 0;
        }
        if (panel_bytes >= limit) continue;
        // warp-private rings: every warp streams its own WB columns, GRP rows per group, ns groups deep
        const size_t per_group = (size_t)(ci.NT / 32) * ci.GRP * ci.WB * ci.elt;
        int ns = (int)std::min<size_t>((limit - panel_bytes) / per_group, 8);
        if (ns < 2) continue;
        const int slab = ci.GRP * ci.WB;
        sp.ring_slab = slab; sp.ring_ns = ns;
        // prefer the deeper ring; at equal depth keep the augmented state in shared memory
        long score = (long)std::min(ns, 4) * 2 + (zg == 0 ? 1 : 0);     // 4 groups in flight cover the L2 latency
        if (score > best_score) { best_score = score; best = sp; best_bytes = panel_bytes + (size_t)ns * per_group; }
    }
    if (best_score < 0) return 0;
    sp = best;
    return best_bytes;
}

// Device facts, cached per device index (a process may drive several GPUs), filled under a mutex.
struct DevFacts { int smem_optin = -1, sm_count = 0, cc_major = 0, cc_minor = 0; };
static DevFacts g_facts[64];
static std::mutex g_facts_mu;
static thread_local int g_smem_optin = -1, g_sm_count = 0, g_cc_major = 0, g_cc_minor = 0;     // facts of the calling thread's current device
int device_facts();
int sm_count() { device_facts(); return g_sm_count; }
int device_facts() {
    int dev = 0;
    NOC_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) return fail(NOC_ERR_ARG, "device index %d out of range", dev);
    std::lock_guard<std::mutex> lock(g_facts_mu);
    DevFacts& f = g_facts[dev];
    if (f.smem_optin < 0) {
        int v = 0;
        NOC_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
        NOC_CUDA(cudaDeviceGetAttribute(&f.sm_count, cudaDevAttrMultiProcessorCount, dev));
        NOC_CUDA(cudaDeviceGetAttribute(&f.cc_major, cudaDevAttrComputeCapabilityMajor, dev));
        NOC_CUDA(cudaDeviceGetAttribute(&f.cc_minor, cudaDevAttrComputeCapabilityMinor, dev));
        // Scratch comes from the device's default stream-ordered pool on every call.  With the default release threshold (0)
        // every synchronisation returns it to the driver and 100 MB inputs are re-allocated per call; keep up to 1 GiB cached
        // (bounded: the pool is shared with the host application and sits outside PyTorch's caching allocator).
        // NOC_POOL_KEEP_MB overrides; documented in include/noc_b200.h.
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
            unsigned long long keep = 1ull << 30;
            if (const char* e = getenv("NOC_POOL_KEEP_MB")) keep = (unsigned long long)atoll(e) << 20;
            unsigned long long cur = 0;
            if (cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &cur) != cudaSuccess || cur < keep)
                cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
        f.smem_optin = v;
    }
    g_smem_optin = f.smem_optin; g_sm_count = f.sm_count; g_cc_major = f.cc_major; g_cc_minor = f.cc_minor;
    return NOC_OK;
}

// Large per-call buffers (the host entry point's device copies of x and of the outputs, the intermediates staging buffers) come
// from a pool of their own, one per device, whose release threshold follows the largest call (bounded by 1/8 of the device's
// memory; NOC_POOL_KEEP_MB, when set, is the bound instead).  In the default pool they were either above the 1 GiB threshold —
// a 2^22-sample swarm50 call (2.5 GB of input) paid the driver for its buffers on EVERY call, 6.2-6.7 s instead of 6.0 s — or cut
// up by the small scratch allocations of the calls in between, so that every few calls a 200 MB buffer had to be mapped afresh
// (sporadic +70 ms on singlequad's 0.37 s calls).
static cudaMemPool_t g_big_pool[64] = {nullptr};
static bool g_big_pool_failed[64] = {false};
int big_reserve(size_t bytes) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return (int)cudaErrorInvalidDevice;
    std::lock_guard<std::mutex> lock(g_facts_mu);
    if (!g_big_pool[dev] && !g_big_pool_failed[dev]) {
        cudaMemPoolProps props;
        memset(&props, 0, sizeof props);
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = dev;
        if (cudaMemPoolCreate(&g_big_pool[dev], &props) != cudaSuccess) { (void)cudaGetLastError(); g_big_pool[dev] = nullptr; g_big_pool_failed[dev] = true; }
    }
    cudaMemPool_t pool = g_big_pool[dev];
    if (!pool) return (int)cudaSuccess;                    // fall back to the default pool (big_alloc)
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) return (int)cudaSuccess;
    unsigned long long cap = (unsigned long long)total_b / 8, want = (unsigned long long)bytes + (64ull << 20), cur = 0;
    if (const char* e = getenv("NOC_POOL_KEEP_MB")) cap = (unsigned long long)atoll(e) << 20;
    if (want > cap) want = cap;
    if (cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &cur) == cudaSuccess && cur < want)
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &want);
    return (int)cudaSuccess;
}
int big_alloc(void** p, size_t bytes, cudaStream_t st) {
    int dev = 0;
    cudaMemPool_t pool = nullptr;
    if (cudaGetDevice(&dev) == cudaSuccess && dev >= 0 && dev < 64) {
        std::lock_guard<std::mutex> lock(g_facts_mu);
        pool = g_big_pool[dev];
    }
    return (int)(pool ? cudaMallocFromPoolAsync(p, bytes ? bytes : 1, pool, st) : cudaMallocAsync(p, bytes ? bytes : 1, st));
}

// candidate configurations in order of preference for (dtype, m); NOC_FORCE_CFG=<id> pins one (tests)
static std::vector<int> candidates(int dtype, int m) {
    const char* f = getenv("NOC_FORCE_CFG");
    if (f && *f) {
        int id = atoi(f);
        if (id >= 0 && id < kNumCfgs && (cfg_is_f64(id) == (dtype == NOC_F64))) return {id};
    }
    if (dtype == NOC_F32) {
        if (m <= 16) return {0, 8, 7, 1, 2, 3};     // measured: the 4-warp tile is faster than the 15-warp one for m = 16
        if (m <= 64) return {7, 1, 2, 3};
        if (m <= 256) return {2, 3};
        return {3};
    }
    if (m <= 64) return {4, 5, 6};
    if (m <= 256) return {5, 6};
    return {6};
}

template <typename real>
static int dispatch(int cfg_id, const RolloutArgs<real>& A, const PhiRaw<real>* raw, int kmode, size_t smem,
                    cudaStream_t st, double* out_sums);
template <>
int dispatch<float>(int cfg_id, const RolloutArgs<float>& A, const PhiRaw<float>* raw, int kmode, size_t smem,
                    cudaStream_t st, double* out_sums) {
    switch (cfg_id) {
        case 0: return launch_cfg_0(A, raw, kmode, smem, st, out_sums);
        case 1: return launch_cfg_1(A, raw, kmode, smem, st, out_sums);
        case 2: return launch_cfg_2(A, raw, kmode, smem, st, out_sums);
        case 3: return launch_cfg_3(A, raw, kmode, smem, st, out_sums);
        case 7: return launch_cfg_7(A, raw, kmode, smem, st, out_sums);
        case 8: return launch_cfg_8(A, raw, kmode, smem, st, out_sums);
    }
    return fail(NOC_ERR_ARG, "bad f32 configuration id %d", cfg_id);
}
template <>
int dispatch<double>(int cfg_id, const RolloutArgs<double>& A, const PhiRaw<double>* raw, int kmode, size_t smem,
                     cudaStream_t st, double* out_sums) {
    switch (cfg_id) {
        case 4: return launch_cfg_4(A, raw, kmode, smem, st, out_sums);
        case 5: return launch_cfg_5(A, raw, kmode, smem, st, out_sums);
        case 6: return launch_cfg_6(A, raw, kmode, smem, st, out_sums);
    }
    return fail(NOC_ERR_ARG, "bad f64 configuration id %d", cfg_id);
}

static int check_prob(const noc_prob_t* pb, int d, ProbPack& pr) {
    if (!pb) return fail(NOC_ERR_ARG, "prob is NULL");
    if (pb->kind < 0 || pb->kind > 2) return fail(NOC_ERR_ARG, "unknown problem kind %d", pb->kind);
    if (pb->obstacle < 0 || pb->obstacle > 3) return fail(NOC_ERR_ARG, "unknown obstacle %d", pb->obstacle);
    const int dims[3] = {2, 3, 12};
    if (pb->agentDim != dims[pb->kind]) return fail(NOC_ERR_ARG, "agentDim %d does not match problem kind %d", pb->agentDim, pb->kind);
    if (pb->nAgents < 1 || pb->nAgents * pb->agentDim != d)
        return fail(NOC_ERR_ARG, "nAgents (%d) * agentDim (%d) != d (%d)", pb->nAgents, pb->agentDim, d);
    if (pb->kind == NOC_PROB_CROSS2D && pb->obstacle == NOC_OBS_BLOCKS) return fail(NOC_ERR_ARG, "'blocks' is a SwarmTraj obstacle");
    if (pb->kind == NOC_PROB_SWARMTRAJ && (pb->obstacle == NOC_OBS_SOFTCORRIDOR || pb->obstacle == NOC_OBS_HARDCORRIDOR))
        return fail(NOC_ERR_ARG, "corridor obstacles are Cross2D obstacles");
    if (pb->kind == NOC_PROB_QUADCOPTER && pb->nAgents > 2 && pb->alph_W > 0.0)
        return fail(NOC_ERR_UNSUPPORTED, "Quadcopter interaction with more than two agents is broken in the reference "
                                         "(Quadcopter.py:144-155 slices the batch) and is not reproduced");
    if (!pb->xtarget) return fail(NOC_ERR_ARG, "prob.xtarget is NULL");
    pr.kind = pb->kind; pr.obstacle = pb->obstacle; pr.training = pb->training ? 1 : 0;
    pr.nAgents = pb->nAgents; pr.agentDim = pb->agentDim;
    pr.nctrl = (pb->kind == NOC_PROB_QUADCOPTER) ? 4 * pb->nAgents : d;
    pr.alph_Q = pb->alph_Q; pr.alph_W = pb->alph_W; pr.r = pb->r; pr.mass = pb->mass; pr.grav = pb->grav;
    // interaction cut-off (python double arithmetic, then rounded to the tensor dtype by the comparison)
    double cut = 2 * pb->r;
    if (pb->training && pb->kind != NOC_PROB_QUADCOPTER)
        cut = (pb->kind == NOC_PROB_SWARMTRAJ && pb->nAgents > 2) ? 3.2 * pb->r : 2.2 * pb->r;
    pr.cutW = cut;
    pr.xtarget = pb->xtarget;
    return NOC_OK;
}

template <typename real>
static int fill_phi(const noc_phi_t* ph, PhiPack<real>& P, PhiRaw<real>& R) {
    if (!ph) return fail(NOC_ERR_ARG, "phi is NULL");
    if (ph->nTh < 2) return fail(NOC_ERR_ARG, "nTh must be an integer >= 2 (src/Phi.py:25-27)");
    if (ph->nTh > MAXL) return fail(NOC_ERR_UNSUPPORTED, "nTh = %d > %d layers", ph->nTh, MAXL);
    if (ph->d < 1 || ph->m < 1 || ph->r < 1) return fail(NOC_ERR_ARG, "bad Phi dims d=%d m=%d r=%d", ph->d, ph->m, ph->r);
    if (!ph->A || !ph->c_w || !ph->c_b || !ph->w || !ph->K || !ph->b) return fail(NOC_ERR_ARG, "phi has NULL tensors");
    P.d = ph->d; P.D = ph->d + 1; P.m = ph->m; P.nTh = ph->nTh; P.r = ph->r;
    P.h = (real)((ph->h > 0.0) ? ph->h : 1.0 / (ph->nTh - 1));
    P.blob = nullptr;
    R.A = (const real*)ph->A; R.c_w = (const real*)ph->c_w; R.c_b = (const real*)ph->c_b; R.w = (const real*)ph->w;
    for (int l = 0; l < MAXL; ++l) { R.K[l] = nullptr; R.b[l] = nullptr; }
    for (int l = 0; l < ph->nTh; ++l) {
        if (!ph->K[l] || !ph->b[l]) return fail(NOC_ERR_ARG, "phi layer %d has NULL tensors", l);
        R.K[l] = (const real*)ph->K[l]; R.b[l] = (const real*)ph->b[l];
    }
    return NOC_OK;
}

// choose a configuration whose panels (+ staged weights or slab ring) fit in shared memory
template <typename real>
static int choose(RolloutArgs<real>& A, int dtype, int kind, int nAgents, int& cfg_id, size_t& smem) {
    int rc = device_facts();
    if (rc) return rc;
    for (int id : candidates(dtype, A.phi.m)) {
        const CfgInfo& ci = kCfgs[id];
        if (!plan_blob(A.phi, ci)) continue;
        smem = plan_smem(A.sp, ci, A.phi, kind, nAgents, (size_t)g_smem_optin - META_BYTES);
        if (smem > 0) { smem += META_BYTES; cfg_id = id; return NOC_OK; }
    }
    return fail(NOC_ERR_NOMEM, "Phi (d=%d, m=%d, nTh=%d) does not fit any tile configuration in %d B of shared memory",
                A.phi.d, A.phi.m, A.phi.nTh, g_smem_optin);
}

static void stage_times_host(double t0, double t1, int nt, double* tab) {
    // replays OCflow.py:25,35,47,50,53 and stepRK4's `h = t1 - t0` (:169) in IEEE double, as Python does
    volatile double h = (t1 - t0) / nt;
    volatile double tk = t0;
    for (int k = 0; k < nt; ++k) {
        volatile double ta = tk, tb = tk + h;
        volatile double hh = tb - ta;
        tk = tk + h;
        volatile double half = hh / 2;
        tab[5 * k + 0] = ta;
        tab[5 * k + 1] = ta + half;
        tab[5 * k + 2] = ta + hh;
        tab[5 * k + 3] = tk - h;
        tab[5 * k + 4] = hh;
    }
}

// ---- tensor-core path (noc_tc_rollout.cuh): fp32, nTh = 2, m <= 128, shapes instantiated in noc_tc_inst.cu
int launch_tc_0(const RolloutCall<float>&);
int launch_tc_1(const RolloutCall<float>&);
int launch_tc_2(const RolloutCall<float>&);
int launch_tc_3(const RolloutCall<float>&);
int launch_tc_4(const RolloutCall<float>&);
int launch_tc_5(const RolloutCall<float>&);
int launch_tc_6(const RolloutCall<float>&);
static int (*const kLaunchTc[])(const RolloutCall<float>&) = {launch_tc_0, launch_tc_1, launch_tc_2, launch_tc_3,
                                                               launch_tc_4, launch_tc_5, launch_tc_6};
static int tc_shape_id(const noc_phi_t* ph, const noc_prob_t* pb) {
    if (ph->nTh != 2 || ph->m < 1 || ph->m > 128) return -1;
    int shape = -1;
    if (pb->kind == NOC_PROB_QUADCOPTER && pb->nAgents == 1 && ph->d == 12) shape = 0;
    if (pb->kind == NOC_PROB_CROSS2D && pb->agentDim == 2 && ph->d == 2 * pb->nAgents) {
        if (pb->nAgents == 2) shape = 1;
        if (pb->nAgents == 4) shape = 2;
        if (pb->nAgents == 12) shape = 3;
        if (pb->nAgents == 6) shape = 4;
        if (pb->nAgents == 8) shape = 5;
        if (pb->nAgents == 10) shape = 6;
    }
    if (shape < 0) return -1;
    const int mp = align_up(ph->m, shape == 0 ? 64 : 16), KS = align_up(ph->d + 2, 16);
    if (tc_smem_bytes(mp, KS) + 1024 > (size_t)g_smem_optin) return -1;      // e.g. d = 24 with m = 128: FMA kernels
    return shape;
}

// ---- streamed tensor-core path (noc_ts_rollout.cuh): fp32, nTh = 2, the 50-agent swarm with 128 < m <= 512
int launch_ts_swarm50(const RolloutCall<float>&);
static bool ts_shape_ok(const noc_phi_t* ph, const noc_prob_t* pb) {
    return ph->nTh == 2 && pb->kind == NOC_PROB_SWARMTRAJ && pb->agentDim == 3 && pb->nAgents == 50 && ph->d == 150 && ph->m > 128 &&
           ph->m <= 512 && ts_smem_bytes_50() <= (size_t)g_smem_optin && g_cc_major == 10;
}

// The kernel family of a forward rollout (NOC_PATH_*, recorded for noc_last_path); *tc_shape is the tensor-core shape id, or
// -1 for the streamed swarm50 kernel.  Small batches (n <= NOC_VEC_MAX: 256, or 64 for swarm50, where the CTA-pair kernel is
// faster beyond that) run one CTA / cluster per sample; the tensor-core kernels take the fp32 shapes they are written for
// (NOC_TC=0 keeps the FMA kernels); everything else runs the FMA tile kernel.  NOC_FORCE_PATH=tile|vec|tc pins a path (tests).
template <typename real>
static int choose_path(const noc_phi_t* ph, const noc_prob_t* pb, long long n, int* tc_shape) {
    const bool f32 = std::is_same<real, float>::value;
    *tc_shape = f32 ? tc_shape_id(ph, pb) : -1;
    const bool ts = f32 && ts_shape_ok(ph, pb);          // never together with a tc shape (SwarmTraj vs Cross2D / Quadcopter)
    const char* vec_env = getenv("NOC_VEC_MAX");
    const char* tc_env = getenv("NOC_TC");
    const char* force = getenv("NOC_FORCE_PATH");
    const bool force_vec = force && !strcmp(force, "vec"), force_tile = force && !strcmp(force, "tile");
    const bool force_tc = force && !strcmp(force, "tc");
    const long long vec_max = vec_env ? atoll(vec_env) : (ts ? 64 : 256);
    bool use_vec = force_vec || (n <= vec_max && !force_tile);
    if (std::max(ph->m, ph->d + 4) > 1024) use_vec = false;
    bool use_tc = false;
    if (*tc_shape >= 0 || ts)
        use_tc = force_tc || (!use_vec && !(tc_env && !strcmp(tc_env, "0")) && !force_tile && !force_vec);
    g_last_path = use_tc ? NOC_PATH_TENSOR : (use_vec ? NOC_PATH_SAMPLE : NOC_PATH_TILE);
    return g_last_path;
}

// FMA tile kernel: the first configuration whose panels fit (choose), NOC_FORCE_CFG pins one
template <typename real>
static int tile_rollout(const RolloutCall<real>& c) {
    RolloutArgs<real> A;
    memset(&A, 0, sizeof A);
    A.phi.d = c.d; A.phi.D = c.d + 1; A.phi.m = c.m; A.phi.nTh = c.nTh; A.phi.r = c.r; A.phi.h = c.h;
    copy_common(A, c);
    A.stepper = c.stepper; A.times = c.times; A.t_end = (real)c.t_end;
    int cfg_id = -1;
    size_t smem = 0;
    const int dtype = std::is_same<real, float>::value ? NOC_F32 : NOC_F64;
    int rc = choose<real>(A, dtype, c.prob.kind, c.prob.nAgents, cfg_id, smem);
    if (rc) return rc;
    return dispatch<real>(cfg_id, A, &c.raw, KMODE_ROLLOUT, smem, c.stream, c.out_sums);
}

template <typename real>
static int ocflow_impl(const noc_phi_t* ph, const noc_prob_t* pb, const void* x, int64_t n, const double* stage_times,
                       double t0, double t1, int nt, int stepper, const double* alph, int mode, void* out_costs,
                       void* zFull, void* ctrlFull, cudaStream_t st) {
    RolloutCall<real> c{};
    PhiPack<real> P;
    int rc = fill_phi<real>(ph, P, c.raw);
    if (rc) return rc;
    rc = check_prob(pb, ph->d, c.prob);
    if (rc) return rc;
    if (!x || n < 1) return fail(NOC_ERR_ARG, "x is NULL or n < 1");
    if (nt < 1) return fail(NOC_ERR_ARG, "nt must be >= 1");
    if (!alph) return fail(NOC_ERR_ARG, "alph is NULL");
    if (stepper != NOC_STEP_NONE && stepper != NOC_STEP_RK1 && stepper != NOC_STEP_RK4)
        return fail(NOC_ERR_ARG, "stepper must be NOC_STEP_NONE, NOC_STEP_RK1 or NOC_STEP_RK4");
    if (mode == NOC_MODE_INTERMEDIATES) { if (!zFull || !ctrlFull) return fail(NOC_ERR_ARG, "intermediates mode needs zFull and ctrlFull"); }
    else if (mode == NOC_MODE_MEAN || mode == NOC_MODE_NOMEAN) { if (!out_costs) return fail(NOC_ERR_ARG, "out_costs is NULL"); }
    else return fail(NOC_ERR_ARG, "unknown mode %d", mode);
    rc = device_facts();
    if (rc) return rc;
    int tc_shape = -1;
    const int path = choose_path<real>(ph, pb, n, &tc_shape);

    std::vector<double> tab((size_t)nt * 5);
    if (stage_times) memcpy(tab.data(), stage_times, sizeof(double) * tab.size());
    else stage_times_host(t0, t1, nt, tab.data());
    ScratchBuf dtab;
    NOC_CUDA(dtab.alloc(sizeof(double) * tab.size(), st));
    NOC_CUDA(cudaMemcpyAsync(dtab.p, tab.data(), sizeof(double) * tab.size(), cudaMemcpyHostToDevice, st));

    c.d = ph->d; c.m = ph->m; c.nTh = ph->nTh; c.r = ph->r; c.h = P.h;
    c.x = (const real*)x; c.n = n; c.host_times = tab.data(); c.times = dtab.as<double>();
    c.nt = nt; c.stepper = stepper; c.mode = mode; c.alph = alph; c.t_end = t1;
    c.out_sums = (mode == NOC_MODE_MEAN) ? (double*)out_costs : nullptr;
    c.out_nomean = (mode == NOC_MODE_NOMEAN) ? (real*)out_costs : nullptr;
    c.zFull = (real*)zFull; c.ctrlFull = (real*)ctrlFull;
    c.smem_limit = g_smem_optin; c.stream = st;
    if (path == NOC_PATH_TENSOR) {
        if constexpr (std::is_same<real, float>::value) rc = (tc_shape >= 0) ? kLaunchTc[tc_shape](c) : launch_ts_swarm50(c);
        else rc = fail(NOC_ERR_UNSUPPORTED, "the tensor-core kernels are fp32 only");      // choose_path does not pick them
    } else if (path == NOC_PATH_SAMPLE) {
        bool took = false;
        rc = lat_rollout<real>(c, &took);
        if (rc == NOC_OK && !took) rc = vec_rollout<real>(c);
    } else
        rc = tile_rollout<real>(c);
    if (rc) return rc;
    NOC_CUDA(dtab.free());
    return NOC_OK;
}

template <typename real>
static int ocflow_host_impl(const noc_phi_t* ph, const noc_prob_t* pb, const void* xh, int64_t n, const double* stage_times,
                            double t0, double t1, int nt, int stepper, const double* alph, int mode, void* out_h,
                            void* z_h, void* c_h, cudaStream_t st) {
    if (!ph || !pb) return fail(NOC_ERR_ARG, "phi / prob is NULL");
    if (!xh || n < 1) return fail(NOC_ERR_ARG, "x is NULL or n < 1");
    const int d = ph->d;
    int nctrl = noc_ctrl_dim(pb, d);
    if (nctrl < 0) return nctrl;
    size_t xb = sizeof(real) * (size_t)n * d;
    size_t ob = (mode == NOC_MODE_MEAN) ? sizeof(double) * 8 : (mode == NOC_MODE_NOMEAN ? sizeof(real) * (size_t)n * 8 : 0);
    size_t zb = (mode == NOC_MODE_INTERMEDIATES) ? sizeof(real) * (size_t)n * (d + 4) * (nt + 1) : 0;
    size_t cb = (mode == NOC_MODE_INTERMEDIATES) ? sizeof(real) * (size_t)n * nctrl * (nt + 1) : 0;
    // Large mean / noMean batches are cut into chunks (multiples of 128 rows, so that the tiling and hence every per-sample
    // result is unchanged): chunk c+1's host->device copy runs on a second stream while chunk c's rollout runs on `st`.
    // Mean mode: one 8-double partial sum per chunk, added on the host in chunk order.  NOC_HOST_CHUNKS overrides the count.
    int nchunk = 1;
    if (mode != NOC_MODE_INTERMEDIATES) {
        nchunk = (int)std::min<long long>(8, std::max<long long>(1, n / 131072));      // >= 128 Ki rows per chunk, at most 8
        if (const char* e = getenv("NOC_HOST_CHUNKS")) nchunk = std::max(1, atoi(e));
        const long long max_chunks = (n + 127) / 128;
        if (nchunk > max_chunks) nchunk = (int)max_chunks;
        if (nchunk > 64) nchunk = 64;
    }
    const long long rows_per = (((n + nchunk - 1) / nchunk + 127) / 128) * 128;
    if (mode == NOC_MODE_MEAN) ob = sizeof(double) * 8 * (size_t)nchunk;
    big_reserve(xb + ob + zb + cb);
    int rc = NOC_OK;
    double sums_h[64 * 8];
    {
        ScratchBuf xd, od, zd, cd;                         // freed at the end of this block, before the synchronisation below
        cudaError_t e = xd.alloc_big(xb, st);
        if (e == cudaSuccess && ob) e = od.alloc_big(ob, st);
        if (e == cudaSuccess && zb) e = zd.alloc_big(zb, st);
        if (e == cudaSuccess && cb) e = cd.alloc_big(cb, st);
        if (e != cudaSuccess) {
            (void)cudaGetLastError();
            return fail(NOC_ERR_NOMEM, "device buffers for the host entry point (%zu + %zu + %zu + %zu B): %s", xb, ob, zb, cb, cudaGetErrorString(e));
        }
        if (nchunk == 1) {
            e = cudaMemcpyAsync(xd.p, xh, xb, cudaMemcpyHostToDevice, st);
            if (e != cudaSuccess) return fail(NOC_ERR_CUDA, "host->device copy failed: %s", cudaGetErrorString(e));
            rc = ocflow_impl<real>(ph, pb, xd.p, n, stage_times, t0, t1, nt, stepper, alph, mode, od.p, zd.p, cd.p, st);
        } else {
            // streams: `cs` copies; chunks alternate between `st` and `as` so that a chunk's last, partly filled wave of tiles
            // overlaps the next chunk's first wave instead of idling SMs
            cudaStream_t cs = nullptr, as = nullptr;
            cudaEvent_t ready = nullptr, joined = nullptr, copied[64] = {nullptr};
            // the two helper streams are created once per host thread and device and reused (creating and destroying them per call
            // showed up as sporadic stalls of the calling thread)
            static thread_local cudaStream_t t_cs[64] = {nullptr}, t_as[64] = {nullptr};
            int dev = 0;
            e = cudaGetDevice(&dev);
            if (e == cudaSuccess && (dev < 0 || dev >= 64)) e = cudaErrorInvalidDevice;
            if (e == cudaSuccess && !t_cs[dev]) e = cudaStreamCreateWithFlags(&t_cs[dev], cudaStreamNonBlocking);
            if (e == cudaSuccess && !t_as[dev]) e = cudaStreamCreateWithFlags(&t_as[dev], cudaStreamNonBlocking);
            if (e == cudaSuccess) { cs = t_cs[dev]; as = t_as[dev]; }
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ready, cudaEventDisableTiming);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&joined, cudaEventDisableTiming);
            if (e == cudaSuccess) e = cudaEventRecord(ready, st);                 // xd / od exist (stream-ordered allocation on st)
            if (e == cudaSuccess) e = cudaStreamWaitEvent(cs, ready, 0);
            if (e == cudaSuccess) e = cudaStreamWaitEvent(as, ready, 0);
            for (int c = 0; c < nchunk && e == cudaSuccess && rc == NOC_OK; ++c) {
                const long long r0 = (long long)c * rows_per, nr = std::min<long long>(rows_per, n - r0);
                if (nr <= 0) { nchunk = c; break; }
                const char* src = (const char*)xh + sizeof(real) * (size_t)r0 * d;
                char* dst = xd.as<char>() + sizeof(real) * (size_t)r0 * d;
                e = cudaMemcpyAsync(dst, src, sizeof(real) * (size_t)nr * d, cudaMemcpyHostToDevice, cs);
                if (e == cudaSuccess) e = cudaEventCreateWithFlags(&copied[c], cudaEventDisableTiming);
                if (e == cudaSuccess) e = cudaEventRecord(copied[c], cs);
                cudaStream_t ks = (c & 1) ? as : st;
                if (e == cudaSuccess) e = cudaStreamWaitEvent(ks, copied[c], 0);
                if (e != cudaSuccess) break;
                void* oc = (mode == NOC_MODE_MEAN) ? (void*)(od.as<double>() + 8 * c) : (void*)(od.as<real>() + 8 * (size_t)r0);
                rc = ocflow_impl<real>(ph, pb, dst, nr, stage_times, t0, t1, nt, stepper, alph, mode, oc, nullptr, nullptr, ks);
            }
            if (e == cudaSuccess && as) e = cudaEventRecord(joined, as);          // st continues after the odd chunks too
            if (e == cudaSuccess && as) e = cudaStreamWaitEvent(st, joined, 0);
            if (e != cudaSuccess && rc == NOC_OK) rc = fail(NOC_ERR_CUDA, "chunked host rollout failed: %s", cudaGetErrorString(e));
            if (cs) cudaStreamSynchronize(cs);
            if (as) cudaStreamSynchronize(as);
            for (int c = 0; c < 64; ++c) if (copied[c]) cudaEventDestroy(copied[c]);
            if (ready) cudaEventDestroy(ready);
            if (joined) cudaEventDestroy(joined);
        }
        if (rc == NOC_OK) {
            if (ob && out_h) e = cudaMemcpyAsync((mode == NOC_MODE_MEAN) ? (void*)sums_h : out_h, od.p, ob, cudaMemcpyDeviceToHost, st);
            if (e == cudaSuccess && zb && z_h) e = cudaMemcpyAsync(z_h, zd.p, zb, cudaMemcpyDeviceToHost, st);
            if (e == cudaSuccess && cb && c_h) e = cudaMemcpyAsync(c_h, cd.p, cb, cudaMemcpyDeviceToHost, st);
            if (e != cudaSuccess) rc = fail(NOC_ERR_CUDA, "device->host copy failed: %s", cudaGetErrorString(e));
        }
    }
    cudaError_t e = cudaStreamSynchronize(st);
    if (rc == NOC_OK && e != cudaSuccess) rc = fail(NOC_ERR_CUDA, "rollout failed: %s", cudaGetErrorString(e));
    if (rc == NOC_OK && mode == NOC_MODE_MEAN && out_h) {          // chunk partials -> [sums, count], fixed order
        double* o = (double*)out_h;
        for (int q = 0; q < 8; ++q) { double a = 0.0; for (int c = 0; c < nchunk; ++c) a += sums_h[8 * c + q]; o[q] = a; }
    }
    return rc;
}

template <typename real>
static int ocflow_grad_impl(const noc_phi_t* ph, const noc_prob_t* pb, const void* x, int64_t n, const double* stage_times,
                            double t0, double t1, int nt, const double* alph, void* out_costs, void* grad, void* grad_x,
                            cudaStream_t st) {
    PhiPack<real> P;
    PhiRaw<real> R;
    ProbPack pr;
    int rc = fill_phi<real>(ph, P, R);
    if (rc) return rc;
    rc = check_prob(pb, ph->d, pr);
    if (rc) return rc;
    if (ph->nTh != 2) return fail(NOC_ERR_UNSUPPORTED, "noc_ocflow_grad: nTh = %d (the adjoint is written for nTh = 2)", ph->nTh);
    if (pb->kind == NOC_PROB_QUADCOPTER && pb->nAgents != 1)
        return fail(NOC_ERR_UNSUPPORTED, "noc_ocflow_grad: Quadcopter with %d agents (one agent only)", pb->nAgents);
    if (!x || n < 1) return fail(NOC_ERR_ARG, "x is NULL or n < 1");
    if (nt < 1) return fail(NOC_ERR_ARG, "nt must be >= 1");
    if (!alph || !out_costs || !grad) return fail(NOC_ERR_ARG, "alph, out_costs or grad is NULL");
    rc = device_facts();
    if (rc) return rc;
    std::vector<double> tab((size_t)nt * 5);
    if (stage_times) memcpy(tab.data(), stage_times, sizeof(double) * tab.size());
    else stage_times_host(t0, t1, nt, tab.data());
    ScratchBuf b_tab;                                      // freed (stream-ordered) on every exit path
    NOC_CUDA(b_tab.alloc(sizeof(double) * tab.size(), st));
    NOC_CUDA(cudaMemcpyAsync(b_tab.p, tab.data(), sizeof(double) * tab.size(), cudaMemcpyHostToDevice, st));
    return grad_rollout<real>(ph->d, ph->m, ph->r, (double)P.h, R, pr, (const real*)x, n, b_tab.as<double>(), nt, alph, t1,
                              (double*)out_costs, (real*)grad, (real*)grad_x, g_smem_optin, st);
}

template <typename real>
static int phi_eval_impl(const noc_phi_t* ph, const void* s, int64_t n, void* out_phi, void* out_grad, cudaStream_t st, int dtype) {
    RolloutArgs<real> A;
    memset(&A, 0, sizeof A);
    PhiRaw<real> R;
    int rc = fill_phi<real>(ph, A.phi, R);
    if (rc) return rc;
    if (!s || n < 1) return fail(NOC_ERR_ARG, "s is NULL or n < 1");
    int cfg_id = -1;
    size_t smem = 0;
    rc = choose<real>(A, dtype, NOC_PROB_CROSS2D, 1, cfg_id, smem);
    if (rc) return rc;
    A.x = (const real*)s; A.n = n; A.nt = 0; A.mode = NOC_MODE_NOMEAN;
    A.out_a = (real*)out_phi; A.out_b = (real*)out_grad;
    return dispatch<real>(cfg_id, A, &R, KMODE_PHI, smem, st, nullptr);
}

template <typename real>
static int phi_vjp_impl(const noc_phi_t* ph, const void* s, int64_t n, const void* seed_phi, const void* seed_grad, void* grad_params,
                        void* grad_s, cudaStream_t st) {
    PhiPack<real> P;
    PhiRaw<real> R;
    int rc = fill_phi<real>(ph, P, R);
    if (rc) return rc;
    if (ph->nTh != 2) return fail(NOC_ERR_UNSUPPORTED, "noc_phi_vjp: nTh = %d (the reverse-mode product is written for nTh = 2)", ph->nTh);
    if (!s || n < 1) return fail(NOC_ERR_ARG, "s is NULL or n < 1");
    if (!grad_params && !grad_s) return NOC_OK;
    rc = device_facts();
    if (rc) return rc;
    return phi_vjp<real>(ph->d, ph->m, ph->r, (double)P.h, R, (const real*)s, n, (const real*)seed_phi, (const real*)seed_grad,
                         (real*)grad_params, (real*)grad_s, g_smem_optin, st);
}

template <typename real>
static int prob_eval_impl(const noc_prob_t* pb, const void* x, const void* p, int64_t n, int d, void* o_lhqw, void* o_g,
                          void* o_c, cudaStream_t st, int dtype) {
    RolloutArgs<real> A;
    memset(&A, 0, sizeof A);
    int rc = check_prob(pb, d, A.prob);
    if (rc) return rc;
    if (!x || !p || n < 1) return fail(NOC_ERR_ARG, "x / p is NULL or n < 1");
    A.phi.d = d; A.phi.D = d + 1; A.phi.m = 1; A.phi.nTh = 2; A.phi.r = 1; A.phi.h = (real)1;
    int cfg_id = -1;
    size_t smem = 0;
    rc = choose<real>(A, dtype, pb->kind, pb->nAgents, cfg_id, smem);
    if (rc) return rc;
    A.phi.blob_len = 0;     // no weights are staged or read in this mode
    A.x = (const real*)x; A.p_in = (const real*)p; A.n = n; A.mode = NOC_MODE_NOMEAN;
    A.out_a = (real*)o_lhqw; A.out_b = (real*)o_g; A.out_c = (real*)o_c;
    return dispatch<real>(cfg_id, A, nullptr, KMODE_PROB, smem, st, nullptr);
}

}  // namespace noc

// ---------------------------------------------------------------------------------------------------
// extern "C"
// ---------------------------------------------------------------------------------------------------
using namespace noc;

extern "C" {

int noc_version(void) { return NOC_ABI_VERSION; }
const char* noc_last_error(void) { return g_err.c_str(); }
int64_t noc_launch_count(void) { return (int64_t)g_launches.load(); }
int noc_last_path(void) { return g_last_path; }

int noc_device_info(int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor, int64_t* smem_optin_bytes) {
    int rc = device_facts();
    if (rc) return rc;
    if (sm_count) *sm_count = g_sm_count;
    if (cc_major) *cc_major = g_cc_major;
    if (cc_minor) *cc_minor = g_cc_minor;
    if (smem_optin_bytes) *smem_optin_bytes = g_smem_optin;
    return NOC_OK;
}

int noc_ctrl_dim(const noc_prob_t* prob, int32_t d) {
    if (!prob) return fail(NOC_ERR_ARG, "prob is NULL");
    if (prob->kind == NOC_PROB_QUADCOPTER) return 4 * prob->nAgents;
    if (prob->kind == NOC_PROB_CROSS2D || prob->kind == NOC_PROB_SWARMTRAJ) return d;
    return fail(NOC_ERR_ARG, "unknown problem kind %d", prob->kind);
}

int noc_stage_times(double t0, double t1, int32_t nt, double* table) {
    if (nt < 1 || !table) return fail(NOC_ERR_ARG, "nt < 1 or table is NULL");
    stage_times_host(t0, t1, nt, table);
    return NOC_OK;
}

int noc_ocflow(const noc_phi_t* phi, const noc_prob_t* prob, const void* x, int64_t n, const double* stage_times, double t0,
               double t1, int32_t nt, int32_t stepper, const double* alph, int32_t mode, int32_t dtype, void* out_costs,
               void* zFull, void* ctrlFull, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == NOC_F32)
        return ocflow_impl<float>(phi, prob, x, n, stage_times, t0, t1, nt, stepper, alph, mode, out_costs, zFull, ctrlFull, st);
    if (dtype == NOC_F64)
        return ocflow_impl<double>(phi, prob, x, n, stage_times, t0, t1, nt, stepper, alph, mode, out_costs, zFull, ctrlFull, st);
    return fail(NOC_ERR_ARG, "dtype must be NOC_F32 or NOC_F64");
}

int noc_ocflow_host(const noc_phi_t* phi, const noc_prob_t* prob, const void* x_host, int64_t n, const double* stage_times,
                    double t0, double t1, int32_t nt, int32_t stepper, const double* alph, int32_t mode, int32_t dtype,
                    void* out_costs_host, void* zFull_host, void* ctrlFull_host, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == NOC_F32)
        return ocflow_host_impl<float>(phi, prob, x_host, n, stage_times, t0, t1, nt, stepper, alph, mode, out_costs_host,
                                       zFull_host, ctrlFull_host, st);
    if (dtype == NOC_F64)
        return ocflow_host_impl<double>(phi, prob, x_host, n, stage_times, t0, t1, nt, stepper, alph, mode, out_costs_host,
                                        zFull_host, ctrlFull_host, st);
    return fail(NOC_ERR_ARG, "dtype must be NOC_F32 or NOC_F64");
}

int noc_ocflow_grad(const noc_phi_t* phi, const noc_prob_t* prob, const void* x, int64_t n, const double* stage_times, double t0,
                    double t1, int32_t nt, const double* alph, int32_t dtype, void* out_costs, void* grad, void* grad_x, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == NOC_F32) return ocflow_grad_impl<float>(phi, prob, x, n, stage_times, t0, t1, nt, alph, out_costs, grad, grad_x, st);
    if (dtype == NOC_F64) return ocflow_grad_impl<double>(phi, prob, x, n, stage_times, t0, t1, nt, alph, out_costs, grad, grad_x, st);
    return fail(NOC_ERR_ARG, "dtype must be NOC_F32 or NOC_F64");
}

int noc_baseline_loss(const noc_prob_t* prob, const void* U, const void* z0, int64_t n, int32_t d, int32_t nt, double alphG,
                      int32_t dtype, void* loss, void* gradU, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    ProbPack pr;
    int rc = check_prob(prob, d, pr);
    if (rc) return rc;
    if (!U || !z0 || !loss || n < 1 || nt < 1) return fail(NOC_ERR_ARG, "U, z0 or loss is NULL, or n < 1, or nt < 1");
    if (prob->kind == NOC_PROB_QUADCOPTER && prob->nAgents != 1)
        return fail(NOC_ERR_UNSUPPORTED, "noc_baseline_loss: Quadcopter with %d agents (baselineQuad.py handles one)", prob->nAgents);
    rc = device_facts();
    if (rc) return rc;
    if (dtype == NOC_F32) return baseline_loss<float>(pr, (const float*)U, (const float*)z0, n, d, nt, alphG, (float*)loss, (float*)gradU, st);
    if (dtype == NOC_F64) return baseline_loss<double>(pr, (const double*)U, (const double*)z0, n, d, nt, alphG, (double*)loss, (double*)gradU, st);
    return fail(NOC_ERR_ARG, "dtype must be NOC_F32 or NOC_F64");
}

int noc_phi_eval(const noc_phi_t* phi, const void* s, int64_t n, int32_t dtype, void* out_phi, void* out_grad, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == NOC_F32) return phi_eval_impl<float>(phi, s, n, out_phi, out_grad, st, dtype);
    if (dtype == NOC_F64) return phi_eval_impl<double>(phi, s, n, out_phi, out_grad, st, dtype);
    return fail(NOC_ERR_ARG, "dtype must be NOC_F32 or NOC_F64");
}

int noc_phi_vjp(const noc_phi_t* phi, const void* s, int64_t n, const void* seed_phi, const void* seed_grad, int32_t dtype,
                void* grad_params, void* grad_s, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == NOC_F32) return phi_vjp_impl<float>(phi, s, n, seed_phi, seed_grad, grad_params, grad_s, st);
    if (dtype == NOC_F64) return phi_vjp_impl<double>(phi, s, n, seed_phi, seed_grad, grad_params, grad_s, st);
    return fail(NOC_ERR_ARG, "dtype must be NOC_F32 or NOC_F64");
}

int noc_prob_eval(const noc_prob_t* prob, const void* x, const void* p, int64_t n, int32_t d, int32_t dtype, void* out_lhqw,
                  void* out_gradpH, void* out_ctrls, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == NOC_F32) return prob_eval_impl<float>(prob, x, p, n, d, out_lhqw, out_gradpH, out_ctrls, st, dtype);
    if (dtype == NOC_F64) return prob_eval_impl<double>(prob, x, p, n, d, out_lhqw, out_gradpH, out_ctrls, st, dtype);
    return fail(NOC_ERR_ARG, "dtype must be NOC_F32 or NOC_F64");
}

int noc_measure_fma_peak(int32_t dtype, double* tflops) {
    if (!tflops) return fail(NOC_ERR_ARG, "tflops is NULL");
    int rc = device_facts();
    if (rc) return rc;
    if (dtype == 4) {                    // packed FFMA2 dependent-chain peak
        const int blocks = g_sm_count * 8, threads = 256, iters = 16384;
        void* o = nullptr;
        NOC_CUDA(cudaMalloc(&o, (size_t)blocks * threads * 4));
        cudaEvent_t a0, a1;
        NOC_CUDA(cudaEventCreate(&a0));
        NOC_CUDA(cudaEventCreate(&a1));
        float bestms = 1e30f;
        for (int rep = 0; rep < 4; ++rep) {
            NOC_CUDA(cudaEventRecord(a0));
            ffma2_peak_kernel<<<blocks, threads>>>((float*)o, iters, 1.0000001f, 1e-9f);
            count_launch();
            NOC_CUDA(cudaEventRecord(a1));
            NOC_CUDA(cudaEventSynchronize(a1));
            float ms = 0;
            NOC_CUDA(cudaEventElapsedTime(&ms, a0, a1));
            if (rep > 0) bestms = std::min(bestms, ms);
        }
        *tflops = 2.0 * 2 * 16 * 8 * (double)iters * blocks * threads / (bestms * 1e-3) / 1e12;
        cudaEventDestroy(a0); cudaEventDestroy(a1); cudaFree(o);
        return NOC_OK;
    }
    if (dtype == 5 || dtype == 6) {      // 8x8 register-tile inner loop with packed FFMA2 at 8 / 16 warps per SM
        const int ksteps = 1 << 15, smem = 64 * 64 * 2 * 4;
        void* o = nullptr;
        NOC_CUDA(cudaMalloc(&o, (size_t)g_sm_count * 512 * 4));
        cudaEvent_t a0, a1;
        NOC_CUDA(cudaEventCreate(&a0));
        NOC_CUDA(cudaEventCreate(&a1));
        float bestms = 1e30f;
        for (int rep = 0; rep < 3; ++rep) {
            NOC_CUDA(cudaEventRecord(a0));
            if (dtype == 5) ffma2_tile_peak_kernel<8><<<g_sm_count, 256, smem>>>((float*)o, ksteps);
            else ffma2_tile_peak_kernel<16><<<g_sm_count, 512, smem>>>((float*)o, ksteps);
            count_launch();
            NOC_CUDA(cudaEventRecord(a1));
            NOC_CUDA(cudaEventSynchronize(a1));
            float ms = 0;
            NOC_CUDA(cudaEventElapsedTime(&ms, a0, a1));
            if (rep > 0) bestms = std::min(bestms, ms);
        }
        const double thr = (dtype == 5) ? 256.0 : 512.0;
        *tflops = 2.0 * 64 * (double)ksteps * g_sm_count * thr / (bestms * 1e-3) / 1e12;
        cudaEventDestroy(a0); cudaEventDestroy(a1); cudaFree(o);
        return NOC_OK;
    }
    if (dtype == 2 || dtype == 3) {      // inner-loop ceiling of the 8x8 register tile at 8 / 16 resident warps per SM
        const int ksteps = 1 << 15, smem = 64 * 64 * 2 * 4;
        void* o = nullptr;
        NOC_CUDA(cudaMalloc(&o, (size_t)g_sm_count * 512 * 4));
        cudaEvent_t a0, a1;
        NOC_CUDA(cudaEventCreate(&a0));
        NOC_CUDA(cudaEventCreate(&a1));
        float bestms = 1e30f;
        for (int rep = 0; rep < 3; ++rep) {
            NOC_CUDA(cudaEventRecord(a0));
            if (dtype == 2) fma_tile_peak_kernel<8><<<g_sm_count, 256, smem>>>((float*)o, ksteps);
            else fma_tile_peak_kernel<16><<<g_sm_count, 512, smem>>>((float*)o, ksteps);
            count_launch();
            NOC_CUDA(cudaEventRecord(a1));
            NOC_CUDA(cudaEventSynchronize(a1));
            float ms = 0;
            NOC_CUDA(cudaEventElapsedTime(&ms, a0, a1));
            if (rep > 0) bestms = std::min(bestms, ms);
        }
        const double thr = (dtype == 2) ? 256.0 : 512.0;
        *tflops = 2.0 * 64 * (double)ksteps * g_sm_count * thr / (bestms * 1e-3) / 1e12;
        cudaEventDestroy(a0); cudaEventDestroy(a1); cudaFree(o);
        return NOC_OK;
    }
    const int blocks = g_sm_count * 8, threads = 256, iters = (dtype == NOC_F64) ? 4096 : 16384;
    void* out = nullptr;
    NOC_CUDA(cudaMalloc(&out, (size_t)blocks * threads * 8));
    cudaEvent_t e0, e1;
    NOC_CUDA(cudaEventCreate(&e0));
    NOC_CUDA(cudaEventCreate(&e1));
    float best = 1e30f;
    for (int rep = 0; rep < 4; ++rep) {
        NOC_CUDA(cudaEventRecord(e0));
        if (dtype == NOC_F64) fma_peak_kernel<double><<<blocks, threads>>>((double*)out, iters, 1.0000001, 1e-9);
        else fma_peak_kernel<float><<<blocks, threads>>>((float*)out, iters, 1.0000001f, 1e-9f);
        count_launch();
        NOC_CUDA(cudaEventRecord(e1));
        NOC_CUDA(cudaEventSynchronize(e1));
        float ms = 0;
        NOC_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        if (rep > 0) best = std::min(best, ms);
    }
    double flops = 2.0 * 16 * 8 * (double)iters * blocks * threads;
    *tflops = flops / (best * 1e-3) / 1e12;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(out);
    return NOC_OK;
}

}  // extern "C"
