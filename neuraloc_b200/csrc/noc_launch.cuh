// noc_launch.cuh — host-side launch plumbing shared by the kernel units and noc_api.cu: the forward rollout request
// (RolloutCall), stream-ordered scratch (ScratchBuf), and the launch of one tile configuration.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <cstring>

#include "../../include/noc_b200.h"
#include "noc_rollout.cuh"

namespace noc {

int fail(int code, const char* fmt, ...);      // sets noc_last_error(), returns code   (noc_api.cu)
void count_launch();                            // kernel-launch counter                 (noc_api.cu)
int sm_count();                                 // SMs of the current device             (noc_api.cu)
int launch_finish(const double* partials, int nblocks, double* out, cudaStream_t st);   // (noc_api.cu)
int big_reserve(size_t bytes);                  // large per-call buffers: their own per-device pool, threshold follows the call (noc_api.cu)
int big_alloc(void** p, size_t bytes, cudaStream_t st);   // cudaError_t as int; freed with cudaFreeAsync

#define NOC_CUDA(expr)                                                                               \
    do {                                                                                             \
        cudaError_t e__ = (expr);                                                                    \
        if (e__ != cudaSuccess)                                                                      \
            return fail(NOC_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
    } while (0)

// stream-ordered scratch that is returned to its pool on every exit path (error returns included); free() releases it early
// and reports the error, for success paths that check the free
struct ScratchBuf {
    void* p = nullptr;
    cudaStream_t st = nullptr;
    ScratchBuf() = default;
    ScratchBuf(const ScratchBuf&) = delete;
    ScratchBuf& operator=(const ScratchBuf&) = delete;
    cudaError_t alloc(size_t bytes, cudaStream_t s) { return kept(cudaMallocAsync(&p, bytes ? bytes : 1, s), s); }
    cudaError_t alloc_big(size_t bytes, cudaStream_t s) { return kept((cudaError_t)big_alloc(&p, bytes, s), s); }   // big_reserve pool
    cudaError_t free() {
        void* q = p;
        p = nullptr;
        return q ? cudaFreeAsync(q, st) : cudaSuccess;
    }
    template <typename T> T* as() const { return static_cast<T*>(p); }
    ~ScratchBuf() { free(); }

  private:
    cudaError_t kept(cudaError_t e, cudaStream_t s) {      // a failed allocation holds nothing
        st = s;
        if (e != cudaSuccess) p = nullptr;
        return e;
    }
};

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
static inline int align_up(int a, int b) { return ceil_div(a, b) * b; }

// tile configurations (see Cfg in noc_rollout.cuh)
//                      real   RO RS WO NWO NWS wsmem
using CfgF_S4 = Cfg<float, 4, 4, 4, 1, 4, true>;    // id 0, m <= 16 : warp-private tiles of 128 samples
using CfgF_S8 = Cfg<float, 8, 4, 4, 1, 4, true>;    // id 1, m <= 64 : warp-private tiles of 128 samples
using CfgF_M = Cfg<float, 8, 8, 8, 2, 4, false>;    // id 2, m <= 128: 128 samples, 2 warps across outputs, streamed weights
using CfgF_L = Cfg<float, 8, 8, 8, 8, 1, false>;    // id 3, m <= 512: 32 samples, 8 warps across outputs, streamed weights
using CfgD_S8 = Cfg<double, 8, 4, 4, 1, 4, true>;   // id 4
using CfgD_M = Cfg<double, 8, 4, 8, 2, 4, false>;   // id 5
using CfgD_L = Cfg<double, 8, 4, 8, 8, 1, false>;   // id 6
using CfgF_S8Z = Cfg<float, 8, 4, 4, 1, 15, true, true>;   // id 7, m <= 64: one 15-warp CTA per SM, warp-private tiles, state in global scratch
using CfgF_S4Z = Cfg<float, 4, 4, 4, 1, 15, true, true>;   // id 8, m <= 16: same

// One forward rollout request (noc_ocflow), validated by the caller; every forward launcher takes it.
template <typename real>
struct RolloutCall {
    int d, m, nTh, r;
    real h;                         // ResNet step, rounded to real
    PhiRaw<real> raw;               // value-network tensors, reference layout (device)
    ProbPack prob;
    const real* x;                  // [n, d] (device)
    long long n;
    const double* host_times;       // stage-time table [nt * 5] (noc_stage_times) on the host ...
    const double* times;            // ... and on the device
    int nt, stepper, mode;
    const double* alph;             // [6] (host)
    double t_end;
    double* out_sums;               // mean: [8] (device), else NULL
    real* out_nomean;               // noMean: [n, 8], else NULL
    real* zFull;                    // intermediates: [n, d + 4, nt + 1], else NULL
    real* ctrlFull;                 // intermediates: [n, nctrl, nt + 1], else NULL
    int smem_limit;                 // opt-in shared memory per block of the device
    cudaStream_t stream;
};

// the fields every kernel argument struct has under these names
template <class Args, typename real>
void copy_common(Args& A, const RolloutCall<real>& c) {
    A.prob = c.prob; A.x = c.x; A.n = c.n; A.nt = c.nt; A.mode = c.mode;
    A.alph0 = (real)c.alph[0]; A.alph3 = (real)c.alph[3]; A.alph4 = (real)c.alph[4]; A.alph5 = (real)c.alph[5];
    A.out_a = c.out_nomean; A.out_b = c.zFull; A.out_c = c.ctrlFull;
}

// small-batch path (noc_vec.cu): one CTA per sample, one thread per hidden unit
template <typename real>
int vec_rollout(const RolloutCall<real>& c);

// deployment-latency path (noc_lat.cu): one thread-block cluster per sample, weights resident in distributed shared memory.
// *took = false: not applicable (nTh != 2, slices do not fit, clusters unavailable) -> use vec_rollout.
template <typename real>
int lat_rollout(const RolloutCall<real>& c, bool* took);

// training step (noc_grad.cu): rollout + discrete adjoint, tiles of 4 or 8 samples per CTA
template <typename real>
int grad_rollout(int d, int m, int r, double h, const PhiRaw<real>& raw, const ProbPack& pr, const real* x, long long n,
                 const double* dtimes, int nt, const double* alph, double t_end, double* out_sums, real* grad, real* grad_x,
                 int smem_limit, cudaStream_t st);

// reverse-mode product of Phi and grad Phi (noc_grad.cu, the training kernel's terminal-block sweeps on one evaluation per row)
template <typename real>
int phi_vjp(int d, int m, int r, double h, const PhiRaw<real>& raw, const real* s, long long n, const real* seed_phi,
            const real* seed_grad, real* grad, real* grad_s, int smem_limit, cudaStream_t st);

// baseline objective (noc_baseline.cu): one warp per sample
template <typename real>
int baseline_loss(const ProbPack& pr, const real* U, const real* z0, long long n, int d, int nt, double alphG, real* loss, real* gradU,
                  cudaStream_t st);

// one translation unit per configuration (noc_inst.cu with -DNOC_CFG_ID=k) defines these
#define NOC_DECL_LAUNCH(ID, REAL) \
    int launch_cfg_##ID(const RolloutArgs<REAL>& A, const PhiRaw<REAL>* raw, int kmode, size_t smem, cudaStream_t st, double* out_sums);
NOC_DECL_LAUNCH(0, float)
NOC_DECL_LAUNCH(1, float)
NOC_DECL_LAUNCH(2, float)
NOC_DECL_LAUNCH(3, float)
NOC_DECL_LAUNCH(4, double)
NOC_DECL_LAUNCH(5, double)
NOC_DECL_LAUNCH(6, double)
NOC_DECL_LAUNCH(7, float)
NOC_DECL_LAUNCH(8, float)

template <class C, typename real>
int launch_cfg(const RolloutArgs<real>& A0, const PhiRaw<real>* raw, int kmode, size_t smem_bytes,
                      cudaStream_t st, double* out_sums) {
    RolloutArgs<real> A = A0;
    auto kern = rollout_kernel<C, real>;
    NOC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
    int per_sm = 0;
    NOC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, C::NT, smem_bytes));
    if (per_sm < 1) return fail(NOC_ERR_NOMEM, "kernel does not fit on an SM (%zu B shared memory)", smem_bytes);
    A.ntiles = (int)((A.n + C::TS - 1) / C::TS);
    int grid = std::min(A.ntiles, per_sm * sm_count());
    if (grid < 1) grid = 1;

    ScratchBuf zscr, blob, partials;
    if (A.sp.z_global && kmode == KMODE_ROLLOUT) {
        A.zstride = 2 * (A.phi.d + 4) * C::TSP;
        NOC_CUDA(zscr.alloc(sizeof(real) * (size_t)A.zstride * grid, st));
        A.zscratch = zscr.as<real>();
    }
    if (raw) {
        NOC_CUDA(blob.alloc(sizeof(real) * (size_t)A.phi.blob_len, st));
        NOC_CUDA(cudaMemsetAsync(blob.p, 0, sizeof(real) * (size_t)A.phi.blob_len, st));
        int work = std::max(A.phi.m * A.phi.m, A.phi.m * A.phi.D);
        int pgrid = std::min(std::max(1, ceil_div(work, 256)), 4 * sm_count());
        pack_phi_kernel<C, real><<<pgrid, 256, 0, st>>>(*raw, A.phi, blob.as<real>());
        count_launch();
        A.phi.blob = blob.as<real>();
    }
    if (kmode == KMODE_ROLLOUT && A.mode == NOC_MODE_MEAN) {
        NOC_CUDA(partials.alloc(sizeof(double) * 8 * (size_t)grid, st));
        A.partials = partials.as<double>();
    }
    kern<<<grid, C::NT, smem_bytes, st>>>(A, kmode);
    count_launch();
    NOC_CUDA(cudaGetLastError());
    if (partials.p) {
        int frc = launch_finish(partials.as<double>(), grid, out_sums, st);
        if (frc) return frc;
        NOC_CUDA(partials.free());
    }
    NOC_CUDA(blob.free());
    NOC_CUDA(zscr.free());
    return NOC_OK;
}

}  // namespace noc
