// noc_grad.cu — the TRAINING step: closed-loop rollout + its exact discrete adjoint in ONE kernel.
//
// Replaces `Jc, cs = OCflow(x0, net, prob, tspan, nt, "rk4", alph); Jc.backward()` (trainOC.py:172-173), i.e. reverse-mode
// differentiation of src/OCflow.py:7-95 through stepRK4 (:157-184), ocOdefun (:104-140), Phi.getGrad (src/Phi.py:99-138) and
// the problems' calcLHQW / calcGradpH in their train-mode variants (Cross2D.py:108-116,139-155, SwarmTraj.py:101-119,140-156,
// Quadcopter.py:65-113).  nTh = 2 (every shipped configuration), stepper 'rk4', fp32 and fp64.
//
// Layout: a CTA owns a tile of TS samples for the whole forward + backward sweep.  Every vector of the network lives in shared
// memory as a panel [unit][TS] (sample contiguous), thread j owns output unit j of every contraction (weights K-major so that
// the lanes of a warp read consecutive addresses; staged in shared memory when the whole blob fits, else read through L1/L2),
// with TS accumulators in registers.  The forward sweep stores the four stage inputs of every RK step ([CTA][step][stage]
// [d][TS], coalesced, reused by the CTA's next tile); the backward sweep re-evaluates grad Phi at each of them and applies the hand-derived adjoint
// (tests/adjoint_ref.py restates the same formulas with torch ops and tests/test_adjoint_formulas.py checks them against
// autograd of the oracle):
//
//     o = K0 s + b0, T0 = tanh(o), u0 = act(o);  a1 = K1 u0 + b1, T1 = tanh(a1);  z1 = w + h K1'(T1*w);  v = T0*z1
//     g = K0'v + A'A s + c_w                                                                        (Phi.py:99-138)
//     psi = abar.(-grad_p H) + cL L + cH |g_t - H|   ->  gbar = d psi/d g,  xdir = d psi/d x            (problem functor)
//     odot = K0 gbar, udot = T0*odot, adot = K1 udot                                                (tangent of the net along gbar)
//     bar_a1 = h w*adot*(1-T1^2) [+ beta h T1*w];  bar_u0 = K1'bar_a1 [+ beta w];  bar_o = (1-T0^2)*odot*z1 + T0*bar_u0
//     sbar = K0'bar_o + A'A gbar [+ beta (A'A s + c_w)]
//     dK1 += (h T1*w)(x)udot + bar_a1(x)u0;  db1 += bar_a1;  dK0 += v(x)gbar + bar_o(x)s;  db0 += bar_o
//     dw += udot + h T1*adot [+ beta u1];  dA += (As)(x)gbar + (A gbar)(x)s [+ beta (As)(x)s];  dc_w += gbar [+ beta s];  dc_b += beta
//
// (the beta terms belong to the terminal block, where Phi itself enters |Phi - alpha_0 G|).  Parameter gradients of a tile are
// reduced over its TS samples in registers and added to the global gradient with one red.global.add per element and evaluation.
// The same kernel, instantiated with VJP = true, differentiates Phi.forward / Phi.getGrad alone (noc_phi_vjp): the terminal
// block's two sweeps once per row, gbar and beta read from memory.
// The L / HJt accumulators of z have constant adjoints (1 and alpha_3), Q and W are reported only (adjoint 0), so the only state
// adjoint is lambda = dJ/dx, a [d][TS] panel.
#include "noc_launch.cuh"
#include <cstdio>
#include <cstdlib>
#include "noc_adjoint.cuh"

namespace noc {

template <typename real>
struct GradPack {
    int d, D, m, r;
    real h;
    const real* blob;          // W1t | Kft | Kr | W4 | sym | b0 | b1 | w | cw | cb | A
    int blob_len;
    int off_W1t;               // [D][m]   K0 transposed:  o = K0 s
    int off_Kft;               // [m][m]   K1 transposed:  a1 = K1 u
    int off_Kr;                // [m][m]   K1 as stored:   K1' y
    int off_W4;                // [m][D]   K0 as stored:   K0' v
    int off_sym;               // [D][D]   A'A
    int off_b0, off_b1, off_w, off_cw, off_cb, off_A;
    // offsets into the gradient vector (reference state_dict order, Phi.py:77-87)
    int g_A, g_cw, g_cb, g_w, g_K0, g_b0, g_K1, g_b1, g_len;
};

template <typename real>
struct GradArgs {
    GradPack<real> phi;
    ProbPack prob;
    const real* x;
    long long n;
    int nt, ntiles;
    const double* times;       // dev [nt*5]
    real alph0, alph3, alph4, alph5, t_end;
    double* partials;          // [ntiles][8] per-tile cost sums (+ count), summed by finish_costs_kernel
    real* grad;                // [g_len] sums over the samples (atomic adds)
    real* grad_x;              // [n][d] or NULL
    real* xsave;               // [grid][nt][4][d][TS]: stage inputs of the tile a CTA is working on (L2-sized: <= 74 MB for swarm50)
    int nsplitD;               // K-slices of the D-wide contractions (K0'v, K0'bar_o)
    int use_v4, deep;          // experiment switches: vector reductions for dK1, eight weight loads in flight
    // shared-memory offsets (elements)
    int o_s, o_g, o_gb, o_q, o_sb, o_xd, o_lam, o_xbn, o_xsum, o_z0, o_za, o_sc, o_red, o_qx, o_as, o_ag, o_bt, o_vm, o_part;
    int o_T0, o_u0, o_T1, o_z1, o_od, o_ad, o_x1, o_x2, o_w;
    // Phi-VJP mode only (x is then s [n][D]): seeds on Phi and on grad Phi (NULL: zero), d psi / d s [n][D] or NULL
    const real* seed_phi;
    const real* seed_grad;
    real* grad_s;
};

template <typename real>
__global__ void pack_phi_grad_kernel(const PhiRaw<real> R, const GradPack<real> P, real* __restrict__ blob) {
    const int D = P.D, m = P.m, r = P.r;
    const int stride = gridDim.x * blockDim.x, t0 = blockIdx.x * blockDim.x + threadIdx.x;
    for (int i = t0; i < m * D; i += stride) {
        int o = i / D, k = i % D;
        real v = R.K[0][i];
        blob[P.off_W1t + k * m + o] = v;
        blob[P.off_W4 + i] = v;
    }
    for (int i = t0; i < m * m; i += stride) {
        int o = i / m, k = i % m;
        real v = R.K[1][i];
        blob[P.off_Kft + k * m + o] = v;
        blob[P.off_Kr + i] = v;
    }
    for (int i = t0; i < D * D; i += stride) {
        int k = i / D, o = i % D;
        real s = real(0);
        for (int q = 0; q < r; ++q) s = r_fma(R.A[q * D + k], R.A[q * D + o], s);
        blob[P.off_sym + i] = s;
    }
    for (int i = t0; i < m; i += stride) { blob[P.off_b0 + i] = R.b[0][i]; blob[P.off_b1 + i] = R.b[1][i]; blob[P.off_w + i] = R.w[i]; }
    for (int i = t0; i < D; i += stride) blob[P.off_cw + i] = R.c_w[i];
    for (int i = t0; i < r * D; i += stride) blob[P.off_A + i] = R.A[i];
    if (t0 == 0) blob[P.off_cb] = R.c_b[0];
}

// one panel row (TS consecutive samples) <-> registers, as 16-byte vectors
template <typename real, int TS>
__device__ __forceinline__ void ld_row(const real* p, real (&v)[TS]) {
    if constexpr (TS * sizeof(real) < 16) {                 // tiles of one or two samples (narrow nets): scalar row loads
#pragma unroll
        for (int i = 0; i < TS; ++i) v[i] = p[i];
    } else if constexpr (sizeof(real) == 4) {
#pragma unroll
        for (int i = 0; i < TS / 4; ++i) {
            float4 t = reinterpret_cast<const float4*>(p)[i];
            v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
        }
    } else {
#pragma unroll
        for (int i = 0; i < TS / 2; ++i) {
            double2 t = reinterpret_cast<const double2*>(p)[i];
            v[2 * i] = t.x; v[2 * i + 1] = t.y;
        }
    }
}

// tanh near saturation.  The adjoint needs BOTH tanh(a) and 1 - tanh(a)^2, and most hidden units of the trained nets are deep in
// saturation (|a| = 5 ... 40), where 1 - T*T from a rounded T keeps no significant digit (T within an ulp of 1 leaves
// 1 - T^2 = 4e-7 with an absolute error of 1e-7).  The panels therefore keep the signed  q = e / (1 + e),  e = exp(-2|a|):
//     tanh(a) = sign(a) (1 - 2q)        1 - tanh(a)^2 = 4 q (1 - q)        (q in [0, 1/2]: no cancellation in either)
// and are rewritten with tanh itself once the derivative has been consumed (the parameter-gradient loops read tanh).
template <typename real>
__device__ __forceinline__ void act_q(real pre, real& av, real& qs) {      // antiderivative of tanh (Phi.py:8-9) and signed q
    const real a = r_abs(pre);
    const real e = r_exp(real(-2) * a);
    av = a + r_log1pe(e);
    qs = copysign(r_div(e, real(1) + e), pre);
}
template <typename real>
__device__ __forceinline__ real q_only(real pre) {
    const real e = r_exp(real(-2) * r_abs(pre));
    return copysign(r_div(e, real(1) + e), pre);
}
template <typename real>
__device__ __forceinline__ real q_tanh(real qs) { return copysign(r_fma(real(-2), r_abs(qs), real(1)), qs); }
template <typename real>
__device__ __forceinline__ real q_dtanh(real qs) { const real q = r_abs(qs); return real(4) * q * (real(1) - q); }

template <typename real>
__device__ __forceinline__ real sgn(real v) { return real((v > real(0)) - (v < real(0))); }

template <typename real>
__device__ __forceinline__ void red_add(real* p, real v) { atomicAdd(p, v); }   // result unused: RED.E.ADD
// four consecutive floats (16-byte aligned) in one reduction: REDG.E.ADD.F32x4
__device__ __forceinline__ void red_add4(float* p, float a, float b, float c, float d) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" :: "l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// gradient sections: accumulation buffer (every section 16-byte aligned, so that rows of K1 take vector reductions) -> the
// caller's compact state_dict-order vector
struct GradSections { int src[8], dst[8], len[8]; };
template <typename real>
__global__ void unpack_grad_kernel(const real* __restrict__ acc, real* __restrict__ out, const GradSections S) {
    const int stride = gridDim.x * blockDim.x, t0 = blockIdx.x * blockDim.x + threadIdx.x;
    for (int q = 0; q < 8; ++q)
        for (int i = t0; i < S.len[q]; i += stride) out[S.dst[q] + i] = acc[S.src[q] + i];
}

// out_j[.] = sum_k W[k*N + j] in[k][.]  for the N outputs; epi(j, acc) runs in the thread that owns output j (j = tid, tid+NT, ...).
// nsplit > 1: the K range is cut into nsplit slices worked on by thread groups of NT / nsplit threads (for N << NT); the partial
// sums meet in `part` ([nsplit][N][TS]).  Every thread of the CTA must call; the caller synchronises before the outputs are read.
template <typename real, int TS, bool WSM, class Epi>
__device__ __forceinline__ void matvec(const real* __restrict__ W, int N, int K, const real* in, real* part, int nsplit,
                                       int tid, int NT, bool deep, Epi epi) {
    auto ldw = [](const real* p) -> real { if constexpr (WSM) return *p; else return __ldg(p); };
    auto dot = [&](int j, int kb, int ke, real (&acc)[TS]) {
#pragma unroll
        for (int s = 0; s < TS; ++s) acc[s] = real(0);
        const real* wp = W + j;
        int k = kb;
        // eight weight loads in flight per thread before their FMAs: a weight element is used by ONE thread (TS FMAs), so the
        // loop is bound by how many bytes the SM keeps in flight towards L2, not by the FMA pipe
        for (; deep && k + 8 <= ke; k += 8) {
            real w8[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) w8[u] = ldw(wp + (size_t)(k + u) * N);
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                real a[TS];
                ld_row<real, TS>(in + (k + u) * TS, a);
#pragma unroll
                for (int s = 0; s < TS; ++s) acc[s] = r_fma(w8[u], a[s], acc[s]);
            }
        }
        for (; k + 2 <= ke; k += 2) {
            real w0 = ldw(wp + (size_t)k * N), w1 = ldw(wp + (size_t)(k + 1) * N);
            real a[TS], b[TS];
            ld_row<real, TS>(in + k * TS, a);
            ld_row<real, TS>(in + (k + 1) * TS, b);
#pragma unroll
            for (int s = 0; s < TS; ++s) { acc[s] = r_fma(w0, a[s], acc[s]); acc[s] = r_fma(w1, b[s], acc[s]); }
        }
        if (k < ke) {
            real w0 = ldw(wp + (size_t)k * N);
            real a[TS];
            ld_row<real, TS>(in + k * TS, a);
#pragma unroll
            for (int s = 0; s < TS; ++s) acc[s] = r_fma(w0, a[s], acc[s]);
        }
    };
    if (nsplit <= 1) {
        for (int j = tid; j < N; j += NT) {
            real acc[TS];
            dot(j, 0, K, acc);
            epi(j, acc);
        }
        return;
    }
    const int G = NT / nsplit, sl = tid / G, jj = tid % G;
    if (sl < nsplit) {
        const int kb = (K * sl) / nsplit, ke = (K * (sl + 1)) / nsplit;
        for (int j = jj; j < N; j += G) {
            real acc[TS];
            dot(j, kb, ke, acc);
#pragma unroll
            for (int s = 0; s < TS; ++s) part[(sl * N + j) * TS + s] = acc[s];
        }
    }
    __syncthreads();
    for (int j = tid; j < N; j += NT) {
        real acc[TS];
#pragma unroll
        for (int s = 0; s < TS; ++s) acc[s] = part[j * TS + s];
        for (int q = 1; q < nsplit; ++q)
#pragma unroll
            for (int s = 0; s < TS; ++s) acc[s] += part[(q * N + j) * TS + s];
        epi(j, acc);
    }
}

// The m-wide contractions (N = m outputs, N even): a thread owns TWO adjacent outputs over HALF of the K range — one 8-byte
// (fp64: 16-byte) weight load and one broadcast row load feed 2 TS FMAs, i.e. half the shared-memory traffic per FMA of matvec()
// (the ncu capture of the first build showed the row loads, not the FMA pipe, as the limiter: short-scoreboard / MIO stalls).
// The upper K-half's partial sums go through `part` ([N][TS]); the lower half's threads finish and run the epilogue of both
// outputs.  Every thread of the CTA must call (block barriers inside).
template <typename real, int TS, bool WSM, class Epi>
__device__ __forceinline__ void matvec2(const real* __restrict__ W, int N, int K, const real* in, real* part, int tid, int NT,
                                        Epi epi) {
    const int G = NT >> 1, sl = tid / G, pp = tid % G, NP = N >> 1;
    const int kb = sl ? (K >> 1) : 0, ke = sl ? K : (K >> 1);
    auto ld2 = [](const real* p, real& x, real& y) {
        if constexpr (sizeof(real) == 4) {
            float2 t;
            if constexpr (WSM) t = *reinterpret_cast<const float2*>(p); else t = __ldg(reinterpret_cast<const float2*>(p));
            x = t.x; y = t.y;
        } else {
            double2 t;
            if constexpr (WSM) t = *reinterpret_cast<const double2*>(p); else t = __ldg(reinterpret_cast<const double2*>(p));
            x = t.x; y = t.y;
        }
    };
    for (int p0 = 0; p0 < NP; p0 += G) {
        const int p = p0 + pp;
        real acc0[TS], acc1[TS];
#pragma unroll
        for (int s = 0; s < TS; ++s) { acc0[s] = real(0); acc1[s] = real(0); }
        if (p < NP) {
            const real* wp = W + 2 * p;
            int k = kb;
            for (; k + 4 <= ke; k += 4) {
                real wx[4], wy[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) ld2(wp + (size_t)(k + u) * N, wx[u], wy[u]);
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    real a[TS];
                    ld_row<real, TS>(in + (k + u) * TS, a);
#pragma unroll
                    for (int s = 0; s < TS; ++s) { acc0[s] = r_fma(wx[u], a[s], acc0[s]); acc1[s] = r_fma(wy[u], a[s], acc1[s]); }
                }
            }
            for (; k < ke; ++k) {
                real wx, wy, a[TS];
                ld2(wp + (size_t)k * N, wx, wy);
                ld_row<real, TS>(in + k * TS, a);
#pragma unroll
                for (int s = 0; s < TS; ++s) { acc0[s] = r_fma(wx, a[s], acc0[s]); acc1[s] = r_fma(wy, a[s], acc1[s]); }
            }
            if (sl == 1) {
#pragma unroll
                for (int s = 0; s < TS; ++s) { part[(2 * p) * TS + s] = acc0[s]; part[(2 * p + 1) * TS + s] = acc1[s]; }
            }
        }
        __syncthreads();
        if (sl == 0 && p < NP) {
            real b0[TS], b1[TS];
            ld_row<real, TS>(part + (2 * p) * TS, b0);
            ld_row<real, TS>(part + (2 * p + 1) * TS, b1);
#pragma unroll
            for (int s = 0; s < TS; ++s) { acc0[s] += b0[s]; acc1[s] += b1[s]; }
            epi(2 * p, acc0);
            epi(2 * p + 1, acc1);
        }
        if (p0 + G < NP) __syncthreads();
    }
}

// VJP = false: the training step (forward sweep, terminal block, backward sweep of every tile).
// VJP = true:  the reverse-mode product of Phi.forward / Phi.getGrad (noc_phi_vjp) — the terminal block's two sweeps on one
//              evaluation per row s_i, with gbar = seed_grad_i and beta = seed_phi_i read from memory, so that sbar is
//              d psi_i / d s_i and the parameter reductions sum d psi_i / d theta for psi_i = a_i Phi(s_i) + B_i . grad Phi(s_i).
template <typename real, int TS, bool WSM, bool VJP>
__global__ void __launch_bounds__(512, 1) rollout_grad_kernel(const GradArgs<real> A) {
    extern __shared__ __align__(16) unsigned char grad_smem[];
    real* sm = reinterpret_cast<real*>(grad_smem);
    const int tid = threadIdx.x, NT = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = NT >> 5;
    // the problem descriptor goes to shared memory: terrain_agent() takes it by reference and is not always inlined, and the address
    // of a kernel parameter would force a local-memory copy of the whole argument struct (an L2 round trip per access)
    __shared__ ProbPack s_prob;
    if (tid == 0) s_prob = A.prob;
    const GradPack<real>& P = A.phi;
    const ProbPack& pr = s_prob;
    const int d = P.d, D = P.D, m = P.m;
    const int smp = tid % TS, part_id = tid / TS, nparts = NT / TS;        // problem phase: NT / TS threads share a sample
    real* s = sm + A.o_s;     real* g = sm + A.o_g;     real* gb = sm + A.o_gb;   real* qv = sm + A.o_q;
    real* sb = sm + A.o_sb;   real* ab = sb;            // the incoming adjoint on dx/dt is consumed before sbar is produced
    real* xd = sm + A.o_xd;   real* lam = sm + A.o_lam; real* xbn = sm + A.o_xbn; real* xsum = sm + A.o_xsum;
    real* z0 = sm + A.o_z0;   real* za = sm + A.o_za;   real* sc = sm + A.o_sc;   real* red = sm + A.o_red;
    real* qx = sm + A.o_qx;   real* as_ = sm + A.o_as;  real* ag_ = sm + A.o_ag;  real* bt = sm + A.o_bt;
    real* vm = sm + A.o_vm;   real* part = sm + A.o_part;
    real* T0 = sm + A.o_T0;   real* u0 = sm + A.o_u0;   real* T1 = sm + A.o_T1;   real* z1 = sm + A.o_z1;
    real* OD = sm + A.o_od;   real* AD = sm + A.o_ad;   real* X1 = sm + A.o_x1;   real* X2 = sm + A.o_x2;
    if (WSM) {
        for (int i = tid; i < P.blob_len; i += NT) sm[A.o_w + i] = P.blob[i];
    }
    const real* wb = WSM ? (sm + A.o_w) : P.blob;
    const real* Wb0 = wb + P.off_b0; const real* Wb1 = wb + P.off_b1; const real* Ww = wb + P.off_w; const real* Wcw = wb + P.off_cw;
    const real h = P.h;
    __syncthreads();

    // per-sample sum over the threads that share a sample (fixed shuffle tree, then warps in fixed order); ends with a barrier
    auto sample_sum = [&](real v) __attribute__((always_inline)) -> real {
#pragma unroll
        for (int off = TS; off < 32; off <<= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
        __syncthreads();
        if (lane < TS) red[warp * TS + lane] = v;
        __syncthreads();
        real t = real(0);
        for (int w = 0; w < nwarps; ++w) t += red[w * TS + smp];
        return t;
    };

    // an m-wide contraction.  Weights from L2 (the wide nets): two outputs per thread over half of K each (measured on swarm50:
    // 34.6 -> 32.9 ms per training iteration).  Weights staged in shared memory (m <= 128): one output per thread — the extra
    // barrier and partial-sum round trip of matvec2 cost more than the saved row loads (singlequad 3.5 -> 4.0 ms).
    auto mwide = [&](const real* Wm, int N, int K, const real* in, auto epi) __attribute__((always_inline)) {
        if constexpr (WSM) matvec<real, TS, WSM>(Wm, N, K, in, part, 1, tid, NT, A.deep != 0, epi);
        else matvec2<real, TS, WSM>(Wm, N, K, in, part, tid, NT, epi);
    };

    // ---- grad Phi at the stage input in `s` -> g (and q = A'A s); terminal: X2 = u1 = u0 + h act(a1)
    auto primal = [&](bool terminal) __attribute__((always_inline)) {
        mwide(wb + P.off_W1t, m, D, s, [&](int j, real (&acc)[TS]) __attribute__((always_inline)) {
            const real b = Wb0[j];
#pragma unroll
            for (int q = 0; q < TS; ++q) { real av, qs; act_q(acc[q] + b, av, qs); u0[j * TS + q] = av; T0[j * TS + q] = qs; }   // T0: q-form
        });
        __syncthreads();
        mwide(wb + P.off_Kft, m, m, u0, [&](int j, real (&acc)[TS]) __attribute__((always_inline)) {
            const real b = Wb1[j], wv = Ww[j];
#pragma unroll
            for (int q = 0; q < TS; ++q) {
                real qs;
                if (terminal) { real av; act_q(acc[q] + b, av, qs); X2[j * TS + q] = u0[j * TS + q] + h * av; }
                else qs = q_only(acc[q] + b);
                T1[j * TS + q] = qs;                                // q-form
                X1[j * TS + q] = q_tanh(qs) * wv;                   // y
            }
        });
        __syncthreads();
        mwide(wb + P.off_Kr, m, m, X1, [&](int j, real (&acc)[TS]) __attribute__((always_inline)) {
            const real wv = Ww[j];
#pragma unroll
            for (int q = 0; q < TS; ++q) { real z = wv + h * acc[q]; z1[j * TS + q] = z; OD[j * TS + q] = q_tanh(T0[j * TS + q]) * z; }   // v
        });
        __syncthreads();
        matvec<real, TS, WSM>(wb + P.off_sym, D, D, s, part, 1, tid, NT, A.deep != 0, [&](int j, real (&acc)[TS]) __attribute__((always_inline)) {
#pragma unroll
            for (int q = 0; q < TS; ++q) qv[j * TS + q] = acc[q];
        });
        matvec<real, TS, WSM>(wb + P.off_W4, D, m, OD, part, A.nsplitD, tid, NT, A.deep != 0, [&](int j, real (&acc)[TS]) __attribute__((always_inline)) {
            const real c = Wcw[j];
#pragma unroll
            for (int q = 0; q < TS; ++q) g[j * TS + q] = (qv[j * TS + q] + acc[q]) + c;
        });
        __syncthreads();
    };

    // ---- calcLHQW at x = s[:d], p = g[:d]  ->  sc = (L, |Phi_t - H|, Q, W), qx (quadcopter rates);
    //      adjoint: also gb = d psi / d g and xd = direct d psi / d x for psi = ab.(-grad_p H) + cL L + cH |g_t - H|
    auto problem = [&](bool adjoint, real cL, real cH) __attribute__((always_inline)) {
        const real vmask = vm[smp];
        cL *= vmask; cH *= vmask;
        if (pr.kind == 2) {                              // Quadcopter.py:65-113, one agent
            if (part_id == 0) {
                auto X = [&](int c) { return s[c * TS + smp]; };
                auto Pp = [&](int c) { return g[c * TS + smp]; };
                real sps, cps, sth, cth, sph, cph;
                r_sincos(X(3), &sps, &cps); r_sincos(X(4), &sth, &cth); r_sincos(X(5), &sph, &cph);
                const real F[3] = {sps * sph + cps * sth * cph, -cps * sph + sps * sth * cph, cth * cph};
                const real fp = F[0] * Pp(6) + F[1] * Pp(7) + F[2] * Pp(8);
                const real u = real(-1.0 / (2.0 * pr.mass)) * fp;
                const real sq = Pp(9) * Pp(9) + Pp(10) * Pp(10) + Pp(11) * Pp(11);
                const real L = real(2) + u * u + real(0.25) * sq;
                const real um = u / real(pr.mass);
                const real xv = X(6) * Pp(0) + X(7) * Pp(1) + X(8) * Pp(2);
                const real xw = X(9) * Pp(3) + X(10) * Pp(4) + X(11) * Pp(5);
                const real H = -L - xv - xw - um * fp + real(pr.grav) * Pp(8) + real(0.5) * sq;
                const real E = g[d * TS + smp] - H;
                sc[SC_L * TS + smp] = L; sc[SC_HJ * TS + smp] = r_abs(E); sc[SC_Q * TS + smp] = real(0); sc[SC_W * TS + smp] = real(0);
                qx[0 * TS + smp] = um; qx[1 * TS + smp] = F[0]; qx[2 * TS + smp] = F[1]; qx[3 * TS + smp] = F[2];
                if (adjoint) {
                    auto Ab = [&](int c) { return ab[c * TS + smp]; };
                    const real k = cH * sgn(E), cLk = cL + k;
                    const real aF = Ab(6) * F[0] + Ab(7) * F[1] + Ab(8) * F[2];
                    const real cfp = -cLk * um + real(2) * k * um - aF / real(2.0 * pr.mass * pr.mass);
                    // dF[c][a] = d F_c / d angle_a, angles (psi, theta, phi) = x[3:6]
                    const real dF[3][3] = {{cps * sph - sps * sth * cph, cps * cth * cph, sps * cph - cps * sth * sph},
                                           {sps * sph + cps * sth * cph, sps * cth * cph, -cps * cph - sps * sth * sph},
                                           {real(0), -sth * cph, -cth * sph}};
#pragma unroll
                    for (int c = 0; c < 3; ++c) {
                        xd[c * TS + smp] = real(0);
                        xd[(3 + c) * TS + smp] = cfp * (dF[0][c] * Pp(6) + dF[1][c] * Pp(7) + dF[2][c] * Pp(8)) +
                                                 um * (dF[0][c] * Ab(6) + dF[1][c] * Ab(7) + dF[2][c] * Ab(8));
                        xd[(6 + c) * TS + smp] = Ab(c) + k * Pp(c);
                        xd[(9 + c) * TS + smp] = Ab(3 + c) + k * Pp(3 + c);
                    }
                    real gbo[12];
#pragma unroll
                    for (int c = 0; c < 3; ++c) {
                        gbo[c] = k * X(6 + c);
                        gbo[3 + c] = k * X(9 + c);
                        gbo[6 + c] = cfp * F[c];
                        gbo[9 + c] = real(-0.5) * Ab(9 + c) - k * Pp(9 + c) + real(0.5) * cLk * Pp(9 + c);
                    }
                    gbo[8] -= k * real(pr.grav);
#pragma unroll
                    for (int c = 0; c < 12; ++c) gb[c * TS + smp] = gbo[c];     // ab aliases nothing of gb: safe to write now
                    gb[d * TS + smp] = k;
                }
            }
            __syncthreads();
            return;
        }
        const int Ag = pr.nAgents, dim = pr.agentDim;
        real pp = real(0), q = real(0), w = real(0);
        for (int j = part_id; j < d; j += nparts) { real p = g[j * TS + smp]; pp = r_fma(p, p, pp); }
        const bool needQ = (pr.obstacle != 0) && (pr.kind == 0 || pr.alph_Q > 0.0);
        const real aQ = needQ ? real(pr.alph_Q) : real(0);
        const bool needW = (pr.alph_W != 0.0) && Ag >= 2;
        const real cut = real(pr.cutW), c2 = real(2 * pr.r * pr.r), inv_r2 = real(1.0 / (pr.r * pr.r)), aW = real(pr.alph_W);
        for (int a = part_id; a < Ag; a += nparts) {
            real xi[3] = {s[(a * dim) * TS + smp], s[(a * dim + 1) * TS + smp], dim == 3 ? s[(a * dim + 2) * TS + smp] : real(0)};
            real gi[3] = {real(0), real(0), real(0)};
            if (needQ) {
                q += terrain_agent<real>(pr, xi[0], xi[1], xi[2]);
                if (adjoint) {
                    real gq[3];
                    terrain_agent_grad<real>(pr, xi[0], xi[1], xi[2], gq);
                    gi[0] = aQ * gq[0]; gi[1] = aQ * gq[1]; gi[2] = aQ * gq[2];
                }
            }
            if (needW) {                                 // Cross2D.py:130-162, SwarmTraj.py:133-164: pairs inside the cut-off
                for (int j = 0; j < Ag; ++j) {
                    if (j == a) continue;
                    real df[3] = {xi[0] - s[(j * dim) * TS + smp], xi[1] - s[(j * dim + 1) * TS + smp],
                                  dim == 3 ? xi[2] - s[(j * dim + 2) * TS + smp] : real(0)};
                    real d2 = r_fma(df[2], df[2], r_fma(df[1], df[1], df[0] * df[0]));
                    if (d2 < cut * cut * real(1.0001)) {
                        real dd = r_sqrt(d2);
                        if (dd < cut) {
                            real e = r_exp(-(dd * dd) / c2);
                            if (j > a && (Ag == 2 || e != real(1))) w += e;      // each pair once; the "== 1" rule (A > 2 only)
                            if (adjoint) { real ce = aW * e * inv_r2; gi[0] -= ce * df[0]; gi[1] -= ce * df[1]; gi[2] -= ce * df[2]; }
                        }
                    }
                }
            }
            if (adjoint)
                for (int c = 0; c < dim; ++c) xd[(a * dim + c) * TS + smp] = gi[c];
        }
        pp = sample_sum(pp);
        if (needQ) q = sample_sum(q);
        if (needW) w = sample_sum(w);
        real Qret, L;
        if (pr.kind == 0) { Qret = real(pr.alph_Q) * q; L = real(0.5) * pp + Qret; }
        else { Qret = (pr.alph_Q > 0.0) ? q : real(0); L = real(0.5) * pp + real(pr.alph_Q) * Qret; }
        if (pr.alph_W != 0.0) L = L + real(pr.alph_W) * w; else w = real(0);
        const real H = -L + pp;
        const real E = g[d * TS + smp] - H;
        if (part_id == 0) { sc[SC_L * TS + smp] = L; sc[SC_HJ * TS + smp] = r_abs(E); sc[SC_Q * TS + smp] = Qret; sc[SC_W * TS + smp] = w; }
        if (adjoint) {
            const real k = cH * sgn(E);
            __syncthreads();                             // every xd row is written
            for (int j = part_id; j < d; j += nparts) {
                gb[j * TS + smp] = (cL - k) * g[j * TS + smp] - ab[j * TS + smp];
                xd[j * TS + smp] *= (cL + k);
            }
            if (part_id == 0) gb[d * TS + smp] = k;
        }
        __syncthreads();
    };

    // ---- second-order sweep: tangent of the net along gb, its reverse, parameter gradients; sbar -> sb.
    //      terminal: bt[.] = beta (the adjoint of Phi itself), X2 = u1.
    auto second_order = [&](bool terminal) __attribute__((always_inline)) {
        mwide(wb + P.off_W1t, m, D, gb, [&](int j, real (&acc)[TS]) __attribute__((always_inline)) {
#pragma unroll
            for (int q = 0; q < TS; ++q) { OD[j * TS + q] = acc[q]; X1[j * TS + q] = q_tanh(T0[j * TS + q]) * acc[q]; }     // odot, udot
        });
        __syncthreads();
        mwide(wb + P.off_Kft, m, m, X1, [&](int j, real (&acc)[TS]) __attribute__((always_inline)) {
            const real wv = Ww[j];
            real wsum = real(0), bsum = real(0);
#pragma unroll
            for (int q = 0; q < TS; ++q) {
                const real ad = acc[q], q1 = T1[j * TS + q], t1 = q_tanh(q1);
                T1[j * TS + q] = t1;                                // from here on (dK1) the panel holds tanh itself
                real ws = X1[j * TS + q] + h * t1 * ad;
                real ba = h * wv * ad * q_dtanh(q1);
                if (terminal) { const real b = bt[q]; ws += b * X2[j * TS + q]; ba += b * h * t1 * wv; }
                AD[j * TS + q] = ba;
                wsum += ws; bsum += ba;
            }
            red_add(A.grad + P.g_w + j, wsum);
            red_add(A.grad + P.g_b1 + j, bsum);
        });
        __syncthreads();
        mwide(wb + P.off_Kr, m, m, AD, [&](int j, real (&acc)[TS]) __attribute__((always_inline)) {
            const real wv = Ww[j];
            real bsum = real(0);
#pragma unroll
            for (int q = 0; q < TS; ++q) {
                real bu = acc[q];
                if (terminal) bu += bt[q] * wv;
                const real q0 = T0[j * TS + q], t0 = q_tanh(q0);
                T0[j * TS + q] = t0;                                // from here on (dK0) the panel holds tanh itself
                const real bo = q_dtanh(q0) * OD[j * TS + q] * z1[j * TS + q] + t0 * bu;
                X2[j * TS + q] = bo;
                bsum += bo;
            }
            red_add(A.grad + P.g_b0 + j, bsum);
        });
        __syncthreads();
        matvec<real, TS, WSM>(wb + P.off_sym, D, D, gb, part, 1, tid, NT, A.deep != 0, [&](int j, real (&acc)[TS]) __attribute__((always_inline)) {
#pragma unroll
            for (int q = 0; q < TS; ++q) sb[j * TS + q] = acc[q];
        });
        matvec<real, TS, WSM>(wb + P.off_W4, D, m, X2, part, A.nsplitD, tid, NT, A.deep != 0, [&](int j, real (&acc)[TS]) __attribute__((always_inline)) {
            const real c = Wcw[j];
            real csum = real(0);
#pragma unroll
            for (int q = 0; q < TS; ++q) {
                real v = sb[j * TS + q] + acc[q];
                real cs = gb[j * TS + q];
                if (terminal) { v += bt[q] * (qv[j * TS + q] + c); cs += bt[q] * s[j * TS + q]; }
                sb[j * TS + q] = v;
                csum += cs;
            }
            red_add(A.grad + P.g_cw + j, csum);
        });
        // A s and A gbar (r x TS each) for dA
        for (int i = tid; i < P.r * TS; i += NT) {
            const int qq = i / TS, si = i % TS;
            const real* Ar = wb + P.off_A + qq * D;
            real a1 = real(0), a2 = real(0);
            for (int c = 0; c < D; ++c) { a1 = r_fma(Ar[c], s[c * TS + si], a1); a2 = r_fma(Ar[c], gb[c * TS + si], a2); }
            as_[i] = a1; ag_[i] = a2;
        }
        __syncthreads();
        // dK1[j][k] += h w_j sum_s T1[j][s] udot[k][s] + sum_s bar_a1[j][s] u0[k][s]
        if (A.use_v4 && sizeof(real) == 4 && (m & 3) == 0 && (NT % (m / 4) == 0 || NT < m / 4)) {
            // fp32: a thread owns FOUR consecutive columns k (its udot / u0 rows in registers) for a slice of the rows j; one
            // 16-byte vector reduction per row (REDG.ADD.F32x4, coalesced over the column groups) and 64 FMAs per pair of row loads
            const int KG = m >> 2, nrg = (NT >= KG) ? NT / KG : 1;
            for (int kg = tid % KG, rg = tid / KG; kg < KG && rg < nrg; kg += NT) {      // NT < KG: column groups in passes
                real ud[4][TS], uu[4][TS];
#pragma unroll
                for (int c = 0; c < 4; ++c) { ld_row<real, TS>(X1 + (4 * kg + c) * TS, ud[c]); ld_row<real, TS>(u0 + (4 * kg + c) * TS, uu[c]); }
                const int jb = (m * rg) / nrg, je = (m * (rg + 1)) / nrg;
                float* gk = reinterpret_cast<float*>(A.grad) + P.g_K1 + 4 * kg;
                for (int j = jb; j < je; ++j) {
                    real t[TS], b[TS];
                    ld_row<real, TS>(T1 + j * TS, t);
                    ld_row<real, TS>(AD + j * TS, b);
                    const real hw = h * Ww[j];
                    float o[4];
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        real a1 = real(0), a2 = real(0);
#pragma unroll
                        for (int q = 0; q < TS; ++q) { a1 = r_fma(t[q], ud[c][q], a1); a2 = r_fma(b[q], uu[c][q], a2); }
                        o[c] = (float)r_fma(hw, a1, a2);
                    }
                    red_add4(gk + (size_t)j * m, o[0], o[1], o[2], o[3]);
                }
            }
        } else {                                                                       // thread = column k: coalesced scalar reds
            for (int k = tid; k < m; k += NT) {
                real ud[TS], uu[TS];
                ld_row<real, TS>(X1 + k * TS, ud);
                ld_row<real, TS>(u0 + k * TS, uu);
                real* gk = A.grad + P.g_K1 + k;
                for (int j = 0; j < m; ++j) {
                    real t[TS], b[TS];
                    ld_row<real, TS>(T1 + j * TS, t);
                    ld_row<real, TS>(AD + j * TS, b);
                    real a1 = real(0), a2 = real(0);
#pragma unroll
                    for (int q = 0; q < TS; ++q) { a1 = r_fma(t[q], ud[q], a1); a2 = r_fma(b[q], uu[q], a2); }
                    red_add(gk + (size_t)j * m, r_fma(h * Ww[j], a1, a2));
                }
            }
        }
        // dK0[j][c] += sum_s v[j][s] gbar[c][s] + bar_o[j][s] s[c][s]                      (thread = column c, rows in slices)
        {
            const int nsl = (A.nsplitD > 1) ? A.nsplitD : 1, G = NT / nsl, sl = tid / G, cc = tid % G;
            if (sl < nsl) {
                const int jb = (m * sl) / nsl, je = (m * (sl + 1)) / nsl;
                for (int c = cc; c < D; c += G) {
                    real gc[TS], scn[TS];
                    ld_row<real, TS>(gb + c * TS, gc);
                    ld_row<real, TS>(s + c * TS, scn);
                    real* gk = A.grad + P.g_K0 + c;
                    for (int j = jb; j < je; ++j) {
                        real t0[TS], zz[TS], bo[TS];
                        ld_row<real, TS>(T0 + j * TS, t0);
                        ld_row<real, TS>(z1 + j * TS, zz);
                        ld_row<real, TS>(X2 + j * TS, bo);
                        real a1 = real(0);
#pragma unroll
                        for (int q = 0; q < TS; ++q) { a1 = r_fma(t0[q] * zz[q], gc[q], a1); a1 = r_fma(bo[q], scn[q], a1); }
                        red_add(gk + (size_t)j * D, a1);
                    }
                }
            }
        }
        // dA[q][c] += sum_s (As)[q][s] gbar[c][s] + (A gbar)[q][s] s[c][s] (+ beta (As)[q][s] s[c][s])
        for (int i = tid; i < P.r * D; i += NT) {
            const int qq = i / D, c = i % D;
            real a1 = real(0);
            for (int q = 0; q < TS; ++q) {
                real asv = as_[qq * TS + q], sv = s[c * TS + q];
                a1 = r_fma(asv, gb[c * TS + q], a1);
                a1 = r_fma(ag_[qq * TS + q], sv, a1);
                if (terminal) a1 = r_fma(bt[q] * asv, sv, a1);
            }
            red_add(A.grad + P.g_A + i, a1);
        }
        if (terminal && tid == 0) {
            real bsum = real(0);
            for (int q = 0; q < TS; ++q) bsum += bt[q];
            red_add(A.grad + P.g_cb, bsum);
        }
        __syncthreads();
    };

    if constexpr (VJP) {
        for (int tile = blockIdx.x; tile < A.ntiles; tile += gridDim.x) {
            const long long base = (long long)tile * TS;
            for (int i = tid; i < D * TS; i += NT) {
                const int c = i / TS, si = i % TS;
                const bool valid = base + si < A.n;
                const long long row = valid ? base + si : A.n - 1;          // pad rows repeat the last row with zero seeds
                s[i] = A.x[row * D + c];
                gb[i] = (valid && A.seed_grad) ? A.seed_grad[row * D + c] : real(0);
            }
            if (tid < TS) bt[tid] = (base + tid < A.n && A.seed_phi) ? A.seed_phi[base + tid] : real(0);
            __syncthreads();
            primal(true);
            second_order(true);
            if (A.grad_s)
                for (int i = tid; i < D * TS; i += NT) {
                    const int c = i / TS, si = i % TS;
                    if (base + si < A.n) A.grad_s[(base + si) * D + c] = sb[i];
                }
        }
        return;
    }

    auto rate = [&](int row, int si) __attribute__((always_inline)) -> real {         // dx/dt = -grad_p H
        if (pr.kind != 2) return -g[row * TS + si];
        if (row < 6) return s[(6 + row) * TS + si];
        if (row < 9) { real gg = -qx[si] * qx[(1 + row - 6) * TS + si]; if (row == 8) gg = gg + real(pr.grav); return -gg; }
        return -(real(0.5) * g[row * TS + si]);
    };

    const real wts[4] = {real(1.0 / 6.0), real(2.0 / 6.0), real(2.0 / 6.0), real(1.0 / 6.0)};
    const int nZ = (d + 4) * TS, nX = d * TS;
    for (int tile = blockIdx.x; tile < A.ntiles; tile += gridDim.x) {
        const long long base = (long long)tile * TS;
        real* xs_tile = A.xsave + (size_t)blockIdx.x * A.nt * 4 * nX;   // per CTA: a tile's forward + backward finish before the next tile starts
        if (tid < TS) vm[tid] = (base + tid < A.n) ? real(1) : real(0);
        for (int i = tid; i < nZ; i += NT) {
            const int r = i / TS, si = i % TS;
            long long row = base + si; if (row >= A.n) row = A.n - 1;              // pad rows repeat the last sample (masked out)
            z0[i] = (r < d) ? A.x[row * d + r] : real(0);
        }
        __syncthreads();
        // ------------------------------------------------ forward sweep (OCflow.py:33-55, stepRK4 :157-184)
        for (int k = 0; k < A.nt; ++k) {
            const double* tt = A.times + 5 * k;
            const real hstep = real(tt[4]);
            for (int i = tid; i < nX; i += NT) s[i] = z0[i];
            if (tid < TS) s[d * TS + tid] = real(tt[0]);
            __syncthreads();
            for (int st = 0; st < 4; ++st) {
                const real cnext = (st < 2) ? real(0.5) : real(1.0);
                const real tnext = (st < 2) ? real(tt[1]) : real(tt[2]);
                real* xsv = xs_tile + (size_t)(k * 4 + st) * nX;
                for (int i = tid; i < nX; i += NT) xsv[i] = s[i];
                primal(false);
                problem(false, real(0), real(0));
                for (int i = tid; i < nZ; i += NT) {
                    const int r = i / TS, si = i % TS;
                    xd[i] = hstep * ((r < d) ? rate(r, si) : sc[(r - d) * TS + si]);
                }
                __syncthreads();
                for (int i = tid; i < nZ; i += NT) {
                    const real kk = xd[i], z0v = z0[i];
                    za[i] = ((st == 0) ? z0v : za[i]) + wts[st] * kk;
                    if (st < 3 && i < nX) s[i] = z0v + cnext * kk;
                }
                if (st < 3 && tid < TS) s[d * TS + tid] = tnext;
                __syncthreads();
            }
            { real* t = z0; z0 = za; za = t; }
        }
        // ------------------------------------------------ terminal block (OCflow.py:58-90) and its adjoint
        for (int i = tid; i < nX; i += NT) s[i] = z0[i];
        if (tid < TS) s[d * TS + tid] = A.t_end;
        __syncthreads();
        primal(true);
        {
            const real* xt = static_cast<const real*>(pr.xtarget);
            real r2 = real(0), hjg = real(0), quad = real(0), lin = real(0), wn = real(0);
            for (int j = part_id; j < d; j += nparts) {
                real res = z0[j * TS + smp] - xt[j];
                r2 = r_fma(res, res, r2);
                hjg += r_abs(g[j * TS + smp] - A.alph0 * res);
            }
            for (int j = part_id; j < D; j += nparts) {
                quad = r_fma(s[j * TS + smp], qv[j * TS + smp], quad);
                lin = r_fma(Wcw[j], s[j * TS + smp], lin);
            }
            for (int j = part_id; j < m; j += nparts) wn = r_fma(Ww[j], X2[j * TS + smp], wn);
            r2 = sample_sum(r2); hjg = sample_sum(hjg); quad = sample_sum(quad); lin = sample_sum(lin); wn = sample_sum(wn);
            const real cG = real(0.5) * r2;
            const real phi1 = wn + real(0.5) * quad + (lin + wb[P.off_cb]);
            const real ef = phi1 - A.alph0 * cG;
            const real vmask = vm[smp];
            const real sf = sgn(ef) * vmask;
            if (part_id == 0) {
                bt[smp] = A.alph4 * sf;
                const real c8[8] = {z0[d * TS + smp], cG, z0[(d + 1) * TS + smp], r_abs(ef), hjg, z0[(d + 2) * TS + smp],
                                    z0[(d + 3) * TS + smp], real(1)};
#pragma unroll
                for (int q = 0; q < 8; ++q) sc[q * TS + smp] = vmask * c8[q];
            }
            for (int j = part_id; j < d; j += nparts) {
                const real res = z0[j * TS + smp] - xt[j];
                const real sg = sgn(g[j * TS + smp] - A.alph0 * res) * vmask;
                gb[j * TS + smp] = A.alph5 * sg;
                xd[j * TS + smp] = A.alph0 * (vmask - A.alph4 * sf) * res - A.alph5 * A.alph0 * sg;
            }
            if (part_id == 0) gb[d * TS + smp] = real(0);
            __syncthreads();
            if (tid < 8) {                               // this tile's cost sums, in double and in sample order
                double t = 0.0;
                for (int q = 0; q < TS; ++q) t += (double)sc[tid * TS + q];
                A.partials[(size_t)tile * 8 + tid] = t;
            }
        }
        second_order(true);
        for (int i = tid; i < nX; i += NT) lam[i] = sb[i] + xd[i];
        __syncthreads();
        // ------------------------------------------------ backward sweep: discrete adjoint of stepRK4
        for (int k = A.nt - 1; k >= 0; --k) {
            const double* tt = A.times + 5 * k;
            const real hstep = real(tt[4]);
            for (int st = 3; st >= 0; --st) {
                const real* xsv = xs_tile + (size_t)(k * 4 + st) * nX;
                const real cx = (st == 3) ? real(0) : ((st == 2) ? real(1) : real(0.5));
                for (int i = tid; i < nX; i += NT) {
                    real kb = wts[st] * lam[i];
                    if (st < 3) kb = r_fma(cx, xbn[i], kb);
                    ab[i] = hstep * kb;
                    s[i] = xsv[i];
                }
                if (tid < TS) s[d * TS + tid] = real(st == 0 ? tt[0] : (st == 3 ? tt[2] : tt[1]));
                __syncthreads();
                primal(false);
                problem(true, hstep * wts[st], hstep * wts[st] * A.alph3);
                second_order(false);
                for (int i = tid; i < nX; i += NT) {
                    const real xb = sb[i] + xd[i];
                    xbn[i] = xb;
                    xsum[i] = (st == 3) ? xb : xsum[i] + xb;
                }
                __syncthreads();
            }
            for (int i = tid; i < nX; i += NT) lam[i] += xsum[i];
            __syncthreads();
        }
        if (A.grad_x)
            for (int i = tid; i < nX; i += NT) {
                const int r = i / TS, si = i % TS;
                if (base + si < A.n) A.grad_x[(base + si) * d + r] = lam[i];
            }
        __syncthreads();
    }
}

// Tile planning and launch, shared by the training step and the Phi VJP: the packed-weight blob, the gradient sections, the tile
// width and the shared-memory layout are the same in both modes.
template <typename real>
struct GradLaunch {
    GradArgs<real> A;
    GradSections GS;
    int TS, NT;
    size_t smem;
    bool wsm;
};

template <typename real>
static int grad_plan(const char* who, int d, int m, int r, double h, long long n, int smem_limit, GradLaunch<real>& G) {
    GradArgs<real>& A = G.A;
    memset(&A, 0, sizeof A);
    GradPack<real>& P = A.phi;
    const int D = d + 1;
    P.d = d; P.D = D; P.m = m; P.r = r; P.h = (real)h;
    int off = 0;
    auto take = [&](int cnt) { int o = off; off += align_up(cnt, 8); return o; };
    P.off_W1t = take(D * m); P.off_Kft = take(m * m); P.off_Kr = take(m * m); P.off_W4 = take(m * D); P.off_sym = take(D * D);
    P.off_b0 = take(m); P.off_b1 = take(m); P.off_w = take(m); P.off_cw = take(D); P.off_cb = take(1); P.off_A = take(r * D);
    P.blob_len = off;
    // the kernel accumulates into a buffer whose sections start on 16-byte boundaries; unpack_grad_kernel compacts it
    GradSections& GS = G.GS;
    int go = 0, co = 0, gi = 0;
    auto gtake = [&](int cnt) { int o = go; GS.src[gi] = go; GS.dst[gi] = co; GS.len[gi] = cnt; ++gi; go += align_up(cnt, 4); co += cnt; return o; };
    P.g_A = gtake(r * D); P.g_cw = gtake(D); P.g_cb = gtake(1); P.g_w = gtake(m); P.g_K0 = gtake(m * D); P.g_b0 = gtake(m);
    P.g_K1 = gtake(m * m); P.g_b1 = gtake(m); P.g_len = go;

    const int NT = std::min(512, std::max(32, align_up(std::max(m, D), 32)));
    if (m > 2048 || (m & 1)) return fail(NOC_ERR_UNSUPPORTED, "%s: m = %d (even widths up to 2048)", who, m);
    auto plan = [&](int TS, size_t& vec_bytes, bool& wsm) -> size_t {
        int so = 0;
        auto stake = [&](int cnt) { int o = so; so += align_up(cnt, 8); return o; };
        A.o_s = stake(D * TS); A.o_g = stake(D * TS); A.o_gb = stake(D * TS); A.o_q = stake(D * TS); A.o_sb = stake(D * TS);
        A.o_xd = stake((d + 4) * TS); A.o_lam = stake(d * TS); A.o_xbn = stake(d * TS); A.o_xsum = stake(d * TS);
        A.o_z0 = stake((d + 4) * TS); A.o_za = stake((d + 4) * TS); A.o_sc = stake(SC_ROWS * TS); A.o_red = stake(32 * TS);
        A.o_qx = stake(4 * TS); A.o_as = stake(r * TS); A.o_ag = stake(r * TS); A.o_bt = stake(TS); A.o_vm = stake(TS);
        A.nsplitD = std::max(1, std::min(4, NT / align_up(D, 32)));
        A.o_part = stake(std::max(A.nsplitD > 1 ? A.nsplitD * D * TS : 8, m * TS));
        A.o_T0 = stake(m * TS); A.o_u0 = stake(m * TS); A.o_T1 = stake(m * TS); A.o_z1 = stake(m * TS);
        A.o_od = stake(m * TS); A.o_ad = stake(m * TS); A.o_x1 = stake(m * TS); A.o_x2 = stake(m * TS);
        A.o_w = so;
        vec_bytes = (size_t)so * sizeof(real);
        wsm = vec_bytes + (size_t)P.blob_len * sizeof(real) <= (size_t)smem_limit;
        return vec_bytes + (wsm ? (size_t)P.blob_len * sizeof(real) : 0);
    };
    // tile width (measured, `bench.py --train`): wide nets want 8 samples per tile — every weight load is amortised over more
    // samples (swarm50, n = 1024: 35 ms with 128 tiles of 8, 50 ms with 256 tiles of 4; singlequad 3.5 vs 5.6 ms); the narrow nets
    // run one or two warps per CTA and want more CTAs instead (softcorridor, n = 1024: 1.5 ms with tiles of 4, 1.9 ms with 8)
    int TS = 8;
    size_t vec_bytes = 0;
    bool wsm = false;
    size_t smem = plan(TS, vec_bytes, wsm);
    const bool fits8 = vec_bytes <= (size_t)smem_limit;
    if (!fits8 || (NT <= 64 && (n + 7) / 8 < 4LL * sm_count())) { TS = 4; smem = plan(TS, vec_bytes, wsm); }
    // ... and tiles of 2 while even tiles of 4 leave the GPU short of warps (measured at the README batch sizes: swap12 2.43 -> 1.99 ms,
    // swap2 1.55 -> 1.41, softcorridor 1.77 -> 1.71; tiles of 1 are slower again: 3.9 / 1.8 / 2.5 ms)
    if (TS == 4 && m <= 64 && wsm && (n + 3) / 4 < 8LL * sm_count()) { TS = 2; smem = plan(TS, vec_bytes, wsm); }
    if (const char* e = getenv("NOC_GRAD_TS")) { int t = atoi(e); if (t == 2 || t == 4 || t == 8) { TS = t; smem = plan(TS, vec_bytes, wsm); } }
    if (TS < 4 && !wsm) return fail(NOC_ERR_UNSUPPORTED, "%s: tiles of %d samples are built for staged weights only", who, TS);
    if (vec_bytes > (size_t)smem_limit)
        return fail(NOC_ERR_NOMEM, "%s: panels of d=%d, m=%d need %zu B of shared memory (> %d)", who, d, m, vec_bytes, smem_limit);
    A.ntiles = (int)((n + TS - 1) / TS);
    if (getenv("NOC_DEBUG"))
        fprintf(stderr, "[noc] %s kernel: n=%lld d=%d m=%d TS=%d NT=%d tiles=%d smem=%zu (panels %zu, weights %s) limit=%d\n", who, n, d, m,
                TS, NT, A.ntiles, smem, vec_bytes, wsm ? "staged" : "L2", smem_limit);
    A.use_v4 = wsm ? 0 : 1; A.deep = 1;
    if (const char* e = getenv("NOC_GRAD_V4")) A.use_v4 = atoi(e);
    if (const char* e = getenv("NOC_GRAD_DEEP")) A.deep = atoi(e);
    G.TS = TS; G.NT = NT; G.smem = smem; G.wsm = wsm;
    return NOC_OK;
}

// weight packing, the kernel of the mode (training: nt RK4 steps per tile; VJP: one evaluation per row) and the compaction of the
// summed parameter gradient into `grad` (NULL: the sums are not wanted)
template <typename real, bool VJP>
static int grad_launch(GradLaunch<real>& G, const PhiRaw<real>& raw, real* grad, int nt, cudaStream_t st) {
    GradArgs<real>& A = G.A;
    GradPack<real>& P = A.phi;
    const int m = P.m, D = P.D, d = P.d, TS = G.TS;
    ScratchBuf b_blob, b_xsave, b_gacc;                    // freed (stream-ordered) on every exit path
    NOC_CUDA(b_blob.alloc(sizeof(real) * (size_t)P.blob_len, st));
    real* blob = b_blob.as<real>();
    NOC_CUDA(cudaMemsetAsync(blob, 0, sizeof(real) * (size_t)P.blob_len, st));
    int pgrid = std::min(std::max(1, ceil_div(std::max(m * m, m * D), 256)), 4 * sm_count());
    pack_phi_grad_kernel<real><<<pgrid, 256, 0, st>>>(raw, P, blob);
    count_launch();
    P.blob = blob;
    NOC_CUDA(b_gacc.alloc(sizeof(real) * (size_t)P.g_len, st));
    real* gacc = b_gacc.as<real>();
    NOC_CUDA(cudaMemsetAsync(gacc, 0, sizeof(real) * (size_t)P.g_len, st));
    A.grad = gacc;
    void (*kern)(const GradArgs<real>) = nullptr;
    if (TS == 8) kern = G.wsm ? rollout_grad_kernel<real, 8, true, VJP> : rollout_grad_kernel<real, 8, false, VJP>;
    else if (TS == 4) kern = G.wsm ? rollout_grad_kernel<real, 4, true, VJP> : rollout_grad_kernel<real, 4, false, VJP>;
    else kern = rollout_grad_kernel<real, 2, true, VJP>;
    NOC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G.smem));
    int per_sm = 0;
    NOC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, G.NT, G.smem));
    if (per_sm < 1) return fail(NOC_ERR_NOMEM, "%s: kernel does not fit on an SM (%zu B shared memory)", VJP ? "noc_phi_vjp" : "noc_ocflow_grad", G.smem);
    const int grid = std::max(1, std::min(A.ntiles, per_sm * sm_count()));
    if (!VJP) {
        NOC_CUDA(b_xsave.alloc(sizeof(real) * (size_t)grid * nt * 4 * d * TS, st));
        A.xsave = b_xsave.as<real>();
    }
    kern<<<grid, G.NT, G.smem, st>>>(A);
    count_launch();
    NOC_CUDA(cudaGetLastError());
    if (grad) {
        unpack_grad_kernel<real><<<std::min(std::max(1, ceil_div(P.g_len, 256)), 4 * sm_count()), 256, 0, st>>>(gacc, grad, G.GS);
        count_launch();
        NOC_CUDA(cudaGetLastError());
    }
    return NOC_OK;
}

template <typename real>
int grad_rollout(int d, int m, int r, double h, const PhiRaw<real>& raw, const ProbPack& pr, const real* x, long long n,
                 const double* dtimes, int nt, const double* alph, double t_end, double* out_sums, real* grad, real* grad_x,
                 int smem_limit, cudaStream_t st) {
    GradLaunch<real> G;
    int rc = grad_plan<real>("noc_ocflow_grad", d, m, r, h, n, smem_limit, G);
    if (rc) return rc;
    GradArgs<real>& A = G.A;
    ScratchBuf b_partials;                                 // freed (stream-ordered) on every exit path
    NOC_CUDA(b_partials.alloc(sizeof(double) * 8 * (size_t)A.ntiles, st));
    A.prob = pr; A.x = x; A.n = n; A.nt = nt; A.times = dtimes;
    A.alph0 = (real)alph[0]; A.alph3 = (real)alph[3]; A.alph4 = (real)alph[4]; A.alph5 = (real)alph[5];
    A.t_end = (real)t_end;
    A.partials = b_partials.as<double>(); A.grad_x = grad_x;
    rc = grad_launch<real, false>(G, raw, grad, nt, st);
    if (rc) return rc;
    return launch_finish(A.partials, A.ntiles, out_sums, st);
}

template <typename real>
int phi_vjp(int d, int m, int r, double h, const PhiRaw<real>& raw, const real* s, long long n, const real* seed_phi,
            const real* seed_grad, real* grad, real* grad_s, int smem_limit, cudaStream_t st) {
    GradLaunch<real> G;
    int rc = grad_plan<real>("noc_phi_vjp", d, m, r, h, n, smem_limit, G);
    if (rc) return rc;
    GradArgs<real>& A = G.A;
    A.x = s; A.n = n; A.seed_phi = seed_phi; A.seed_grad = seed_grad; A.grad_s = grad_s;
    return grad_launch<real, true>(G, raw, grad, 0, st);
}

// one object per precision (Makefile: -DNOC_GRAD_ONLY=32 / 64) so that the two sets of instantiations compile in parallel
#if !defined(NOC_GRAD_ONLY) || NOC_GRAD_ONLY == 32
template int grad_rollout<float>(int, int, int, double, const PhiRaw<float>&, const ProbPack&, const float*, long long, const double*, int,
                                 const double*, double, double*, float*, float*, int, cudaStream_t);
template int phi_vjp<float>(int, int, int, double, const PhiRaw<float>&, const float*, long long, const float*, const float*, float*, float*,
                            int, cudaStream_t);
#endif
#if !defined(NOC_GRAD_ONLY) || NOC_GRAD_ONLY == 64
template int grad_rollout<double>(int, int, int, double, const PhiRaw<double>&, const ProbPack&, const double*, long long, const double*, int,
                                  const double*, double, double*, double*, double*, int, cudaStream_t);
template int phi_vjp<double>(int, int, int, double, const PhiRaw<double>&, const double*, long long, const double*, const double*, double*,
                             double*, int, cudaStream_t);
#endif

}  // namespace noc
