// noc_vec.cu — the small-batch ("deployment") rollout kernel: ONE CTA PER SAMPLE, one thread per hidden unit.
//
// The tile kernel (noc_rollout.cuh) gives every thread an outputs x samples register tile, which is the right shape
// for 10^5..10^7 samples but makes a batch of one pay for a whole tile of samples and run as a single warp's serial
// instruction stream.  timeDeployment/timeOC.py times exactly one OCflow(xInit) call (SURVEY.md §6.1), so for small
// batches the contractions are laid out the other way round: every grad-Phi contraction is a matrix-vector product
// whose input vector sits in shared memory and whose output unit j belongs to thread j; the weights are read
// K-major (coalesced over j) from a staged shared-memory copy when they fit (all nets but swarm50) or from L2.
// Same arithmetic, same quirks, same outputs as the tile kernel; the host picks the path by batch size.
#include "noc_launch.cuh"

namespace noc {

template <typename real>
struct VecPack {
    int d, D, m, nTh, r;
    real h;
    const real* blob;
    int blob_len;
    int off_W1t;               // [D][m]   W1t[k][o] = K0[o][k]
    int off_Kft[MAXL];         // [m][m]   Kft[k][o] = K_i[o][k]
    int off_Kr[MAXL];          // [m][m]   K_i as stored: out k' = sum_j K_i[j][k'] y[j]
    int off_sym;               // [D][D]   A'A
    int off_W4;                // [m][D]   K0 as stored
    int off_b[MAXL], off_w, off_cw, off_cb;
};

template <typename real>
struct VecArgs {
    VecPack<real> phi;
    ProbPack prob;
    const real* x;
    long long n;
    int nt, stepper, mode;
    const double* times;
    real alph0, alph3, alph4, alph5, t_end;
    double* partials;          // mean mode: [n][8] per-sample costs (+ count 1), summed by finish_costs_kernel
    real* out_a; real* out_b; real* out_c;
    // element offsets of the shared-memory vectors
    int o_s, o_u, o_u2, o_t, o_zb, o_g, o_q, o_z0, o_za, o_sc, o_red, o_qx, o_w;
};

template <typename real>
__global__ void pack_phi_plain_kernel(const PhiRaw<real> R, const VecPack<real> P, real* __restrict__ blob) {
    const int D = P.D, m = P.m, nTh = P.nTh, r = P.r;
    const int stride = gridDim.x * blockDim.x, t0 = blockIdx.x * blockDim.x + threadIdx.x;
    for (int i = t0; i < m * D; i += stride) {
        int o = i / D, k = i % D;
        real v = R.K[0][i];
        blob[P.off_W1t + k * m + o] = v;
        blob[P.off_W4 + i] = v;
    }
    for (int l = 1; l < nTh; ++l)
        for (int i = t0; i < m * m; i += stride) {
            int o = i / m, k = i % m;
            real v = R.K[l][i];
            blob[P.off_Kft[l] + k * m + o] = v;
            blob[P.off_Kr[l] + i] = v;
        }
    for (int i = t0; i < D * D; i += stride) {
        int k = i / D, o = i % D;
        real s = real(0);
        for (int q = 0; q < r; ++q) s = r_fma(R.A[q * D + k], R.A[q * D + o], s);
        blob[P.off_sym + i] = s;
    }
    for (int l = 0; l < nTh; ++l)
        for (int i = t0; i < m; i += stride) blob[P.off_b[l] + i] = R.b[l][i];
    for (int i = t0; i < m; i += stride) blob[P.off_w + i] = R.w[i];
    for (int i = t0; i < D; i += stride) blob[P.off_cw + i] = R.c_w[i];
    if (t0 == 0) blob[P.off_cb] = R.c_b[0];
}

// deterministic block-wide sum: every thread returns the same total (fixed shuffle tree + fixed warp order)
template <bool ONEWARP>
__device__ __forceinline__ void cta_sync() {
    if (ONEWARP) __syncwarp(); else __syncthreads();
}

template <typename real, bool ONEWARP>
__device__ __forceinline__ real block_sum(real v, real* red, int tid, int nthreads) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    if (ONEWARP) return v;                 // nets with m, d+4 <= 32 run as a single warp: no shared-memory stage
    __syncthreads();                       // previous users of `red` are done
    if ((tid & 31) == 0) red[tid >> 5] = v;
    __syncthreads();
    real s = real(0);
    for (int w = 0; w < (nthreads >> 5); ++w) s += red[w];
    return s;
}

// out_j = sum_k W[k][j] in[k] for my column j (W points at column j of row 0, row stride N)
template <typename real, bool WSM>
__device__ __forceinline__ real gemv_col(const real* __restrict__ W, int N, const real* in, int K) {
    real a0 = real(0), a1 = real(0), a2 = real(0), a3 = real(0);
    int k = 0;
    for (; k + 4 <= K; k += 4) {
        real w0, w1, w2, w3;
        if (WSM) { w0 = W[k * N]; w1 = W[(k + 1) * N]; w2 = W[(k + 2) * N]; w3 = W[(k + 3) * N]; }
        else { w0 = __ldg(W + k * N); w1 = __ldg(W + (k + 1) * N); w2 = __ldg(W + (k + 2) * N); w3 = __ldg(W + (k + 3) * N); }
        a0 = r_fma(w0, in[k], a0); a1 = r_fma(w1, in[k + 1], a1);
        a2 = r_fma(w2, in[k + 2], a2); a3 = r_fma(w3, in[k + 3], a3);
    }
    for (; k < K; ++k) a0 = r_fma(WSM ? W[k * N] : __ldg(W + k * N), in[k], a0);
    return (a0 + a1) + (a2 + a3);
}

template <typename real, bool WSM, bool ONEWARP>
__device__ __forceinline__ void rollout_vec_body(const VecArgs<real>& A) {
    extern __shared__ __align__(16) unsigned char vec_smem[];
    real* sm = reinterpret_cast<real*>(vec_smem);
    const int tid = threadIdx.x, NT = blockDim.x;
    const VecPack<real>& P = A.phi;
    const ProbPack& pr = A.prob;
    const int d = P.d, D = P.D, m = P.m, nTh = P.nTh;
    real* s = sm + A.o_s;      real* g = sm + A.o_g;     real* qv = sm + A.o_q;
    real* tbuf = sm + A.o_t;   real* zbv = sm + A.o_zb;  real* sc = sm + A.o_sc;
    real* red = sm + A.o_red;  real* qx = sm + A.o_qx;
    real* z0 = sm + A.o_z0;    real* za = sm + A.o_za;
    if (WSM) {
        for (int i = tid; i < P.blob_len; i += NT) sm[A.o_w + i] = P.blob[i];
    }
    const real* wb = WSM ? (sm + A.o_w) : P.blob;
    cta_sync<ONEWARP>();

    // grad Phi (Phi.py:99-138) of the s = [x,t] in `s` -> g; terminal also Phi's pieces: returns w . u_last
    auto chain = [&](bool terminal) -> real {
        real* u = sm + A.o_u;
        real* u2 = sm + A.o_u2;
        real phiN = real(0);
        if (tid < m) {                               // opening layer (Phi.py:114-115)
            real pre = gemv_col<real, WSM>(wb + P.off_W1t + tid, m, s, D) + wb[P.off_b[0] + tid];
            real av, tv;
            act_tanh(pre, av, tv);
            u[tid] = av;
            tbuf[tid] = tv;
        }
        cta_sync<ONEWARP>();
        for (int i = 1; i < nTh; ++i) {              // forward layers (Phi.py:118-120)
            const bool last = (i == nTh - 1);
            real part = real(0);
            if (tid < m) {
                real pre = gemv_col<real, WSM>(wb + P.off_Kft[i] + tid, m, u, m) + wb[P.off_b[i] + tid];
                if (!last) {
                    real av, tv;
                    act_tanh(pre, av, tv);
                    tbuf[i * m + tid] = tv;
                    u2[tid] = u[tid] + P.h * av;
                } else {
                    real wv = wb[P.off_w + tid];
                    if (terminal) {
                        real av, tv;
                        act_tanh(pre, av, tv);
                        part = wv * (u[tid] + P.h * av);
                        u2[tid] = tv * wv;
                    } else {
                        u2[tid] = tanh_only(pre) * wv;
                    }
                }
            }
            if (terminal && last) phiN = block_sum<real, ONEWARP>(part, red, tid, NT);
            cta_sync<ONEWARP>();
            real* t = u; u = u2; u2 = t;
        }
        for (int i = nTh - 1; i >= 1; --i) {         // reverse sweep (Phi.py:124-131); u holds y
            if (tid < m) {
                real acc = gemv_col<real, WSM>(wb + P.off_Kr[i] + tid, m, u, m);
                real zi = ((i == nTh - 1) ? wb[P.off_w + tid] : zbv[tid]) + P.h * acc;
                if (i > 1) zbv[tid] = zi;
                u2[tid] = tbuf[(i - 1) * m + tid] * zi;
            }
            cta_sync<ONEWARP>();
            real* t = u; u = u2; u2 = t;
        }
        if (tid < D) {                               // grad = A'A s + K0' v + c_w' (Phi.py:133-136)
            real q = gemv_col<real, WSM>(wb + P.off_sym + tid, D, s, D);
            if (terminal) qv[tid] = q;
            g[tid] = (q + gemv_col<real, WSM>(wb + P.off_W4 + tid, D, u, m)) + wb[P.off_cw + tid];
        }
        cta_sync<ONEWARP>();
        return phiN;
    };

    // L, |Phi_t - H|, Q, W -> sc[0..3] from x = s[:d], p = g[:d] (calcLHQW of the three problem classes)
    auto problem = [&]() {
        if (pr.kind == 2) {                          // Quadcopter.py:86-113 (one thread; a handful of flops)
            if (tid == 0) {
                real H = real(0), Q = real(0), W = real(0);
                real L = real(pr.alph_Q) * Q;
                if (pr.alph_W > 0.0) {
                    if (pr.nAgents == 2) {
                        real d2 = real(0);
                        for (int c = 0; c < 3; ++c) { real df = s[c] - s[12 + c]; d2 = r_fma(df, df, d2); }
                        real dd = r_sqrt(d2);
                        if (dd < real(2 * pr.r)) W = r_exp(-(dd * dd) / real(2 * pr.r * pr.r));
                    }
                    L = L + real(pr.alph_W) * W;
                }
                for (int a = 0; a < pr.nAgents; ++a) {
                    const real* x = s + 12 * a;
                    const real* p = g + 12 * a;
                    real sps, cps, sth, cth, sph, cph;
                    r_sincos(x[3], &sps, &cps); r_sincos(x[4], &sth, &cth); r_sincos(x[5], &sph, &cph);
                    real f7 = sps * sph + cps * sth * cph, f8 = -cps * sph + sps * sth * cph, f9 = cth * cph;
                    real fp = f7 * p[6] + f8 * p[7] + f9 * p[8];
                    real u = real(-1.0 / (2.0 * pr.mass)) * fp;
                    real sq = p[9] * p[9] + p[10] * p[10] + p[11] * p[11];
                    L = L + real(2) + u * u + real(0.25) * sq;
                    real um = u / real(pr.mass);
                    real xv = x[6] * p[0] + x[7] * p[1] + x[8] * p[2];
                    real xw = x[9] * p[3] + x[10] * p[4] + x[11] * p[5];
                    H = H - L - xv - xw - um * fp + real(pr.grav) * p[8] + real(0.5) * sq;
                    qx[5 * a] = um; qx[5 * a + 1] = f7; qx[5 * a + 2] = f8; qx[5 * a + 3] = f9; qx[5 * a + 4] = u;
                }
                sc[SC_L] = L; sc[SC_HJ] = r_abs(g[d] - H); sc[SC_Q] = Q; sc[SC_W] = W;
            }
            cta_sync<ONEWARP>();
            return;
        }
        const int Ag = pr.nAgents, dim = pr.agentDim;
        real pp = block_sum<real, ONEWARP>((tid < d) ? g[tid] * g[tid] : real(0), red, tid, NT);
        real q = real(0), w = real(0);
        const bool needQ = (pr.obstacle != 0) && (pr.kind == 0 || pr.alph_Q > 0.0);
        if (needQ) {
            real mine = real(0);
            for (int a = tid; a < Ag; a += NT) mine += terrain_agent<real>(pr, s[a * dim], s[a * dim + 1], dim == 3 ? s[a * dim + 2] : real(0));
            q = block_sum<real, ONEWARP>(mine, red, tid, NT);
        }
        if (pr.alph_W != 0.0 && Ag >= 2) {
            const real cut = real(pr.cutW), c2 = real(2 * pr.r * pr.r);
            real mine = real(0);
            const int npairs = Ag * (Ag - 1) / 2;
            for (int p = tid; p < npairs; p += NT) {
                int i = 0, rem = p;
                while (rem >= Ag - 1 - i) { rem -= Ag - 1 - i; ++i; }
                const int j = i + 1 + rem;
                real d2 = real(0);
                for (int c = 0; c < dim; ++c) { real df = s[i * dim + c] - s[j * dim + c]; d2 = r_fma(df, df, d2); }
                real dd = r_sqrt(d2);
                if (dd < cut) {
                    real e = r_exp(-(dd * dd) / c2);
                    if (Ag == 2 || e != real(1)) mine += e;     // the "== 1" rule applies to the A > 2 branch only
                }
            }
            w = block_sum<real, ONEWARP>(mine, red, tid, NT);
        }
        if (tid == 0) {
            real Qret, L;
            if (pr.kind == 0) { Qret = real(pr.alph_Q) * q; L = real(0.5) * pp + Qret; }
            else { Qret = (pr.alph_Q > 0.0) ? q : real(0); L = real(0.5) * pp + real(pr.alph_Q) * Qret; }
            if (pr.alph_W != 0.0) L = L + real(pr.alph_W) * w; else w = real(0);
            real H = -L + pp;
            sc[SC_L] = L; sc[SC_HJ] = r_abs(g[d] - H); sc[SC_Q] = Qret; sc[SC_W] = w;
        }
        cta_sync<ONEWARP>();
    };
    auto rate = [&](int row) -> real {               // dx/dt = -grad_p H
        if (pr.kind != 2) return -g[row];
        int a = row / 12, c = row % 12;
        if (c < 6) return s[a * 12 + 6 + c];
        if (c < 9) { real gg = -qx[5 * a] * qx[5 * a + 1 + (c - 6)]; if (c == 8) gg = gg + real(pr.grav); return -gg; }
        return -(real(0.5) * g[row]);
    };
    auto control = [&](int c) -> real {
        if (pr.kind != 2) return -g[c];
        int a = c / 4, q = c % 4;
        return (q == 0) ? qx[5 * a + 4] : real(-0.5) * g[a * 12 + 8 + q];
    };

    const int nstage = (A.stepper == 4) ? 4 : (A.stepper == 1 ? 1 : 0);
    const bool inter = (A.mode == 2);
    const int ntp1 = A.nt + 1;
    for (long long smp = blockIdx.x; smp < A.n; smp += gridDim.x) {
        if (tid < d) z0[tid] = A.x[smp * d + tid];
        else if (tid < d + 4) z0[tid] = real(0);
        cta_sync<ONEWARP>();
        if (inter) {
            if (tid < d + 4) A.out_b[(smp * (d + 4) + tid) * ntp1] = z0[tid];
            for (int c = tid; c < pr.nctrl; c += NT) A.out_c[(smp * pr.nctrl + c) * ntp1] = real(0);
        }
        for (int k = 0; k < A.nt; ++k) {
            const double* tt = A.times + 5 * k;
            const real hstep = real(tt[4]);
            if (nstage > 0) {
                if (tid < d) s[tid] = z0[tid];
                if (tid == d) s[d] = real(tt[0]);
                cta_sync<ONEWARP>();
            }
            for (int st = 0; st < nstage; ++st) {
                real wgt, cnext, tnext;
                if (nstage == 1) { wgt = real(1); cnext = real(0); tnext = real(0); }
                else if (st == 0) { wgt = real(1.0 / 6.0); cnext = real(0.5); tnext = real(tt[1]); }
                else if (st == 1) { wgt = real(2.0 / 6.0); cnext = real(0.5); tnext = real(tt[1]); }
                else if (st == 2) { wgt = real(2.0 / 6.0); cnext = real(1.0); tnext = real(tt[2]); }
                else { wgt = real(1.0 / 6.0); cnext = real(0); tnext = real(0); }
                const bool lastst = (st == nstage - 1);
                chain(false);
                problem();
                real kk = real(0), z0v = real(0);
                if (tid < d + 4) {
                    kk = hstep * ((tid < d) ? rate(tid) : sc[tid - d]);
                    z0v = z0[tid];
                }
                cta_sync<ONEWARP>();                     // every rate() has read s before s is rewritten
                if (tid < d + 4) {
                    za[tid] = ((st == 0) ? z0v : za[tid]) + wgt * kk;
                    if (!lastst && tid < d) s[tid] = z0v + cnext * kk;
                }
                if (!lastst && tid == d) s[d] = tnext;
                cta_sync<ONEWARP>();
            }
            if (nstage > 0) { real* t = z0; z0 = za; za = t; }
            if (inter) {
                if (tid < d + 4) A.out_b[(smp * (d + 4) + tid) * ntp1 + (k + 1)] = z0[tid];
                if (tid < d) s[tid] = z0[tid];
                if (tid == d) s[d] = real(tt[3]);
                cta_sync<ONEWARP>();
                chain(false);
                if (pr.kind == 2) problem();
                for (int c = tid; c < pr.nctrl; c += NT) A.out_c[(smp * pr.nctrl + c) * ntp1 + (k + 1)] = control(c);
                cta_sync<ONEWARP>();
            }
        }
        // terminal block (OCflow.py:58-90)
        if (tid < d) s[tid] = z0[tid];
        if (tid == d) s[d] = A.t_end;
        cta_sync<ONEWARP>();
        const real phiN = chain(true);
        const real* xt = static_cast<const real*>(pr.xtarget);
        real res = (tid < d) ? (z0[tid] - xt[tid]) : real(0);
        real cG = real(0.5) * block_sum<real, ONEWARP>(res * res, red, tid, NT);
        real hjg = block_sum<real, ONEWARP>((tid < d) ? r_abs(g[tid] - A.alph0 * res) : real(0), red, tid, NT);
        real quad = block_sum<real, ONEWARP>((tid < D) ? s[tid] * qv[tid] : real(0), red, tid, NT);
        real lin = block_sum<real, ONEWARP>((tid < D) ? wb[P.off_cw + tid] * s[tid] : real(0), red, tid, NT);
        if (tid == 0) {
            real phi1 = phiN + real(0.5) * quad + (lin + wb[P.off_cb]);
            real c[7] = {z0[d], cG, z0[d + 1], r_abs(phi1 - A.alph0 * cG), hjg, z0[d + 2], z0[d + 3]};
            if (A.mode == 0) {
                for (int q = 0; q < 7; ++q) A.partials[smp * 8 + q] = (double)c[q];
                A.partials[smp * 8 + 7] = 1.0;
            } else if (A.mode == 1) {
                real* o = A.out_a + smp * 8;
                o[0] = c[0] + A.alph0 * c[1] + A.alph3 * c[2] + A.alph4 * c[3] + A.alph5 * c[4];
                for (int q = 0; q < 7; ++q) o[1 + q] = c[q];
            }
        }
        cta_sync<ONEWARP>();
    }
}

template <typename real, bool WSM, bool ONEWARP>
__global__ void rollout_vec_kernel(const VecArgs<real> A) { rollout_vec_body<real, WSM, ONEWARP>(A); }

// The same kernel built for 1024 threads per block (at most 64 registers per thread).  Left to itself the compiler gives the
// fp64 kernels 96-116 registers, which leaves room for 544-672 threads per block, not for the 1024 that m up to 1024 needs:
// vec_rollout takes this copy for exactly the blocks the other one cannot launch.
template <typename real, bool WSM>
__global__ void __launch_bounds__(1024) rollout_vec_kernel_1024(const VecArgs<real> A) { rollout_vec_body<real, WSM, false>(A); }

template <typename real>
int vec_rollout(const RolloutCall<real>& c) {
    const int d = c.d, m = c.m, nTh = c.nTh;
    const long long n = c.n;
    cudaStream_t st = c.stream;
    VecArgs<real> A;
    memset(&A, 0, sizeof A);
    VecPack<real>& P = A.phi;
    P.d = d; P.D = d + 1; P.m = m; P.nTh = nTh; P.r = c.r; P.h = c.h;
    const int D = d + 1;
    int off = 0;
    auto take = [&](int cnt) { int o = off; off += align_up(cnt, 8); return o; };
    P.off_W1t = take(D * m);
    for (int l = 1; l < nTh; ++l) { P.off_Kft[l] = take(m * m); P.off_Kr[l] = take(m * m); }
    P.off_sym = take(D * D);
    P.off_W4 = take(m * D);
    for (int l = 0; l < nTh; ++l) P.off_b[l] = take(m);
    P.off_w = take(m); P.off_cw = take(D); P.off_cb = take(1);
    P.blob_len = off;
    // shared-memory vectors
    int so = 0;
    auto stake = [&](int cnt) { int o = so; so += align_up(cnt, 8); return o; };
    const int nthreads = std::min(1024, std::max(32, align_up(std::max(std::max(m, D), d + 4), 32)));
    A.o_s = stake(D); A.o_u = stake(m); A.o_u2 = stake(m); A.o_t = stake(std::max(1, nTh - 1) * m); A.o_zb = stake(m);
    A.o_g = stake(D); A.o_q = stake(D); A.o_z0 = stake(d + 4); A.o_za = stake(d + 4); A.o_sc = stake(8); A.o_red = stake(32);
    A.o_qx = stake(5 * std::max(1, c.prob.nAgents)); A.o_w = so;
    const size_t vec_bytes = (size_t)so * sizeof(real);
    const bool wsm = vec_bytes + (size_t)P.blob_len * sizeof(real) <= (size_t)c.smem_limit;
    const size_t smem = vec_bytes + (wsm ? (size_t)P.blob_len * sizeof(real) : 0);

    ScratchBuf blob, partials;
    NOC_CUDA(blob.alloc(sizeof(real) * (size_t)P.blob_len, st));
    NOC_CUDA(cudaMemsetAsync(blob.p, 0, sizeof(real) * (size_t)P.blob_len, st));
    int pgrid = std::min(std::max(1, ceil_div(std::max(m * m, m * D), 256)), 4 * sm_count());
    pack_phi_plain_kernel<real><<<pgrid, 256, 0, st>>>(c.raw, P, blob.as<real>());
    count_launch();
    P.blob = blob.as<real>();
    copy_common(A, c);
    A.stepper = c.stepper; A.times = c.times; A.t_end = (real)c.t_end;
    if (c.mode == NOC_MODE_MEAN) {
        NOC_CUDA(partials.alloc(sizeof(double) * 8 * (size_t)n, st));
        A.partials = partials.as<double>();
    }
    const bool onewarp = wsm && nthreads == 32;
    auto kern = onewarp ? rollout_vec_kernel<real, true, true>
                        : (wsm ? rollout_vec_kernel<real, true, false> : rollout_vec_kernel<real, false, false>);
    cudaFuncAttributes fa;
    NOC_CUDA(cudaFuncGetAttributes(&fa, kern));
    if (nthreads > fa.maxThreadsPerBlock)
        kern = wsm ? rollout_vec_kernel_1024<real, true> : rollout_vec_kernel_1024<real, false>;
    NOC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int grid = (int)std::min<long long>(n, 16LL * sm_count());
    kern<<<grid, nthreads, smem, st>>>(A);
    count_launch();
    NOC_CUDA(cudaGetLastError());
    if (partials.p) {
        int frc = launch_finish(partials.as<double>(), (int)n, c.out_sums, st);
        if (frc) return frc;
        NOC_CUDA(partials.free());
    }
    NOC_CUDA(blob.free());
    return NOC_OK;
}

template int vec_rollout<float>(const RolloutCall<float>&);
template int vec_rollout<double>(const RolloutCall<double>&);

}  // namespace noc
