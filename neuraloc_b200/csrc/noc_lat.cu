// noc_lat.cu — the deployment-latency rollout kernel: ONE THREAD-BLOCK CLUSTER PER SAMPLE, weights resident in (distributed)
// shared memory, several threads per output.  timeDeployment/timeOC.py:76-81 times ONE OCflow(xInit) call: 4 nt + 1
// dependent grad-Phi evaluations of four dependent matrix-vector products each (Phi.py:99-138), i.e. a latency chain, not a
// throughput problem.  The one-CTA-per-sample kernel (noc_vec.cu) runs it with one thread per hidden unit — for the small nets
// that is a single warp fetching ~1 700 instructions per evaluation (7 us), for swarm50 it streams 2.7 MB of weights per
// evaluation from L2 through one SM (49 us).  Here:
//   * every contraction is split over `TPO` threads per output (float4 loads of a padded, conflict-free row slice + a shuffle
//     tree), 256 threads per CTA;
//   * the hidden units (and the gradient components) are partitioned over the NC CTAs of a cluster; each CTA keeps ITS rows of
//     K0, K1, K1', K0', A'A in shared memory for the whole rollout (swarm50: 16 CTAs x 186 KB), so nothing is re-read from L2;
//   * after each contraction the CTAs exchange their slice of the result: every CTA bulk-copies its slice into every peer's
//     copy of the vector through distributed shared memory (cp.async.bulk shared::cta -> shared::cluster, 16 copies issued by
//     16 threads) and each peer's mbarrier counts the bytes -- an all-gather of m or D floats without a cluster-wide barrier
//     (barrier.cluster with its MEMBAR was 35 % of the stall samples of the first version); NC = 1 (all nets up to m = 128)
//     degenerates to __syncthreads();
//   * the per-sample work (calcLHQW, RK update, terminal block) is done redundantly by every CTA of the cluster, so no further
//     exchange is needed; rank 0 writes the outputs.
// nTh = 2 networks (all pretrained ones); anything else, or a shape whose slices do not fit, stays on noc_vec.cu.
#include <cooperative_groups.h>

#include <cstdio>
#include <cstdlib>

#include "noc_launch.cuh"
#include "noc_tc.cuh"

namespace cg = cooperative_groups;

namespace noc {

template <typename real>
struct LatArgs {
    int d, D, m, r, NC, mc, dc, Kp_D, Kp_m;      // mc / dc: hidden units / gradient components per CTA; Kp_*: padded row lengths
    real h;
    const real* blob;                              // [NC][slice_len]: per-rank weight slices (lat_pack_kernel)
    int slice_len;
    int off_W1, off_b0, off_K1f, off_b1, off_w, off_K1r, off_W4, off_sym, off_cw, off_cb;   // element offsets inside a slice
    ProbPack prob;
    const real* x;
    long long n;
    int nt, stepper, mode;
    const double* times;
    real alph0, alph3, alph4, alph5, t_end;
    double* partials;
    real* out_a; real* out_b; real* out_c;
    int o_s, o_u, o_y, o_v, o_t, o_g, o_q, o_z0, o_za, o_sc, o_red, o_qx, o_tmp, o_phi, o_w;   // shared-memory element offsets
};

template <typename real>
__global__ void lat_pack_kernel(const PhiRaw<real> R, const LatArgs<real> A, real* __restrict__ blob) {
    const int D = A.D, m = A.m, mc = A.mc, dc = A.dc, KD = A.Kp_D, Km = A.Kp_m;
    const int rank = blockIdx.y;
    real* B = blob + (size_t)rank * A.slice_len;
    const int stride = gridDim.x * blockDim.x, t0 = blockIdx.x * blockDim.x + threadIdx.x;
    for (int i = t0; i < mc * KD; i += stride) {              // W1[j][k] = K0[u][k]
        const int j = i / KD, k = i % KD, u = rank * mc + j;
        B[A.off_W1 + i] = (u < m && k < D) ? R.K[0][u * D + k] : real(0);
    }
    for (int i = t0; i < mc * Km; i += stride) {              // K1f[j][k] = K1[u][k];  K1r[j][k] = K1[k][u]
        const int j = i / Km, k = i % Km, u = rank * mc + j;
        B[A.off_K1f + i] = (u < m && k < m) ? R.K[1][u * m + k] : real(0);
        B[A.off_K1r + i] = (u < m && k < m) ? R.K[1][k * m + u] : real(0);
    }
    for (int i = t0; i < dc * Km; i += stride) {              // W4[c][k] = K0[k][comp]
        const int c = i / Km, k = i % Km, comp = rank * dc + c;
        B[A.off_W4 + i] = (comp < D && k < m) ? R.K[0][k * D + comp] : real(0);
    }
    for (int i = t0; i < dc * KD; i += stride) {              // sym[c][k] = (A'A)[comp][k]
        const int c = i / KD, k = i % KD, comp = rank * dc + c;
        real s = real(0);
        if (comp < D && k < D) for (int q = 0; q < A.r; ++q) s = r_fma(R.A[q * D + k], R.A[q * D + comp], s);
        B[A.off_sym + i] = s;
    }
    for (int j = t0; j < mc; j += stride) {
        const int u = rank * mc + j;
        B[A.off_b0 + j] = (u < m) ? R.b[0][u] : real(0);
        B[A.off_b1 + j] = (u < m) ? R.b[1][u] : real(0);
        B[A.off_w + j] = (u < m) ? R.w[u] : real(0);
    }
    for (int c = t0; c < dc; c += stride) { const int comp = rank * dc + c; B[A.off_cw + c] = (comp < D) ? R.c_w[comp] : real(0); }
    if (t0 == 0) B[A.off_cb] = R.c_b[0];
}

// out = sum_k W[row][k] in[k] for one output row, split over TPO consecutive lanes (p = my index among them): vector loads of
// 16 bytes, a shuffle tree at the end; every lane of the group returns the sum.  Rows are padded (zeros) to Kp, a multiple of
// 4 with Kp % 32 == 8 so that the groups of a warp hit distinct banks; `in` is readable (zeros) up to Kp.
template <typename real>
__device__ __forceinline__ real gemv_split(const real* __restrict__ Wrow, const real* __restrict__ in, int Kp, int TPO, int p) {
    constexpr int V = 16 / (int)sizeof(real);
    real a0 = real(0), a1 = real(0);
    const int nv = Kp / V;
    int q = p;
    for (; q + TPO < nv; q += 2 * TPO) {
        real w0[V], x0[V], w1[V], x1[V];
        *reinterpret_cast<float4*>(w0) = *reinterpret_cast<const float4*>(Wrow + q * V);
        *reinterpret_cast<float4*>(x0) = *reinterpret_cast<const float4*>(in + q * V);
        *reinterpret_cast<float4*>(w1) = *reinterpret_cast<const float4*>(Wrow + (q + TPO) * V);
        *reinterpret_cast<float4*>(x1) = *reinterpret_cast<const float4*>(in + (q + TPO) * V);
#pragma unroll
        for (int e = 0; e < V; ++e) { a0 = r_fma(w0[e], x0[e], a0); a1 = r_fma(w1[e], x1[e], a1); }
    }
    for (; q < nv; q += TPO) {
        real w0[V], x0[V];
        *reinterpret_cast<float4*>(w0) = *reinterpret_cast<const float4*>(Wrow + q * V);
        *reinterpret_cast<float4*>(x0) = *reinterpret_cast<const float4*>(in + q * V);
#pragma unroll
        for (int e = 0; e < V; ++e) a0 = r_fma(w0[e], x0[e], a0);
    }
    real a = a0 + a1;
    for (int off = TPO >> 1; off > 0; off >>= 1) a += __shfl_xor_sync(0xffffffffu, a, off);
    return a;
}

template <typename real>
__device__ __forceinline__ real lat_block_sum(real v, real* red, int tid, int nthreads) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    __syncthreads();
    if ((tid & 31) == 0) red[tid >> 5] = v;
    __syncthreads();
    real s = real(0);
    for (int w = 0; w < (nthreads >> 5); ++w) s += red[w];
    return s;
}

template <typename real, bool CL>
__global__ void __launch_bounds__(256, 1) rollout_lat_kernel(const LatArgs<real> A) {
    extern __shared__ __align__(16) unsigned char lat_smem[];
    real* sm = reinterpret_cast<real*>(lat_smem);
    constexpr int NT = 256;
    const int tid = threadIdx.x;
    __shared__ ProbPack spr;                            // (a reference to the kernel parameter would be a local-memory copy:
    if (tid == 0) spr = A.prob;                         //  an L2 round trip per field read inside terrain_agent)
    __syncthreads();
    const ProbPack& pr = spr;
    const int d = A.d, D = A.D, m = A.m, NC = A.NC, mc = A.mc, dc = A.dc, KD = A.Kp_D, Km = A.Kp_m;
    unsigned rank = 0, cluster_id = blockIdx.x, nclusters = gridDim.x;
    if (CL) {
        cg::cluster_group cl = cg::this_cluster();
        rank = cl.block_rank();
        cluster_id = blockIdx.x / NC; nclusters = gridDim.x / NC;
    }
    real* s = sm + A.o_s;      real* ub = sm + A.o_u;    real* yb = sm + A.o_y;    real* vb = sm + A.o_v;
    real* t0b = sm + A.o_t;    real* g = sm + A.o_g;     real* qv = sm + A.o_q;    real* sc = sm + A.o_sc;
    real* red = sm + A.o_red;  real* qx = sm + A.o_qx;   real* tmp = sm + A.o_tmp; real* phib = sm + A.o_phi;
    real* z0 = sm + A.o_z0;    real* za = sm + A.o_za;   real* wsl = sm + A.o_w;
    __shared__ __align__(8) unsigned long long gbar[4];   // one mbarrier per exchanged vector (u0, y, v, grad)
    int gphase = 0;
    if (CL && tid == 0) { for (int k = 0; k < 4; ++k) mbar_init(smem_u32(&gbar[k]), 1); fence_mbar_init_cluster(); }
    // my weight slice -> shared memory (once), vectors zeroed (the padded tails are read by gemv_split)
    {
        const real* src = A.blob + (size_t)rank * A.slice_len;
        for (int i = tid; i < A.slice_len; i += NT) wsl[i] = src[i];
        for (int i = tid; i < A.o_w; i += NT) sm[i] = real(0);
    }
    const real* W1 = wsl + A.off_W1;  const real* K1f = wsl + A.off_K1f; const real* K1r = wsl + A.off_K1r;
    const real* W4 = wsl + A.off_W4;  const real* sym = wsl + A.off_sym;
    const real* b0 = wsl + A.off_b0;  const real* b1 = wsl + A.off_b1;   const real* wv = wsl + A.off_w;
    const real* cw = wsl + A.off_cw;
    auto sync_all = [&] {
        if (CL) { cg::this_cluster().sync(); } else { __syncthreads(); }
    };
    sync_all();
    // exchange: the thread that holds output `e` of my slice stores it as element rank*cnt + e of `dst` in EVERY CTA of the
    // cluster (distributed-shared-memory stores), then one cluster barrier publishes the vector (publish_sync)
    // (single CTA: stored directly; cluster: staged in this exchange's own `tmp` slot and bulk-copied to every peer)
    const int tslot = A.o_phi - A.o_tmp >= 0 ? (A.o_phi - A.o_tmp) / 4 : 0;       // elements per tmp slot
    auto put_all = [&](int k, real* dst, int cnt, int e, real v, int second = 0) {
        if (CL) tmp[k * tslot + second * cnt + e] = v; else dst[rank * cnt + e] = v;
    };
    auto publish_sync = [&](int k, real* dst, int cnt, real* dst2 = nullptr) {
        if (CL) {
            fence_async_smem();                          // my tmp writes -> visible to the bulk-copy engine
            __syncthreads();
            const unsigned bytes = (unsigned)(cnt * sizeof(real));
            if (tid == 0) mbar_arrive_expect_tx(smem_u32(&gbar[k]), bytes * NC * (dst2 ? 2 : 1));
            if (tid < NC) {
                const unsigned peer_bar = mapa_shared(smem_u32(&gbar[k]), tid);
                dsmem_bulk_copy(mapa_shared(smem_u32(dst + rank * cnt), tid), smem_u32(tmp + k * tslot), bytes, peer_bar);
                if (dst2) dsmem_bulk_copy(mapa_shared(smem_u32(dst2 + rank * cnt), tid), smem_u32(tmp + k * tslot + cnt), bytes, peer_bar);
            }
            mbar_wait_cluster(smem_u32(&gbar[k]), gphase, 400 + k);
        } else __syncthreads();
    };
    // threads per output for the m-wide and the D-wide contractions
    int TPOm = 1; while (TPOm * 2 * mc <= NT && TPOm < 32) TPOm *= 2;
    int TPOd = 1; while (TPOd * 2 * dc <= NT && TPOd < 32) TPOd *= 2;
    const int om = tid / TPOm, pm = tid % TPOm, od = tid / TPOd, pd = tid % TPOd;
    const int omc = om < mc ? om : mc - 1, odc = od < dc ? od : dc - 1;        // every thread runs the contractions (full-warp shuffles)

    // grad Phi (Phi.py:99-138, nTh = 2) of s = [x, t] -> g (all D components in every CTA); terminal: returns w . u_1 as well
    auto chain = [&](bool terminal) -> real {
        {                                                   // opening layer: o = K0 s + b0 (own units)
            const real pre = gemv_split<real>(W1 + omc * KD, s, KD, TPOm, pm) + b0[omc];
            if (om < mc && pm == 0) { real av, tv; act_tanh(pre, av, tv); put_all(0, ub, mc, om, av); t0b[om] = tv; }
        }
        publish_sync(0, ub, mc);                               // u0, all units
        real part = real(0);
        {                                                   // a1 = K1 u0 + b1 -> y = tanh(a1) w
            const real pre = gemv_split<real>(K1f + omc * Km, ub, Km, TPOm, pm) + b1[omc];
            if (om < mc && pm == 0) {
                if (terminal) { real av, tv; act_tanh(pre, av, tv); part = wv[om] * (ub[rank * mc + om] + A.h * av); put_all(1, yb, mc, om, tv * wv[om]); }
                else put_all(1, yb, mc, om, tanh_only(pre) * wv[om]);
            }
        }
        real phiN = real(0);
        if (terminal) {                                     // w . (u0 + h act(a1)): block sum, then over the cluster
            const real mine = lat_block_sum<real>(part, red, tid, NT);
            if (CL) {
                cg::cluster_group cl = cg::this_cluster();
                if (tid < NC) { real* remote = cl.map_shared_rank(phib, tid); remote[rank] = mine; }
                cl.sync();                                  // (once per rollout) publishes phib
            } else if (tid == 0) phib[0] = mine;
        }
        publish_sync(1, yb, mc);                            // y, all units
        if (terminal) { for (int r = 0; r < NC; ++r) phiN += phib[r]; }
        {                                                   // z1 = w + h K1' y -> v = tanh(o) z1 (own units)
            const real acc = gemv_split<real>(K1r + omc * Km, yb, Km, TPOm, pm);
            if (om < mc && pm == 0) put_all(2, vb, mc, om, t0b[om] * (wv[om] + A.h * acc));
        }
        publish_sync(2, vb, mc);                               // v, all units
        {                                                   // grad = A'A s + K0' v + c_w (own components)
            const real q = gemv_split<real>(sym + odc * KD, s, KD, TPOd, pd);
            const real k0v = gemv_split<real>(W4 + odc * Km, vb, Km, TPOd, pd);
            if (od < dc && pd == 0) { put_all(3, g, dc, od, (q + k0v) + cw[od]); put_all(3, qv, dc, od, q, 1); }
        }
        publish_sync(3, g, dc, qv);
        gphase ^= 1;                            // g and q = A'A s, all components, in every CTA
        return phiN;
    };

    // L, |Phi_t - H|, Q, W -> sc[0..3] from x = s[:d], p = g[:d] (calcLHQW of the three problem classes); as in noc_vec.cu
    const bool needQ = (pr.obstacle != 0) && (pr.kind == 0 || pr.alph_Q > 0.0), hasW = (pr.alph_W != 0.0), posQ = (pr.alph_Q > 0.0);
    const real f_alphQ = real(pr.alph_Q), f_alphW = real(pr.alph_W), f_cut = real(pr.cutW), f_c2 = real(2 * pr.r * pr.r);
    const real f_guard = f_cut * f_cut * real(1.0001);
    const real f_mass = real(pr.mass), f_grav = real(pr.grav), f_uscale = real(-1.0 / (2.0 * pr.mass)), f_cutq = real(2 * pr.r);
    const int p_kind = pr.kind, Ag = pr.nAgents, dim = pr.agentDim, nctrl = pr.nctrl;
    auto problem = [&]() {
        if (p_kind == 2) {                           // Quadcopter.py:86-113 (one thread; a handful of flops)
            if (tid == 0) {
                real H = real(0), Q = real(0), W = real(0);
                real L = f_alphQ * Q;
                if (pr.alph_W > 0.0) {
                    if (Ag == 2) {
                        real d2 = real(0);
                        for (int c = 0; c < 3; ++c) { real df = s[c] - s[12 + c]; d2 = r_fma(df, df, d2); }
                        real dd = r_sqrt(d2);
                        if (dd < f_cutq) W = r_exp(-(dd * dd) / f_c2);
                    }
                    L = L + f_alphW * W;
                }
                for (int a = 0; a < Ag; ++a) {
                    const real* x = s + 12 * a;
                    const real* p = g + 12 * a;
                    real sps, cps, sth, cth, sph, cph;
                    r_sincos(x[3], &sps, &cps); r_sincos(x[4], &sth, &cth); r_sincos(x[5], &sph, &cph);
                    real f7 = sps * sph + cps * sth * cph, f8 = -cps * sph + sps * sth * cph, f9 = cth * cph;
                    real fp = f7 * p[6] + f8 * p[7] + f9 * p[8];
                    real u = f_uscale * fp;
                    real sq = p[9] * p[9] + p[10] * p[10] + p[11] * p[11];
                    L = L + real(2) + u * u + real(0.25) * sq;
                    real um = u / f_mass;
                    real xv = x[6] * p[0] + x[7] * p[1] + x[8] * p[2];
                    real xw = x[9] * p[3] + x[10] * p[4] + x[11] * p[5];
                    H = H - L - xv - xw - um * fp + f_grav * p[8] + real(0.5) * sq;
                    qx[5 * a] = um; qx[5 * a + 1] = f7; qx[5 * a + 2] = f8; qx[5 * a + 3] = f9; qx[5 * a + 4] = u;
                }
                sc[SC_L] = L; sc[SC_HJ] = r_abs(g[d] - H); sc[SC_Q] = Q; sc[SC_W] = W;
            }
            __syncthreads();
            return;
        }
        real ppm = real(0), qm = real(0), wm = real(0);
        for (int c = tid; c < d; c += NT) ppm = r_fma(g[c], g[c], ppm);
        if (needQ)
            for (int a = tid; a < Ag; a += NT) qm += terrain_agent<real>(pr, s[a * dim], s[a * dim + 1], dim == 3 ? s[a * dim + 2] : real(0));
        if (hasW && Ag >= 2) {
            // pairs (i, j > i): thread group `gi` takes the rows gi and A-2-gi (together A pairs: balanced), j strided inside the
            // group -- no index decoding, at most ceil(A / TPR) pairs per thread
            const int nfold = Ag / 2;                                 // row pairs (gi, A-2-gi); the middle row of an even count alone
            int TPR = 1; while (TPR * 2 * nfold <= NT && TPR < 32) TPR *= 2;
            for (int gi = tid / TPR; gi < nfold; gi += NT / TPR)
                for (int t = tid % TPR; t < Ag; t += TPR) {
                    // the t-th pair of the folded row: first the A-1-gi pairs of row gi, then the gi+1 pairs of row A-2-gi
                    int i, j;
                    if (t < Ag - 1 - gi) { i = gi; j = gi + 1 + t; }
                    else {
                        if (2 * gi == Ag - 2) continue;               // the middle row is its own partner: counted once
                        i = Ag - 2 - gi; j = i + 1 + (t - (Ag - 1 - gi));
                    }
                    real d2 = real(0);
                    for (int c = 0; c < dim; ++c) { real df = s[i * dim + c] - s[j * dim + c]; d2 = r_fma(df, df, d2); }
                    if (d2 < f_guard) {                         // (widened squared cut-off first: the exact test needs a sqrt)
                        real dd = r_sqrt(d2);
                        if (dd < f_cut) {
                            real e = r_exp(-(dd * dd) / f_c2);
                            if (Ag == 2 || e != real(1)) wm += e;   // the "== 1" rule applies to the A > 2 branch only
                        }
                    }
                }
        }
        // one block reduction for the three sums (fixed shuffle tree + fixed warp order: deterministic)
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            ppm += __shfl_xor_sync(0xffffffffu, ppm, off); qm += __shfl_xor_sync(0xffffffffu, qm, off); wm += __shfl_xor_sync(0xffffffffu, wm, off);
        }
        if ((tid & 31) == 0) { red[tid >> 5] = ppm; red[8 + (tid >> 5)] = qm; red[16 + (tid >> 5)] = wm; }
        __syncthreads();
        real pp = real(0), q = real(0), w = real(0);
        if (tid == 0)
            for (int k8 = 0; k8 < NT / 32; ++k8) { pp += red[k8]; q += red[8 + k8]; w += red[16 + k8]; }
        if (tid == 0) {
            real Qret, L;
            if (p_kind == 0) { Qret = f_alphQ * q; L = real(0.5) * pp + Qret; }
            else { Qret = posQ ? q : real(0); L = real(0.5) * pp + f_alphQ * Qret; }
            if (hasW) L = L + f_alphW * w; else w = real(0);
            real H = -L + pp;
            sc[SC_L] = L; sc[SC_HJ] = r_abs(g[d] - H); sc[SC_Q] = Qret; sc[SC_W] = w;
        }
        __syncthreads();
    };
    auto rate = [&](int row) -> real {               // dx/dt = -grad_p H
        if (p_kind != 2) return -g[row];
        int a = row / 12, c = row % 12;
        if (c < 6) return s[a * 12 + 6 + c];
        if (c < 9) { real gg = -qx[5 * a] * qx[5 * a + 1 + (c - 6)]; if (c == 8) gg = gg + f_grav; return -gg; }
        return -(real(0.5) * g[row]);
    };
    auto control = [&](int c) -> real {
        if (p_kind != 2) return -g[c];
        int a = c / 4, q = c % 4;
        return (q == 0) ? qx[5 * a + 4] : real(-0.5) * g[a * 12 + 8 + q];
    };

    const int nstage = (A.stepper == 4) ? 4 : (A.stepper == 1 ? 1 : 0);
    const bool inter = (A.mode == 2), writer = (rank == 0);
    const int ntp1 = A.nt + 1;
    for (long long smp = cluster_id; smp < A.n; smp += nclusters) {
        for (int c = tid; c < d + 4; c += NT) z0[c] = (c < d) ? A.x[smp * d + c] : real(0);
        __syncthreads();
        if (inter && writer) {
            for (int c = tid; c < d + 4; c += NT) A.out_b[(smp * (d + 4) + c) * ntp1] = z0[c];
            for (int c = tid; c < nctrl; c += NT) A.out_c[(smp * nctrl + c) * ntp1] = real(0);
        }
        for (int k = 0; k < A.nt; ++k) {
            const double* tt = A.times + 5 * k;
            const real hstep = real(tt[4]);
            const real ts[4] = {real(tt[0]), real(tt[1]), real(tt[2]), real(tt[3])};
            if (nstage > 0) {
                for (int c = tid; c <= d; c += NT) s[c] = (c < d) ? z0[c] : ts[0];
                __syncthreads();
            }
            for (int st = 0; st < nstage; ++st) {
                real wgt, cnext, tnext;
                if (nstage == 1) { wgt = real(1); cnext = real(0); tnext = real(0); }
                else if (st == 0) { wgt = real(1.0 / 6.0); cnext = real(0.5); tnext = ts[1]; }
                else if (st == 1) { wgt = real(2.0 / 6.0); cnext = real(0.5); tnext = ts[1]; }
                else if (st == 2) { wgt = real(2.0 / 6.0); cnext = real(1.0); tnext = ts[2]; }
                else { wgt = real(1.0 / 6.0); cnext = real(0); tnext = real(0); }
                const bool lastst = (st == nstage - 1);
                chain(false);
                problem();
                real kk = real(0), z0v = real(0);            // (d + 4 <= 256 components: one per thread)
                if (tid < d + 4) {
                    kk = hstep * ((tid < d) ? rate(tid) : sc[tid - d]);
                    z0v = z0[tid];
                }
                __syncthreads();                             // every rate() has read s before s is rewritten
                if (tid < d + 4) {
                    za[tid] = ((st == 0) ? z0v : za[tid]) + wgt * kk;
                    if (!lastst && tid < d) s[tid] = z0v + cnext * kk;
                }
                if (!lastst && tid == d) s[d] = tnext;
                __syncthreads();
            }
            if (nstage > 0) { real* t = z0; z0 = za; za = t; }
            if (inter) {
                if (writer) for (int c = tid; c < d + 4; c += NT) A.out_b[(smp * (d + 4) + c) * ntp1 + (k + 1)] = z0[c];
                for (int c = tid; c <= d; c += NT) s[c] = (c < d) ? z0[c] : ts[3];
                __syncthreads();
                chain(false);
                if (p_kind == 2) problem();
                if (writer) for (int c = tid; c < nctrl; c += NT) A.out_c[(smp * nctrl + c) * ntp1 + (k + 1)] = control(c);
                __syncthreads();
            }
        }
        // terminal block (OCflow.py:58-90)
        for (int c = tid; c <= d; c += NT) s[c] = (c < d) ? z0[c] : A.t_end;
        __syncthreads();
        const real phiN = chain(true);
        const real* xt = static_cast<const real*>(pr.xtarget);
        const real res = (tid < d) ? (z0[tid] - xt[tid]) : real(0);
        const real cG = real(0.5) * lat_block_sum<real>(res * res, red, tid, NT);
        const real hjg = lat_block_sum<real>((tid < d) ? r_abs(g[tid] - A.alph0 * res) : real(0), red, tid, NT);
        const real quad = lat_block_sum<real>((tid < D) ? s[tid] * qv[tid] : real(0), red, tid, NT);
        // c_w . s: every CTA holds only its slice of c_w; g - (K0'v + A'A s) would be circular, so gather it through tmp
        real lin;
        {
            real mine = real(0);
            if (tid < dc && (int)rank * dc + tid < D) mine = cw[tid] * s[rank * dc + tid];
            const real part = lat_block_sum<real>(mine, red, tid, NT);
            if (CL) {
                cg::cluster_group cl = cg::this_cluster();
                if (tid < NC) cl.map_shared_rank(phib, tid)[NC + rank] = part;
                cl.sync();
                lin = real(0);
                for (int r = 0; r < NC; ++r) lin += phib[NC + r];
            } else lin = part;
        }
        if (tid == 0 && writer) {
            real phi1 = phiN + real(0.5) * quad + (lin + wsl[A.off_cb]);
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
        sync_all();                                            // phib / vectors are reused by the next sample
    }
}

static inline int lat_pad(int K, int elt) {       // multiple of 16 bytes, and (in 4-byte words) congruent 8 mod 32
    const int V = 16 / elt;
    int Kp = (K + V - 1) / V * V;
    while ((Kp * elt / 4) % 32 != 8) Kp += V;
    return Kp;
}

// returns NOC_OK and *took = true when the cluster kernel ran; *took = false means "not applicable, use noc_vec.cu"
template <typename real>
int lat_rollout(const RolloutCall<real>& c, bool* took) {
    const int d = c.d, m = c.m;
    const long long n = c.n;
    cudaStream_t st = c.stream;
    *took = false;
    if (c.nTh != 2 || d + 4 > 256 || getenv("NOC_NO_LAT")) return NOC_OK;
    LatArgs<real> A;
    memset(&A, 0, sizeof A);
    const int D = d + 1, elt = (int)sizeof(real);
    A.d = d; A.D = D; A.m = m; A.r = c.r; A.h = c.h;
    A.Kp_D = lat_pad(D, elt); A.Kp_m = lat_pad(m, elt);
    int NC = 0;
    size_t smem = 0;
    auto plan = [&](int nc) -> bool {                          // slice + vector layout for a cluster of nc CTAs; true if it fits
        const int V = 16 / elt;                               // slices are bulk-copied: multiples of 16 bytes
        const int mc = (nc > 1) ? align_up(ceil_div(m, nc), V) : m, dc = (nc > 1) ? align_up(ceil_div(D, nc), V) : D;
        if (mc > 256 || 2 * dc > 256) return false;
        int off = 0;
        auto take = [&](int cnt) { int o = off; off += align_up(cnt, 8); return o; };
        A.off_W1 = take(mc * A.Kp_D); A.off_K1f = take(mc * A.Kp_m); A.off_K1r = take(mc * A.Kp_m); A.off_W4 = take(dc * A.Kp_m);
        A.off_sym = take(dc * A.Kp_D); A.off_b0 = take(mc); A.off_b1 = take(mc); A.off_w = take(mc); A.off_cw = take(dc); A.off_cb = take(1);
        A.slice_len = off;
        int so = 0;
        auto stake = [&](int cnt) { int o = so; so += align_up(cnt, 8); return o; };
        const int mfull = mc * nc, dfull = dc * nc;
        A.o_s = stake(std::max(A.Kp_D, dfull)); A.o_u = stake(std::max(A.Kp_m, mfull)); A.o_y = stake(std::max(A.Kp_m, mfull));
        A.o_v = stake(std::max(A.Kp_m, mfull)); A.o_t = stake(mc); A.o_g = stake(std::max(A.Kp_D, dfull)); A.o_q = stake(std::max(A.Kp_D, dfull));
        A.o_z0 = stake(d + 4); A.o_za = stake(d + 4); A.o_sc = stake(8); A.o_red = stake(32); A.o_qx = stake(5 * std::max(1, c.prob.nAgents));
        A.o_tmp = stake(4 * align_up(std::max(mc, 2 * dc), 8)); A.o_phi = stake(2 * 16); A.o_w = so;      // four exchange slots
        smem = (size_t)(so + A.slice_len) * elt;
        if (smem > (size_t)c.smem_limit) return false;
        NC = nc; A.mc = mc; A.dc = dc;
        return true;
    };
    int first = 1;
    if (const char* e = getenv("NOC_LAT_NC")) { const int want = atoi(e); if (want >= 1 && want <= 16 && (want & (want - 1)) == 0) first = want; }
    for (int nc = first; nc <= 16 && NC == 0; nc *= 2) plan(nc);       // the smallest cluster whose slices fit
    if (NC == 0) return NOC_OK;
    A.NC = NC;
    auto kern = (NC > 1) ? rollout_lat_kernel<real, true> : rollout_lat_kernel<real, false>;
    NOC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (NC > 8) {
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess) { (void)cudaGetLastError(); return NOC_OK; }
    }
    // how many clusters can run at once (for the grid); 0 = this cluster size cannot be scheduled: leave it to noc_vec.cu
    int nclusters = (int)std::min<long long>(n, std::max(1, sm_count() / NC));
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof cfg);
    cudaLaunchAttribute attr[1];
    cfg.gridDim = dim3(nclusters * NC); cfg.blockDim = dim3(256); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    if (NC > 1) {
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = NC; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        int maxc = 0;
        if (cudaOccupancyMaxActiveClusters(&maxc, kern, &cfg) != cudaSuccess || maxc < 1) { (void)cudaGetLastError(); return NOC_OK; }
        nclusters = (int)std::min<long long>(n, maxc);
        cfg.gridDim = dim3(nclusters * NC);
    }
    ScratchBuf blob, partials;
    NOC_CUDA(blob.alloc(sizeof(real) * (size_t)A.slice_len * NC, st));
    lat_pack_kernel<real><<<dim3(std::max(1, std::min(64, ceil_div(A.mc * A.Kp_m, 256))), NC), 256, 0, st>>>(c.raw, A, blob.as<real>());
    count_launch();
    A.blob = blob.as<real>();
    copy_common(A, c);
    A.stepper = c.stepper; A.times = c.times; A.t_end = (real)c.t_end;
    if (c.mode == NOC_MODE_MEAN) {
        NOC_CUDA(partials.alloc(sizeof(double) * 8 * (size_t)n, st));
        A.partials = partials.as<double>();
    }
    if (getenv("NOC_DEBUG")) fprintf(stderr, "[noc] latency kernel: cluster of %d, %d units + %d components per CTA, smem %zu B, %d clusters\n", NC, A.mc, A.dc, smem, nclusters);
    NOC_CUDA(cudaLaunchKernelEx(&cfg, kern, A));
    count_launch();
    NOC_CUDA(cudaGetLastError());
    if (partials.p) {
        int frc = launch_finish(partials.as<double>(), (int)n, c.out_sums, st);
        if (frc) return frc;
        NOC_CUDA(partials.free());
    }
    NOC_CUDA(blob.free());
    *took = true;
    return NOC_OK;
}

template int lat_rollout<float>(const RolloutCall<float>&, bool*);
template int lat_rollout<double>(const RolloutCall<double>&, bool*);

}  // namespace noc
