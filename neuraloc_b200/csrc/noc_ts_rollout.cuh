// noc_ts_rollout.cuh — tensor-core rollout for WIDE value networks (swarm50: d = 150, m = 512, nTh = 2; src/Phi.py:99-138,
// src/problem/SwarmTraj.py:68-164, src/OCflow.py:7-184), fp32 in / fp32 out: CTA pairs (cta_group::2), TMA-streamed
// weights, activations handed from the epilogue warps to the tensor core chunk by chunk.
//
// Why a different kernel from noc_tc_rollout.cuh: at m = 512 nothing is resident.  One hidden vector of one sample is 2 KB in
// fp32, so a 128-sample tile needs 256 KB for ONE accumulator (all of TMEM) and 256 KB for ONE split activation operand
// (more than shared memory); K1 alone is 1 MB as split 16-bit planes.  So:
//   * a CTA PAIR shares each tile of 128 samples: every MMA is cta_group::2 with M = 128 (64 samples from each CTA), N = 256;
//     each CTA's TMEM then holds [64 samples x 512 units] in 256 columns (2x2 layout: lanes 0-63 = columns [0,N/2) of the
//     instruction, lanes 64-127 = [N/2,N)), i.e. TWO accumulator regions R0 / R1 that the four contractions ping-pong between
//     (GEMM-1 -> R0, GEMM-2 -> R1, GEMM-3 -> R0, GEMM-4 -> R1), so the epilogue of one contraction overlaps the MMAs of the next;
//   * the weights stream from L2 through a ring of 16 KB stages filled by cp.async.bulk.tensor (TMA, 2-SM form: each CTA loads
//     its half of B's N rows, both report to the leader's mbarrier); the stream order is fixed (GEMM-1..4 of every evaluation),
//     pre-packed once per call as split fp16 planes in exactly the shared-memory image each stage needs;
//   * an epilogue turns 32 accumulator columns per thread into the next contraction's A operand (activation, fp16 split,
//     canonical no-swizzle UMMA layout) and hands over K-slabs of 128 units through mbarriers: the MMA issuer consumes slab i
//     while the epilogue warps produce slab i+1 (two slab buffers);
//   * tanh(o) (needed again after GEMM-3), the step-start state z0 and the RK accumulator live in a per-CTA global scratch
//     (L2-resident, coalesced [row][64 samples]); the stage input x lives in shared memory in fp32 (pair distances need it exact).
//
// Precision: every fp32 operand is split into TWO fp16 terms (hi + lo, ~2^-23 relative; weights are pre-scaled per matrix by a
// power of two so that their lo parts stay in fp16's normal range; the scale is undone exactly in the epilogue) and each logical
// product is three MMAs (hi*hi, hi*lo, lo*hi; the dropped lo*lo term is O(2^-24)) into one fp32 TMEM accumulator.
//
// Warp roles (320 threads): warps 0-7 epilogue / per-sample work (4 threads per sample: TMEM lane half x column half),
// warp 8 TMA producer (both CTAs), warp 9 MMA issuer (leader CTA only; allocates TMEM in both).  (10 warps leave 168 registers
// per thread; handing the two service warps' registers to the epilogue warps with setmaxnreg made ptxas spill MORE.)
#pragma once
#include <cuda.h>

#include <type_traits>

#include "noc_launch.cuh"
#include "noc_tc.cuh"
#include "noc_tc_rollout.cuh"

namespace noc {

template <int NA_>
struct TsShape {
    static constexpr int NA = NA_, DIM = 3;
    static constexpr int d = NA * DIM, D = d + 1, NZ = d + 4;
    static constexpr int KS = ((d + 2 + 31) / 32) * 32;       // K of the stage-input operand S = [x, t, 1, 0..]; also N of GEMM-4
    static constexpr int CPT = KS / 4;                         // gradient components per thread (4 threads per sample)
    static constexpr int MP = 512;                             // hidden width, zero-padded
    static constexpr int NT = 320;
    static constexpr int NK1 = KS / 16;                        // k-steps of GEMM-1 (and of S.symb' in GEMM-4)
    static constexpr int NS1 = 2 * (KS / 32);                  // stages: GEMM-1 = [nh][2 k-steps]
    static constexpr int NS2 = 32;                             // GEMM-2 / GEMM-3 = [slab][k-step]
    static constexpr int NK4 = 32 + NK1;                       // k-steps of GEMM-4 = V.K0 (32) then S.symb' (NK1)
    static constexpr int NS4 = (NK4 + 2) / 3;                  // three k-steps per stage
    static constexpr int NSTAGE = NS1 + 2 * NS2 + NS4;         // stages per grad-Phi evaluation
    static constexpr int STAGE_BYTES = 16384, NSLOT = 4;
    static constexpr int SBO_S = (KS / 8) * 128, PLANE_S = 8 * SBO_S;     // S operand: [64 x KS] per plane
    static constexpr int G4_PLANE = (KS / 2) * 32;                         // one k-step of GEMM-4's B: [KS/2 rows x 16 k]
    static_assert(CPT == 32 || CPT == 40, "gradient components per thread: 32 or 40");
    static_assert(3 * 2 * G4_PLANE <= STAGE_BYTES, "GEMM-4 stage");
    // shared-memory map (bytes from the 1024-aligned base)
    static constexpr int oX = 0;                                // 2 slabs x (hi, lo) x [64 x 128] fp16
    static constexpr int oS = oX + 2 * 32768;
    static constexpr int oW = oS + 2 * PLANE_S;
    static constexpr int oXS = oW + NSLOT * STAGE_BYTES;        // x of the current stage input, fp32 [d][64]
    static constexpr int oRED = oXS + d * 64 * 4;               // [6][4][64] partial sums + [64] Phi_t
    static constexpr int oB1 = oRED + (6 * 4 + 1) * 64 * 4;
    static constexpr int oWV = oB1 + MP * 4;
    static constexpr int oSRED = oWV + MP * 4;                  // [2][8] per-warp cost sums
    static constexpr int oBAR = oSRED + 192;                    // + [8] running sums of this CTA
    static constexpr int SMEM = oBAR + 32 * 8;
    // per-CTA global scratch (floats): tanh(o) [MP][64], u0 at the terminal evaluation [MP][64], z0 [d][64], RK accumulator [d][64]
    static constexpr int SCR = 2 * MP * 64 + 2 * d * 64;
};

struct TsArgs {
    int m;
    float h;
    const float *b1, *w, *c_w, *c_b;        // reference layout, fp32, device
    const float* scales;                    // device [6]: s1, s2, s4 (powers of two) and their reciprocals
    ProbPack prob;
    const float* x;
    long long n;
    int nt, mode;
    const TcEval* evals;
    int nevals;
    float alph0, alph3, alph4, alph5;
    double* partials;
    float *out_a, *out_b, *out_c;
    float* stage;                            // intermediates: tile-major staging [tile][step][row][128 samples] (coalesced), or NULL
    float* scratch;
    int ntiles;                              // tiles of 128 samples, one per CTA pair per round
    // problem constants rounded to fp32 on the host (a double compare / convert in the loop costs ~50x an fp32 instruction here)
    float f_alphQ, f_alphW, f_cut, f_c2, thr[10];
    int hasQ, hasW, posQ, obstacle, training;
    long long* trace;                        // NOC_TS_TRACE: [20 roles][256][2] (tag, clock) of blocks 0-1 during evaluation 5, or NULL
};

// hidden unit of k-index kk (0..127) of activation slab ji (0..3): the order in which the epilogue threads produce units
// (thread group gq = kk / 32 owns TMEM columns of instruction half gq / 2, lane half gq % 2)
__host__ __device__ inline int ts_unit(int ji, int kk) {
    const int gq = kk >> 5;
    return 256 * (gq >> 1) + 128 * (gq & 1) + 32 * ji + (kk & 31);
}

// ------------------------------------------------------------------------------------------------------------------
// weight packing: reference layout -> the streamed blob [rank][stage][16 KB] of split fp16 planes (see the file header)
// ------------------------------------------------------------------------------------------------------------------
struct TsPackArgs {
    int m, D, r;
    const float *K0, *b0, *K1, *A, *c_w;
    unsigned* maxbits;                      // [3] running max |.| of K0b, K1, (K0 | symb) as float bits
    float* scales;                          // [9]: scales, reciprocals, accumulate-bias corrections (ulps * 2^-23)
    unsigned char* blob;
    float bias[3];                          // relative compensation of the accumulate bias of GEMM-1, GEMM-2/3, GEMM-4
};

__device__ __forceinline__ float ts_symb(const TsPackArgs& P, int comp, int k) {      // [A'A | c_w] (Phi.py:110,136)
    if (comp >= P.D) return 0.f;
    if (k < P.D) { float s = 0.f; for (int q = 0; q < P.r; ++q) s = fmaf(P.A[q * P.D + k], P.A[q * P.D + comp], s); return s; }
    return (k == P.D) ? P.c_w[comp] : 0.f;
}

static __global__ void ts_absmax_kernel(const TsPackArgs P) {
    float m1 = 0.f, m2 = 0.f, m4 = 0.f;
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    for (int i = tid; i < P.m * P.D; i += nth) { const float v = fabsf(P.K0[i]); m1 = fmaxf(m1, v); m4 = fmaxf(m4, v); }
    for (int i = tid; i < P.m; i += nth) m1 = fmaxf(m1, fabsf(P.b0[i]));
    for (int i = tid; i < P.m * P.m; i += nth) m2 = fmaxf(m2, fabsf(P.K1[i]));
    for (int i = tid; i < P.D * (P.D + 1); i += nth) m4 = fmaxf(m4, fabsf(ts_symb(P, i / (P.D + 1), i % (P.D + 1))));
    for (int off = 16; off > 0; off >>= 1) {
        m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, off));
        m2 = fmaxf(m2, __shfl_xor_sync(0xffffffffu, m2, off));
        m4 = fmaxf(m4, __shfl_xor_sync(0xffffffffu, m4, off));
    }
    if ((threadIdx.x & 31) == 0) {          // non-negative floats order like their bit patterns
        atomicMax(P.maxbits + 0, __float_as_uint(m1));
        atomicMax(P.maxbits + 1, __float_as_uint(m2));
        atomicMax(P.maxbits + 2, __float_as_uint(m4));
    }
}
static __global__ void ts_scales_kernel(const TsPackArgs P) {
    if (threadIdx.x < 3) {
        const float mx = __uint_as_float(P.maxbits[threadIdx.x]);
        float s = 1.f;
        if (mx > 0.f && mx < 3.0e38f) s = exp2f((float)(13 - ilogbf(mx)));      // scaled max in [2^13, 2^14)
        P.scales[threadIdx.x] = s;
#ifdef NOC_TS_ULP_UNBIAS
        P.scales[3 + threadIdx.x] = 1.f / s;
        P.scales[6 + threadIdx.x] = P.bias[threadIdx.x] * (0.22f / 0.159f);        // relative shrink -> ulps * 2^-23
#else
        P.scales[3 + threadIdx.x] = (1.f / s) * (1.f + P.bias[threadIdx.x]);
        P.scales[6 + threadIdx.x] = 0.f;
#endif
    }
}

template <class SH>
static __global__ void __launch_bounds__(256) ts_pack_kernel(const TsPackArgs P) {
    constexpr int KS = SH::KS;
    const int gid = blockIdx.x * blockDim.x + threadIdx.x;
    const int j = gid & 511, st = (gid >> 9) % SH::NSTAGE, c = (gid >> 9) / SH::NSTAGE;
    if (c >= 2) return;
    unsigned char* stage = P.blob + ((size_t)c * SH::NSTAGE + st) * SH::STAGE_BYTES;
    const float s1 = P.scales[0], s2 = P.scales[1], s4 = P.scales[2];
    const int m = P.m, D = P.D;
    float v[8];
    int off_hi, lo_delta;
    if (st < SH::NS1) {                                      // GEMM-1: B[n = unit][k] = K0b = [K0 | b0 | 0]
        const int nh = st / (KS / 32), sp = st % (KS / 32);
        const int n = j >> 2, kc = j & 3, u = 256 * nh + 128 * c + n;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int k = 32 * sp + 8 * kc + e;
            v[e] = (u < m) ? (k < D ? P.K0[u * D + k] : (k == D ? P.b0[u] : 0.f)) * s1 : 0.f;
        }
        off_hi = (n >> 3) * 512 + kc * 128 + (n & 7) * 16; lo_delta = 8192;
    } else if (st < SH::NS1 + 2 * SH::NS2) {                 // GEMM-2: K1[u_out][u_in];  GEMM-3: K1[u_in][u_out]
        const bool fwd = st < SH::NS1 + SH::NS2;
        const int s2i = (st - SH::NS1) % SH::NS2, ji = s2i >> 3, ks = s2i & 7;
        const int nh = j >> 8, n = (j >> 1) & 127, kc = j & 1, uo = 256 * nh + 128 * c + n;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int ui = ts_unit(ji, 16 * ks + 8 * kc + e);
            v[e] = (uo < m && ui < m) ? (fwd ? P.K1[uo * m + ui] : P.K1[ui * m + uo]) * s2 : 0.f;
        }
        off_hi = nh * 8192 + (n >> 3) * 256 + kc * 128 + (n & 7) * 16; lo_delta = 4096;
    } else {                                                 // GEMM-4: B[n = component][k]: K0[u_in][comp] then [A'A | c_w][comp][k]
        const int s4i = st - SH::NS1 - 2 * SH::NS2;
        const int per = (KS / 2) * 2;                        // chunks per k-step plane
        if (j >= 3 * per) return;
        const int t = j / per, jj = j % per, n = jj >> 1, kc = jj & 1, g = 3 * s4i + t, comp = (KS / 2) * c + n;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            float val = 0.f;
            if (g < 32) { const int ui = ts_unit(g >> 3, 16 * (g & 7) + 8 * kc + e); if (ui < m && comp < D) val = P.K0[ui * D + comp]; }
            else if (g < SH::NK4) val = ts_symb(P, comp, 16 * (g - 32) + 8 * kc + e);
            v[e] = val * s4;
        }
        off_hi = (t * 2) * SH::G4_PLANE + (n >> 3) * 256 + kc * 128 + (n & 7) * 16; lo_delta = SH::G4_PLANE;
    }
    uint4 hi, lo;
    split2_f16(v[0], v[1], hi.x, lo.x); split2_f16(v[2], v[3], hi.y, lo.y);
    split2_f16(v[4], v[5], hi.z, lo.z); split2_f16(v[6], v[7], hi.w, lo.w);
    *reinterpret_cast<uint4*>(stage + off_hi) = hi;
    *reinterpret_cast<uint4*>(stage + off_hi + lo_delta) = lo;
}

// ------------------------------------------------------------------------------------------------------------------
// the rollout kernel
// ------------------------------------------------------------------------------------------------------------------
enum { TS_WFULL = 0, TS_WEMPTY = 4, TS_XFULL = 8, TS_XEMPTY = 10, TS_SFULL = 12, TS_ACC = 13, TS_NBAR = 18 };

// three MMAs of one k-step: hi*hi, hi*lo, lo*hi (planes are `alo` / `blo` 16-byte units after the hi planes)
__device__ __forceinline__ void ts_mma3(unsigned dt, unsigned long long a, unsigned alo, unsigned long long b, unsigned blo, unsigned idesc, int acc) {
    umma2_f16(dt, a, b, idesc, acc);
    umma2_f16(dt, a, b + blo, idesc, 1);
    umma2_f16(dt, a + alo, b, idesc, 1);
}

// Accumulate-bias compensation.  The tensor core's fp32 accumulate rounds toward zero (below 1/4 ulp) on every MMA, so a
// K = 512 contraction issued as 96 accumulating MMAs comes out ~21 ulp SHORT, the same way for every sample -- a systematic
// error that shows up 1:1 in the mean terminal cost G.  Measured: -0.137 ulp per MMA on bf16 data (scripts/tc_bias_probe.py),
// -0.22 ulp per MMA = a mean relative shrink of 1.89e-8 per MMA for this kernel's fp16 planes, constant to +-1.5 % across step
// counts, input distributions and networks (scripts/ts_bias_robust.py).  The mean shrink of each contraction is undone by
// folding (1 + 1.89e-8 * #MMAs) into the reciprocal weight scale its epilogue applies anyway (no extra instruction); the
// per-element variant below (add kappa ulps away from zero; -DNOC_TS_ULP_UNBIAS) measured the same residual.
#ifdef NOC_TS_ULP_UNBIAS
__device__ __forceinline__ float ts_unbias(float v, float kq) {
    return fmaf(__uint_as_float(__float_as_uint(v) & 0xff800000u), kq, v);       // v + sign(v) * kappa * ulp(v), kq = kappa * 2^-23
}
#else
__device__ __forceinline__ float ts_unbias(float v, float) { return v; }
#endif

// Interaction cost of one sample (SwarmTraj.py:147-162): this thread owns the agent rows i = part, part + 4, ... and pairs
// each with every j > i.  The rows are processed in blocks of up to four (i0, i0 + 4, i0 + 8, i0 + 12) so that one load of
// agent j serves four pairs -- eight warps walking 1225 pairs per sample with three shared-memory loads per pair were bound
// by the shared-memory pipe (which the tensor core reads its operands through as well).  Per block only the minimum squared
// distance is tracked, branch-free; a block with a pair inside the slightly widened cut-off (rare, and the same blocks in every
// lane: the samples of a tile are perturbations of one formation) is redone exactly -- sqrt, cut-off, exp, the "== 1" rule --
// row by row in the reference's (i, j) order.  ts_pairs() runs the blocks whose first row lies in [ib, ie).
__device__ __forceinline__ float ts_pair_block(const float* xs, int A, int i0, int nr, float cut, float c2, float guard, float w) {
    float xi[4][3];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int i = (r < nr) ? i0 + 4 * r : i0;
#pragma unroll
        for (int c = 0; c < 3; ++c) xi[r][c] = xs[(3 * i + c) * 64];
    }
    const int ilast = i0 + 4 * (nr - 1);
    float dm[4] = {guard, guard, guard, guard};            // one running minimum per row: four short dependency chains
    int j = i0 + 1;
    for (; j <= ilast && j < A; ++j) {                      // j between the rows of the block: row r pairs with j only if j > i_r
        const float xj0 = xs[(3 * j) * 64], xj1 = xs[(3 * j + 1) * 64], xj2 = xs[(3 * j + 2) * 64];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const float d0 = xi[r][0] - xj0, d1 = xi[r][1] - xj1, d2c = xi[r][2] - xj2;
            const float d2 = fmaf(d2c, d2c, fmaf(d1, d1, fmaf(d0, d0, 0.f)));
            if (r < nr && j > i0 + 4 * r) dm[r] = fminf(dm[r], d2);
        }
    }
#pragma unroll 1
    for (; j + 4 <= A; j += 4) {                           // j beyond the last row: every row of the block pairs with it
        float xj[4][3];
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int c = 0; c < 3; ++c) xj[u][c] = xs[(3 * (j + u) + c) * 64];
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const float d0 = xi[r][0] - xj[u][0], d1 = xi[r][1] - xj[u][1], d2c = xi[r][2] - xj[u][2];
                dm[r] = fminf(dm[r], fmaf(d2c, d2c, fmaf(d1, d1, fmaf(d0, d0, 0.f))));   // rows r >= nr repeat row 0: harmless
            }
    }
    for (; j < A; ++j) {
        const float xj0 = xs[(3 * j) * 64], xj1 = xs[(3 * j + 1) * 64], xj2 = xs[(3 * j + 2) * 64];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const float d0 = xi[r][0] - xj0, d1 = xi[r][1] - xj1, d2c = xi[r][2] - xj2;
            dm[r] = fminf(dm[r], fmaf(d2c, d2c, fmaf(d1, d1, fmaf(d0, d0, 0.f))));
        }
    }
    // exact pass over the rows that have a pair inside the guard (four distances per branch), in (i, j) order
#pragma unroll 1
    for (int r = 0; r < nr; ++r) {
        const float dmr = (r == 0) ? dm[0] : (r == 1 ? dm[1] : (r == 2 ? dm[2] : dm[3]));
        if (!(dmr < guard)) continue;
        const int i = i0 + 4 * r;
        const float a0 = xs[(3 * i) * 64], a1 = xs[(3 * i + 1) * 64], a2 = xs[(3 * i + 2) * 64];
#pragma unroll 1
        for (int jj = i + 1; jj < A; jj += 4) {
            float d2[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int jc = (jj + u < A) ? jj + u : A - 1;
                const float d0 = a0 - xs[(3 * jc) * 64], d1 = a1 - xs[(3 * jc + 1) * 64], d2c = a2 - xs[(3 * jc + 2) * 64];
                d2[u] = (jj + u < A) ? fmaf(d2c, d2c, fmaf(d1, d1, fmaf(d0, d0, 0.f))) : guard;
            }
            if (fminf(fminf(d2[0], d2[1]), fminf(d2[2], d2[3])) < guard) {
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (d2[u] < guard) {
                        const float dd = sqrtf(d2[u]);
                        if (dd < cut) {
                            const float e = r_exp(-(dd * dd) / c2);
                            if (e != 1.f) w += e;       // pairs whose Gaussian rounds to 1 are dropped (mask2)
                        }
                    }
            }
        }
    }
    return w;
}
__device__ __forceinline__ float ts_pairs(const float* xs, int A, int part, int ib, int ie, float cut, float c2, float w) {
    const float guard = cut * cut * 1.0001f;
    for (int i0 = ib + part; i0 < ie && i0 < A - 1; i0 += 16) {
        int nr = (A - 1 - i0 + 3) / 4;                      // rows i0, i0 + 4, ... below A - 1
        nr = nr > 4 ? 4 : nr;
        w = ts_pair_block(xs, A, i0, nr, cut, c2, guard, w);
    }
    return w;
}

// Per-agent terrain cost of SwarmTraj ('blocks', SwarmTraj.py:90-122) with the problem constants in registers.  (The shared
// terrain_agent() takes the problem descriptor by reference: here that put a copy of the kernel parameter in local memory and
// every field read became an L2 round trip -- 7 000 cycles per evaluation for 13 agents in the first trace.)
__device__ __forceinline__ float ts_terrain(int obstacle, bool training, const float (&t)[10], float x0, float x1, float x2) {
    if (obstacle != 3) return 0.f;
    if (!training) {                    // bitwise &, |: no short-circuit branches (ten dependent branches per agent otherwise)
        const bool in = ((x0 < 2.0f) & (x0 > -2.0f) & (x1 < 0.5f) & (x1 > -0.5f) & (x2 < 7.0f)) |
                        ((x0 < 4.0f) & (x0 > 2.0f) & (x1 < 1.0f) & (x1 > -1.0f) & (x2 < 4.0f));
        return in ? 1.f : 0.f;
    }
    // thresholds inflated by r, rounded from double on the host: t = {2+r, -2-r, .5+r, -.5-r, 7+r, 4+r, 2-r, 1+r, -1-r, 4+r}
    const bool in = ((x0 < t[0]) & (x0 > t[1]) & (x1 < t[2]) & (x1 > t[3]) & (x2 < t[4])) |
                    ((x0 < t[5]) & (x0 > t[6]) & (x1 < t[7]) & (x1 > t[8]) & (x2 < t[9]));
    if (!in) return 0.f;
    return (gauss3<float>(x0, x1, x2, 0.f, 0.f, 2.f, 9.f, 3.f, 9.f) + gauss3<float>(x0, x1, x2, 2.5f, 0.f, 2.f, 9.f, 3.f, 3.f)) + 999.f;
}

__device__ __forceinline__ void ts_bar_epi() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

template <class SH, bool INTER>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(SH::NT, 1) rollout_ts_kernel(const TsArgs A, const __grid_constant__ CUtensorMap tmapW) {
    constexpr int d = SH::d, D = SH::D, NZ = SH::NZ, KS = SH::KS, CPT = SH::CPT, MP = SH::MP;
    extern __shared__ __align__(1024) unsigned char smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int warp_u = __shfl_sync(0xffffffffu, warp, 0);
    const unsigned rank = cluster_ctarank();
    const ProbPack& pr = A.prob;
    unsigned char* sX = smem + SH::oX;
    unsigned char* sS = smem + SH::oS;
    unsigned char* sW = smem + SH::oW;
    float* sxs = reinterpret_cast<float*>(smem + SH::oXS);
    float* sred = reinterpret_cast<float*>(smem + SH::oRED);      // [6][4][64], then gt [64]
    float* sgt = sred + 6 * 4 * 64;
    float* sb1 = reinterpret_cast<float*>(smem + SH::oB1);
    float* swv = reinterpret_cast<float*>(smem + SH::oWV);
    double* scost = reinterpret_cast<double*>(smem + SH::oSRED);
    unsigned long long* bars = reinterpret_cast<unsigned long long*>(smem + SH::oBAR);
    unsigned* tmem_slot = reinterpret_cast<unsigned*>(bars + TS_NBAR);
    const unsigned bar0 = smem_u32(bars);
    auto bar = [&](int i) { return bar0 + 8u * (unsigned)i; };
    // development aid: time stamps of one evaluation of block 0 (role 0/1: epilogue warps 0 / 7, 2: MMA issuer, 3: TMA producer)
    // (compiled in with -DNOC_TS_TRACE_BUILD and switched on with NOC_TS_TRACE=1)
    int trole = -1, tidx = 0;
    bool ton = false;
#ifdef NOC_TS_TRACE_BUILD
    if (A.trace && blockIdx.x < 2 && lane == 0) trole = (int)blockIdx.x * 10 + warp;     // role = 10 * CTA + warp (8: TMA, 9: MMA)
    auto TR = [&](int tag) {
        if (ton && tidx < 256) { A.trace[(trole * 256 + tidx) * 2] = tag; A.trace[(trole * 256 + tidx) * 2 + 1] = clock64(); ++tidx; }
    };
#else
    auto TR = [&](int) {};
    (void)trole; (void)tidx; (void)ton;
#endif

    if (tid == 0) {
        for (int i = 0; i < 4; ++i) { mbar_init(bar(TS_WFULL + i), 1); mbar_init(bar(TS_WEMPTY + i), 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(bar(TS_XFULL + i), 16); mbar_init(bar(TS_XEMPTY + i), 1); }
        mbar_init(bar(TS_SFULL), 16);
        for (int i = 0; i < 5; ++i) mbar_init(bar(TS_ACC + i), 1);
        fence_mbar_init_cluster();
    }
    if (warp == 9) tmem_alloc2(smem_u32(tmem_slot), 512);
    if (warp == 8 && lane == 0) tma_prefetch_desc(&tmapW);
    for (int i = tid; i < MP; i += SH::NT) { sb1[i] = (i < A.m) ? A.b1[i] : 0.f; swv[i] = (i < A.m) ? A.w[i] : 0.f; }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const unsigned tbase = *tmem_slot;
    const unsigned R0 = tbase, R1 = tbase + 256;
    const int ncl = (int)cluster_count_x(), cl = (int)cluster_id_x();

    if (warp_u == 8) {
        // ================= TMA producer: the same NSTAGE stages for every evaluation of every tile =================
        if (elect_one_sync()) {
            const unsigned wfull_leader = mapa_shared(bar(TS_WFULL), 0);
            unsigned cnt = 0;
            for (int tile = cl; tile < A.ntiles; tile += ncl)
                for (int it = 0; it < A.nevals; ++it)
                    for (int st = 0; st < SH::NSTAGE; ++st, ++cnt) {
                        const unsigned slot = cnt & 3, par = (cnt >> 2) & 1;
                        ton = (trole % 10 == 8 && tile == cl && it == 5);
                        mbar_wait_cluster(bar(TS_WEMPTY + slot), par ^ 1, 100 + slot);
                        if ((st & 7) == 0) TR(st);
                        if (rank == 0) mbar_arrive_expect_tx(bar(TS_WFULL + slot), 2 * SH::STAGE_BYTES);
                        tma2_load_2d(smem_u32(sW + slot * SH::STAGE_BYTES), &tmapW, wfull_leader + 8 * slot, 0,
                                     (int)((rank * SH::NSTAGE + st) * 128));
                    }
        }
        __syncwarp();
    } else if (warp_u == 9) {
        // ================= MMA issuer (leader CTA) =================
        if (rank == 0) {
            const unsigned idN = umma_idesc_f16(128, 256), idG = umma_idesc_f16(128, KS);
            const unsigned long long dX0 = umma_desc(smem_u32(sX), 128, 2048), dS = umma_desc(smem_u32(sS), 128, SH::SBO_S);
            constexpr unsigned qX = 16384 >> 4, qS = SH::PLANE_S >> 4, slabq = 32768 >> 4;
            unsigned wcnt = 0, xcnt0 = 0, xcnt1 = 0, scnt = 0;
            auto wait_w = [&]() -> unsigned {
                const unsigned slot = wcnt & 3, par = (wcnt >> 2) & 1;
                mbar_wait_cluster(bar(TS_WFULL + slot), par, 200 + slot);
                ++wcnt;
                tc_fence_after();
                return slot;
            };
            auto wait_x = [&](int b) {
                unsigned& c = b ? xcnt1 : xcnt0;
                mbar_wait_cluster(bar(TS_XFULL + b), c & 1, 210 + b);
                ++c;
                tc_fence_after();
            };
            for (int tile = cl; tile < A.ntiles; tile += ncl)
                for (int it = 0; it < A.nevals; ++it) {
                    const bool term = (it == A.nevals - 1);
                    ton = (trole % 10 == 9 && tile == cl && it == 5);
                    TR(0);
                    // ---- GEMM-1: O = S . K0b'  -> R0, committed per instruction half
                    mbar_wait_cluster(bar(TS_SFULL), scnt & 1, 220); ++scnt;
                    tc_fence_after();
                    TR(1);
                    for (int nh = 0; nh < 2; ++nh) {
                        for (int sp = 0; sp < KS / 32; ++sp) {
                            const unsigned slot = wait_w();
                            if (elect_one_sync()) {
                                const unsigned long long dB = umma_desc(smem_u32(sW + slot * SH::STAGE_BYTES), 128, 512);
#pragma unroll
                                for (int t = 0; t < 2; ++t)
                                    ts_mma3(R0 + 128 * nh, dS + (2 * sp + t) * 16, qS, dB + t * 16, 8192 >> 4, idN, (sp | t) > 0);
                                umma2_commit_mc(bar(TS_WEMPTY + slot), 3);
                            }
                            __syncwarp();
                        }
                        if (elect_one_sync()) umma2_commit_mc(bar(TS_ACC + nh), 3);
                        __syncwarp();
                        TR(10 + nh);
                    }
                    // ---- GEMM-2: A1 = U0 . K1' -> R1;  GEMM-3: Z1 = Y . K1 -> R0   (activation slabs as they are produced)
                    for (int gm = 0; gm < 2; ++gm) {
                        const unsigned Rd = gm == 0 ? R1 : R0;
                        for (int ji = 0; ji < 4; ++ji) {
                            const int b = ji & 1;
                            TR(100 * (gm + 1) + 10 * ji);
                            wait_x(b);
                            TR(100 * (gm + 1) + 10 * ji + 1);
                            for (int ks = 0; ks < 8; ++ks) {
                                const unsigned slot = wait_w();
                                if (elect_one_sync()) {
                                    const unsigned long long dB = umma_desc(smem_u32(sW + slot * SH::STAGE_BYTES), 128, 256);
                                    const unsigned long long dA = dX0 + b * slabq + ks * 16;
#pragma unroll
                                    for (int nh = 0; nh < 2; ++nh)
                                        ts_mma3(Rd + 128 * nh, dA, qX, dB + nh * (8192 >> 4), 4096 >> 4, idN, (ji | ks) > 0);
                                    umma2_commit_mc(bar(TS_WEMPTY + slot), 3);
                                    if (ks == 7) umma2_commit_mc(bar(TS_XEMPTY + b), 3);
                                }
                                __syncwarp();
                            }
                        }
                        if (elect_one_sync()) umma2_commit_mc(bar(TS_ACC + 2 + gm), 3);
                        __syncwarp();
                        TR(100 * (gm + 1) + 50);
                    }
                    // ---- GEMM-4: G = V . K0 + S . [A'A | c_w]' -> R1 (terminal evaluation: the S part apart, at R1 + 128)
                    for (int s4 = 0; s4 < SH::NS4; ++s4) {
                        const unsigned slot = wait_w();
                        for (int t = 0; t < 3; ++t) {
                            const int g = 3 * s4 + t;
                            if (g >= SH::NK4) break;
                            if (g < 32 && (g & 7) == 0) { TR(300 + g); wait_x((g >> 3) & 1); TR(301 + g); }
                            if (elect_one_sync()) {
                                const unsigned long long dB = umma_desc(smem_u32(sW + slot * SH::STAGE_BYTES + t * 2 * SH::G4_PLANE), 128, 256);
                                if (g < 32) {
                                    const int b = (g >> 3) & 1;
                                    ts_mma3(R1, dX0 + b * slabq + (g & 7) * 16, qX, dB, SH::G4_PLANE >> 4, idG, g > 0);
                                    if ((g & 7) == 7) umma2_commit_mc(bar(TS_XEMPTY + b), 3);
                                } else {
                                    ts_mma3(term ? R1 + 128 : R1, dS + (g - 32) * 16, qS, dB, SH::G4_PLANE >> 4, idG, term ? (g > 32) : 1);
                                }
                            }
                            __syncwarp();
                        }
                        if (elect_one_sync()) umma2_commit_mc(bar(TS_WEMPTY + slot), 3);
                        __syncwarp();
                    }
                    if (elect_one_sync()) umma2_commit_mc(bar(TS_ACC + 4), 3);
                    __syncwarp();
                    TR(350);
                }
        }
    } else if (warp_u < 8) {
        // ================= epilogue / per-sample warps =================
        const int qd = warp & 3, wh = warp >> 2;
        const int s = 32 * (qd & 1) + lane, q = qd >> 1, gq = 2 * wh + q;
        const unsigned lane_bits = (unsigned)(32 * qd) << 16;
        const int ubase = 256 * wh + 128 * q;                 // my hidden units: ubase + j, j in [0,128), TMEM column 128*wh + j
        const int cbase = (KS / 2) * q + CPT * wh;            // my gradient components [cbase, cbase + CPT), TMEM column CPT*wh + i
        const unsigned colH = 128 * wh, colG = CPT * wh;
        float* scr = A.scratch + (size_t)blockIdx.x * SH::SCR;
        float4* t0s = reinterpret_cast<float4*>(scr);
        float4* u0s = reinterpret_cast<float4*>(scr + MP * 64);
        float* z0s = scr + 2 * MP * 64;
        float* zas = z0s + d * 64;
        const float is1 = A.scales[3], is2 = A.scales[4], is4 = A.scales[5];
        const float kq1 = A.scales[6], kq2 = A.scales[7], kq4 = A.scales[8];
        const unsigned xfull_leader = mapa_shared(bar(TS_XFULL), 0), sfull_leader = mapa_shared(bar(TS_SFULL), 0);
        const bool hasQ = A.hasQ != 0, hasW = A.hasW != 0, posQ = A.posQ != 0;
        const float f_alphQ = A.f_alphQ, f_alphW = A.f_alphW, f_cut = A.f_cut, f_c2 = A.f_c2;
        const float hnet = A.h;
        const int p_obstacle = A.obstacle;
        const bool p_training = A.training != 0;
        unsigned xcnt0 = 0, xcnt1 = 0, acnt = 0;
        double* csum = scost + 16;                              // [7] cost sums + sample count of this CTA (thread warp 6, lane 0)
        if (warp == 6 && lane < 8) csum[lane] = 0.0;
        const int ntp1 = A.nt + 1;
        // intermediates: trajectory column `col` of row c of (zFull | ctrlFull).  With the staging buffer a warp writes 128
        // contiguous bytes per (step, row) and tc_untile_kernel transposes into the reference layout [n, rows, nt+1] afterwards;
        // without it (allocation failed) every thread writes its strided 4-byte element.
        auto put_z = [&](int tile, long long gs, int c, int col, float v) {
            if (A.stage) A.stage[(((size_t)tile * ntp1 + col) * (NZ + d) + c) * 128 + 64 * rank + s] = v;
            else A.out_b[(gs * NZ + c) * ntp1 + col] = v;
        };
        auto put_u = [&](int tile, long long gs, int c, int col, float v) {
            if (A.stage) A.stage[(((size_t)tile * ntp1 + col) * (NZ + d) + NZ + c) * 128 + 64 * rank + s] = v;
            else A.out_c[(gs * d + c) * ntp1 + col] = v;
        };

        // write 32 values (units ubase + 32 ji + [0,32)) as one thread's part of activation slab `b`, then hand the slab over
        auto put_slab = [&](int b, const float* v) {
            unsigned char* base = sX + b * 32768 + (s >> 3) * 2048 + (4 * gq) * 128 + (s & 7) * 16;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                uint4 hi, lo;
                split2_f16(v[8 * c], v[8 * c + 1], hi.x, lo.x); split2_f16(v[8 * c + 2], v[8 * c + 3], hi.y, lo.y);
                split2_f16(v[8 * c + 4], v[8 * c + 5], hi.z, lo.z); split2_f16(v[8 * c + 6], v[8 * c + 7], hi.w, lo.w);
                *reinterpret_cast<uint4*>(base + c * 128) = hi;
                *reinterpret_cast<uint4*>(base + 16384 + c * 128) = lo;
            }
            fence_async_smem();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(xfull_leader + 8 * b);
        };
        auto wait_slab_free = [&](int b) {
            unsigned& c = b ? xcnt1 : xcnt0;
            mbar_wait_cluster(bar(TS_XEMPTY + b), (c & 1) ^ 1, 300 + b);
            ++c;
        };
        auto wait_acc = [&](int g) { mbar_wait_cluster(bar(TS_ACC + g), acnt & 1, 310 + g); tc_fence_after(); };
        // my CPT/8 chunks of the stage-input operand S = [x, t, 1, 0..] from the fp32 x in shared memory
        auto put_S = [&](float tnext) {
#pragma unroll
            for (int c = 0; c < CPT / 8; ++c) {
                float v[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const int k = cbase + 8 * c + e;
                    v[e] = (k < d) ? sxs[(k < d ? k : 0) * 64 + s] : (k == d ? tnext : (k == D ? 1.f : 0.f));
                }
                uint4 hi, lo;
                split2_f16(v[0], v[1], hi.x, lo.x); split2_f16(v[2], v[3], hi.y, lo.y);
                split2_f16(v[4], v[5], hi.z, lo.z); split2_f16(v[6], v[7], hi.w, lo.w);
                unsigned char* p = sS + (s >> 3) * SH::SBO_S + ((cbase >> 3) + c) * 128 + (s & 7) * 16;
                *reinterpret_cast<uint4*>(p) = hi;
                *reinterpret_cast<uint4*>(p + SH::PLANE_S) = lo;
            }
            fence_async_smem();
        };
        auto arrive_S = [&] {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(sfull_leader);
        };

        for (int tile = cl; tile < A.ntiles; tile += ncl) {
            const long long s0 = (long long)tile * 128 + 64 * rank;
            const long long left = A.n - s0;
            const int nvalid = left >= 64 ? 64 : (left > 0 ? (int)left : 0);
            const bool valid = s < nvalid;
            long long gs = s0 + s;                               // padding rows replay the last sample (results unused)
            if (gs > A.n - 1) gs = A.n - 1;
            const float4* etab = reinterpret_cast<const float4*>(A.evals);
            float zq0[4] = {0.f, 0.f, 0.f, 0.f}, zqa[4] = {0.f, 0.f, 0.f, 0.f};   // [L, HJt, Q, W] integrals (gq == 3 thread)
            // ---- tile start: x -> z0 scratch, fp32 stage input, S operand of the first evaluation
#pragma unroll
            for (int i = 0; i < CPT; ++i) {
                const int c = cbase + i;
                if (c < d) {
                    const float xv = A.x[gs * d + c];
                    __stcg(z0s + c * 64 + s, xv);
                    sxs[c * 64 + s] = xv;
                    if (INTER && valid) { put_z(tile, gs, c, 0, xv); put_u(tile, gs, c, 0, 0.f); }
                }
            }
            if (INTER && valid && gq == 3) {
#pragma unroll
                for (int c = d; c < NZ; ++c) put_z(tile, gs, c, 0, 0.f);
            }
            put_S(__ldg(etab).x);
            ts_bar_epi();
            arrive_S();

            float phi1 = 0.f;
            for (int it = 0; it < A.nevals; ++it) {
                const float4 ef = __ldg(etab + 2 * it);
                const int4 ei = __ldg(reinterpret_cast<const int4*>(etab + 2 * it + 1));
                const float tcur = ef.x, wgt = ef.y, cnext = ef.z, hstep = ef.w;
                const int k = ei.x, kind = ei.y, first = ei.z, last = ei.w;
                const bool term = (kind == 2);
                ton = (trole >= 0 && trole % 10 < 8 && tile == cl && it == 5);
                TR(0);
                // ---- problem terms that need only x (SwarmTraj.py:90-164): computed in three pieces in the gaps where these
                //      warps would wait for the tensor core (after each of the epilogues 1-3 the last two slabs are still in flight)
                float qpart = 0.f, wpart = 0.f;
                // ---- epilogue 1: u0 = act(o) -> slabs, tanh(o) -> scratch
                TR(1);
                wait_acc(wh);
                TR(2);
#pragma unroll 1
                for (int ji = 0; ji < 4; ++ji) {
                    float v[32], tt[32];
                    tmem_ld32(R0 + lane_bits + colH + 32 * ji, v);
                    TR(100 + 10 * ji);
                    wait_slab_free(ji & 1);
                    TR(101 + 10 * ji);
#pragma unroll
                    for (int i = 0; i < 32; ++i) act_tanh(ts_unbias(v[i], kq1) * is1, v[i], tt[i]);
                    const int g4 = ((ubase + 32 * ji) >> 2) * 64 + s;
#pragma unroll
                    for (int i = 0; i < 8; ++i) __stcg(t0s + g4 + 64 * i, make_float4(tt[4 * i], tt[4 * i + 1], tt[4 * i + 2], tt[4 * i + 3]));
                    if (term) {
#pragma unroll
                        for (int i = 0; i < 8; ++i) __stcg(u0s + g4 + 64 * i, make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]));
                    }
                    put_slab(ji & 1, v);
                }
                // ---- epilogue 2: y = tanh(a1 + b1) * w -> slabs   (terminal: also w . (u0 + h act(a1 + b1)), Phi.py:50,96)
                float phiN = 0.f;
                TR(140);
                if (!term) {
                    if (hasQ)
                        for (int a = gq; a < SH::NA; a += 4)
                            qpart += ts_terrain(p_obstacle, p_training, A.thr, sxs[(3 * a) * 64 + s], sxs[(3 * a + 1) * 64 + s], sxs[(3 * a + 2) * 64 + s]);
                    TR(141);
                    if (hasW) wpart = ts_pairs(sxs + s, SH::NA, gq, 0, 16, f_cut, f_c2, wpart);
                }
                TR(150);
                wait_acc(2);
                TR(151);
#pragma unroll 1
                for (int ji = 0; ji < 4; ++ji) {
                    float v[32];
                    tmem_ld32(R1 + lane_bits + colH + 32 * ji, v);
                    TR(200 + 10 * ji);
                    wait_slab_free(ji & 1);
                    TR(201 + 10 * ji);
                    const int u0i = ubase + 32 * ji;
                    if (term) {
                        const int g4 = (u0i >> 2) * 64 + s;
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const float4 uu = __ldcg(u0s + g4 + 64 * i);
                            const float u4[4] = {uu.x, uu.y, uu.z, uu.w};
#pragma unroll
                            for (int e = 0; e < 4; ++e) {
                                float av, tv;
                                act_tanh(fmaf(ts_unbias(v[4 * i + e], kq2), is2, sb1[u0i + 4 * i + e]), av, tv);
                                const float wv = swv[u0i + 4 * i + e];
                                phiN = fmaf(wv, u4[e] + hnet * av, phiN);
                                v[4 * i + e] = tv * wv;
                            }
                        }
                    } else {
#pragma unroll
                        for (int i = 0; i < 32; i += 4) {
                            const float4 b4 = *reinterpret_cast<const float4*>(sb1 + u0i + i), w4 = *reinterpret_cast<const float4*>(swv + u0i + i);
                            v[i] = tanh_only(fmaf(ts_unbias(v[i], kq2), is2, b4.x)) * w4.x;
                            v[i + 1] = tanh_only(fmaf(ts_unbias(v[i + 1], kq2), is2, b4.y)) * w4.y;
                            v[i + 2] = tanh_only(fmaf(ts_unbias(v[i + 2], kq2), is2, b4.z)) * w4.z;
                            v[i + 3] = tanh_only(fmaf(ts_unbias(v[i + 3], kq2), is2, b4.w)) * w4.w;
                        }
                    }
                    put_slab(ji & 1, v);
                }
                // ---- epilogue 3: v = tanh(o) * (w + h z1) -> slabs
                if (!term && hasW) wpart = ts_pairs(sxs + s, SH::NA, gq, 16, 32, f_cut, f_c2, wpart);
                TR(250);
                wait_acc(3);
                TR(251);
                const float hs = hnet * is2;
#pragma unroll 1
                for (int ji = 0; ji < 4; ++ji) {
                    float v[32];
                    const int u0i = ubase + 32 * ji, g4 = (u0i >> 2) * 64 + s;
                    float4 t4[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) t4[i] = __ldcg(t0s + g4 + 64 * i);
                    tmem_ld32(R0 + lane_bits + colH + 32 * ji, v);
                    TR(300 + 10 * ji);
                    wait_slab_free(ji & 1);
                    TR(301 + 10 * ji);
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float4 w4 = *reinterpret_cast<const float4*>(swv + u0i + 4 * i);
                        v[4 * i] = t4[i].x * fmaf(hs, ts_unbias(v[4 * i], kq2), w4.x);
                        v[4 * i + 1] = t4[i].y * fmaf(hs, ts_unbias(v[4 * i + 1], kq2), w4.y);
                        v[4 * i + 2] = t4[i].z * fmaf(hs, ts_unbias(v[4 * i + 2], kq2), w4.z);
                        v[4 * i + 3] = t4[i].w * fmaf(hs, ts_unbias(v[4 * i + 3], kq2), w4.w);
                    }
                    put_slab(ji & 1, v);
                }
                // ---- epilogue 4: grad Phi -> costs, RK update, next stage input
                if (!term && hasW) wpart = ts_pairs(sxs + s, SH::NA, gq, 32, SH::NA, f_cut, f_c2, wpart);
                // every warp is done reading this evaluation's x (pair terms) and the previous evaluation's partial sums before
                // any warp overwrites them below: GEMM-4's completion does not imply it (the slabs it needs were handed over
                // before the last piece of the pair loop).  compute-sanitizer racecheck found this one.
                ts_bar_epi();
                TR(350);
                wait_acc(4);
                TR(351);
                ++acnt;
                float g[CPT];
                {
                    unsigned r32[32];
                    tmem_ld32_issue(R1 + lane_bits + colG, r32);
                    if constexpr (CPT == 40) {
                        unsigned r8[8];
                        tmem_ld8_issue(R1 + lane_bits + colG + 32, r8);
                        tmem_wait_ld();
#pragma unroll
                        for (int i = 0; i < 8; ++i) g[32 + i] = ts_unbias(__uint_as_float(r8[i]), kq4) * is4;
                    } else {
                        tmem_wait_ld();
                    }
#pragma unroll
                    for (int i = 0; i < 32; ++i) g[i] = ts_unbias(__uint_as_float(r32[i]), kq4) * is4;
                }
                TR(360);
                if (!term) {
                    float pp = 0.f;
#pragma unroll
                    for (int i = 0; i < CPT; ++i) if (cbase + i < d) pp = fmaf(g[i], g[i], pp);
                    sred[(0 * 4 + gq) * 64 + s] = pp;
                    sred[(1 * 4 + gq) * 64 + s] = qpart;
                    sred[(2 * 4 + gq) * 64 + s] = wpart;
                    if (gq == 3) sgt[s] = g[d - ((KS / 2) + CPT)];         // Phi_t = component d of grad Phi
                    TR(370);
                    if (INTER && kind == 1) {                              // controls at the new state, OLD time (quirk 3)
                        if (valid) {
#pragma unroll
                            for (int i = 0; i < CPT; ++i) {
                                const int c = cbase + i;
                                if (c < d) {
                                    put_z(tile, gs, c, k + 1, __ldcg(z0s + c * 64 + s));
                                    put_u(tile, gs, c, k + 1, -g[i]);
                                }
                            }
                            if (gq == 3) {
#pragma unroll
                                for (int c = 0; c < 4; ++c) put_z(tile, gs, d + c, k + 1, zq0[c]);
                            }
                        }
                    } else {
                        // RK combination of my state components (OCflow.py:143-184); dx = -grad_p H = -p (SwarmTraj.py:68-69).
                        // z0 / the RK accumulator come from the L2 scratch in four batches, the next batch's loads in flight while
                        // this one is combined (no long-lived register arrays: they spilled, and a spill is an L2 round trip here).
                        constexpr int NB = (CPT == 40) ? 5 : 4, BQ = CPT / NB;
                        auto rk = [&](auto FIRST, auto LAST) {
                            constexpr bool F = decltype(FIRST)::value, L = decltype(LAST)::value;
                            float zb[2][BQ], za2[2][BQ];
                            auto fetch = [&](int b, float (&a0)[BQ], float (&a1)[BQ]) {
#pragma unroll
                                for (int i = 0; i < BQ; ++i) {
                                    const int c = cbase + b * BQ + i;
                                    a0[i] = (c < d && (F || !L)) ? __ldcg(z0s + c * 64 + s) : 0.f;
                                    a1[i] = (c < d && !F) ? __ldcg(zas + c * 64 + s) : 0.f;
                                }
                            };
                            fetch(0, zb[0], za2[0]);
#pragma unroll
                            for (int b = 0; b < NB; ++b) {
                                if (b + 1 < NB) fetch(b + 1, zb[(b + 1) & 1], za2[(b + 1) & 1]);
#pragma unroll
                                for (int i = 0; i < BQ; ++i) {
                                    const int ii = b * BQ + i, c = cbase + ii;
                                    if (c < d) {
                                        const float kk = hstep * (-g[ii]);
                                        const float za1 = (F ? zb[b & 1][i] : za2[b & 1][i]) + wgt * kk;
                                        float xn;
                                        if (!L) { __stcg(zas + c * 64 + s, za1); xn = zb[b & 1][i] + cnext * kk; }
                                        else { __stcg(z0s + c * 64 + s, za1); xn = za1; }
                                        sxs[c * 64 + s] = xn;
                                    }
                                }
                            }
                        };
                        if (first) { if (last) rk(std::true_type{}, std::true_type{}); else rk(std::true_type{}, std::false_type{}); }
                        else { if (last) rk(std::false_type{}, std::true_type{}); else rk(std::false_type{}, std::false_type{}); }
                    }
                    TR(400);
                    put_S(__ldg(etab + 2 * (it + 1)).x);
                    TR(401);
                    ts_bar_epi();
                    TR(402);
                    if (gq == 3 && !(INTER && kind == 1)) {                // L, H, the four cost rates (SwarmTraj.py:71-87, OCflow.py:130-138)
                        float pps = 0.f, qs = 0.f, ws = 0.f;
#pragma unroll
                        for (int p = 0; p < 4; ++p) { pps += sred[(0 * 4 + p) * 64 + s]; qs += sred[(1 * 4 + p) * 64 + s]; ws += sred[(2 * 4 + p) * 64 + s]; }
                        const float Qret = posQ ? qs : 0.f;
                        float L = 0.5f * pps + f_alphQ * Qret;
                        if (hasW) L = L + f_alphW * ws; else ws = 0.f;
                        const float H = -L + pps;
                        const float rate[4] = {L, fabsf(sgt[s] - H), Qret, ws};
#pragma unroll
                        for (int c = 0; c < 4; ++c) {
                            const float kk = hstep * rate[c];
                            zqa[c] = (first ? zq0[c] : zqa[c]) + wgt * kk;
                            if (last) zq0[c] = zqa[c];
                        }
                    }
                    arrive_S();
                    TR(403);
                    continue;
                }
                // ---- terminal block (OCflow.py:58-90): x(T) in shared memory, g = grad Phi(x(T), T)
                float gqv[CPT];
                {
                    unsigned r32[32];
                    tmem_ld32_issue(R1 + 128 + lane_bits + colG, r32);
                    if constexpr (CPT == 40) {
                        unsigned r8[8];
                        tmem_ld8_issue(R1 + 128 + lane_bits + colG + 32, r8);
                        tmem_wait_ld();
#pragma unroll
                        for (int i = 0; i < 8; ++i) gqv[32 + i] = __uint_as_float(r8[i]) * is4;
                    } else {
                        tmem_wait_ld();
                    }
#pragma unroll
                    for (int i = 0; i < 32; ++i) gqv[i] = __uint_as_float(r32[i]) * is4;
                }
                const float* xt = static_cast<const float*>(pr.xtarget);
                float cG = 0.f, hjg = 0.f, quad = 0.f, lin = 0.f;
#pragma unroll
                for (int i = 0; i < CPT; ++i) {
                    const int c = cbase + i;
                    if (c < D) {
                        const float cw = __ldg(A.c_w + c);
                        const float sv = (c < d) ? sxs[(c < d ? c : 0) * 64 + s] : tcur;
                        const float gfull = g[i] + gqv[i];                   // V.K0 + (A'A s + c_w)
                        quad = fmaf(sv, gqv[i] - cw, quad);
                        lin = fmaf(cw, sv, lin);
                        if (c < d) {
                            const float res = sv - __ldg(xt + c);
                            cG = fmaf(res, res, cG);
                            hjg += fabsf(gfull - A.alph0 * res);
                        }
                    }
                }
                sred[(0 * 4 + gq) * 64 + s] = cG; sred[(1 * 4 + gq) * 64 + s] = hjg; sred[(2 * 4 + gq) * 64 + s] = quad;
                sred[(3 * 4 + gq) * 64 + s] = lin; sred[(4 * 4 + gq) * 64 + s] = phiN;
                ts_bar_epi();
                if (gq == 3) {
                    float t5[5];
#pragma unroll
                    for (int r5 = 0; r5 < 5; ++r5) t5[r5] = ((sred[(r5 * 4 + 0) * 64 + s] + sred[(r5 * 4 + 1) * 64 + s]) + sred[(r5 * 4 + 2) * 64 + s]) + sred[(r5 * 4 + 3) * 64 + s];
                    const float cGh = 0.5f * t5[0];
                    phi1 = t5[4] + 0.5f * t5[2] + (t5[3] + A.c_b[0]);           // Phi = w.u1 + 0.5 s'A'A s + c_w.s + c_b (Phi.py:96)
                    const float cost[7] = {zq0[0], cGh, zq0[1], fabsf(phi1 - A.alph0 * cGh), t5[1], zq0[2], zq0[3]};
                    if (A.mode == NOC_MODE_MEAN) {
#pragma unroll
                        for (int q7 = 0; q7 < 7; ++q7) {
                            double vsum = valid ? (double)cost[q7] : 0.0;      // double: the sums must not depend on the tiling
#pragma unroll
                            for (int off = 16; off > 0; off >>= 1) vsum += __shfl_xor_sync(0xffffffffu, vsum, off);
                            if (lane == 0) scost[(qd & 1) * 8 + q7] = vsum;
                        }
                    } else if (A.mode == NOC_MODE_NOMEAN && valid) {
                        float* o = A.out_a + gs * 8;
                        o[0] = cost[0] + A.alph0 * cost[1] + A.alph3 * cost[2] + A.alph4 * cost[3] + A.alph5 * cost[4];   // OCflow.py:75
#pragma unroll
                        for (int q7 = 0; q7 < 7; ++q7) o[1 + q7] = cost[q7];
                    }
                }
                ts_bar_epi();
                if (A.mode == NOC_MODE_MEAN && warp == 6 && lane == 0) {
                    for (int q7 = 0; q7 < 7; ++q7) csum[q7] += scost[q7] + scost[8 + q7];
                    csum[7] += (double)nvalid;
                }
            }
        }
        if (A.mode == NOC_MODE_MEAN && A.partials && warp == 6 && lane == 0) {
            for (int q7 = 0; q7 < 8; ++q7) A.partials[blockIdx.x * 8 + q7] = csum[q7];
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 9) tmem_dealloc2(tbase, 512);
}

// ------------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------------
typedef CUresult (*ts_encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static inline ts_encode_fn ts_get_encode() {
    static ts_encode_fn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
            fn = (ts_encode_fn)p;
    }
    return fn;
}

static inline size_t ts_smem_bytes_50() { return (size_t)TsShape<50>::SMEM; }

template <class SH>
int launch_ts(const RolloutCall<float>& c) {
    cudaStream_t st = c.stream;
    const ProbPack& pr = c.prob;
    TsArgs A;
    memset(&A, 0, sizeof A);
    copy_common(A, c);
    A.m = c.m; A.h = c.h;
    A.b1 = c.raw.b[1]; A.w = c.raw.w; A.c_w = c.raw.c_w; A.c_b = c.raw.c_b;
    A.f_alphQ = (float)pr.alph_Q; A.f_alphW = (float)pr.alph_W; A.f_cut = (float)pr.cutW; A.f_c2 = (float)(2 * pr.r * pr.r);
    A.hasQ = (pr.obstacle != 0) && (pr.alph_Q > 0.0); A.hasW = (pr.alph_W != 0.0); A.posQ = (pr.alph_Q > 0.0);
    A.obstacle = pr.obstacle; A.training = pr.training;
    {
        const double r = pr.r;                     // SwarmTraj.py:101-119: the boxes inflated by r (train mode)
        const double t[10] = {2.0 + r, -2.0 - r, 0.5 + r, -0.5 - r, 7.0 + r, 4.0 + r, 2.0 - r, 1.0 + r, -1.0 - r, 4.0 + r};
        for (int i = 0; i < 10; ++i) A.thr[i] = (float)t[i];
    }
    ScratchBuf evals, blob, aux, scratch, partials, stage;     // aux: [3] max bits, [6] scales (+ pad)
    NOC_CUDA(tc_upload_evals(c, A, evals));
    const size_t smem = SH::SMEM;
    auto kern = (A.mode == NOC_MODE_INTERMEDIATES) ? rollout_ts_kernel<SH, true> : rollout_ts_kernel<SH, false>;
    if (smem > (size_t)c.smem_limit) return fail(NOC_ERR_NOMEM, "streamed tensor-core rollout needs %zu B of shared memory", smem);
    ts_encode_fn encode = ts_get_encode();
    if (!encode) return fail(NOC_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
    NOC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    A.ntiles = (int)((A.n + 127) / 128);
    const int clusters = std::max(1, std::min(A.ntiles, sm_count() / 2));
    const int grid = 2 * clusters;
    const size_t blob_bytes = (size_t)2 * SH::NSTAGE * SH::STAGE_BYTES;
    NOC_CUDA(blob.alloc(blob_bytes, st));
    NOC_CUDA(aux.alloc(64, st));
    NOC_CUDA(scratch.alloc(sizeof(float) * (size_t)SH::SCR * grid, st));
    NOC_CUDA(cudaMemsetAsync(blob.p, 0, blob_bytes, st));
    NOC_CUDA(cudaMemsetAsync(aux.p, 0, 64, st));
    TsPackArgs P;
    P.m = A.m; P.D = c.d + 1; P.r = c.r;
    P.K0 = c.raw.K[0]; P.b0 = c.raw.b[0]; P.K1 = c.raw.K[1]; P.A = c.raw.A; P.c_w = c.raw.c_w;
    P.maxbits = aux.as<unsigned>(); P.scales = aux.as<float>() + 4; P.blob = blob.as<unsigned char>();
    {
        // The tensor core's fp32 accumulate rounds toward zero: measured -0.137 ulp of the result per accumulating MMA
        // (scripts/tc_bias_probe.py), i.e. a relative shrink of 0.137 * 0.72 * 2^-23 = 1.18e-8 per MMA on average over the
        // mantissa.  A K = 512 contraction is 96 MMAs; the mean shrink is undone in the epilogue scale (zero-mean residual).
        double f[3] = {1.0, 1.0, 1.0};
        if (const char* e = getenv("NOC_TS_BIAS")) {
            const int got = sscanf(e, "%lf,%lf,%lf", &f[0], &f[1], &f[2]);
            if (got == 1) f[1] = f[2] = f[0];
        }
        const double per = 1.89e-8;                            // mean relative shrink per accumulating MMA (see ts_unbias)
        P.bias[0] = (float)(per * f[0] * 3 * SH::NK1); P.bias[1] = (float)(per * f[1] * 3 * 32); P.bias[2] = (float)(per * f[2] * 3 * SH::NK4);
    }
    ts_absmax_kernel<<<64, 256, 0, st>>>(P);
    count_launch();
    ts_scales_kernel<<<1, 32, 0, st>>>(P);
    count_launch();
    ts_pack_kernel<SH><<<(2 * SH::NSTAGE * 512 + 255) / 256, 256, 0, st>>>(P);
    count_launch();
    NOC_CUDA(cudaGetLastError());
    // the blob as a 2-D tensor of 128-byte rows; one stage = one box of 128 rows (the exact shared-memory image)
    CUtensorMap tmap;
    const cuuint64_t gdim[2] = {64, (cuuint64_t)(blob_bytes / 128)};
    const cuuint64_t gstr[1] = {128};
    const cuuint32_t box[2] = {64, 128}, estr[2] = {1, 1};
    CUresult cr = encode(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT16, 2, blob.p, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) return fail(NOC_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)cr);
    A.scales = P.scales;
    A.scratch = scratch.as<float>();
    if (A.mode == NOC_MODE_MEAN) {
        NOC_CUDA(partials.alloc(sizeof(double) * 8 * (size_t)grid, st));
        NOC_CUDA(cudaMemsetAsync(partials.p, 0, sizeof(double) * 8 * (size_t)grid, st));
        A.partials = partials.as<double>();
    }
    if (getenv("NOC_DEBUG"))
        fprintf(stderr, "[noc] ts rollout: smem=%zu grid=%d (clusters of 2) tiles=%d stages/eval=%d evals=%d\n", smem, grid, A.ntiles,
                SH::NSTAGE, A.nevals);
    // intermediates: stage the trajectories tile-major (coalesced) and transpose afterwards; if the staging buffer (as large as
    // the outputs) cannot be allocated the kernel writes the reference layout directly (strided, slower, same result)
    if (A.mode == NOC_MODE_INTERMEDIATES && !getenv("NOC_TS_NOSTAGE")) {
        const size_t bytes = sizeof(float) * (size_t)A.ntiles * (A.nt + 1) * (SH::NZ + SH::d) * 128;
        big_reserve(bytes);                              // repeated intermediates calls reuse the staging buffer instead of paying the driver
        if (stage.alloc_big(bytes, st) != cudaSuccess) (void)cudaGetLastError();
    }
    A.stage = stage.as<float>();
    long long* trace = nullptr;
    if (getenv("NOC_TS_TRACE")) {
        NOC_CUDA(cudaMalloc((void**)&trace, sizeof(long long) * 20 * 256 * 2));
        NOC_CUDA(cudaMemset(trace, 0, sizeof(long long) * 20 * 256 * 2));
        A.trace = trace;
    }
    kern<<<grid, SH::NT, smem, st>>>(A, tmap);
    count_launch();
    NOC_CUDA(cudaGetLastError());
    if (trace) {
        std::vector<long long> h(20 * 256 * 2);
        NOC_CUDA(cudaStreamSynchronize(st));
        NOC_CUDA(cudaMemcpy(h.data(), trace, sizeof(long long) * h.size(), cudaMemcpyDeviceToHost));
        long long t0 = 0;
        for (int r = 0; r < 20; ++r) for (int i = 0; i < 256; ++i) { long long c = h[(r * 256 + i) * 2 + 1]; if (c && (!t0 || c < t0)) t0 = c; }
        for (int r = 0; r < 20; ++r) {
            fprintf(stderr, "[noc trace] role %d:", r);
            for (int i = 0; i < 256 && h[(r * 256 + i) * 2 + 1]; ++i) fprintf(stderr, " %lld@%lld", h[(r * 256 + i) * 2], h[(r * 256 + i) * 2 + 1] - t0);
            fprintf(stderr, "\n");
        }
        cudaFree(trace);
    }
    if (stage.p) {
        tc_untile_kernel<<<dim3(A.ntiles, SH::NZ + SH::d), 128, 0, st>>>(A.stage, A.out_b, A.out_c, A.n, A.nt + 1, SH::NZ, SH::d);
        count_launch();
        NOC_CUDA(cudaGetLastError());
        NOC_CUDA(stage.free());
    }
    if (partials.p) {
        int frc = launch_finish(A.partials, grid, c.out_sums, st);
        if (frc) return frc;
        NOC_CUDA(partials.free());
    }
    NOC_CUDA(scratch.free());
    NOC_CUDA(aux.free());
    NOC_CUDA(blob.free());
    NOC_CUDA(evals.free());
    return NOC_OK;
}

}  // namespace noc
