// noc_tc_rollout.cuh — tensor-core (tcgen05 / TMEM) rollout kernel, fp32 in / fp32 out, for value networks with
// nTh = 2 and m <= 128 on problems whose state fits one thread's registers (d <= 24).
//
// One CTA owns a tile of 128 samples; THREAD r IS SAMPLE r (SPLIT > 1: SPLIT threads per sample, each owning 1/SPLIT of the
// hidden units in the epilogues and all of them keeping the per-sample state): it keeps the augmented state
// z = [x, L, HJt, Q, W] and the RK accumulator in registers for all nt steps (the accumulator parked in spare TMEM columns
// during an evaluation for wide states), evaluates the problem terms (calcLHQW / calcGradpH / calcCtrls) in registers, and is
// an epilogue thread of TMEM lane r.  The four contractions of one grad-Phi evaluation
// (Phi.py:99-138) run on the 5th-generation tensor cores with M = 128 samples:
//     GEMM-1  O  [128 x m]  = S [128 x KS] . K0b'     S = [x, t, 1, 0..]  (the 1-column folds the bias b0 in)
//     GEMM-2  A1 [128 x m]  = U0 [128 x m] . K1'      B = K1 read K-major
//     GEMM-3  Z1 [128 x m]  = Y  [128 x m] . K1       B = the SAME K1 buffer read MN-major
//     GEMM-4  G  [128 x KS] = V  [128 x m] . K0b (MN-major view of the GEMM-1 buffer)  +  S . symb'  (A'A and c_w)
// The accumulator lives in TMEM (fp32); tanh(o) is parked in TMEM between GEMM-1 and GEMM-3.
//
// Precision: every fp32 operand is split into two fp16 terms (hi + lo, 22 significant bits) and each logical product is three
// MMAs (hi.hi, hi.lo, lo.hi; the dropped lo.lo term is O(2^-22)), because a single bf16 / tf32 pass breaks the 1e-5
// per-step-state tolerance (SURVEY.md H1).  fp16's narrow exponent is handled with per-matrix power-of-two scales computed at
// set-up (largest weight of a matrix -> [2^13, 2^14), so that the lo plane stays in the normal range; the Y / V operands
// carry the scale of w the same way); the reciprocal scales are folded into constants the epilogues apply anyway.  The
// tensor core's fp32 accumulate rounds toward zero (measured: a mean relative shrink of 1.89e-8 per accumulating MMA,
// scripts/tc_bias_probe.py, scripts/ts_bias_robust.py); the mean is undone in the same reciprocal scales.  (Round 1 used three
// bf16 planes and six MMAs per product into two accumulators: twice the tensor work, 1.5x the split / store work and twice
// the TMEM loads for the same measured accuracy.)
//
// Operands are written by the epilogue threads straight into the canonical no-swizzle UMMA layout (8-row x 16-byte core
// matrices), one elected lane issues the MMAs, and tcgen05.commit signals an mbarrier all epilogue threads wait on.
// Several CTAs share an SM when shared memory and TMEM columns allow, so one tile's epilogue overlaps another's MMAs.
#pragma once
#include "noc_launch.cuh"
#include "noc_tc.cuh"

#include <cstdio>
#include <cstdlib>
#include <vector>

namespace noc {

// One entry per grad-Phi evaluation of a rollout, in execution order: the RK stages of every step (OCflow.py:157-184),
// the control evaluation after each step when intermediates are requested (:51-55), and the terminal evaluation (:58).
// Times and RK weights are the reference's python doubles rounded to fp32 once, on the host.
struct __align__(16) TcEval {
    float t, wgt, cnext, h;         // evaluation time, weight of this stage in the RK sum, coefficient of the next stage input, step
    int k, kind, first, last;       // step index; 0 = RK stage, 1 = controls, 2 = terminal; first / last stage of its step
};

struct TcArgs {
    int m, mp;                      // hidden width and its padded value (multiple of the epilogue chunk)
    float h;
    const float *K0, *b0, *K1, *b1, *w, *A, *c_w, *c_b;   // reference layout (fp32, device)
    int r;
    ProbPack prob;
    const float* x;
    long long n;
    int nt, stepper, mode;
    const TcEval* evals;            // flat sequence of Phi evaluations of one rollout (host-built, see tc_build_evals)
    int nevals;
    float alph0, alph3, alph4, alph5, t_end;
    double* partials;
    float* out_a; float* out_b; float* out_c;
    float* stage;                   // intermediates: tile-major staging buffer [tile][step][row][128 samples] (coalesced), or NULL
    int ntiles, tmem_cols;
    float bias_f;                   // multiplier of the accumulate-bias compensation (1; experiments: NOC_TC_BIAS)
    float sx;                       // power-of-two scale of the S = [x, t, 1] operand (fp16 range, see the header)
    int park_col;                   // PARK shapes: column of the parked RK accumulator inside the main block, or -1 = own 32-column block
};

// problem shapes the kernel is instantiated for
template <int KIND_, int NA_, int CH_, int MINB_, int SPLIT_ = 1>
struct TcShape {
    static constexpr int KIND = KIND_, NA = NA_;
    static constexpr int DIM = (KIND == 2) ? 12 : (KIND == 0 ? 2 : 3);
    static constexpr int d = NA * DIM, D = d + 1, NZ = d + 4;
    static constexpr int KS = ((D + 1 + 15) / 16) * 16;           // K of the S operand: [x, t, 1] zero-padded
    static constexpr int NCTRL = (KIND == 2) ? 4 * NA : d;
    static constexpr int CH = CH_;                                 // epilogue chunk (TMEM columns per load)
    static constexpr int MINB = MINB_;
    static constexpr int SPLIT = SPLIT_;                           // threads per sample: each owns 1/SPLIT of the hidden units in the epilogues
    static constexpr int NT = 128 * SPLIT;
    // wide states: the RK accumulator is parked in 32 extra TMEM columns during each evaluation instead of being
    // spilled to local memory by the compiler (L1 is tiny next to ~200 KB of shared memory: every spill was an L2 trip)
    static constexpr bool PARK = ((NZ > 20) && (NZ <= 32) && SPLIT == 1) || (KIND == 2);
    static constexpr int PW = (NZ <= 16) ? 16 : 32;                 // parked columns per thread
    static_assert(KIND != 2 || NA == 1, "one quadcopter");
};

// write 8 consecutive K-elements (one 16-byte chunk) of row `row` of an A/B operand, both split planes (hi, lo)
__device__ __forceinline__ void store_chunk2(unsigned char* base, int plane_bytes, int row, int k0, int K, const float* v) {
    uint4 h, l;
    split2_f16(v[0], v[1], h.x, l.x);
    split2_f16(v[2], v[3], h.y, l.y);
    split2_f16(v[4], v[5], h.z, l.z);
    split2_f16(v[6], v[7], h.w, l.w);
    const int off = il_off(row, k0, K);
    *reinterpret_cast<uint4*>(base + off) = h;
    *reinterpret_cast<uint4*>(base + plane_bytes + off) = l;
}
__device__ __forceinline__ void unpack_f16x2(unsigned p, float& a, float& b) {
    asm("{\n\t.reg .b16 l, u;\n\tmov.b32 {l, u}, %2;\n\tcvt.f32.f16 %0, l;\n\tcvt.f32.f16 %1, u;\n\t}\n" : "=f"(a), "=f"(b) : "r"(p));
}
__device__ __forceinline__ void load_chunk2(const unsigned char* base, int plane_bytes, int row, int k0, int K, float* v) {
    const int off = il_off(row, k0, K);
    const uint4 a = *reinterpret_cast<const uint4*>(base + off), b = *reinterpret_cast<const uint4*>(base + plane_bytes + off);
    const unsigned pa[4] = {a.x, a.y, a.z, a.w}, pb[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        float h0, h1, l0, l1;
        unpack_f16x2(pa[i], h0, h1);
        unpack_f16x2(pb[i], l0, l1);
        v[2 * i] = h0 + l0;
        v[2 * i + 1] = h1 + l1;
    }
}

// one logical fp32 product block: three fp16 MMAs over the two planes of A and B (same descriptor geometry per plane) into
// one accumulator.  `ad` / `bd` are the descriptors of the hi planes; the start-address field is the low 14 bits (16-byte
// units), so the lo plane or another k-block is an integer add.
__device__ __forceinline__ void mma3(unsigned dt, unsigned long long ad, unsigned a_plane16, unsigned long long bd, unsigned b_plane16,
                                     unsigned idesc, int accumulate) {
    umma_bf16(dt, ad, bd, idesc, accumulate);                      // hi.hi   (kind::f16; the operand formats are in idesc)
    umma_bf16(dt, ad, bd + b_plane16, idesc, 1);                   // hi.lo
    umma_bf16(dt, ad + a_plane16, bd, idesc, 1);                   // lo.hi
}
// kind::f16 instruction descriptor, fp16 x fp16 -> f32, A K-major, B K- or MN-major
__device__ __forceinline__ unsigned umma_idesc_f16_b(int M, int N, int b_mn_major) {
    return (1u << 4) | ((unsigned)b_mn_major << 16) | ((unsigned)(N >> 3) << 17) | ((unsigned)(M >> 4) << 24);
}
// power-of-two scale that puts a matrix whose largest magnitude is `mx` into [2^e, 2^(e+1))
__device__ __forceinline__ float pow2_scale(float mx, int e) {
    return (mx > 0.f && mx < 3.0e38f) ? exp2f((float)(e - ilogbf(mx))) : 1.f;
}

template <int CH>
__device__ __forceinline__ void tmem_ld(unsigned ta, float* v) {
    unsigned r[CH];
    if constexpr (CH == 32) tmem_ld32_issue(ta, r); else tmem_ld16_issue(ta, r);
    tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < CH; ++i) v[i] = __uint_as_float(r[i]);
}
// two loads, one wait
template <int CH>
__device__ __forceinline__ void tmem_ld2(unsigned ta, float* v, unsigned tb, float* w) {
    unsigned r[CH], q[CH];
    if constexpr (CH == 32) { tmem_ld32_issue(ta, r); tmem_ld32_issue(tb, q); }
    else { tmem_ld16_issue(ta, r); tmem_ld16_issue(tb, q); }
    tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < CH; ++i) { v[i] = __uint_as_float(r[i]); w[i] = __uint_as_float(q[i]); }
}
template <int CH>
__device__ __forceinline__ void tmem_st(unsigned ta, const float* v) {
    unsigned r[CH];
#pragma unroll
    for (int i = 0; i < CH; ++i) r[i] = __float_as_uint(v[i]);
    if constexpr (CH == 32) tmem_st32_bits(ta, r); else tmem_st16_bits(ta, r);
}

// bytes of dynamic shared memory for (mp, KS)
static inline size_t tc_smem_bytes(int mp, int KS) {
    return 2 * ((size_t)mp * mp * 2 + (size_t)mp * KS * 2 + (size_t)KS * KS * 2 + (size_t)128 * mp * 2 + (size_t)128 * KS * 2) +
           sizeof(float) * (3 * (size_t)mp + KS + 32 + 3 * 128);
}
static inline int tc_tmem_cols(int mp, int KS) {      // accumulator | tanh(o) (the terminal evaluation's S.symb' reuses it)
    int need = 2 * std::max(mp, KS), c = 32;
    while (c < need) c *= 2;
    return c;
}

// INTER: the intermediates=True build (trajectory + control outputs); the mean / noMean build carries none of that code
template <class SH, bool INTER>
__global__ void __launch_bounds__(SH::NT, SH::MINB) rollout_tc_kernel(const TcArgs A) {
    constexpr int d = SH::d, D = SH::D, KS = SH::KS, NZ = SH::NZ, NCTRL = SH::NCTRL, CH = SH::CH, KIND = SH::KIND;
    constexpr int SPLIT = SH::SPLIT, NT = SH::NT;
    extern __shared__ __align__(1024) unsigned char smem[];
    const int tid = threadIdx.x, warp = tid >> 5;
    const int row = tid & 127, hf = tid >> 7;                  // my sample (= TMEM lane) and my share of the hidden units
    const int warp_u = __shfl_sync(0xffffffffu, warp, 0);      // the same value, known to the compiler as warp-uniform
    const int m = A.m, mp = A.mp;
    const ProbPack& pr = A.prob;
    // shared-memory map (bytes); every operand has two planes (hi, lo)
    const int pK1 = mp * mp * 2, pK0 = mp * KS * 2, pX = 128 * mp * 2;
    constexpr int pSy = KS * KS * 2, pS = 128 * KS * 2;
    unsigned char* sK1 = smem;
    unsigned char* sK0 = sK1 + 2 * pK1;
    unsigned char* sSy = sK0 + 2 * pK0;
    unsigned char* sX = sSy + 2 * pSy;
    unsigned char* sS = sX + 2 * pX;
    float* sb1 = reinterpret_cast<float*>(sS + 2 * pS);
    float* sb1c = sb1 + mp;                              // b1 * 2 log2(e): the bias as tanh2_w() wants it
    float* sw = sb1c + mp;                               // w * s_w (see below)
    float* scw = sw + mp;                                // KS floats
    float* sred = scw + KS;                              // 4 warps x 8
    float* sphi = sred + 32;                             // (SPLIT - 1) x 128: partial w.u1 of the other threads of a sample
    __shared__ __align__(8) unsigned long long mbar;
    __shared__ unsigned tmem_base_s, tmem_park_s;
    __shared__ unsigned smax[4];                         // bit patterns of max |K1|, |K0b|, |symb|, |w|
    __shared__ double sredd[32];                         // 4 sample warps x 8 cost sums of a tile (mean mode)

    // ---- one-time per CTA: weights -> scaled, split fp16 operands in canonical layout (padded units have zero weights:
    //      they contribute exactly nothing to any contraction, see DESIGN.md)
    // pass 1: symb = [A'A | c_w] in fp32 (parked in the X operand's space, free until the first evaluation) and the largest
    // magnitude of each matrix
    float* symb = reinterpret_cast<float*>(sX);          // [KS][KS], symb[n = k'][k]: (A'A)[k][k'] | c_w[k'] in column D | 0
    if (tid < 4) smax[tid] = 0u;
    __syncthreads();
    {
        float m1 = 0.f, m0 = 0.f, ms = 0.f, mw = 0.f;
        for (int i = tid; i < m * m; i += NT) m1 = fmaxf(m1, fabsf(A.K1[i]));
        for (int i = tid; i < m * D; i += NT) m0 = fmaxf(m0, fabsf(A.K0[i]));
        for (int i = tid; i < m; i += NT) { m0 = fmaxf(m0, fabsf(A.b0[i])); mw = fmaxf(mw, fabsf(A.w[i])); }
        for (int i = tid; i < KS * KS; i += NT) {
            const int kp = i / KS, k = i % KS;
            float v = 0.f;
            if (kp < D && k < D) { for (int q = 0; q < A.r; ++q) v = fmaf(A.A[q * D + k], A.A[q * D + kp], v); }
            else if (kp < D && k == D) v = A.c_w[kp];
            symb[i] = v;
            ms = fmaxf(ms, fabsf(v));
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, off)); m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, off));
            ms = fmaxf(ms, __shfl_xor_sync(0xffffffffu, ms, off)); mw = fmaxf(mw, __shfl_xor_sync(0xffffffffu, mw, off));
        }
        if ((tid & 31) == 0) {                           // non-negative floats order like their bit patterns (NaN sorts above inf)
            atomicMax(&smax[0], __float_as_uint(m1)); atomicMax(&smax[1], __float_as_uint(m0));
            atomicMax(&smax[2], __float_as_uint(ms)); atomicMax(&smax[3], __float_as_uint(mw));
        }
    }
    __syncthreads();
    // Scales (powers of two, the same in every thread and every CTA).  K1 -> s1.  Y and V carry s_w (w is stored pre-scaled, so
    // the epilogues pay nothing for it), hence GEMM-4's accumulator holds s_w s0 g and symb, which lands in the same
    // accumulator from the unscaled S, is scaled by s_w s0; s0 keeps both K0b and that product below 2^14.
    const float s_w = pow2_scale(__uint_as_float(smax[3]), 6);
    const float s1 = pow2_scale(__uint_as_float(smax[0]), 13);
    const float sx = A.sx;
    const float s0 = pow2_scale(fmaxf(__uint_as_float(smax[1]), __uint_as_float(smax[2]) * (s_w / sx)), 13);
    const float ssy = s0 * s_w;                          // scale of GEMM-4's accumulator; symb itself carries ssy / sx
    // reciprocal scales with the accumulate-bias compensation of each contraction folded in (3 MMAs per 16-deep k-block)
    const float kShrink = 1.89e-8f * A.bias_f;
    const float r_o = (1.f / (s0 * sx)) * (1.f + kShrink * 3.f * (KS / 16));             // GEMM-1: o = acc r_o
    const float r_a = (1.f / s1) * (1.f + kShrink * 3.f * (mp / 16));                    // GEMM-2: a1 = acc r_a;  GEMM-3: s_w z1 = acc r_a
    const float r_g = (1.f / ssy) * (1.f + kShrink * 3.f * ((mp + KS) / 16));            // GEMM-4: g = acc r_g
    const float r_q = (1.f / ssy) * (1.f + kShrink * 3.f * (KS / 16));                   // terminal S.symb' on its own
    const float r_ac = r_a * kTwoLog2e;                  // ... for tanh2_w()
    const float hz = A.h * r_a;                          // s_w v = tanh(o) (s_w w + h (s_w z1))
    const float inv_sw = 1.f / s_w, ssym = ssy / sx;
    for (int i = tid; i < mp * (mp / 8); i += NT) {     // K1[o][k0..k0+8)
        const int o = i / (mp / 8), k0 = (i % (mp / 8)) * 8;
        float v[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) v[e] = (o < m && k0 + e < m) ? A.K1[o * m + k0 + e] * s1 : 0.f;
        store_chunk2(sK1, pK1, o, k0, mp, v);
    }
    for (int i = tid; i < mp * (KS / 8); i += NT) {     // K0b[j][k]: K0 | b0 | 0
        const int j = i / (KS / 8), k0 = (i % (KS / 8)) * 8;
        float v[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) { const int k = k0 + e; v[e] = (j >= m) ? 0.f : ((k < D) ? A.K0[j * D + k] : (k == D ? A.b0[j] : 0.f)) * s0; }
        store_chunk2(sK0, pK0, j, k0, KS, v);
    }
    for (int i = tid; i < KS * (KS / 8); i += NT) {
        const int kp = i / (KS / 8), k0 = (i % (KS / 8)) * 8;
        float v[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) v[e] = symb[kp * KS + k0 + e] * ssym;
        store_chunk2(sSy, pSy, kp, k0, KS, v);
    }
    for (int i = tid; i < mp; i += NT) {
        const float bv = (i < m) ? A.b1[i] : 0.f;
        sb1[i] = bv; sb1c[i] = bv * kTwoLog2e; sw[i] = (i < m) ? A.w[i] * s_w : 0.f;
    }
    if (tid < KS) scw[tid] = (tid < D) ? A.c_w[tid] : 0.f;
    if (warp == 0) {
        const bool own = SH::PARK && A.park_col < 0;
        tmem_alloc(smem_u32(&tmem_base_s), A.tmem_cols, !own);
        if (own) tmem_alloc(smem_u32(&tmem_park_s), 32, true);        // (own block only for SPLIT == 1, PW == 32 shapes)
    }
    if (tid == 0) mbar_init(smem_u32(&mbar), 1);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const int C = (mp > KS) ? mp : KS;
    const unsigned tacc = tmem_base_s;                   // the accumulator, columns [0, C)
    const unsigned tpark = !SH::PARK ? 0u : (A.park_col < 0 ? tmem_park_s : tacc + (unsigned)A.park_col) + (unsigned)(hf * SH::PW);
    const unsigned tT0 = tacc + C;                       // tanh(o); at the terminal evaluation afterwards S.symb'
    const unsigned lane_bits = (unsigned)((warp & 3) * 32) << 16;
    const unsigned mb = smem_u32(&mbar);
    int phase = 0;
    const unsigned idesc_m_k = umma_idesc_f16_b(128, mp, 0), idesc_m_mn = umma_idesc_f16_b(128, mp, 1);
    const unsigned idesc_s_mn = umma_idesc_f16_b(128, KS, 1), idesc_s_k = umma_idesc_f16_b(128, KS, 0);
    const unsigned sboM = (unsigned)(mp >> 3) * 128;     // 8-row-group stride of an operand with K = mp
    constexpr unsigned sboS = (unsigned)(KS >> 3) * 128; // ... with K = KS
    // hi-plane descriptors (k-block 0); the lo plane and k-blocks are reached by adding 16-byte-unit offsets
    const unsigned long long dX = umma_desc(smem_u32(sX), 128, sboM), dS = umma_desc(smem_u32(sS), 128, sboS);
    const unsigned long long dK1k = umma_desc(smem_u32(sK1), 128, sboM), dK1n = umma_desc(smem_u32(sK1), sboM, 128);
    const unsigned long long dK0k = umma_desc(smem_u32(sK0), 128, sboS), dK0n = umma_desc(smem_u32(sK0), sboS, 128);
    const unsigned long long dSy = umma_desc(smem_u32(sSy), 128, sboS);
    const unsigned qX = pX >> 4, qS = pS >> 4, qK1 = pK1 >> 4, qK0 = pK0 >> 4, qSy = pSy >> 4;    // plane strides, 16-byte units
    const unsigned kK1n = (2 * sboM) >> 4;               // k-block step of K1 read MN-major (16 rows)
    constexpr unsigned kK0n = (2 * sboS) >> 4;           // ... of K0b read MN-major

    // publish my operand writes and let thread 0 issue `issue`; mma_wait() then blocks until the tensor core is done
    // The issuing warp rotates with the GEMM (warp g issues GEMM-g): the MMA issue instructions are then spread over
    // four warps instead of lengthening warp 0's critical path in every round.  Ordering is safe: each GEMM is issued
    // after a block barrier that follows every thread's wait on the previous GEMM's commit.
    auto mma_issue = [&](int who, auto issue) {
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (warp_u == who) {                             // warp-uniform branch, then one elected lane
            if (elect_one_sync()) {
                tc_fence_after();
                issue();
                umma_commit(mb);
            }
            __syncwarp();
        }
    };
    auto mma_wait = [&] {
        mbar_wait(mb, phase);
        phase ^= 1;
        tc_fence_after();
    };
    auto run_mma = [&](int who, auto issue) { mma_issue(who, issue); mma_wait(); };

    // calcLHQW / calcGradpH / calcCtrls in registers, in two parts (Cross2D.py:69-87,133-165; Quadcopter.py:65-113,160-197).
    // Part 1 needs only x and runs while GEMM-1 is in flight: the terrain and interaction costs (q, w) of Cross2D, or the
    // thrust direction (f7, f8, f9) of the quadcopter, returned in xq[0..3).
    // the problem's python-double parameters, rounded to fp32 once (the reference rounds them to the tensor dtype at use);
    // left as doubles inside the loop they cost FP64-pipe compares / converts in every evaluation
    const bool hasQ = (pr.obstacle != 0) && (pr.kind == 0 || pr.alph_Q > 0.0), hasW = (pr.alph_W != 0.0), posQ = (pr.alph_Q > 0.0);
    const float f_alphQ = float(pr.alph_Q), f_alphW = float(pr.alph_W), f_cut = float(pr.cutW), f_c2 = float(2 * pr.r * pr.r);
    const float f_mass = float(pr.mass), f_grav = float(pr.grav), f_uscale = float(-1.0 / (2.0 * pr.mass));
    auto problem_x = [&](const float (&x)[d], float (&xq)[3]) {
        if constexpr (KIND == 2) {
            float sps, cps, sth, cth, sph, cph;
            sincosf(x[3], &sps, &cps); sincosf(x[4], &sth, &cth); sincosf(x[5], &sph, &cph);
            xq[0] = sps * sph + cps * sth * cph; xq[1] = -cps * sph + sps * sth * cph; xq[2] = cth * cph;
        } else {
            constexpr int NA = SH::NA, DIM = SH::DIM;
            float q = 0.f, w = 0.f;
            if (hasQ) {
#pragma unroll
                for (int a = 0; a < NA; ++a) q += terrain_agent<float>(pr, x[a * DIM], x[a * DIM + 1], DIM == 3 ? x[a * DIM + DIM - 1] : 0.f);
            }
            if (hasW && NA >= 2) {
                const float cut = f_cut, c2 = f_c2;
                if constexpr (NA == 2) {               // Cross2D.py:133-145: no "== 1" rule here
                    float d2 = 0.f;
#pragma unroll
                    for (int c = 0; c < DIM; ++c) { const float df = x[c] - x[DIM + c]; d2 = fmaf(df, df, d2); }
                    const float dd = sqrtf(d2);
                    if (dd < cut) w = r_exp(-(dd * dd) / c2);
                } else {                               // Cross2D.py:147-160; same fast path as interaction_pairs()
                    const float guard = cut * cut * 1.0001f;
                    float dmin = guard;
#pragma unroll
                    for (int i = 0; i < NA - 1; ++i)
#pragma unroll
                        for (int j = i + 1; j < NA; ++j) {
                            float d2 = 0.f;
#pragma unroll
                            for (int c = 0; c < DIM; ++c) { const float df = x[i * DIM + c] - x[j * DIM + c]; d2 = fmaf(df, df, d2); }
                            dmin = fminf(dmin, d2);
                        }
                    if (dmin < guard) {                // rare: redo the pairs exactly, in the same order
#pragma unroll
                        for (int i = 0; i < NA - 1; ++i)
#pragma unroll
                            for (int j = i + 1; j < NA; ++j) {
                                float d2 = 0.f;
#pragma unroll
                                for (int c = 0; c < DIM; ++c) { const float df = x[i * DIM + c] - x[j * DIM + c]; d2 = fmaf(df, df, d2); }
                                if (d2 < guard) {
                                    const float dd = sqrtf(d2);
                                    if (dd < cut) {
                                        const float e = r_exp(-(dd * dd) / c2);
                                        if (e != 1.f) w += e;      // pairs whose Gaussian rounds to 1 are dropped (mask2)
                                    }
                                }
                            }
                    }
                }
            }
            xq[0] = q; xq[1] = w; xq[2] = 0.f;
        }
    };
    // grad Phi at s = [xs, t]; problem_x(xs) runs between the issue of GEMM-1 and the wait for it
    const int cbeg = hf * (mp / SPLIT), cend = cbeg + mp / SPLIT;      // my hidden units
    auto chain = [&](const float (&xs)[d], float t, float (&g)[KS], bool terminal, float& phi_out, float (&xq)[3]) {
#pragma unroll
        for (int c0 = 0; c0 < KS; c0 += 8) {             // S operand row: [x, t, 1, 0..]
            if (SPLIT > 1 && ((c0 >> 3) % SPLIT) != hf) continue;
            float v[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) { const int k = c0 + e; v[e] = sx * ((k < d) ? xs[k < d ? k : 0] : (k == d ? t : (k == D ? 1.f : 0.f))); }
            store_chunk2(sS, pS, row, c0, KS, v);
        }
        mma_issue(0, [&] {                               // GEMM-1: s0 O = S . K0b'
#pragma unroll
            for (int kb = 0; kb < KS / 16; ++kb) mma3(tacc, dS + kb * 16, qS, dK0k + kb * 16, qK0, idesc_m_k, kb > 0);
        });
        if (!terminal) problem_x(xs, xq);
        mma_wait();
        for (int c0 = cbeg; c0 < cend; c0 += CH) {            // u0 = act(o) -> X operand, tanh(o) -> TMEM
            float v[CH], tt[CH];
            tmem_ld<CH>(tacc + lane_bits + c0, v);
#pragma unroll
            for (int i = 0; i < CH; i += 2) {
                float2 av, tv;
                act_tanh2(make_float2(v[i], v[i + 1]), make_float2(r_o, r_o), av, tv);
                v[i] = av.x; v[i + 1] = av.y; tt[i] = tv.x; tt[i + 1] = tv.y;
            }
            tmem_st<CH>(tT0 + lane_bits + c0, tt);
#pragma unroll
            for (int q = 0; q < CH / 8; ++q) store_chunk2(sX, pX, row, c0 + q * 8, mp, v + q * 8);
        }
        run_mma(1, [&] {                                 // GEMM-2: s1 A1 = U0 . K1'  (B K-major)
            for (int kb = 0; kb < mp / 16; ++kb) mma3(tacc, dX + kb * 16, qX, dK1k + kb * 16, qK1, idesc_m_k, kb > 0);
        });
        float phiN = 0.f;
        for (int c0 = cbeg; c0 < cend; c0 += CH) {            // s_w y = tanh(a1 + b1) * (s_w w) -> X operand
            float v[CH];
            tmem_ld<CH>(tacc + lane_bits + c0, v);
#pragma unroll
            for (int q = 0; q < CH / 8; ++q) {
                float u8[8];
                if (terminal) load_chunk2(sX, pX, row, c0 + q * 8, mp, u8);      // u0, before it is overwritten
                float b8[8], w8[8];                       // 16-byte loads of the bias and w (16-byte aligned by construction)
                const float* sb = terminal ? sb1 : sb1c;
                *reinterpret_cast<float4*>(b8) = *reinterpret_cast<const float4*>(sb + c0 + q * 8);
                *reinterpret_cast<float4*>(b8 + 4) = *reinterpret_cast<const float4*>(sb + c0 + q * 8 + 4);
                *reinterpret_cast<float4*>(w8) = *reinterpret_cast<const float4*>(sw + c0 + q * 8);
                *reinterpret_cast<float4*>(w8 + 4) = *reinterpret_cast<const float4*>(sw + c0 + q * 8 + 4);
                if (terminal) {
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        float av, tv;
                        act_tanh(fmaf(v[q * 8 + e], r_a, b8[e]), av, tv);
                        phiN = fmaf(w8[e], u8[e] + A.h * av, phiN);        // s_w w.u1 (unscaled at the end)
                        v[q * 8 + e] = tv * w8[e];
                    }
                } else {
#pragma unroll
                    for (int e = 0; e < 8; e += 2) {
                        const float2 y = tanh2_w(make_float2(v[q * 8 + e], v[q * 8 + e + 1]), make_float2(r_ac, r_ac),
                                                 make_float2(b8[e], b8[e + 1]), make_float2(w8[e], w8[e + 1]));
                        v[q * 8 + e] = y.x; v[q * 8 + e + 1] = y.y;
                    }
                }
                store_chunk2(sX, pX, row, c0 + q * 8, mp, v + q * 8);
            }
        }
        if (SPLIT > 1 && terminal && hf > 0) sphi[(hf - 1) * 128 + row] = phiN;
        run_mma(2, [&] {                                 // GEMM-3: s_w s1 Z1 = (s_w Y) . K1  (the same buffer, MN-major)
            for (int kb = 0; kb < mp / 16; ++kb) mma3(tacc, dX + kb * 16, qX, dK1n + kb * kK1n, qK1, idesc_m_mn, kb > 0);
        });
        for (int c0 = cbeg; c0 < cend; c0 += CH) {            // s_w v = tanh(o) * (s_w w + h s_w z1acc) -> X operand
            float v[CH], tt[CH];
            tmem_ld2<CH>(tacc + lane_bits + c0, v, tT0 + lane_bits + c0, tt);
#pragma unroll
            for (int i = 0; i < CH; i += 4) {
                const float4 w4 = *reinterpret_cast<const float4*>(sw + c0 + i);
                const float2 a = __fmul2_rn(make_float2(tt[i], tt[i + 1]), __ffma2_rn(make_float2(hz, hz), make_float2(v[i], v[i + 1]), make_float2(w4.x, w4.y)));
                const float2 b = __fmul2_rn(make_float2(tt[i + 2], tt[i + 3]), __ffma2_rn(make_float2(hz, hz), make_float2(v[i + 2], v[i + 3]), make_float2(w4.z, w4.w)));
                v[i] = a.x; v[i + 1] = a.y; v[i + 2] = b.x; v[i + 3] = b.y;
            }
#pragma unroll
            for (int q = 0; q < CH / 8; ++q) store_chunk2(sX, pX, row, c0 + q * 8, mp, v + q * 8);
        }
        run_mma(3, [&] {                                 // GEMM-4: s_w s0 G = (s_w V) . K0b (MN-major view) + S . (s_w s0 symb)'
            for (int kb = 0; kb < mp / 16; ++kb) mma3(tacc, dX + kb * 16, qX, dK0n + kb * kK0n, qK0, idesc_s_mn, kb > 0);
            // the terminal evaluation needs S.symb' on its own (Phi's quadratic term): it goes to the free tanh columns
            const unsigned qm = terminal ? tT0 : tacc;
#pragma unroll
            for (int kb = 0; kb < KS / 16; ++kb) mma3(qm, dS + kb * 16, qS, dSy + kb * 16, qSy, idesc_s_k, terminal ? (kb > 0) : 1);
        });
        const float rg = terminal ? (1.f / ssy) * (1.f + kShrink * 3.f * (mp / 16)) : r_g;
#pragma unroll
        for (int c0 = 0; c0 < KS; c0 += 16) {
            tmem_ld<16>(tacc + lane_bits + c0, g + c0);
#pragma unroll
            for (int i = 0; i < 16; i += 2) {
                const float2 gg = __fmul2_rn(make_float2(g[c0 + i], g[c0 + i + 1]), make_float2(rg, rg));
                g[c0 + i] = gg.x; g[c0 + i + 1] = gg.y;
            }
        }
        if (terminal) {                                   // Phi = w.u1 + 0.5 s'A'A s + c_w.s + c_b  (Phi.py:96)
            float gq[KS];
#pragma unroll
            for (int c0 = 0; c0 < KS; c0 += 16) tmem_ld<16>(tT0 + lane_bits + c0, gq + c0);
            float quad = 0.f, lin = 0.f;
#pragma unroll
            for (int k = 0; k < D; ++k) {
                const float sv = (k < d) ? xs[k < d ? k : 0] : t, gk = gq[k] * r_q;
                quad = fmaf(sv, gk - scw[k], quad);      // gq carries c_w (column D of symb)
                lin = fmaf(scw[k], sv, lin);
                g[k] += gk;
            }
            if (SPLIT > 1) {                              // written before GEMM-3's barrier; only the hf = 0 thread's sum is used
#pragma unroll
                for (int q = 1; q < SPLIT; ++q) phiN += sphi[(q - 1) * 128 + row];
            }
            phi_out = phiN * inv_sw + 0.5f * quad + (lin + A.c_b[0]);
        }
    };

    // Part 2, after grad Phi: dx = -grad_p H, cost rates L, HJ = |Phi_t - H|, Q, W; uctrl = the quadcopter thrust
    auto problem = [&](const float (&x)[d], const float (&g)[KS], const float (&xq)[3], float (&dx)[d], float (&rate)[4], float& uctrl) {
        if constexpr (KIND == 2) {
            const float f7 = xq[0], f8 = xq[1], f9 = xq[2];
            const float fp = f7 * g[6] + f8 * g[7] + f9 * g[8];
            const float u = f_uscale * fp;
            const float sq = g[9] * g[9] + g[10] * g[10] + g[11] * g[11];
            float L = f_alphQ * 0.f;
            L = L + 2.f + u * u + 0.25f * sq;
            const float um = u / f_mass;
            const float xv = x[6] * g[0] + x[7] * g[1] + x[8] * g[2];
            const float xw = x[9] * g[3] + x[10] * g[4] + x[11] * g[5];
            const float H = 0.f - L - xv - xw - um * fp + f_grav * g[8] + 0.5f * sq;
            rate[0] = L; rate[1] = fabsf(g[d] - H); rate[2] = 0.f; rate[3] = 0.f;
#pragma unroll
            for (int c = 0; c < 6; ++c) dx[c] = x[6 + c];
            dx[6] = -(-um * f7); dx[7] = -(-um * f8); dx[8] = -(-um * f9 + f_grav);
#pragma unroll
            for (int c = 9; c < 12; ++c) dx[c] = -(0.5f * g[c]);
            uctrl = u;
        } else {
            float pp = 0.f, w = xq[1];
            const float q = xq[0];
#pragma unroll
            for (int r = 0; r < d; ++r) pp = fmaf(g[r], g[r], pp);
            float Qret, L;
            if (pr.kind == 0) { Qret = f_alphQ * q; L = 0.5f * pp + Qret; }     // Cross2D returns Q pre-scaled (quirk 6)
            else { Qret = posQ ? q : 0.f; L = 0.5f * pp + f_alphQ * Qret; }
            if (hasW) L = L + f_alphW * w; else w = 0.f;
            const float H = -L + pp;
            rate[0] = L; rate[1] = fabsf(g[d] - H); rate[2] = Qret; rate[3] = w;
#pragma unroll
            for (int c = 0; c < d; ++c) dx[c] = -g[c];
            uctrl = 0.f;
        }
    };

    double csum[7] = {0, 0, 0, 0, 0, 0, 0};
    long long cnt = 0;
    constexpr bool inter = INTER;
    const int ntp1 = A.nt + 1;
    for (int tile = blockIdx.x; tile < A.ntiles; tile += gridDim.x) {
        const long long s0 = (long long)tile * 128;
        const int nvalid = (int)((A.n - s0 < 128) ? (A.n - s0) : 128);
        const bool valid = row < nvalid;
        const bool writer = valid && hf == 0;                          // one thread per sample writes results
        const long long gs = s0 + (valid ? row : nvalid - 1);        // padding threads replay the last valid sample
        float z0[NZ], za[SH::PARK ? SH::PW : NZ];
        if (SH::PARK) {
#pragma unroll
            for (int c = 0; c < SH::PW; ++c) za[c] = 0.f;
        }
#pragma unroll
        for (int c = 0; c < d; ++c) z0[c] = A.x[gs * d + c];
#pragma unroll
        for (int c = d; c < NZ; ++c) z0[c] = 0.f;
        // intermediates: trajectory column `col` of (row c of zFull | row c of ctrlFull).  With a staging buffer the warp
        // writes 128 contiguous bytes per (step, row) and tc_untile_kernel transposes into the reference layout
        // [n, rows, nt+1] afterwards; without one (allocation failed) each thread writes its strided 4-byte element.
        // (addresses are recomputed at each use: nothing of this stays live in the mean / noMean modes)
        auto put_z = [&](int c, int col, float v) {
            if (A.stage) A.stage[(((size_t)tile * ntp1 + col) * (NZ + NCTRL) + c) * 128 + row] = v;
            else A.out_b[(gs * NZ + c) * ntp1 + col] = v;
        };
        auto put_u = [&](int c, int col, float v) {
            if (A.stage) A.stage[(((size_t)tile * ntp1 + col) * (NZ + NCTRL) + NZ + c) * 128 + row] = v;
            else A.out_c[(gs * NCTRL + c) * ntp1 + col] = v;
        };
        if (inter && writer) {                                         // zFull[:,:,0] = z, ctrlFull[:,:,0] = 0 (OCflow.py:37-43)
#pragma unroll
            for (int c = 0; c < NZ; ++c) put_z(c, 0, z0[c]);
#pragma unroll
            for (int c = 0; c < NCTRL; ++c) put_u(c, 0, 0.f);
        }
        // ONE call site for the chain: the evaluations of a rollout are a flat host-built sequence (TcEval); `xs` always
        // holds the next evaluation's input.
        float g[KS], dx[d], xs[d], phi1 = 0.f;
#pragma unroll
        for (int c = 0; c < d; ++c) xs[c] = z0[c];
        const float4* etab = reinterpret_cast<const float4*>(A.evals);
        for (int it = 0; it < A.nevals; ++it) {
            const float4 ef = __ldg(etab + 2 * it);
            const int4 ei = __ldg(reinterpret_cast<const int4*>(etab + 2 * it + 1));
            const float tcur = ef.x, wgt = ef.y, cnext = ef.z, hstep = ef.w;
            const int k = ei.x, kind = ei.y, first = ei.z, last = ei.w;
            const bool term = (kind == 2);
            float xq[3];
            if (SH::PARK) tmem_st<SH::PW>(tpark + lane_bits, za);
            chain(xs, tcur, g, term, phi1, xq);
            if (SH::PARK) tmem_ld<SH::PW>(tpark + lane_bits, za);
            if (term) break;
            float rate[4], uc;
            problem(xs, g, xq, dx, rate, uc);
            if (INTER && kind == 1) {                                // controls at the new state, OLD time (quirk 3)
                if (writer) {
#pragma unroll
                    for (int c = 0; c < NZ; ++c) put_z(c, k + 1, z0[c]);
                    if constexpr (KIND == 2) {
                        put_u(0, k + 1, uc);
#pragma unroll
                        for (int c = 1; c < 4; ++c) put_u(c, k + 1, -0.5f * g[8 + c]);
                    } else {
#pragma unroll
                        for (int c = 0; c < d; ++c) put_u(c, k + 1, -g[c]);
                    }
                }
                continue;
            }
#pragma unroll
            for (int c = 0; c < NZ; ++c) {                           // RK combination (OCflow.py:143-184)
                float kk;
                if (c < d) kk = (KIND == 2) ? hstep * dx[c < d ? c : 0] : hstep * (-g[c]);
                else kk = hstep * rate[c >= d ? c - d : 0];
                za[c] = (first ? z0[c] : za[c]) + wgt * kk;
                if (c < d) dx[c < d ? c : 0] = kk;
            }
            if (!last) {
#pragma unroll
                for (int c = 0; c < d; ++c) xs[c] = z0[c] + cnext * dx[c];
            } else {
#pragma unroll
                for (int c = 0; c < NZ; ++c) z0[c] = za[c];
#pragma unroll
                for (int c = 0; c < d; ++c) xs[c] = z0[c];
            }
        }
        // terminal block (OCflow.py:58-90): xs = x(T), g = grad Phi(x(T), T), phi1 = Phi(x(T), T)
        const float* xt = static_cast<const float*>(pr.xtarget);
        float cG = 0.f, hjg = 0.f;
#pragma unroll
        for (int c = 0; c < d; ++c) {
            const float res = xs[c] - xt[c];
            cG = fmaf(res, res, cG);
            hjg += fabsf(g[c] - A.alph0 * res);
        }
        cG *= 0.5f;
        const float cost[7] = {z0[d], cG, z0[d + 1], fabsf(phi1 - A.alph0 * cG), hjg, z0[d + 2], z0[d + 3]};
        if (A.mode == 0) {
            // deterministic CTA sum: lanes -> warp (shuffle tree), warps -> thread 0 in fixed order
#pragma unroll
            for (int q = 0; q < 7; ++q) {
                double v = valid ? (double)cost[q] : 0.0;              // double: the sums must not depend on the tiling
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
                if ((tid & 31) == 0 && hf == 0) sredd[warp * 8 + q] = v;
            }
            __syncthreads();
            if (tid == 0) {
                for (int q = 0; q < 7; ++q) csum[q] += ((sredd[q] + sredd[8 + q]) + sredd[16 + q]) + sredd[24 + q];
                cnt += nvalid;
            }
            __syncthreads();
        } else if (A.mode == 1 && writer) {
            float* o = A.out_a + gs * 8;
            o[0] = cost[0] + A.alph0 * cost[1] + A.alph3 * cost[2] + A.alph4 * cost[3] + A.alph5 * cost[4];   // OCflow.py:75
#pragma unroll
            for (int q = 0; q < 7; ++q) o[1 + q] = cost[q];
        }
    }
    if (A.mode == 0 && A.partials && tid == 0) {
        for (int q = 0; q < 7; ++q) A.partials[blockIdx.x * 8 + q] = csum[q];
        A.partials[blockIdx.x * 8 + 7] = (double)cnt;
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tmem_dealloc(tacc, A.tmem_cols);
        if (SH::PARK && A.park_col < 0) tmem_dealloc(tpark, 32);
    }
}

// host: the flat evaluation sequence of one rollout from the stage-time table (nt x 5 doubles, noc_stage_times)
static inline void tc_build_evals(const double* tab, int nt, int stepper, bool inter, double t_end, std::vector<TcEval>& ev) {
    const int nstage = (stepper == NOC_STEP_RK4) ? 4 : (stepper == NOC_STEP_RK1 ? 1 : 0);
    ev.clear();
    for (int k = 0; k < nt; ++k) {
        const double* tt = tab + 5 * k;
        for (int st = 0; st < nstage; ++st) {
            TcEval e;
            e.h = (float)tt[4]; e.k = k; e.kind = 0; e.first = (st == 0); e.last = (st == nstage - 1);
            e.t = (float)tt[0]; e.wgt = 1.f; e.cnext = 0.f;
            if (nstage == 4) {                                      // OCflow.py:172-182
                const double w[4] = {1.0 / 6.0, 2.0 / 6.0, 2.0 / 6.0, 1.0 / 6.0}, c[4] = {0.5, 0.5, 1.0, 0.0};
                const double ts[4] = {tt[0], tt[1], tt[1], tt[2]};
                e.t = (float)ts[st]; e.wgt = (float)w[st]; e.cnext = (float)c[st];
            }
            ev.push_back(e);
        }
        if (inter) {
            TcEval e;
            e.t = (float)tt[3]; e.wgt = 0.f; e.cnext = 0.f; e.h = (float)tt[4]; e.k = k; e.kind = 1; e.first = 0; e.last = 0;
            ev.push_back(e);
        }
    }
    TcEval e;
    e.t = (float)t_end; e.wgt = 0.f; e.cnext = 0.f; e.h = 0.f; e.k = 0; e.kind = 2; e.first = 0; e.last = 0;
    ev.push_back(e);
}

// builds the evaluation sequence of the rollout `c` and uploads it (stream-ordered) into `buf` for A.evals / A.nevals
template <class Args>
cudaError_t tc_upload_evals(const RolloutCall<float>& c, Args& A, ScratchBuf& buf) {
    std::vector<TcEval> ev;
    tc_build_evals(c.host_times, c.nt, c.stepper, c.mode == NOC_MODE_INTERMEDIATES, c.t_end, ev);
    A.nevals = (int)ev.size();
    cudaError_t e = buf.alloc(sizeof(TcEval) * ev.size(), c.stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(buf.p, ev.data(), sizeof(TcEval) * ev.size(), cudaMemcpyHostToDevice, c.stream);   // pageable: staged before return
    A.evals = buf.as<TcEval>();
    return e;
}

// staging buffer [tile][step][row][128] -> zFull [n, NZ, ntp1] and ctrlFull [n, NCTRL, ntp1] (last dim contiguous).
// One block per (tile, row): coalesced 512-byte reads, a padded shared-memory transpose, (nt+1)-float contiguous writes.
constexpr int kUntileSteps = 64;
static __global__ void __launch_bounds__(128) tc_untile_kernel(const float* __restrict__ stage, float* __restrict__ zFull,
                                                               float* __restrict__ ctrlFull, long long n, int ntp1, int NZ, int NCTRL) {
    __shared__ float tl[kUntileSteps * 129];
    const int t = blockIdx.x, r = blockIdx.y, R = NZ + NCTRL, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long s0 = (long long)t * 128;
    const int nvalid = (int)((n - s0 < 128) ? (n - s0) : 128);
    float* out = (r < NZ) ? zFull : ctrlFull;
    const int rr = (r < NZ) ? r : r - NZ, RR = (r < NZ) ? NZ : NCTRL;
    for (int k0 = 0; k0 < ntp1; k0 += kUntileSteps) {
        const int kc = (ntp1 - k0 < kUntileSteps) ? (ntp1 - k0) : kUntileSteps;
        if ((int)threadIdx.x < nvalid)
            for (int k = 0; k < kc; ++k) tl[k * 129 + threadIdx.x] = stage[(((size_t)t * ntp1 + k0 + k) * R + r) * 128 + threadIdx.x];
        __syncthreads();
        for (int l = warp; l < nvalid; l += 4)
            for (int k = lane; k < kc; k += 32) out[((s0 + l) * RR + rr) * ntp1 + k0 + k] = tl[k * 129 + l];
        __syncthreads();
    }
}

template <class SH>
int launch_tc(const RolloutCall<float>& c) {
    const int smem_limit = c.smem_limit;
    cudaStream_t st = c.stream;
    TcArgs A;
    memset(&A, 0, sizeof A);
    copy_common(A, c);
    A.m = c.m; A.mp = align_up(c.m, SH::KIND == 2 ? 64 : 16); A.h = c.h; A.r = c.r;   // mp: as tc_shape_id (noc_api.cu)
    A.K0 = c.raw.K[0]; A.b0 = c.raw.b[0]; A.K1 = c.raw.K[1]; A.b1 = c.raw.b[1]; A.w = c.raw.w; A.A = c.raw.A; A.c_w = c.raw.c_w; A.c_b = c.raw.c_b;
    A.stepper = c.stepper; A.t_end = (float)c.t_end;
    ScratchBuf evals, partials, stage;
    NOC_CUDA(tc_upload_evals(c, A, evals));
    const size_t smem = tc_smem_bytes(A.mp, SH::KS);
    auto kern = (A.mode == NOC_MODE_INTERMEDIATES) ? rollout_tc_kernel<SH, true> : rollout_tc_kernel<SH, false>;
    if (smem + 1024 > (size_t)smem_limit) return fail(NOC_ERR_NOMEM, "tensor-core rollout needs %zu B of shared memory", smem);
    NOC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // resident CTAs per SM from the kernel's own resource use (registers, shared memory incl. the 1 KB the driver reserves
    // per block, TMEM columns: a CTA that cannot get its columns would only wait in tcgen05.alloc)
    int occ_api = 0;
    NOC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_api, kern, SH::NT, smem));
    cudaFuncAttributes fa;
    NOC_CUDA(cudaFuncGetAttributes(&fa, kern));
    int dev = 0, regs_sm = 65536, smem_sm = 233472;
    NOC_CUDA(cudaGetDevice(&dev));
    NOC_CUDA(cudaDeviceGetAttribute(&regs_sm, cudaDevAttrMaxRegistersPerMultiprocessor, dev));
    NOC_CUDA(cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev));
    // TMEM columns: accumulator | tanh(o), in one power-of-two block; PARK shapes add the parked
    // RK accumulator: in the block's spare columns when there are any, else (one thread per sample, 32 columns) in a second
    // 32-column block so that e.g. swap12 stays at 160 columns = 3 CTAs per SM, else by growing the block
    const int tmem_used = 2 * std::max(A.mp, SH::KS), park_need = SH::PW * SH::SPLIT;
    A.tmem_cols = tc_tmem_cols(A.mp, SH::KS);
    {   // scale 2^e of the S operand (states beyond 2^(15-e) would overflow fp16: 1024 at the default; experiments: NOC_TC_SX = e)
        int ex = 5;
        if (const char* e = getenv("NOC_TC_SX")) ex = atoi(e);
        A.sx = ldexpf(1.f, ex);
        A.bias_f = 1.f;
        if (const char* e = getenv("NOC_TC_BIAS")) A.bias_f = (float)atof(e);
    }
    A.park_col = -1;
    if (SH::PARK) {
        if (A.tmem_cols - tmem_used >= park_need) A.park_col = tmem_used;
        else if (park_need != 32) {
            while (A.tmem_cols - tmem_used < park_need) A.tmem_cols *= 2;
            if (A.tmem_cols > 512) return fail(NOC_ERR_NOMEM, "no TMEM columns left for the parked state");
            A.park_col = tmem_used;
        }
    }
    const int by_regs = regs_sm / (align_up(std::max(fa.numRegs, 1), 8) * SH::NT);
    const int tmem_per_cta = A.tmem_cols + ((SH::PARK && A.park_col < 0) ? 32 : 0);
    // A CTA that cannot get its TMEM columns blocks inside tcgen05.alloc, and PARK shapes allocate in two steps: if more CTAs
    // than 512 / tmem_per_cta ever shared an SM (this launch's, or another stream's launch of the same kernel) they could each
    // hold the first block and wait forever for the second.  Make it structurally impossible: shared memory is the per-SM
    // resource every co-resident CTA needs, so request enough of it that at most 512 / tmem_per_cta CTAs fit.
    size_t smem_req = smem;
    {
        const int cap = std::max(1, 512 / tmem_per_cta);
        if ((int)(smem_sm / (smem_req + fa.sharedSizeBytes + 1024)) > cap) {
            smem_req = (size_t)smem_sm / cap - fa.sharedSizeBytes - 1024;
            smem_req = std::min(smem_req, (size_t)smem_limit) & ~(size_t)15;
            while ((int)(smem_sm / (smem_req + fa.sharedSizeBytes + 1024)) > cap && smem_req + 16 <= (size_t)smem_limit) smem_req += 16;
            NOC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_req));
        }
    }
    const int by_smem = (int)(smem_sm / (smem_req + fa.sharedSizeBytes + 1024));
    int per_sm = std::min(std::min(by_regs, by_smem), 512 / tmem_per_cta);
    if (getenv("NOC_DEBUG"))
        fprintf(stderr, "[noc] tc occupancy: api=%d regs=%d (->%d) smem->%d tmem->%d\n", occ_api, fa.numRegs, by_regs, by_smem, 512 / tmem_per_cta);
    if (per_sm < 1) return fail(NOC_ERR_NOMEM, "tensor-core rollout does not fit on an SM");
    A.ntiles = (int)((A.n + 127) / 128);
    const int grid = std::max(1, std::min(A.ntiles, per_sm * sm_count()));
    if (getenv("NOC_DEBUG"))
        fprintf(stderr, "[noc] tc rollout: mp=%d KS=%d smem=%zu tmem_cols=%d CTAs/SM=%d grid=%d tiles=%d\n", A.mp, SH::KS, smem,
                A.tmem_cols, per_sm, grid, A.ntiles);
    if (A.mode == NOC_MODE_MEAN) {
        NOC_CUDA(partials.alloc(sizeof(double) * 8 * (size_t)grid, st));
        A.partials = partials.as<double>();
    }
    // intermediates: stage the trajectories tile-major (coalesced) and transpose afterwards; if the staging buffer (as large
    // as the outputs) cannot be allocated the kernel writes the reference layout directly (strided, slower, same result)
    if (A.mode == NOC_MODE_INTERMEDIATES) {
        const size_t bytes = sizeof(float) * (size_t)A.ntiles * (A.nt + 1) * (SH::NZ + SH::NCTRL) * 128;
        big_reserve(bytes);                              // repeated intermediates calls reuse the staging buffer instead of paying the driver
        if (stage.alloc_big(bytes, st) != cudaSuccess) (void)cudaGetLastError();
    }
    A.stage = stage.as<float>();
    kern<<<grid, SH::NT, smem_req, st>>>(A);
    count_launch();
    NOC_CUDA(cudaGetLastError());
    if (stage.p) {
        tc_untile_kernel<<<dim3(A.ntiles, SH::NZ + SH::NCTRL), 128, 0, st>>>(A.stage, A.out_b, A.out_c, A.n, A.nt + 1, SH::NZ, SH::NCTRL);
        count_launch();
        NOC_CUDA(cudaGetLastError());
        NOC_CUDA(stage.free());
    }
    if (partials.p) {
        int frc = launch_finish(A.partials, grid, c.out_sums, st);
        if (frc) return frc;
        NOC_CUDA(partials.free());
    }
    NOC_CUDA(evals.free());
    return NOC_OK;
}

}  // namespace noc
