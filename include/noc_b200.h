/*
 * noc_b200.h — C ABI of the B200-native NeuralOC rollout library (libnoc_b200.so).
 *
 * The reference (donken/NeuralOC) is pure Python on PyTorch and has NO FFI; the drop-in boundary
 * for its hot path is the Python function
 *
 *     OCflow(x, Phi, prob, tspan, nt, stepper="rk4", alph=[1.0]*6, intermediates=False, noMean=False)
 *                                                                        -- src/OCflow.py:7
 *
 * plus the duck-typed Phi (src/Phi.py:56-138) and problem objects (src/problem/*.py) it receives.
 * Each entry point below names the reference interface it replaces.  A maintainer binds these
 * with ctypes (see INTEGRATION.md); neuraloc_b200/_cabi.py is exactly that binding.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types cross this boundary
 *   - every function returns NOC_OK (0) or a negative noc_status; the message of the last error
 *     of the calling thread is available from noc_last_error(); nothing ever calls exit()
 *   - "dev" pointers are CUDA device pointers on the current device, "host" pointers are host
 *     memory (pinned or pageable); `stream` is a cudaStream_t passed as void* (NULL = default stream)
 *   - dtype: NOC_F32 or NOC_F64 selects the arithmetic type of x, of all Phi / problem tensors and
 *     of the per-sample / trajectory outputs (the reference's --prec single|double)
 *   - all matrices are row-major and contiguous, in the reference's own checkpoint layout
 *     (src/Phi.py:77-87, 32-36): no re-layout is required of the caller
 *   - re-entrant and stream-ordered: work is enqueued on `stream`; only the *_host variants and
 *     noc_measure_* synchronise
 *   - scratch is allocated stream-ordered (cudaMallocAsync) from the device's default memory pool; on first use of a device
 *     the library raises that pool's release threshold to 1 GiB (env NOC_POOL_KEEP_MB overrides) so that freed scratch is
 *     reused instead of being returned to the driver at every synchronisation — a process-wide setting of that device's pool;
 *     the large per-call buffers (noc_ocflow_host's device copies of x and of the outputs, the intermediates staging buffers)
 *     come from a second, library-owned pool per device whose threshold follows the largest call (at most 1/8 of the device's
 *     memory, or NOC_POOL_KEEP_MB), so that repeated calls on multi-GB host batches do not pay the driver for them every time
 *   - there is no CPU implementation behind any of these: without a CUDA device they fail with
 *     NOC_ERR_CUDA
 */
#ifndef NOC_B200_H
#define NOC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NOC_ABI_VERSION 1

typedef enum noc_status {
    NOC_OK = 0,
    NOC_ERR_ARG = -1,          /* invalid argument (null pointer, negative size, bad enum) */
    NOC_ERR_UNSUPPORTED = -2,  /* valid in the reference but not instantiated here (message says what) */
    NOC_ERR_CUDA = -3,         /* a CUDA runtime call failed / no device */
    NOC_ERR_NOMEM = -4         /* shared-memory or device-memory budget exceeded */
} noc_status;

enum { NOC_F32 = 0, NOC_F64 = 1 };

/* problem classes: src/problem/Cross2D.py, SwarmTraj.py, Quadcopter.py */
enum { NOC_PROB_CROSS2D = 0, NOC_PROB_SWARMTRAJ = 1, NOC_PROB_QUADCOPTER = 2 };
/* prob.obstacle strings: None, 'softcorridor', 'hardcorridor' (Cross2D.py:43-52), 'blocks' (SwarmTraj.py:47-51) */
enum { NOC_OBS_NONE = 0, NOC_OBS_SOFTCORRIDOR = 1, NOC_OBS_HARDCORRIDOR = 2, NOC_OBS_BLOCKS = 3 };
/* stepper: 'rk4' (OCflow.py:157-184), 'rk1' (:143-155); any other string integrates nothing (:46-49) */
enum { NOC_STEP_NONE = 0, NOC_STEP_RK1 = 1, NOC_STEP_RK4 = 4 };
/* return modes of OCflow: default means (:80-95), noMean=True (:66-76), intermediates=True (:37-55,92-93) */
enum { NOC_MODE_MEAN = 0, NOC_MODE_NOMEAN = 1, NOC_MODE_INTERMEDIATES = 2 };

/* The value network Phi(s) = w'N(s) + 0.5 s'A'A s + c_w's + c_b, s = [x, t]   (src/Phi.py:56-96).
 * Replaces reading `Phi.A, Phi.c, Phi.w, Phi.N.layers[i]` of the live nn.Module. */
typedef struct noc_phi_t {
    int32_t d;        /* space dimension; the net input is D = d + 1                              */
    int32_t m;        /* hidden width                                                               */
    int32_t nTh;      /* number of ResNet layers, >= 2 (Phi.py:25-27)                               */
    int32_t r;        /* rows of A = min(10, d+1) (Phi.py:75)                                       */
    double h;         /* ResNet step N.h = 1/(nTh-1) (Phi.py:38); <= 0 means "use 1/(nTh-1)"        */
    const void* A;    /* dev [r, D]          state_dict key "A"                                     */
    const void* c_w;  /* dev [1, D]          "c.weight"                                             */
    const void* c_b;  /* dev [1]             "c.bias"                                               */
    const void* w;    /* dev [1, m]          "w.weight"                                             */
    const void* const* K;  /* HOST array of nTh dev pointers: K[0] [m, D] "N.layers.0.weight", K[i] [m, m] */
    const void* const* b;  /* HOST array of nTh dev pointers: b[i] [m]    "N.layers.i.bias"        */
} noc_phi_t;

/* The duck-typed problem object (attributes read by OCflow through calcLHQW / calcGradpH / calcCtrls /
 * xtarget: Cross2D.py:30-52, SwarmTraj.py:36-51, Quadcopter.py:37-48). */
typedef struct noc_prob_t {
    int32_t kind;       /* NOC_PROB_*                                                               */
    int32_t obstacle;   /* NOC_OBS_*                                                                */
    int32_t training;   /* prob.training: 0 after prob.eval(), 1 after prob.train()                 */
    int32_t nAgents;
    int32_t agentDim;   /* 2 (Cross2D), 3 (SwarmTraj), 12 (Quadcopter)                              */
    double alph_Q, alph_W, r;
    double mass, grav;  /* Quadcopter only (Quadcopter.py:37)                                       */
    const void* xtarget; /* dev [d], dtype-typed                                                    */
} noc_prob_t;

int noc_version(void);                 /* NOC_ABI_VERSION of the loaded library */
const char* noc_last_error(void);      /* thread-local, never NULL */

/* Device facts used by the host side (bench / tests): SM count, compute capability, shared memory per block. */
int noc_device_info(int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor, int64_t* smem_optin_bytes);

/* Number of control channels calcCtrls returns for this problem: d (Cross2D.py:164, SwarmTraj.py:166)
 * or 4 * nAgents (Quadcopter.py:165-174). Negative on error. */
int noc_ctrl_dim(const noc_prob_t* prob, int32_t d);

/* Fill `table` (HOST, nt * 5 doubles) with, per step k: t_a, t_a + h'/2, t_a + h', t_ctrl, h' where the values
 * replay the reference's double arithmetic `tk += h`, `h' = (tk + h) - tk` (OCflow.py:25,35,47,50,53,169). */
int noc_stage_times(double t0, double t1, int32_t nt, double* table);

/*
 * noc_ocflow — replaces OCflow(x, Phi, prob, tspan, nt, stepper, alph, intermediates, noMean), src/OCflow.py:7-95,
 * i.e. stepRK4/stepRK1 (:143-184), ocOdefun (:104-140), Phi.getGrad / Phi.forward (Phi.py:91-138) and
 * prob.calcLHQW / calcGradpH / calcCtrls, as ONE persistent kernel launch (+ a 1-block finishing reduction in mean mode, a
 * weight-packing kernel for the FMA kernels, a layout transpose of the trajectories for the tensor-core kernel's
 * intermediates mode).
 *
 *   x            dev [n, d]
 *   stage_times  HOST [nt * 5] from noc_stage_times(), or NULL to have it computed from (t0, t1, nt)
 *   alph         HOST [6]; only alph[0], [3], [4], [5] are used (quirk 7: Q/W weights live in prob)
 *   mode == NOC_MODE_MEAN:          out_costs dev [8] DOUBLE = sums over the n samples of
 *                                   [L, G, HJt, HJfin, HJgrad, Q, W] followed by the sample count n
 *                                   (divide by the count for the reference's means; sums so that shards add)
 *   mode == NOC_MODE_NOMEAN:        out_costs dev [n, 8] dtype-typed rows [Jc, L, G, HJt, HJfin, HJgrad, Q, W]
 *   mode == NOC_MODE_INTERMEDIATES: zFull dev [n, d+4, nt+1], ctrlFull dev [n, nCtrl, nt+1] (last dim contiguous),
 *                                   out_costs may be NULL
 */
int noc_ocflow(const noc_phi_t* phi, const noc_prob_t* prob, const void* x, int64_t n,
               const double* stage_times, double t0, double t1, int32_t nt, int32_t stepper,
               const double* alph, int32_t mode, int32_t dtype,
               void* out_costs, void* zFull, void* ctrlFull, void* stream);

/* Same call with HOST buffers for x and for every output (what evalOC.py / timeOC.py pass: CPU tensors).
 * Copies x host->device, runs noc_ocflow on `stream`, copies the results back and synchronises `stream`.
 * Mean / noMean batches of >= 256 Ki rows are processed as up to 8 row chunks (multiples of 128 rows: per-sample results are
 * unchanged; mean-mode chunk sums are added on the host in chunk order) so that a chunk's copy overlaps the previous chunk's
 * rollout; the chunks use two internal streams ordered after / before `stream` (created once per host thread and device, reused).
 * phi / prob tensors stay device pointers (uploaded once by the caller). */
int noc_ocflow_host(const noc_phi_t* phi, const noc_prob_t* prob, const void* x_host, int64_t n,
                    const double* stage_times, double t0, double t1, int32_t nt, int32_t stepper,
                    const double* alph, int32_t mode, int32_t dtype,
                    void* out_costs_host, void* zFull_host, void* ctrlFull_host, void* stream);

/* noc_phi_eval — replaces Phi.forward (Phi.py:91-96) and Phi.getGrad (Phi.py:99-138) on a batch.
 *   s dev [n, d+1]; out_phi dev [n] or NULL; out_grad dev [n, d+1] or NULL. */
int noc_phi_eval(const noc_phi_t* phi, const void* s, int64_t n, int32_t dtype,
                 void* out_phi, void* out_grad, void* stream);

/*
 * noc_phi_vjp — reverse-mode product of Phi.forward (Phi.py:91-96) and Phi.getGrad (Phi.py:99-138) on a batch: what
 * `torch.autograd.grad` of a loss built from net(s) and net.getGrad(s) needs.  For rows s_i = [x_i, t_i], a seed a on Phi and a
 * seed B on grad_s Phi, with  psi_i = a_i Phi(s_i) + B_i . grad_s Phi(s_i):
 *
 *   s            dev [n, d+1]
 *   seed_phi     dev [n] (a) or NULL (zero)
 *   seed_grad    dev [n, d+1] (B) or NULL (zero)
 *   grad_params  dev [P] or NULL: SUMS over the rows of d psi_i / d parameter, in noc_ocflow_grad's order and length
 *                (A, c.weight, c.bias, w.weight, N.layers.0.weight, N.layers.0.bias, N.layers.1.weight, N.layers.1.bias).
 *                Overwritten, not accumulated; floating-point atomics: reproducible to rounding, not bitwise.
 *   grad_s       dev [n, d+1] or NULL: d psi_i / d s_i = a_i grad Phi(s_i) + Hess Phi(s_i) B_i (last column: d / dt)
 *
 * One launch of the training kernel's second-order sweep per call (+ weight packing and the gradient compaction).  nTh == 2
 * only (NOC_ERR_UNSUPPORTED otherwise), even widths m, fp32 and fp64.
 */
int noc_phi_vjp(const noc_phi_t* phi, const void* s, int64_t n, const void* seed_phi,
                const void* seed_grad, int32_t dtype, void* grad_params, void* grad_s, void* stream);

/* noc_prob_eval — replaces prob.calcLHQW(x,p), prob.calcGradpH(x,p), prob.calcCtrls(x,p) on a batch.
 *   x, p dev [n, d]; out_lhqw dev [n, 4] = (L, H, Q, W); out_gradpH dev [n, d]; out_ctrls dev [n, nCtrl];
 *   any output may be NULL. */
int noc_prob_eval(const noc_prob_t* prob, const void* x, const void* p, int64_t n, int32_t d, int32_t dtype,
                  void* out_lhqw, void* out_gradpH, void* out_ctrls, void* stream);

/* Roofline denominators measured on the device the library runs on (SURVEY.md H10): a register-resident
 * FMA micro-benchmark on all SMs. Returns TFLOP/s (2 flops per FMA) in *tflops. Synchronises. */
int noc_measure_fma_peak(int32_t dtype, double* tflops);

/* Self-test of the Blackwell tensor-core building blocks (tcgen05.mma with TMEM accumulators, no-swizzle shared-memory
 * descriptors in both majors, tcgen05.ld/st, tcgen05.commit -> mbarrier): one CTA computes D[128,N] = A[128,K] * B in bf16
 * with fp32 accumulation.  B is [N,K] (b_mn_major = 0) or [K,N] read MN-major (b_mn_major = 1).  All pointers dev.
 * Diagnostics for the building blocks of the tensor-core rollout kernel; not used by noc_ocflow. */
int noc_tc_probe(const void* A_bf16, const void* B_bf16, void* D_f32, int32_t N, int32_t K, int32_t b_mn_major,
                 int32_t roundtrip_tmem, void* stream);

/* noc_sample_rho0 — replaces the host-side draw of the initial states, `xInit + cvt(var0 * torch.randn(n, d))`
 * (src/initProb.py:27-28,107-120,196-203 and resample, :252-262; the quadcopter perturbs its first 3 columns only, :132-140):
 *   x[i, c] = center[c] + (c < noise_cols ? var0 * N(0,1) : 0)   for the rows row0 .. row0 + n - 1 of the (virtual) full batch.
 * Counter-based Philox4x32-10 + Box-Muller: row i, column c uses word (i d + c) % 4 of counter block (i d + c) / 4 under
 * key = seed, so a shard (row0, n) reproduces exactly its rows of the full batch and the result does not depend on the
 * launch geometry.  The stream differs from torch's generators: parity with the reference is distributional (tests).
 *   center dev [d] dtype-typed; x dev [n, d]; noise_cols < 0 or > d means d. */
int noc_sample_rho0(const void* center, int32_t d, int32_t noise_cols, double var0, uint64_t seed, int64_t row0, int64_t n,
                    int32_t dtype, void* x, void* stream);

/* The raw generator behind noc_sample_rho0 (known-answer tests): out_u32 dev [4 * ngroups] = Philox4x32-10 of the
 * counter blocks group0 .. group0 + ngroups - 1 (counter = (lo32, hi32, 0, 0), key = (lo32(seed), hi32(seed))). */
int noc_philox_raw(uint64_t seed, int64_t group0, int64_t ngroups, void* out_u32, void* stream);

/*
 * noc_ocflow_grad — replaces one training evaluation, `Jc, cs = OCflow(x0, net, prob, tspan, nt, "rk4", alph); Jc.backward()`
 * (trainOC.py:172-173): the rollout of noc_ocflow in mean mode AND the exact reverse-mode gradient of the sum over the samples
 * of the per-sample objective  L + alph[0] G + alph[3] HJt + alph[4] HJfin + alph[5] HJgrad  (OCflow.py:75) with respect to every
 * Phi parameter and, optionally, the initial states — the discrete adjoint of stepRK4 (OCflow.py:157-184) with the second-order
 * terms of Phi.getGrad (Phi.py:99-138) and the derivatives of calcLHQW / calcGradpH (train- or eval-mode, as prob->training
 * says).  One kernel launch (forward sweep, terminal block, backward sweep) + a weight-packing kernel + the cost reduction.
 * nTh == 2 and stepper 'rk4' only; Quadcopter with one agent only (NOC_ERR_UNSUPPORTED otherwise).
 *
 *   out_costs  dev [8] DOUBLE: sums of [L, G, HJt, HJfin, HJgrad, Q, W] and the sample count, as noc_ocflow's mean mode
 *   grad       dev [P] dtype-typed, P = r D + D + 1 + m + m D + m + m m + m: SUMS over the samples of d objective / d parameter,
 *              concatenated in the reference's state_dict order (Phi.py:77-87): A, c.weight, c.bias, w.weight,
 *              N.layers.0.weight, N.layers.0.bias, N.layers.1.weight, N.layers.1.bias.  Divide by the sample count for the
 *              gradient of the reference's mean objective (sums so that shards add).  Overwritten, not accumulated.
 *              Accumulated with floating-point atomics: reproducible to rounding, not bitwise.
 *   grad_x     dev [n, d] or NULL: d (sample's objective) / d x
 */
int noc_ocflow_grad(const noc_phi_t* phi, const noc_prob_t* prob, const void* x, int64_t n,
                    const double* stage_times, double t0, double t1, int32_t nt, const double* alph, int32_t dtype,
                    void* out_costs, void* grad, void* grad_x, void* stream);

/*
 * noc_baseline_loss — replaces the baseline's discrete-control objective for a batch of initial states:
 * loss_fun(U, Z_0, prob, nt, alphG) (baseline2D.py:42-63, timeBaseline.py:50-70; Cross2D / SwarmTraj problems:
 * Z += h U_i, loss += h L(Z, U_i) with L from calcLHQW, + alphG G(Z_nt)) and compute_loss(ctrls, x0, prob, alphG) with dyn
 * (baselineQuad.py:40-72; one quadcopter: x += h dyn(c_i, x), J += h (2 + |c_i|^2), + alphG 0.5 |x - xtarget|^2), h = 1/nt,
 * and — when gradU is not NULL — `err.backward()` of the optimisation loops (baseline2D.py:97-102, baselineQuad.py:80-86).
 * The reference evaluates one initial state per Python call; here every sample of the batch is one warp of one launch.
 *   U      dev [n, nt, nc]   controls, nc = d (Cross2D, SwarmTraj) or 4 (Quadcopter: thrust, three torques)
 *   z0     dev [n, d]        initial states
 *   loss   dev [n]           per-sample objective
 *   gradU  dev [n, nt, nc] or NULL: d loss[i] / d U[i]
 */
int noc_baseline_loss(const noc_prob_t* prob, const void* U, const void* z0, int64_t n, int32_t d, int32_t nt, double alphG,
                      int32_t dtype, void* loss, void* gradU, void* stream);

/* Which kernel family the calling thread's last noc_ocflow / noc_ocflow_host call ran (-1 before the first call):
 * the FMA sample-tile kernel, the one-CTA-per-sample small-batch kernel, or the tensor-core kernel.  The choice is made
 * from the shapes and the batch size; env NOC_TC=0 disables the tensor-core kernel, NOC_FORCE_PATH=tile|vec|tc pins one. */
enum { NOC_PATH_TILE = 0, NOC_PATH_SAMPLE = 1, NOC_PATH_TENSOR = 2 };
int noc_last_path(void);

/* Kernel-launch counter (number of CUDA kernels this library launched in this process); bench.py reports it. */
int64_t noc_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* NOC_B200_H */
