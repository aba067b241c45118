/*
 * qlnlp.h -- C ABI of the B200 batched evaluator for the planar-quadruped landing NLP.
 *
 * This is the drop-in boundary: a host program (the reference's Julia `HybridNLP`, a Python
 * harness, Ipopt's C interface, ...) binds exactly these symbols.  Each entry point names the
 * reference interface it replaces (paths relative to the reference checkout's src/).
 * INTEGRATION.md shows the `ccall` methods a maintainer adds next to src/moi.jl.
 *
 * Conventions
 *   - plain C types only; all arrays are fp64 / int64, caller-owned, never retained;
 *   - every function returns 0 on success, a QLNLP_E* code otherwise, and never throws or exits;
 *     qlnlp_last_error() returns a message for the calling thread's last failure;
 *   - indices handed to the caller are 1-BASED (Julia / MOI convention, moi.jl:31-33);
 *   - one handle may be driven by one host thread at a time (Ipopt calls back from one thread);
 *     different handles are independent;
 *   - every call leaves the calling thread's current CUDA device as it found it;
 *   - streams and CUDA graphs (the *_device entry points): a handle may launch on any number of streams, and
 *     launches on different streams may run at once.  Launches may be captured into CUDA graphs, and a graph may be
 *     replayed on any stream, concurrently with anything else the handle does, including replays of other graphs
 *     captured on the same stream and eager launches on the capture stream: each graph owns the work counter and
 *     the scratch its launches use.  Up to 1,024 graphs per handle may hold launches at once (a capture beyond that
 *     is refused with QLNLP_EINVAL); a graph gives its counter back when it and its executable instantiations are
 *     destroyed, and must not outlive its handle.  Replay one executable instantiation of a graph at a time.
 *     First-use set-up allocates and synchronises, which a capture cannot hold: the first call of a handle, its first
 *     kinematic evaluation, its first KKT call of any of the three kinds (one-shot solve, factor, factored solve) and
 *     the first ragged launch over a set of classes are refused with
 *     QLNLP_EINVAL inside a capture (the caller's capture stays valid).  Warm the handle outside the capture by
 *     making each kind of call it will capture once, on any stream;
 *   - there is NO CPU fallback: evaluation entry points fail with QLNLP_ENODEVICE when no
 *     sm_100 device / driver is present.  Structure, dimension and bound queries are pure host
 *     integer logic and work anywhere.
 *
 * Layouts (SURVEY.md section 8a)
 *   Z     n_nlp = 20N-5        knot k (1-based): x_k at 20(k-1)+1..+15, u_k at 20(k-1)+16..+20   nlp.jl:38-39
 *   g     m_nlp = 18N-k_trans+16   blocks init|term|dyn|contact-first|contact-other|final-ctrl|body-pos   nlp.jl:48-63
 *   grad  n_nlp
 *   jac   QLNLP_JAC_SPARSE_BLOCK: nnz = 529N-k_trans-87 values = the entries constraints.jl:212-291
 *         assigns, in the reference's column-major order (row fastest);
 *         QLNLP_JAC_DENSE: the full m_nlp x n_nlp column-major grid the reference reports
 *         (moi.jl:31-33), unassigned entries written as 0 -- single evaluations only.
 */
#ifndef QLNLP_H
#define QLNLP_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QLNLP_VERSION 2

enum {
    QLNLP_OK = 0,
    QLNLP_EINVAL = 1,     /* bad argument (NULL, out-of-range N/k_trans/init_mode, misaligned ld) */
    QLNLP_ENODEVICE = 2,  /* no usable CUDA device / driver: the product has no CPU path */
    QLNLP_ECUDA = 3,      /* a CUDA runtime call failed; see qlnlp_last_error() */
    QLNLP_ENOMEM = 4
};

enum {
    QLNLP_JAC_SPARSE_BLOCK = 0,   /* the entries jac_c! assigns (zeros of the identity / RK4 blocks included) */
    QLNLP_JAC_DENSE = 1,          /* the reference's full m_nlp x n_nlp grid; single evaluations only */
    QLNLP_JAC_SPARSE_TRUE = 2     /* only structurally non-zero entries: identity blocks as diagonals, RK4 blocks
                                     as their mode pattern (71/71/57 entries, 56 at the jump knot); 4,840 values
                                     instead of 32,161 at the default instance, same column-major order */
};

/* OR this into `jac_mode` at qlnlp_create to switch on the kinematic (leg-length) rows the reference carries
 * COMMENTED OUT (nlp.jl:60,70; constraints.jl:115-138,276-288): cinds[8] = 2 rows per knot, norm(pb - p1) and
 * norm(pb - p2) with bounds [0, l1 + l2 + lb/2].  m_nlp grows by 2N, every Jacobian pattern by 8N entries (merged
 * into the column-major order).  Default off = the reference as it runs.  Not available for ragged launches,
 * registered output rows and the Hessian; this path is not tuned (the Jacobian values take a second pass). */
#define QLNLP_WITH_KINEMATICS 0x100

/* planar_quadruped.jl:11-20 */
typedef struct {
    double g, mb, mf, lb, l1, l2;
} qlnlp_model;

/* The fields of HybridNLP (nlp.jl:13-33) the evaluators read, plus the per-knot QuadraticCost
 * tables (quadratic_cost.jl:16-22; Q and R as diagonals), knot-major, N rows each; row N-1 is the
 * terminal cost (costs.jl:15,33). */
typedef struct {
    int64_t N;          /* knot points                                  nlp.jl:16 */
    int64_t k_trans;    /* first knot of mode 3, 1 <= k_trans <= N      nlp.jl:19 */
    int64_t init_mode;  /* 1 or 2                                       nlp.jl:18 */
    qlnlp_model model;
    double x0[15];      /* nlp.jl:20 */
    double xf[15];      /* nlp.jl:21 */
    const double* Q;    /* [N][15] */
    const double* R;    /* [N][5]  */
    const double* q;    /* [N][15] */
    const double* r;    /* [N][5]  */
    const double* c;    /* [N]     */
} qlnlp_problem_desc;

typedef struct qlnlp_handle_s* qlnlp_handle;

/* HybridNLP(model, obj, init_mode, k_trans, N, x0, xf)            nlp.jl:33-83
 * `device` is the CUDA ordinal used by every later call on the handle (bound lazily, at the first
 * evaluation).  `jac_mode` selects what qlnlp_eval_constraint_jacobian / jacobian_structure report.
 * Values: divisions by the model constants go through a reciprocal (csrc/fastdiv.h), exact while every numerator
 * has |a| >= 2^-969 and a/mf, a/Ib ... stay clear of overflow (all of the landing problem's range).  Inputs that
 * drive values to the ends of the double range may see one ulp, +0 for -0, or NaN where IEEE division gives +-Inf;
 * with the environment variable QLNLP_IEEE_DIV=1 set when the handle is created, the kernels divide IEEE-exactly. */
int qlnlp_create(const qlnlp_problem_desc* desc, int device, int jac_mode, qlnlp_handle* out);
int qlnlp_destroy(qlnlp_handle h);

/* The same evaluator spread over several GPUs of one process (SURVEY.md 8e: the problems are independent, so a batch
 * is split into contiguous shards, qlnlp_shard_bounds, one per device, with no exchange between the devices).
 * `devices` lists ndev distinct CUDA ordinals.  On such a handle
 *   - qlnlp_eval_batch_host shards the caller's batch itself: one driver thread + one pipeline per device, and the
 *     host cores are split between the devices;
 *   - qlnlp_eval_batch_device_multi launches one shard per device on device-resident arrays;
 *   - the single-evaluation callbacks and the integer queries use the first device;
 *   - qlnlp_eval_batch_device / qlnlp_eval_ragged_device are refused (they take one device's pointers). */
int qlnlp_create_multi(const qlnlp_problem_desc* desc, const int* devices, int ndev, int jac_mode, qlnlp_handle* out);
/* devices of the handle (1 for qlnlp_create); fills at most cap ordinals */
int qlnlp_devices(qlnlp_handle h, int* devices, int cap, int* ndev);
/* shard `shard` of `nshards` covers evaluations [lo, hi): contiguous and balanced, the first B % nshards shards hold
 * one extra evaluation */
int qlnlp_shard_bounds(int64_t B, int nshards, int shard, int64_t* lo, int64_t* hi);
/* tuning knobs: "host_chunk" (evaluations per pipeline stage of the host-pointer path, default 512), "host_threads"
 * (row-builder threads per device, 0 = this handle's share of the CPUs the process may use), "pin_threads" (0/1),
 * "x_cache" (0/1: serve repeated single-evaluation callbacks at the same x from the last evaluation), "compressible"
 * (0/1, default 1: qlnlp_device_alloc asks for compressible memory where the device offers it; 0 gives cudaMalloc
 * memory, for outputs that must be exported with cudaIpcGetMemHandle or shared through torch.multiprocessing, which
 * cuMemCreate memory does not support; the Python layer's outputs follow it too) */
int qlnlp_set_option(qlnlp_handle h, const char* name, int64_t value);

/* num_primals / num_duals                                          nlp.jl:86-87
 * nnz = length of the structure for the handle's jac_mode; nnz_block = SPARSE_BLOCK count. */
int qlnlp_dims(qlnlp_handle h, int64_t* n_nlp, int64_t* m_nlp, int64_t* nnz, int64_t* nnz_block);

/* MOI.jacobian_structure(nlp)                                      moi.jl:31-33
 * Fills rows[nnz], cols[nnz], 1-based, in value order.  Host-only integer logic. */
int qlnlp_jacobian_structure(qlnlp_handle h, int64_t* rows, int64_t* cols);

/* constraint bounds nlp.lb / nlp.ub                                nlp.jl:66-69 */
int qlnlp_constraint_bounds(qlnlp_handle h, double* lb, double* ub);
/* the variable bounds solve() installs                             moi.jl:51-67 */
int qlnlp_variable_bounds(qlnlp_handle h, double* xl, double* xu);

/* ---- single evaluations on HOST pointers: the four MOI callbacks -------------------------
 * Ipopt asks for f, grad f, g and the Jacobian values of an iterate in separate callbacks.  The first callback at a
 * new x evaluates all four with ONE launch (one H2D copy, one kernel, one D2H copy) and keeps the results; callbacks
 * that follow with the same x (compared bit for bit; 9.7 KB at the default instance) are served from that cache, so
 * a caller need not track Ipopt's new_x flag.  The evaluator keeps no other state between calls. */
/* MOI.eval_objective(prob, x)               -> eval_f              moi.jl:1-3   costs.jl:6-16 */
int qlnlp_eval_objective(qlnlp_handle h, const double* x, double* f);
/* MOI.eval_objective_gradient(prob, grad, x) -> grad_f!            moi.jl:5-8   costs.jl:23-34 */
int qlnlp_eval_objective_gradient(qlnlp_handle h, const double* x, double* grad);
/* MOI.eval_constraint(prob, g, x)           -> eval_c!             moi.jl:10-13 constraints.jl:145-158 */
int qlnlp_eval_constraint(qlnlp_handle h, const double* x, double* g);
/* MOI.eval_constraint_jacobian(prob, vals, x) -> jac_c!            moi.jl:15-24 constraints.jl:212-291
 * vals has qlnlp_dims().nnz entries in jacobian_structure order. */
int qlnlp_eval_constraint_jacobian(qlnlp_handle h, const double* x, double* vals);
/* all four at once (any output may be NULL): what the callbacks above do at a new x            moi.jl:1-24 */
int qlnlp_eval_all(qlnlp_handle h, const double* x, double* f, double* grad, double* g, double* vals);

/* ---- Lagrangian Hessian: what MOI.eval_hessian_lagrangian / hessian_lagrangian_structure need to offer [:Hess] ----
 * NOT in the reference: src/moi.jl:26-28 advertises [:Grad, :Jac] and Ipopt runs L-BFGS (src/main.ipynb:219).
 *   H = sigma * Hess f(x) + sum_r lambda_r * Hess g_r(x)
 * with f as eval_f computes it (costs.jl:6-16; its true second derivatives, d/dh of h*stagecost included) and g as
 * eval_c! (constraints.jl:145-158; lambda in that order).  H is block diagonal, one 20x20 block per knot; the
 * structure is the lower triangle restricted to the structural non-zeros of each knot's mode, 1-based (row, col),
 * column-major (3,355 entries at the default instance). */
int qlnlp_hessian_nnz(qlnlp_handle h, int64_t* nnz);
int qlnlp_hessian_structure(qlnlp_handle h, int64_t* rows, int64_t* cols);
/* one evaluation on HOST pointers: x[n_nlp], lambda[m_nlp] -> vals[nnz_hess] */
int qlnlp_eval_hessian_lagrangian(qlnlp_handle h, const double* x, double sigma, const double* lambda, double* vals);
/* B evaluations on DEVICE pointers: Z[B][ldz], sigma[B] (NULL: 1.0), lambda[B][ldlambda], H[B][ldh]; enqueued on
 * `stream`, not synchronised.  H 16-byte aligned with even ldh takes the TMA store path. */
int qlnlp_eval_hessian_batch_device(qlnlp_handle h, int64_t B, const double* Z, int64_t ldz, const double* sigma,
                                    const double* lambda, int64_t ldlambda, double* H, int64_t ldh, void* stream);

/* Initial guesses of a sweep on the device (notebook cell 7, src/main.ipynb:181-196; SURVEY.md 8f N2):
 * Z[b] = `base` (the class guess: packZ(nlp, Xguess, Uref) for the handle's own x0, n_nlp doubles) with the first 14
 * states of knots 1..k_trans replaced by  x0[b] + (xterm - x0[b]) / (k_trans - 1) * (k - 1).  Device pointers. */
int qlnlp_initial_guess_batch_device(qlnlp_handle h, int64_t B, const double* base, const double* x0, double* Z,
                                     int64_t ldz, void* stream);

/* ---- batched evaluation (B independent decision vectors; no reference equivalent) -------- */
typedef struct {
    const double* Z;   int64_t ldz;     /* [B][ldz],    ldz    >= n_nlp          (required).  With Z 16-byte aligned
                                           and ldz even (> n_nlp, which is odd) a row is fetched with one TMA load that
                                           also READS the padding element Z[b][n_nlp]. */
    const double* x0;                   /* [B][15] per-evaluation initial state, or NULL -> desc.x0 */
    const double* xf;                   /* [B][15] per-evaluation final state,   or NULL -> desc.xf */
    double* f;                          /* [B]                                    or NULL: skip */
    double* grad;      int64_t ldgrad;  /* [B][ldgrad], ldgrad >= n_nlp           or NULL: skip */
    double* g;         int64_t ldg;     /* [B][ldg],    ldg    >= m_nlp           or NULL: skip */
    double* jac;       int64_t ldjac;   /* [B][ldjac],  ldjac  >= nnz             or NULL: skip
                                           values in the handle's sparse pattern (SPARSE_TRUE handles:
                                           nnz_true; SPARSE_BLOCK and DENSE handles: nnz_block).
                                           The TMA bulk-store path needs jac
                                           16-byte aligned and ldjac even; otherwise a slower
                                           plain-store path is used. */
} qlnlp_batch_io;

/* All pointers are DEVICE pointers on the handle's device; the launch is enqueued on `stream`
 * (a cudaStream_t passed as void*, NULL = default stream) and the call returns without
 * synchronising.  One fused kernel evaluates everything requested. */
int qlnlp_eval_batch_device(qlnlp_handle h, int64_t B, const qlnlp_batch_io* io, void* stream);

/* ---- matrix-free products: what MOI.eval_constraint_jacobian_product, eval_constraint_jacobian_transpose_product and
 * eval_hessian_lagrangian_product need to offer [:JacVec] / [:HessVec].  NOT in the reference (moi.jl:26-28).
 *   J     the Jacobian the handle reports, quirks included (Q2: the zeroed time row at the jump knot, Q4: the body
 *         row's d/dtheta branches on theta > 0), with the 2N kinematic rows on a QLNLP_WITH_KINEMATICS handle; w and
 *         J'y have n_nlp entries, y and Jw m_nlp (kinematic rows included).  The same for every jac_mode.
 *   H     the matrix qlnlp_eval_hessian_* returns (its lower triangle, mirrored), same sigma / lambda conventions;
 *         handles with kinematic rows are refused, as by the Hessian.
 * Summation order (the bits are defined): every output entry is the left fold, starting from the first term, of
 * RN(entry * vector) terms added with RN(a + b), no fused multiply-add, over the structurally non-zero entries (the
 * SPARSE_TRUE pattern; for H the entries of qlnlp_hessian_structure and their mirror images):
 *   (J w)_r   row r's entries in ascending column order (a defect row: the RK4 block's 20 columns, then -w_(k+1));
 *   (J'y)_c   column c's entries in ascending row order (the order of the column inside the SPARSE_BLOCK values);
 *   (H v)_i   row i of the knot's symmetric block in ascending column order.
 * The result does not depend on B, the batch position, leading dimensions, alignment or the entry point used. */
typedef struct {
    const double* w;  int64_t ldw;     /* [B][ldw >= n_nlp]   or NULL: no J w */
    double* jw;       int64_t ldjw;    /* [B][ldjw >= m_nlp]  required iff w */
    const double* y;  int64_t ldy;     /* [B][ldy >= m_nlp]   or NULL: no J'y */
    double* jty;      int64_t ldjty;   /* [B][ldjty >= n_nlp] required iff y */
} qlnlp_product_io;
/* DEVICE pointers, enqueued on `stream`, not synchronised.  io->jac must be NULL; io->Z, x0, xf, f, grad, g as in
 * qlnlp_eval_batch_device: one fused launch evaluates everything requested.  Single-device handles only. */
int qlnlp_eval_jacobian_products_batch_device(qlnlp_handle h, int64_t B, const qlnlp_batch_io* io,
                                              const qlnlp_product_io* pv, void* stream);
/* DEVICE pointers: Z[B][ldz], sigma[B] (NULL: 1.0), lambda[B][ldlambda], V[B][ldv], HV[B][ldhv >= n_nlp] */
int qlnlp_eval_hessian_product_batch_device(qlnlp_handle h, int64_t B, const double* Z, int64_t ldz, const double* sigma,
                                            const double* lambda, int64_t ldlambda, const double* V, int64_t ldv,
                                            double* HV, int64_t ldhv, void* stream);
/* the MOI callbacks: HOST pointers, synchronous, one evaluation on the handle's first device */
int qlnlp_eval_constraint_jacobian_product(qlnlp_handle h, const double* x, const double* w, double* jw);
int qlnlp_eval_constraint_jacobian_transpose_product(qlnlp_handle h, const double* x, const double* y, double* jty);
int qlnlp_eval_hessian_lagrangian_product(qlnlp_handle h, const double* x, const double* v, double sigma,
                                          const double* lambda, double* hv);

/* ---- batched Newton step: the regularised KKT system of each problem (no reference counterpart; the reference hands
 * it to Ipopt's sparse factorisation).  For every problem b of a SPARSE_TRUE handle, solve
 *     [ W + diag(sx)   J'       ] [ px ]   [ r1 ]
 *     [ J             -diag(dc) ] [ pl ] = [ r2 ]
 *   W    hess[b]: the values qlnlp_eval_hessian_batch_device writes (lower triangle in qlnlp_hessian_structure
 *        order), used mirrored;
 *   J    jac[b]: SPARSE_TRUE values in qlnlp_jacobian_structure order, as qlnlp_eval_batch_device writes them on a
 *        SPARSE_TRUE handle, used as given (quirks Q2 and Q4 included);
 *   sx   [n_nlp] >= 0, the primal diagonal (barrier term + delta_w), or NULL: 0;
 *   dc   [m_nlp] > 0 on EVERY row, the constraint diagonal (delta_c + slack terms; equality rows carry a
 *        regularisation: the quasi-definite form).
 * Method: M = W + diag(sx) + J' diag(dc)^-1 J is block tridiagonal with 20x20 blocks (15x15 at knot N); its Cholesky
 * factor is formed knot by knot, then M px = r1 + J' (r2 ./ dc) and pl = (J px - r2) ./ dc.
 * status[b]:  0  success;
 *             k  (1-based knot) the diagonal block of knot k in the factorisation had a pivot <= 0 or not finite.
 *                With dc > 0, M is positive definite exactly when the KKT matrix has inertia (n_nlp, m_nlp, 0)
 *                (Haynsworth), so k > 0 is the "wrong inertia" signal: raise delta_w and solve again;
 *            -1  a dc entry is <= 0 or not finite.
 *   px[b] and pl[b] of a problem with status != 0 are written as NaN.
 * One fixed operation order per problem: the bits do not depend on B, the batch position, leading dimensions,
 * alignment or the stream.  DEVICE pointers, 8-byte aligned (status 4-byte); enqueued on `stream`, not
 * synchronised.  Refused (QLNLP_EINVAL): SPARSE_BLOCK / DENSE handles, QLNLP_WITH_KINEMATICS handles, multi-device
 * handles.  The factor scratch (1,840 B per knot per resident warp) is allocated at the first call on a stream; a
 * captured solve allocates its own inside the graph. */
typedef struct {
    const double* hess; int64_t ldhess;   /* [B][ldhess >= nnz_hess] */
    const double* jac;  int64_t ldjac;    /* [B][ldjac  >= nnz (SPARSE_TRUE)] */
    const double* sx;   int64_t ldsx;     /* [B][ldsx   >= n_nlp]   or NULL */
    const double* dc;   int64_t lddc;     /* [B][lddc   >= m_nlp] */
    const double* r1;   int64_t ldr1;     /* [B][ldr1   >= n_nlp] */
    const double* r2;   int64_t ldr2;     /* [B][ldr2   >= m_nlp] */
    double* px;         int64_t ldpx;     /* [B][ldpx   >= n_nlp] */
    double* pl;         int64_t ldpl;     /* [B][ldpl   >= m_nlp] */
    int32_t* status;                      /* [B] */
} qlnlp_kkt_io;
int qlnlp_kkt_solve_batch_device(qlnlp_handle h, int64_t B, const qlnlp_kkt_io* io, void* stream);

/* The same solve split in two: factorise once, then solve any number of right-hand sides against the kept factor
 * (iterative refinement, predictor and corrector, second-order corrections).  A factor followed by a factored solve
 * gives the bits qlnlp_kkt_solve_batch_device gives for the same inputs.
 *
 * A factor row holds, in a layout that belongs to the library, L_kk of every knot (210 doubles, packed), the 15x20
 * off-diagonal factor X_k of every knot but the last (300), the problem's SPARSE_TRUE J values and dc, its status and
 * a stamp of its class (N, k_trans, init_mode):
 *     size = 4 + 210 N + 300 (N - 1) + nnz (SPARSE_TRUE) + m_nlp   doubles
 * 36,747 doubles (293,976 B) per problem at the default instance (N = 61, k_trans = 21), 19.3 GB at B = 65,536.
 * qlnlp_kkt_factor_size reports it.  A factor is self-contained: overwriting hess, jac, sx or dc after factorising
 * changes no later solve.  A row with status 0 is written in full; entries beyond `size` are never written.  The handles qlnlp_kkt_solve_batch_device
 * refuses are refused by the three calls below too.  Neither kernel needs scratch: the factor lives in caller memory. */
int qlnlp_kkt_factor_size(qlnlp_handle h, int64_t* doubles);
typedef struct {
    const double* hess; int64_t ldhess;   /* [B][ldhess >= nnz_hess] */
    const double* jac;  int64_t ldjac;    /* [B][ldjac  >= nnz (SPARSE_TRUE)] */
    const double* sx;   int64_t ldsx;     /* [B][ldsx   >= n_nlp]   or NULL */
    const double* dc;   int64_t lddc;     /* [B][lddc   >= m_nlp] */
    double* factor;     int64_t ldfactor; /* [B][ldfactor >= qlnlp_kkt_factor_size] */
    int32_t* status;                      /* [B] as qlnlp_kkt_solve_batch_device: 0, the failing knot k, or -1 */
} qlnlp_kkt_factor_io;
/* Factorises B problems (inputs as qlnlp_kkt_solve_batch_device).  DEVICE pointers, enqueued on `stream`. */
int qlnlp_kkt_factor_batch_device(qlnlp_handle h, int64_t B, const qlnlp_kkt_factor_io* io, void* stream);
typedef struct {
    const double* factor; int64_t ldfactor; int64_t nfactor;   /* [nfactor][ldfactor]: rows of factors */
    const int64_t* index;                 /* [R] factor row of each right-hand side, or NULL: row i uses factor i */
    const double* r1;   int64_t ldr1;     /* [R][ldr1 >= n_nlp] */
    const double* r2;   int64_t ldr2;     /* [R][ldr2 >= m_nlp] */
    double* px;         int64_t ldpx;     /* [R][ldpx >= n_nlp] */
    double* pl;         int64_t ldpl;     /* [R][ldpl >= m_nlp] */
    int32_t* status;                      /* [R] */
} qlnlp_kkt_rhs_io;
/* Solves R right-hand sides; row i against the factor of row index[i] (or i), so several right-hand sides may share
 * one factor and a subset of the problems may be solved alone.  status[i]:
 *      0  success;
 *      k > 0 or -1  the factor's own status, copied;
 *     -2  index[i] (or i) outside [0, nfactor);
 *     -3  the factor's class stamp is not this handle's class.
 * px[i] and pl[i] of a row with status != 0 are written as NaN.  DEVICE pointers, enqueued on `stream`. */
int qlnlp_kkt_solve_factored_batch_device(qlnlp_handle h, int64_t R, const qlnlp_kkt_rhs_io* io, void* stream);

/* Accuracy.  The step comes from the condensed form M, which loses what W + diag(sx) holds below eps ||J' D^-1 J||: px
 * loses digits when dc is small relative to ||J||^2 / ||W + diag(sx)||, and pl with it.  Measured on a B200 against an
 * extended-precision solve of K (tests/test_gpu_kkt_accuracy.py, DESIGN.md section 5), errors relative to the largest
 * entry of each block, N = 2 .. 1024:
 *   normwise backward error ||r - K z||_inf / (||K||_inf ||z||_inf + ||r||_inf), z = [px; pl]: <= 1e-13 with dc_eq >=
 *     1e-6 and inequality dc in [1e-2, 1]; up to 5e-12 at smaller dc_eq, and up to 7e-11 when the inequality dc span
 *     1e-10 .. 1e2 (an active set).  The one-shot and factored solves are not backward stable at such scalings.
 *   px: 1e-14 at dc >= 1e-2 (sx in [1, 10]); 3e-10 at dc_eq = 1e-6; 2e-6 at dc_eq = 1e-8 with sx over 1e-8 .. 1e8;
 *     4e-4 at dc_eq = 1e-12, and no digit at all with an active set and wide sx.
 * Iterative refinement with the residual below and the kept factor (HybridNLP.kkt_solve_refined_batch, 3 steps) brings
 * px and pl to 1e-14 and the componentwise backward error to 3.2e-16 wherever dc_eq >= 1e-8 (2 steps: up to 4.9e-14).
 * At dc_eq <= 1e-10 each step gains only 1 .. 3 digits although Skeel's condition of K times eps is 1e-15 there: the
 * condensed factor, not K, limits it.  Where the factor is too far from K (dc_eq = 1e-12 with an active set and wide sx)
 * refinement diverges; the refined solve keeps a step only when it halves the componentwise backward error, so it
 * returns the unrefined step there, which has no correct digit.
 *
 * Residual of the system: s1 = r1 - (W + diag(sx)) px - J' pl,  s2 = r2 - J px + dc .* pl, for B problems, with W, J,
 * sx, dc as the solve takes them.  Each entry is the left fold, starting from r, of fused multiply-adds
 * acc = RN(acc - a * v), one per term, in this order:
 *   s1_i  the row of i's knot block of W (mirrored) in ascending column order, its diagonal entry rounded once as
 *         RN(W_ii + sx_i); then J' pl over the rows that touch i's knot in the order of kkt_slot_row (qlnlp_kkt.cuh);
 *   s2_r  row r's entries in ascending column order (a defect row: the RK4 block's 20 columns, then -x_(k+1)), then
 *         + dc_r pl_r.
 * The knot-local blocks may hold structural zeros; they add exact zeros for finite px and pl.  The result is within
 * gamma_t (|r| + |K| |z|) of the exact residual, t = 1 + the structural terms of the entry (at most 56 in s1, 23 in
 * s2), and its bits do not depend on B, the batch position, leading dimensions or alignment.  NaN in px or pl (a failed
 * solve's rows) gives NaN residual rows.  DEVICE pointers, 8-byte aligned, enqueued on `stream`; the handles the KKT
 * solve refuses are refused. */
typedef struct {
    const double* hess; int64_t ldhess;   /* [B][ldhess >= nnz_hess] */
    const double* jac;  int64_t ldjac;    /* [B][ldjac  >= nnz (SPARSE_TRUE)] */
    const double* sx;   int64_t ldsx;     /* [B][ldsx   >= n_nlp]   or NULL */
    const double* dc;   int64_t lddc;     /* [B][lddc   >= m_nlp] */
    const double* r1;   int64_t ldr1;     /* [B][ldr1   >= n_nlp] */
    const double* r2;   int64_t ldr2;     /* [B][ldr2   >= m_nlp] */
    const double* px;   int64_t ldpx;     /* [B][ldpx   >= n_nlp] */
    const double* pl;   int64_t ldpl;     /* [B][ldpl   >= m_nlp] */
    double* s1;         int64_t lds1;     /* [B][lds1   >= n_nlp] */
    double* s2;         int64_t lds2;     /* [B][lds2   >= m_nlp] */
} qlnlp_kkt_residual_io;
int qlnlp_kkt_residual_batch_device(qlnlp_handle h, int64_t B, const qlnlp_kkt_residual_io* io, void* stream);

/* Ragged batches: problems of different size (several handles = several (N, k_trans, init_mode) classes) packed
 * back to back in flat arrays.  One call evaluates the B problems of THIS handle's class; the b-th of them is problem
 * number i = index[b] (or b when index is NULL) of the flat batch and its rows start at
 *   io->Z + z_off[i],  io->grad + z_off[i],  io->g + g_off[i],  io->jac + jac_off[i]     (offsets in doubles)
 * while io->f, io->x0, io->xf are indexed by i.  The ld fields of io are ignored.  All pointers are device pointers.
 * Rows whose jac address is 16-byte aligned take the TMA store path, the others the plain one. */
typedef struct {
    const int64_t* index;    /* [B] or NULL */
    const int64_t* z_off;    /* [number of problems] */
    const int64_t* g_off;    /* required when io->g is set */
    const int64_t* jac_off;  /* required when io->jac is set */
    int64_t flags;           /* QLNLP_RAGGED_Z_PADDED: every z_off is even and every Z row is followed by at least one
                                readable double (rows padded to an even length): Z is then fetched with TMA loads */
} qlnlp_ragged_io;
#define QLNLP_RAGGED_Z_PADDED 1
int qlnlp_eval_ragged_device(qlnlp_handle h, int64_t B, const qlnlp_batch_io* io, const qlnlp_ragged_io* rg, void* stream);
/* The whole mixed batch in ONE launch: problem i belongs to the class of handles[class_of[i]] (all handles on one
 * device, same Jacobian pattern).  The B evaluations of the launch are the problems index[0..B) (or 0..B-1); a warp
 * swaps class records when the class changes from one of its evaluations to the next, so order `index` by class
 * (largest horizon first balances the tail).  class_of is a device array of int32; the handles must stay alive while
 * launches that name them are in flight. */
int qlnlp_eval_ragged_classes(const qlnlp_handle* handles, int nclasses, int64_t B, const qlnlp_batch_io* io,
                              const qlnlp_ragged_io* rg, const int32_t* class_of, void* stream);

/* One shard per device of a multi-device handle (or the single device of a plain one): B[i] evaluations on the
 * DEVICE pointers of io[i], which live on device i of the handle, enqueued on streams[i] (NULL array or entry = that
 * device's default stream).  Not synchronised; qlnlp_synchronize waits for every device of the handle. */
int qlnlp_eval_batch_device_multi(qlnlp_handle h, const int64_t* B, const qlnlp_batch_io* io, void* const* streams);
int qlnlp_synchronize(qlnlp_handle h);

/* All pointers are HOST pointers.  Copies Z (and x0/xf) to the device, evaluates, copies the requested outputs back,
 * and returns when they are in place.  Work is pipelined in chunks over four streams so copies overlap the kernel;
 * pinned (page-locked) host arrays make the copies asynchronous (qlnlp_host_pin).  For batches >= 64 only the
 * VALUE-DEPENDENT Jacobian entries cross PCIe (2,794 of the 32,161 SPARSE_BLOCK values at the default instance): a
 * persistent pool of host threads assembles the caller's rows from the constant image of the pattern (zeros, +-1)
 * and those entries, written a 64-byte line at a time with non-temporal stores -- identical rows, no host
 * arithmetic.  On a multi-device handle the batch is split into one contiguous shard per device. */
int qlnlp_eval_batch_host(qlnlp_handle h, int64_t B, const qlnlp_batch_io* io);

/* Registered output rows.  jac_c! itself assigns only part of the caller's matrix and relies on the rest of the
 * buffer keeping its zeros (constraints.jl:212-291 never clears it).  A host caller that reuses one `jac` array
 * for every batch can do the same here: qlnlp_host_output_register writes the constant image of the handle's
 * pattern into the B rows once; later qlnlp_eval_batch_host calls whose io->jac points at a row of that buffer
 * (same ldjac) rewrite only the 64-byte lines that hold a value-dependent entry (42 % of a SPARSE_BLOCK row at the
 * default instance).  The caller must not overwrite the rows in between (reading them is fine); unregister, or
 * register again, after doing so.  The resulting rows are identical to the unregistered ones. */
int qlnlp_host_output_register(qlnlp_handle h, double* jac, int64_t ldjac, int64_t B);
int qlnlp_host_output_unregister(qlnlp_handle h, double* jac);
/* page-lock / unlock a caller-owned host array (cudaHostRegister) so that copies to and from it are asynchronous */
int qlnlp_host_pin(void* ptr, int64_t bytes);
int qlnlp_host_unpin(void* ptr);
/* page-locked host memory on 2 MB pages where the kernel grants them (2 MB aligned, zero-filled).  Rows of 257 KB
 * each touch 63 small pages; on a virtualised host the page walks of the row builder then cost as much as its stores.
 * Free with qlnlp_host_free(ptr, same byte count). */
int qlnlp_host_alloc(int64_t bytes, void** out);
int qlnlp_host_free(void* ptr, int64_t bytes);
/* Device memory for the evaluator's outputs on the handle's device (for a multi-device handle: the calling thread's
 * current device, which must be one of the handle's).  Where the device reports CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_
 * SUPPORTED the block is compressible (cuMemCreate with CU_MEM_ALLOCATION_COMP_GENERIC, rounded up to the allocation
 * granularity): the compression is lossless and invisible to kernels and copies, and it cuts the DRAM traffic of
 * zero-rich rows such as the SPARSE_BLOCK Jacobian's.  Otherwise, when the driver declines a compressible block
 * (compressible backing is limited), or after qlnlp_set_option(h, "compressible", 0), the block is plain cudaMalloc
 * memory.  A compressible block is mapped read-write for its device and for every device that can access it peer to
 * peer, as cudaMalloc memory is; it cannot be exported with cudaIpcGetMemHandle (so neither shared through
 * torch.multiprocessing).  Blocks are at least 256-byte aligned.  Each call is a driver allocation: callers that
 * allocate per evaluation should keep and reuse their blocks (the Python layer draws its outputs from a caching pool
 * over these blocks).  Caller-owned buffers behave exactly as before; callers who want the gain allocate their
 * outputs here.  Returns QLNLP_ENODEVICE without a device. */
int qlnlp_device_alloc(qlnlp_handle h, int64_t bytes, void** out);
/* Frees a qlnlp_device_alloc block (NULL is a no-op).  Needs no handle: a block may outlive the handle it was
 * allocated through.  Waits for the block's device, as cudaFree does.  QLNLP_EINVAL for any other pointer. */
int qlnlp_device_free(void* ptr);
/* For a pointer inside a qlnlp_device_alloc block: [0] 1 if the block is compressible, [1] its device, [2] its length
 * in bytes.  QLNLP_EINVAL for any other pointer. */
int qlnlp_device_alloc_info(const void* ptr, int64_t info[3]);
/* host path facts: [0] row-builder threads per device, [1] Jacobian doubles per evaluation that cross PCIe,
 * [2] doubles per row, [3] 64-byte lines rewritten per registered row, [4] lines per row, [5] AVX-512 writer in use,
 * [6] rows assembled so far, [7] lines written so far */
int qlnlp_host_path_info(qlnlp_handle h, int64_t info[8]);

/* Launch geometry of the last batched launch (for benchmarks / profiles): blocks, threads per
 * block, dynamic shared memory per block, resident blocks per SM, SM count. */
int qlnlp_launch_info(qlnlp_handle h, int64_t info[5]);

const char* qlnlp_last_error(void);
int qlnlp_version(void);

#ifdef __cplusplus
}
#endif
#endif
