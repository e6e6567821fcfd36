/* b200lops.h -- C ABI of libb200lops.so
 *
 * B200-native (sm_100a) kernels + NCCL collectives for the pylops-mpi
 * distributed matvec/rmatvec hot path.  Plain pointers and sizes only: every
 * buffer is a raw DEVICE pointer owned by the caller (unless a parameter is
 * explicitly named *_host), every stream is a cudaStream_t passed as void*.
 * Every entry point returns 0 on success, a cudaError_t (1..999) on a CUDA
 * failure, 1000+ncclResult_t on an NCCL failure, or a B2_ERR_* code; none
 * throws, none frees or retains caller memory past the call (handles such as
 * b2_ctx / b2_comm own their private workspaces and have *_destroy).
 *
 * Each declaration cites the reference interface (file:line relative to
 * pylops_mpi/ of PyLops/pylops-mpi @ fb5b7d4) it replaces.
 */
#ifndef B200LOPS_H
#define B200LOPS_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2_VERSION 100

/* element types */
enum { B2_F32 = 0, B2_F64 = 1, B2_C64 = 2, B2_C128 = 3, B2_BF16 = 4, B2_I64 = 5 };
/* reduction operators (mpi4py MPI.SUM / MPI.MAX / MPI.MIN, utils/_nccl.py:23-43) */
enum { B2_SUM = 0, B2_MAX = 1, B2_MIN = 2 };
/* local part of DistributedArray._compute_vector_norm, DistributedArray.py:688-758 */
enum { B2_NRM_COUNT_NONZERO = 0, B2_NRM_SUM_ABS = 1, B2_NRM_SUM_SQ = 2,
       B2_NRM_MAX_ABS = 3, B2_NRM_MIN_ABS = 4, B2_NRM_SUM_POW = 5 };
/* MPIFirstDerivative kinds, basicoperators/FirstDerivative.py:104-127 */
enum { B2_FD_FORWARD = 0, B2_FD_BACKWARD = 1, B2_FD_CENTERED = 2 };
/* op(A) for gemv/gemm */
enum { B2_OP_N = 0, B2_OP_T = 1, B2_OP_H = 2 };
enum { B2_THRESH_NONE = 0, B2_THRESH_SOFT = 1, B2_THRESH_HARD = 2, B2_THRESH_HALF = 3 };

/* error codes >= 2000 are library-level */
enum { B2_OK = 0, B2_ERR_DTYPE = 2001, B2_ERR_ARG = 2002, B2_ERR_HALO = 2003,
       B2_ERR_WORKSPACE = 2004, B2_ERR_UNSUPPORTED = 2005, B2_ERR_ALIGN = 2006 };

/* per-device context: SM count + the reduction workspace (per-CTA partials, ticket counter) shared by b2_dot /
 * b2_norm_partial / b2_dot_multi / b2_sparse_update / the transposed b2_gemv.  Calls that use the workspace must be
 * stream-ordered with respect to each other: use one b2_ctx per stream that issues reductions concurrently. */
typedef struct b2_ctx b2_ctx;
typedef struct b2_comm b2_comm;          /* one NCCL communicator (world, mask group, grid row / col) */
typedef struct b2_peer b2_peer;          /* peer-memory mailbox group for one-shot SCALAR all-reduces */
typedef struct b2_peer_vec b2_peer_vec;  /* peer-memory mailboxes for one-shot VECTOR all-reduces */

int b2_version(void);
const char* b2_strerror(int code);

/* ---- context --------------------------------------------------------- */
int b2_ctx_create(int device, b2_ctx** out);
int b2_ctx_destroy(b2_ctx* ctx);
int b2_ctx_sm_count(const b2_ctx* ctx, int* out);

/* ---- element-wise (DistributedArray.py:574-652, 809-837: add, iadd,
 *      multiply, __neg__, conj, copy, zeros_like) ------------------------- */
/* out = a * op(x) + b * y ; a,b are (re,im) host pairs; y may be NULL (b ignored);
 * op = conj when conj_x != 0.  out may alias x or y. */
int b2_lincomb(b2_ctx* ctx, void* out, const double a[2], const void* x, const double b[2],
               const void* y, size_t n, int dtype, int conj_x, void* stream);
/* Same with DEVICE-resident real scalars: a = a_scale * (*a_dev) (a_dev may be NULL -> 1),
 * b likewise; lets a solver iteration run with no host round-trip
 * (optimization/cls_basic.py:389-397 does five .item() syncs per iteration). */
int b2_lincomb_dev(b2_ctx* ctx, void* out, const double* a_dev, double a_scale, const void* x,
                   const double* b_dev, double b_scale, const void* y, size_t n, int dtype,
                   void* stream);
/* b2_lincomb_dev fused with the reduction the CGLS recurrence needs next: out = a x + b y (real device scalars) and
 * norm2_dev[0] = sum |out|^2 (float64, local partial; norm2_dev[1] = 0 for complex dtypes so that the caller's
 * (re, im) slot layout is kept).  x.x after x += a c, s.s after s -= a q, c.c after c = r + b c
 * (cls_basic.py:389-401): one pass and one launch each instead of two.  Shares the ctx reduction workspace. */
int b2_lincomb_dev_norm2(b2_ctx* ctx, void* out, const double* a_dev, double a_scale, const void* x,
                         const double* b_dev, double b_scale, const void* y, size_t n, int dtype,
                         double* norm2_dev, void* stream);
/* out = op(x) * y element-wise (DistributedArray.multiply, :630-652) */
int b2_mul(b2_ctx* ctx, void* out, const void* x, const void* y, size_t n, int dtype,
           int conj_x, void* stream);
int b2_fill(b2_ctx* ctx, void* out, const double v[2], size_t n, int dtype, void* stream);

/* ---- local reductions (the per-rank half of DistributedArray.dot :654-686
 *      and _compute_vector_norm :688-758); results are float64 in DEVICE
 *      memory, accumulated in float64 in a fixed (deterministic) order ----- */
/* out_dev[0..1] = sum_i op(x_i) * y_i  (re, im); op = conj when conj_x (numpy.vdot) */
int b2_dot(b2_ctx* ctx, const void* x, const void* y, size_t n, int dtype, int conj_x,
           double* out_dev, void* stream);
/* out_dev[0] = local partial for the requested norm kind (p only for SUM_POW) */
int b2_norm_partial(b2_ctx* ctx, const void* x, size_t n, int dtype, int kind, double p,
                    double* out_dev, void* stream);
/* axis-wise variant (DistributedArray.norm(ord, axis=...), DistributedArray.py:688-758, 796-807): x is the local block
 * viewed as [n_outer][n_axis][n_inner]; out_dev[o * n_inner + i] = float64 partial over the middle axis for the same
 * norm kinds (the caller combines partials across ranks when the axis is the partition axis and takes the root) */
int b2_norm_axis(b2_ctx* ctx, const void* x, size_t n_outer, size_t n_axis, size_t n_inner, int dtype, int kind,
                 double p, double* out_dev, void* stream);
/* k dot products <x_j, y_j> in ONE launch: out_dev[0..k) for real dtypes, out_dev[0..2k) as
 * (re, im) pairs for complex dtypes (CGLS needs q.q and c.c
 * together, r.r / s.s / x.x together -- cls_basic.py:389, 394-401) */
int b2_dot_multi(b2_ctx* ctx, int k, const void* const* xs, const void* const* ys, size_t n,
                 int dtype, int conj_x, double* out_dev, void* stream);

/* out = |num / (den1 + alpha * den2)| on DEVICE scalars (den2 may be NULL): the CGLS step length
 * a = kold / (q.q + damp c.c) and ratio b = k / kold (cls_basic.py:389, 395) with no host sync */
int b2_scalar_div(double* out_dev, const double* num_dev, const double* den1_dev,
                  const double* den2_dev, double alpha, void* stream);

/* Device-side history of solver scalars: hist[it * nvals + j] = |src[j * stride]| (skipped when it >= cap), then the
 * optional scalar copy *copy_dst = *copy_src (kold <- k, cls_basic.py:397) and ++(*it_dev) (uint64).  With it a block of
 * CGLS iterations (cls_basic.py:370-404) needs no host synchronisation and can be replayed as a CUDA graph. */
int b2_history_push(const double* src_dev, int nvals, int stride, double* hist_dev, void* it_dev, size_t cap,
                    double* copy_dst_dev, const double* copy_src_dev, void* stream);

/* ---- ISTA / FISTA model update ("next" row; optimization/cls_sparsity.py:270-343, 578-662) in ONE pass:
 *   u = base + alpha*g (g may be NULL);  v = threshold_kind(u, thresh) (_apply_thresh, cls_sparsity.py:21-46);
 *   xnew = v;  znew = v + c*(v - xold) (znew may be NULL; FISTA's auxiliary model, :640-644);
 *   sums_dev[0] = sum|v - xold|^2 (0 if xold NULL), sums_dev[1] = sum|v| -- local partials of the update norm
 *   (:331) and the l1 cost (:333).  xnew/znew may alias base/xold.  HALF is real-only. */
int b2_sparse_update(b2_ctx* ctx, const void* base, const void* g, double alpha, const void* xold,
                     double thresh, int kind, void* xnew, void* znew, double c, double* sums_dev,
                     size_t n, int dtype, void* stream);

/* ---- MPIFirstDerivative per-rank apply (FirstDerivative.py:129-319) -------
 * x,y: this rank's row block [nrows_local x ncols] (C order) of the global
 * [nrows_global x ncols] array, global row offset row0.  halo_lo holds the n_lo
 * rows immediately before row0, halo_hi the n_hi rows immediately after the
 * block (the add_ghost_cells payload, DistributedArray.py:876-953); NULL / 0
 * at the global edges.  Complex arrays: pass the real dtype and 2*ncols. */
int b2_first_derivative(b2_ctx* ctx, const void* x, void* y, const void* halo_lo, int n_lo,
                        const void* halo_hi, int n_hi, size_t nrows_local, size_t ncols,
                        size_t row0, size_t nrows_global, int kind, int order, int edge,
                        double sampling, int adjoint, int dtype, void* stream);
/* rows of halo each side needs (1 or 2) */
int b2_first_derivative_halo(int kind, int order, int adjoint, int* need_lo, int* need_hi);
/* MPISecondDerivative per-rank apply (basicoperators/SecondDerivative.py:125-257): same contract as
 * b2_first_derivative (row block + up to 2 halo rows per side, exact-transpose adjoint), scale 1/sampling^2 */
int b2_second_derivative(b2_ctx* ctx, const void* x, void* y, const void* halo_lo, int n_lo,
                         const void* halo_hi, int n_hi, size_t nrows_local, size_t ncols, size_t row0,
                         size_t nrows_global, int kind, int edge, double sampling, int adjoint, int dtype,
                         void* stream);
int b2_second_derivative_halo(int kind, int edge, int adjoint, int* need_lo, int* need_hi);
/* rank-local first (deriv=1) / second (deriv=2) derivative along the MIDDLE axis of a C-ordered
 * [n_outer][n_axis][n_inner] block: the non-partitioned directions of MPILaplacian / MPIGradient
 * (Laplacian.py:97-126, Gradient.py:101-119 wrap a serial pylops derivative per rank) */
int b2_derivative_axis(b2_ctx* ctx, const void* x, void* y, size_t n_outer, size_t n_axis, size_t n_inner,
                       int deriv, int kind, int order, int edge, double sampling, int adjoint, int dtype,
                       void* stream);
/* rank-local 1-D convolution with a real filter along the MIDDLE axis of a C-ordered [n_outer][n_axis][n_inner]
 * block: the pylops.signalprocessing.Convolve1D that MPIBlockDiag applies per rank (tutorials/reflectivity.py:75,
 * basicoperators/BlockDiag.py:127-129).  taps: nh DEVICE values of the data's precision (dtype B2_F32 | B2_F64;
 * complex data: pass the real dtype with the (re, im) pairs folded into n_inner).  Zero outside [0, n_axis):
 *   forward:  y[i] = sum_k taps[k] x[i + offset - k]
 *   adjoint:  y[j] = sum_k taps[k] x[j - offset + k]     (the exact transpose)
 * Any offset; 1 <= nh <= B2_CONV_MAX_TAPS (else B2_ERR_UNSUPPORTED).  x and y must not overlap.  Each output sums
 * its taps in a fixed order in the data's precision: results are identical from run to run. */
#define B2_CONV_MAX_TAPS 2048
int b2_convolve1d(b2_ctx* ctx, const void* x, void* y, size_t n_outer, size_t n_axis, size_t n_inner,
                  const void* taps, int nh, long long offset, int adjoint, int dtype, void* stream);
/* Peer-memory halo exchange fused INTO the stencil kernel (replaces the add_ghost_cells Send/Recv pairs of
 * DistributedArray.py:876-953 as used by FirstDerivative.py:221-247, 276-319 and SecondDerivative.py): every rank
 * owns a box of b2_halo_bytes(cap) bytes in IPC-mapped memory (b2_symm_alloc + b2_ipc_*); boxes_host[r] is rank r's
 * box as mapped in this process.  b2_derivative_peer is ONE launch per apply: the first CTAs push the boundary rows
 * into the neighbours' boxes over NVLink and publish a flag, the CTAs of the first / last row chunk run last and
 * wait for it.  Collective: same call sequence on every rank of the handle, all on one stream; each rank must
 * own >= 2 rows; 2 * ncols * sizeof(dtype) must fit in cap_bytes.  deriv = 1 | 2 (first | second derivative). */
typedef struct b2_halo b2_halo;
size_t b2_halo_bytes(size_t cap_bytes);
int b2_halo_create(int rank, int size, void* const* boxes_host, size_t cap_bytes, b2_halo** out);
int b2_halo_destroy(b2_halo* h);
int b2_derivative_peer(b2_ctx* ctx, b2_halo* h, const void* x, void* y, size_t nrows_local, size_t ncols,
                       size_t row0, size_t nrows_global, int deriv, int kind, int order, int edge, double sampling,
                       int adjoint, int dtype, void* stream);
/* Same operator on HOST buffers (pageable or pinned).  x_host / y_host address the
 * GLOBAL [nrows_global x ncols] arrays (to_dist keeps the global array replicated on
 * every rank's host, DistributedArray.py:440-459); this call processes rows
 * [row_begin, row_end) and only touches rows [row_begin-2, row_end+2) of x_host and
 * [row_begin, row_end) of y_host.  Row chunks go through the device with H2D /
 * kernel / D2H overlapped on three streams.  This is the host-buffer plugin entry
 * the end-to-end benchmark times. */
int b2_first_derivative_host(b2_ctx* ctx, const void* x_host, void* y_host, size_t nrows_global,
                             size_t ncols, size_t row_begin, size_t row_end, int kind, int order,
                             int edge, double sampling, int adjoint, int dtype);

/* ---- dense per-rank matvec (the pylops.MatrixMult block inside MPIBlockDiag /
 *      MPIVStack, BlockDiag.py:127-129,139-141; VStack.py:129-131,144-145; and
 *      the M==1 tile product of MPIMatrixMult, MatrixMult.py:366-370,670) ----
 * y[m or n] = op(A[m x n, row-major, leading dim lda]) x ; dtype_a in
 * {F32,F64,C64,C128,BF16}; x,y have dtype_xy (BF16 A pairs with F32 x/y). */
int b2_gemv(b2_ctx* ctx, const void* A, size_t lda, size_t m, size_t n, const void* x, void* y,
            int op, int dtype_a, int dtype_xy, void* stream);

/* ---- dense tile product on tcgen05 tensor cores (MPIMatrixMult with M>1,
 *      MatrixMult.py:663-670, 742-763): C[m x n] (+)= op(A) B, A,B bf16,
 *      C fp32, all row-major ------------------------------------------------ */
int b2_gemm_bf16(b2_ctx* ctx, const void* A, size_t lda, const void* B, size_t ldb, float* C,
                 size_t ldc, size_t m, size_t n, size_t k, int op_a, int accumulate,
                 void* stream);
/* Stationary-A MPIMatrixMult (round 2): A tiles are operator state and never move; per apply the small operand is
 * all-gathered (cast to bf16 on the fly) and the partial products are reduce-scattered by the GEMM epilogue itself.
 *   b2_cast_bf16_multi: float32 tile -> bfloat16, stored to ndst <= 8 destinations (local or IPC-mapped peers):
 *                       the X / Y panel broadcasts of MatrixMult.py:663-670, 742-763 as ONE read of the tile.
 *   b2_gemm_bf16_seg  : op(A) B on tcgen05 with the output columns cut into nseg <= 8 segments of seg_cols
 *                       (multiple of 32) columns, segment c written to segs_host[c] (leading dimension ldc) -- peer
 *                       GPUs' staging buffers, i.e. the reduce-scatter rides on the epilogue's NVLink stores.
 *   b2_sum_slots      : out[rows x cols] = sum_s slots[s * slot_stride + r * ld_in + c] in slot order. */
int b2_cast_bf16_multi(b2_ctx* ctx, const float* src, size_t ld_src, size_t rows, size_t cols,
                       void* const* dsts_host, int ndst, size_t ld_dst, void* stream);
int b2_gemm_bf16_seg(b2_ctx* ctx, const void* A, size_t lda, const void* B, size_t ldb, float* const* segs_host,
                     int nseg, size_t seg_cols, size_t ldc, size_t m, size_t n, size_t k, int op_a, void* stream);
int b2_sum_slots(b2_ctx* ctx, const float* slots, size_t slot_stride, int nslots, size_t ld_in, float* out,
                 size_t rows, size_t cols, void* stream);
/* generic SIMT tile product for the dtypes tensor cores do not serve
 * (f32/f64/c64/c128 parity cases of tests/test_matrixmult.py) */
int b2_gemm(b2_ctx* ctx, const void* A, size_t lda, const void* B, size_t ldb, void* C, size_t ldc,
            size_t m, size_t n, size_t k, int op_a, int accumulate, int dtype, void* stream);

/* ---- MPIFredholm1 per-rank batched product (Fredholm1.py:119-129, 147-167):
 *      y[s] = op(G[s]) x[s] for s < nsl ; G[s] is nx x ny, x[s] is (ny|nx) x nz */
int b2_batched_gemm(b2_ctx* ctx, const void* G, const void* x, void* y, size_t nsl, size_t nx,
                    size_t ny, size_t nz, int adjoint, int dtype, void* stream);

/* Fused product + all-gather over NVLink peer memory: the epilogue stores every output element to
 * y (local) and to the same offset of `npeers` peer buffers (IPC-mapped; peers_host[d] already points
 * at the position matching y).  Replaces product-then-Allgather of Fredholm1.py:122-132 by ONE kernel;
 * completion across ranks = any stream-ordered collective after it (e.g. a 1-element b2_allreduce). */
int b2_batched_gemm_allgather(b2_ctx* ctx, const void* G, const void* x, void* y, void* const* peers_host,
                              int npeers, size_t nsl, size_t nx, size_t ny, size_t nz, int adjoint,
                              int dtype, void* stream);
/* Tensor-core (tcgen05) plan for the same product, float32 / complex64 only (Fredholm1.py:119-129, 147-167).
 * G is operator state: plan creation splits G and G^H (the reference's `saveGt`, :105-106) ONCE into three bf16
 * planes each ("bf16x3": 24 significant bits, six MMAs per k-step -> float32-class accuracy on the bf16 tensor
 * pipe); complex64 runs as one real product over the (re,im)-interleaved views.  b2_fredholm_apply packs x
 * (one small kernel) and runs the batched product; with npeers > 0 the epilogue also stores every output
 * element to the same offset of the peers' IPC-mapped buffers (fused Allgather of Fredholm1.py:131-132,
 * completion = any stream-ordered cross-rank barrier after it).  The plan owns its device workspaces; applies
 * of one plan must be stream-ordered.  G must stay valid only during b2_fredholm_plan_create. */
typedef struct b2_fredholm_plan b2_fredholm_plan;
int b2_fredholm_plan_create(b2_ctx* ctx, const void* G, size_t nsl, size_t nx, size_t ny, size_t nz, int dtype,
                            b2_fredholm_plan** out);
int b2_fredholm_plan_destroy(b2_fredholm_plan* plan);
int b2_fredholm_apply(b2_fredholm_plan* plan, const void* x, void* y, void* const* peers_host, int npeers,
                      int adjoint, void* stream);
/* profiling aid: parts = 1 packs x only, 2 = product on the planes of the previous pack, 3 = both */
int b2_fredholm_apply_parts(b2_fredholm_plan* plan, const void* x, void* y, int adjoint, int parts, void* stream);
/* peer-mappable device buffers (cudaMalloc) and CUDA IPC handle plumbing (64-byte handles) */
int b2_symm_alloc(size_t bytes, void** out);
int b2_symm_free(void* p);
int b2_ipc_get_handle(void* p, void* handle64_host);
int b2_ipc_open_handle(const void* handle64_host, void** out);
int b2_ipc_close_handle(void* p);

/* One-shot all-reduce of k <= 8 float64 scalars over NVLink peer memory (no NCCL): the collective half
 * of DistributedArray.dot / norm (DistributedArray.py:684-686, 714-757) and of the CGLS step scalars.
 * slots_host[r] = rank r's mailbox (b2_symm_alloc of b2_peer_slots_bytes(), IPC-mapped here). */
size_t b2_peer_slots_bytes(void);
int b2_peer_create(int rank, int size, void* const* slots_host, b2_peer** out);
int b2_peer_destroy(b2_peer* peer);
int b2_peer_allreduce(b2_peer* peer, double* vals_dev, int k, int op, void* stream);

/* One-shot SUM all-reduce of a small vector (<= b2_peer_vec_max_bytes()) over peer memory: the array
 * Allreduce of MPIVStack._rmatvec (VStack.py:146-148) / MatrixMult.py:420-426 in the latency regime.
 * boxes_host[r] = rank r's mailbox (b2_symm_alloc of b2_peer_vec_bytes(), IPC-mapped here). */
size_t b2_peer_vec_bytes(void);
size_t b2_peer_vec_max_bytes(void);
int b2_peer_vec_create(int rank, int size, void* const* boxes_host, b2_peer_vec** out);
int b2_peer_vec_destroy(b2_peer_vec* h);
int b2_peer_vec_allreduce(b2_peer_vec* h, void* buf_dev, size_t n, int dtype, void* stream);

/* One-shot Allgather(v) over the same mailboxes (every chunk <= b2_peer_vec_max_bytes()): recv = concatenation of the
 * ranks' counts_host[r] elements.  The latency-regime replacement of the pad-to-max NCCL gather of
 * utils/_nccl.py:363-403 (e.g. the 128 KB model vector of MPIMatrixMult's single-column apply). */
int b2_peer_vec_allgatherv(b2_peer_vec* h, const void* send, void* recv, const size_t* counts_host, int dtype,
                           void* stream);

/* ---- NCCL collectives (utils/_nccl.py:98-403, utils/_mpi.py:21-344,
 *      Distributed.py:35-349) --------------------------------------------- */
int b2_get_unique_id(void* id128_host);                       /* _nccl.py:98-132 */
int b2_comm_create(int rank, int size, const void* id128_host, int device, b2_comm** out);
int b2_comm_split(b2_comm* comm, int color, int key, b2_comm** out);   /* _nccl.py:135-165 */
int b2_comm_destroy(b2_comm* comm);
int b2_comm_rank(const b2_comm* comm, int* rank, int* size);
int b2_allreduce(b2_comm* comm, const void* send, void* recv, size_t n, int dtype, int op,
                 void* stream);                               /* _nccl.py:203-240 */
int b2_allgather(b2_comm* comm, const void* send, void* recv, size_t n_per_rank, int dtype,
                 void* stream);                               /* _nccl.py:167-200 */
/* uneven gather without the reference's pad-to-max (_nccl.py:363-403): rank r
 * contributes counts[r] elements; recv is the plain concatenation */
int b2_allgatherv(b2_comm* comm, const void* send, void* recv, const size_t* counts_host,
                  int dtype, void* stream);
/* same, with explicit placement: rank r's counts[r] elements land at recv + offsets[r] (elements);
 * send may alias its own destination (in-place).  Enables chunked gather overlapped with compute. */
int b2_allgatherv_at(b2_comm* comm, const void* send, void* recv, const size_t* counts_host,
                     const size_t* offsets_host, int dtype, void* stream);
int b2_bcast(b2_comm* comm, void* buf, size_t n, int dtype, int root, void* stream);  /* :243-262 */
int b2_send(b2_comm* comm, const void* buf, size_t n, int dtype, int peer, void* stream); /* :265-286 */
int b2_recv(b2_comm* comm, void* buf, size_t n, int dtype, int peer, void* stream);       /* :289-316 */
int b2_group_start(void);
int b2_group_end(void);

#ifdef __cplusplus
}
#endif
#endif /* B200LOPS_H */
