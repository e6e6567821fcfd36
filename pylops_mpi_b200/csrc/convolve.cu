// Batched 1-D convolution with a real filter along the middle axis of a C-ordered [n_outer][n_axis][n_inner]
// block: the rank-local pylops.signalprocessing.Convolve1D that MPIBlockDiag applies per rank
// (tutorials/reflectivity.py:75, BlockDiag.py:127-129).
//
//   forward: y[i] = sum_k h[k] x[i + offset - k]         (x = 0 outside [0, n_axis))
//   adjoint: x[j] = sum_k h[k] y[j - offset + k]
//
// Both are written as one correlation  out[i] = sum_q g[q] in[i - shift + q]  with
//   forward: g[q] = h[nh-1-q], shift = nh-1-offset;    adjoint: g[q] = h[q], shift = offset,
// so the adjoint is the exact transpose of the forward and one kernel serves both.  Every output sums its taps in
// increasing q with one FMA per tap in the data's precision: results do not depend on the launch shape.
//
// Two launch shapes:
//  * n_inner == 1 (time is the last axis): a CTA owns a TILE-sample piece of one row.  It stages the piece plus its
//    nhp-sample halo in shared memory (16-byte loads, zero outside the row), then each thread keeps R consecutive
//    outputs in registers and sweeps the taps R at a time over a 2R-sample register window, so one 16-byte
//    shared-memory read feeds 4R (float) / 2R (double) FMAs.  The window is padded by 16 bytes every 128 bytes so the
//    threads' R-strided 16-byte reads hit distinct banks.
//  * n_inner > 1: each thread owns a 16-byte inner column vector (one element when the columns are not 16-byte
//    aligned) and RB consecutive outputs along the axis; it marches its window along the axis through the L1
//    (cached loads: the CTA's axis groups overlap by the halo).  CTAs walk down the axis of one column block before
//    moving to the next, so the halo rows a CTA shares with the previous one come from L2.
#include "common.cuh"

namespace {

constexpr int CONV_R = 8;                         // outputs per thread, rows regime (also the tap padding)
constexpr int CONV_THREADS = 128;
constexpr int CONV_TILE = CONV_THREADS * CONV_R;  // outputs per CTA, rows regime
constexpr int CONV_RB = 4;                        // outputs per thread, columns regime
constexpr int CONV_CX = 32, CONV_CY = 8;          // columns regime CTA: 32 column vectors x 8 axis groups
constexpr int CONV_CTILE = CONV_CY * CONV_RB;     // axis outputs per CTA, columns regime

template <typename T>
__host__ __device__ constexpr int vlen() { return 16 / (int)sizeof(T); }

// padded shared-memory index: 16 bytes of padding after every 128 bytes
template <typename T>
__device__ __forceinline__ int sidx(int m) { return m + (m / (8 * vlen<T>())) * vlen<T>(); }

template <typename T>
__host__ __device__ inline int padded_len(int L) { return L + (L / (8 * vlen<T>()) + 1) * vlen<T>(); }

// 16-byte shared-memory read of V consecutive T (through uint4 so that it is one LDS.128, not V scalar reads)
template <typename T>
__device__ __forceinline__ void lds16(T* dst, const T* src) {
  *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(src);
}

// floor(a / b) for b > 0
__device__ __forceinline__ long long floordiv(long long a, long long b) { return a >= 0 ? a / b : -((-a + b - 1) / b); }

// taps in correlation order, zero-padded to nhp (a multiple of CONV_R)
template <typename T>
__device__ __forceinline__ void load_taps(T* gs, const T* __restrict__ h, int nh, int nhp, int flip, int tid, int nthr) {
  for (int q = tid; q < nhp; q += nthr) gs[q] = q < nh ? h[flip ? nh - 1 - q : q] : T(0);
}

template <typename T, bool VLD, bool VST>
__global__ void __launch_bounds__(CONV_THREADS)
conv_rows_kernel(const T* __restrict__ x, T* __restrict__ y, long long n_axis, long long tiles_per_row,
                 const T* __restrict__ h, int nh, int nhp, long long shift, int flip) {
  constexpr int V = vlen<T>();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* gs = reinterpret_cast<T*>(smem_raw);
  T* xs = gs + nhp;
  const long long row = blockIdx.x / tiles_per_row;
  const long long i0 = (blockIdx.x % tiles_per_row) * CONV_TILE;
  const long long lo = i0 - shift;                 // row coordinate of window sample 0
  const int L = CONV_TILE + nhp;
  load_taps(gs, h, nh, nhp, flip, threadIdx.x, CONV_THREADS);
  const long long rbeg = row * n_axis;             // flat index of the row's first sample
  if (VLD) {
    // 16-byte chunks (aligned in the flat array) covering the window; partial chunks at the row ends go scalar
    const long long a = rbeg + lo;
    const long long a0 = floordiv(a, V) * V;
    const int nchunks = (int)((a + L - a0 + V - 1) / V);
    for (int c = threadIdx.x; c < nchunks; c += CONV_THREADS) {
      const long long e0 = a0 + (long long)c * V;  // flat index of the chunk
      const long long p0 = e0 - rbeg;              // its row coordinate
      T v[V];
      if (p0 >= 0 && p0 + V <= n_axis) {
        Vec16<T> t = load_vec(x + e0);
#pragma unroll
        for (int j = 0; j < V; ++j) v[j] = t.v[j];
      } else {
#pragma unroll
        for (int j = 0; j < V; ++j) v[j] = (p0 + j >= 0 && p0 + j < n_axis) ? x[e0 + j] : T(0);
      }
#pragma unroll
      for (int j = 0; j < V; ++j) {
        const long long m = e0 + j - a;
        if (m >= 0 && m < L) xs[sidx<T>((int)m)] = v[j];
      }
    }
  } else {
    for (int m = threadIdx.x; m < L; m += CONV_THREADS) {
      const long long p = lo + m;
      xs[sidx<T>(m)] = (p >= 0 && p < n_axis) ? x[rbeg + p] : T(0);
    }
  }
  __syncthreads();

  const int base = threadIdx.x * CONV_R;
  __align__(16) T acc[CONV_R];
  __align__(16) T w[2 * CONV_R];
#pragma unroll
  for (int r = 0; r < CONV_R; ++r) acc[r] = T(0);
#pragma unroll
  for (int j = 0; j < CONV_R; j += V) lds16(&w[j], &xs[sidx<T>(base + j)]);
  for (int q0 = 0; q0 < nhp; q0 += CONV_R) {
    __align__(16) T g[CONV_R];
#pragma unroll
    for (int j = 0; j < CONV_R; j += V) {
      lds16(&w[CONV_R + j], &xs[sidx<T>(base + q0 + CONV_R + j)]);
      lds16(&g[j], &gs[q0 + j]);
    }
#pragma unroll
    for (int k = 0; k < CONV_R; ++k)
#pragma unroll
      for (int r = 0; r < CONV_R; ++r) acc[r] = fma(g[k], w[r + k], acc[r]);
#pragma unroll
    for (int j = 0; j < CONV_R; ++j) w[j] = w[CONV_R + j];
  }

  const long long i = i0 + base;                   // row coordinate of acc[0]
  T* yr = y + rbeg;
  if (VST) {                                       // n_axis % V == 0: a chunk is wholly in or out of the row
#pragma unroll
    for (int j = 0; j < CONV_R; j += V)
      if (i + j < n_axis) store_vec(yr + i + j, *reinterpret_cast<const Vec16<T>*>(&acc[j]));
  } else {
#pragma unroll
    for (int r = 0; r < CONV_R; ++r)
      if (i + r < n_axis) yr[i + r] = acc[r];
  }
}

template <typename T, int W>
struct ColVec {
  T v[W];
};

template <typename T, int W>
__device__ __forceinline__ ColVec<T, W> load_col(const T* p) {
  ColVec<T, W> o;
  if constexpr (W == 1) {
    o.v[0] = __ldg(p);
  } else if constexpr (sizeof(T) == 4) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(p));
    o.v[0] = t.x; o.v[1] = t.y; o.v[2] = t.z; o.v[3] = t.w;
  } else {
    const double2 t = __ldg(reinterpret_cast<const double2*>(p));
    o.v[0] = t.x; o.v[1] = t.y;
  }
  return o;
}

// W = elements per thread column: 16 / sizeof(T) when the columns are 16-byte aligned, else 1
template <typename T, int W>
__global__ void __launch_bounds__(CONV_CX * CONV_CY)
conv_cols_kernel(const T* __restrict__ x, T* __restrict__ y, long long n_axis, long long n_inner, long long axis_tiles,
                 long long col_tiles, const T* __restrict__ h, int nh, int nhp, long long shift, int flip) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* gs = reinterpret_cast<T*>(smem_raw);
  const int tid = threadIdx.y * CONV_CX + threadIdx.x;
  load_taps(gs, h, nh, nhp, flip, tid, CONV_CX * CONV_CY);
  __syncthreads();
  long long b = blockIdx.x;
  const long long at = b % axis_tiles;
  b /= axis_tiles;
  const long long ct = b % col_tiles;
  const long long o = b / col_tiles;
  const long long col = (ct * CONV_CX + threadIdx.x) * W;
  const long long i0 = at * CONV_CTILE + (long long)threadIdx.y * CONV_RB;
  if (col >= n_inner || i0 >= n_axis) return;
  const T* xo = x + o * n_axis * n_inner + col;
  T* yo = y + o * n_axis * n_inner + col;
  const long long lo = i0 - shift;                 // axis coordinate of window sample 0

  auto load = [&](long long m) {
    const long long p = lo + m;
    ColVec<T, W> v;
    if (p >= 0 && p < n_axis) return load_col<T, W>(xo + p * n_inner);
#pragma unroll
    for (int e = 0; e < W; ++e) v.v[e] = T(0);
    return v;
  };

  ColVec<T, W> acc[CONV_RB], w[2 * CONV_RB];
#pragma unroll
  for (int r = 0; r < CONV_RB; ++r)
#pragma unroll
    for (int e = 0; e < W; ++e) acc[r].v[e] = T(0);
#pragma unroll
  for (int j = 0; j < CONV_RB; ++j) w[j] = load(j);
  for (int q0 = 0; q0 < nhp; q0 += CONV_RB) {
#pragma unroll
    for (int j = 0; j < CONV_RB; ++j) w[CONV_RB + j] = load(q0 + CONV_RB + j);
#pragma unroll
    for (int k = 0; k < CONV_RB; ++k) {
      const T g = gs[q0 + k];
#pragma unroll
      for (int r = 0; r < CONV_RB; ++r)
#pragma unroll
        for (int e = 0; e < W; ++e) acc[r].v[e] = fma(g, w[r + k].v[e], acc[r].v[e]);
    }
#pragma unroll
    for (int j = 0; j < CONV_RB; ++j) w[j] = w[CONV_RB + j];
  }
#pragma unroll
  for (int r = 0; r < CONV_RB; ++r) {
    if (i0 + r >= n_axis) break;
    T* p = yo + (i0 + r) * n_inner;
    if constexpr (W == 1) {
      *p = acc[r].v[0];
    } else {
      store_vec(p, *reinterpret_cast<const Vec16<T>*>(&acc[r]));
    }
  }
}

template <typename T>
int launch_conv(const void* x, void* y, size_t n_outer, size_t n_axis, size_t n_inner, const void* taps, int nh,
                long long shift, int flip, cudaStream_t st) {
  constexpr int V = vlen<T>();
  const int nhp = (nh + CONV_R - 1) / CONV_R * CONV_R;
  const T* xp = (const T*)x;
  T* yp = (T*)y;
  const T* hp = (const T*)taps;
  if (n_inner == 1) {
    const long long tiles = ((long long)n_axis + CONV_TILE - 1) / CONV_TILE;
    const size_t smem = (size_t)(nhp + padded_len<T>(CONV_TILE + nhp)) * sizeof(T);
    const bool vld = b2_aligned16(x), vst = b2_aligned16(y) && n_axis % V == 0;
    const dim3 grid((unsigned)(tiles * (long long)n_outer));
#define B2_CONV_ROWS(VL, VS) \
    conv_rows_kernel<T, VL, VS><<<grid, CONV_THREADS, smem, st>>>(xp, yp, (long long)n_axis, tiles, hp, nh, nhp, shift, flip)
    if (vld && vst) B2_CONV_ROWS(true, true);
    else if (vld) B2_CONV_ROWS(true, false);
    else if (vst) B2_CONV_ROWS(false, true);
    else B2_CONV_ROWS(false, false);
#undef B2_CONV_ROWS
  } else {
    const bool vec = b2_aligned16(x) && b2_aligned16(y) && n_inner % V == 0;
    const long long ncv = vec ? (long long)(n_inner / V) : (long long)n_inner;
    const long long col_tiles = (ncv + CONV_CX - 1) / CONV_CX;
    const long long axis_tiles = ((long long)n_axis + CONV_CTILE - 1) / CONV_CTILE;
    const size_t smem = (size_t)nhp * sizeof(T);
    const dim3 grid((unsigned)(axis_tiles * col_tiles * (long long)n_outer)), block(CONV_CX, CONV_CY);
    if (vec)
      conv_cols_kernel<T, V><<<grid, block, smem, st>>>(xp, yp, (long long)n_axis, (long long)n_inner, axis_tiles,
                                                         col_tiles, hp, nh, nhp, shift, flip);
    else
      conv_cols_kernel<T, 1><<<grid, block, smem, st>>>(xp, yp, (long long)n_axis, (long long)n_inner, axis_tiles,
                                                         col_tiles, hp, nh, nhp, shift, flip);
  }
  B2_LAUNCH_CHECK();
  return B2_OK;
}

}  // namespace

extern "C" int b2_convolve1d(b2_ctx* ctx, const void* x, void* y, size_t n_outer, size_t n_axis, size_t n_inner,
                             const void* taps, int nh, long long offset, int adjoint, int dtype, void* stream) {
  if (!ctx) return B2_ERR_ARG;
  if (nh < 1) return B2_ERR_ARG;
  if (nh > B2_CONV_MAX_TAPS) return B2_ERR_UNSUPPORTED;
  if (dtype != B2_F32 && dtype != B2_F64) return B2_ERR_DTYPE;
  if (n_outer == 0 || n_axis == 0 || n_inner == 0) return B2_OK;
  if (!x || !y || !taps) return B2_ERR_ARG;
  const size_t bytes = n_outer * n_axis * n_inner * b2_dtype_size(dtype);
  if ((const char*)x < (const char*)y + bytes && (const char*)y < (const char*)x + bytes) return B2_ERR_ARG;  // no in-place
  // grid size: one CTA per tile, gridDim.x <= 2^31 - 1
  const long long tiles = n_inner == 1
      ? (long long)((n_axis + CONV_TILE - 1) / CONV_TILE) * (long long)n_outer
      : (long long)((n_axis + CONV_CTILE - 1) / CONV_CTILE) * (long long)((n_inner + CONV_CX - 1) / CONV_CX) *
            (long long)n_outer;
  if (tiles > 0x7fffffffLL) return B2_ERR_UNSUPPORTED;
  const long long shift = adjoint ? offset : (long long)nh - 1 - offset;
  const int flip = adjoint ? 0 : 1;
  cudaStream_t st = (cudaStream_t)stream;
  return dtype == B2_F32 ? launch_conv<float>(x, y, n_outer, n_axis, n_inner, taps, nh, shift, flip, st)
                         : launch_conv<double>(x, y, n_outer, n_axis, n_inner, taps, nh, shift, flip, st);
}
