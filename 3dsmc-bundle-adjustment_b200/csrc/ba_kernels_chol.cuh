// ba_kernels_chol.cuh -- blocked dense Cholesky for the explicit Schur complement of LARGE REF-mode
// problems (free intrinsics make the reduced system a dense-bordered matrix, so the reference's
// "global optimisation" call -- windowOptimize(cfg, 0, keyframes.size() - 1, ...), src/main.cpp:179-182
// -- needs an exact dense solve beyond the single-CTA kernel's 1024 unknowns).
//
// Right-looking, 64 x 64 fp64 tiles, lower triangle of the row-major n x n matrix, in place:
//   for k = 0 .. nt-1:   k_chol_potrf2  diagonal tile (one CTA: register-resident L D L^T, yields L_kk and L_kk^-1)
//                        k_chol_trsm2   tiles (i, k), i > k:  L_ik = A_ik L_kk^-T   (a product with L_kk^-1)
//                        k_chol_update  tiles (i, j), k < j <= i:  A_ij -= L_ik L_jk^T
//                                       (256 threads, 4 x 4 outputs each, both operand tiles in shared memory)
// then k_chol_solve2: blocked forward / backward substitution through the stored L_kk^-1 tiles and the scatter into y_c / y_k.
// On one GPU the steps are software-pipelined over three streams (ba_gpu.cu: factor_blocked_lookahead2): the diagonal kernel
// brings its own tile up to date (fused prologue), so it is the only kernel on the critical chain.
// The first versions (left-looking diagonal tile, one-thread-per-row panel, substitution with grid barriers) were removed;
// the timings quoted below for them are the measurements that replaced them.
// Every sum has a fixed order (no atomics).  == the exact step of Ceres DENSE_SCHUR / SPARSE_SCHUR.
#pragma once
#include "ba_kernels.cuh"

#define CH_NB 64
#define CH_LD (CH_NB + 1)

// trailing update with panel k, A_ij -= L_ik L_jk^T, of the lower-triangle tiles (i, j), kmap < j <= i (linear CTA index ->
// tile), or, with single_col, of the tiles (i, kmap + 1) only.  kmap = k: the whole trailing matrix; the look-ahead
// schedule splits it into the next column (single_col) and the rest (kmap = k + 1).
// Bsub != nullptr (single_col only, look-ahead schedule): the column operand L_{k+1,k} comes from the side buffer and the
// diagonal tile (k + 1, k + 1) is left to the fused k_chol_potrf2: tiles (i, k + 1), i >= k + 2.
// BAND-AWARE tile rows.  The reduced matrix of a keyframe SEQUENCE is block-banded (a landmark track is a run of neighbouring
// keyframes) with the 4 intrinsics columns as a dense border at the end; Cholesky creates no fill outside band + border.
// For tile column k the tile rows that can be non-zero below the diagonal are the n_band rows k + 1 .. k + n_band and the
// border rows bord0 .. (last); "active row" t of a launch maps to tile row ch_row(first, t, n_band, bord0), first = k + 1 (or
// k + 2 for the bulk of the look-ahead schedule).  A dense matrix is the special case n_band = all rows, no border rows.
__device__ __forceinline__ int ch_row(int first, int t, int n_band, int bord0) { return t < n_band ? first + t : bord0 + (t - n_band); }
#define CH_KH 32               // the 64-deep inner product in two halves: 34 KB of shared memory per CTA instead of 67 KB
#define CH_HLD (CH_KH + 1)
#define CH_UPD_SMEM ((size_t)2 * CH_NB * CH_HLD * 8)
__global__ void __launch_bounds__(256, 4)
k_chol_update(int n, double *__restrict__ A, const double *__restrict__ Bsub, int k, int kmap, int single_col, int n_band, int bord0,
              const LmState *st, int gate) {
  if (!gate_open(st, gate) || st->lin_fail) return;
  extern __shared__ double sh[];
  double *As = sh, *Bs = sh + CH_NB * CH_HLD;
  // triangular decode: b = ti (ti + 1) / 2 + tj
  const int b = blockIdx.x;
  int ti = Bsub ? b + 1 : b, tj = 0;
  if (!single_col) {
    ti = (int)((sqrt(8.0 * (double)b + 1.0) - 1.0) * 0.5);
    while ((ti + 1) * (ti + 2) / 2 <= b) ++ti;
    while (ti * (ti + 1) / 2 > b) --ti;
    tj = b - ti * (ti + 1) / 2;
  }
  const int i0 = ch_row(kmap + 1, ti, n_band, bord0) * CH_NB, c0 = ch_row(kmap + 1, tj, n_band, bord0) * CH_NB, j0 = k * CH_NB;
  const int kk = min(CH_NB, n - j0);
  const int tid = threadIdx.x;
  const int ty = tid >> 4, tx = tid & 15;
  double acc[4][4];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[r][c] = 0.0;
  for (int h = 0; h < CH_NB / CH_KH; ++h) {
    if (h) __syncthreads();
    for (int idx = tid; idx < CH_NB * CH_KH; idx += 256) {
      const int r = idx >> 5, c = (idx & 31) + h * CH_KH;
      As[r * CH_HLD + (idx & 31)] = (i0 + r < n && c < kk) ? A[(size_t)(i0 + r) * n + j0 + c] : 0.0;
      Bs[r * CH_HLD + (idx & 31)] = Bsub ? Bsub[r * CH_NB + c] : ((c0 + r < n && c < kk) ? A[(size_t)(c0 + r) * n + j0 + c] : 0.0);
    }
    __syncthreads();
    for (int q = 0; q < CH_KH; ++q) {  // q ascending over both halves: the same sum per entry as one 64-deep pass
      double a[4], bb[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) a[r] = As[(ty * 4 + r) * CH_HLD + q];
#pragma unroll
      for (int c = 0; c < 4; ++c) bb[c] = Bs[(tx + 16 * c) * CH_HLD + q];  // columns tx, tx+16, ..: 16 distinct banks (odd stride)
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[r][c] += a[r] * bb[c];
    }
  }
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int row = i0 + ty * 4 + r;
    if (row >= n) continue;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int col = c0 + tx + 16 * c;
      if (col < n && col <= row) A[(size_t)row * n + col] -= acc[r][c];
    }
  }
}

// (Measured and rejected: a 128 x 128 super-tile version of this kernel -- 512 threads, 8 x 4 outputs each, every panel
// tile loaded half as often, 12 instead of 16 shared-memory loads per 32 multiply-adds.  Alone it is faster per tile, but
// its 133 KB CTAs fill an SM for their whole run, so the CTAs of the look-ahead chain (diagonal tile, panel, next column)
// wait for one to drain: 800-keyframe REF step 7.23 ms against 6.43 ms with the 64 x 64 tiles, three CTAs per SM.
// Also rejected: 128 threads with 8 x 4 outputs and both operand tiles transposed in shared memory (LDS.128 operands, 5 instead
// of 8 shared-memory wavefronts per warp and inner-product step): 7.10 ms against 6.18 ms -- with 12 instead of 24 warps per
// SM the kernel is bound by latency, not by the LSU / fp64 pipes.)

// =====================================================================
// Windowed problems (n <= BA_LDLT_MAX_N): the whole reduced-system solve in ONE CTA with the matrix in
// shared memory.  A = L D L^T, right-looking, no square roots:
//   * the right-hand side rides along as row n of the matrix, so the forward substitution L w = b is
//     part of the elimination (row n ends up holding w);
//   * column j is only READ during step j (trailing entries take  A_ik -= (A_ij / d_j) A_kj), so one
//     barrier per column suffices; every thread forms 1/d_j itself from the shared pivot;
//   * leading dimension odd: the strided column reads A_kj are bank-conflict free for 8-byte words;
//   * the back substitution L^T y = D^-1 w runs in warp 0 with register-resident w (lane l owns rows
//     l, l+32, ...) and one shuffle broadcast per unknown instead of a CTA barrier.
// The critical path per column is barrier + 1/d + one fused multiply-add (about 250 cycles) instead of a
// j-long dependent FMA chain, a square root and two barriers (the removed single-CTA column Cholesky: 135 us at n = 118).
// Every sum has a fixed order.  == the exact step of Ceres DENSE_SCHUR / SPARSE_SCHUR.
// =====================================================================
#define BA_LDLT_MAX_N 160
#define BA_LDLT_SLOTS (BA_LDLT_MAX_N / 32)
static_assert(BA_LDLT_MAX_N <= 160, "k_ldlt_solve: phases cover at most 5 row tiles");
__host__ __device__ inline int ldlt_ld(int n) { return n | 1; }
__host__ __device__ inline size_t ldlt_smem_bytes(int n) { return ((size_t)(n + 1) * ldlt_ld(n) + 2 * (size_t)(n + 8)) * 8; }

// One elimination step with NT = ceil((n - j) / 32) row tiles (compile-time: the j loop is split into phases).
// The trailing update is a grid of 32 x 32 tiles, row = warp, column = lane: tile (ti, tk) holds entry
// (i, k) = (j + 1 + warp + 32 ti, j + 1 + lane + 32 tk); tk < ti, and tk == ti for lane <= warp, lie in the lower
// triangle.  Only the last tile row / column can leave the matrix: its loads go to a clamped (valid) address and
// its stores are predicated.  All loads of a step are issued before the first multiply-add (the compiler cannot
// move the column reads across the trailing stores itself: same array).
template <int NT>
__device__ __forceinline__ void ldlt_step(double *__restrict__ A, double *__restrict__ invd, int ld, int n, int j, int warp,
                                          int lane, double rd) {
  const int i0 = j + 1 + warp, k0 = j + 1 + lane;
  const int base = i0 * ld + k0;                 // entry (i0, k0)
  const int cbi = base - lane - 1;               // (i0, j)
  const int cbk = k0 * ld + j;                   // (k0, j)
  const int ld32 = 32 * ld;
  const bool row_ok = i0 + 32 * (NT - 1) <= n;   // last tile row inside the matrix (rows .. n)
  const bool col_ok = k0 + 32 * (NT - 1) < n;    // last tile column inside the matrix (columns .. n-1)
  double li[NT], ck[NT], a[NT * (NT + 1) / 2];
#pragma unroll
  for (int t = 0; t < NT; ++t) {
    li[t] = (t < NT - 1 || row_ok) ? A[cbi + t * ld32] : 0.0;
    ck[t] = (t < NT - 1 || col_ok) ? A[cbk + t * ld32] : 0.0;
  }
#pragma unroll
  for (int ti = 0, u = 0; ti < NT; ++ti)
#pragma unroll
    for (int tk = 0; tk <= ti; ++tk, ++u)
      a[u] = ((ti < NT - 1 || row_ok) && (tk < NT - 1 || col_ok)) ? A[base + ti * ld32 + tk * 32] : 0.0;
#pragma unroll
  for (int ti = 0, u = 0; ti < NT; ++ti) {
    const double l = li[ti] * rd;
#pragma unroll
    for (int tk = 0; tk <= ti; ++tk, ++u) {
      const double v = a[u] - l * ck[tk];
      bool ok = true;
      if (ti == NT - 1) ok = ok && row_ok;
      if (tk == NT - 1) ok = ok && col_ok;
      if (tk == ti) ok = ok && lane <= warp;
      if (ok) A[base + ti * ld32 + tk * 32] = v;
      // the owner of the next pivot (entry (j+1, j+1)) publishes its reciprocal: nobody else needs to form it.
      // -1 marks a non-positive pivot; +inf gives 0 and NaN stays NaN, both fail the "> 0" test of the next step
      if (ti == 0 && tk == 0 && (warp | lane) == 0 && j + 1 < n) invd[j + 1] = v > 0.0 ? __drcp_rn(v) : -1.0;
    }
  }
}

__global__ void __launch_bounds__(1024)
k_ldlt_solve(int n, const double *__restrict__ Sg, const double *__restrict__ rhs, int n_cam, int n_free,
             const int32_t *__restrict__ cam_slot, int nk, double *__restrict__ yc, double *__restrict__ yk, LmState *st,
             int gate) {
  if (!gate_open(st, gate)) return;
  if (st->lin_fail) return;
  extern __shared__ double smd[];
  const int ld = ldlt_ld(n);
  double *A = smd;                           // (n + 1) x ld, lower triangle; row n = right-hand side
  double *invd = smd + (size_t)(n + 1) * ld;  // n + 8
  double *ysh = invd + n + 8;                 // n + 8
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;  // launched with exactly 32 warps
  for (int i = warp; i < n; i += 32)
    for (int k = lane; k <= i; k += 32) A[i * ld + k] = Sg[(size_t)i * n + k];
  for (int k = tid; k < n; k += 1024) A[n * ld + k] = rhs[k];
  if (tid == 0) {
    const double d = A[0];  // written by this thread
    invd[0] = d > 0.0 ? __drcp_rn(d) : -1.0;
  }
  bool bad = false;
  int j = 0;
#define BA_LDLT_PHASE(NT)                                                  \
  for (; !bad && j < n && ((n - j + 31) >> 5) == NT; ++j) {                \
    __syncthreads();                                                       \
    const double rd = invd[j];                                             \
    if (!(rd > 0.0)) { /* same value in every thread: uniform exit */      \
      bad = true;                                                          \
      break;                                                               \
    }                                                                      \
    ldlt_step<NT>(A, invd, ld, n, j, warp, lane, rd);                      \
  }
  BA_LDLT_PHASE(5)
  BA_LDLT_PHASE(4)
  BA_LDLT_PHASE(3)
  BA_LDLT_PHASE(2)
  BA_LDLT_PHASE(1)
#undef BA_LDLT_PHASE
  if (bad) {
    if (tid == 0) st->lin_fail = 1;
    return;
  }
  __syncthreads();
  if (warp == 0) {
    double w[BA_LDLT_SLOTS], iv[BA_LDLT_SLOTS];
#pragma unroll
    for (int s = 0; s < BA_LDLT_SLOTS; ++s) {
      const int i = lane + 32 * s;
      w[s] = i < n ? A[n * ld + i] : 0.0;
      iv[s] = i < n ? invd[i] : 0.0;
    }
#pragma unroll
    for (int s = BA_LDLT_SLOTS - 1; s >= 0; --s) {
      if (32 * s >= n) continue;
#pragma unroll 4
      for (int kk = 31; kk >= 0; --kk) {
        const int k = 32 * s + kk;
        if (k >= n) continue;
        const double y = __shfl_sync(0xffffffffu, w[s] * iv[s], kk);
        const double *Ak = A + k * ld;
        if (lane == kk) ysh[k] = y;
        if (lane < kk) w[s] -= Ak[32 * s + lane] * y;
#pragma unroll
        for (int s2 = 0; s2 < BA_LDLT_SLOTS; ++s2)
          if (s2 < s) w[s2] -= Ak[32 * s2 + lane] * y;
      }
    }
  }
  __syncthreads();
  for (int c = tid; c < n_cam; c += blockDim.x) {
    const int slot = cam_slot[c];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      const double v = slot >= 0 ? ysh[6 * slot + k] : 0.0;
      if (!isfinite(v)) st->lin_fail = 1;
      yc[6 * (size_t)c + k] = v;
    }
  }
  if (tid < 4) yk[tid] = nk ? ysh[6 * n_free + tid] : 0.0;
}

// =====================================================================
// Register-resident variant (the one in force).  k_ldlt_solve above keeps the trailing matrix in shared memory
// and is bound by shared-memory bandwidth (n^3/6 entries loaded and stored once each: 58 of its 67 us at n = 118).
// Here every thread OWNS the entries (i, k) = (warp + 32 ti, lane + 32 tk), tk <= ti, in registers for the whole
// factorisation (NT (NT + 1) / 2 <= 15 doubles); only the pivot column travels through shared memory:
//   step j:  barrier; read column j (c_k by lane, c_i by warp: broadcast) and 1 / d_j; a_ik -= (c_i / d_j) c_k on
//            the live tiles (tile columns >= j / 32: compile-time phases); the owners of column j + 1 (lane ==
//            (j + 1) % 32) store it to its permanent slot C[(j + 1) ldc + i], the owner of the next pivot also
//            stores its reciprocal.
// No predicates in the update: entries of finished rows / columns and of the upper halves of the diagonal tiles
// keep being "updated" with whatever the finished part of the column slot holds -- they are never read again.
// The stored columns C are L D (column-major, ldc odd: the row-wise reads of the back substitution are
// bank-conflict free); row n carries the right-hand side, so C[j ldc + n] = w_j (L w = b) at the end.
// =====================================================================
// (Measured and rejected: replacing the CTA barrier of a step by a split arrive / wait on a shared-memory mbarrier, so that
// column j + 1 is published before the bulk of the update with column j -- bit-identical factor, but slower: cfg 2
// 8,003 -> 7,695 LM it/s with 1,024 pollers, 4,723 with one poller per warp + __syncwarp; bar.sync is cheaper than the
// mbarrier round trip it would hide.)
#define BA_LDLT2_MAX_N 159
__host__ __device__ inline int ldlt2_ldc(int n) { return (n + 1) | 1; }
__host__ __device__ inline int ldlt2_tiles(int n) { return (n + 1 + 31) / 32; }
__host__ __device__ inline size_t ldlt2_smem_bytes(int n) {
  return ((size_t)n * ldlt2_ldc(n) + 32 * ldlt2_tiles(n) + 2 * (size_t)(n + 8)) * 8;
}
#define LDLT2_IDX(ti, tk) ((ti) * ((ti) + 1) / 2 + (tk))

template <int NT, int P, int PUB>
__device__ __forceinline__ bool ldlt2_step(double (&a)[NT * (NT + 1) / 2], double *__restrict__ C, double *__restrict__ invd,
                                           int ldc, int n, int nrows, int j, int warp, int lane) {
  __syncthreads();
  const double *cj = C + j * ldc;
  const double rd = invd[j];
  if (!(rd > 0.0)) return false;  // -1: non-positive pivot, 0: infinite pivot, NaN; the same value in every thread
  double ck[NT];
#pragma unroll
  for (int t = P; t < NT; ++t) ck[t] = cj[lane + 32 * t];
#pragma unroll
  for (int ti = P; ti < NT; ++ti) {
    const double l = cj[warp + 32 * ti] * rd;
#pragma unroll
    for (int tk = P; tk <= ti; ++tk) a[LDLT2_IDX(ti, tk)] -= l * ck[tk];
  }
  const int jn = j + 1;
  if (jn < n && lane == (jn & 31)) {  // this lane owns column jn in every warp
    double *cn = C + jn * ldc;
#pragma unroll
    for (int ti = PUB; ti < NT; ++ti) {
      const int i = warp + 32 * ti;
      if (i >= jn && i < nrows) cn[i] = a[LDLT2_IDX(ti, PUB)];  // nrows = n + 1 (solve) or n + m (potrf: identity rows)
    }
    if (warp == lane) {
      const double d = a[LDLT2_IDX(PUB, PUB)];
      invd[jn] = d > 0.0 ? __drcp_rn(d) : -1.0;
    }
  }
  return true;
}

template <int NT, int P>
__device__ __forceinline__ bool ldlt2_phase(double (&a)[NT * (NT + 1) / 2], double *__restrict__ C, double *__restrict__ invd,
                                            int ldc, int n, int nrows, int warp, int lane) {
  if constexpr (P < NT) {
    const int jend = min(32 * P + 31, n);
    for (int j = 32 * P; j < jend; ++j)
      if (!ldlt2_step<NT, P, P>(a, C, invd, ldc, n, nrows, j, warp, lane)) return false;
    if (32 * P + 31 < n)  // the last column of the tile column publishes into the next one
      if (!ldlt2_step<NT, P, (P + 1 < NT ? P + 1 : P)>(a, C, invd, ldc, n, nrows, 32 * P + 31, warp, lane)) return false;
    return ldlt2_phase<NT, P + 1>(a, C, invd, ldc, n, nrows, warp, lane);
  } else {
    return true;
  }
}

template <int NT>
__global__ void __launch_bounds__(1024)
k_ldlt2_solve(int n, const double *__restrict__ Sg, const double *__restrict__ rhs, int n_cam, int n_free,
              const int32_t *__restrict__ cam_slot, int nk, double *__restrict__ yc, double *__restrict__ yk, LmState *st,
              int gate) {
  if (!gate_open(st, gate)) return;
  if (st->lin_fail) return;
  extern __shared__ double smd[];
  const int ldc = ldlt2_ldc(n);
  double *C = smd;                                      // n columns of ldc (+ 32 NT: reads of the last tile row)
  double *invd = smd + (size_t)n * ldc + 32 * NT;       // n + 8
  double *ysh = invd + n + 8;                           // n + 8
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;  // launched with exactly 32 warps
  double a[NT * (NT + 1) / 2];
#pragma unroll
  for (int ti = 0; ti < NT; ++ti)
#pragma unroll
    for (int tk = 0; tk <= ti; ++tk) {
      const int i = warp + 32 * ti, k = lane + 32 * tk;
      double v = 0.0;
      if (k < n) {
        if (i < n) v = Sg[(size_t)i * n + k];
        else if (i == n) v = rhs[k];
      }
      a[LDLT2_IDX(ti, tk)] = v;
    }
  if (lane == 0) {  // column 0
#pragma unroll
    for (int ti = 0; ti < NT; ++ti) {
      const int i = warp + 32 * ti;
      if (i <= n) C[i] = a[LDLT2_IDX(ti, 0)];
    }
    if (warp == 0) invd[0] = a[0] > 0.0 ? __drcp_rn(a[0]) : -1.0;
  }
  const bool ok = ldlt2_phase<NT, 0>(a, C, invd, ldc, n, n + 1, warp, lane);
  if (!ok) {
    if (tid == 0) st->lin_fail = 1;
    return;
  }
  __syncthreads();
  if (warp == 0) {
    // L^T y = D^-1 w: lane l owns rows l + 32 s; y_k broadcast by shuffle, c_ki = C[i ldc + k]
    double w[NT], iv[NT];
#pragma unroll
    for (int s = 0; s < NT; ++s) {
      const int i = lane + 32 * s;
      w[s] = i < n ? C[i * ldc + n] : 0.0;
      iv[s] = i < n ? invd[i] : 0.0;
    }
#pragma unroll
    for (int s = NT - 1; s >= 0; --s) {
      if (32 * s >= n) continue;
#pragma unroll 4
      for (int kk = 31; kk >= 0; --kk) {
        const int k = 32 * s + kk;
        if (k >= n) continue;
        const double y = __shfl_sync(0xffffffffu, w[s] * iv[s], kk);
        if (lane == kk) ysh[k] = y;
        if (lane < kk) w[s] -= C[(32 * s + lane) * ldc + k] * y;
#pragma unroll
        for (int s2 = 0; s2 < NT; ++s2)
          if (s2 < s) w[s2] -= C[(32 * s2 + lane) * ldc + k] * y;
      }
    }
  }
  __syncthreads();
  for (int c = tid; c < n_cam; c += 1024) {
    const int slot = cam_slot[c];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      const double v = slot >= 0 ? ysh[6 * slot + k] : 0.0;
      if (!isfinite(v)) st->lin_fail = 1;
      yc[6 * (size_t)c + k] = v;
    }
  }
  if (tid < 4) yk[tid] = nk ? ysh[6 * n_free + tid] : 0.0;
}


// =====================================================================
// Diagonal tile and panel of the blocked factorisation, second version (in force):
//  * k_chol_potrf2: the register-resident L D L^T above applied to the m x m diagonal tile (m <= 64) with m extra
//    rows holding the identity: row m + r ends up as column r of the unit factor's inverse, so the kernel writes
//    both the Cholesky factor L = Lu D^1/2 (back into A) and L^-1 = D^-1/2 Lu^-1 (into Linv, dense 64 x 64, zeros above
//    the diagonal) in ~64 barrier steps.  The removed left-looking version (one thread per row): 45 us per tile.
//  * k_chol_trsm2: the panel X = A_ik L^-T as a 64 x 64 x 64 product with L^-1 (256 threads, 4 x 4 outputs each)
//    instead of one thread per row walking a 64-step substitution with j-long dependent chains (63 us per launch).
// =====================================================================
#define CH_P2_LDC 129
// fuse != 0 (look-ahead schedule, k > 0): the kernel first brings its own diagonal tile up to date, so that the chain
// diagonal tile k - 1 -> diagonal tile k has no other kernel in it:
//   L_{k,k-1} = A_{k,k-1} L_{k-1,k-1}^-T   (A_{k,k-1} is still the un-solved tile: k_chol_trsm2 writes this panel tile to a side
//                                          buffer, never in place, so nothing overwrites what this kernel reads)
//   D = A_kk - L_{k,k-1} L_{k,k-1}^T       (the update k_chol_update would have applied)
// with the same operation order per entry as k_chol_trsm2 / k_chol_update (sums over q ascending from zero), i.e. the same bits.
__host__ __device__ inline size_t chol_potrf2_smem_bytes() {
  return ((size_t)CH_NB * CH_P2_LDC + 128 + 2 * (CH_NB + 8) + 2 * CH_NB * CH_LD) * 8;
}

__global__ void __launch_bounds__(1024)
k_chol_potrf2(int n, double *__restrict__ A, double *__restrict__ Linv, int k, int fuse, LmState *st, int gate) {
  if (!gate_open(st, gate) || st->lin_fail) return;
  constexpr int NT = 4;
  extern __shared__ double smd[];
  double *C = smd;                                   // m columns of CH_P2_LDC (+ 128: reads of the last tile rows)
  double *invd = smd + (size_t)CH_NB * CH_P2_LDC + 128;
  double *Xs = invd + 2 * (CH_NB + 8);               // fused prologue: A_{k,k-1}, then L_{k,k-1}
  double *Ds = Xs + CH_NB * CH_LD;                   // fused prologue: L_{k-1,k-1}^-1, then the updated diagonal tile
  const int j0 = k * CH_NB, m = min(CH_NB, n - j0);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool fused = fuse && k > 0;
  if (fused) {
    const int jp = j0 - CH_NB;
    const double *Lp = Linv - (size_t)CH_NB * CH_NB;  // L^-1 of the previous diagonal tile (Linv points at this tile's slot)
    for (int idx = tid; idx < CH_NB * CH_NB; idx += 1024) {
      const int r = idx >> 6, c = idx & 63;
      Xs[r * CH_LD + c] = r < m ? A[(size_t)(j0 + r) * n + jp + c] : 0.0;
      Ds[r * CH_LD + c] = Lp[idx];
    }
    __syncthreads();
    const int r = tid >> 4, cg = tid & 15;
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    for (int q = 0; q < CH_NB; ++q) {
      const double x = Xs[r * CH_LD + q];
#pragma unroll
      for (int cc = 0; cc < 4; ++cc) acc[cc] += x * Ds[(cg + 16 * cc) * CH_LD + q];
    }
    __syncthreads();
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) Xs[r * CH_LD + cg + 16 * cc] = acc[cc];
    __syncthreads();
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) acc[cc] = 0.0;
    for (int q = 0; q < CH_NB; ++q) {
      const double x = Xs[r * CH_LD + q];
#pragma unroll
      for (int cc = 0; cc < 4; ++cc) acc[cc] += x * Xs[(cg + 16 * cc) * CH_LD + q];
    }
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) {
      const int c = cg + 16 * cc;
      double d = 0.0;
      if (r < m && c <= r) {
        d = A[(size_t)(j0 + r) * n + j0 + c];
        d -= acc[cc];
      }
      Ds[r * CH_LD + c] = d;
    }
    __syncthreads();
  }
  double a[NT * (NT + 1) / 2];
#pragma unroll
  for (int ti = 0; ti < NT; ++ti)
#pragma unroll
    for (int tk = 0; tk <= ti; ++tk) {
      const int i = warp + 32 * ti, c = lane + 32 * tk;
      double v = 0.0;
      if (c < m) {
        if (i < m) {  // the lower triangle is current
          if (fused) v = c <= i ? Ds[i * CH_LD + c] : Ds[c * CH_LD + i];
          else v = c <= i ? A[(size_t)(j0 + i) * n + j0 + c] : A[(size_t)(j0 + c) * n + j0 + i];
        } else if (i - m == c) v = 1.0;
      }
      a[LDLT2_IDX(ti, tk)] = v;
    }
  if (lane == 0) {
#pragma unroll
    for (int ti = 0; ti < NT; ++ti) {
      const int i = warp + 32 * ti;
      if (i < 2 * m) C[i] = a[LDLT2_IDX(ti, 0)];
    }
    if (warp == 0) invd[0] = a[0] > 0.0 ? __drcp_rn(a[0]) : -1.0;
  }
  const bool ok = ldlt2_phase<NT, 0>(a, C, invd, CH_P2_LDC, m, 2 * m, warp, lane);
  if (!ok) {
    if (tid == 0) st->lin_fail = 1;
    return;
  }
  __syncthreads();
  for (int idx = tid; idx < CH_NB * CH_NB; idx += 1024) {
    const int i = idx >> 6, j = idx & 63;  // (row, column) of L resp. L^-1
    double li = 0.0;
    if (i < m && j < m && j <= i) {
      const double sj = sqrt(invd[j]);
      A[(size_t)(j0 + i) * n + j0 + j] = i == j ? 1.0 / sj : C[j * CH_P2_LDC + i] * sj;  // L_ij = c_ij / sqrt(d_j), L_jj = sqrt(d_j)
      li = C[i * CH_P2_LDC + m + j] * sqrt(invd[i]);  // (L^-1)_ij = (Lu^-1)_ij / sqrt(d_i); identity row m + j, column i
    }
    Linv[idx] = li;
  }
}

// Lsub != nullptr (look-ahead schedule): the tile right below the diagonal, (k + 1, k), goes to Lsub (dense 64 x 64) instead
// of in place -- the fused k_chol_potrf2 of step k + 1 reads the un-solved tile concurrently; k_chol_fixup stores it at the end.
__global__ void __launch_bounds__(256)
k_chol_trsm2(int n, double *__restrict__ A, const double *__restrict__ Linv, double *__restrict__ Lsub, int k, int n_band, int bord0,
             const LmState *st, int gate) {
  if (!gate_open(st, gate) || st->lin_fail) return;
  extern __shared__ double sh[];
  double *As = sh, *Bs = sh + CH_NB * CH_LD;
  const int j0 = k * CH_NB, kk = min(CH_NB, n - j0);
  const int i0 = ch_row(k + 1, blockIdx.x, n_band, bord0) * CH_NB;
  const int tid = threadIdx.x;
  for (int idx = tid; idx < CH_NB * CH_NB; idx += 256) {
    const int r = idx >> 6, c = idx & 63;
    As[r * CH_LD + c] = (i0 + r < n && c < kk) ? A[(size_t)(i0 + r) * n + j0 + c] : 0.0;
    Bs[r * CH_LD + c] = Linv[idx];  // row r of L^-1 (zero beyond the tile and above the diagonal)
  }
  __syncthreads();
  const int ty = tid >> 4, tx = tid & 15;
  double acc[4][4];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[r][c] = 0.0;
  for (int q = 0; q < CH_NB; ++q) {  // X[r][c] = sum_q A[r][q] Linv[c][q]
    double av[4], bb[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) av[r] = As[(ty * 4 + r) * CH_LD + q];
#pragma unroll
    for (int c = 0; c < 4; ++c) bb[c] = Bs[(tx + 16 * c) * CH_LD + q];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[r][c] += av[r] * bb[c];
  }
  if (Lsub && blockIdx.x == 0) {
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) Lsub[(ty * 4 + r) * CH_NB + tx + 16 * c] = acc[r][c];  // zero beyond the matrix
    return;
  }
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int row = i0 + ty * 4 + r;
    if (row >= n) continue;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int col = tx + 16 * c;
      if (col < kk) A[(size_t)row * n + j0 + col] = acc[r][c];
    }
  }
}

// look-ahead schedule: the panel tiles right below the diagonal, kept aside during the factorisation, into the matrix
__global__ void __launch_bounds__(256)
k_chol_fixup(int n, double *__restrict__ A, const double *__restrict__ Lsub, const LmState *st, int gate) {
  if (!gate_open(st, gate) || st->lin_fail) return;
  const int k = blockIdx.x + 1, j0 = k * CH_NB, jp = j0 - CH_NB;
  const double *L = Lsub + (size_t)k * CH_NB * CH_NB;
  for (int idx = threadIdx.x; idx < CH_NB * CH_NB; idx += 256) {
    const int r = idx >> 6, c = idx & 63;
    if (j0 + r < n) A[(size_t)(j0 + r) * n + jp + c] = L[idx];
  }
}

// =====================================================================
// Blocked substitution, second version (in force): L z = b, L^T y = z over the 64 x 64 tiles WITHOUT grid barriers
// and without a sequential triangular solve per diagonal tile.
//  * k_chol_potrf2 leaves L_kk^-1 of every diagonal tile (Linv + 4096 k), so a diagonal step is a 64 x 64 product:
//    z_k = L_kk^-1 v_k (forward), y_k = L_kk^-T v_k (backward).
//  * tile row (forward) / tile column (backward) t belongs to CTA t % gridDim.x for the whole pass; its running
//    right-hand side v_t never leaves that CTA's shared memory, so only the 64 solved values of a step travel:
//    published as 16-byte FLAG-IN-DATA slots {value, tag} with one vector store each and polled by the consumers
//    (no fence, no separate flag, no barrier: one L2 round trip per step).
//  * the owner of the NEXT diagonal tile applies the step to that tile first and publishes the next 64 values
//    before touching its other tiles; the tile it needs (and L^-1 of its diagonal tile) is already in registers
//    when the awaited values arrive (the loads are issued before the wait).
// Critical path per step: poll -> 64 x 64 product -> 64 x 64 product -> publish (about 3 us) instead of a tile load,
// 64 two-barrier substitution steps in one CTA and two grid barriers (33 us: 5.0 of the 13.2 ms of an exact LM step
// at n = 4798).  Every sum has a fixed order (per thread 16 products in two chains, then a fixed tree).
// Cooperative launch only for co-residency (consumers spin on producers); gridDim.x * CH_S2_OWN >= tile count.
// =====================================================================
#define CH_S2_OWN 4
struct __align__(16) ChSlot {
  double v;
  unsigned long long tag;
};
__device__ __forceinline__ void ch_publish(ChSlot *p, double v) {
  asm volatile("st.volatile.global.v2.u64 [%0], {%1, %2};" ::"l"(p), "l"(__double_as_longlong(v)), "l"(1ull) : "memory");
}
__device__ __forceinline__ double ch_wait(const ChSlot *p) {
  unsigned long long a, b;
  do {
    asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "l"(p) : "memory");
  } while (b != 1ull);
  return __longlong_as_double((long long)a);
}
// row layout: thread (r = tid >> 2, part = tid & 3) holds A[r0 + r][c0 + 4 q + part], q = 0..15 (a quarter-warp reads
// whole 32-byte sectors); column layout: thread (c = tid & 63, g = tid >> 6) holds A[r0 + g + 4 q][c0 + c]
__device__ __forceinline__ void ch_load_rows(const double *__restrict__ A, int ld, int nr, int nc, int r0, int c0, int tid,
                                             double (&reg)[16]) {
  const int r = r0 + (tid >> 2), part = tid & 3;
#pragma unroll
  for (int q = 0; q < 16; ++q) {
    const int c = c0 + 4 * q + part;
    reg[q] = (r < nr && c < nc) ? A[(size_t)r * ld + c] : 0.0;
  }
}
__device__ __forceinline__ void ch_load_cols(const double *__restrict__ A, int ld, int nr, int nc, int r0, int c0, int tid,
                                             double (&reg)[16]) {
  const int c = c0 + (tid & 63), g = tid >> 6;
#pragma unroll
  for (int q = 0; q < 16; ++q) {
    const int r = r0 + g + 4 * q;
    reg[q] = (r < nr && c < nc) ? A[(size_t)r * ld + c] : 0.0;
  }
}
// sum_c A[r][c] x[c] for the thread's row; identical in the four threads of a row
__device__ __forceinline__ double ch_dot_rows(const double (&reg)[16], const double *__restrict__ x, int tid) {
  const int part = tid & 3;
  double s0 = 0.0, s1 = 0.0;
#pragma unroll
  for (int q = 0; q < 16; q += 2) {
    s0 += reg[q] * x[4 * q + part];
    s1 += reg[q + 1] * x[4 * q + 4 + part];
  }
  double s = s0 + s1;
  s += __shfl_xor_sync(0xffffffffu, s, 1);
  s += __shfl_xor_sync(0xffffffffu, s, 2);
  return s;
}
// partial of sum_r A[r][c] x[r] over the thread's 16 rows -> red[g][c]; the caller adds the four groups in order
__device__ __forceinline__ void ch_dot_cols(const double (&reg)[16], const double *__restrict__ x, int tid, double *red) {
  const int g = tid >> 6;
  double s0 = 0.0, s1 = 0.0;
#pragma unroll
  for (int q = 0; q < 16; q += 2) {
    s0 += reg[q] * x[g + 4 * q];
    s1 += reg[q + 1] * x[g + 4 * q + 4];
  }
  red[g * CH_NB + (tid & 63)] = s0 + s1;
}

__global__ void __launch_bounds__(256)
k_chol_solve2(int n, const double *__restrict__ A, const double *__restrict__ Linv, const double *__restrict__ rhs,
              ChSlot *fwd, ChSlot *bwd /* [nt * 64] each, zeroed before the launch */, int n_cam, int n_free,
              const int32_t *__restrict__ cam_slot, int nk, double *__restrict__ yc, double *__restrict__ yk, LmState *st,
              int gate) {
  if (!gate_open(st, gate) || st->lin_fail) return;  // identical on every CTA
  __shared__ double vs[CH_S2_OWN][CH_NB];  // running right-hand side of the owned tiles, then their solved values
  __shared__ double xb[2][CH_NB];          // the solved values of step k (buffer k & 1)
  __shared__ double red[4 * CH_NB];
  const int tid = threadIdx.x, b = blockIdx.x, G = gridDim.x;
  const int nt = (n + CH_NB - 1) / CH_NB;
  double Lr[16], Ir[16];
  if (b < nt) {
    for (int idx = tid; idx < CH_S2_OWN * CH_NB; idx += 256) {
      const int t = b + (idx >> 6) * G, i = t * CH_NB + (idx & 63);
      vs[idx >> 6][idx & 63] = (t < nt && i < n) ? rhs[i] : 0.0;
    }
    __syncthreads();
    // ---------------- forward: L z = b
    if (b == 0) {  // z_0 = L_00^-1 v_0
      ch_load_rows(Linv, CH_NB, CH_NB, CH_NB, 0, 0, tid, Ir);
      const double z = ch_dot_rows(Ir, vs[0], tid);
      __syncthreads();
      if ((tid & 3) == 0) {
        vs[0][tid >> 2] = z;
        xb[0][tid >> 2] = z;
        ch_publish(fwd + (tid >> 2), z);
      }
      __syncthreads();
    }
    for (int k = 0; k + 1 < nt; ++k) {
      // first owned tile row below k
      int i = k + 1 <= b ? b : b + ((k + 1 - b + G - 1) / G) * G;
      if (i >= nt) break;  // no tile rows left below k: this CTA's part of the pass is done
      const bool diag_next = i == k + 1;
      ch_load_rows(A, n, n, n, i * CH_NB, k * CH_NB, tid, Lr);
      if (diag_next) ch_load_rows(Linv + (size_t)i * CH_NB * CH_NB, CH_NB, CH_NB, CH_NB, 0, 0, tid, Ir);
      double *x = xb[k & 1];
      if (k % G != b && tid < CH_NB) x[tid] = ch_wait(fwd + k * CH_NB + tid);
      __syncthreads();
      for (; i < nt; i += G) {
        const int slot = (i - b) / G;
        const double s = ch_dot_rows(Lr, x, tid);
        if ((tid & 3) == 0) vs[slot][tid >> 2] -= s;
        if (i == k + 1) {  // the next diagonal tile is mine: solve it and publish before anything else
          __syncthreads();
          const double z = ch_dot_rows(Ir, vs[slot], tid);
          __syncthreads();
          if ((tid & 3) == 0) {
            vs[slot][tid >> 2] = z;
            xb[(k + 1) & 1][tid >> 2] = z;
            ch_publish(fwd + (k + 1) * CH_NB + (tid >> 2), z);
          }
        }
        if (i + G < nt) ch_load_rows(A, n, n, n, (i + G) * CH_NB, k * CH_NB, tid, Lr);
      }
      __syncthreads();
    }
    // ---------------- backward: L^T y = z (vs holds z of the owned tiles)
    if ((nt - 1) % G == b) {
      const int slot = (nt - 1 - b) / G;
      ch_load_cols(Linv + (size_t)(nt - 1) * CH_NB * CH_NB, CH_NB, CH_NB, CH_NB, 0, 0, tid, Ir);
      ch_dot_cols(Ir, vs[slot], tid, red);
      __syncthreads();
      if (tid < CH_NB) {
        const double y = ((red[tid] + red[CH_NB + tid]) + red[2 * CH_NB + tid]) + red[3 * CH_NB + tid];
        vs[slot][tid] = y;
        xb[(nt - 1) & 1][tid] = y;
        ch_publish(bwd + (nt - 1) * CH_NB + tid, y);
      }
      __syncthreads();
    }
    for (int i = nt - 1; i >= 1; --i) {
      // last owned tile column left of i
      int k = -1;
      if (b <= i - 1) k = b + ((i - 1 - b) / G) * G;
      if (k < 0) break;  // no tile columns left of i
      const bool diag_next = k == i - 1;
      ch_load_cols(A, n, n, n, i * CH_NB, k * CH_NB, tid, Lr);
      if (diag_next) ch_load_cols(Linv + (size_t)k * CH_NB * CH_NB, CH_NB, CH_NB, CH_NB, 0, 0, tid, Ir);
      double *x = xb[i & 1];
      if (i % G != b && tid < CH_NB) x[tid] = ch_wait(bwd + i * CH_NB + tid);
      __syncthreads();
      for (; k >= 0; k -= G) {
        const int slot = (k - b) / G;
        ch_dot_cols(Lr, x, tid, red);
        __syncthreads();
        if (tid < CH_NB) vs[slot][tid] -= ((red[tid] + red[CH_NB + tid]) + red[2 * CH_NB + tid]) + red[3 * CH_NB + tid];
        __syncthreads();
        if (k == i - 1) {
          ch_dot_cols(Ir, vs[slot], tid, red);
          __syncthreads();
          if (tid < CH_NB) {
            const double y = ((red[tid] + red[CH_NB + tid]) + red[2 * CH_NB + tid]) + red[3 * CH_NB + tid];
            vs[slot][tid] = y;
            xb[(i - 1) & 1][tid] = y;
            ch_publish(bwd + (i - 1) * CH_NB + tid, y);
          }
          __syncthreads();
        }
        if (k - G >= 0) ch_load_cols(A, n, n, n, i * CH_NB, (k - G) * CH_NB, tid, Lr);
      }
      __syncthreads();
    }
  }
  // ---------------- scatter (every CTA; a value is read when its tag has arrived)
  const int gtid = b * 256 + tid, nthr = G * 256;
  for (int c = gtid; c < n_cam; c += nthr) {
    const int slot = cam_slot[c];
#pragma unroll
    for (int q = 0; q < 6; ++q) {
      const double x = slot >= 0 ? ch_wait(bwd + 6 * slot + q) : 0.0;
      if (!isfinite(x)) st->lin_fail = 1;
      yc[6 * (size_t)c + q] = x;
    }
  }
  if (gtid < 4) yk[gtid] = nk ? ch_wait(bwd + 6 * n_free + gtid) : 0.0;
}
