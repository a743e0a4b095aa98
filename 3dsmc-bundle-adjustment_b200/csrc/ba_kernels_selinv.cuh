// ba_kernels_selinv.cuh -- covariance of the estimate (ba_gpu_covariance): the inverse of the undamped Gauss-Newton Hessian
// on the pattern of the sparse Cholesky factor, by SELECTED INVERSION over the supernodal tree of ba_kernels_spchol.cuh.
//
// Reduced system [[A, B], [B^T, C]] (A = L L^T over the free cameras, B the 6 x 4 camera-intrinsics border, C the 4 x 4
// corner), factorised by the same tree as an LM step with zero damping.  Per node (own cameras O, border cameras Bd; the
// panel holds L_OO and L_BO), top-down, parents before children (Takahashi recurrence):
//     Y    = L_BO L_OO^-1
//     S_BO = -S_BB Y                         (S_BB gathered from the parent's front through `rel`, the reverse of extend-add)
//     S_OO = L_OO^-T L_OO^-1 - Y^T S_BO
// where S denotes A^-1.  The Sigma front of a node is written over its own factor storage: S_OO and S_BO into the panel
// (same layout), S_BB into the update-matrix slot (dense NB6 x NB6, full).  No L of a node is read after its own inversion
// (the children read only their own panels and the parent's Sigma front), and the next solve re-factorises.
// Y goes to a panel-shaped scratch buffer (border rows only).
// Intrinsics border: X = A^-1 B = L^-T Z (backward substitution, one column at a time, k_spchol_solve), T = C - Z^T Z,
//     Sigma_kk = T^-1,  Sigma_ck = -X T^-1,  Sigma_cc(a, b) = (A^-1)_ab + X_a T^-1 X_b^T.
// Points: Sigma_pp = V^-1 + V^-1 (W_p^T Sigma_RR W_p) V^-1 over the observation pairs of the point.
// Everything is Jacobi-scaled on the device; the outputs are unscaled (Sigma = diag(s) Sigma_s diag(s)).
// Every sum has a fixed order and no float atomics are used: the results are bit-identical from run to run.
#pragma once
#include "ba_kernels_spchol.cuh"

struct SelInv {
  const int32_t *node, *rel;
  const double *linv;  // inverse pivot blocks by elimination position [36 n_cam] (row-major 6 x 6, lower)
  double *panel, *U;   // factor panels / update-matrix slots on entry; Sigma fronts on exit
  double *Y;           // Y = L_BO L_OO^-1: border rows of a panel-shaped buffer
  const int2 *queue;   // (node, kind): kind >= 0 product tile, -1 prepare, -3 finish
  int n_items;
  const int32_t *tiles;
  int *ticket, *pdone, *tdone, *sdone;
};
inline size_t si_smem(int m, int nb) {
  const size_t C6 = 6 * (size_t)m, NB6 = 6 * (size_t)nb;
  return std::max(C6 * C6 + 6 * C6, NB6 * C6) * 8 + 64;
}

// element (R, Cc) (local scalar row / column in the node's (own, border) list) of a finished Sigma front
__device__ __forceinline__ double si_front(const double *Pp, const double *Up, int LD, int C6, int NB6, int R, int Cc) {
  if (Cc < C6) return __ldcg(Pp + (size_t)Cc * LD + R);
  if (R < C6) return __ldcg(Pp + (size_t)R * LD + Cc);
  return __ldcg(Up + (size_t)(Cc - C6) * NB6 + (R - C6));
}

// prepare(node): L_OO^-1 in shared memory, S_OO <- L_OO^-T L_OO^-1 (into the panel's own rows), Y = L_BO L_OO^-1, then --
// after the parent's Sigma front is complete -- S_BB gathered into the update-matrix slot
__device__ __forceinline__ void si_prepare(const SelInv &a, int id, double *sm) {
  const int tid = threadIdx.x;
  const int32_t *N = a.node + (size_t)id * SPSYM_NODE_INTS;
  const int k0 = N[SPN_K0], m = N[SPN_M], nb = N[SPN_NB];
  const int LD = 6 * (m + nb), C6 = 6 * m, NB6 = 6 * nb;
  double *Pg = a.panel + 36 * spc_off(N, SPN_PANEL_LO);
  double *Ls = sm;                   // L_OO, column-major C6 x C6; becomes L_OO^-1 column block by column block
  double *G = Ls + (size_t)C6 * C6;  // C6 x 6 partial products of the current column block
  for (int idx = tid; idx < C6 * C6; idx += SPC_THREADS) {
    const int c = idx / C6, r = idx - c * C6;
    Ls[idx] = r >= c ? __ldcg(Pg + (size_t)c * LD + r) : 0.0;
  }
  __syncthreads();
  // L^-1 in place, block columns right to left: Linv_ij = -(sum_{k=j+1..i} Linv_ik L_kj) T_j, Linv_jj = T_j
  for (int j = m - 1; j >= 0; --j) {
    const int r0 = 6 * (j + 1), nr = C6 - r0;
    for (int idx = tid; idx < 6 * nr; idx += SPC_THREADS) {
      const int cc = idx / nr, R = r0 + (idx - cc * nr);
      double s = 0.0;
      for (int K = r0; K <= R; ++K) s += Ls[(size_t)K * C6 + R] * Ls[(size_t)(6 * j + cc) * C6 + K];
      G[(size_t)cc * C6 + R] = s;
    }
    __syncthreads();
    const double *T = a.linv + 36 * (size_t)(k0 + j);
    for (int idx = tid; idx < 6 * nr; idx += SPC_THREADS) {
      const int cc = idx / nr, R = r0 + (idx - cc * nr);
      double s = 0.0;
#pragma unroll
      for (int c2 = 0; c2 < 6; ++c2) s += G[(size_t)c2 * C6 + R] * __ldcg(T + c2 * 6 + cc);
      Ls[(size_t)(6 * j + cc) * C6 + R] = -s;
    }
    if (tid < 36) {
      const int r = tid / 6, c = tid - 6 * r;
      Ls[(size_t)(6 * j + c) * C6 + 6 * j + r] = __ldcg(T + tid);
    }
    __syncthreads();
  }
  // S_OO <- Linv^T Linv (lower triangle computed, both written: exactly symmetric)
  for (int idx = tid; idx < C6 * C6; idx += SPC_THREADS) {
    const int b = idx / C6, r = idx - b * C6;
    if (r < b) continue;
    double s = 0.0;
    for (int K = r; K < C6; ++K) s += Ls[(size_t)r * C6 + K] * Ls[(size_t)b * C6 + K];
    Pg[(size_t)b * LD + r] = s;
    Pg[(size_t)r * LD + b] = s;
  }
  // Y = L_BO Linv: Y[r][c] = sum_{K >= c} L_BO[r][K] Linv[K][c]
  double *Yg = a.Y + 36 * spc_off(N, SPN_PANEL_LO);
  for (int idx = tid; idx < NB6 * C6; idx += SPC_THREADS) {
    const int c = idx / NB6, r = idx - c * NB6;
    double s = 0.0;
    for (int K = c; K < C6; ++K) s += __ldcg(Pg + (size_t)K * LD + C6 + r) * Ls[(size_t)c * C6 + K];
    Yg[(size_t)c * LD + C6 + r] = s;
  }
  if (nb == 0) return;
  const int par = N[SPN_PARENT];
  if (tid == 0) spc_wait_ge(a.sdone + par, 1);
  __syncthreads();
  const int32_t *Pn = a.node + (size_t)par * SPSYM_NODE_INTS;
  const int pC6 = 6 * Pn[SPN_M], pNB6 = 6 * Pn[SPN_NB], pLD = pC6 + pNB6;
  const double *Pp = a.panel + 36 * spc_off(Pn, SPN_PANEL_LO), *Up = a.U + 36 * spc_off(Pn, SPN_U_LO);
  const int32_t *rel = a.rel + N[SPN_REL];
  double *Ug = a.U + 36 * spc_off(N, SPN_U_LO);
  for (int idx = tid; idx < NB6 * NB6; idx += SPC_THREADS) {
    const int col = idx / NB6, row = idx - col * NB6;
    const int i = row / 6, j = col / 6;
    Ug[idx] = si_front(Pp, Up, pLD, pC6, pNB6, 6 * __ldg(rel + i) + row - 6 * i, 6 * __ldg(rel + j) + col - 6 * j);
  }
}

// tile `tile` of `tiles` of S_BO = -S_BB Y (3 x 6 output pieces, Y row-major in shared memory, S_BB read by columns:
// it is symmetric), into the panel's border rows
__device__ __forceinline__ void si_tile(const SelInv &a, int id, int tile, int tiles, double *sm) {
  const int tid = threadIdx.x;
  const int32_t *N = a.node + (size_t)id * SPSYM_NODE_INTS;
  const int m = N[SPN_M], nb = N[SPN_NB];
  const int LD = 6 * (m + nb), C6 = 6 * m, NB6 = 6 * nb;
  double *Pg = a.panel + 36 * spc_off(N, SPN_PANEL_LO);
  const double *Yg = a.Y + 36 * spc_off(N, SPN_PANEL_LO);
  const double *Ug = a.U + 36 * spc_off(N, SPN_U_LO);
  double *Ys = sm;  // Ys[k * C6 + c] = Y[k][c]
  for (int idx = tid; idx < NB6 * C6; idx += SPC_THREADS) {
    const int c = idx / NB6, k = idx - c * NB6;
    Ys[(size_t)k * C6 + c] = __ldcg(Yg + (size_t)c * LD + C6 + k);
  }
  __syncthreads();
  const int rg = NB6 / 3, n_pieces = rg * m;
  for (int p = tile * SPC_THREADS + tid; p < n_pieces; p += tiles * SPC_THREADS) {
    const int cbk = p / rg, ra = 3 * (p - cbk * rg), cb = 6 * cbk;
    double acc[3][6];
#pragma unroll
    for (int x = 0; x < 3; ++x)
#pragma unroll
      for (int y = 0; y < 6; ++y) acc[x][y] = 0.0;
    for (int k = 0; k < NB6; ++k) {
      const double *uc = Ug + (size_t)k * NB6 + ra;
      const double a0 = __ldcg(uc), a1 = __ldcg(uc + 1), a2 = __ldcg(uc + 2);
      const double *yr = Ys + (size_t)k * C6 + cb;
#pragma unroll
      for (int y = 0; y < 6; ++y) {
        const double bv = yr[y];
        acc[0][y] += a0 * bv;
        acc[1][y] += a1 * bv;
        acc[2][y] += a2 * bv;
      }
    }
#pragma unroll
    for (int y = 0; y < 6; ++y)
#pragma unroll
      for (int x = 0; x < 3; ++x) Pg[(size_t)(cb + y) * LD + C6 + ra + x] = -acc[x][y];
  }
}

// finish(node): S_OO -= Y^T S_BO (lower triangle computed, both written)
__device__ __forceinline__ void si_finish(const SelInv &a, int id) {
  const int tid = threadIdx.x;
  const int32_t *N = a.node + (size_t)id * SPSYM_NODE_INTS;
  const int m = N[SPN_M], nb = N[SPN_NB];
  if (nb == 0) return;
  const int LD = 6 * (m + nb), C6 = 6 * m, NB6 = 6 * nb;
  double *Pg = a.panel + 36 * spc_off(N, SPN_PANEL_LO);
  const double *Yg = a.Y + 36 * spc_off(N, SPN_PANEL_LO);
  for (int idx = tid; idx < C6 * C6; idx += SPC_THREADS) {
    const int b = idx / C6, r = idx - b * C6;
    if (r < b) continue;
    const double *yc = Yg + (size_t)r * LD + C6, *sc = Pg + (size_t)b * LD + C6;
    double s = 0.0;
    for (int k = 0; k < NB6; ++k) s += __ldcg(yc + k) * __ldcg(sc + k);
    const double v = __ldcg(Pg + (size_t)b * LD + r) - s;
    Pg[(size_t)b * LD + r] = v;
    Pg[(size_t)r * LD + b] = v;
  }
}

// The selected inversion in ONE persistent launch (the scheme of k_spchol_tree, top-down): a block takes the next item from a
// ticket counter and waits on integer completion counters:
//     prepare(n)  its own part (L_OO^-1, Y) at once; the gather of S_BB after finish(parent(n))
//     tile(n, t)  after prepare(n)
//     finish(n)   after prepare(n) and every tile of n
// The queue holds the levels top-down (per level: prepare items, tiles, finish items): every item waits only for items with
// a smaller queue index, so there is no deadlock whatever the number of resident blocks.
__global__ void __launch_bounds__(SPC_THREADS, 1) k_selinv_tree(SelInv a) {
  extern __shared__ __align__(16) double si_sm[];
  __shared__ int s_item;
  const int tid = threadIdx.x;
  for (;;) {
    __syncthreads();
    if (tid == 0) s_item = atomicAdd(a.ticket, 1);
    __syncthreads();
    const int it = s_item;
    if (it >= a.n_items) return;
    const int2 q = a.queue[it];
    const int id = q.x;
    if (q.y == -1) {
      si_prepare(a, id, si_sm);
      __syncthreads();
      if (tid == 0) {
        __threadfence();
        atomicExch(a.pdone + id, 1);
      }
    } else if (q.y >= 0) {
      if (tid == 0) spc_wait_ge(a.pdone + id, 1);
      __syncthreads();
      si_tile(a, id, q.y, a.tiles[id], si_sm);
      __syncthreads();
      if (tid == 0) {
        __threadfence();
        atomicAdd(a.tdone + id, 1);
      }
    } else {
      if (tid == 0) {
        spc_wait_ge(a.pdone + id, 1);  // (a node without tiles -- a root -- has no other path to its own prepare item)
        spc_wait_ge(a.tdone + id, a.tiles[id]);
      }
      __syncthreads();
      si_finish(a, id);
      __syncthreads();
      if (tid == 0) {
        __threadfence();
        atomicExch(a.sdone + id, 1);
      }
    }
  }
}

// column q of Z (by position, 6 x 4 row-major per position) as a right-hand side of the backward substitution
__global__ void __launch_bounds__(BA_THREADS) k_cov_zcol(int n6, int q, const double *__restrict__ Zb, double *__restrict__ zq) {
  const int i = blockIdx.x * BA_THREADS + threadIdx.x;
  if (i < n6) zq[i] = Zb[4 * (size_t)i + q];
}

// T = C - Z^T Z (partials of k_spb_reduce added in block order) and T^-1 by a 4 x 4 Cholesky (one thread).  A non-positive or
// non-finite pivot sets lin_fail.
__global__ void k_cov_border(int nblk, const double *__restrict__ part, const double *__restrict__ kk, double *__restrict__ Tinv,
                             LmState *st) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  double s[10];
  for (int k = 0; k < 10; ++k) {
    double v = 0.0;
    for (int b = 0; b < nblk; ++b) v += part[14 * (size_t)b + k];
    s[k] = v;
  }
  double T[4][4];
  int u = 0;
  for (int i = 0; i < 4; ++i)
    for (int c = i; c < 4; ++c) {
      T[i][c] = kk[i * 4 + c] - s[u++];
      T[c][i] = T[i][c];
    }
  double L[4][4] = {{0.0}}, Li[4][4] = {{0.0}};
  bool ok = true;
  for (int j = 0; j < 4; ++j) {
    double d = T[j][j];
    for (int k = 0; k < j; ++k) d -= L[j][k] * L[j][k];
    if (!(d > 0.0) || !isfinite(d)) ok = false;
    L[j][j] = ok ? sqrt(d) : 1.0;
    for (int i = j + 1; i < 4; ++i) {
      double x = T[i][j];
      for (int k = 0; k < j; ++k) x -= L[i][k] * L[j][k];
      L[i][j] = x / L[j][j];
    }
  }
  for (int c = 0; c < 4; ++c)
    for (int i = c; i < 4; ++i) {
      double x = i == c ? 1.0 : 0.0;
      for (int k = c; k < i; ++k) x -= L[i][k] * Li[k][c];
      Li[i][c] = x / L[i][i];
    }
  for (int i = 0; i < 4; ++i)
    for (int c = i; c < 4; ++c) {
      double v = 0.0;
      for (int k = c; k < 4; ++k) v += Li[k][i] * Li[k][c];
      Tinv[i * 4 + c] = v;
      Tinv[c * 4 + i] = v;
    }
  if (!ok) st->lin_fail = 1;
}

// Sigma (scaled) on every stored block of S: the finished fronts (through the block's entry record: node, local row, local
// column, flags 1 = transposed / 2 = diagonal) plus the border correction X_i T^-1 X_j^T.  Diagonal blocks are computed on
// their upper triangle and mirrored: exactly symmetric.
__global__ void __launch_bounds__(BA_THREADS)
k_cov_blocks(int n_blk, const int4 *__restrict__ brec, const int32_t *__restrict__ blk_i, const int32_t *__restrict__ blk_j,
             const int32_t *__restrict__ node, const double *__restrict__ panel, const int32_t *__restrict__ pos, int n_cam,
             const double *__restrict__ X, const double *__restrict__ Tinv, double *__restrict__ covS) {
  const int idx = blockIdx.x * BA_THREADS + threadIdx.x;
  if (idx >= n_blk * 36) return;
  const int b = idx / 36, e = idx - 36 * b;
  int x = e / 6, y = e - 6 * (e / 6);
  const int4 r = brec[b];
  const int32_t *N = node + (size_t)r.x * SPSYM_NODE_INTS;
  const int LD = 6 * (N[SPN_M] + N[SPN_NB]);
  const double *Pg = panel + 36 * spc_off(N, SPN_PANEL_LO);
  double v;
  if (r.w & 2) {
    if (x > y) {
      const int t = x;
      x = y;
      y = t;
    }
    v = Pg[(size_t)(6 * r.z + y) * LD + 6 * r.z + x];
  } else if (r.w & 1) {
    v = Pg[(size_t)(6 * r.z + x) * LD + 6 * r.y + y];
  } else {
    v = Pg[(size_t)(6 * r.z + y) * LD + 6 * r.y + x];
  }
  if (X) {
    const size_t n6 = 6 * (size_t)n_cam, ri = 6 * (size_t)pos[blk_i[b]] + x, rj = 6 * (size_t)pos[blk_j[b]] + y;
    double s = 0.0;
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      double t = 0.0;
#pragma unroll
      for (int q = 0; q < 4; ++q) t += Tinv[p * 4 + q] * X[q * n6 + rj];
      s += X[p * n6 + ri] * t;
    }
    v += s;
  }
  covS[idx] = v;
}

// stored block of S for the camera pair (i <= j): binary search of column j in row i's entries (ascending columns), -1 if none
__device__ __forceinline__ int cov_find_block(const int32_t *__restrict__ ent_ptr, const int2 *__restrict__ ent, int i, int j) {
  int lo = ent_ptr[i], hi = ent_ptr[i + 1];
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (ent[mid].y < j)
      lo = mid + 1;
    else
      hi = mid;
  }
  return (lo < ent_ptr[i + 1] && ent[lo].y == j) ? (int)((uint32_t)ent[lo].x & 0x7fffffffu) : -1;
}

// per camera: Sigma_cc (unscaled, from its diagonal block) and Sigma_ck = -X_c T^-1 (scaled -> ck, unscaled -> cam_intr); the
// fixed camera's blocks are zero
__global__ void __launch_bounds__(BA_THREADS)
k_cov_cam(int n_cam, int fixed_cam, int nk, const int32_t *__restrict__ diag, const double *__restrict__ covS,
          const int32_t *__restrict__ pos, const double *__restrict__ X, const double *__restrict__ Tinv, const double *__restrict__ sc,
          const double *__restrict__ sk, double *__restrict__ ck, double *__restrict__ cam_out, double *__restrict__ ci_out) {
  const int idx = blockIdx.x * BA_THREADS + threadIdx.x;
  if (idx >= n_cam * 60) return;
  const int c = idx / 60, e = idx - 60 * c;
  const bool fixed = c == fixed_cam;
  if (e < 36) {
    const int x = e / 6, y = e - 6 * (e / 6), b = diag[c];
    cam_out[36 * (size_t)c + e] = (fixed || b < 0) ? 0.0 : covS[36 * (size_t)b + e] * (sc[6 * (size_t)c + x] * sc[6 * (size_t)c + y]);
  } else {
    const int q = e - 36, x = q / 4, k = q - 4 * (q / 4);
    double v = 0.0;
    if (nk && !fixed) {
      const size_t n6 = 6 * (size_t)n_cam, rc = 6 * (size_t)pos[c] + x;
      double s = 0.0;
#pragma unroll
      for (int p = 0; p < 4; ++p) s += X[p * n6 + rc] * Tinv[p * 4 + k];
      v = -s;
    }
    ck[24 * (size_t)c + q] = v;
    ci_out[24 * (size_t)c + q] = v * (sc[6 * (size_t)c + x] * sk[k]);
  }
}

// Cov(delta_a, delta_b) of the requested camera pairs (unscaled); a pair of cameras that share no point sets *bad
__global__ void __launch_bounds__(BA_THREADS)
k_cov_pairs(int n_pairs, const int32_t *__restrict__ cam_a, const int32_t *__restrict__ cam_b, int fixed_cam,
            const int32_t *__restrict__ ent_ptr, const int2 *__restrict__ ent, const double *__restrict__ covS,
            const double *__restrict__ sc, double *__restrict__ out, int *bad) {
  const int idx = blockIdx.x * BA_THREADS + threadIdx.x;
  if (idx >= n_pairs * 36) return;
  const int pi = idx / 36, e = idx - 36 * pi, x = e / 6, y = e - 6 * (e / 6);
  const int a = cam_a[pi], b = cam_b[pi];
  double v = 0.0;
  if (a != fixed_cam && b != fixed_cam) {
    const int blk = cov_find_block(ent_ptr, ent, min(a, b), max(a, b));
    if (blk < 0) {
      *bad = 1;  // (every writer stores the same value)
    } else {
      v = (a <= b ? covS[36 * (size_t)blk + 6 * x + y] : covS[36 * (size_t)blk + 6 * y + x]) *
          (sc[6 * (size_t)a + x] * sc[6 * (size_t)b + y]);
    }
  }
  out[idx] = v;
}

// Sigma_pp = V^-1 + V^-1 M V^-1, M = W_p^T Sigma_RR W_p over the point's observation pairs (point-major, cameras ascending),
// plus the intrinsics terms; one thread per point, pairs in slot order.  Unscaled, exactly symmetric.
__global__ void __launch_bounds__(BA_THREADS)
k_cov_points(int n_pt, int fixed_cam, int nk, const int32_t *__restrict__ pt_rowptr, const int32_t *__restrict__ pm_cam,
             const int32_t *__restrict__ perm, const double *__restrict__ W, const double *__restrict__ Wk,
             const double *__restrict__ Vinv, const int32_t *__restrict__ ent_ptr, const int2 *__restrict__ ent,
             const double *__restrict__ covS, const double *__restrict__ ck, const double *__restrict__ Tinv,
             const double *__restrict__ sp, double *__restrict__ out) {
  const int p = blockIdx.x * BA_THREADS + threadIdx.x;
  if (p >= n_pt) return;
  double M[3][3];
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int s = 0; s < 3; ++s) M[r][s] = 0.0;
  double wk[4][3];
#pragma unroll
  for (int k = 0; k < 4; ++k)
#pragma unroll
    for (int s = 0; s < 3; ++s) wk[k][s] = nk ? Wk[12 * (size_t)p + 3 * k + s] : 0.0;
  const int s0 = pt_rowptr[p], s1 = pt_rowptr[p + 1];
  for (int sa = s0; sa < s1; ++sa) {
    const int ca = pm_cam[sa];
    if (ca == fixed_cam) continue;
    const double *Wa = W + 18 * (size_t)perm[sa];
    for (int sb = sa; sb < s1; ++sb) {
      const int cb = pm_cam[sb];
      if (cb == fixed_cam) continue;
      const int blk = cov_find_block(ent_ptr, ent, ca, cb);
      if (blk < 0) continue;
      const double *Sg = covS + 36 * (size_t)blk, *Wb = W + 18 * (size_t)perm[sb];
      double t[6][3];  // Sigma_ab W_b
#pragma unroll
      for (int r = 0; r < 6; ++r)
#pragma unroll
        for (int s = 0; s < 3; ++s) {
          double v = 0.0;
#pragma unroll
          for (int k = 0; k < 6; ++k) v += Sg[6 * r + k] * Wb[3 * k + s];
          t[r][s] = v;
        }
#pragma unroll
      for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int s = 0; s < 3; ++s) {
          double v = 0.0, w = 0.0;
#pragma unroll
          for (int k = 0; k < 6; ++k) {
            v += Wa[3 * k + r] * t[k][s];
            w += Wa[3 * k + s] * t[k][r];
          }
          M[r][s] += sb == sa ? v : v + w;
        }
    }
    if (nk) {
      const double *C = ck + 24 * (size_t)ca;
      double t[6][3];  // Sigma_ck W_k
#pragma unroll
      for (int r = 0; r < 6; ++r)
#pragma unroll
        for (int s = 0; s < 3; ++s) {
          double v = 0.0;
#pragma unroll
          for (int k = 0; k < 4; ++k) v += C[4 * r + k] * wk[k][s];
          t[r][s] = v;
        }
#pragma unroll
      for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int s = 0; s < 3; ++s) {
          double v = 0.0, w = 0.0;
#pragma unroll
          for (int k = 0; k < 6; ++k) {
            v += Wa[3 * k + r] * t[k][s];
            w += Wa[3 * k + s] * t[k][r];
          }
          M[r][s] += v + w;
        }
    }
  }
  if (nk) {
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int s = 0; s < 3; ++s) {
        double v = 0.0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          double t = 0.0;
#pragma unroll
          for (int l = 0; l < 4; ++l) t += Tinv[4 * k + l] * wk[l][s];
          v += wk[k][r] * t;
        }
        M[r][s] += v;
      }
  }
  const double *vp = Vinv + 6 * (size_t)p;
  const double Vi[3][3] = {{vp[0], vp[1], vp[2]}, {vp[1], vp[3], vp[4]}, {vp[2], vp[4], vp[5]}};
  double VM[3][3];
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int s = 0; s < 3; ++s) VM[r][s] = Vi[r][0] * M[0][s] + Vi[r][1] * M[1][s] + Vi[r][2] * M[2][s];
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int s = r; s < 3; ++s) {
      const double v = (Vi[r][s] + (VM[r][0] * Vi[0][s] + VM[r][1] * Vi[1][s] + VM[r][2] * Vi[2][s])) *
                       (sp[3 * (size_t)p + r] * sp[3 * (size_t)p + s]);
      out[9 * (size_t)p + 3 * r + s] = v;
      out[9 * (size_t)p + 3 * s + r] = v;
    }
}
