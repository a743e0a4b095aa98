// ba_kernels_spchol.cuh -- NUMERIC phase of the exact sparse Cholesky of the reduced camera system
// (BA_SOLVER_SPARSE_SCHUR_CHOLESKY): what the reference asks Ceres for with linear_solver_type = SPARSE_SCHUR
// (headers/BundleAdjustmentConfig.h:62; ceres::Solve at src/OptimizationUtils.cpp:300) -- the explicit block-sparse
// S of ba_kernels_sparse.cuh factorised exactly instead of handed to PCG.
//
// Supernodal multifrontal Cholesky over the nested-dissection tree built on the host (ba_sparse_symbolic.h), as ONE persistent
// launch (k_spchol_tree, below) that works through a queue of factor, update and solve items with completion counters:
//   * ONE thread block per factor item (a tree node); a node starts as soon as its children's update matrices are done.
//   * A node's FRONT PANEL ((own + border) x own cameras, dense, scalar column-major, leading dimension LD = 6 (m + nb))
//     lives in shared memory for the whole elimination of its m own cameras: assembled from the stored blocks of S
//     (+ LM damping on the diagonal) minus the children's update matrices (extend-add through the host-built index maps),
//     then factorised right-looking with 6x6 pivot blocks.  One thread owns one scalar ROW of the panel: a step costs it
//     six contiguous loads of its pivot-column entries (kept row-major in a side buffer LT), and per trailing block column
//     36 warp-broadcast loads of the pivot rows + a conflict-free read-modify-write of its six entries.
//   * The 6x6 pivot block is factorised by warp 0 with shuffles (lane = row) while the other warps still run the
//     trailing update of the previous step (look-ahead): two CTA barriers per eliminated camera.
//   * The right-hand side rides along as one more row (forward substitution fused into the factorisation).  With free
//     intrinsics (REF cost) it is R = 5 rows: b_c and the four columns of the camera-intrinsics border B, so the forward
//     substitution yields z = L^-1 b_c and Z = L^-1 B; the 4x4 border system T y_k = t (T = C - Z^T Z, t = b_k - Z^T z)
//     is solved between factorisation and backward substitution (k_spb_reduce / k_spb_solve), and the backward
//     substitution solves L^T y_c = z - Z y_k.  The symbolic phase, the tree and the supernodes are the same for R = 1, 5.
//   * The panel goes to HBM/L2 for the backward substitution; the node's update matrix U = L_B L_B^T (+ what its children
//     pass through) -- two thirds of the multiply-adds, no dependent chain -- is formed by several update items per node
//     (spc_update_node), for the parent's extend-add.
// Backward substitution: parents before children (solve items of the tree; the covariance's border columns run the queue's
// solve items alone, one launch per column); L_OO and the stored inverses of the pivot blocks come back into shared memory,
// the border product is a warp-per-column reduction over the panel in L2.
// Every sum has a fixed order: results are bit-identical from run to run and across ranks.
#pragma once
#include "ba_kernels_sparse.cuh"
#include "ba_sparse_symbolic.h"

#define SPC_THREADS 512
#define SPC_WARPS (SPC_THREADS / 32)
// capacity of a front in 6x6 blocks: (m + nb) (m + 1) [panel + the row-major pivot column LT] <= SPC_CAP_BLOCKS, m <= SPC_MAX_OWN
#define SPC_CAP_BLOCKS 770
#define SPC_MAX_OWN 24

struct SpChol {
  const int32_t *node, *bord, *children, *rel, *inv, *aent, *perm;
  const double *S, *dsq, *b;  // stored upper blocks of S, LM damping D^2 [6 n_cam], right-hand side [6 n_cam] (by camera)
  double *panel, *U, *ru;     // per node: factor panel, update matrix (dense lower incl. full diagonal blocks), rhs update [6 nb]
  double *z, *linv, *ypos;    // by elimination position: forward-substituted rhs [6], inverse pivot blocks [36], solution [6]
  double *yc;                 // solution by camera [6 n_cam]
  unsigned long long *prof;   // nullable (BA_SPCHOL_PROF=1): ns per phase of thread block 0 of every factor launch, summed
  // intrinsics border (R = 5; nullptr otherwise): B by camera [24 n_cam] (6 x 4 row-major per camera), Z = L^-1 B by
  // elimination position [24 n_cam] (6 x 4 row-major per position), y_k [4] (read by the backward substitution)
  const double *Bc;
  double *Zb;
  const double *yk;
};
#define SPC_TICK(slot)                                          \
  if (a.prof && prof_block && tid == 0) {                       \
    unsigned long long t1_;                                     \
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t1_));      \
    a.prof[slot] += t1_ - t0_;                                  \
    t0_ = t1_;                                                  \
  }

__host__ __device__ inline size_t spc_off(const int32_t *N, int lo) { return ((size_t)N[lo + 1] << 31) | (size_t)N[lo]; }
// (R: right-hand-side rows, 1 or 5)
inline size_t spc_factor_smem(int m, int nb, int R = 1) { return ((size_t)36 * (m + nb) * (m + 1) + 6 * m * R + 72 + 8) * 8; }
inline size_t spc_solve_smem(int m, int nb) { return ((size_t)36 * m * m + 36 * m + 6 * nb + 12 * m + 8) * 8; }

// right-hand side b = -g_c - sum (J_c^T J_p V^-1 g_p partials) and LM damping D^2 = (sqrt(diag / radius))^2 per camera column
__global__ void __launch_bounds__(BA_THREADS)
k_spchol_rhs(int n_cam, const int32_t *__restrict__ item_ptr, const double *__restrict__ part, const double *__restrict__ gc,
             const double *__restrict__ dc, double *__restrict__ b, double *__restrict__ dsq, LmState *st, int gate, int keep_b) {
  if (!gate_open(st, gate)) return;
  const int c = blockIdx.x * BA_THREADS + threadIdx.x;
  if (c == 0) st->pcg_iters_last = 0;
  if (c >= n_cam) return;
  const double radius = st->radius;
  if (!keep_b) {
    double s[6], g[6], bv[6];
    sum_items6(item_ptr, part, c, s);
    load6(gc + 6 * (size_t)c, g);
#pragma unroll
    for (int k = 0; k < 6; ++k) bv[k] = -g[k] - s[k];
    store6(b + 6 * (size_t)c, bv);
  }
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    const double D = sqrt(dc[6 * (size_t)c + k] / radius);
    dsq[6 * (size_t)c + k] = D * D;
  }
}

// Cholesky of the 6x6 pivot block k of the panel by one warp (lane = row, lanes 0..5 carry data): L back into the panel
// (upper triangle zeroed), T = L^-1 (lower, row-major) to Tout and to linv_g.  Returns false on a non-positive pivot.
__device__ __forceinline__ bool spc_chol6(double *P, int LD, int k, int lane, double *Tout, double *linv_g) {
  double row[6], invd[6];
  const int r = lane < 6 ? lane : 0;
  double *D = P + (size_t)(6 * k) * LD + 6 * k;  // D[c * LD + r] = block(r, c)
#pragma unroll
  for (int c = 0; c < 6; ++c) row[c] = (c <= r) ? D[(size_t)c * LD + r] : 0.0;
  bool ok = true;
#pragma unroll
  for (int c = 0; c < 6; ++c) {
    const double dcc = __shfl_sync(BA_FULL, row[c], c);
    if (!(dcc > 0.0) || !isfinite(dcc)) ok = false;
    // one reciprocal square root instead of a square root and a division on the dependent chain of the six columns
    const double inv = rsqrt(dcc);
    const double s = dcc * inv;
    invd[c] = inv;
    if (lane == c)
      row[c] = s;
    else if (lane > c)
      row[c] *= inv;
#pragma unroll
    for (int c2 = c + 1; c2 < 6; ++c2) {
      const double v = __shfl_sync(BA_FULL, row[c], c2);
      if (lane >= c2) row[c2] -= row[c] * v;
    }
  }
  if (lane < 6) {
#pragma unroll
    for (int c = 0; c < 6; ++c) D[(size_t)c * LD + lane] = (c <= lane) ? row[c] : 0.0;
  }
  __syncwarp();
  if (lane < 6) {
    // column `lane` of T = L^-1 by forward substitution (the reciprocals of the diagonal are in registers)
    double t[6];
#pragma unroll
    for (int rr = 0; rr < 6; ++rr) {
      if (rr < lane) {
        t[rr] = 0.0;
      } else if (rr == lane) {
        t[rr] = invd[rr];
      } else {
        double acc = 0.0;
#pragma unroll
        for (int q = 0; q < 6; ++q)
          if (q < rr && q >= lane) acc += D[(size_t)q * LD + rr] * t[q];
        t[rr] = -acc * invd[rr];
      }
    }
#pragma unroll
    for (int rr = 0; rr < 6; ++rr) {
      Tout[rr * 6 + lane] = t[rr];
      linv_g[rr * 6 + lane] = t[rr];
    }
  }
  __syncwarp();
  return ok;
}

// six consecutive doubles from shared memory, 16-byte aligned (rows of the row-major pivot column): three LDS.128
__device__ __forceinline__ void spc_ld6(const double *p, double v[6]) {
  const double2 *q = reinterpret_cast<const double2 *>(p);
  const double2 a = q[0], b = q[1], c = q[2];
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; v[4] = c.x; v[5] = c.y;
}

// (i, j), i >= j, of the p-th lower block in row-major order of the lower triangle
__device__ __forceinline__ void spc_tri(int p, int &i, int &j) {
  int r = (int)((sqrt(8.0 * (double)p + 1.0) - 1.0) * 0.5);
  while (r * (r + 1) / 2 > p) --r;
  while ((r + 1) * (r + 2) / 2 <= p) ++r;
  i = r;
  j = p - r * (r + 1) / 2;
}

// the take / wait / publish steps of the persistent tree kernels (k_spchol_tree, k_selinv_tree).  Take: the next queue item
// from the ticket counter, between two barriers (the first: the previous item's shared memory is no longer in use).
__device__ __forceinline__ int spc_take(int *ticket, int *s_item) {
  __syncthreads();
  if (threadIdx.x == 0) *s_item = atomicAdd(ticket, 1);
  __syncthreads();
  return *s_item;
}
// wait (one thread) until a completion counter reaches `want`
__device__ __forceinline__ void spc_wait_ge(const int *flag, int want) {
  int v;
  for (;;) {
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
    if (v >= want) return;
    __nanosleep(64);
  }
}
// publish an item: barrier (every thread's writes of the item are issued), device-scope fence, then the counter -- set to 1
// for the one item of its kind a node has, one more for a tile
__device__ __forceinline__ void spc_publish(int *counter, bool tile) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    if (tile)
      atomicAdd(counter, 1);
    else
      atomicExch(counter, 1);
  }
}
// factorisation of the front of node `id` by the calling thread block (SPC_THREADS threads, spc_factor_smem bytes at spc_sm)
// (udone / tiles: completion counters of k_spchol_tree -- the node waits for its children's update matrices only AFTER it has
//  assembled its stored blocks of S, which do not depend on them)
// NR right-hand-side rows (1: b; 5: b and the four border columns), row r of the own cameras at zf[r * C6 ..]
template <int NR>
__device__ __forceinline__ void spc_factor_node(const SpChol &a, int id, bool prof_block, LmState *st, double *spc_sm,
                                                const int *udone, const int32_t *tiles) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int32_t *N = a.node + (size_t)id * SPSYM_NODE_INTS;
  const int k0 = N[SPN_K0], m = N[SPN_M], nb = N[SPN_NB];
  const int LD = 6 * (m + nb), C6 = 6 * m;
  double *P = spc_sm;                    // panel, column-major, LD x C6
  double *LT = P + (size_t)LD * C6;      // current pivot column block, row-major: LT[R * 6 + c]
  double *zf = LT + (size_t)LD * 6;      // right-hand-side rows of the own cameras
  double *Tb = zf + NR * C6;             // two inverse pivot blocks (ping-pong)

  unsigned long long t0_ = 0;
  if (a.prof && prof_block && tid == 0) asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t0_));
  // ---- phase 0: clear, right-hand side
  for (int i = tid; i < LD * C6; i += SPC_THREADS) P[i] = 0.0;
  for (int i = tid; i < NR * C6; i += SPC_THREADS) {
    const int r = i / C6, j = i - r * C6;
    const int cam = a.perm[k0 + j / 6];
    zf[i] = r == 0 ? a.b[6 * (size_t)cam + j % 6] : a.Bc[24 * (size_t)cam + (j % 6) * 4 + r - 1];
  }
  __syncthreads();
  // ---- phase 1a: stored blocks of S (one thread per scalar, entry records through 16-byte broadcast loads), damping on
  //      the diagonal.  Independent iterations: unrolled so that several dependent load chains are in flight.
  {
    const int4 *E4 = reinterpret_cast<const int4 *>(a.aent) + N[SPN_AENT];
    const int ne36 = 36 * N[SPN_NAENT];
#pragma unroll 4
    for (int idx = tid; idx < ne36; idx += SPC_THREADS) {
      const int e = idx / 36, t = idx - 36 * e, r6 = t / 6, c6 = t - 6 * r6;
      const int4 en = __ldg(E4 + e);  // (block | flags, local row, local column, camera of the column)
      const uint32_t code = (uint32_t)en.x, blk = code & 0x3fffffffu;
      double v = 0.0;
      if (code & 0x40000000u) {  // diagonal block: symmetrised from its upper triangle (as k_sp_minv does) + D^2
        if (blk != 0x3fffffffu) v = a.S[36 * (size_t)blk + (r6 <= c6 ? r6 * 6 + c6 : c6 * 6 + r6)];
        if (r6 == c6) v += a.dsq[6 * (size_t)en.w + r6];
      } else if (code & 0x80000000u) {
        v = a.S[36 * (size_t)blk + c6 * 6 + r6];
      } else {
        v = a.S[36 * (size_t)blk + r6 * 6 + c6];
      }
      P[(size_t)(6 * en.z + c6) * LD + 6 * en.y + r6] = v;
    }
  }
  if (tid == 0)
    for (int ci = 0; ci < N[SPN_NCHILD]; ++ci) {
      const int ch = a.children[N[SPN_CHILD] + ci];
      spc_wait_ge(udone + ch, tiles[ch]);
    }
  __syncthreads();
  SPC_TICK(0)
  // ---- phase 1b: extend-add of the children (one after the other: fixed order; inside a child the map is injective).
  //      rel is ascending, so the child's border cameras that are OWN cameras of this node come first: only those block
  //      columns land in the panel (the rest of the child's update matrix passes through to this node's, spc_update_node)
  for (int ci = 0; ci < N[SPN_NCHILD]; ++ci) {
    const int ch = a.children[N[SPN_CHILD] + ci];
    const int32_t *Cn = a.node + (size_t)ch * SPSYM_NODE_INTS;
    const int nbc = Cn[SPN_NB], nbc6 = 6 * nbc;
    const int32_t *rel = a.rel + Cn[SPN_REL];
    int n_in = 0;  // first border index with rel >= m (binary search, same on every thread)
    {
      int lo = 0, hi = nbc;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(rel + mid) < m)
          lo = mid + 1;
        else
          hi = mid;
      }
      n_in = lo;
    }
    const double *Uc = a.U + 36 * spc_off(Cn, SPN_U_LO);
    const double *ruc = a.ru + 6 * NR * (size_t)Cn[SPN_BORD];  // (row r of the child's rhs update at ruc[r * nbc6 ..])
    // one warp per scalar column of the child's update matrix (block lower triangle: rows from the column's own block
    // down), lanes along the rows: coalesced reads of the column from L2, up to four independent loads in flight per lane
    // before the first one is consumed (this gather was the longest piece of a node's critical path: one dependent
    // round trip to L2 per element in the first version)
    for (int col = warp; col < 6 * n_in; col += SPC_WARPS) {
      const int j = col / 6, cj = col - 6 * j;
      const int rj = __ldg(rel + j);
      const double *ucol = Uc + (size_t)col * nbc6;
      double *pcol = P + (size_t)(6 * rj + cj) * LD;
      for (int row0 = 6 * j; row0 < nbc6; row0 += 128) {
        double v[4];
        int dst[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int row = row0 + lane + 32 * u;
          v[u] = 0.0;
          dst[u] = -1;
          if (row < nbc6) {
            v[u] = __ldcg(ucol + row);
            const int i = row / 6;
            dst[u] = 6 * __ldg(rel + i) + (row - 6 * i);
          }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (dst[u] >= 0) pcol[dst[u]] -= v[u];
      }
    }
    for (int idx = tid; idx < NR * 6 * n_in; idx += SPC_THREADS) {
      const int r = idx / (6 * n_in), e = idx - r * 6 * n_in;
      zf[r * C6 + 6 * __ldg(rel + e / 6) + e % 6] -= __ldcg(ruc + (size_t)r * nbc6 + e);
    }
    __syncthreads();
  }
  SPC_TICK(1)
  // ---- phase 2: right-looking factorisation, 6 columns (one camera) per step
  bool ok = true;
  if (warp == 0) ok = spc_chol6(P, LD, 0, lane, Tb, a.linv + 36 * (size_t)k0);
  __syncthreads();
  for (int k = 0; k < m; ++k) {
    const double *T = Tb + (k & 1) * 36;
    // (b) pivot column: rows below the pivot block times T^T; forward substitution of the pivot's right-hand side
    for (int R = 6 * (k + 1) + tid; R < LD; R += SPC_THREADS) {
      double x[6];
#pragma unroll
      for (int c = 0; c < 6; ++c) x[c] = P[(size_t)(6 * k + c) * LD + R];
#pragma unroll
      for (int bb = 0; bb < 6; ++bb) {
        double o = 0.0;
#pragma unroll
        for (int c = 0; c < 6; ++c)
          if (c <= bb) o += x[c] * T[bb * 6 + c];
        P[(size_t)(6 * k + bb) * LD + R] = o;
        LT[R * 6 + bb] = o;
      }
    }
    if (warp == 0) {
      // lane = (rhs row r, component l): 6 NR <= 30 lanes
      const int r = lane / 6, l = lane - 6 * r;
      double *zr = zf + r * C6 + 6 * k;
      double v = 0.0;
      if (lane < 6 * NR) {
#pragma unroll
        for (int c = 0; c < 6; ++c)
          if (c <= l) v += T[l * 6 + c] * zr[c];
      }
      __syncwarp();
      if (lane < 6 * NR) zr[l] = v;
    }
    __syncthreads();
    if (k + 1 == m) break;
    // (c) trailing update with column k.  Warp 0: the rows of the next pivot block, then its Cholesky (look-ahead);
    //     the other warps: one scalar row each (and a share of the block columns when rows are fewer than threads)
    if (warp == 0) {
      if (lane < 6) {
        const int R = 6 * (k + 1) + lane, j = k + 1;
        double x[6];
        spc_ld6(LT + R * 6, x);
#pragma unroll
        for (int bb = 0; bb < 6; ++bb) {
          double lj[6];
          spc_ld6(LT + (6 * j + bb) * 6, lj);
          double s = 0.0;
#pragma unroll
          for (int c = 0; c < 6; ++c) s += x[c] * lj[c];
          P[(size_t)(6 * j + bb) * LD + R] -= s;
        }
#pragma unroll
        for (int r = 0; r < NR; ++r) {
          double s = 0.0;
#pragma unroll
          for (int c = 0; c < 6; ++c) s += x[c] * zf[r * C6 + 6 * k + c];
          zf[r * C6 + R] -= s;
        }
      }
      __syncwarp();
      ok = spc_chol6(P, LD, k + 1, lane, Tb + ((k + 1) & 1) * 36, a.linv + 36 * (size_t)(k0 + k + 1)) && ok;
    } else {
      // own rows (R < C6: their block-column range ends at their own block) one per thread; border rows (all block columns)
      // two per thread, so that the pivot rows lj -- warp-broadcast loads -- are fetched once for two rows
      const int base = 6 * (k + 2), avail = SPC_THREADS - 32;
      const int n_own = C6 > base ? C6 - base : 0;
      const int b0 = C6 > base ? C6 : base, n_bord = LD - b0, n_pair = (n_bord + 1) >> 1;
      const int n_it = n_own + n_pair;
      if (n_it > 0) {
        int G = avail / n_it;
        G = G < 1 ? 1 : (G > 4 ? 4 : G);
        for (int t = tid - 32; t < G * n_it; t += avail) {
          const int g = t / n_it, u = t - g * n_it;
          if (u < n_own) {
            const int R = base + u;
            const int jmax = R / 6;  // (< m: an own row)
            double x[6];
            spc_ld6(LT + R * 6, x);
            for (int j = k + 1 + g; j <= jmax; j += G) {
#pragma unroll
              for (int bb = 0; bb < 6; ++bb) {
                double lj[6];
                spc_ld6(LT + (6 * j + bb) * 6, lj);
                double s = 0.0;
#pragma unroll
                for (int c = 0; c < 6; ++c) s += x[c] * lj[c];
                P[(size_t)(6 * j + bb) * LD + R] -= s;
              }
            }
            if (g == 0) {
#pragma unroll
              for (int r = 0; r < NR; ++r) {
                double s = 0.0;
#pragma unroll
                for (int c = 0; c < 6; ++c) s += x[c] * zf[r * C6 + 6 * k + c];
                zf[r * C6 + R] -= s;
              }
            }
          } else {
            const int R1 = b0 + (u - n_own), R2 = R1 + n_pair;
            const bool two = R2 < LD;
            double x1[6], x2[6];
            spc_ld6(LT + R1 * 6, x1);
            spc_ld6(LT + (two ? R2 : R1) * 6, x2);
            for (int j = k + 1 + g; j < m; j += G) {
#pragma unroll
              for (int bb = 0; bb < 6; ++bb) {
                double lj[6];
                spc_ld6(LT + (6 * j + bb) * 6, lj);
                double s1 = 0.0, s2 = 0.0;
#pragma unroll
                for (int c = 0; c < 6; ++c) {
                  s1 += x1[c] * lj[c];
                  s2 += x2[c] * lj[c];
                }
                double *pc = P + (size_t)(6 * j + bb) * LD;
                pc[R1] -= s1;
                if (two) pc[R2] -= s2;
              }
            }
          }
        }
      }
    }
    __syncthreads();
  }
  if (warp == 0 && lane == 0 && !ok) st->lin_fail = 1;
  SPC_TICK(2)
  // ---- phase 3: panel and forward-substituted right-hand side to global memory
  {
    double *Pg = a.panel + 36 * spc_off(N, SPN_PANEL_LO);
    for (int i = tid; i < LD * C6; i += SPC_THREADS) Pg[i] = P[i];
    for (int i = tid; i < C6; i += SPC_THREADS) a.z[6 * (size_t)k0 + i] = zf[i];
    if (NR > 1)
      for (int i = tid; i < (NR - 1) * C6; i += SPC_THREADS) {
        const int q = i / C6, j = i - q * C6;
        a.Zb[4 * (6 * (size_t)k0 + j) + q] = zf[(q + 1) * C6 + j];
      }
  }
  __syncthreads();
  SPC_TICK(3)
  if (a.prof && prof_block && tid == 0) a.prof[4] += 1;
}

// Update matrix of a node, after its panel is factorised: U = L_B L_B^T + what the children pass through (block lower
// triangle, full diagonal blocks) and the right-hand side update ru = L_B z + children.  This is two thirds of a node's
// multiply-adds and has no dependent chain, so it is split into `tiles` items per node: the upper levels of the tree have
// fewer nodes than the GPU has SMs.  Every item loads the node's border rows of the panel (L2-resident, just written) into
// shared memory and takes every tiles-th chunk of the 3 x 6 output pieces.
inline size_t spc_update_smem(int m, int nb, int R = 1) { return ((size_t)36 * nb * m + 6 * m * R + 8) * 8; }
// tile `tile` of `tiles` of the update matrix of node `id`, by the calling thread block; NR right-hand-side rows
template <int NR>
__device__ __forceinline__ void spc_update_node(const SpChol &a, int id, int tile, int tiles, double *spc_sm) {
  const int tid = threadIdx.x;
  const int32_t *N = a.node + (size_t)id * SPSYM_NODE_INTS;
  const int k0 = N[SPN_K0], m = N[SPN_M], nb = N[SPN_NB];
  if (nb == 0) return;
  const int LD = 6 * (m + nb), C6 = 6 * m, NB6 = 6 * nb;
  double *LB = spc_sm;              // border rows of the panel, column-major NB6 x C6
  double *zf = LB + (size_t)NB6 * C6;
  {
    const double *Pg = a.panel + 36 * spc_off(N, SPN_PANEL_LO) + C6;
#pragma unroll 8
    for (int idx = tid; idx < NB6 * C6; idx += SPC_THREADS) {
      const int c = idx / NB6, r = idx - c * NB6;
      LB[idx] = __ldcg(Pg + (size_t)c * LD + r);  // (L2: written by another thread block of this or the previous launch)
    }
    for (int i = tid; i < C6; i += SPC_THREADS) zf[i] = __ldcg(a.z + 6 * (size_t)k0 + i);
    if (NR > 1)
      for (int i = tid; i < (NR - 1) * C6; i += SPC_THREADS) {
        const int q = i / C6, j = i - q * C6;
        zf[(q + 1) * C6 + j] = __ldcg(a.Zb + 4 * (6 * (size_t)k0 + j) + q);
      }
  }
  __syncthreads();
  double *Ug = a.U + 36 * spc_off(N, SPN_U_LO);
  const int n_items = nb * (nb + 1);
  const int nch = N[SPN_NCHILD];
  for (int idx = tile * SPC_THREADS + tid; idx < n_items; idx += tiles * SPC_THREADS) {
    int i, j;
    spc_tri(idx >> 1, i, j);
    const int h = idx & 1;
    const int ra = 6 * i + 3 * h, rb = 6 * j;
    double acc[3][6];
#pragma unroll
    for (int x = 0; x < 3; ++x)
#pragma unroll
      for (int y = 0; y < 6; ++y) acc[x][y] = 0.0;
#pragma unroll 2
    for (int c = 0; c < C6; ++c) {
      const double *col = LB + (size_t)c * NB6;
      const double a0 = col[ra], a1 = col[ra + 1], a2 = col[ra + 2];
      const double2 b01 = *reinterpret_cast<const double2 *>(col + rb), b23 = *reinterpret_cast<const double2 *>(col + rb + 2),
                    b45 = *reinterpret_cast<const double2 *>(col + rb + 4);
      const double bv[6] = {b01.x, b01.y, b23.x, b23.y, b45.x, b45.y};
#pragma unroll
      for (int y = 0; y < 6; ++y) {
        acc[0][y] += a0 * bv[y];
        acc[1][y] += a1 * bv[y];
        acc[2][y] += a2 * bv[y];
      }
    }
    for (int ci = 0; ci < nch; ++ci) {
      const int ch = a.children[N[SPN_CHILD] + ci];
      const int32_t *Cn = a.node + (size_t)ch * SPSYM_NODE_INTS;
      const int32_t *inv = a.inv + Cn[SPN_INV];
      const int ii = inv[i], jj = inv[j];
      if (ii < 0 || jj < 0) continue;
      const int nbc6 = 6 * Cn[SPN_NB];
      const double *Uc = a.U + 36 * spc_off(Cn, SPN_U_LO);
#pragma unroll
      for (int y = 0; y < 6; ++y)
#pragma unroll
        for (int x = 0; x < 3; ++x) acc[x][y] += __ldcg(Uc + (size_t)(6 * jj + y) * nbc6 + 6 * ii + 3 * h + x);
    }
#pragma unroll
    for (int y = 0; y < 6; ++y)
#pragma unroll
      for (int x = 0; x < 3; ++x) Ug[(size_t)(rb + y) * NB6 + ra + x] = acc[x][y];
  }
  // rhs updates: row r of the node at ru[6 NR bord + r NB6 ..]
  double *rug = a.ru + 6 * NR * (size_t)N[SPN_BORD];
  for (int idx = tile * SPC_THREADS + tid; idx < NR * NB6; idx += tiles * SPC_THREADS) {
    const int r = idx / NB6, e = idx - r * NB6;
    const double *zr = zf + r * C6;
    double s = 0.0;
    for (int c = 0; c < C6; ++c) s += LB[(size_t)c * NB6 + e] * zr[c];
    for (int ci = 0; ci < nch; ++ci) {
      const int ch = a.children[N[SPN_CHILD] + ci];
      const int32_t *Cn = a.node + (size_t)ch * SPSYM_NODE_INTS;
      const int ii = a.inv[Cn[SPN_INV] + e / 6];
      if (ii >= 0) s += __ldcg(a.ru + 6 * NR * (size_t)Cn[SPN_BORD] + (size_t)r * 6 * Cn[SPN_NB] + 6 * ii + e % 6);
    }
    rug[idx] = s;
  }
}

// backward substitution of one node (its parent is done): y_O = L_OO^-T (z_O - L_BO^T y_B)
__device__ __forceinline__ void spc_solve_node(const SpChol &a, int id, LmState *st, double *spc_sm) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int32_t *N = a.node + (size_t)id * SPSYM_NODE_INTS;
  const int k0 = N[SPN_K0], m = N[SPN_M], nb = N[SPN_NB];
  const int LD = 6 * (m + nb), C6 = 6 * m, NB6 = 6 * nb;
  double *Loo = spc_sm;               // own part of the panel, column-major C6 x C6
  double *Ti = Loo + (size_t)C6 * C6;  // inverse pivot blocks
  double *yB = Ti + 36 * m;
  double *w = yB + NB6;
  double *y = w + C6;
  const double *Pg = a.panel + 36 * spc_off(N, SPN_PANEL_LO);
  const int32_t *bord = a.bord + N[SPN_BORD];
  for (int idx = tid; idx < C6 * C6; idx += SPC_THREADS) {
    const int c = idx / C6, r = idx - c * C6;
    Loo[idx] = __ldcg(Pg + (size_t)c * LD + r);
  }
  for (int i = tid; i < 36 * m; i += SPC_THREADS) Ti[i] = __ldcg(a.linv + 36 * (size_t)k0 + i);
  for (int i = tid; i < NB6; i += SPC_THREADS) yB[i] = __ldcg(a.ypos + 6 * (size_t)bord[i / 6] + i % 6);
  for (int i = tid; i < C6; i += SPC_THREADS) {
    double v = __ldcg(a.z + 6 * (size_t)k0 + i);
    if (a.Zb) {  // intrinsics border: L^T y_c = z - Z y_k
      const double *zr = a.Zb + 4 * (6 * (size_t)k0 + i);
      v -= ((__ldcg(zr) * __ldcg(a.yk) + __ldcg(zr + 1) * __ldcg(a.yk + 1)) + __ldcg(zr + 2) * __ldcg(a.yk + 2)) + __ldcg(zr + 3) * __ldcg(a.yk + 3);
    }
    w[i] = v;
    y[i] = 0.0;
  }
  __syncthreads();
  // w -= L_BO^T y_B: one warp per column, lanes stride the border rows (coalesced reads of the panel)
  for (int c = warp; c < C6; c += SPC_WARPS) {
    const double *col = Pg + (size_t)c * LD + C6;
    double s = 0.0;
    for (int R = lane; R < NB6; R += 32) s += __ldcg(col + R) * yB[R];
    s = warp_sum(s);
    if (lane == 0) w[c] -= s;
  }
  __syncthreads();
  if (warp == 0) {
    for (int k = m - 1; k >= 0; --k) {
      double part[6] = {0, 0, 0, 0, 0, 0};
      for (int R = 6 * (k + 1) + lane; R < C6; R += 32) {
        const double yr = y[R];
#pragma unroll
        for (int c = 0; c < 6; ++c) part[c] += Loo[(size_t)(6 * k + c) * C6 + R] * yr;
      }
#pragma unroll
      for (int c = 0; c < 6; ++c) part[c] = warp_sum(part[c]);
      if (lane < 6) {
        const double *T = Ti + 36 * k;
        double v = 0.0;
#pragma unroll
        for (int c = 0; c < 6; ++c)
          if (c >= lane) v += T[c * 6 + lane] * (w[6 * k + c] - part[c]);
        y[6 * k + lane] = v;
      }
      __syncwarp();
    }
  }
  __syncthreads();
  for (int i = tid; i < C6; i += SPC_THREADS) {
    const double v = y[i];
    if (!isfinite(v)) st->lin_fail = 1;
    a.ypos[6 * (size_t)k0 + i] = v;
    a.yc[6 * (size_t)a.perm[k0 + i / 6] + i % 6] = v;
  }
}

// ---------------------------------------------------------------------------------------------
// The whole linear solve in ONE launch: a persistent grid (one thread block per SM) works through a queue of items --
// factor(node), update(node, tile), solve(node) -- in an order in which every item follows the items it depends on
// (levels bottom-up for the factorisation, top-down for the backward substitution).  A block takes the next item from
// a ticket counter and waits on integer completion counters in global memory:
//     factor(n)     after every update tile of every child of n
//     update(n, t)  after factor(n)
//     solve(n)      after solve(parent(n))   (roots: after their own factor)
// Items are handed out dynamically, so an item is only ever held by a RUNNING block and every item it waits for has a
// smaller queue index, i.e. was taken earlier by a running block: no deadlock, whatever the number of resident blocks.
// Compared with one launch per tree level this removes 3 x levels launches and, more important, lets a node start as
// soon as ITS children are done instead of when the slowest node of the level below is: the linear solve is bound by
// the longest root-to-leaf chain of the tree, not by the sum of the per-level maxima.
// The queue is built on the host (spq_cholesky, ba_sparse_symbolic.h; tests/test_tree_queue_order.py checks the order).
// Counters are zeroed by the host before the launch; producers publish with a device-scope fence before the counter
// update, consumers read other blocks' results through L2 (__ldcg).
// ---------------------------------------------------------------------------------------------
struct SpTree {
  const int2 *queue;       // (node, kind): kind >= 0 update tile, -1 factor, -2 solve
  int n_items;
  const int32_t *tiles;    // update tiles per node (0: no border)
  int *ticket, *fdone, *udone, *sdone;
};
template <int NR>
__global__ void __launch_bounds__(SPC_THREADS, 1)
k_spchol_tree(SpChol a, SpTree t, LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  extern __shared__ __align__(16) double spc_sm[];
  __shared__ int s_item;
  const int tid = threadIdx.x;
  for (;;) {
    const int it = spc_take(t.ticket, &s_item);
    if (it >= t.n_items) return;
    const int2 q = t.queue[it];
    const int id = q.x;
    const int32_t *N = a.node + (size_t)id * SPSYM_NODE_INTS;
    if (q.y == -1) {
      spc_factor_node<NR>(a, id, it == 0, st, spc_sm, t.udone, t.tiles);
      spc_publish(t.fdone + id, false);
    } else if (q.y >= 0) {
      if (tid == 0) spc_wait_ge(t.fdone + id, 1);
      __syncthreads();
      spc_update_node<NR>(a, id, q.y, t.tiles[id], spc_sm);
      spc_publish(t.udone + id, true);
    } else {
      if (tid == 0) {
        const int par = N[SPN_PARENT];
        if (par >= 0)
          spc_wait_ge(t.sdone + par, 1);
        else
          spc_wait_ge(t.fdone + id, 1);
      }
      __syncthreads();
      spc_solve_node(a, id, st, spc_sm);
      spc_publish(t.sdone + id, false);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Distributed factorisation (one subtree group per rank, top part replicated): the step is assembled by ONE all-reduce
// over yc -- every camera's six values are non-zero on exactly one rank (own subtrees; the top part's cameras, which
// every rank computed bit-identically, are kept by rank 0 only), so the sum is exact and identical on all ranks.  The
// linear-solver failure flag rides in the extra slot yc[6 n_cam].
// ---------------------------------------------------------------------------------------------
__global__ void k_spchol_dist_pre(int n_cam, int n_top, const int32_t *topcams, int rank, double *yc, LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (rank != 0 && i < 6 * n_top) yc[6 * (size_t)topcams[i / 6] + i % 6] = 0.0;
  if (i == 0) yc[6 * (size_t)n_cam] = st->lin_fail ? 1.0 : 0.0;
}
__global__ void k_spchol_dist_post(int n_cam, const double *yc, LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  if (threadIdx.x == 0 && yc[6 * (size_t)n_cam] != 0.0) st->lin_fail = 1;
}

// ---------------------------------------------------------------------------------------------
// Sparse Cholesky of the REF / DEPTH / INTR cost (depth prior and / or free intrinsics, planes store): the explicit path's
// per-observation W = Jc^T Jp and WV = W V^-1 (k_obs_W, already Jacobi-scaled) summed into the device-built block structure
// (build_pair_blocks), the camera-intrinsics border B, the corner C and the right-hand side assembled by camera, and the
// 4 x 4 border system solved between the forward and the backward substitution.
// ---------------------------------------------------------------------------------------------
// values of S from the planes: one warp per block, S_b = -sum_pairs WV_a W_b^T in the fixed pair order of the block
// (lanes stride the pairs, then the recursive-halving warp sum); k_sp_add_diag then puts U on the diagonal blocks
__global__ void __launch_bounds__(BA_THREADS)
k_sp_schur_planes(int n_blk, const int32_t *__restrict__ blk_ptr, const unsigned long long *__restrict__ pairs,
                  const double *__restrict__ W, const double *__restrict__ WV, double *__restrict__ S, const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  const int b = (int)((blockIdx.x * (size_t)BA_THREADS + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (b >= n_blk) return;
  double acc[36];
#pragma unroll
  for (int k = 0; k < 36; ++k) acc[k] = 0.0;
  const int e1 = blk_ptr[b + 1];
  for (int e = blk_ptr[b] + lane; e < e1; e += 32) {
    const unsigned long long pr = __ldg(pairs + e);
    const double *wv = WV + 18 * (size_t)(pr >> 32), *w = W + 18 * (size_t)(pr & 0xffffffffu);
    double A[18], B[18];
#pragma unroll
    for (int k = 0; k < 18; ++k) {
      A[k] = __ldg(wv + k);
      B[k] = __ldg(w + k);
    }
#pragma unroll
    for (int r = 0; r < 6; ++r)
#pragma unroll
      for (int c = 0; c < 6; ++c) acc[r * 6 + c] += A[3 * r] * B[3 * c] + A[3 * r + 1] * B[3 * c + 1] + A[3 * r + 2] * B[3 * c + 2];
  }
  int idx, cnt;
  sp_reduce_scatter36(acc, lane, idx, cnt);
  double *Sb = S + 36 * (size_t)b + idx;
  if (cnt > 0) Sb[0] = -acc[0];
  if (cnt > 1) Sb[1] = -acc[1];
}

// right-hand side, border and corner by camera: k_explicit_assemble<NK>'s arithmetic with the destinations of the sparse
// solve.  b[6 c] = -g_c + W V^-1 g_p; (NK) B[24 c] = U_ck - sum WV Wk^T (zero for the fixed camera), kk[0..15] = C (damped),
// kk[16..19] = b_k.  Item partials are added in item order, point-tile partials in tile order.
template <int NK>
__global__ void __launch_bounds__(BA_THREADS)
k_spb_assemble(int n_cam, int fixed_cam, const int32_t *__restrict__ item_ptr, const double *__restrict__ part_cam, int nblk_pt,
               const double *__restrict__ part_kk, const double *__restrict__ gc, const double *__restrict__ Uck,
               const double *__restrict__ Ukk, const double *__restrict__ gk, const double *__restrict__ dk, double *__restrict__ b,
               double *__restrict__ Bc, double *__restrict__ kk, const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  constexpr int NV = 6 + (NK ? 24 : 0);
  const int idx = blockIdx.x * BA_THREADS + threadIdx.x;
  if (idx < n_cam * NV) {
    const int c = idx / NV, k = idx - c * NV;
    const bool fixed = c == fixed_cam;
    double acc = 0.0;
    for (int it = item_ptr[c]; it < item_ptr[c + 1]; ++it) acc += part_cam[(size_t)it * NV + k];
    if (k < 6)
      b[6 * (size_t)c + k] = fixed ? 0.0 : -gc[6 * (size_t)c + k] + acc;
    else if (NK)
      Bc[24 * (size_t)c + k - 6] = fixed ? 0.0 : Uck[24 * (size_t)c + k - 6] - acc;
  } else if (NK && idx < n_cam * NV + 14) {
    const int k = idx - n_cam * NV;
    double v = 0.0;
    for (int t = 0; t < nblk_pt; ++t) v += part_kk[14 * (size_t)t + k];
    if (k < 10) {
      int a = 0, r = k;  // k-th entry of the row-major upper triangle of the 4 x 4 block -> (a, b)
      while (r >= 4 - a) {
        r -= 4 - a;
        ++a;
      }
      const int b2 = a + r;
      double x = Ukk[a * 4 + b2] - v;
      if (a == b2) {
        const double D = sqrt(dk[a] / st->radius);
        x += D * D;
      }
      kk[a * 4 + b2] = x;
      kk[b2 * 4 + a] = x;
    } else {
      kk[16 + k - 10] = -gk[k - 10] + v;
    }
  }
}

// border reduction after the forward substitution: per thread block, over its elimination positions (one per thread),
// Z^T Z (10 upper entries) and Z^T z (4), block sums in a fixed tree -> part[14 blockIdx.x ..]
__global__ void __launch_bounds__(BA_THREADS)
k_spb_reduce(int n_pos, const double *__restrict__ Zb, const double *__restrict__ z, double *__restrict__ part, const LmState *st,
             int gate) {
  if (!gate_open(st, gate)) return;
  __shared__ double red[BA_WARPS + 1];
  const int p = blockIdx.x * BA_THREADS + threadIdx.x;
  double v[14];
#pragma unroll
  for (int k = 0; k < 14; ++k) v[k] = 0.0;
  if (p < n_pos) {
#pragma unroll
    for (int r = 0; r < 6; ++r) {
      double zr[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) zr[q] = __ldcg(Zb + 4 * (6 * (size_t)p + r) + q);
      const double zz = __ldcg(z + 6 * (size_t)p + r);
      int u = 0;
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int c = a; c < 4; ++c) v[u++] += zr[a] * zr[c];
#pragma unroll
      for (int a = 0; a < 4; ++a) v[10 + a] += zr[a] * zz;
    }
  }
#pragma unroll
  for (int k = 0; k < 14; ++k) {
    const double s = block_sum(v[k], red);
    if (threadIdx.x == 0) part[14 * (size_t)blockIdx.x + k] = s;
  }
}

// the border system, one warp: partials added in block order, T = C - Z^T Z, t = b_k - Z^T z, y_k = T^-1 t by a 4 x 4
// Cholesky.  A non-positive or non-finite pivot sets lin_fail (y_k = 0 then).
__global__ void __launch_bounds__(32)
k_spb_solve(int nblk, const double *__restrict__ part, const double *__restrict__ kk, double *__restrict__ yk, LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  __shared__ double s[14];
  const int lane = threadIdx.x;
  if (lane < 14) {
    double v = 0.0;
    for (int b = 0; b < nblk; ++b) v += __ldcg(part + 14 * (size_t)b + lane);
    s[lane] = v;
  }
  __syncwarp();
  if (lane != 0) return;
  double T[4][4], t[4];
  int u = 0;
  for (int a = 0; a < 4; ++a)
    for (int c = a; c < 4; ++c) {
      T[a][c] = kk[a * 4 + c] - s[u++];
      T[c][a] = T[a][c];
    }
  for (int a = 0; a < 4; ++a) t[a] = kk[16 + a] - s[10 + a];
  bool ok = true;
  for (int j = 0; j < 4; ++j) {  // L in the lower triangle of T
    double d = T[j][j];
    for (int k = 0; k < j; ++k) d -= T[j][k] * T[j][k];
    if (!(d > 0.0) || !isfinite(d)) {
      ok = false;
      break;
    }
    T[j][j] = sqrt(d);
    for (int i = j + 1; i < 4; ++i) {
      double x = T[i][j];
      for (int k = 0; k < j; ++k) x -= T[i][k] * T[j][k];
      T[i][j] = x / T[j][j];
    }
  }
  double y[4] = {0.0, 0.0, 0.0, 0.0};
  if (ok) {
    for (int i = 0; i < 4; ++i) {
      double x = t[i];
      for (int k = 0; k < i; ++k) x -= T[i][k] * y[k];
      y[i] = x / T[i][i];
    }
    for (int i = 3; i >= 0; --i) {
      double x = y[i];
      for (int k = i + 1; k < 4; ++k) x -= T[k][i] * y[k];
      y[i] = x / T[i][i];
    }
    for (int i = 0; i < 4; ++i) ok = ok && isfinite(y[i]);
  }
  if (!ok) {
    st->lin_fail = 1;
    for (int i = 0; i < 4; ++i) y[i] = 0.0;
  }
  for (int i = 0; i < 4; ++i) yk[i] = y[i];
}
