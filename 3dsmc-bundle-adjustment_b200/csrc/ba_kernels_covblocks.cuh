// ba_kernels_covblocks.cuh -- covariance of ANY two parameter blocks (ba_gpu_covariance_blocks): camera pairs that share no
// point, camera-point, point-point, and everything ba_gpu_covariance returns, without the selected inversion.
//
// With A = L L^T (the supernodal factor of ba_kernels_spchol.cuh, Jacobi-scaled, zero damping) and E_c the six unit columns of
// camera c, F_c = L^-1 E_c is non-zero only on the own rows of the nodes on the path from c's node to its root, and
//     (A^-1)_ab = F_a^T F_b = sum over the nodes common to both paths (the lowest common ancestor .. the root) of F_a[n]^T F_b[n].
// The intrinsics border adds X_a T^-1 X_b^T (X = L^-T Z, T = C - Z^T Z: ba_kernels_selinv.cuh), and the points follow from the
// reduced-camera blocks: Sigma(R, p) = -Sigma_RR W_p V_p^-1, Sigma(p, q) = delta_pq V_p^-1 + V_p^-1 W_p^T Sigma_RR W_q V_q^-1.
//
// k_cb_forward: the multi-source forward substitution F_s = L^-1 E_s.  Items (node, group of up to CB_GROUP sources whose
// paths pass through the node), one tree level per launch, bottom-up.  An item builds each source's front right-hand side --
// E_s at the source's own node, otherwise the border part that the child on the source's path carried up, through the
// child's rel / inv maps -- solves the own block with the panel and the stored inverse pivot blocks (left-looking), stores
// z_O into F and carries r_B - L_BO z_O to the parent.  SIMT: every column's arithmetic has a fixed order that does not
// depend on the group, the pass or the thread mapping, so a source's F has the same bits whatever else is requested.
// k_cb_blocks: one warp per requested block, in the canonical orientation (camera < point < intrinsics, then index); path dot
// products root to lca, rows ascending; the point compositions on the fly; unscaled.  No float atomics.
#pragma once
#include "ba_kernels_selinv.cuh"

#define CB_THREADS 128
#define CB_GROUP 8               // sources per forward item (48 right-hand-side columns)
#define CB_WARPS (CB_THREADS / 32)
#define CB_ENT_INTS 8            // path entry: node, previous entry (-1 at the source's node), own block of the source there
                                 // (-1 elsewhere), F offset, carry offset (6x6 blocks), node level, 2 unused
inline size_t cb_forward_smem(int max_m) { return ((size_t)6 * max_m + 6) * 6 * CB_GROUP * 8; }

struct CbFwd {
  const int32_t *node, *rel, *inv;
  const double *panel, *linv;
  const int32_t *ent;
  const int2 *items;  // (first entry, entries): consecutive entries of one node
  double *F, *carry;  // F: C6 x 6 row-major per entry; carry: NB6 x 6 row-major per entry
};

__global__ void __launch_bounds__(CB_THREADS) k_cb_forward(CbFwd a, int item0) {
  extern __shared__ __align__(16) double cb_sm[];
  __shared__ int s_own[CB_GROUP], s_f[CB_GROUP], s_c[CB_GROUP], s_pc[CB_GROUP], s_pn[CB_GROUP];
  const int tid = threadIdx.x;
  const int2 it = a.items[item0 + blockIdx.x];
  const int g = it.y, nc = 6 * g;
  const int32_t *E0 = a.ent + (size_t)CB_ENT_INTS * it.x;
  const int id = E0[0];
  const int32_t *N = a.node + (size_t)id * SPSYM_NODE_INTS;
  const int k0 = N[SPN_K0], m = N[SPN_M], nb = N[SPN_NB];
  const int LD = 6 * (m + nb), C6 = 6 * m, NB6 = 6 * nb;
  const double *Pg = a.panel + 36 * spc_off(N, SPN_PANEL_LO);
  double *z = cb_sm;                 // own rows, z[R * nc + col]
  double *v = z + (size_t)C6 * nc;   // the current pivot block's rows before the pivot inverse, v[r * nc + col]
  if (tid < g) {
    const int32_t *E = E0 + CB_ENT_INTS * tid;
    s_own[tid] = E[2];
    s_f[tid] = E[3];
    s_c[tid] = E[4];
    const int prev = E[1];
    s_pn[tid] = prev >= 0 ? a.ent[(size_t)CB_ENT_INTS * prev] : -1;          // child on the path
    s_pc[tid] = prev >= 0 ? a.ent[(size_t)CB_ENT_INTS * prev + 4] : 0;       // its carry
  }
  for (int i = tid; i < C6 * nc; i += CB_THREADS) z[i] = 0.0;
  __syncthreads();
  // right-hand side of the own rows: E_s, or the child's carried border rows that are own cameras here
  for (int j = 0; j < g; ++j) {
    if (s_own[j] >= 0) {
      if (tid < 6) z[(size_t)(6 * s_own[j] + tid) * nc + 6 * j + tid] = 1.0;
    } else {
      const int32_t *Cn = a.node + (size_t)s_pn[j] * SPSYM_NODE_INTS;
      const int32_t *rel = a.rel + Cn[SPN_REL];
      const double *cr = a.carry + 36 * (size_t)s_pc[j];
      for (int idx = tid; idx < 36 * Cn[SPN_NB]; idx += CB_THREADS) {
        const int i = idx / 36, t = idx - 36 * i, x = t / 6, c = t - 6 * x, ri = __ldg(rel + i);
        if (ri < m) z[(size_t)(6 * ri + x) * nc + 6 * j + c] = __ldcg(cr + idx);
      }
    }
  }
  __syncthreads();
  // own block, left-looking: v = r_k - L_k,<k z_<k, z_k = T_k v
  for (int k = 0; k < m; ++k) {
    for (int idx = tid; idx < 6 * nc; idx += CB_THREADS) {
      const int r = idx / nc, col = idx - r * nc, R = 6 * k + r;
      double s = z[(size_t)R * nc + col];
      for (int c = 0; c < 6 * k; ++c) s -= __ldg(Pg + (size_t)c * LD + R) * z[(size_t)c * nc + col];
      v[idx] = s;
    }
    __syncthreads();
    const double *T = a.linv + 36 * (size_t)(k0 + k);
    for (int idx = tid; idx < 6 * nc; idx += CB_THREADS) {
      const int l = idx / nc, col = idx - l * nc;
      double s = 0.0;
      for (int c = 0; c <= l; ++c) s += __ldg(T + 6 * l + c) * v[(size_t)c * nc + col];
      z[(size_t)(6 * k + l) * nc + col] = s;
    }
    __syncthreads();
  }
  for (int idx = tid; idx < C6 * nc; idx += CB_THREADS) {
    const int R = idx / nc, col = idx - R * nc, j = col / 6;
    a.F[36 * (size_t)s_f[j] + 6 * R + (col - 6 * j)] = z[idx];
  }
  // border rows: r_B (the child's carried rows that are border cameras here, through inv) - L_BO z_O
  for (int idx = tid; idx < NB6 * nc; idx += CB_THREADS) {
    const int Rb = idx / nc, col = idx - Rb * nc, j = col / 6, c = col - 6 * j, i = Rb / 6;
    double s = 0.0;
    if (s_own[j] < 0) {
      const int32_t *Cn = a.node + (size_t)s_pn[j] * SPSYM_NODE_INTS;
      const int ii = __ldg(a.inv + Cn[SPN_INV] + i);
      if (ii >= 0) s = __ldcg(a.carry + 36 * (size_t)s_pc[j] + 36 * ii + 6 * (Rb - 6 * i) + c);
    }
    const double *lb = Pg + C6 + Rb;
    for (int c2 = 0; c2 < C6; ++c2) s -= __ldg(lb + (size_t)c2 * LD) * z[(size_t)c2 * nc + col];
    a.carry[36 * (size_t)s_c[j] + 6 * Rb + c] = s;
  }
}

// observation slots of the requested points: (first slot, slot count) per point, then the cameras of those slots
__global__ void __launch_bounds__(BA_THREADS)
k_cb_obs_range(int n, const int32_t *__restrict__ pts, const int32_t *__restrict__ pt_rowptr, int2 *__restrict__ out) {
  const int i = blockIdx.x * BA_THREADS + threadIdx.x;
  if (i < n) out[i] = make_int2(pt_rowptr[pts[i]], pt_rowptr[pts[i] + 1] - pt_rowptr[pts[i]]);
}
__global__ void __launch_bounds__(BA_THREADS)
k_cb_obs_cams(int n, const int32_t *__restrict__ slot, const int32_t *__restrict__ pm_cam, int32_t *__restrict__ out) {
  const int i = blockIdx.x * BA_THREADS + threadIdx.x;
  if (i < n) out[i] = pm_cam[slot[i]];
}

enum { CB_CAM = 0, CB_PT = 1, CB_INTR = 2 };  // (== BA_COV_CAMERA / POINT / INTRINSICS)

struct CbBlk {
  const int32_t *ent, *src_ptr, *src_ent, *cam_src, *node;
  const double *F;
  const int32_t *pos;
  const double *X, *Tinv;
  int nk, n_cam, fixed_cam;
  const int32_t *pt_rowptr, *pm_cam, *perm;
  const double *W, *Wk, *Vinv, *sc, *sp, *sk;
  const int4 *req;          // canonical (kind a, index a, kind b, index b)
  const long long *off;     // output offset in doubles; bit 62 set: the caller asked for (b, a) -- write the transpose
  int n_req;
  double *out;
};

// scaled Sigma(a, b) of two free cameras into S (row-major 6x6), by the calling warp: lane < 18 owns entries 2 lane, 2 lane + 1
__device__ __forceinline__ void cb_cc(const CbBlk &a, int ca, int cb, double *S, int lane) {
  if (lane < 18) {
    const int x = (2 * lane) / 6, y = 2 * lane - 6 * x;
    const int sa = a.cam_src[ca], sb = a.cam_src[cb];
    const int pa = a.src_ptr[sa], pb = a.src_ptr[sb];
    int i = a.src_ptr[sa + 1] - pa - 1, j = a.src_ptr[sb + 1] - pb - 1;
    double s0 = 0.0, s1 = 0.0;
    // root to lca (paths are stored bottom-up); different roots: no common node
    while (i >= 0 && j >= 0) {
      const int32_t *Ea = a.ent + (size_t)CB_ENT_INTS * a.src_ent[pa + i], *Eb = a.ent + (size_t)CB_ENT_INTS * a.src_ent[pb + j];
      if (Ea[0] != Eb[0]) break;
      const int C6 = 6 * a.node[(size_t)Ea[0] * SPSYM_NODE_INTS + SPN_M];
      const double *fa = a.F + 36 * (size_t)Ea[3] + x, *fb = a.F + 36 * (size_t)Eb[3] + y;
      for (int R = 0; R < C6; ++R) {
        const double va = fa[6 * R];
        s0 += va * fb[6 * R];
        s1 += va * fb[6 * R + 1];
      }
      --i;
      --j;
    }
    if (a.nk) {
      const size_t n6 = 6 * (size_t)a.n_cam, ra = 6 * (size_t)a.pos[ca] + x, rb = 6 * (size_t)a.pos[cb] + y;
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        double t0 = 0.0, t1 = 0.0;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          t0 += a.Tinv[p * 4 + q] * a.X[q * n6 + rb];
          t1 += a.Tinv[p * 4 + q] * a.X[q * n6 + rb + 1];
        }
        s0 += a.X[p * n6 + ra] * t0;
        s1 += a.X[p * n6 + ra] * t1;
      }
    }
    S[6 * x + y] = s0;
    S[6 * x + y + 1] = s1;
  }
  __syncwarp();
}

// scaled Sigma(c, k) = -X_c T^-1 of a free camera into S (row-major 6x4): k_cov_cam's arithmetic
__device__ __forceinline__ void cb_ck(const CbBlk &a, int c, double *S, int lane) {
  if (lane < 24) {
    const int x = lane / 4, k = lane - 4 * x;
    const size_t n6 = 6 * (size_t)a.n_cam, rc = 6 * (size_t)a.pos[c] + x;
    double s = 0.0;
#pragma unroll
    for (int p = 0; p < 4; ++p) s += a.X[p * n6 + rc] * a.Tinv[p * 4 + k];
    S[lane] = -s;
  }
  __syncwarp();
}

__device__ __forceinline__ void cb_vinv(const double *Vinv, int p, double V[3][3]) {
  const double *vp = Vinv + 6 * (size_t)p;
  V[0][0] = vp[0]; V[0][1] = vp[1]; V[0][2] = vp[2];
  V[1][0] = vp[1]; V[1][1] = vp[3]; V[1][2] = vp[4];
  V[2][0] = vp[2]; V[2][1] = vp[4]; V[2][2] = vp[5];
}

__global__ void __launch_bounds__(CB_THREADS) k_cb_blocks(CbBlk a) {
  __shared__ double s_S[CB_WARPS][36], s_A[CB_WARPS][36];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int r = blockIdx.x * CB_WARPS + w;
  if (r >= a.n_req) return;
  double *S = s_S[w], *A = s_A[w];
  const int4 q = a.req[r];
  const long long o = a.off[r];
  const bool flip = (o >> 62) & 1;
  double *out = a.out + (o & ((1ll << 62) - 1));
  const int da = q.x == CB_CAM ? 6 : q.x == CB_PT ? 3 : 4, db = q.z == CB_CAM ? 6 : q.z == CB_PT ? 3 : 4;
  const bool fa = q.x == CB_CAM && q.y == a.fixed_cam, fb = q.z == CB_CAM && q.w == a.fixed_cam;
  // value (x, y) of the canonical block (da x db) goes to out[x db + y], or to out[y da + x] when flipped
  auto put = [&](int x, int y, double v) { out[flip ? y * da + x : x * db + y] = v; };
  if (fa || fb || (!a.nk && (q.x == CB_INTR || q.z == CB_INTR))) {  // constant blocks
    for (int e = lane; e < da * db; e += 32) out[e] = 0.0;
    return;
  }
  if (q.x == CB_CAM && q.z == CB_CAM) {
    cb_cc(a, q.y, q.w, S, lane);
    for (int e = lane; e < 36; e += 32) {
      int x = e / 6, y = e - 6 * x;
      const double v = q.y == q.w && x > y ? S[6 * y + x] : S[e];  // (a diagonal block: its upper triangle, mirrored)
      put(x, y, v * (a.sc[6 * (size_t)q.y + x] * a.sc[6 * (size_t)q.w + y]));
    }
  } else if (q.x == CB_CAM && q.z == CB_INTR) {
    cb_ck(a, q.y, S, lane);
    if (lane < 24) put(lane / 4, lane % 4, S[lane] * (a.sc[6 * (size_t)q.y + lane / 4] * a.sk[lane % 4]));
  } else if (q.x == CB_INTR) {
    if (lane < 16) put(lane / 4, lane % 4, a.Tinv[lane] * (a.sk[lane / 4] * a.sk[lane % 4]));
  } else if (q.x == CB_CAM && q.z == CB_PT) {
    // Sigma(a, p) = -(sum_o Sigma(a, c_o) W_o + Sigma(a, k) W_k) V_p^-1
    const int c = q.y, p = q.w, x = lane / 3, y = lane - 3 * (lane / 3);
    double acc = 0.0;
    for (int sl = a.pt_rowptr[p]; sl < a.pt_rowptr[p + 1]; ++sl) {
      const int co = a.pm_cam[sl];
      if (co == a.fixed_cam) continue;
      cb_cc(a, c, co, S, lane);
      if (lane < 18) {
        const double *Wo = a.W + 18 * (size_t)a.perm[sl];
        double t = 0.0;
#pragma unroll
        for (int k = 0; k < 6; ++k) t += S[6 * x + k] * Wo[3 * k + y];
        acc += t;
      }
      __syncwarp();
    }
    if (a.nk) {
      cb_ck(a, c, S, lane);
      if (lane < 18) {
        double t = 0.0;
#pragma unroll
        for (int k = 0; k < 4; ++k) t += S[4 * x + k] * a.Wk[12 * (size_t)p + 3 * k + y];
        acc += t;
      }
    }
    if (lane < 18) A[lane] = acc;
    __syncwarp();
    if (lane < 18) {
      double V[3][3];
      cb_vinv(a.Vinv, p, V);
      const double v = -(A[3 * x] * V[0][y] + A[3 * x + 1] * V[1][y] + A[3 * x + 2] * V[2][y]);
      put(x, y, v * (a.sc[6 * (size_t)c + x] * a.sp[3 * (size_t)p + y]));
    }
  } else if (q.x == CB_PT && q.z == CB_INTR) {
    // Sigma(p, k) = -V_p^-1 (sum_o W_o^T Sigma(c_o, k) + W_k^T Sigma_kk)
    const int p = q.y, x = lane / 4, k = lane - 4 * (lane / 4);
    double acc = 0.0;
    for (int sl = a.pt_rowptr[p]; sl < a.pt_rowptr[p + 1]; ++sl) {
      const int co = a.pm_cam[sl];
      if (co == a.fixed_cam) continue;
      cb_ck(a, co, S, lane);
      if (lane < 12) {
        const double *Wo = a.W + 18 * (size_t)a.perm[sl];
        double t = 0.0;
#pragma unroll
        for (int u = 0; u < 6; ++u) t += Wo[3 * u + x] * S[4 * u + k];
        acc += t;
      }
      __syncwarp();
    }
    if (lane < 12) {
      double t = 0.0;
#pragma unroll
      for (int l = 0; l < 4; ++l) t += a.Wk[12 * (size_t)p + 3 * l + x] * a.Tinv[4 * l + k];
      A[lane] = acc + t;
    }
    __syncwarp();
    if (lane < 12) {
      double V[3][3];
      cb_vinv(a.Vinv, p, V);
      const double v = -(V[x][0] * A[k] + V[x][1] * A[4 + k] + V[x][2] * A[8 + k]);
      put(x, k, v * (a.sp[3 * (size_t)p + x] * a.sk[k]));
    }
  } else {
    // Sigma(p, q) = delta_pq V_p^-1 + V_p^-1 M V_q^-1, M = W_p^T Sigma_RR W_q (camera pairs, then the intrinsics terms)
    const int p = q.y, pq = q.w, x = lane / 3, y = lane - 3 * (lane / 3);
    const double *wkp = a.Wk + 12 * (size_t)p, *wkq = a.Wk + 12 * (size_t)pq;
    double M = 0.0;
    for (int s1 = a.pt_rowptr[p]; s1 < a.pt_rowptr[p + 1]; ++s1) {
      const int c1 = a.pm_cam[s1];
      if (c1 == a.fixed_cam) continue;
      const double *W1 = a.W + 18 * (size_t)a.perm[s1];
      for (int s2 = a.pt_rowptr[pq]; s2 < a.pt_rowptr[pq + 1]; ++s2) {
        const int c2 = a.pm_cam[s2];
        if (c2 == a.fixed_cam) continue;
        cb_cc(a, c1, c2, S, lane);
        if (lane < 9) {
          const double *W2 = a.W + 18 * (size_t)a.perm[s2];
          double t = 0.0;
#pragma unroll
          for (int k = 0; k < 6; ++k) {
            double u = 0.0;
#pragma unroll
            for (int l = 0; l < 6; ++l) u += S[6 * k + l] * W2[3 * l + y];
            t += W1[3 * k + x] * u;
          }
          M += t;
        }
        __syncwarp();
      }
      if (a.nk) {  // W_o^T Sigma(c_o, k) W_kq
        cb_ck(a, c1, S, lane);
        if (lane < 9) {
          double t = 0.0;
#pragma unroll
          for (int k = 0; k < 6; ++k) {
            double u = 0.0;
#pragma unroll
            for (int l = 0; l < 4; ++l) u += S[4 * k + l] * wkq[3 * l + y];
            t += W1[3 * k + x] * u;
          }
          M += t;
        }
        __syncwarp();
      }
    }
    if (a.nk) {
      for (int s2 = a.pt_rowptr[pq]; s2 < a.pt_rowptr[pq + 1]; ++s2) {  // W_kp^T Sigma(k, c_o') W_o'
        const int c2 = a.pm_cam[s2];
        if (c2 == a.fixed_cam) continue;
        cb_ck(a, c2, S, lane);
        if (lane < 9) {
          const double *W2 = a.W + 18 * (size_t)a.perm[s2];
          double t = 0.0;
#pragma unroll
          for (int l = 0; l < 4; ++l) {
            double u = 0.0;
#pragma unroll
            for (int k = 0; k < 6; ++k) u += S[4 * k + l] * W2[3 * k + y];
            t += wkp[3 * l + x] * u;
          }
          M += t;
        }
        __syncwarp();
      }
      if (lane < 9) {  // W_kp^T T^-1 W_kq
        double t = 0.0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          double u = 0.0;
#pragma unroll
          for (int l = 0; l < 4; ++l) u += a.Tinv[4 * k + l] * wkq[3 * l + y];
          t += wkp[3 * k + x] * u;
        }
        M += t;
      }
    }
    if (lane < 9) A[lane] = M;
    __syncwarp();
    double Vp[3][3], Vq[3][3];
    cb_vinv(a.Vinv, p, Vp);
    cb_vinv(a.Vinv, pq, Vq);
    if (lane < 9) S[lane] = Vp[x][0] * A[y] + Vp[x][1] * A[3 + y] + Vp[x][2] * A[6 + y];  // V_p^-1 M
    __syncwarp();
    if (lane < 9) {
      const int xx = p == pq && x > y ? y : x, yy = p == pq && x > y ? x : y;  // (a diagonal block: upper triangle, mirrored)
      double v = S[3 * xx] * Vq[0][yy] + S[3 * xx + 1] * Vq[1][yy] + S[3 * xx + 2] * Vq[2][yy];
      if (p == pq) v += Vp[xx][yy];
      put(x, y, v * (a.sp[3 * (size_t)p + xx] * a.sp[3 * (size_t)pq + yy]));
    }
  }
}
