// ba_kernels.cuh -- hand-written sm_100a kernels of the windowed-BA hot path.
//
// Replaces what ceres::Solve does for the reference's problem
// (src/OptimizationUtils.cpp:300): residual + Jacobian evaluation of the cost
// functors (:25-49, :72-94, :116-125) chained with the SE3 local
// parameterisation (headers/sophus/local_parameterization_se3.hpp:17-37), Huber
// correction, normal-equation blocks, Schur complement, linear solve and the
// Levenberg-Marquardt controller.  fp64 throughout, no global floating-point
// atomics: every reduction has a fixed order.  Tensor cores only where a block is a
// dense fp64 contraction: k_sp_schur (ba_kernels_sparse.cuh) sums with fp64 DMMA.
//
// Gating: every kernel of the LM pipeline first looks at the device-resident
// controller state, so the host can enqueue whole iterations without waiting
// for the accept/reject decision.
#pragma once
#include "ba_common.cuh"

enum { GATE_RUN = 0, GATE_ACCEPTED = 1, GATE_PCG = 2, GATE_PCG_RESET = 3, GATE_SCALE = 4 };

// Programmatic dependent launch: the windowed LM iteration is a chain of ~20 small dependent kernels, so every kernel of
// the iteration is launched with programmatic stream serialisation (ba_gpu.cu: LAUNCH with ctx->pdl).  Its CTAs may become
// resident while the previous kernel still runs; nothing is read or written before this wait returns (= the previous
// grid has completed and its writes are visible), and the kernel's own dependents are released at once, so their launch
// latency overlaps this kernel's execution.  Without the launch attribute both instructions are no-ops.
__device__ __forceinline__ void pdl_wait() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

__device__ __forceinline__ bool gate_open(const LmState *st, int gate, int reset_period = 0) {
  pdl_wait();
  if (st->done) return false;
  switch (gate) {
    case GATE_ACCEPTED: return st->accepted != 0;
    case GATE_PCG: return st->pcg_done == 0;
    case GATE_PCG_RESET: return st->pcg_done == 0 && reset_period > 0 && (st->pcg_it % reset_period) == 0;
    case GATE_SCALE: return st->have_scale == 0;
    default: return true;
  }
}

// =====================================================================
// Index construction (device-built, integer-exact)
// =====================================================================
// histogram of pt_idx / cam_idx + validation (camera-sorted, in range)
// The camera CSR comes straight from the sorted camera list (cam_rowptr[c] = first observation with camera >= c: the
// thread at a camera boundary writes the pointers of the cameras that start there), not from a histogram: 8 M atomic
// increments on 10 k counters, 32 lanes of a warp on the same address, took 1.0 ms at config 5.
__global__ void __launch_bounds__(BA_THREADS) k_index_count(int n_obs, int n_cam, int n_pt, const int32_t *__restrict__ cam_idx,
                                                           const int32_t *__restrict__ pt_idx, int32_t *pt_cnt,
                                                           int32_t *cam_rowptr, int32_t *err) {
  const int i = blockIdx.x * BA_THREADS + threadIdx.x;
  if (i >= n_obs) return;
  const int c = cam_idx[i], p = pt_idx[i];
  const int prev = i > 0 ? cam_idx[i - 1] : -1;
  if (c < 0 || c >= n_cam || p < 0 || p >= n_pt || (i > 0 && c < prev)) {
    atomicOr(err, 1);
    return;
  }
  atomicAdd(&pt_cnt[p], 1);
  if (prev < c)  // (an invalid predecessor raises the error flag itself; the clamp only keeps these writes in range)
    for (int cc = prev < -1 ? 0 : prev + 1; cc <= c; ++cc) cam_rowptr[cc] = i;
  if (i == n_obs - 1)
    for (int cc = c + 1; cc <= n_cam; ++cc) cam_rowptr[cc] = n_obs;
}

// single-CTA exclusive scan: out[0..n] (n+1 entries) from cnt[0..n)
__global__ void __launch_bounds__(1024) k_exclusive_scan(int n, const int32_t *__restrict__ cnt, int32_t *__restrict__ out) {
  __shared__ int32_t wsum[32];
  __shared__ int32_t carry_s;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int base = 0; base < n; base += 1024) {
    const int i = base + threadIdx.x;
    const int v = i < n ? cnt[i] : 0;
    int x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(BA_FULL, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) wsum[w] = x;
    __syncthreads();
    if (w == 0) {
      int s = wsum[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(BA_FULL, s, o);
        if (lane >= o) s += y;
      }
      wsum[lane] = s;
    }
    __syncthreads();
    const int carry = carry_s;
    const int incl = x + (w > 0 ? wsum[w - 1] : 0) + carry;
    if (i < n) out[i] = incl - v;
    __syncthreads();
    if (threadIdx.x == 1023) carry_s = incl;
    __syncthreads();
  }
  if (threadIdx.x == 0) out[n] = carry_s;
}

// unordered bucket fill (integer atomics), made canonical by k_index_sort
// (same validity predicate as k_index_count: an observation that was not counted must not be filled either, or the
// cursor would run past its bucket / index outside the arrays before the host has read the error flag)
__global__ void __launch_bounds__(BA_THREADS) k_index_fill(int n_obs, int n_cam, int n_pt, const int32_t *__restrict__ cam_idx,
                                                          const int32_t *__restrict__ pt_idx,
                                                          const int32_t *__restrict__ pt_rowptr, int32_t *cursor,
                                                          int32_t *perm) {
  const int i = blockIdx.x * BA_THREADS + threadIdx.x;
  if (i >= n_obs) return;
  const int c = cam_idx[i], p = pt_idx[i];
  if (c < 0 || c >= n_cam || p < 0 || p >= n_pt || (i > 0 && c < cam_idx[i - 1])) return;
  const int pos = atomicAdd(&cursor[p], 1);
  perm[pt_rowptr[p] + pos] = i;
}
// ascending sort of every point's bucket == the STABLE counting sort of pt_idx
__global__ void __launch_bounds__(BA_THREADS) k_index_sort(int n_pt, const int32_t *__restrict__ pt_rowptr, int32_t *perm) {
  const int p = blockIdx.x * BA_THREADS + threadIdx.x;
  if (p >= n_pt) return;
  const int b = pt_rowptr[p], e = pt_rowptr[p + 1];
  for (int i = b + 1; i < e; ++i) {
    const int v = perm[i];
    int j = i - 1;
    while (j >= b && perm[j] > v) {
      perm[j + 1] = perm[j];
      --j;
    }
    perm[j + 1] = v;
  }
}
// point-major copies of the observation arrays
__global__ void __launch_bounds__(BA_THREADS) k_index_gather(int n_pt, int n_obs, const int32_t *__restrict__ pt_rowptr,
                                                            const int32_t *__restrict__ perm,
                                                            const int32_t *__restrict__ cam_idx, const double2 *__restrict__ uv,
                                                            const double *__restrict__ depth, int32_t *pm_cam, int32_t *pm_pt,
                                                            double2 *pm_uv, double *pm_depth) {
  const int p = blockIdx.x * BA_THREADS + threadIdx.x;
  if (p >= n_pt) return;
  for (int s = pt_rowptr[p]; s < pt_rowptr[p + 1]; ++s) {
    const int i = perm[s];
    pm_cam[s] = cam_idx[i];
    pm_pt[s] = p;
    pm_uv[s] = uv[i];
    if (depth) pm_depth[s] = depth[i];
  }
}
// camera-major work items: runs of <= item_obs (<= BA_ITEM_OBS) observations of one camera; small problems get
// shorter runs so that the warp-per-item kernels still fill the GPU (chosen at upload)
__global__ void __launch_bounds__(BA_THREADS) k_item_count(int n_cam, int item_obs, const int32_t *__restrict__ cam_rowptr, int32_t *item_cnt) {
  const int c = blockIdx.x * BA_THREADS + threadIdx.x;
  if (c >= n_cam) return;
  const int n = cam_rowptr[c + 1] - cam_rowptr[c];
  item_cnt[c] = (n + item_obs - 1) / item_obs;
}
__global__ void __launch_bounds__(BA_THREADS) k_item_fill(int n_cam, int item_obs, const int32_t *__restrict__ cam_rowptr,
                                                         const int32_t *__restrict__ item_ptr, BaItem *items) {
  const int c = blockIdx.x * BA_THREADS + threadIdx.x;
  if (c >= n_cam) return;
  const int b = cam_rowptr[c], e = cam_rowptr[c + 1];
  int k = item_ptr[c];
  for (int s = b; s < e; s += item_obs, ++k) {
    BaItem it;
    it.cam = c;
    it.begin = s;
    it.end = min(e, s + item_obs);
    it.pad = 0;
    items[k] = it;
  }
}

// =====================================================================
// Residuals + analytic Jacobians (the "Jacobian-eval" kernel)
// =====================================================================
// One thread per observation.  Algorithmic traffic NS mode: 208 B/obs
// (uv 16 + idx 8 + point 24 read; r 16 + Jc 96 + Jp 48 written).
//   r  = sqrt(w) (pi(K, R^T (p - t)) - z)             (:25-49)
//   rd = sqrt(wd) (d - Z)                             (:72-94)
//   d r / d delta = A [-I | [p_C]x]   (right perturbation T exp(delta))
//   d r / d p     = A R^T
// then Huber corrector sqrt(rho') and the Jacobi column scaling.
template <int DEPTH, int NK, int COST>
__global__ void __launch_bounds__(BA_THREADS)
k_linearize(int n_obs, const int32_t *__restrict__ cam_idx, const int32_t *__restrict__ pt_idx,
            const double2 *__restrict__ uv, const double *__restrict__ depth, const double *__restrict__ pose,
            const double *__restrict__ pt, const double *__restrict__ intr, const double *__restrict__ sc,
            const double *__restrict__ sp, const double *__restrict__ sk, CostParams cp, JPlanes J,
            double *__restrict__ cost_part, LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  __shared__ double red[BA_WARPS + 1];
  const int i = blockIdx.x * BA_THREADS + threadIdx.x;
  double cost = 0.0;
  if (i < n_obs) {
    const int c = cam_idx[i], p = pt_idx[i];
    const double *P = pose + 7 * (size_t)c;
    const double q[4] = {ldg1(P), ldg1(P + 1), ldg1(P + 2), ldg1(P + 3)};
    double R[9];
    quat_to_R(q, R);
    const double *X3 = pt + 3 * (size_t)p;
    const double d0 = ldg1(X3) - ldg1(P + 4), d1 = ldg1(X3 + 1) - ldg1(P + 5), d2 = ldg1(X3 + 2) - ldg1(P + 6);
    const double X = (R[0] * d0 + R[3] * d1) + R[6] * d2;
    const double Y = (R[1] * d0 + R[4] * d1) + R[7] * d2;
    const double Z = (R[2] * d0 + R[5] * d1) + R[8] * d2;
    const double iz = 1.0 / Z;
    const double fx = ldg1(intr), fy = ldg1(intr + 1), cx = ldg1(intr + 2), cy = ldg1(intr + 3);
    const double xz = X * iz, yz = Y * iz;
    const double2 m = lds2(uv + i);
    double r0 = cp.sw_repr * ((fx * xz + cx) - m.x);
    double r1 = cp.sw_repr * ((fy * yz + cy) - m.y);
    double rho0;
    const double hs = huber_scale(cp.hub_repr, r0 * r0 + r1 * r1, rho0);
    cost = 0.5 * rho0;
    r0 *= hs;
    r1 *= hs;
    const double w = cp.sw_repr * hs;
    const double a = w * fx * iz, b = w * fy * iz;
    const bool fixed = (c == cp.fixed_cam);
    const double *S = sc + 6 * (size_t)c;
    const double s0 = ldg1(S), s1 = ldg1(S + 1), s2 = ldg1(S + 2), s3 = ldg1(S + 3), s4 = ldg1(S + 4), s5 = ldg1(S + 5);
    const double *SP = sp + 3 * (size_t)p;
    const double sp0 = ldg1(SP), sp1 = ldg1(SP + 1), sp2 = ldg1(SP + 2);
    sts2(J.r + i, make_double2(r0, r1));
    if (!fixed) {
      sts2(J.Jc[0] + i, make_double2(-a * s0, 0.0));
      sts2(J.Jc[1] + i, make_double2(0.0, -b * s1));
      sts2(J.Jc[2] + i, make_double2(a * xz * s2, b * yz * s2));
      sts2(J.Jc[3] + i, make_double2(a * X * yz * s3, (w * fy) * (1.0 + yz * yz) * s3));
      sts2(J.Jc[4] + i, make_double2(-(w * fx) * (1.0 + xz * xz) * s4, -b * X * yz * s4));
      sts2(J.Jc[5] + i, make_double2(a * Y * s5, -b * X * s5));
    } else {
      const double2 z2 = make_double2(0.0, 0.0);
#pragma unroll
      for (int k = 0; k < 6; ++k) sts2(J.Jc[k] + i, z2);
    }
    sts2(J.Jp[0] + i, make_double2(a * (R[0] - xz * R[2]) * sp0, b * (R[1] - yz * R[2]) * sp0));
    sts2(J.Jp[1] + i, make_double2(a * (R[3] - xz * R[5]) * sp1, b * (R[4] - yz * R[5]) * sp1));
    sts2(J.Jp[2] + i, make_double2(a * (R[6] - xz * R[8]) * sp2, b * (R[7] - yz * R[8]) * sp2));
    bool bad = !(isfinite(r0) && isfinite(r1) && isfinite(iz));
    if (DEPTH) {
      double r2 = cp.sw_unpr * (lds1(depth + i) - Z);
      double rho0d;
      const double hd = huber_scale(cp.hub_unpr, r2 * r2, rho0d);
      cost += 0.5 * rho0d;
      r2 *= hd;
      const double w3 = cp.sw_unpr * hd;
      sts1(J.r3 + i, r2);
      if (!fixed) {
        sts1(J.Jc3[0] + i, 0.0);
        sts1(J.Jc3[1] + i, 0.0);
        sts1(J.Jc3[2] + i, w3 * s2);
        sts1(J.Jc3[3] + i, w3 * Y * s3);
        sts1(J.Jc3[4] + i, -w3 * X * s4);
        sts1(J.Jc3[5] + i, 0.0);
      } else {
#pragma unroll
        for (int k = 0; k < 6; ++k) sts1(J.Jc3[k] + i, 0.0);
      }
      sts1(J.Jp3[0] + i, -w3 * R[2] * sp0);
      sts1(J.Jp3[1] + i, -w3 * R[5] * sp1);
      sts1(J.Jp3[2] + i, -w3 * R[8] * sp2);
      bad = bad || !isfinite(r2);
    }
    if (NK) {
      sts2(J.Jk[0] + i, make_double2(w * xz * ldg1(sk), w * yz * ldg1(sk + 1)));
      sts2(J.Jk[1] + i, make_double2(w * ldg1(sk + 2), w * ldg1(sk + 3)));
    }
    if (bad) st->eval_fail = 1;
  }
  if (COST) {
    const double s = block_sum(cost, red);
    if (threadIdx.x == 0) cost_part[blockIdx.x] = s;
  }
}

// cost-only evaluation of a candidate point (T=double path of the functors)
template <int DEPTH>
__global__ void __launch_bounds__(BA_THREADS)
k_cost(int n_obs, const int32_t *__restrict__ cam_idx, const int32_t *__restrict__ pt_idx, const double2 *__restrict__ uv,
       const double *__restrict__ depth, const double *__restrict__ pose, const double *__restrict__ pt,
       const double *__restrict__ intr, CostParams cp, double *__restrict__ cost_part, const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  __shared__ double red[BA_WARPS + 1];
  const int i = blockIdx.x * BA_THREADS + threadIdx.x;
  double cost = 0.0;
  if (i < n_obs) {
    const int c = cam_idx[i], p = pt_idx[i];
    const double *P = pose + 7 * (size_t)c;
    const double q[4] = {ldg1(P), ldg1(P + 1), ldg1(P + 2), ldg1(P + 3)};
    double R[9];
    quat_to_R(q, R);
    const double *X3 = pt + 3 * (size_t)p;
    const double d0 = ldg1(X3) - ldg1(P + 4), d1 = ldg1(X3 + 1) - ldg1(P + 5), d2 = ldg1(X3 + 2) - ldg1(P + 6);
    const double X = (R[0] * d0 + R[3] * d1) + R[6] * d2;
    const double Y = (R[1] * d0 + R[4] * d1) + R[7] * d2;
    const double Z = (R[2] * d0 + R[5] * d1) + R[8] * d2;
    const double iz = 1.0 / Z;
    const double2 m = lds2(uv + i);
    const double r0 = cp.sw_repr * ((ldg1(intr) * (X * iz) + ldg1(intr + 2)) - m.x);
    const double r1 = cp.sw_repr * ((ldg1(intr + 1) * (Y * iz) + ldg1(intr + 3)) - m.y);
    double rho0;
    huber_scale(cp.hub_repr, r0 * r0 + r1 * r1, rho0);
    cost = 0.5 * rho0;
    if (DEPTH) {
      const double r2 = cp.sw_unpr * (lds1(depth + i) - Z);
      huber_scale(cp.hub_unpr, r2 * r2, rho0);
      cost += 0.5 * rho0;
    }
  }
  const double s = block_sum(cost, red);
  if (threadIdx.x == 0) cost_part[blockIdx.x] = s;
}

// =====================================================================
// Normal-equation blocks, camera side: warp-shuffle segmented reduction
// =====================================================================
// One warp per work item (a run of observations of one camera): lanes stride
// over the run with coalesced 128-bit loads, accumulate in registers, then a
// butterfly shuffle reduction; lane 0 writes the item partial.  A second tiny
// kernel adds the item partials of a camera in fixed order.
//   per item: U (21 upper entries of Jc^T Jc), g (6) [, U_ck 24, U_kk 6, g_k 4]
template <int NK>
struct CamBlk {
  static const int NV = 27 + (NK ? 34 : 0);
};

template <int DEPTH, int NK>
__global__ void __launch_bounds__(BA_THREADS)
k_cam_blocks(int n_items, const BaItem *__restrict__ items, JPlanes J, double *__restrict__ part, const LmState *st,
             int gate) {
  if (!gate_open(st, gate)) return;
  const int wid = (blockIdx.x * BA_THREADS + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (wid >= n_items) return;
  const BaItem it = items[wid];
  constexpr int NV = CamBlk<NK>::NV;
  double acc[NV];
#pragma unroll
  for (int k = 0; k < NV; ++k) acc[k] = 0.0;
  for (int i = it.begin + lane; i < it.end; i += 32) {
    double2 jc[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) jc[k] = lds2(J.Jc[k] + i);
    const double2 r = lds2(J.r + i);
    int u = 0;
#pragma unroll
    for (int a = 0; a < 6; ++a)
#pragma unroll
      for (int b = a; b < 6; ++b) acc[u++] += jc[a].x * jc[b].x + jc[a].y * jc[b].y;
#pragma unroll
    for (int a = 0; a < 6; ++a) acc[21 + a] += jc[a].x * r.x + jc[a].y * r.y;
    if (DEPTH) {
      double j3[6];
#pragma unroll
      for (int k = 0; k < 6; ++k) j3[k] = lds1(J.Jc3[k] + i);
      const double r3 = lds1(J.r3 + i);
      u = 0;
#pragma unroll
      for (int a = 0; a < 6; ++a)
#pragma unroll
        for (int b = a; b < 6; ++b) acc[u++] += j3[a] * j3[b];
#pragma unroll
      for (int a = 0; a < 6; ++a) acc[21 + a] += j3[a] * r3;
    }
    if (NK) {
      const double2 k0 = lds2(J.Jk[0] + i), k1 = lds2(J.Jk[1] + i);
      // Jk row0 = [k0.x 0 k1.x 0], row1 = [0 k0.y 0 k1.y]
#pragma unroll
      for (int a = 0; a < 6; ++a) {
        acc[27 + a * 4 + 0] += jc[a].x * k0.x;
        acc[27 + a * 4 + 1] += jc[a].y * k0.y;
        acc[27 + a * 4 + 2] += jc[a].x * k1.x;
        acc[27 + a * 4 + 3] += jc[a].y * k1.y;
      }
      acc[51] += k0.x * k0.x;  // (0,0)
      acc[52] += k0.x * k1.x;  // (0,2)
      acc[53] += k1.x * k1.x;  // (2,2)
      acc[54] += k0.y * k0.y;  // (1,1)
      acc[55] += k0.y * k1.y;  // (1,3)
      acc[56] += k1.y * k1.y;  // (3,3)
      acc[57] += k0.x * r.x;
      acc[58] += k0.y * r.y;
      acc[59] += k1.x * r.x;
      acc[60] += k1.y * r.y;
    }
  }
  // warp sum by recursive halving (27 / 61 butterflies otherwise): every lane writes the one or two entries it ends up with
  int idx, cnt;
  warp_reduce_scatter<NV>(acc, lane, idx, cnt);
  double *o = part + (size_t)wid * NV + idx;
  if (cnt > 0) o[0] = acc[0];
  if (NV > 32 && cnt > 1) o[1] = acc[1];
}

// per camera: add item partials in order; U (full 6x6), g_c, U_ck, clamped LM diagonal
template <int NK>
__device__ __forceinline__ void d_k_cam_blocks_fin(int bid, int n_cam, const int32_t *__restrict__ item_ptr, const double *__restrict__ part, double *__restrict__ U,
                 double *__restrict__ gc, double *__restrict__ Uck, double *__restrict__ dc, LmOptions lo,
                 const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  // one thread per (camera, value): a camera's item partials are added in item order (coalesced across values)
  constexpr int NV = CamBlk<NK>::NV;
  constexpr int NL = 27 + (NK ? 24 : 0);
  const int idx = bid * BA_THREADS + threadIdx.x;
  if (idx >= n_cam * NL) return;
  const int c = idx / NL, k = idx - c * NL;
  double acc = 0.0;
  for (int it = item_ptr[c]; it < item_ptr[c + 1]; ++it) acc += part[(size_t)it * NV + k];
  if (k < 21) {
    int a = 0, r = k;  // k-th entry of the row-major upper triangle -> (a, b)
    while (r >= 6 - a) {
      r -= 6 - a;
      ++a;
    }
    const int b2 = a + r;
    double *Uc = U + 36 * (size_t)c;
    Uc[a * 6 + b2] = acc;
    Uc[b2 * 6 + a] = acc;
    if (a == b2) dc[6 * (size_t)c + a] = fmin(fmax(acc, lo.min_lm_diagonal), lo.max_lm_diagonal);
  } else if (k < 27) {
    gc[6 * (size_t)c + k - 21] = acc;
  } else if (NK) {
    Uck[24 * (size_t)c + k - 27] = acc;
  }
}
template <int NK>
__global__ void __launch_bounds__(BA_THREADS)
k_cam_blocks_fin(int n_cam, const int32_t *__restrict__ item_ptr, const double *__restrict__ part, double *__restrict__ U,
                 double *__restrict__ gc, double *__restrict__ Uck, double *__restrict__ dc, LmOptions lo,
                 const LmState *st, int gate) {
  d_k_cam_blocks_fin<NK>(blockIdx.x, n_cam, item_ptr, part, U, gc, Uck, dc, lo, st, gate);
}

// intrinsics block: U_kk (4x4), g_k, LM diagonal; single CTA, fixed order.
// Adds the IntrinsicsPrior (:116-125) residual r_k = sqrt(w)(prior - intr) with
// Jacobian -sqrt(w) I (column-scaled by sk).
__device__ __forceinline__ void d_k_kk_fin(int bid, int n_items, const double *__restrict__ part, const double *__restrict__ intr, const double *__restrict__ intr_prior,
         const double *__restrict__ sk, CostParams cp, LmOptions lo, double *__restrict__ Ukk, double *__restrict__ gk,
         double *__restrict__ dk, double *__restrict__ rk, double *__restrict__ Jkk, const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  // one warp per value (lanes stride the items, butterfly sum): one pass instead of ten CTA-wide reductions
  __shared__ double vs[10];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int k = warp; k < 10; k += BA_WARPS) {
    double s = 0.0;
    for (int i = lane; i < n_items; i += 32) s += part[(size_t)i * CamBlk<4>::NV + 51 + k];
    s = warp_sum(s);
    if (lane == 0) vs[k] = s;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double v[10];
    for (int k = 0; k < 10; ++k) v[k] = vs[k];
    double K[16];
    for (int k = 0; k < 16; ++k) K[k] = 0.0;
    K[0] = v[0];
    K[2] = K[8] = v[1];
    K[10] = v[2];
    K[5] = v[3];
    K[7] = K[13] = v[4];
    K[15] = v[5];
    double g[4] = {v[6], v[7], v[8], v[9]};
    for (int k = 0; k < 4; ++k) {
      const double r = cp.sw_intr * (intr_prior[k] - intr[k]);
      const double j = -cp.sw_intr * sk[k];
      rk[k] = r;
      Jkk[k] = j;
      K[k * 5] += j * j;
      g[k] += j * r;
    }
    for (int k = 0; k < 16; ++k) Ukk[k] = K[k];
    for (int k = 0; k < 4; ++k) {
      gk[k] = g[k];
      dk[k] = fmin(fmax(K[k * 5], lo.min_lm_diagonal), lo.max_lm_diagonal);
    }
  }
}
__global__ void __launch_bounds__(BA_THREADS)
k_kk_fin(int n_items, const double *__restrict__ part, const double *__restrict__ intr, const double *__restrict__ intr_prior,
         const double *__restrict__ sk, CostParams cp, LmOptions lo, double *__restrict__ Ukk, double *__restrict__ gk,
         double *__restrict__ dk, double *__restrict__ rk, double *__restrict__ Jkk, const LmState *st, int gate) {
  d_k_kk_fin(blockIdx.x, n_items, part, intr, intr_prior, sk, cp, lo, Ukk, gk, dk, rk, Jkk, st, gate);
}

// REF mode: the two finishing kernels above are independent -> one launch (CTAs [0, nb_cam) finish the camera
// blocks, the last CTA the intrinsics block); one launch less on the critical path of the windowed LM iteration
__global__ void __launch_bounds__(BA_THREADS)
k_cam_kk_fin(int nb_cam, int n_cam, const int32_t *__restrict__ item_ptr, const double *__restrict__ part, double *__restrict__ U,
             double *__restrict__ gc, double *__restrict__ Uck, double *__restrict__ dc, int n_items,
             const double *__restrict__ intr, const double *__restrict__ intr_prior, const double *__restrict__ sk, CostParams cp,
             LmOptions lo, double *__restrict__ Ukk, double *__restrict__ gk, double *__restrict__ dk, double *__restrict__ rk,
             double *__restrict__ Jkk, const LmState *st, int gate) {
  if ((int)blockIdx.x < nb_cam)
    d_k_cam_blocks_fin<4>(blockIdx.x, n_cam, item_ptr, part, U, gc, Uck, dc, lo, st, gate);
  else
    d_k_kk_fin(0, n_items, part, intr, intr_prior, sk, cp, lo, Ukk, gk, dk, rk, Jkk, st, gate);
}

// =====================================================================
// Point-major tile reduction
// =====================================================================
// A CTA owns BA_TILE_PTS consecutive points.  Its observations (contiguous in
// the point-major copy) are processed one per thread with coalesced plane
// loads; the per-observation NV-vector goes to shared memory and one thread
// per point adds its run in order -- the summation order of a sequential loop
// over the stable point-major permutation, with no atomics.
template <int NV, int TOBS, class Contrib, class Finish>
__device__ __forceinline__ void tile_point_reduce(int n_pt, const int32_t *__restrict__ pt_rowptr, double *sm /*[NV*TOBS]*/,
                                                  Contrib contrib, Finish finish, int tile_pts = BA_TILE_PTS) {
  // tile_pts <= BA_TILE_PTS: the planes-store kernels of small problems run with shorter tiles (more CTAs)
  const int p0 = blockIdx.x * tile_pts;
  const int p1 = min(n_pt, p0 + tile_pts);
  const int o0 = pt_rowptr[p0], o1 = pt_rowptr[p1];
  const int p = p0 + threadIdx.x;
  const bool own = p < p1;
  int pb = 0, pe = 0;
  if (own) {
    pb = pt_rowptr[p];
    pe = pt_rowptr[p + 1];
  }
  double sum[NV];
#pragma unroll
  for (int k = 0; k < NV; ++k) sum[k] = 0.0;
  for (int cs = o0; cs < o1; cs += TOBS) {
    for (int l = threadIdx.x; l < TOBS; l += BA_THREADS) {
      const int s = cs + l;
      if (s < o1) {
        double v[NV];
        contrib(s, v);
#pragma unroll
        for (int k = 0; k < NV; ++k) sm[k * TOBS + l] = v[k];
      }
    }
    __syncthreads();
    if (own) {
      const int b = max(pb, cs), e = min(pe, cs + TOBS);
      for (int s = b; s < e; ++s) {
        const int l = s - cs;
#pragma unroll
        for (int k = 0; k < NV; ++k) sum[k] += sm[k * TOBS + l];
      }
    }
    __syncthreads();
  }
  if (own) finish(p, sum);
}

// V_p = sum Jp^T Jp (packed sym 6), g_p = sum Jp^T r, [Wk_p = sum Jk^T Jp (4x3)],
// clamped LM diagonal of the point columns
template <int DEPTH, int NK>
__global__ void __launch_bounds__(BA_THREADS)
k_pt_blocks(int n_pt, int tile_pts, const int32_t *__restrict__ pt_rowptr, JPlanes J, double *__restrict__ V,
            double *__restrict__ gp, double *__restrict__ Wk, double *__restrict__ dp, LmOptions lo, const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  constexpr int NV = 9 + (NK ? 12 : 0);
  constexpr int TOBS = NK ? 256 : 512;
  __shared__ double sm[NV * TOBS];
  tile_point_reduce<NV, TOBS>(
      n_pt, pt_rowptr, sm,
      [&](int s, double *v) {
        double2 jp[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) jp[k] = lds2(J.Jp[k] + s);
        const double2 r = lds2(J.r + s);
        v[0] = jp[0].x * jp[0].x + jp[0].y * jp[0].y;
        v[1] = jp[0].x * jp[1].x + jp[0].y * jp[1].y;
        v[2] = jp[0].x * jp[2].x + jp[0].y * jp[2].y;
        v[3] = jp[1].x * jp[1].x + jp[1].y * jp[1].y;
        v[4] = jp[1].x * jp[2].x + jp[1].y * jp[2].y;
        v[5] = jp[2].x * jp[2].x + jp[2].y * jp[2].y;
#pragma unroll
        for (int k = 0; k < 3; ++k) v[6 + k] = jp[k].x * r.x + jp[k].y * r.y;
        if (DEPTH) {
          double j3[3];
#pragma unroll
          for (int k = 0; k < 3; ++k) j3[k] = lds1(J.Jp3[k] + s);
          const double r3 = lds1(J.r3 + s);
          v[0] += j3[0] * j3[0];
          v[1] += j3[0] * j3[1];
          v[2] += j3[0] * j3[2];
          v[3] += j3[1] * j3[1];
          v[4] += j3[1] * j3[2];
          v[5] += j3[2] * j3[2];
#pragma unroll
          for (int k = 0; k < 3; ++k) v[6 + k] += j3[k] * r3;
        }
        if (NK) {
          const double2 k0 = lds2(J.Jk[0] + s), k1 = lds2(J.Jk[1] + s);
#pragma unroll
          for (int b = 0; b < 3; ++b) {
            v[9 + 0 * 3 + b] = k0.x * jp[b].x;
            v[9 + 1 * 3 + b] = k0.y * jp[b].y;
            v[9 + 2 * 3 + b] = k1.x * jp[b].x;
            v[9 + 3 * 3 + b] = k1.y * jp[b].y;
          }
        }
      },
      [&](int p, const double *sum) {
#pragma unroll
        for (int k = 0; k < 6; ++k) V[6 * (size_t)p + k] = sum[k];
#pragma unroll
        for (int k = 0; k < 3; ++k) gp[3 * (size_t)p + k] = sum[6 + k];
        dp[3 * (size_t)p + 0] = fmin(fmax(sum[0], lo.min_lm_diagonal), lo.max_lm_diagonal);
        dp[3 * (size_t)p + 1] = fmin(fmax(sum[3], lo.min_lm_diagonal), lo.max_lm_diagonal);
        dp[3 * (size_t)p + 2] = fmin(fmax(sum[5], lo.min_lm_diagonal), lo.max_lm_diagonal);
        if (NK) {
#pragma unroll
          for (int k = 0; k < 12; ++k) Wk[12 * (size_t)p + k] = sum[9 + k];
        }
      },
      tile_pts);
}

// V_p + D_p^2 -> V_p^-1 (in-register 3x3 Cholesky inverse), tg_p = V_p^-1 g_p
// D = sqrt(diag / radius) as LevenbergMarquardtStrategy::ComputeStep
__global__ void __launch_bounds__(BA_THREADS)
k_point_inverse(int n_pt, const double *__restrict__ V, const double *__restrict__ dp, const double *__restrict__ gp,
                double *__restrict__ Vinv, double *__restrict__ tg, LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  const int p = blockIdx.x * BA_THREADS + threadIdx.x;
  if (p >= n_pt) return;
  const double radius = st->radius;
  double v[6], vi[6];
#pragma unroll
  for (int k = 0; k < 6; ++k) v[k] = V[6 * (size_t)p + k];
  const double D0 = sqrt(dp[3 * (size_t)p] / radius), D1 = sqrt(dp[3 * (size_t)p + 1] / radius),
               D2 = sqrt(dp[3 * (size_t)p + 2] / radius);
  v[0] += D0 * D0;
  v[3] += D1 * D1;
  v[5] += D2 * D2;
  if (!spd3_inverse(v, vi)) {
    st->lin_fail = 1;
#pragma unroll
    for (int k = 0; k < 6; ++k) vi[k] = 0.0;
  }
#pragma unroll
  for (int k = 0; k < 6; ++k) Vinv[6 * (size_t)p + k] = vi[k];
  const double g[3] = {gp[3 * (size_t)p], gp[3 * (size_t)p + 1], gp[3 * (size_t)p + 2]};
  double t[3];
  sym3_mul(vi, g, t);
  tg[3 * (size_t)p] = t[0];
  tg[3 * (size_t)p + 1] = t[1];
  tg[3 * (size_t)p + 2] = t[2];
}

// =====================================================================
// Implicit Schur complement, pass 1 (point-major):
//   MODE 0: t_p  = V_p^-1 sum_o Jp^T (Jc x_c)                (matvec)
//   MODE 1: y_p  = V_p^-1 (-g_p - sum_o Jp^T (Jc y_c + Jk y_k))  (back-substitution)
// Algorithmic traffic NS: 144 B/obs (planes) + 4 (cam idx) + 72 B/point.
// =====================================================================
template <int DEPTH, int NK, int MODE>
__global__ void __launch_bounds__(BA_THREADS)
k_schur_pass1(int n_pt, int tile_pts, const int32_t *__restrict__ pt_rowptr, const int32_t *__restrict__ pm_cam, JPlanes J,
              const double *__restrict__ x, const double *__restrict__ yk, const double *__restrict__ Vinv,
              const double *__restrict__ gp, double *__restrict__ out, const LmState *st, int gate, int reset_period) {
  if (!gate_open(st, gate, reset_period)) return;
  constexpr int TOBS = 512;
  __shared__ double sm[3 * TOBS];
  double k_y[4] = {0, 0, 0, 0};
  if (NK && MODE == 1) {
#pragma unroll
    for (int k = 0; k < 4; ++k) k_y[k] = yk[k];
  }
  tile_point_reduce<3, TOBS>(
      n_pt, pt_rowptr, sm,
      [&](int s, double *v) {
        const int c = pm_cam[s];
        const double2 *xc = reinterpret_cast<const double2 *>(x + 6 * (size_t)c);
        const double2 x01 = ldg2(xc), x23 = ldg2(xc + 1), x45 = ldg2(xc + 2);
        double2 jc[6], jp[3];
#pragma unroll
        for (int k = 0; k < 6; ++k) jc[k] = lds2(J.Jc[k] + s);
#pragma unroll
        for (int k = 0; k < 3; ++k) jp[k] = lds2(J.Jp[k] + s);
        const double xx[6] = {x01.x, x01.y, x23.x, x23.y, x45.x, x45.y};
        double a0 = 0.0, a1 = 0.0;
#pragma unroll
        for (int k = 0; k < 6; ++k) {
          a0 += jc[k].x * xx[k];
          a1 += jc[k].y * xx[k];
        }
        if (NK && MODE == 1) {
          const double2 k0 = lds2(J.Jk[0] + s), k1 = lds2(J.Jk[1] + s);
          a0 += k0.x * k_y[0] + k1.x * k_y[2];
          a1 += k0.y * k_y[1] + k1.y * k_y[3];
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) v[k] = jp[k].x * a0 + jp[k].y * a1;
        if (DEPTH) {
          double a2 = 0.0;
#pragma unroll
          for (int k = 0; k < 6; ++k) a2 += lds1(J.Jc3[k] + s) * xx[k];
#pragma unroll
          for (int k = 0; k < 3; ++k) v[k] += lds1(J.Jp3[k] + s) * a2;
        }
      },
      [&](int p, const double *sum) {
        double vi[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) vi[k] = Vinv[6 * (size_t)p + k];
        double b[3] = {sum[0], sum[1], sum[2]}, t[3];
        if (MODE == 1) {
#pragma unroll
          for (int k = 0; k < 3; ++k) b[k] = -gp[3 * (size_t)p + k] - sum[k];
        }
        sym3_mul(vi, b, t);
        out[3 * (size_t)p] = t[0];
        out[3 * (size_t)p + 1] = t[1];
        out[3 * (size_t)p + 2] = t[2];
      },
      tile_pts);
}

// =====================================================================
// Implicit Schur complement, pass 2 (camera-major work items):
//   part[item] = sum_o Jc^T (alpha Jc x_c - Jp t_p)
// alpha = 1: matvec (U x - W V^-1 W^T x, the U term comes for free);
// alpha = 0 with t = V^-1 g_p: the reduced right-hand side.
// Algorithmic traffic NS: 144 B/obs + 4 (pt idx) + 24 (t_p gather).
// =====================================================================
template <int DEPTH>
__global__ void __launch_bounds__(BA_THREADS)
k_schur_pass2(int n_items, const BaItem *__restrict__ items, const int32_t *__restrict__ pt_idx, JPlanes J,
              const double *__restrict__ x, const double *__restrict__ t, double alpha, double *__restrict__ part,
              const LmState *st, int gate, int reset_period) {
  if (!gate_open(st, gate, reset_period)) return;
  const int wid = (blockIdx.x * BA_THREADS + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (wid >= n_items) return;
  const BaItem it = items[wid];
  double xx[6];
  {
    const double2 *xc = reinterpret_cast<const double2 *>(x + 6 * (size_t)it.cam);
    const double2 x01 = ldg2(xc), x23 = ldg2(xc + 1), x45 = ldg2(xc + 2);
    xx[0] = alpha * x01.x;
    xx[1] = alpha * x01.y;
    xx[2] = alpha * x23.x;
    xx[3] = alpha * x23.y;
    xx[4] = alpha * x45.x;
    xx[5] = alpha * x45.y;
  }
  double acc[6] = {0, 0, 0, 0, 0, 0};
  for (int i = it.begin + lane; i < it.end; i += 32) {
    const int p = __ldg(pt_idx + i);
    double2 jc[6], jp[3];
#pragma unroll
    for (int k = 0; k < 6; ++k) jc[k] = lds2(J.Jc[k] + i);
#pragma unroll
    for (int k = 0; k < 3; ++k) jp[k] = lds2(J.Jp[k] + i);
    const double t0 = ldg1(t + 3 * (size_t)p), t1 = ldg1(t + 3 * (size_t)p + 1), t2 = ldg1(t + 3 * (size_t)p + 2);
    double a0 = -(jp[0].x * t0 + jp[1].x * t1 + jp[2].x * t2);
    double a1 = -(jp[0].y * t0 + jp[1].y * t1 + jp[2].y * t2);
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      a0 += jc[k].x * xx[k];
      a1 += jc[k].y * xx[k];
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) acc[k] += jc[k].x * a0 + jc[k].y * a1;
    if (DEPTH) {
      double j3[6];
#pragma unroll
      for (int k = 0; k < 6; ++k) j3[k] = lds1(J.Jc3[k] + i);
      double a2 = -(lds1(J.Jp3[0] + i) * t0 + lds1(J.Jp3[1] + i) * t1 + lds1(J.Jp3[2] + i) * t2);
#pragma unroll
      for (int k = 0; k < 6; ++k) a2 += j3[k] * xx[k];
#pragma unroll
      for (int k = 0; k < 6; ++k) acc[k] += j3[k] * a2;
    }
  }
#pragma unroll
  for (int k = 0; k < 6; ++k) acc[k] = warp_sum(acc[k]);
  if (lane == 0) {
    double *o = part + 6 * (size_t)wid;
#pragma unroll
    for (int k = 0; k < 6; ++k) o[k] = acc[k];
  }
}

// =====================================================================
// SCHUR_JACOBI preconditioner: inverse of the 6x6 diagonal blocks of S
// =====================================================================
// per item: sum_o W V^-1 W^T with W = Jc^T Jp (6x3); 21 upper entries
template <int DEPTH>
__global__ void __launch_bounds__(BA_THREADS)
k_schur_diag(int n_items, const BaItem *__restrict__ items, const int32_t *__restrict__ pt_idx, JPlanes J,
             const double *__restrict__ Vinv, double *__restrict__ part, const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  const int wid = (blockIdx.x * BA_THREADS + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (wid >= n_items) return;
  const BaItem it = items[wid];
  double acc[21];
#pragma unroll
  for (int k = 0; k < 21; ++k) acc[k] = 0.0;
  for (int i = it.begin + lane; i < it.end; i += 32) {
    const int p = __ldg(pt_idx + i);
    double2 jc[6], jp[3];
#pragma unroll
    for (int k = 0; k < 6; ++k) jc[k] = lds2(J.Jc[k] + i);
#pragma unroll
    for (int k = 0; k < 3; ++k) jp[k] = lds2(J.Jp[k] + i);
    double vi[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) vi[k] = ldg1(Vinv + 6 * (size_t)p + k);
    double W[6][3];
#pragma unroll
    for (int a = 0; a < 6; ++a)
#pragma unroll
      for (int b = 0; b < 3; ++b) W[a][b] = jc[a].x * jp[b].x + jc[a].y * jp[b].y;
    if (DEPTH) {
      double j3[6], p3[3];
#pragma unroll
      for (int k = 0; k < 6; ++k) j3[k] = lds1(J.Jc3[k] + i);
#pragma unroll
      for (int k = 0; k < 3; ++k) p3[k] = lds1(J.Jp3[k] + i);
#pragma unroll
      for (int a = 0; a < 6; ++a)
#pragma unroll
        for (int b = 0; b < 3; ++b) W[a][b] += j3[a] * p3[b];
    }
    double WV[6][3];
#pragma unroll
    for (int a = 0; a < 6; ++a) sym3_mul(vi, W[a], WV[a]);
    int u = 0;
#pragma unroll
    for (int a = 0; a < 6; ++a)
#pragma unroll
      for (int b = a; b < 6; ++b) acc[u++] += WV[a][0] * W[b][0] + WV[a][1] * W[b][1] + WV[a][2] * W[b][2];
  }
#pragma unroll
  for (int k = 0; k < 21; ++k) acc[k] = warp_sum(acc[k]);
  if (lane == 0) {
    double *o = part + 21 * (size_t)wid;
#pragma unroll
    for (int k = 0; k < 21; ++k) o[k] = acc[k];
  }
}

// 6x6 SPD inverse through Cholesky (ceres InvertPSDMatrix); A row-major
__device__ __forceinline__ bool spd6_inverse(const double A[36], double Ai[36]) {
  double L[36];
#pragma unroll
  for (int k = 0; k < 36; ++k) L[k] = A[k];
  bool ok = true;
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    double d = L[j * 6 + j];
#pragma unroll
    for (int k = 0; k < j; ++k) d -= L[j * 6 + k] * L[j * 6 + k];
    if (!(d > 0.0) || !isfinite(d)) ok = false;
    d = sqrt(d);
    L[j * 6 + j] = d;
    const double inv = 1.0 / d;
#pragma unroll
    for (int i = j + 1; i < 6; ++i) {
      double s = L[i * 6 + j];
#pragma unroll
      for (int k = 0; k < j; ++k) s -= L[i * 6 + k] * L[j * 6 + k];
      L[i * 6 + j] = s * inv;
    }
  }
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    double col[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      double s = (i == j) ? 1.0 : 0.0;
#pragma unroll
      for (int k = 0; k < i; ++k) s -= L[i * 6 + k] * col[k];
      col[i] = s / L[i * 6 + i];
    }
#pragma unroll
    for (int i = 5; i >= 0; --i) {
      double s = col[i];
#pragma unroll
      for (int k = i + 1; k < 6; ++k) s -= L[k * 6 + i] * col[k];
      col[i] = s / L[i * 6 + i];
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) Ai[i * 6 + j] = col[i];
  }
  return ok;
}

__global__ void __launch_bounds__(BA_THREADS)
k_schur_diag_fin(int n_cam, const int32_t *__restrict__ item_ptr, const double *__restrict__ part,
                 const double *__restrict__ U, const double *__restrict__ dc, double *__restrict__ Minv,
                 double *__restrict__ dsq /* D^2 per column, may be null */, LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  const int c = blockIdx.x * BA_THREADS + threadIdx.x;
  if (c >= n_cam) return;
  const double radius = st->radius;
  double acc[21];
#pragma unroll
  for (int k = 0; k < 21; ++k) acc[k] = 0.0;
  for (int it = item_ptr[c]; it < item_ptr[c + 1]; ++it) {
#pragma unroll
    for (int k = 0; k < 21; ++k) acc[k] += part[21 * (size_t)it + k];
  }
  double B[36], Bi[36];
  int u = 0;
#pragma unroll
  for (int a = 0; a < 6; ++a)
#pragma unroll
    for (int b = a; b < 6; ++b) {
      const double v = U[36 * (size_t)c + a * 6 + b] - acc[u++];
      B[a * 6 + b] = v;
      B[b * 6 + a] = v;
    }
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    const double D = sqrt(dc[6 * (size_t)c + k] / radius);
    B[k * 6 + k] += D * D;
    if (dsq) dsq[6 * (size_t)c + k] = D * D;
  }
  if (!spd6_inverse(B, Bi)) st->lin_fail = 1;
#pragma unroll
  for (int k = 0; k < 36; ++k) Minv[36 * (size_t)c + k] = Bi[k];
}

// =====================================================================
// Reduced-system vectors: one thread per camera (6 components in registers)
// =====================================================================
__device__ __forceinline__ void load6(const double *p, double v[6]) {
  const double2 *q = reinterpret_cast<const double2 *>(p);
  const double2 a = q[0], b = q[1], c = q[2];
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; v[4] = c.x; v[5] = c.y;
}
__device__ __forceinline__ void store6(double *p, const double v[6]) {
  double2 *q = reinterpret_cast<double2 *>(p);
  q[0] = make_double2(v[0], v[1]);
  q[1] = make_double2(v[2], v[3]);
  q[2] = make_double2(v[4], v[5]);
}
__device__ __forceinline__ void sum_items6(const int32_t *item_ptr, const double *part, int c, double s[6]) {
#pragma unroll
  for (int k = 0; k < 6; ++k) s[k] = 0.0;
  for (int it = item_ptr[c]; it < item_ptr[c + 1]; ++it) {
    double v[6];
    load6(part + 6 * (size_t)it, v);
#pragma unroll
    for (int k = 0; k < 6; ++k) s[k] += v[k];
  }
}
__device__ __forceinline__ void minv_mul(const double *Minv, int c, const double r[6], double z[6]) {
  const double *M = Minv + 36 * (size_t)c;
#pragma unroll
  for (int a = 0; a < 6; ++a) {
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < 6; ++k) s += M[a * 6 + k] * r[k];
    z[a] = s;
  }
}

// b = -g_c - part (part = -sum Jc^T Jp V^-1 g_p), then PCG start: x = 0, r = b,
// z = M^-1 r, per-CTA partials of r.z and b.b
__global__ void __launch_bounds__(BA_THREADS)
k_pcg_init(int n_cam, const int32_t *__restrict__ item_ptr, const double *__restrict__ part, const double *__restrict__ gc,
           const double *__restrict__ Minv, double *__restrict__ b, double *__restrict__ x, double *__restrict__ r,
           double *__restrict__ z, double *__restrict__ part_rho, double *__restrict__ part_bb, const LmState *st,
           int gate) {
  if (!gate_open(st, gate)) return;
  __shared__ double red[BA_WARPS + 1];
  const int c = blockIdx.x * BA_THREADS + threadIdx.x;
  double rho = 0.0, bb = 0.0;
  if (c < n_cam) {
    double s[6], g[6], bv[6], zv[6], zero[6] = {0, 0, 0, 0, 0, 0};
    sum_items6(item_ptr, part, c, s);
    load6(gc + 6 * (size_t)c, g);
#pragma unroll
    for (int k = 0; k < 6; ++k) bv[k] = -g[k] - s[k];
    minv_mul(Minv, c, bv, zv);
    store6(b + 6 * (size_t)c, bv);
    store6(r + 6 * (size_t)c, bv);
    store6(x + 6 * (size_t)c, zero);
    store6(z + 6 * (size_t)c, zv);
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      rho += bv[k] * zv[k];
      bb += bv[k] * bv[k];
    }
  }
  const double s1 = block_sum(rho, red);
  const double s2 = block_sum(bb, red);
  if (threadIdx.x == 0) {
    part_rho[blockIdx.x] = s1;
    part_bb[blockIdx.x] = s2;
  }
}

// single CTA: PCG controller reset ("Convergence. |b| = 0" shortcut included)
__global__ void __launch_bounds__(BA_THREADS)
k_pcg_start(int nblk, const double *__restrict__ part_bb, const double *__restrict__ part_rho, LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  __shared__ double red[BA_WARPS + 2];
  const double bb = block_sum_array(part_bb, nblk, red);
  const double rho = block_sum_array(part_rho, nblk, red);
  if (threadIdx.x == 0) {
    st->pcg_it = 1;
    st->pcg_fail = 0;
    st->pcg_break = 0;
    st->pcg_Q0 = 0.0;
    st->pcg_rho = rho;
    st->pcg_beta = 0.0;
    st->pcg_counter = 0;
    st->pcg_iters_last = 0;
    st->pcg_done = (bb == 0.0 || st->lin_fail) ? 1 : 0;
    if (!isfinite(bb)) {
      st->pcg_done = 1;
      st->lin_fail = 1;
    } else if (bb != 0.0 && (rho == 0.0 || !isfinite(rho))) {  // IsZeroOrInfinity(rho): solver failure
      st->pcg_done = 1;
      st->lin_fail = 1;
      st->pcg_iters_last = 1;
    }
  }
}

// direction update p = z + beta p (beta = rho / last_rho from the controller)
__global__ void __launch_bounds__(BA_THREADS)
k_pcg_dir(int n_cam, const double *__restrict__ z, double *__restrict__ p, const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  const int c = blockIdx.x * BA_THREADS + threadIdx.x;
  if (c >= n_cam) return;
  const int it = st->pcg_it;
  const double beta = st->pcg_beta;
  double zv[6], pv[6];
  load6(z + 6 * (size_t)c, zv);
  if (it > 1) {
    load6(p + 6 * (size_t)c, pv);
#pragma unroll
    for (int k = 0; k < 6; ++k) pv[k] = zv[k] + beta * pv[k];
  } else {
#pragma unroll
    for (int k = 0; k < 6; ++k) pv[k] = zv[k];
  }
  store6(p + 6 * (size_t)c, pv);
}

// q = S p from the pass-2 item partials (+ LM damping), per-CTA partials of p.q
__global__ void __launch_bounds__(BA_THREADS)
k_pcg_q(int n_cam, const int32_t *__restrict__ item_ptr, const double *__restrict__ part, const double *__restrict__ dc,
        const double *__restrict__ p, double *__restrict__ q, double *__restrict__ part_pq, const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  __shared__ double red[BA_WARPS + 1];
  const int c = blockIdx.x * BA_THREADS + threadIdx.x;
  const double radius = st->radius;
  double pq = 0.0;
  if (c < n_cam) {
    double s[6], pv[6], d[6];
    sum_items6(item_ptr, part, c, s);
    load6(p + 6 * (size_t)c, pv);
    load6(dc + 6 * (size_t)c, d);
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      const double D = sqrt(d[k] / radius);
      s[k] += D * D * pv[k];
      pq += pv[k] * s[k];
    }
    store6(q + 6 * (size_t)c, s);
  }
  const double s1 = block_sum(pq, red);
  if (threadIdx.x == 0) part_pq[blockIdx.x] = s1;
}

// Tail of a PCG iteration, run by the LAST CTA to finish (integer ticket, the
// floating-point sums stay in fixed order): quadratic-model termination of
// conjugate_gradients_solver.cc, then rho / beta of the next iteration.
__device__ __forceinline__ void pcg_controller(int nblk, double *part_rho, double *part_Q, double *red, const LmOptions &lo,
                                               LmState *st) {
  __shared__ int is_last;
  if (threadIdx.x == 0) {
    __threadfence();
    const int t = atomicAdd(&st->pcg_counter, 1);
    is_last = (t == nblk - 1);
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  double v = 0.0, w = 0.0;
  for (int i = threadIdx.x; i < nblk; i += blockDim.x) {
    v += __ldcg(part_rho + i);
    w += __ldcg(part_Q + i);
  }
  v = warp_sum(v);
  w = warp_sum(w);
  const int wid = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) {
    red[wid] = v;
    red[BA_WARPS + 2 + wid] = w;
  }
  __syncthreads();
  if (threadIdx.x != 0) return;
  double rho_new = 0.0, xq = 0.0;
  for (int i = 0; i < BA_WARPS; ++i) {
    rho_new += red[i];
    xq += red[BA_WARPS + 2 + i];
  }
  st->pcg_counter = 0;
  const int it = st->pcg_it;
  st->pcg_iters_last = it;
  const double Q1 = -1.0 * xq;
  const double zeta = it * (Q1 - st->pcg_Q0) / Q1;
  if (zeta < lo.eta && it >= lo.min_pcg) {
    st->pcg_done = 1;
    return;
  }
  st->pcg_Q0 = Q1;
  if (it >= lo.max_pcg) {
    st->pcg_done = 1;
    return;
  }
  // next iteration: rho = r.z, beta = rho / last_rho (IsZeroOrInfinity -> failure)
  const double beta = rho_new / st->pcg_rho;
  if (rho_new == 0.0 || !isfinite(rho_new) || beta == 0.0 || !isfinite(beta)) {
    st->pcg_iters_last = it + 1;
    st->pcg_done = 1;
    st->lin_fail = 1;
    return;
  }
  st->pcg_rho = rho_new;
  st->pcg_beta = beta;
  st->pcg_it = it + 1;
}

// alpha = rho / p.q ; x += alpha p ; r -= alpha q ; z = M^-1 r ; partials of r.z and
// x.(b + r); the last CTA runs the controller.  On a residual-reset iteration only x
// is updated here (r is recomputed from b - S x by k_pcg_reset).
__global__ void __launch_bounds__(BA_THREADS)
k_pcg_step(int n_cam, int nblk, const double *__restrict__ part_pq, const double *__restrict__ p,
           const double *__restrict__ q, const double *__restrict__ b, const double *__restrict__ Minv,
           double *__restrict__ x, double *__restrict__ r, double *__restrict__ z, double *part_rho, double *part_Q,
           LmOptions lo, LmState *st, int gate, int reset) {
  if (!gate_open(st, gate)) return;
  __shared__ double red[2 * BA_WARPS + 4];
  const double pq = block_sum_array(part_pq, nblk, red);
  const double rho = st->pcg_rho;
  if (pq <= 0.0 || isinf(pq) || isnan(pq)) {  // NO_CONVERGENCE: keep x, stop
    if (blockIdx.x == 0 && threadIdx.x == 0) {
      st->pcg_iters_last = st->pcg_it;
      st->pcg_break = 1;
      st->pcg_done = 1;  // safe: every CTA takes this branch from its own (identical) sum
    }
    return;
  }
  const double alpha = rho / pq;
  if (isinf(alpha)) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
      st->pcg_iters_last = st->pcg_it;
      st->pcg_done = 1;
      st->lin_fail = 1;
    }
    return;
  }
  const int c = blockIdx.x * BA_THREADS + threadIdx.x;
  double rz = 0.0, xq = 0.0;
  if (c < n_cam) {
    double xv[6], pv[6];
    load6(x + 6 * (size_t)c, xv);
    load6(p + 6 * (size_t)c, pv);
#pragma unroll
    for (int k = 0; k < 6; ++k) xv[k] = xv[k] + alpha * pv[k];
    store6(x + 6 * (size_t)c, xv);
    if (!reset) {
      double rv[6], qv[6], bv[6], zv[6];
      load6(r + 6 * (size_t)c, rv);
      load6(q + 6 * (size_t)c, qv);
      load6(b + 6 * (size_t)c, bv);
#pragma unroll
      for (int k = 0; k < 6; ++k) rv[k] = rv[k] - alpha * qv[k];
      store6(r + 6 * (size_t)c, rv);
      minv_mul(Minv, c, rv, zv);
      store6(z + 6 * (size_t)c, zv);
#pragma unroll
      for (int k = 0; k < 6; ++k) {
        rz += rv[k] * zv[k];
        xq += xv[k] * (bv[k] + rv[k]);
      }
    }
  }
  if (reset) return;
  const double s1 = block_sum(rz, red);
  const double s2 = block_sum(xq, red);
  if (threadIdx.x == 0) {
    part_rho[blockIdx.x] = s1;
    part_Q[blockIdx.x] = s2;
  }
  pcg_controller(nblk, part_rho, part_Q, red, lo, st);
}

// residual reset (every residual_reset_period iterations): r = b - S x
__global__ void __launch_bounds__(BA_THREADS)
k_pcg_reset(int n_cam, int nblk, const int32_t *__restrict__ item_ptr, const double *__restrict__ part,
            const double *__restrict__ dc, const double *__restrict__ x, const double *__restrict__ b,
            const double *__restrict__ Minv, double *__restrict__ r, double *__restrict__ z, double *part_rho,
            double *part_Q, LmOptions lo, LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  __shared__ double red[2 * BA_WARPS + 4];
  const int c = blockIdx.x * BA_THREADS + threadIdx.x;
  const double radius = st->radius;
  double rz = 0.0, xq = 0.0;
  if (c < n_cam) {
    double s[6], xv[6], d[6], bv[6], rv[6], zv[6];
    sum_items6(item_ptr, part, c, s);
    load6(x + 6 * (size_t)c, xv);
    load6(dc + 6 * (size_t)c, d);
    load6(b + 6 * (size_t)c, bv);
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      const double D = sqrt(d[k] / radius);
      s[k] += D * D * xv[k];
      rv[k] = bv[k] - s[k];
    }
    store6(r + 6 * (size_t)c, rv);
    minv_mul(Minv, c, rv, zv);
    store6(z + 6 * (size_t)c, zv);
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      rz += rv[k] * zv[k];
      xq += xv[k] * (bv[k] + rv[k]);
    }
  }
  const double s1 = block_sum(rz, red);
  const double s2 = block_sum(xq, red);
  if (threadIdx.x == 0) {
    part_rho[blockIdx.x] = s1;
    part_Q[blockIdx.x] = s2;
  }
  pcg_controller(nblk, part_rho, part_Q, red, lo, st);
}

// y_c = x (PCG solution); non-finite solution = linear solver failure
__global__ void __launch_bounds__(BA_THREADS)
k_pcg_finish(int n, const double *__restrict__ x, double *__restrict__ yc, LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  const int i = blockIdx.x * BA_THREADS + threadIdx.x;
  if (i == 0) st->total_lin_iters += st->pcg_iters_last;
  if (i >= n) return;
  const double v = x[i];
  if (!isfinite(v)) st->lin_fail = 1;
  yc[i] = v;
}

// =====================================================================
// Parameter-space kernels.  "Entries": [0,n_cam) cameras, [n_cam,n_cam+n_pt)
// points, then one entry for the intrinsics block.
// =====================================================================
// gradient max norm |x [+] (-g) - x|_inf (unscaled gradient g = g_s / scale) and |x|^2
__global__ void __launch_bounds__(BA_THREADS)
k_state_norms(int n_cam, int n_pt, int nk, int fixed_cam, const double *__restrict__ pose, const double *__restrict__ pt,
              const double *__restrict__ intr, const double *__restrict__ gc, const double *__restrict__ gp,
              const double *__restrict__ gk, const double *__restrict__ sc, const double *__restrict__ sp,
              const double *__restrict__ sk, double *__restrict__ part_gmax, double *__restrict__ part_xn,
              const LmState *st, int gate, double cam_weight) {
  if (!gate_open(st, gate)) return;
  __shared__ double red[BA_WARPS + 1];
  const int e = blockIdx.x * BA_THREADS + threadIdx.x;
  double gm = 0.0, xn = 0.0;
  if (e < n_cam) {
    if (e != fixed_cam) {
      double T[7], d[6], o[7];
#pragma unroll
      for (int k = 0; k < 7; ++k) T[k] = pose[7 * (size_t)e + k];
#pragma unroll
      for (int k = 0; k < 6; ++k) d[k] = -(gc[6 * (size_t)e + k] / sc[6 * (size_t)e + k]);
      se3_plus(T, d, o);
#pragma unroll
      for (int k = 0; k < 7; ++k) {
        gm = fmax(gm, fabs(T[k] - o[k]));
        xn += cam_weight * (T[k] * T[k]);
      }
    }
  } else if (e < n_cam + n_pt) {
    const size_t p = (size_t)(e - n_cam);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      gm = fmax(gm, fabs(gp[3 * p + k] / sp[3 * p + k]));
      const double v = pt[3 * p + k];
      xn += v * v;
    }
  } else if (e == n_cam + n_pt && nk) {
    for (int k = 0; k < 4; ++k) {
      gm = fmax(gm, fabs(gk[k] / sk[k]));
      xn += cam_weight * (intr[k] * intr[k]);
    }
  }
  const double m = block_max(gm, red);
  const double s = block_sum(xn, red);
  if (threadIdx.x == 0) {
    part_gmax[blockIdx.x] = m;
    part_xn[blockIdx.x] = s;
  }
}

// Jacobi column scaling, fixed at iteration 0: 1 / (1 + sqrt(sum_i J_ij^2))
__global__ void __launch_bounds__(BA_THREADS)
k_make_scale(int n_cam, int n_pt, int nk, const double *__restrict__ U, const double *__restrict__ V,
             const double *__restrict__ Ukk, double *__restrict__ sc, double *__restrict__ sp, double *__restrict__ sk,
             const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  const int e = blockIdx.x * BA_THREADS + threadIdx.x;
  if (e < n_cam) {
#pragma unroll
    for (int k = 0; k < 6; ++k) sc[6 * (size_t)e + k] = 1.0 / (1.0 + sqrt(U[36 * (size_t)e + 7 * k]));
  } else if (e < n_cam + n_pt) {
    const size_t p = (size_t)(e - n_cam);
    sp[3 * p + 0] = 1.0 / (1.0 + sqrt(V[6 * p + 0]));
    sp[3 * p + 1] = 1.0 / (1.0 + sqrt(V[6 * p + 3]));
    sp[3 * p + 2] = 1.0 / (1.0 + sqrt(V[6 * p + 5]));
  } else if (e == n_cam + n_pt && nk) {
    for (int k = 0; k < 4; ++k) sk[k] = 1.0 / (1.0 + sqrt(Ukk[5 * k]));
  }
}
__global__ void k_set_have_scale(LmState *st) {
  pdl_wait();
  if (st->done) return;
  st->have_scale = 1;
}

// candidate x+ = x [+] (y .* scale): SE3 plus for poses
// (local_parameterization_se3.hpp:17-24), addition for points / intrinsics;
// per-CTA partials of |x+ - x|^2 in the ambient space
__global__ void __launch_bounds__(BA_THREADS)
k_candidate(int n_cam, int n_pt, int nk, int fixed_cam, const double *__restrict__ pose, const double *__restrict__ pt,
            const double *__restrict__ intr, const double *__restrict__ yc, const double *__restrict__ yp,
            const double *__restrict__ yk, const double *__restrict__ sc, const double *__restrict__ sp,
            const double *__restrict__ sk, double *__restrict__ pose_c, double *__restrict__ pt_c,
            double *__restrict__ intr_c, double *__restrict__ part_step, const LmState *st, int gate, double cam_weight) {
  if (!gate_open(st, gate)) return;
  __shared__ double red[BA_WARPS + 1];
  const int e = blockIdx.x * BA_THREADS + threadIdx.x;
  double sn = 0.0;
  if (e < n_cam) {
    double T[7], o[7];
#pragma unroll
    for (int k = 0; k < 7; ++k) T[k] = pose[7 * (size_t)e + k];
    if (e != fixed_cam) {
      double d[6];
#pragma unroll
      for (int k = 0; k < 6; ++k) d[k] = yc[6 * (size_t)e + k] * sc[6 * (size_t)e + k];
      se3_plus(T, d, o);
#pragma unroll
      for (int k = 0; k < 7; ++k) {
        const double df = T[k] - o[k];
        sn += cam_weight * (df * df);
      }
    } else {
#pragma unroll
      for (int k = 0; k < 7; ++k) o[k] = T[k];
    }
#pragma unroll
    for (int k = 0; k < 7; ++k) pose_c[7 * (size_t)e + k] = o[k];
  } else if (e < n_cam + n_pt) {
    const size_t p = (size_t)(e - n_cam);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const double x = pt[3 * p + k];
      const double c = x + yp[3 * p + k] * sp[3 * p + k];
      pt_c[3 * p + k] = c;
      const double df = x - c;
      sn += df * df;
    }
  } else if (e == n_cam + n_pt) {
    for (int k = 0; k < 4; ++k) {
      const double x = intr[k];
      const double c = nk ? x + yk[k] * sk[k] : x;
      intr_c[k] = c;
      const double df = x - c;
      sn += cam_weight * (df * df);
    }
  }
  const double s = block_sum(sn, red);
  if (threadIdx.x == 0) part_step[blockIdx.x] = s;
}

// accepted step: x <- x+
__global__ void __launch_bounds__(BA_THREADS)
k_accept(int n_cam, int n_pt, double *__restrict__ pose, double *__restrict__ pt, double *__restrict__ intr,
         const double *__restrict__ pose_c, const double *__restrict__ pt_c, const double *__restrict__ intr_c,
         const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  const int e = blockIdx.x * BA_THREADS + threadIdx.x;
  if (e < n_cam) {
#pragma unroll
    for (int k = 0; k < 7; ++k) pose[7 * (size_t)e + k] = pose_c[7 * (size_t)e + k];
  } else if (e < n_cam + n_pt) {
    const size_t p = (size_t)(e - n_cam);
#pragma unroll
    for (int k = 0; k < 3; ++k) pt[3 * p + k] = pt_c[3 * p + k];
  } else if (e == n_cam + n_pt) {
    for (int k = 0; k < 4; ++k) intr[k] = intr_c[k];
  }
}

// model_cost_change = -(J y).(r + J y / 2): per-CTA partials of sum m (r + m/2)
template <int DEPTH, int NK>
__global__ void __launch_bounds__(BA_THREADS)
k_model_cost(int n_obs, const int32_t *__restrict__ cam_idx, const int32_t *__restrict__ pt_idx, JPlanes J,
             const double *__restrict__ yc, const double *__restrict__ yp, const double *__restrict__ yk,
             double *__restrict__ part, const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  __shared__ double red[BA_WARPS + 1];
  const int i = blockIdx.x * BA_THREADS + threadIdx.x;
  double acc = 0.0;
  if (i < n_obs) {
    const int c = cam_idx[i], p = pt_idx[i];
    double y[6];
    load6(yc + 6 * (size_t)c, y);
    const double q0 = ldg1(yp + 3 * (size_t)p), q1 = ldg1(yp + 3 * (size_t)p + 1), q2 = ldg1(yp + 3 * (size_t)p + 2);
    double2 jp[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) jp[k] = lds2(J.Jp[k] + i);
    double m0 = jp[0].x * q0 + jp[1].x * q1 + jp[2].x * q2;
    double m1 = jp[0].y * q0 + jp[1].y * q1 + jp[2].y * q2;
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      const double2 jc = lds2(J.Jc[k] + i);
      m0 += jc.x * y[k];
      m1 += jc.y * y[k];
    }
    if (NK) {
      const double2 k0 = lds2(J.Jk[0] + i), k1 = lds2(J.Jk[1] + i);
      m0 += k0.x * yk[0] + k1.x * yk[2];
      m1 += k0.y * yk[1] + k1.y * yk[3];
    }
    const double2 r = lds2(J.r + i);
    acc = m0 * (r.x + m0 / 2.0) + m1 * (r.y + m1 / 2.0);
    if (DEPTH) {
      double m2 = lds1(J.Jp3[0] + i) * q0 + lds1(J.Jp3[1] + i) * q1 + lds1(J.Jp3[2] + i) * q2;
#pragma unroll
      for (int k = 0; k < 6; ++k) m2 += lds1(J.Jc3[k] + i) * y[k];
      acc += m2 * (lds1(J.r3 + i) + m2 / 2.0);
    }
  }
  const double s = block_sum(acc, red);
  if (threadIdx.x == 0) part[blockIdx.x] = s;
}

// =====================================================================
// Levenberg-Marquardt controller (single CTA kernels)
// =====================================================================
__device__ __forceinline__ void push_trace(LmState *st, BaIterRec *trace, int cap, const BaIterRec &r) {
  if (st->n_trace < cap) trace[st->n_trace] = r;
  st->n_trace++;
}
__device__ __forceinline__ double block_max_array(const double *part, int n, double *smem) {
  double a[4] = {0, 0, 0, 0};
  const int bd = blockDim.x;
  int i = threadIdx.x;
  for (; i + 3 * bd < n; i += 4 * bd) {  // four loads in flight (the maximum does not depend on the order)
    const double t0 = part[i], t1 = part[i + bd], t2 = part[i + 2 * bd], t3 = part[i + 3 * bd];
    a[0] = fmax(a[0], t0);
    a[1] = fmax(a[1], t1);
    a[2] = fmax(a[2], t2);
    a[3] = fmax(a[3], t3);
  }
  for (; i < n; i += bd) a[0] = fmax(a[0], part[i]);
  double v = fmax(fmax(a[0], a[1]), fmax(a[2], a[3]));
  v = warp_max(v);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) smem[w] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int i = 0; i < BA_WARPS; ++i) s = fmax(s, smem[i]);
    smem[BA_WARPS] = s;
  }
  __syncthreads();
  return smem[BA_WARPS];
}

__global__ void k_lm_init(LmState *st, double initial_radius) {
  pdl_wait();
  LmState s;
  memset(&s, 0, sizeof(s));
  s.radius = initial_radius;
  s.decrease_factor = 2.0;
  s.pcg_done = 1;
  *st = s;
}

// IterationZero: cost, gradient norm, |x|; gradient-tolerance check
__global__ void __launch_bounds__(BA_THREADS)
k_lm_iter0(int nblk_obs, int nblk_ent, int nk, const double *__restrict__ part_cost, const double *__restrict__ part_gmax,
           const double *__restrict__ part_xn, const double *__restrict__ rk, LmOptions lo, LmState *st,
           BaIterRec *trace) {
  pdl_wait();
  __shared__ double red[BA_WARPS + 2];
  double cost = block_sum_array(part_cost, nblk_obs, red);
  const double gmax = block_max_array(part_gmax, nblk_ent, red);
  const double xn = block_sum_array(part_xn, nblk_ent, red);
  if (threadIdx.x != 0) return;
  if (nk) {
    double s = 0.0;
    for (int k = 0; k < 4; ++k) s += rk[k] * rk[k];
    cost = 0.5 * s + cost;
  }
  st->x_cost = cost;
  st->initial_cost = cost;
  st->gmax = gmax;
  st->x_norm = sqrt(xn);
  BaIterRec r;
  memset(&r, 0, sizeof(r));
  r.cost = cost;
  r.gradient_max_norm = gmax;
  r.radius = st->radius;
  r.step_is_valid = 1;
  r.step_is_successful = 1;
  push_trace(st, trace, lo.trace_cap, r);
  st->iter = 1;
  st->last_successful = 1;
  st->termination = 0;
  if (st->eval_fail || !isfinite(cost)) {
    st->done = 1;
    st->termination = 5;
  } else if (gmax <= lo.gradient_tolerance) {
    st->done = 1;
    st->termination = 1;
  }
}

// top of the minimizer loop (FinalizeIterationAndCheckIfMinimizerCanContinue).  Evaluated by the thread that ENDS
// the previous iteration (k_lm_control when the step is not accepted, k_lm_post when it is; k_lm_begin after
// iteration zero): one launch less per iteration, and the termination flag is already set when the host polls
// after the last iteration (no trailing gated-off iteration).
__device__ __forceinline__ void lm_begin(const LmOptions &lo, LmState *st) {
  if (st->done) return;
  if (st->iter - 1 >= lo.max_num_iterations) {
    st->done = 1;
    st->termination = 0;
    return;
  }
  if (st->last_successful && st->gmax <= lo.gradient_tolerance) {
    st->done = 1;
    st->termination = 1;
    return;
  }
  if (st->radius <= lo.min_radius) {
    st->done = 1;
    st->termination = 4;
    return;
  }
  st->accepted = 0;
  st->lin_fail = 0;
  st->pcg_iters_last = 0;
}
__global__ void k_lm_begin(LmOptions lo, LmState *st) {
  pdl_wait();
  lm_begin(lo, st);
}

// step evaluation: model cost change, tolerances, relative decrease, radius
// update (LevenbergMarquardtStrategy::StepAccepted / StepRejected)
__device__ __forceinline__ void lm_control_thread0(double msum, double step2, double cand, int nk, const double *__restrict__ rk,
                                                   const double *__restrict__ Jkk, const double *__restrict__ yk,
                                                   const double *__restrict__ intr_c, const double *__restrict__ intr_prior,
                                                   double sw_intr, const LmOptions &lo, LmState *st, BaIterRec *trace) {
  BaIterRec r;
  memset(&r, 0, sizeof(r));
  r.iteration = st->iter;
  r.linear_iters = st->pcg_iters_last;
  if (nk) {
    double pm = 0.0, s = 0.0;
    for (int k = 0; k < 4; ++k) {
      const double m = Jkk[k] * yk[k];
      pm += m * (rk[k] + m / 2.0);
      const double rc = sw_intr * (intr_prior[k] - intr_c[k]);
      s += rc * rc;
    }
    msum = pm + msum;
    cand = 0.5 * s + cand;
  }
  const double mcc = st->lin_fail ? 0.0 : -msum;
  const bool valid = !st->lin_fail && (mcc > 0.0);
  r.model_cost_change = mcc;
  r.step_is_valid = valid ? 1 : 0;
  st->accepted = 0;
  if (!valid) {
    st->invalid_run++;
    r.cost = st->x_cost;
    r.gradient_max_norm = st->gmax;
    st->last_successful = 0;
    if (st->invalid_run >= lo.max_invalid) {
      st->done = 1;
      st->termination = 5;
      r.radius = st->radius;
      push_trace(st, trace, lo.trace_cap, r);
      return;
    }
    st->radius = st->radius / st->decrease_factor;
    st->decrease_factor *= 2.0;
    r.radius = st->radius;
    st->num_unsuccessful++;
    push_trace(st, trace, lo.trace_cap, r);
    st->iter++;
    return;
  }
  st->invalid_run = 0;
  if (!isfinite(cand)) cand = DBL_MAX;
  r.step_norm = sqrt(step2);
  r.radius = st->radius;
  r.cost = st->x_cost;
  r.gradient_max_norm = st->gmax;
  if (r.step_norm <= lo.parameter_tolerance * (st->x_norm + lo.parameter_tolerance)) {
    st->done = 1;
    st->termination = 2;
    push_trace(st, trace, lo.trace_cap, r);
    return;
  }
  r.cost_change = st->x_cost - cand;
  if (fabs(r.cost_change) <= lo.function_tolerance * st->x_cost) {
    st->done = 1;
    st->termination = 3;
    push_trace(st, trace, lo.trace_cap, r);
    return;
  }
  r.relative_decrease = r.cost_change / mcc;
  if (r.relative_decrease > lo.min_relative_decrease) {
    st->accepted = 1;
    const double t = 2.0 * r.relative_decrease - 1.0;
    st->radius = st->radius / fmax(1.0 / 3.0, 1.0 - t * t * t);
    st->radius = fmin(lo.max_radius, st->radius);
    st->decrease_factor = 2.0;
    st->num_successful++;
    r.step_is_successful = 1;
    r.radius = st->radius;
    st->pending = r;  // completed by k_lm_post after relinearisation
  } else {
    st->last_successful = 0;
    st->radius = st->radius / st->decrease_factor;
    st->decrease_factor *= 2.0;
    st->num_unsuccessful++;
    r.radius = st->radius;
    push_trace(st, trace, lo.trace_cap, r);
  }
  st->iter++;
}
__global__ void __launch_bounds__(BA_THREADS)
k_lm_control(int nblk_obs, int nblk_ent, int nk, const double *__restrict__ part_mcc, const double *__restrict__ part_step,
             const double *__restrict__ part_cost, const double *__restrict__ rk, const double *__restrict__ Jkk,
             const double *__restrict__ yk, const double *__restrict__ intr_c, const double *__restrict__ intr_prior,
             double sw_intr, LmOptions lo, LmState *st, BaIterRec *trace) {
  pdl_wait();
  if (st->done) return;
  __shared__ double red[BA_WARPS + 2];
  const double msum = block_sum_array(part_mcc, nblk_obs, red);
  const double step2 = block_sum_array(part_step, nblk_ent, red);
  const double cand = block_sum_array(part_cost, nblk_obs, red);
  if (threadIdx.x != 0) return;
  lm_control_thread0(msum, step2, cand, nk, rk, Jkk, yk, intr_c, intr_prior, sw_intr, lo, st, trace);
  if (!st->accepted) lm_begin(lo, st);  // not accepted (or finished): the iteration ends here
}

// after the relinearisation of an accepted step
__global__ void __launch_bounds__(BA_THREADS)
k_lm_post(int nblk_obs, int nblk_ent, int nk, const double *__restrict__ part_cost, const double *__restrict__ part_gmax,
          const double *__restrict__ part_xn, const double *__restrict__ rk, LmOptions lo, LmState *st,
          BaIterRec *trace, int gate) {
  if (!gate_open(st, gate)) return;
  __shared__ double red[BA_WARPS + 2];
  double cost = block_sum_array(part_cost, nblk_obs, red);
  const double gmax = block_max_array(part_gmax, nblk_ent, red);
  const double xn = block_sum_array(part_xn, nblk_ent, red);
  if (threadIdx.x != 0) return;
  if (nk) {
    double s = 0.0;
    for (int k = 0; k < 4; ++k) s += rk[k] * rk[k];
    cost = 0.5 * s + cost;
  }
  st->x_cost = cost;
  st->gmax = gmax;
  st->x_norm = sqrt(xn);
  st->last_successful = 1;
  BaIterRec r = st->pending;
  r.cost = cost;
  r.gradient_max_norm = gmax;
  push_trace(st, trace, lo.trace_cap, r);
  if (st->eval_fail || !isfinite(cost)) {
    st->done = 1;
    st->termination = 5;
  }
  lm_begin(lo, st);  // an accepted iteration ends here
}

// =====================================================================
// Explicit Schur complement (windowed problems) + dense Cholesky
//   S = [U + D^2] - sum_p W_p V_p^-1 W_p^T     (schur_eliminator_impl.h)
// with the 4 intrinsics columns as one extra "camera-side" block (REF mode).
// =====================================================================
// per observation (camera-major): W = Jc^T Jp (6x3) and WV = W V_p^-1
template <int DEPTH>
__global__ void __launch_bounds__(BA_THREADS)
k_obs_W(int n_obs, const int32_t *__restrict__ pt_idx, JPlanes J, const double *__restrict__ V, const double *__restrict__ dp,
        double *__restrict__ W, double *__restrict__ WV, const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;  // (64-thread CTAs on windows: one CTA per SM)
  if (i >= n_obs) return;
  const int p = pt_idx[i];
  // V_p^-1 is re-derived here from V_p and the LM diagonal with k_point_inverse's arithmetic (identical bits), so that
  // kernel runs beside this one on the side stream instead of in front of it
  double vi[6];
  {
    const double radius = st->radius;
    double v[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) v[k] = V[6 * (size_t)p + k];
    const double D0 = sqrt(dp[3 * (size_t)p] / radius), D1 = sqrt(dp[3 * (size_t)p + 1] / radius),
                 D2 = sqrt(dp[3 * (size_t)p + 2] / radius);
    v[0] += D0 * D0;
    v[3] += D1 * D1;
    v[5] += D2 * D2;
    if (!spd3_inverse(v, vi)) {
#pragma unroll
      for (int k = 0; k < 6; ++k) vi[k] = 0.0;
    }
  }
  double2 jc[6], jp[3];
#pragma unroll
  for (int k = 0; k < 6; ++k) jc[k] = lds2(J.Jc[k] + i);
#pragma unroll
  for (int k = 0; k < 3; ++k) jp[k] = lds2(J.Jp[k] + i);
  double w[6][3];
#pragma unroll
  for (int a = 0; a < 6; ++a)
#pragma unroll
    for (int b = 0; b < 3; ++b) w[a][b] = jc[a].x * jp[b].x + jc[a].y * jp[b].y;
  if (DEPTH) {
#pragma unroll
    for (int a = 0; a < 6; ++a) {
      const double j3 = lds1(J.Jc3[a] + i);
#pragma unroll
      for (int b = 0; b < 3; ++b) w[a][b] += j3 * lds1(J.Jp3[b] + i);
    }
  }
#pragma unroll
  for (int a = 0; a < 6; ++a) {
    double wv[3];
    sym3_mul(vi, w[a], wv);
#pragma unroll
    for (int b = 0; b < 3; ++b) {
      W[18 * (size_t)i + a * 3 + b] = w[a][b];
      WV[18 * (size_t)i + a * 3 + b] = wv[b];
    }
  }
}

// camera-side vectors of the reduced system, one warp per work item:
//   rhs_c += W_o (V^-1 g_p)          (6)
//   S_ck  += WV_o Wk_p^T             (6x4, REF mode)
template <int NK>
__device__ __forceinline__ void d_k_explicit_cam(int bid, int n_items, const BaItem *__restrict__ items, const int32_t *__restrict__ pt_idx,
               const double *__restrict__ W, const double *__restrict__ WV, const double *__restrict__ tg,
               const double *__restrict__ Wk, double *__restrict__ part, const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  const int wid = (bid * BA_THREADS + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (wid >= n_items) return;
  const BaItem it = items[wid];
  constexpr int NV = 6 + (NK ? 24 : 0);
  double acc[NV];
#pragma unroll
  for (int k = 0; k < NV; ++k) acc[k] = 0.0;
  for (int i = it.begin + lane; i < it.end; i += 32) {
    const int p = pt_idx[i];
    const double t0 = tg[3 * (size_t)p], t1 = tg[3 * (size_t)p + 1], t2 = tg[3 * (size_t)p + 2];
#pragma unroll
    for (int a = 0; a < 6; ++a) {
      const double *w = W + 18 * (size_t)i + 3 * a;
      acc[a] += w[0] * t0 + w[1] * t1 + w[2] * t2;
    }
    if (NK) {
      const double *wk = Wk + 12 * (size_t)p;
#pragma unroll
      for (int a = 0; a < 6; ++a) {
        const double *wv = WV + 18 * (size_t)i + 3 * a;
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[6 + a * 4 + b] += wv[0] * wk[3 * b] + wv[1] * wk[3 * b + 1] + wv[2] * wk[3 * b + 2];
      }
    }
  }
#pragma unroll
  for (int k = 0; k < NV; ++k) acc[k] = warp_sum(acc[k]);
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < NV; ++k) part[(size_t)wid * NV + k] = acc[k];
  }
}
template <int NK>
__global__ void __launch_bounds__(BA_THREADS)
k_explicit_cam(int n_items, const BaItem *__restrict__ items, const int32_t *__restrict__ pt_idx,
               const double *__restrict__ W, const double *__restrict__ WV, const double *__restrict__ tg,
               const double *__restrict__ Wk, double *__restrict__ part, const LmState *st, int gate) {
  d_k_explicit_cam<NK>(blockIdx.x, n_items, items, pt_idx, W, WV, tg, Wk, part, st, gate);
}

// intrinsics corner: per-CTA partials over points of Wk V^-1 Wk^T (10 upper
// entries) and Wk (V^-1 g_p) (4)
__device__ __forceinline__ void d_k_explicit_kk(int bid, int n_pt, const double *__restrict__ Wk, const double *__restrict__ Vinv, const double *__restrict__ tg,
              double *__restrict__ part, const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  __shared__ double red[BA_WARPS + 1];
  const int p = bid * BA_THREADS + threadIdx.x;
  double v[14];
#pragma unroll
  for (int k = 0; k < 14; ++k) v[k] = 0.0;
  if (p < n_pt) {
    double vi[6], wk[4][3], wv[4][3];
#pragma unroll
    for (int k = 0; k < 6; ++k) vi[k] = Vinv[6 * (size_t)p + k];
#pragma unroll
    for (int a = 0; a < 4; ++a) {
#pragma unroll
      for (int b = 0; b < 3; ++b) wk[a][b] = Wk[12 * (size_t)p + 3 * a + b];
      sym3_mul(vi, wk[a], wv[a]);
    }
    int u = 0;
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = a; b < 4; ++b) v[u++] = wv[a][0] * wk[b][0] + wv[a][1] * wk[b][1] + wv[a][2] * wk[b][2];
#pragma unroll
    for (int a = 0; a < 4; ++a)
      v[10 + a] = wk[a][0] * tg[3 * (size_t)p] + wk[a][1] * tg[3 * (size_t)p + 1] + wk[a][2] * tg[3 * (size_t)p + 2];
  }
#pragma unroll
  for (int k = 0; k < 14; ++k) {
    const double s = block_sum(v[k], red);
    if (threadIdx.x == 0) part[14 * (size_t)bid + k] = s;
  }
}
__global__ void __launch_bounds__(BA_THREADS)
k_explicit_kk(int n_pt, const double *__restrict__ Wk, const double *__restrict__ Vinv, const double *__restrict__ tg,
              double *__restrict__ part, const LmState *st, int gate) {
  d_k_explicit_kk(blockIdx.x, n_pt, Wk, Vinv, tg, part, st, gate);
}

// REF mode: camera-side vectors and the intrinsics corner in one launch (CTAs [0, nb_item) / [nb_item, ..))
__global__ void __launch_bounds__(BA_THREADS)
k_explicit_cam_kk(int nb_item, int n_items, const BaItem *__restrict__ items, const int32_t *__restrict__ pt_idx,
                  const double *__restrict__ W, const double *__restrict__ WV, const double *__restrict__ tg,
                  const double *__restrict__ Wk, double *__restrict__ part, int n_pt, const double *__restrict__ Vinv,
                  double *__restrict__ part_kk, const LmState *st, int gate) {
  if ((int)blockIdx.x < nb_item)
    d_k_explicit_cam<4>(blockIdx.x, n_items, items, pt_idx, W, WV, tg, Wk, part, st, gate);
  else
    d_k_explicit_kk(blockIdx.x - nb_item, n_pt, Wk, Vinv, tg, part_kk, st, gate);
}

// camera-camera blocks: one CTA per block (ci <= cj) of the block-sparse pair structure (keys ci * n_cam + cj, pair
// ranges blk_ptr, pairs (ia << 32) | ib in point-major order, *n_keys blocks), then n_xdiag empty diagonal blocks of free
// cameras without observations (keys xdiag); CTAs past the table return.
// thread = (entry of the 6x6 block, slice of the pair run); fixed-order
// reduction over the slices in shared memory.
//   S_ij = [i==j] (U_i + D_i^2) - sum_{(a,b)} WV_a W_b^T        (i, j: camera slots)
// SLICES = 28 (1008 threads) when the blocks are few and their pair runs long (windows), 7 otherwise
template <int SLICES>
__global__ void __launch_bounds__(SLICES * 36, 2048 / (SLICES * 36))  // (32 registers: 2 / 8 CTAs per SM)
k_schur_pairs(int n, int n_cam, int fixed_cam, const int32_t *__restrict__ n_keys, const unsigned long long *__restrict__ keys,
              const int32_t *__restrict__ blk_ptr, const unsigned long long *__restrict__ xdiag, int n_xdiag,
              const unsigned long long *__restrict__ pairs, const double *__restrict__ W,
              const double *__restrict__ WV, const double *__restrict__ U, const double *__restrict__ dc,
              double *__restrict__ S, const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  __shared__ double sm[SLICES * 36];
  const int blk = blockIdx.x;
  // (blk_ptr holds an entry for every launched CTA: the range loads go out together with the block count)
  const int nk = *n_keys, p0 = blk_ptr[blk], p1 = blk_ptr[blk + 1];
  if (blk >= nk + n_xdiag) return;
  const bool own = blk < nk;
  const int e = threadIdx.x % 36, sl = threadIdx.x / 36;
  const int row = e / 6, col = e % 6;
  // the loop is bound by the index -> block gather latency: four pairs per round, all index loads issued before
  // the first block load; the slice's partial is (even pairs) + (odd pairs), a fixed order
  double acc0 = 0.0, acc1 = 0.0;
  const int k1 = own ? p1 : 0;
  for (int k = (own ? p0 : 0) + sl; k < k1; k += 4 * SLICES) {
    int ia[4], ib[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int kk = k + u * SLICES;
      const int2 v = kk < k1 ? reinterpret_cast<const int2 *>(pairs)[kk] : make_int2(0, -1);  // (low word ib, high word ia)
      ia[u] = v.y;
      ib[u] = v.x;
    }
    double t[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      t[u] = 0.0;
      if (ia[u] >= 0) {
        const double *wv = WV + 18 * (size_t)ia[u] + 3 * row;
        const double *w = W + 18 * (size_t)ib[u] + 3 * col;
        t[u] = wv[0] * w[0] + wv[1] * w[1] + wv[2] * w[2];
      }
    }
    acc0 += t[0];
    acc1 += t[1];
    acc0 += t[2];
    acc1 += t[3];
  }
  sm[sl * 36 + e] = acc0 + acc1;
  __syncthreads();
  if (threadIdx.x < 36) {
    double s = 0.0;
#pragma unroll
    for (int q = 0; q < SLICES; ++q) s += sm[q * 36 + e];
    const uint32_t key = (uint32_t)(own ? keys[blk] : xdiag[blk - nk]);  // (dense S: n_cam <= BA_EXPLICIT_MAX_DIM / 6, so n_cam^2 < 2^32)
    const int c = (int)(key / (uint32_t)n_cam), cj = (int)(key % (uint32_t)n_cam);
    const int i = fixed_cam >= 0 && c > fixed_cam ? c - 1 : c, j = fixed_cam >= 0 && cj > fixed_cam ? cj - 1 : cj;
    double v = -s;
    if (i == j) {
      v += U[36 * (size_t)c + e];
      if (row == col) {
        const double D = sqrt(dc[6 * (size_t)c + row] / st->radius);
        v += D * D;
      }
    }
    S[(size_t)(6 * i + row) * n + 6 * j + col] = v;
    if (i != j) S[(size_t)(6 * j + col) * n + 6 * i + row] = v;
  }
}

// borders + right-hand side.  One thread per (camera, value): 6 right-hand-side entries and (REF mode) the 6 x 4
// border block of a free camera, item partials added in item order; 14 more threads own the intrinsics corner
// (10 upper entries of the 4 x 4 block + 4 right-hand-side entries, point-tile partials added in tile order).
//   rhs = -g + W V^-1 g_p
template <int NK>
__global__ void __launch_bounds__(BA_THREADS)
k_explicit_assemble(int n_cam, int n_free, int n, const int32_t *__restrict__ cam_slot, const int32_t *__restrict__ item_ptr,
                    const double *__restrict__ part_cam, int nblk_pt, const double *__restrict__ part_kk,
                    const double *__restrict__ gc, const double *__restrict__ Uck, const double *__restrict__ Ukk,
                    const double *__restrict__ gk, const double *__restrict__ dk, double *__restrict__ S,
                    double *__restrict__ rhs, const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  constexpr int NV = 6 + (NK ? 24 : 0);
  const int idx = blockIdx.x * BA_THREADS + threadIdx.x;
  const int koff = 6 * n_free;
  if (idx < n_cam * NV) {
    const int c = idx / NV, k = idx - c * NV;
    const int slot = cam_slot[c];
    if (slot < 0) return;
    double acc = 0.0;
    for (int it = item_ptr[c]; it < item_ptr[c + 1]; ++it) acc += part_cam[(size_t)it * NV + k];
    if (k < 6) {
      rhs[6 * slot + k] = -gc[6 * (size_t)c + k] + acc;
    } else if (NK) {
      const int a = (k - 6) >> 2, b = (k - 6) & 3;
      const double v = Uck[24 * (size_t)c + k - 6] - acc;
      S[(size_t)(6 * slot + a) * n + koff + b] = v;
      S[(size_t)(koff + b) * n + 6 * slot + a] = v;
    }
  } else if (NK && idx < n_cam * NV + 14) {
    const int k = idx - n_cam * NV;
    double v = 0.0;
    for (int b = 0; b < nblk_pt; ++b) v += part_kk[14 * (size_t)b + k];
    if (k < 10) {
      int a = 0, r = k;  // k-th entry of the row-major upper triangle of the 4 x 4 block -> (a, b)
      while (r >= 4 - a) {
        r -= 4 - a;
        ++a;
      }
      const int b = a + r;
      double x = Ukk[a * 4 + b] - v;
      if (a == b) {
        const double D = sqrt(dk[a] / st->radius);
        x += D * D;
      }
      S[(size_t)(koff + a) * n + koff + b] = x;
      S[(size_t)(koff + b) * n + koff + a] = x;
    } else {
      rhs[koff + k - 10] = -gk[k - 10] + v;
    }
  }
}

// =====================================================================
// Multi-GPU glue (points sharded across ranks, SURVEY.md 8e): local
// per-camera sums / scalars are packed into dense buffers that NCCL all-reduces
// in place; the single-GPU kernels then consume them through an identity
// item_ptr (one "item" per camera) or a 1-entry partial array.
// =====================================================================
template <int NV>
__global__ void __launch_bounds__(BA_THREADS)
k_sum_items(int n_cam, const int32_t *__restrict__ item_ptr, const double *__restrict__ part, double *__restrict__ out,
            const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  const int idx = blockIdx.x * BA_THREADS + threadIdx.x;
  if (idx >= n_cam * NV) return;
  const int c = idx / NV, k = idx - c * NV;
  double s = 0.0;
  for (int it = item_ptr[c]; it < item_ptr[c + 1]; ++it) s += part[(size_t)it * NV + k];
  out[idx] = s;
}
__global__ void __launch_bounds__(BA_THREADS)
k_reduce_partials(int n, const double *__restrict__ part, double *__restrict__ out, int is_max, const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  __shared__ double red[BA_WARPS + 2];
  const double v = is_max ? block_max_array(part, n, red) : block_sum_array(part, n, red);
  if (threadIdx.x == 0) out[0] = v;
}
__global__ void k_flags_pack(const LmState *st, double *out) {
  pdl_wait();
  out[0] = (double)st->eval_fail;
  out[1] = (double)st->lin_fail;
}
__global__ void k_flags_unpack(LmState *st, const double *in) {
  pdl_wait();
  if (in[0] != 0.0) st->eval_fail = 1;
  if (in[1] != 0.0) st->lin_fail = 1;
}
__global__ void k_iota(int n, int32_t *p) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = i;
}
