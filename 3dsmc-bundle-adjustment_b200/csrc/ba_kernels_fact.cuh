// ba_kernels_fact.cuh -- FACTORED Jacobian store for the large NS-mode problems
// (reprojection only, fixed intrinsics, implicit-Schur PCG: configs 3-5).
//
// The 2x6 / 2x3 Jacobian blocks of one observation are functions of FOUR
// per-observation numbers and of per-camera / per-point data:
//     g = (X/Z, Y/Z, 1/Z, w)        w = sqrt(weight) * sqrt(rho'(s))  (Huber)
//     Jc = diag(w fx, w fy) [ -iz  0  iz xz   xz yz   -(1+xz^2)   yz ] diag(s_c)
//                           [  0 -iz  iz yz  1+yz^2    -xz yz    -xz ]
//     Jp = diag(w fx iz, w fy iz) [ R^T row0 - xz R^T row2 ] diag(s_p)
//                                 [ R^T row1 - yz R^T row2 ]
// (Appendix B of SURVEY.md; s_c, s_p = Jacobi column scales, R = R(q) of the
// camera).  Instead of materialising 144 B of Jacobian per observation, the store
// keeps per observation one 32-byte record g (one 256-bit load or store) and the
// 16-byte residual r, and every consumer rebuilds the entries in registers.  The
// point scale s_p is folded into per-point quantities (V^-1, t, y_p are kept
// pre-scaled) so the camera-major kernels never gather it.
//
// Layout and readers:
//   geo  per camera: R (from k_cam_geo, the one R every projection uses) and s_c.
//   Fc_  camera-major r / g, written by kf_linearize; read by kf_cam_blocks,
//        kf_schur_pass2, kf_schur_diag and k_sp_schur.
//   Fp_  point-major r / g, only for the implicit solver (its PCG product runs
//        kf_schur_pass1 every iteration); filled by kf_pt_linearize<1, .>.
//        The block-sparse solvers neither allocate nor fill it: kf_pt_linearize<0, .>
//        reduces V, g_p straight from the projection, and the step evaluation
//        kf_step_eval projects again.  All projections go through
//        project_obs with R from geo, so a recomputed g equals the stored one bit for bit.
#pragma once
#include "ba_kernels.cuh"

struct FPlanes {
  double2 *r;  // robustified residual (r0, r1)
  double4 *g;  // (X/Z, Y/Z, 1/Z, w), 32-byte records
};

// per-camera record, 16 doubles = one 128-byte line: R (9, row-major), s (6, zero
// for the constant pose :299 so that its Jacobian columns vanish), pad
#define BA_CAMREC 16
// shared-memory staging of a point tile's camera run (kf_pt_linearize, kf_schur_pass1, kf_step_eval): at most BA_STAGE_CAMS
// cameras
#define BA_STAGE_CAMS 96
#define BA_STAGE_REC 18
struct CamRec {
  double R[9];
  double s[6];
};
__device__ __forceinline__ void load_camrec(const double *__restrict__ geo, int c, CamRec &cr) {
  const double2 *p = reinterpret_cast<const double2 *>(geo + (size_t)BA_CAMREC * c);
  const double2 a = ldg2(p), b = ldg2(p + 1), d = ldg2(p + 2), e = ldg2(p + 3), f = ldg2(p + 4), g = ldg2(p + 5),
                h = ldg2(p + 6), i = ldg2(p + 7);
  cr.R[0] = a.x; cr.R[1] = a.y; cr.R[2] = b.x; cr.R[3] = b.y; cr.R[4] = d.x; cr.R[5] = d.y; cr.R[6] = e.x; cr.R[7] = e.y;
  cr.R[8] = f.x; cr.s[0] = f.y; cr.s[1] = g.x; cr.s[2] = g.y; cr.s[3] = h.x; cr.s[4] = h.y; cr.s[5] = i.x;
}

__global__ void __launch_bounds__(BA_THREADS)
k_cam_geo(int n_cam, int fixed_cam, const double *__restrict__ pose, const double *__restrict__ sc, double *__restrict__ geo,
          const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  const int c = blockIdx.x * BA_THREADS + threadIdx.x;
  if (c >= n_cam) return;
  const double q[4] = {pose[7 * (size_t)c], pose[7 * (size_t)c + 1], pose[7 * (size_t)c + 2], pose[7 * (size_t)c + 3]};
  double R[9];
  quat_to_R(q, R);
  double *o = geo + (size_t)BA_CAMREC * c;
#pragma unroll
  for (int k = 0; k < 9; ++k) o[k] = R[k];
#pragma unroll
  for (int k = 0; k < 6; ++k) o[9 + k] = (c == fixed_cam) ? 0.0 : sc[6 * (size_t)c + k];
  o[15] = 0.0;
}

// packed per-camera input of pass 1: (s .* v)(6), R (9), pad
__global__ void __launch_bounds__(BA_THREADS)
k_pack_camx(int n_cam, const double *__restrict__ v, const double *__restrict__ geo, double *__restrict__ camx,
            const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  const int c = blockIdx.x * BA_THREADS + threadIdx.x;
  if (c >= n_cam) return;
  const double *g = geo + (size_t)BA_CAMREC * c;
  double *o = camx + (size_t)BA_CAMREC * c;
#pragma unroll
  for (int k = 0; k < 6; ++k) o[k] = g[9 + k] * v[6 * (size_t)c + k];
#pragma unroll
  for (int k = 0; k < 9; ++k) o[6 + k] = g[k];
  o[15] = 0.0;
}

// rows of diag(w fx, w fy)^-1 Jc diag(s)^-1 applied to a 6-vector / transposed
struct ObsGeo {
  double xz, yz, iz, wfx, wfy;
};
__device__ __forceinline__ void jc_dot(const ObsGeo &o, const double x[6], double &a0, double &a1) {
  a0 = o.wfx * (o.iz * (o.xz * x[2] - x[0]) + (o.xz * o.yz) * x[3] - (1.0 + o.xz * o.xz) * x[4] + o.yz * x[5]);
  a1 = o.wfy * (o.iz * (o.yz * x[2] - x[1]) + (1.0 + o.yz * o.yz) * x[3] - (o.xz * o.yz) * x[4] - o.xz * x[5]);
}
// acc += (Jc diag(s)^-1)^T (a0, a1)
__device__ __forceinline__ void jc_tacc(const ObsGeo &o, double a0, double a1, double acc[6]) {
  const double c0 = o.wfx * a0, c1 = o.wfy * a1;
  acc[0] -= o.iz * c0;
  acc[1] -= o.iz * c1;
  acc[2] += o.iz * (o.xz * c0 + o.yz * c1);
  acc[3] += (o.xz * o.yz) * c0 + (1.0 + o.yz * o.yz) * c1;
  acc[4] -= (1.0 + o.xz * o.xz) * c0 + (o.xz * o.yz) * c1;
  acc[5] += o.yz * c0 - o.xz * c1;
}
// (Jp diag(s_p)^-1) t = diag(wfx iz, wfy iz) [u0 - xz u2; u1 - yz u2], u = R^T t
__device__ __forceinline__ void jp_dot(const ObsGeo &o, const double R[9], const double t[3], double &b0, double &b1) {
  const double u0 = (R[0] * t[0] + R[3] * t[1]) + R[6] * t[2];
  const double u1 = (R[1] * t[0] + R[4] * t[1]) + R[7] * t[2];
  const double u2 = (R[2] * t[0] + R[5] * t[1]) + R[8] * t[2];
  b0 = (o.wfx * o.iz) * (u0 - o.xz * u2);
  b1 = (o.wfy * o.iz) * (u1 - o.yz * u2);
}
// (Jp diag(s_p)^-1)^T (a0, a1) = R (al0, al1, -(xz al0 + yz al1))
__device__ __forceinline__ void jp_tmul(const ObsGeo &o, const double R[9], double a0, double a1, double v[3]) {
  const double al0 = (o.wfx * o.iz) * a0, al1 = (o.wfy * o.iz) * a1;
  const double al2 = -(o.xz * al0 + o.yz * al1);
  v[0] = (R[0] * al0 + R[1] * al1) + R[2] * al2;
  v[1] = (R[3] * al0 + R[4] * al1) + R[5] * al2;
  v[2] = (R[6] * al0 + R[7] * al1) + R[8] * al2;
}
// 256-bit accesses of the 32-byte g record (LDG.E.256 / STG.E.256 on sm_100a): streaming load, L1 load, streaming store
__device__ __forceinline__ double4 lds4(const double4 *p) {
  double4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(v.x), "=d"(v.y), "=d"(v.z), "=d"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ double4 ldg4(const double4 *p) {
  double4 v;
  asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(v.x), "=d"(v.y), "=d"(v.z), "=d"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ void sts4(double4 *p, double4 v) {
  asm volatile("st.global.L1::no_allocate.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(p), "d"(v.x), "d"(v.y), "d"(v.z), "d"(v.w));
}
__device__ __forceinline__ ObsGeo obs_geo(double4 g, double fx, double fy) {
  ObsGeo o;
  o.xz = g.x;
  o.yz = g.y;
  o.iz = g.z;
  o.wfx = g.w * fx;
  o.wfy = g.w * fy;
  return o;
}
__device__ __forceinline__ ObsGeo load_geo(const FPlanes &F, int i, double fx, double fy) { return obs_geo(lds4(F.g + i), fx, fy); }

// R of camera c as k_cam_geo stored it
__device__ __forceinline__ void load_R(const double *__restrict__ geo, int c, double R[9]) {
  const double2 *p = reinterpret_cast<const double2 *>(geo + (size_t)BA_CAMREC * c);
  const double2 a = ldg2(p), b = ldg2(p + 1), d = ldg2(p + 2), e = ldg2(p + 3);
  R[0] = a.x; R[1] = a.y; R[2] = b.x; R[3] = b.y; R[4] = d.x; R[5] = d.y; R[6] = e.x; R[7] = e.y;
  R[8] = ldg1(geo + (size_t)BA_CAMREC * c + 8);
}

// The projection of one observation: camera rotation R (from geo) and centre C, point X, measurement m, intrinsics
// K = (fx, fy, cx, cy).  Every linearisation of the factored store and the back-substitution's recompute go through this
// one function, so the g they form agree bit for bit.
struct ObsProj {
  double r0, r1;       // robustified residual
  double xz, yz, iz, w;  // the g record
  double rho;          // rho(s), the cost term is rho / 2
};
__device__ __forceinline__ ObsProj project_obs(const double R[9], const double C[3], const double X3[3], double2 m,
                                               double4 K, const CostParams &cp) {
  const double d0 = X3[0] - C[0], d1 = X3[1] - C[1], d2 = X3[2] - C[2];
  const double X = (R[0] * d0 + R[3] * d1) + R[6] * d2;
  const double Y = (R[1] * d0 + R[4] * d1) + R[7] * d2;
  const double Z = (R[2] * d0 + R[5] * d1) + R[8] * d2;
  ObsProj o;
  o.iz = 1.0 / Z;
  o.xz = X * o.iz;
  o.yz = Y * o.iz;
  const double r0 = cp.sw_repr * ((K.x * o.xz + K.z) - m.x);
  const double r1 = cp.sw_repr * ((K.y * o.yz + K.w) - m.y);
  const double hs = huber_scale(cp.hub_repr, r0 * r0 + r1 * r1, o.rho);
  o.r0 = r0 * hs;
  o.r1 = r1 * hs;
  o.w = cp.sw_repr * hs;
  return o;
}
__device__ __forceinline__ double4 load_intr(const double *__restrict__ intr) {
  return make_double4(ldg1(intr), ldg1(intr + 1), ldg1(intr + 2), ldg1(intr + 3));
}
__device__ __forceinline__ void load_pt(const double *__restrict__ pt, int p, double X3[3]) {
  const double *q = pt + 3 * (size_t)p;
  X3[0] = ldg1(q);
  X3[1] = ldg1(q + 1);
  X3[2] = ldg1(q + 2);
}

// ------------------------------------------------------------------ linearise (camera-major)
// 96 B/obs: uv 16 + idx 8 + point 24 read; r 16 + g 32 written (R and centre are per camera: broadcast within an item)
__global__ void __launch_bounds__(BA_THREADS)
kf_linearize(int n_obs, const int32_t *__restrict__ cam_idx, const int32_t *__restrict__ pt_idx,
             const double2 *__restrict__ uv, const double *__restrict__ pose, const double *__restrict__ pt,
             const double *__restrict__ geo, const double *__restrict__ intr, CostParams cp, FPlanes F,
             double *__restrict__ cost_part, LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  __shared__ double red[BA_WARPS + 1];
  const int i = blockIdx.x * BA_THREADS + threadIdx.x;
  double cost = 0.0;
  if (i < n_obs) {
    const int c = cam_idx[i];
    double R[9], X3[3];
    load_R(geo, c, R);
    const double *P = pose + 7 * (size_t)c;
    const double C[3] = {ldg1(P + 4), ldg1(P + 5), ldg1(P + 6)};
    load_pt(pt, pt_idx[i], X3);
    const ObsProj o = project_obs(R, C, X3, lds2(uv + i), load_intr(intr), cp);
    cost = 0.5 * o.rho;
    sts2(F.r + i, make_double2(o.r0, o.r1));
    sts4(F.g + i, make_double4(o.xz, o.yz, o.iz, o.w));
    if (!(isfinite(o.r0) && isfinite(o.r1) && isfinite(o.iz))) st->eval_fail = 1;
  }
  const double s = block_sum(cost, red);
  if (threadIdx.x == 0) cost_part[blockIdx.x] = s;
}

// ------------------------------------------------------------------ camera blocks
// U (21) + g (6) per work item; Jc rebuilt from g and the camera's column scale
__global__ void __launch_bounds__(BA_THREADS)
kf_cam_blocks(int n_items, const BaItem *__restrict__ items, FPlanes F, const double *__restrict__ geo,
              const double *__restrict__ intr, double *__restrict__ part, const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  const int wid = (blockIdx.x * BA_THREADS + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (wid >= n_items) return;
  const BaItem it = items[wid];
  const double fx = ldg1(intr), fy = ldg1(intr + 1);
  double acc[27];
#pragma unroll
  for (int k = 0; k < 27; ++k) acc[k] = 0.0;
  for (int i = it.begin + lane; i < it.end; i += 32) {
    const ObsGeo o = load_geo(F, i, fx, fy);
    const double2 r = lds2(F.r + i);
    // rows of Jc diag(s)^-1
    const double j0[6] = {-o.wfx * o.iz, 0.0, o.wfx * o.iz * o.xz, o.wfx * o.xz * o.yz, -o.wfx * (1.0 + o.xz * o.xz), o.wfx * o.yz};
    const double j1[6] = {0.0, -o.wfy * o.iz, o.wfy * o.iz * o.yz, o.wfy * (1.0 + o.yz * o.yz), -o.wfy * o.xz * o.yz, -o.wfy * o.xz};
    int u = 0;
#pragma unroll
    for (int a = 0; a < 6; ++a)
#pragma unroll
      for (int b = a; b < 6; ++b) {
        acc[u] = fma(j1[a], j1[b], fma(j0[a], j0[b], acc[u]));
        ++u;
      }
#pragma unroll
    for (int a = 0; a < 6; ++a) acc[21 + a] = fma(j1[a], r.y, fma(j0[a], r.x, acc[21 + a]));
  }
  {
    // apply the column scale once per item and lane (compile-time indices): U_ab *= s_a s_b, g_a *= s_a; then the warp sum by
    // recursive halving (27 butterflies were half of this kernel's instructions): lane l writes the entry it ends up with
    const double *s = geo + (size_t)BA_CAMREC * it.cam + 9;
    double sv[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) sv[k] = ldg1(s + k);
    int u = 0;
#pragma unroll
    for (int a = 0; a < 6; ++a)
#pragma unroll
      for (int b = a; b < 6; ++b) {
        acc[u] *= sv[a] * sv[b];
        ++u;
      }
#pragma unroll
    for (int a = 0; a < 6; ++a) acc[21 + a] *= sv[a];
    int idx, cnt;
    warp_reduce_scatter<27>(acc, lane, idx, cnt);
    if (cnt > 0) part[(size_t)wid * 27 + idx] = acc[0];
  }
}

// ------------------------------------------------------------------ point-major linearisation
// V_p (6), g_p (3) and the clamped LM diagonal, reduced straight from the projection: no record plane is written and read
// back.  The point's column scale is applied once.  The tile's cameras (R 9, centre 3) are staged in shared memory as in
// kf_schur_pass1; STAGED = 0 gathers them from geo and pose.  STORE = 1 also writes the point-major r / g records, which
// only the implicit solver's product reads.  Algorithmic traffic: 48 B/obs (uv 16, cam and point idx 8, point 24; + 48 B
// written with STORE) + 72 B/point.
#define BA_LIN_REC 12
template <int STORE, int STAGED>
__global__ void __launch_bounds__(BA_THREADS, 3)
kf_pt_linearize(int n_pt, const int32_t *__restrict__ pt_rowptr, const int32_t *__restrict__ pm_cam,
                const int32_t *__restrict__ pm_pt, const double2 *__restrict__ pm_uv, const double *__restrict__ pose,
                const double *__restrict__ pt, const double *__restrict__ geo, const int32_t *__restrict__ tile_lo,
                const int32_t *__restrict__ tile_span, const double *__restrict__ intr, CostParams cp,
                const double *__restrict__ sp, FPlanes F, double *__restrict__ V, double *__restrict__ gp,
                double *__restrict__ dp, LmOptions lo, const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  constexpr int TOBS = 512;
  __shared__ double sm[9 * TOBS];
  __shared__ __align__(16) double rec[STAGED ? BA_STAGE_CAMS * BA_LIN_REC : 2];
  int cam_lo = 0;
  if (STAGED) {
    cam_lo = tile_lo[blockIdx.x];
    const int n = tile_span[blockIdx.x];
    for (int idx = threadIdx.x; idx < n * BA_LIN_REC; idx += BA_THREADS) {
      const int rc = idx / BA_LIN_REC, k = idx - rc * BA_LIN_REC;
      const size_t c = (size_t)(cam_lo + rc);
      rec[idx] = k < 9 ? geo[c * BA_CAMREC + k] : pose[7 * c + 4 + (k - 9)];
    }
    __syncthreads();
  }
  const double4 K = load_intr(intr);
  tile_point_reduce<9, TOBS>(
      n_pt, pt_rowptr, sm,
      [&](int s, double *v) {
        const int c = pm_cam[s];
        double R[9], C[3], X3[3];
        if (STAGED) {
          const double2 *cr = reinterpret_cast<const double2 *>(rec + (c - cam_lo) * BA_LIN_REC);
          const double2 a = cr[0], b = cr[1], d = cr[2], e = cr[3], f = cr[4], g = cr[5];
          R[0] = a.x; R[1] = a.y; R[2] = b.x; R[3] = b.y; R[4] = d.x; R[5] = d.y; R[6] = e.x; R[7] = e.y; R[8] = f.x;
          C[0] = f.y; C[1] = g.x; C[2] = g.y;
        } else {
          load_R(geo, c, R);
          const double *P = pose + 7 * (size_t)c;
          C[0] = ldg1(P + 4); C[1] = ldg1(P + 5); C[2] = ldg1(P + 6);
        }
        load_pt(pt, pm_pt[s], X3);
        const ObsProj pr = project_obs(R, C, X3, lds2(pm_uv + s), K, cp);
        if (STORE) {
          sts2(F.r + s, make_double2(pr.r0, pr.r1));
          sts4(F.g + s, make_double4(pr.xz, pr.yz, pr.iz, pr.w));
        }
        const ObsGeo o = obs_geo(make_double4(pr.xz, pr.yz, pr.iz, pr.w), K.x, K.y);
        const double a = o.wfx * o.iz, b = o.wfy * o.iz;
        double p0[3], p1[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          p0[k] = a * (R[3 * k] - o.xz * R[3 * k + 2]);
          p1[k] = b * (R[3 * k + 1] - o.yz * R[3 * k + 2]);
        }
        v[0] = p0[0] * p0[0] + p1[0] * p1[0];
        v[1] = p0[0] * p0[1] + p1[0] * p1[1];
        v[2] = p0[0] * p0[2] + p1[0] * p1[2];
        v[3] = p0[1] * p0[1] + p1[1] * p1[1];
        v[4] = p0[1] * p0[2] + p1[1] * p1[2];
        v[5] = p0[2] * p0[2] + p1[2] * p1[2];
#pragma unroll
        for (int k = 0; k < 3; ++k) v[6 + k] = p0[k] * pr.r0 + p1[k] * pr.r1;
      },
      [&](int p, const double *sum) {
        const double s0 = sp[3 * (size_t)p], s1 = sp[3 * (size_t)p + 1], s2 = sp[3 * (size_t)p + 2];
        const double v[6] = {sum[0] * (s0 * s0), sum[1] * (s0 * s1), sum[2] * (s0 * s2),
                             sum[3] * (s1 * s1), sum[4] * (s1 * s2), sum[5] * (s2 * s2)};
#pragma unroll
        for (int k = 0; k < 6; ++k) V[6 * (size_t)p + k] = v[k];
        gp[3 * (size_t)p] = sum[6] * s0;
        gp[3 * (size_t)p + 1] = sum[7] * s1;
        gp[3 * (size_t)p + 2] = sum[8] * s2;
        dp[3 * (size_t)p + 0] = fmin(fmax(v[0], lo.min_lm_diagonal), lo.max_lm_diagonal);
        dp[3 * (size_t)p + 1] = fmin(fmax(v[3], lo.min_lm_diagonal), lo.max_lm_diagonal);
        dp[3 * (size_t)p + 2] = fmin(fmax(v[5], lo.min_lm_diagonal), lo.max_lm_diagonal);
      });
}

// V^-1 as k_point_inverse, plus the pre-scaled copies the camera-major kernels use:
//   Vs = diag(s) V^-1 diag(s)   and   tgs = s .* (V^-1 g_p)
__global__ void __launch_bounds__(BA_THREADS)
kf_point_inverse(int n_pt, const double *__restrict__ V, const double *__restrict__ dp, const double *__restrict__ gp,
                 const double *__restrict__ sp, double *__restrict__ Vinv, double *__restrict__ Vs, double *__restrict__ tgs,
                 LmState *st, int gate) {
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
  const double s0 = sp[3 * (size_t)p], s1 = sp[3 * (size_t)p + 1], s2 = sp[3 * (size_t)p + 2];
#pragma unroll
  for (int k = 0; k < 6; ++k) Vinv[6 * (size_t)p + k] = vi[k];
  Vs[6 * (size_t)p + 0] = vi[0] * (s0 * s0);
  Vs[6 * (size_t)p + 1] = vi[1] * (s0 * s1);
  Vs[6 * (size_t)p + 2] = vi[2] * (s0 * s2);
  Vs[6 * (size_t)p + 3] = vi[3] * (s1 * s1);
  Vs[6 * (size_t)p + 4] = vi[4] * (s1 * s2);
  Vs[6 * (size_t)p + 5] = vi[5] * (s2 * s2);
  const double g[3] = {gp[3 * (size_t)p], gp[3 * (size_t)p + 1], gp[3 * (size_t)p + 2]};
  double t[3];
  sym3_mul(vi, g, t);
  *(reinterpret_cast<double4 *>(tgs) + p) = make_double4(t[0] * s0, t[1] * s1, t[2] * s2, 0.0);
}

// ------------------------------------------------------------------ pass 1 (point-major)
//   ts_p = s .* V^-1 (s .* sum_o Jpu^T (Jc x_c))      (the implicit solver's matvec)
// Algorithmic traffic: 36 B/obs (g 32 + cam idx 4) + 80 B/point.
// The per-camera operand (s.*x (6), R (9)) of every
// observation comes from SHARED MEMORY: a tile of 128 consecutive points touches a
// short run of cameras (tracks are runs of consecutive keyframes, points are numbered
// by first appearance), so the CTA stages that run once, 144-byte records (bank-conflict
// free for 8 consecutive cameras).  STAGED = 0 is the fallback for inputs whose
// tiles span more than BA_STAGE_CAMS cameras: the records are gathered through L1.
// kf_step_eval (below) stages the same way.

// per point tile: first camera and number of cameras spanned by its observations
__global__ void __launch_bounds__(BA_THREADS)
k_tile_cam_range(int n_pt, const int32_t *__restrict__ pt_rowptr, const int32_t *__restrict__ pm_cam, int32_t *__restrict__ tile_lo,
                 int32_t *__restrict__ tile_span, int32_t *max_span) {
  __shared__ int lo_s[BA_WARPS], hi_s[BA_WARPS];
  const int p0 = blockIdx.x * BA_TILE_PTS, p1 = min(n_pt, p0 + BA_TILE_PTS);
  const int o0 = pt_rowptr[p0], o1 = pt_rowptr[p1];
  int lo = 0x7fffffff, hi = -1;
  for (int s = o0 + threadIdx.x; s < o1; s += BA_THREADS) {
    const int c = pm_cam[s];
    lo = min(lo, c);
    hi = max(hi, c);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    lo = min(lo, __shfl_xor_sync(BA_FULL, lo, o));
    hi = max(hi, __shfl_xor_sync(BA_FULL, hi, o));
  }
  if ((threadIdx.x & 31) == 0) {
    lo_s[threadIdx.x >> 5] = lo;
    hi_s[threadIdx.x >> 5] = hi;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 0; w < BA_WARPS; ++w) {
      lo = min(lo, lo_s[w]);
      hi = max(hi, hi_s[w]);
    }
    const int span = hi >= lo ? hi - lo + 1 : 0;
    tile_lo[blockIdx.x] = hi >= lo ? lo : 0;
    tile_span[blockIdx.x] = span;
    atomicMax(max_span, span);
  }
}

template <int STAGED>
__global__ void __launch_bounds__(BA_THREADS, 5)
kf_schur_pass1(int n_pt, const int32_t *__restrict__ pt_rowptr, const int32_t *__restrict__ pm_cam, FPlanes F,
               const double *__restrict__ geo, const double *__restrict__ x, const double *__restrict__ camx,
               const int32_t *__restrict__ tile_lo, const int32_t *__restrict__ tile_span, const double *__restrict__ intr,
               const double *__restrict__ Vinv, const double *__restrict__ sp, double *__restrict__ out_s, const LmState *st,
               int gate) {
  if (!gate_open(st, gate)) return;
  constexpr int TOBS = 512;
  __shared__ double sm[3 * TOBS];
  __shared__ __align__(16) double rec[STAGED ? BA_STAGE_CAMS * BA_STAGE_REC : 2];
  const double4 K = load_intr(intr);
  int cam_lo = 0;
  if (STAGED) {
    constexpr int NREC = 16;
    cam_lo = tile_lo[blockIdx.x];
    const int n = tile_span[blockIdx.x];
    for (int idx = threadIdx.x; idx < n * NREC; idx += BA_THREADS) {
      const int rc = idx / NREC, k = idx - rc * NREC;
      const size_t c = (size_t)(cam_lo + rc);
      double v;
      if (k < 6)
        v = geo[c * BA_CAMREC + 9 + k] * x[c * 6 + k];
      else if (k < 15)
        v = geo[c * BA_CAMREC + (k - 6)];
      else
        v = 0.0;
      rec[rc * BA_STAGE_REC + k] = v;
    }
    __syncthreads();
  }
  tile_point_reduce<3, TOBS>(
      n_pt, pt_rowptr, sm,
      [&](int s, double *v) {
        const int c = pm_cam[s];
        double2 c0, c1, c2, c3, c4, c5, c6, c7;
        if (STAGED) {
          const double2 *cx = reinterpret_cast<const double2 *>(rec + (c - cam_lo) * BA_STAGE_REC);
          c0 = cx[0]; c1 = cx[1]; c2 = cx[2]; c3 = cx[3]; c4 = cx[4]; c5 = cx[5]; c6 = cx[6]; c7 = cx[7];
        } else {
          const double2 *cx = reinterpret_cast<const double2 *>(camx + (size_t)BA_CAMREC * c);
          c0 = ldg2(cx); c1 = ldg2(cx + 1); c2 = ldg2(cx + 2); c3 = ldg2(cx + 3); c4 = ldg2(cx + 4); c5 = ldg2(cx + 5);
          c6 = ldg2(cx + 6); c7 = ldg2(cx + 7);
        }
        const double xx[6] = {c0.x, c0.y, c1.x, c1.y, c2.x, c2.y};
        const double R[9] = {c3.x, c3.y, c4.x, c4.y, c5.x, c5.y, c6.x, c6.y, c7.x};
        const ObsGeo o = load_geo(F, s, K.x, K.y);
        double a0, a1;
        jc_dot(o, xx, a0, a1);
        jp_tmul(o, R, a0, a1, v);
      },
      [&](int p, const double *sum) {
        double vi[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) vi[k] = Vinv[6 * (size_t)p + k];
        const double s[3] = {sp[3 * (size_t)p], sp[3 * (size_t)p + 1], sp[3 * (size_t)p + 2]};
        double b[3], t[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) b[k] = s[k] * sum[k];
        sym3_mul(vi, b, t);
        // pre-scaled copy, padded to 32 bytes: one 256-bit gather per observation in pass 2
        double4 *o4 = reinterpret_cast<double4 *>(out_s) + p;
        *o4 = make_double4(s[0] * t[0], s[1] * t[1], s[2] * t[2], 0.0);
      });
}

// 256-bit read-only gather (LDG.E.256 on sm_100a)
__device__ __forceinline__ void ldg256(const double *p, double &a, double &b, double &c) {
  double d;
  asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p));
  (void)d;  // padding lane of the 32-byte record
}

// ------------------------------------------------------------------ pass 2 (camera-major items)
//   part[item] = s_c .* sum_o Jcu^T (alpha Jcu (s_c .* x_c) - Jpu ts_p)
// Algorithmic traffic: 36 B/obs (g 32 + pt idx 4) + ts_p gather 32 B/obs.
__global__ void __launch_bounds__(BA_THREADS, 3)
kf_schur_pass2(int n_items, const BaItem *__restrict__ items, const int32_t *__restrict__ pt_idx, FPlanes F,
               const double *__restrict__ geo, const double *__restrict__ intr, const double *__restrict__ x,
               const double *__restrict__ ts, double alpha, double *__restrict__ part, const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  const int wid = (blockIdx.x * BA_THREADS + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (wid >= n_items) return;
  const BaItem it = items[wid];
  const double fx = ldg1(intr), fy = ldg1(intr + 1);
  CamRec cr;
  load_camrec(geo, it.cam, cr);
  double xs[6];
  {
    double xv[6];
    load6(x + 6 * (size_t)it.cam, xv);
#pragma unroll
    for (int k = 0; k < 6; ++k) xs[k] = alpha * (cr.s[k] * xv[k]);
  }
  double acc[6] = {0, 0, 0, 0, 0, 0};
  int i = it.begin + lane;
  // two observations per lane and trip: both index loads, then both gathers, in flight together
  for (; i + 32 < it.end; i += 64) {
    const int pa = __ldg(pt_idx + i), pb = __ldg(pt_idx + i + 32);
    const ObsGeo oa = load_geo(F, i, fx, fy), ob = load_geo(F, i + 32, fx, fy);
    double ta[3], tb[3];
    ldg256(ts + 4 * (size_t)pa, ta[0], ta[1], ta[2]);
    ldg256(ts + 4 * (size_t)pb, tb[0], tb[1], tb[2]);
    double a0, a1, b0, b1;
    jc_dot(oa, xs, a0, a1);
    jp_dot(oa, cr.R, ta, b0, b1);
    jc_tacc(oa, a0 - b0, a1 - b1, acc);
    jc_dot(ob, xs, a0, a1);
    jp_dot(ob, cr.R, tb, b0, b1);
    jc_tacc(ob, a0 - b0, a1 - b1, acc);
  }
  if (i < it.end) {
    const int p = __ldg(pt_idx + i);
    const ObsGeo o = load_geo(F, i, fx, fy);
    double t[3];
    ldg256(ts + 4 * (size_t)p, t[0], t[1], t[2]);
    double a0, a1, b0, b1;
    jc_dot(o, xs, a0, a1);
    jp_dot(o, cr.R, t, b0, b1);
    jc_tacc(o, a0 - b0, a1 - b1, acc);
  }
#pragma unroll
  for (int k = 0; k < 6; ++k) acc[k] = warp_sum(acc[k]);
  if (lane == 0) {
    double *o = part + 6 * (size_t)wid;
#pragma unroll
    for (int k = 0; k < 6; ++k) o[k] = acc[k] * cr.s[k];
  }
}

// ------------------------------------------------------------------ SCHUR_JACOBI partials
__global__ void __launch_bounds__(BA_THREADS)
kf_schur_diag(int n_items, const BaItem *__restrict__ items, const int32_t *__restrict__ pt_idx, FPlanes F,
              const double *__restrict__ geo, const double *__restrict__ intr, const double *__restrict__ Vs,
              double *__restrict__ part, const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  const int wid = (blockIdx.x * BA_THREADS + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (wid >= n_items) return;
  const BaItem it = items[wid];
  const double fx = ldg1(intr), fy = ldg1(intr + 1);
  CamRec cr;
  load_camrec(geo, it.cam, cr);
  double acc[21];
#pragma unroll
  for (int k = 0; k < 21; ++k) acc[k] = 0.0;
  for (int i = it.begin + lane; i < it.end; i += 32) {
    const int p = __ldg(pt_idx + i);
    const ObsGeo o = load_geo(F, i, fx, fy);
    double vi[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) vi[k] = ldg1(Vs + 6 * (size_t)p + k);
    const double j0[6] = {-o.wfx * o.iz, 0.0, o.wfx * o.iz * o.xz, o.wfx * o.xz * o.yz, -o.wfx * (1.0 + o.xz * o.xz), o.wfx * o.yz};
    const double j1[6] = {0.0, -o.wfy * o.iz, o.wfy * o.iz * o.yz, o.wfy * (1.0 + o.yz * o.yz), -o.wfy * o.xz * o.yz, -o.wfy * o.xz};
    const double a = o.wfx * o.iz, b = o.wfy * o.iz;
    double p0[3], p1[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      p0[k] = a * (cr.R[3 * k] - o.xz * cr.R[3 * k + 2]);
      p1[k] = b * (cr.R[3 * k + 1] - o.yz * cr.R[3 * k + 2]);
    }
    double W[6][3], WV[6][3];
#pragma unroll
    for (int r = 0; r < 6; ++r) {
#pragma unroll
      for (int k = 0; k < 3; ++k) W[r][k] = j0[r] * p0[k] + j1[r] * p1[k];
      sym3_mul(vi, W[r], WV[r]);
    }
    int u = 0;
#pragma unroll
    for (int r = 0; r < 6; ++r)
#pragma unroll
      for (int c = r; c < 6; ++c) acc[u++] += WV[r][0] * W[c][0] + WV[r][1] * W[c][1] + WV[r][2] * W[c][2];
  }
#pragma unroll
  for (int k = 0; k < 21; ++k) acc[k] = warp_sum(acc[k]);
  if (lane == 0) {
    double *o = part + 21 * (size_t)wid;
    int u = 0;
#pragma unroll
    for (int r = 0; r < 6; ++r)
#pragma unroll
      for (int c = r; c < 6; ++c) {
        o[u] = acc[u] * (cr.s[r] * cr.s[c]);
        ++u;
      }
  }
}

// ------------------------------------------------------------------ step evaluation
// One point-major pass over a tile of BA_TILE_PTS points evaluates the LM step:
//   1. back-substitution  y_p = V^-1 (-g_p - s .* sum_o Jpu^T (Jc y_c)),  ys_p = s .* y_p  (J rebuilt by project_obs from
//      the inputs of kf_pt_linearize, so it is the J the linearisation used);
//   2. candidate point  pt_c = p + y_p .* s_p  and its share of |x+ - x|^2;
//   3. per observation, the model cost term m (r + m / 2), m = Jc (s_c .* y_c) + Jp ys_p (r and J projected again: the
//      bits kf_linearize stored), and the candidate cost rho / 2 at (pose_c, pt_c) (k_cost's arithmetic): two more loops
//      over the tile's observations, whose indices and measurements then come from L2.
// The candidate cameras pose_c come first (k_candidate over the cameras and the intrinsics entry only).  Per-tile partials of
// the three sums (fixed-order block sums, no atomics) go to part_mcc, part_step[step_off + tile] and part_cand.  The camera
// run is staged as in kf_schur_pass1: s.*y_c, R and centre (18 doubles), and the candidate camera's R(q+) and centre (12);
// STAGED = 0 gathers s.*y_c and R from camx (k_pack_camx), the centre from pose, and forms R(q+) per observation.
// Algorithmic traffic: 24 B/obs (uv 16, cam and point idx 8) + 224 B/point (pt 24, V^-1 48, s_p 24, g_p 24 read; y_p 24,
// ys_p 32, pt_c 24 written; the tile's points once more through L2 are not counted).
#define BA_CAND_REC 12
template <int STAGED>
__global__ void __launch_bounds__(BA_THREADS, 3)
kf_step_eval(int n_pt, const int32_t *__restrict__ pt_rowptr, const int32_t *__restrict__ pm_cam,
             const int32_t *__restrict__ pm_pt, const double2 *__restrict__ pm_uv, const double *__restrict__ pose,
             const double *__restrict__ pt, CostParams cp, const double *__restrict__ geo, const double *__restrict__ yc,
             const double *__restrict__ camx, const double *__restrict__ pose_c, const int32_t *__restrict__ tile_lo,
             const int32_t *__restrict__ tile_span, const double *__restrict__ intr, const double *__restrict__ intr_c,
             const double *__restrict__ Vinv, const double *__restrict__ sp, const double *__restrict__ gp,
             double *__restrict__ yp, double *__restrict__ ys, double *__restrict__ pt_c, double *__restrict__ part_mcc,
             double *__restrict__ part_step, int step_off, double *__restrict__ part_cand, const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  constexpr int TOBS = 512, PREC = 9;  // per point of the tile, after the reduction: X (3), ys (3), pt_c (3)
  static_assert(PREC * BA_TILE_PTS <= 3 * TOBS, "point records reuse the reduction buffer");
  __shared__ double sm[3 * TOBS];
  __shared__ __align__(16) double rec[STAGED ? BA_STAGE_CAMS * BA_STAGE_REC : 2];
  __shared__ __align__(16) double recc[STAGED ? BA_STAGE_CAMS * BA_CAND_REC : 2];
  __shared__ double red[BA_WARPS + 1];
  const double4 K = load_intr(intr);
  int cam_lo = 0;
  if (STAGED) {
    cam_lo = tile_lo[blockIdx.x];
    const int n = tile_span[blockIdx.x];
    for (int idx = threadIdx.x; idx < n * BA_STAGE_REC; idx += BA_THREADS) {
      const int rc = idx / BA_STAGE_REC, k = idx - rc * BA_STAGE_REC;
      const size_t c = (size_t)(cam_lo + rc);
      double v;
      if (k < 6)
        v = geo[c * BA_CAMREC + 9 + k] * yc[c * 6 + k];
      else if (k < 15)
        v = geo[c * BA_CAMREC + (k - 6)];
      else
        v = pose[7 * c + 4 + (k - 15)];
      rec[idx] = v;
    }
    for (int rc = threadIdx.x; rc < n; rc += BA_THREADS) {
      const double *P = pose_c + 7 * (size_t)(cam_lo + rc);
      const double q[4] = {P[0], P[1], P[2], P[3]};
      double *o = recc + rc * BA_CAND_REC;
      quat_to_R(q, o);
      o[9] = P[4]; o[10] = P[5]; o[11] = P[6];
    }
    __syncthreads();
  }
  // the current camera of observation s: s.*y_c, R, centre
  auto cam = [&](int c, double xx[6], double R[9], double C[3]) {
    double2 c0, c1, c2, c3, c4, c5, c6, c7;
    if (STAGED) {
      const double2 *cx = reinterpret_cast<const double2 *>(rec + (c - cam_lo) * BA_STAGE_REC);
      c0 = cx[0]; c1 = cx[1]; c2 = cx[2]; c3 = cx[3]; c4 = cx[4]; c5 = cx[5]; c6 = cx[6]; c7 = cx[7];
      const double2 c8 = cx[8];
      C[0] = c7.y; C[1] = c8.x; C[2] = c8.y;
    } else {
      const double2 *cx = reinterpret_cast<const double2 *>(camx + (size_t)BA_CAMREC * c);
      c0 = ldg2(cx); c1 = ldg2(cx + 1); c2 = ldg2(cx + 2); c3 = ldg2(cx + 3); c4 = ldg2(cx + 4); c5 = ldg2(cx + 5);
      c6 = ldg2(cx + 6); c7 = ldg2(cx + 7);
      const double *P = pose + 7 * (size_t)c;
      C[0] = ldg1(P + 4); C[1] = ldg1(P + 5); C[2] = ldg1(P + 6);
    }
    xx[0] = c0.x; xx[1] = c0.y; xx[2] = c1.x; xx[3] = c1.y; xx[4] = c2.x; xx[5] = c2.y;
    R[0] = c3.x; R[1] = c3.y; R[2] = c4.x; R[3] = c4.y; R[4] = c5.x; R[5] = c5.y; R[6] = c6.x; R[7] = c6.y; R[8] = c7.x;
  };
  const int p0 = blockIdx.x * BA_TILE_PTS, p1 = min(n_pt, p0 + BA_TILE_PTS);
  tile_point_reduce<3, TOBS>(
      n_pt, pt_rowptr, sm,
      [&](int s, double *v) {
        double xx[6], R[9], C[3], X3[3];
        cam(pm_cam[s], xx, R, C);
        load_pt(pt, pm_pt[s], X3);
        const ObsProj pr = project_obs(R, C, X3, lds2(pm_uv + s), K, cp);
        const ObsGeo o = obs_geo(make_double4(pr.xz, pr.yz, pr.iz, pr.w), K.x, K.y);
        double a0, a1;
        jc_dot(o, xx, a0, a1);
        jp_tmul(o, R, a0, a1, v);
      },
      [&](int p, const double *sum) {
        double vi[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) vi[k] = Vinv[6 * (size_t)p + k];
        const double s[3] = {sp[3 * (size_t)p], sp[3 * (size_t)p + 1], sp[3 * (size_t)p + 2]};
        double b[3], t[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) b[k] = s[k] * sum[k];
#pragma unroll
        for (int k = 0; k < 3; ++k) b[k] = -gp[3 * (size_t)p + k] - b[k];
        sym3_mul(vi, b, t);
        // the point's record for the loops below; the candidate point with k_candidate's arithmetic
        double *q = sm + PREC * (p - p0);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          yp[3 * (size_t)p + k] = t[k];
          const double x = pt[3 * (size_t)p + k];
          const double c = fma(t[k], s[k], x);  // (contracted as in k_candidate; s * t, rounded, is also formed below)
          pt_c[3 * (size_t)p + k] = c;
          q[k] = x;
          q[3 + k] = s[k] * t[k];
          q[6 + k] = c;
        }
        // pre-scaled copy, padded to 32 bytes: one 256-bit gather per observation in pass 2
        *(reinterpret_cast<double4 *>(ys) + p) = make_double4(q[3], q[4], q[5], 0.0);
      });
  __syncthreads();
  // the tile's share of |x+ - x|^2, written before the observation loops so that it holds no register through them
  double sn = 0.0;
  if (p0 + (int)threadIdx.x < p1) {
    const double *q = sm + PREC * threadIdx.x;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const double df = q[k] - q[6 + k];
      sn += df * df;
    }
  }
  sn = block_sum(sn, red);
  if (threadIdx.x == 0) part_step[step_off + blockIdx.x] = sn;
  // model cost change and candidate cost over the tile's observations: two loops, so that neither holds the other's
  // camera in registers (one loop spills at 80 registers)
  const double4 Kc = load_intr(intr_c);
  double mcc = 0.0, cand = 0.0;
  for (int s = pt_rowptr[p0] + threadIdx.x, o1 = pt_rowptr[p1]; s < o1; s += BA_THREADS) {
    const int c = pm_cam[s];
    const double *q = sm + PREC * (pm_pt[s] - p0);
    const double2 m = ldg2(pm_uv + s);
    double xx[6], R[9], C[3];
    cam(c, xx, R, C);
    {
      const double X3[3] = {q[0], q[1], q[2]}, t[3] = {q[3], q[4], q[5]};
      const ObsProj pr = project_obs(R, C, X3, m, K, cp);
      const ObsGeo o = obs_geo(make_double4(pr.xz, pr.yz, pr.iz, pr.w), K.x, K.y);
      double a0, a1, b0, b1;
      jc_dot(o, xx, a0, a1);
      jp_dot(o, R, t, b0, b1);
      const double m0 = a0 + b0, m1 = a1 + b1;
      mcc += m0 * (pr.r0 + m0 / 2.0) + m1 * (pr.r1 + m1 / 2.0);
    }
  }
  for (int s = pt_rowptr[p0] + threadIdx.x, o1 = pt_rowptr[p1]; s < o1; s += BA_THREADS) {
    const int c = pm_cam[s];
    const double *q = sm + PREC * (pm_pt[s] - p0);
    const double2 m = ldg2(pm_uv + s);
    double Rc[9], Cc[3];
    if (STAGED) {
      const double2 *cx = reinterpret_cast<const double2 *>(recc + (c - cam_lo) * BA_CAND_REC);
      const double2 a = cx[0], b = cx[1], d = cx[2], e = cx[3], f = cx[4], g = cx[5];
      Rc[0] = a.x; Rc[1] = a.y; Rc[2] = b.x; Rc[3] = b.y; Rc[4] = d.x; Rc[5] = d.y; Rc[6] = e.x; Rc[7] = e.y; Rc[8] = f.x;
      Cc[0] = f.y; Cc[1] = g.x; Cc[2] = g.y;
    } else {
      const double *P = pose_c + 7 * (size_t)c;
      const double q[4] = {ldg1(P), ldg1(P + 1), ldg1(P + 2), ldg1(P + 3)};
      quat_to_R(q, Rc);
      Cc[0] = ldg1(P + 4); Cc[1] = ldg1(P + 5); Cc[2] = ldg1(P + 6);
    }
    const double Xc[3] = {q[6], q[7], q[8]};
    cand += 0.5 * project_obs(Rc, Cc, Xc, m, Kc, cp).rho;
  }
  const double s_mcc = block_sum(mcc, red);
  const double s_cand = block_sum(cand, red);
  if (threadIdx.x == 0) {
    part_mcc[blockIdx.x] = s_mcc;
    part_cand[blockIdx.x] = s_cand;
  }
}
