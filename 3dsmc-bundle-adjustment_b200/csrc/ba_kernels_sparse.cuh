// ba_kernels_sparse.cuh -- EXPLICIT block-sparse Schur complement + PCG
// (BA_SOLVER_SPARSE_SCHUR_PCG): the reduced camera system of the large NS-mode
// problems formed once per LM iteration as a block-sparse symmetric matrix
//
//     S_ij = delta_ij U_i - sum_{p seen by i and j} W_ip V_p^-1 W_jp^T        (6x6 blocks)
//
// and multiplied by a block-CSR kernel inside PCG (== Ceres ITERATIVE_SCHUR with
// use_explicit_schur_complement, and the structure SPARSE_SCHUR factorises:
// src/OptimizationUtils.cpp:300 with linear_solver_type = SPARSE_SCHUR,
// headers/BundleAdjustmentConfig.h:63).  Sequential-SLAM problems have a very
// sparse S (config 5: 156k upper blocks = 45 MB for 10k cameras, L2-resident),
// so one PCG iteration reads tens of MB instead of streaming every observation.
//
// Structure (built once per upload, integer-only, on the device):
//   pairs   : for every point, all (a <= b) pairs of its free-camera observations
//             (point-major positions), keyed by (cam_a, cam_b); stable radix sort
//             by key => the pair list of every block, in point-major order
//             (the fixed summation order of the block)
//   blocks  : the distinct keys (upper triangle incl. diagonal), blk_ptr into pairs
//   rows    : per camera the entries (block, transposed?) in ascending column order
// Values: one warp per block walks its pair list; Jacobian entries are rebuilt from
// the factored point-major store (ba_kernels_fact.cuh).
#pragma once
#include "ba_kernels_fact.cuh"

// pairs per point: k (k + 1) / 2 over its free-camera observations
__global__ void __launch_bounds__(BA_THREADS)
k_sp_count(int n_pt, const int32_t *__restrict__ pt_rowptr, const int32_t *__restrict__ pm_cam, int fixed_cam,
           long long *__restrict__ cnt) {
  const int p = blockIdx.x * BA_THREADS + threadIdx.x;
  if (p > n_pt) return;
  long long k = 0, extra = 0;
  if (p < n_pt) {
    int prev = -1, run = 0;
    for (int s = pt_rowptr[p]; s < pt_rowptr[p + 1]; ++s) {
      const int c = pm_cam[s];
      if (c == fixed_cam) continue;
      ++k;
      run = (c == prev) ? run + 1 : 0;  // a camera seeing the point twice: both orders of the pair
      extra += run;
      prev = c;
    }
  }
  cnt[p] = k * (k + 1) / 2 + extra;  // cnt[n_pt] = 0: the scan's last entry is the total
}

__global__ void __launch_bounds__(BA_THREADS)
k_sp_emit(int n_pt, int n_cam, const int32_t *__restrict__ pt_rowptr, const int32_t *__restrict__ pm_cam,
          const int32_t *__restrict__ perm /* point-major slot -> canonical observation index */, int fixed_cam,
          const long long *__restrict__ off, unsigned long long *__restrict__ keys, unsigned long long *__restrict__ vals) {
  const int p = blockIdx.x * BA_THREADS + threadIdx.x;
  if (p >= n_pt) return;
  long long w = off[p];
  const int b0 = pt_rowptr[p], e0 = pt_rowptr[p + 1];
  for (int a = b0; a < e0; ++a) {
    const int ca = pm_cam[a];
    if (ca == fixed_cam) continue;
    for (int b = a; b < e0; ++b) {
      const int cb = pm_cam[b];
      if (cb == fixed_cam) continue;
      // cameras ascend inside a point's run (stable sort of a camera-major list): ca <= cb
      // pair records carry canonical (camera-major) observation indices: the a side indexes the row camera's own run
      const unsigned ia = (unsigned)perm[a], ib = (unsigned)perm[b];
      keys[w] = (unsigned long long)ca * (unsigned long long)n_cam + (unsigned long long)cb;
      vals[w] = ((unsigned long long)ia << 32) | ib;
      ++w;
      if (ca == cb && a != b) {  // same camera twice: the diagonal block also needs W_b V^-1 W_a^T
        keys[w] = keys[w - 1];
        vals[w] = ((unsigned long long)ib << 32) | ia;
        ++w;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Pair list of the DENSE explicit solver (windowed problems), built on the device instead of by the host loop
// of build_pair_list(): same enumeration as k_sp_emit, keyed by the dense upper-triangle index of the camera
// SLOT pair, values = the two CANONICAL (camera-major) observation indices; the per-block counts come from
// integer atomics (the counts, not the order, so the result is deterministic), the order inside a block from the
// stable radix sort = ascending point, as the host loop produces.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int ex_slot(int c, int fixed_cam) { return c == fixed_cam ? -1 : (fixed_cam >= 0 && c > fixed_cam ? c - 1 : c); }
__device__ __forceinline__ int ex_bidx(int i, int j, int nf) { return i * nf - i * (i - 1) / 2 + (j - i); }

__global__ void __launch_bounds__(BA_THREADS)
k_ex_emit(int n_pt, int nf, const int32_t *__restrict__ pt_rowptr, const int32_t *__restrict__ pm_cam,
          const int32_t *__restrict__ perm, int fixed_cam, const long long *__restrict__ off, uint32_t *__restrict__ keys,
          unsigned long long *__restrict__ vals, int32_t *blk_cnt) {
  const int p = blockIdx.x * BA_THREADS + threadIdx.x;
  if (p >= n_pt) return;
  long long w = off[p];
  const int b0 = pt_rowptr[p], e0 = pt_rowptr[p + 1];
  for (int a = b0; a < e0; ++a) {
    const int sa = ex_slot(pm_cam[a], fixed_cam);
    if (sa < 0) continue;
    const unsigned oa = (unsigned)perm[a];
    for (int b = a; b < e0; ++b) {
      const int sb = ex_slot(pm_cam[b], fixed_cam);
      if (sb < 0) continue;
      // cameras ascend inside a point's run (stable sort of a camera-major list): sa <= sb
      const int key = ex_bidx(sa, sb, nf);
      const unsigned ob = (unsigned)perm[b];
      keys[w] = (uint32_t)key;
      vals[w] = ((unsigned long long)oa << 32) | ob;
      ++w;
      int n = 1;
      if (sa == sb && a != b) {  // same camera twice: the diagonal block also needs W_b V^-1 W_a^T
        keys[w] = (uint32_t)key;
        vals[w] = ((unsigned long long)ob << 32) | oa;
        ++w;
        n = 2;
      }
      atomicAdd(&blk_cnt[key], n);
    }
  }
}

// sorted values -> pair_a / pair_b; block table of the dense upper triangle (every block listed; empty
// off-diagonal ones are skipped by k_schur_pairs)
__global__ void __launch_bounds__(BA_THREADS)
k_ex_finish(int n_pairs, const unsigned long long *__restrict__ vals, int32_t *__restrict__ pair_a, int32_t *__restrict__ pair_b,
            int nf, int fixed_cam, int32_t *__restrict__ blk_i, int32_t *__restrict__ blk_j, int32_t *__restrict__ blk_cam) {
  const int t = blockIdx.x * BA_THREADS + threadIdx.x;
  if (t < n_pairs) {
    const unsigned long long v = vals[t];
    pair_a[t] = (int32_t)(v >> 32);
    pair_b[t] = (int32_t)(v & 0xffffffffu);
  }
  if (t < nf * nf) {
    const int i = t / nf, j = t - i * nf;
    if (j >= i) {
      const int k = ex_bidx(i, j, nf);
      blk_i[k] = i;
      blk_j[k] = j;
      blk_cam[k] = (fixed_cam >= 0 && i >= fixed_cam) ? i + 1 : i;
    }
  }
}

// decode the distinct keys; per-row counts of upper and transposed entries
__global__ void __launch_bounds__(BA_THREADS)
k_sp_blocks(int n_blk, int n_cam, const unsigned long long *__restrict__ ukeys, int32_t *__restrict__ blk_i,
            int32_t *__restrict__ blk_j, int32_t *row_ucnt, int32_t *row_tcnt, unsigned long long *__restrict__ tkeys,
            int32_t *__restrict__ tvals) {
  const int b = blockIdx.x * BA_THREADS + threadIdx.x;
  if (b >= n_blk) return;
  const unsigned long long k = ukeys[b];
  const int i = (int)(k / (unsigned long long)n_cam), j = (int)(k % (unsigned long long)n_cam);
  blk_i[b] = i;
  blk_j[b] = j;
  atomicAdd(row_ucnt + i, 1);
  if (i != j) atomicAdd(row_tcnt + j, 1);
  // transposed list: sorted by (j, i); diagonal blocks get the largest key and are dropped
  tkeys[b] = i != j ? (unsigned long long)j * (unsigned long long)n_cam + (unsigned long long)i : ~0ull;
  tvals[b] = b;
}

// row r: transposed entries (columns < r, ascending) then upper entries (columns >= r, ascending)
// entry = (block index with bit 31 set when the block is used transposed, column)
__global__ void __launch_bounds__(BA_THREADS)
k_sp_entries(int n_cam, const int32_t *__restrict__ row_ustart, const int32_t *__restrict__ row_tstart,
             const int32_t *__restrict__ tvals_sorted, const int32_t *__restrict__ blk_i, const int32_t *__restrict__ blk_j,
             int32_t *__restrict__ ent_ptr, int2 *__restrict__ ent) {
  const int r = blockIdx.x * BA_THREADS + threadIdx.x;
  if (r > n_cam) return;
  const int base = row_ustart[r] + row_tstart[r];
  ent_ptr[r] = base;
  if (r == n_cam) return;
  int w = base;
  for (int e = row_tstart[r]; e < row_tstart[r + 1]; ++e, ++w) {
    const int b = tvals_sorted[e];
    ent[w] = make_int2((int)((uint32_t)b | 0x80000000u), blk_i[b]);
  }
  for (int b = row_ustart[r]; b < row_ustart[r + 1]; ++b, ++w) ent[w] = make_int2(b, blk_j[b]);
}

// sort keys of the PCG row order: rows by DECREASING entry count (ties by row index)
__global__ void __launch_bounds__(BA_THREADS)
k_sp_row_keys(int n_cam, const int32_t *__restrict__ ent_ptr, unsigned long long *__restrict__ keys, int32_t *__restrict__ vals) {
  const int r = blockIdx.x * BA_THREADS + threadIdx.x;
  if (r >= n_cam) return;
  const unsigned int cnt = (unsigned int)(ent_ptr[r + 1] - ent_ptr[r]);
  keys[r] = ((unsigned long long)(0xffffffffu - cnt) << 32) | (unsigned int)r;
  vals[r] = r;
}

// ------------------------------------------------------------------ values
// One warp per (local) block.  S_b = [i == j] U_i - diag(s_i) (sum_pairs W_a Vs_p W_b^T) diag(s_j),
// W_o = jr0_o (x) p0_o + jr1_o (x) p1_o (un-scaled rows rebuilt from the factored store).
// Through the 2x2 core M = P_a Vs P_b^T:  W_a Vs W_b^T = [jr0_a jr1_a] M [jr0_b jr1_b]^T.
__device__ __forceinline__ void sp_rows(const ObsGeo &o, const double R[9], double jr0[6], double jr1[6], double p0[3],
                                        double p1[3]) {
  jr0[0] = -o.wfx * o.iz; jr0[1] = 0.0; jr0[2] = o.wfx * o.iz * o.xz; jr0[3] = o.wfx * o.xz * o.yz;
  jr0[4] = -o.wfx * (1.0 + o.xz * o.xz); jr0[5] = o.wfx * o.yz;
  jr1[0] = 0.0; jr1[1] = -o.wfy * o.iz; jr1[2] = o.wfy * o.iz * o.yz; jr1[3] = o.wfy * (1.0 + o.yz * o.yz);
  jr1[4] = -o.wfy * o.xz * o.yz; jr1[5] = -o.wfy * o.xz;
  const double a = o.wfx * o.iz, b = o.wfy * o.iz;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    p0[k] = a * (R[3 * k] - o.xz * R[3 * k + 2]);
    p1[k] = b * (R[3 * k + 1] - o.yz * R[3 * k + 2]);
  }
}

// local block -> index in the common (all-rank) block list
__global__ void __launch_bounds__(BA_THREADS)
k_sp_lookup(int n_local, const unsigned long long *__restrict__ lkeys, int n_global, const unsigned long long *__restrict__ gkeys,
            int32_t *__restrict__ gid) {
  const int b = blockIdx.x * BA_THREADS + threadIdx.x;
  if (b >= n_local) return;
  const unsigned long long k = lkeys[b];
  int lo = 0, hi = n_global - 1;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (gkeys[mid] < k)
      lo = mid + 1;
    else
      hi = mid;
  }
  gid[b] = lo;
}
// diagonal block of every camera row (its first upper entry, if that is (c, c)), else -1
__global__ void __launch_bounds__(BA_THREADS)
k_sp_diag_index(int n_cam, const int32_t *__restrict__ row_ustart, const int32_t *__restrict__ blk_j, int32_t *__restrict__ diag) {
  const int c = blockIdx.x * BA_THREADS + threadIdx.x;
  if (c >= n_cam) return;
  const int b = row_ustart[c];
  diag[c] = (b < row_ustart[c + 1] && blk_j[b] == c) ? b : -1;
}
__global__ void __launch_bounds__(BA_THREADS)
k_sp_add_diag(int n_cam, const int32_t *__restrict__ diag, const double *__restrict__ U, double *__restrict__ S, const LmState *st,
              int gate) {
  if (!gate_open(st, gate)) return;
  const int i = blockIdx.x * BA_THREADS + threadIdx.x;
  if (i >= n_cam * 36) return;
  const int c = i / 36, k = i - 36 * c;
  const int b = diag[c];
  if (b >= 0) S[36 * (size_t)b + k] += U[36 * (size_t)c + k];
}

// gather (unpack = 0) / scatter (unpack = 1) of the blocks of S that are summed over ranks in the distributed factorisation
__global__ void __launch_bounds__(BA_THREADS)
k_sp_xpack(int nx, const int32_t *__restrict__ xidx, double *__restrict__ S, double *__restrict__ xbuf, int unpack, const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  const int i = blockIdx.x * BA_THREADS + threadIdx.x;
  if (i >= nx * 36) return;
  const int b = i / 36, k = i - 36 * b;
  double *src = S + 36 * (size_t)xidx[b] + k;
  if (unpack)
    *src = xbuf[i];
  else
    xbuf[i] = *src;
}

// point of every pair (gathered once per upload: one level less in the dependent-load chain of k_sp_schur)
__global__ void __launch_bounds__(BA_THREADS)
k_sp_pair_points(long long n_pairs, const unsigned long long *__restrict__ pairs, const int32_t *__restrict__ pt_idx,
                 int32_t *__restrict__ pair_pt) {
  const long long e = (long long)blockIdx.x * BA_THREADS + threadIdx.x;
  if (e < n_pairs) pair_pt[e] = pt_idx[(int)(pairs[e] >> 32)];  // (canonical observation index -> point)
}

// Persistent warps fetch blocks from a shared ticket counter (integer atomic): block sizes range from a
// handful of pairs to ~800 (diagonal blocks), a static block -> warp map leaves most warps of a CTA idle
// behind its largest block.  The order in which blocks are PROCESSED does not touch the result: every
// block is summed by one warp in its fixed pair order.
// SCHUR_JACOBI preconditioner straight from the explicit matrix: M_c^-1 = (S_cc + D_c^2)^-1 (the diagonal
// block already holds U_c - sum W V^-1 W^T), and the damping D^2 the product adds per column.
__global__ void __launch_bounds__(BA_THREADS)
k_sp_minv(int n_cam, const int32_t *__restrict__ diag, const double *__restrict__ S, const double *__restrict__ dc,
          double *__restrict__ Minv, double *__restrict__ dsq, LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  const int c = blockIdx.x * BA_THREADS + threadIdx.x;
  if (c >= n_cam) return;
  const double radius = st->radius;
  const int b = diag[c];
  double B[36], Bi[36];
  if (b >= 0) {
    const double *Sb = S + 36 * (size_t)b;
    // symmetrise from the upper triangle, as the packed partial sums of k_schur_diag_fin do
#pragma unroll
    for (int a = 0; a < 6; ++a)
#pragma unroll
      for (int k = a; k < 6; ++k) {
        const double v = Sb[a * 6 + k];
        B[a * 6 + k] = v;
        B[k * 6 + a] = v;
      }
  } else {
#pragma unroll
    for (int k = 0; k < 36; ++k) B[k] = 0.0;
  }
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    const double D = sqrt(dc[6 * (size_t)c + k] / radius);
    B[k * 6 + k] += D * D;
    dsq[6 * (size_t)c + k] = D * D;
  }
  if (!spd6_inverse(B, Bi)) st->lin_fail = 1;
#pragma unroll
  for (int k = 0; k < 36; ++k) Minv[36 * (size_t)c + k] = Bi[k];
}

// Blocks are handed out in CHUNKS of consecutive blocks (sorted by (row camera, column camera): a chunk is about two
// camera rows): the CTA takes a chunk from the global ticket counter, its warps take blocks of the chunk from a
// shared-memory counter (the diagonal block -- the longest pair list of a row -- comes first).  All warps of a CTA then
// gather the factored records of the SAME cameras' observations at the same time, through L1-allocating loads: the
// row camera's records are read by every block of the row and hit L1 after the first touch (ncu, round 1 version with
// one global ticket per block and L1-bypassing loads: 36 % of the stall samples on these gathers at 8 warps per SM;
// 1.43 -> 1.24 ms at config 5).  Pair records hold CANONICAL (camera-major) observation indices, so both sides of a
// block index the contiguous run of one camera in the camera-major factored planes.
// Measured and rejected in round 2 (config 5, same results): two CTAs per SM at 128 registers (accumulators spill to
// local memory: 1.57 ms); one camera ROW per CTA with the row's a side -- rows of Jc and Vs p-rows, 18 doubles per
// observation -- staged in shared memory, chunked work items and prefetched b-side records (40 B and ~140 multiply-adds
// per pair instead of 124 B and ~190, but three CTA-wide phases per row at 8 warps per SM: 1.92 ms); a two-trip software
// pipeline of the gathers in this kernel (252 registers: 1.36 ms).
#define BA_SPS_CHUNK 32
// Sum over the warp of 36 per-lane values by recursive halving: at every level a lane keeps one half of its values and
// receives the partner's partial sums of that half.  Afterwards lane l holds the complete sums of the entries
// idx .. idx + cnt - 1 (cnt <= 2) in acc[0..1]; the 36 entries are spread over the 32 lanes.
__device__ __forceinline__ void sp_reduce_scatter36(double (&acc)[36], int lane, int &idx, int &cnt) {
#define SP_HALVE(N, H, MASK)                                                        \
  {                                                                                 \
    const bool up = (lane & MASK) != 0;                                             \
    _Pragma("unroll") for (int i = 0; i < H; ++i) {                                 \
      const double lo = acc[i], hi = (i + H < N) ? acc[i + H] : 0.0;                \
      const double keep = up ? hi : lo, send = up ? lo : hi;                        \
      acc[i] = keep + __shfl_xor_sync(BA_FULL, send, MASK);                         \
    }                                                                               \
  }
  SP_HALVE(36, 18, 16)
  SP_HALVE(18, 9, 8)
  SP_HALVE(9, 5, 4)
  SP_HALVE(5, 3, 2)
  SP_HALVE(3, 2, 1)
#undef SP_HALVE
  idx = ((lane & 16) ? 18 : 0) + ((lane & 8) ? 9 : 0) + ((lane & 4) ? 5 : 0) + ((lane & 2) ? 3 : 0) + ((lane & 1) ? 2 : 0);
  int c = (lane & 4) ? 4 : 5;
  c = (lane & 2) ? c - 3 : 3;
  cnt = (lane & 1) ? (c > 2 ? c - 2 : 0) : (c < 2 ? c : 2);
}
__device__ __forceinline__ ObsGeo load_geo_l1(const FPlanes &F, int i, double fx, double fy) {
  const double2 a = __ldg(F.g0 + i), b = __ldg(F.g1 + i);
  ObsGeo o;
  o.xz = a.x;
  o.yz = a.y;
  o.iz = b.x;
  o.wfx = b.y * fx;
  o.wfy = b.y * fy;
  return o;
}
// The round-2 kernel: every lane holds the 36 accumulators of the block (238 registers, 8 warps per SM).  Kept only to
// alternate with k_sp_schur in one process (BA_SPS_SIMT=1, read at create); no solver selects it.
__global__ void __launch_bounds__(BA_THREADS)
k_sp_schur_simt(int n_blk, int n_cam, const int32_t *__restrict__ blk_ptr, const unsigned long long *__restrict__ lkeys,
           const int32_t *__restrict__ gid, const unsigned long long *__restrict__ pairs, const int32_t *__restrict__ pair_pt,
           FPlanes F, const double *__restrict__ geo, const double *__restrict__ intr, const double *__restrict__ Vs,
           double *__restrict__ S, int *ticket, const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  __shared__ int s_chunk, s_next;
  const int lane = threadIdx.x & 31;
  const double fx = ldg1(intr), fy = ldg1(intr + 1);
  for (;;) {
    __syncthreads();  // every warp is done with the previous chunk's counter
    if (threadIdx.x == 0) {
      s_chunk = atomicAdd(ticket, 1);
      s_next = 0;
    }
    __syncthreads();
    const int c0 = s_chunk * BA_SPS_CHUNK;
    if (c0 >= n_blk) return;
    const int cend = c0 + BA_SPS_CHUNK < n_blk ? c0 + BA_SPS_CHUNK : n_blk;
    for (;;) {
      int b = 0;
      if (lane == 0) b = c0 + atomicAdd(&s_next, 1);
      b = __shfl_sync(BA_FULL, b, 0);
      if (b >= cend) break;
      const unsigned long long key = lkeys[b];
      const int ci = (int)(key / (unsigned long long)n_cam), cj = (int)(key % (unsigned long long)n_cam);
      CamRec ri, rj;
      load_camrec(geo, ci, ri);
      load_camrec(geo, cj, rj);
      double acc[36];
#pragma unroll
      for (int k = 0; k < 36; ++k) acc[k] = 0.0;
      const int e1 = blk_ptr[b + 1];
      int e = blk_ptr[b] + lane;
      unsigned long long pr = 0;
      int p = 0;
      if (e < e1) {
        pr = pairs[e];
        p = __ldg(pair_pt + e);
      }
      while (e < e1) {
        // the next trip's pair record is fetched before this trip's gathers are consumed
        const int en = e + 32;
        unsigned long long prn = 0;
        int pn = 0;
        if (en < e1) {
          prn = pairs[en];
          pn = __ldg(pair_pt + en);
        }
        const int oa = (int)(pr >> 32), ob = (int)(pr & 0xffffffffu);
        double vs[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) vs[k] = ldg1(Vs + 6 * (size_t)p + k);
        const ObsGeo ga = load_geo_l1(F, oa, fx, fy), gb = load_geo_l1(F, ob, fx, fy);
        double a0[6], a1[6], pa0[3], pa1[3], b0[6], b1[6], pb0[3], pb1[3];
        sp_rows(ga, ri.R, a0, a1, pa0, pa1);
        sp_rows(gb, rj.R, b0, b1, pb0, pb1);
        double v0[3], v1[3];
        sym3_mul(vs, pa0, v0);
        sym3_mul(vs, pa1, v1);
        const double m00 = v0[0] * pb0[0] + v0[1] * pb0[1] + v0[2] * pb0[2];
        const double m01 = v0[0] * pb1[0] + v0[1] * pb1[1] + v0[2] * pb1[2];
        const double m10 = v1[0] * pb0[0] + v1[1] * pb0[1] + v1[2] * pb0[2];
        const double m11 = v1[0] * pb1[0] + v1[1] * pb1[1] + v1[2] * pb1[2];
#pragma unroll
        for (int c = 0; c < 6; ++c) {
          const double h0 = m00 * b0[c] + m01 * b1[c], h1 = m10 * b0[c] + m11 * b1[c];
#pragma unroll
          // (kept as product-sum + add: an fma chain through acc -- two DFMA instead of DMUL + DFMA + DADD -- measured slower,
          //  1.03 -> 1.13 ms: with two warps per scheduler the longer dependent chain per accumulator costs more than the instruction)
          for (int r = 0; r < 6; ++r) acc[r * 6 + c] += a0[r] * h0 + a1[r] * h1;
        }
        pr = prn;
        p = pn;
        e = en;
      }
      // column scales (compile-time indices), then the warp sum as a recursive halving: every lane ends up with at most two
      // COMPLETE entries of the block (37 shuffled doubles instead of the 180 of 36 butterflies; SASS of the butterfly
      // version: 722 SHFL, a quarter of the instructions of a block with ~155 pairs).  Fixed tree: deterministic.
#pragma unroll
      for (int k = 0; k < 36; ++k) acc[k] *= ri.s[k / 6] * rj.s[k % 6];
      int idx, cnt;
      sp_reduce_scatter36(acc, lane, idx, cnt);
      double *Sb = S + 36 * (size_t)gid[b] + idx;
      if (cnt > 0) Sb[0] = -acc[0];  // k_sp_add_diag puts U on the diagonal blocks
      if (cnt > 1) Sb[1] = -acc[1];
    }
  }
}

// Per block, S_b = -diag(s_i) [sum_pairs A_p^T H_p] diag(s_j) with A_p = [a0; a1] (2 x 6, rows of Jc in camera i) and
// H_p = M_p [b0; b1] (2 x 6, the 2x2 core times the rows of Jc in camera j): a dense fp64 contraction of 6 x 2n by 2n x 6,
// which is what mma.m8n8k4.f64 (DMMA) computes, two pairs per instruction, into an 8 x 8 accumulator (the 6 x 6 block
// padded) of 2 registers per lane.  The warp walks the block's pairs in trips of 32: lane j stages pair e0 + j -- the
// same gathers and arithmetic as k_sp_schur_simt -- as 12 double2 (a_t[r], h_t[r]) in its warp's slab, then the warp
// runs ceil(n / 2) DMMA steps over the slab.  Lanes past the block's end stage zeros, so an odd tail's second pair adds 0.
// Every block is summed in one fixed order (pair order, then the steps in order): bit-identical from run to run.
// Slab: entry q = 6 t + r of pair p at q * BA_SPS_LD + p.  A lane stages with 12 stores of consecutive double2 across the
// warp, and in step s lane (r = l >> 2, k = l & 3) reads entry (6 (k & 1) + r, 2 s + (k >> 1)) with one 16-byte load; with a
// row stride of 34 (= 2 mod 8 in 16-byte bank groups) the 8 lanes of each quarter-warp hit 8 distinct bank groups, for the
// stores and for the loads (a stride of 32 puts 4 of them on one group).
// Registers: 122, no spills, two CTAs (16 warps) per SM.  Three CTAs (80 registers) spill even with the rotations moved to
// shared memory and the pair-record prefetch dropped (16 to 40 bytes).
#define BA_SPS_LD 34
#define BA_SPS_SMEM (BA_THREADS / 32 * 12 * BA_SPS_LD * 16)
__device__ __forceinline__ void dmma_m8n8k4(double &d0, double &d1, double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}
__global__ void __launch_bounds__(BA_THREADS, 2)
k_sp_schur(int n_blk, int n_cam, const int32_t *__restrict__ blk_ptr, const unsigned long long *__restrict__ lkeys,
           const int32_t *__restrict__ gid, const unsigned long long *__restrict__ pairs, const int32_t *__restrict__ pair_pt,
           FPlanes F, const double *__restrict__ geo, const double *__restrict__ intr, const double *__restrict__ Vs,
           double *__restrict__ S, int *ticket, const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  extern __shared__ double2 sps_slab[];
  __shared__ int s_chunk, s_next;
  const int lane = threadIdx.x & 31, r = lane >> 2, k = lane & 3;
  double2 *slab = sps_slab + (threadIdx.x >> 5) * (12 * BA_SPS_LD);
  const double2 *frag = slab + (6 * (k & 1) + r) * BA_SPS_LD + (k >> 1);  // this lane's A / B operand in step 0
  const double fx = ldg1(intr), fy = ldg1(intr + 1);
  for (;;) {
    __syncthreads();  // every warp is done with the previous chunk's counter
    if (threadIdx.x == 0) {
      s_chunk = atomicAdd(ticket, 1);
      s_next = 0;
    }
    __syncthreads();
    const int c0 = s_chunk * BA_SPS_CHUNK;
    if (c0 >= n_blk) return;
    const int cend = c0 + BA_SPS_CHUNK < n_blk ? c0 + BA_SPS_CHUNK : n_blk;
    for (;;) {
      int b = 0;
      if (lane == 0) b = c0 + atomicAdd(&s_next, 1);
      b = __shfl_sync(BA_FULL, b, 0);
      if (b >= cend) break;
      const unsigned long long key = lkeys[b];
      const int ci = (int)(key / (unsigned long long)n_cam), cj = (int)(key % (unsigned long long)n_cam);
      CamRec ri, rj;
      load_camrec(geo, ci, ri);
      load_camrec(geo, cj, rj);
      double d0 = 0.0, d1 = 0.0;
      const int e1 = blk_ptr[b + 1];
      int e0 = blk_ptr[b];
      unsigned long long pr = 0;
      int p = 0;
      if (e0 + lane < e1) {
        pr = pairs[e0 + lane];
        p = __ldg(pair_pt + e0 + lane);
      }
      for (; e0 < e1; e0 += 32) {
        // the next trip's pair record is fetched before this trip's gathers are consumed
        const int en = e0 + 32 + lane;
        unsigned long long prn = 0;
        int pn = 0;
        if (en < e1) {
          prn = pairs[en];
          pn = __ldg(pair_pt + en);
        }
        // a lane past the block's end stages zeros: zero geometry (weights included) zeroes its rows and its core
        ObsGeo ga = {0.0, 0.0, 0.0, 0.0, 0.0}, gb = ga;
        double vs[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        if (e0 + lane < e1) {
          // Vs as three 16-byte loads (the record is 48 B, 16-byte aligned): every load instruction of these gathers touches
          // up to 32 different lines, and the L1 work of the six 8-byte loads was a third of the kernel's gather traffic
          const double2 *v2 = reinterpret_cast<const double2 *>(Vs) + 3 * (size_t)p;
          const double2 v01 = ldg2(v2), v23 = ldg2(v2 + 1), v45 = ldg2(v2 + 2);
          vs[0] = v01.x; vs[1] = v01.y; vs[2] = v23.x; vs[3] = v23.y; vs[4] = v45.x; vs[5] = v45.y;
          ga = load_geo_l1(F, (int)(pr >> 32), fx, fy);
          gb = load_geo_l1(F, (int)(pr & 0xffffffffu), fx, fy);
        }
        double a0[6], a1[6], pa0[3], pa1[3], b0[6], b1[6], pb0[3], pb1[3];
        sp_rows(ga, ri.R, a0, a1, pa0, pa1);
        sp_rows(gb, rj.R, b0, b1, pb0, pb1);
        double v0[3], v1[3];
        sym3_mul(vs, pa0, v0);
        sym3_mul(vs, pa1, v1);
        const double m00 = v0[0] * pb0[0] + v0[1] * pb0[1] + v0[2] * pb0[2];
        const double m01 = v0[0] * pb1[0] + v0[1] * pb1[1] + v0[2] * pb1[2];
        const double m10 = v1[0] * pb0[0] + v1[1] * pb0[1] + v1[2] * pb0[2];
        const double m11 = v1[0] * pb1[0] + v1[1] * pb1[1] + v1[2] * pb1[2];
#pragma unroll
        for (int c = 0; c < 6; ++c) {
          slab[c * BA_SPS_LD + lane] = make_double2(a0[c], m00 * b0[c] + m01 * b1[c]);
          slab[(6 + c) * BA_SPS_LD + lane] = make_double2(a1[c], m10 * b0[c] + m11 * b1[c]);
        }
        __syncwarp();
        const int n_step = ((e1 - e0 < 32 ? e1 - e0 : 32) + 1) >> 1;
        for (int s = 0; s < n_step; ++s) {
          double av = 0.0, bv = 0.0;  // rows / columns 6 and 7 of the padded block
          if (r < 6) {
            const double2 v = frag[2 * s];
            av = v.x;
            bv = v.y;
          }
          dmma_m8n8k4(d0, d1, av, bv);
        }
        __syncwarp();  // the slab is read before the next trip overwrites it
        pr = prn;
        p = pn;
      }
      // lane l holds entries (r, 2k) and (r, 2k + 1) of the block: scales, then -S (k_sp_add_diag puts U on the diagonal)
      if (r < 6 && k < 3) {
        const double *si = geo + BA_CAMREC * (size_t)ci + 9, *sj = geo + BA_CAMREC * (size_t)cj + 9;
        const double s_r = ldg1(si + r);
        *reinterpret_cast<double2 *>(S + 36 * (size_t)gid[b] + 6 * r + 2 * k) =
            make_double2(-(d0 * (s_r * ldg1(sj + 2 * k))), -(d1 * (s_r * ldg1(sj + 2 * k + 1))));
      }
    }
  }
}

// ------------------------------------------------------------------ y = S x  (without the LM damping)
// One warp per camera row; a lane multiplies whole 6x6 blocks (256-bit loads), the
// lane partials are combined by a fixed butterfly.  v = za (+ beta * pb) is formed on the
// fly (PCG direction update fused into the product); CG = 1 reads the vectors through L2
// (ld.global.cg) because other CTAs of the same launch wrote them.
__device__ __forceinline__ void ld256(const double *p, double &a, double &b, double &c, double &d) {
  asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p));
}
__device__ __forceinline__ void load6cg(const double *p, double v[6]) {
  const double2 *q = reinterpret_cast<const double2 *>(p);
  const double2 a = __ldcg(q), b = __ldcg(q + 1), c = __ldcg(q + 2);
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; v[4] = c.x; v[5] = c.y;
}
template <int CG>
__device__ __forceinline__ void bsr_row(int r, int lane, const int32_t *__restrict__ ent_ptr, const int2 *__restrict__ ent,
                                        const double *__restrict__ S, const double *za, const double *pb, double beta, bool use_pb,
                                        double acc[6]) {
#pragma unroll
  for (int k = 0; k < 6; ++k) acc[k] = 0.0;
  for (int e = __ldg(ent_ptr + r) + lane; e < __ldg(ent_ptr + r + 1); e += 32) {
    const int2 en = __ldg(ent + e);
    const double *B = S + 36 * (size_t)((uint32_t)en.x & 0x7fffffffu);
    double m[36], xv[6];
#pragma unroll
    for (int k = 0; k < 9; ++k) ld256(B + 4 * k, m[4 * k], m[4 * k + 1], m[4 * k + 2], m[4 * k + 3]);
    if (CG)
      load6cg(za + 6 * (size_t)en.y, xv);
    else
      load6(za + 6 * (size_t)en.y, xv);
    if (use_pb) {
      double pv[6];
      if (CG)
        load6cg(pb + 6 * (size_t)en.y, pv);
      else
        load6(pb + 6 * (size_t)en.y, pv);
#pragma unroll
      for (int k = 0; k < 6; ++k) xv[k] = xv[k] + beta * pv[k];
    }
    if ((uint32_t)en.x & 0x80000000u) {
#pragma unroll
      for (int a = 0; a < 6; ++a)
#pragma unroll
        for (int k = 0; k < 6; ++k) acc[a] += m[k * 6 + a] * xv[k];
    } else {
#pragma unroll
      for (int a = 0; a < 6; ++a)
#pragma unroll
        for (int k = 0; k < 6; ++k) acc[a] += m[a * 6 + k] * xv[k];
    }
  }
#pragma unroll
  for (int k = 0; k < 6; ++k) acc[k] = warp_sum(acc[k]);
}
__device__ __forceinline__ double pick6(const double a[6], int k) {
  return k == 0 ? a[0] : k == 1 ? a[1] : k == 2 ? a[2] : k == 3 ? a[3] : k == 4 ? a[4] : a[5];
}

// Experimental mapping (BA_SPMV6=1; measurement for the next step of the persistent PCG, DESIGN section 10): a block is shared
// by SIX lanes -- lane a of a group forms component a of (S_ij x_j), reading one 48-byte block row (or one strided column when
// the block is used transposed) -- and five groups walk the row's entries.  ~40 registers instead of ~230, so six times as many
// warps per SM keep loads in flight; the lanes of the same component are added in group order (fixed).
__global__ void __launch_bounds__(BA_THREADS)
k_bsr_spmv6(int n_cam, const int32_t *__restrict__ ent_ptr, const int2 *__restrict__ ent, const double *__restrict__ S,
            const double *__restrict__ x, double *__restrict__ y, const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  const int r = (blockIdx.x * BA_THREADS + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (r >= n_cam) return;
  const int g = lane / 6, a = lane - 6 * g;
  const int b0 = __ldg(ent_ptr + r), e0 = __ldg(ent_ptr + r + 1);
  double acc = 0.0;
  if (g < 5) {
#pragma unroll 4
    for (int e = b0 + g; e < e0; e += 5) {
      const int2 en = __ldg(ent + e);
      const double *B = S + 36 * (size_t)((uint32_t)en.x & 0x7fffffffu);
      double xv[6], m[6];
      load6(x + 6 * (size_t)en.y, xv);
      if ((uint32_t)en.x & 0x80000000u) {
#pragma unroll
        for (int k = 0; k < 6; ++k) m[k] = __ldg(B + 6 * k + a);
      } else {
        const double2 *row = reinterpret_cast<const double2 *>(B + 6 * a);
        const double2 m0 = __ldg(row), m1 = __ldg(row + 1), m2 = __ldg(row + 2);
        m[0] = m0.x; m[1] = m0.y; m[2] = m1.x; m[3] = m1.y; m[4] = m2.x; m[5] = m2.y;
      }
      double sdot = 0.0;
#pragma unroll
      for (int k = 0; k < 6; ++k) sdot += m[k] * xv[k];
      acc += sdot;
    }
  }
  double sum = acc;
#pragma unroll
  for (int gg = 1; gg < 5; ++gg) sum += __shfl_sync(BA_FULL, acc, (lane + 6 * gg) & 31);
  if (lane < 6) y[6 * (size_t)r + lane] = sum;
}

__global__ void __launch_bounds__(BA_THREADS)
k_bsr_spmv(int n_cam, const int32_t *__restrict__ ent_ptr, const int2 *__restrict__ ent, const double *__restrict__ S,
           const double *__restrict__ x, double *__restrict__ y, const LmState *st, int gate) {
  if (!gate_open(st, gate)) return;
  const int r = (blockIdx.x * BA_THREADS + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (r >= n_cam) return;
  double acc[6];
  bsr_row<0>(r, lane, ent_ptr, ent, S, x, x, 0.0, false, acc);
  if (lane == 0) store6(y + 6 * (size_t)r, acc);
}

// ------------------------------------------------------------------ persistent PCG
// The whole preconditioned-CG solve of one LM iteration in ONE cooperative launch:
// with S explicit a PCG iteration is ~10 us of work, so four launches per iteration
// (direction, product, q, step) plus a host poll every few iterations would leave the
// GPU idle most of the time.  Persistent CTAs (all co-resident) run
//     phase I   p = z + beta p_old (ping-pong buffers), q = S p + D^2 p, per-row p.q
//               (warps walk rows independently: no CTA barrier inside the phase)
//     phase II  alpha, x += alpha p, r -= alpha q, z = M^-1 r, partials of r.z and x.(b + r)
// separated by grid barriers (monotonic arrival counter, release/acquire through L2);
// every CTA then evaluates the Ceres CG controller (conjugate_gradients_solver.cc: quadratic
// model termination, rho / beta) from the same partials in the same order, so all CTAs
// take identical decisions with no broadcast.  Every residual_reset_period iterations
// r = b - S x is recomputed (one extra product).  Partials have a fixed granularity
// (rows, 256-camera blocks) => results do not depend on the grid size.
__device__ __forceinline__ void grid_barrier(unsigned int *bar, unsigned int &epoch) {
  __syncthreads();
  if (threadIdx.x == 0) {
    epoch += gridDim.x;
    __threadfence();
    atomicAdd(bar, 1u);
    while (*((volatile unsigned int *)bar) < epoch) {
    }
    __threadfence();
  }
  __syncthreads();
}
// every thread of the CTA gets sum(part[0..n)), part written by other CTAs
__device__ __forceinline__ double block_sum_array_cg(const double *part, int n, double *smem /*>=BA_WARPS+1*/) {
  double v = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) v += __ldcg(part + i);
  v = warp_sum(v);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) smem[w] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int i = 0; i < BA_WARPS; ++i) s += smem[i];
    smem[BA_WARPS] = s;
  }
  __syncthreads();
  return smem[BA_WARPS];
}

// one 6x6 block (or its transpose) times v = za[col] (+ beta pb[col]), accumulated into acc
__device__ __forceinline__ void bsr_entry(const int2 en, const double *__restrict__ S, const double *za, const double *pb,
                                          double beta, bool use_pb, double acc[6]) {
  const double *B = S + 36 * (size_t)((uint32_t)en.x & 0x7fffffffu);
  double m[36], xv[6];
#pragma unroll
  for (int k = 0; k < 9; ++k) ld256(B + 4 * k, m[4 * k], m[4 * k + 1], m[4 * k + 2], m[4 * k + 3]);
  load6cg(za + 6 * (size_t)en.y, xv);
  if (use_pb) {
    double pv[6];
    load6cg(pb + 6 * (size_t)en.y, pv);
#pragma unroll
    for (int k = 0; k < 6; ++k) xv[k] = xv[k] + beta * pv[k];
  }
  if ((uint32_t)en.x & 0x80000000u) {
#pragma unroll
    for (int a = 0; a < 6; ++a)
#pragma unroll
      for (int k = 0; k < 6; ++k) acc[a] += m[k * 6 + a] * xv[k];
  } else {
#pragma unroll
    for (int a = 0; a < 6; ++a)
#pragma unroll
      for (int k = 0; k < 6; ++k) acc[a] += m[a * 6 + k] * xv[k];
  }
}

// rows gw, gw + nw, ... of out = S v + dsq .* v with v = za (+ beta pb).  The row pointers
// are fetched two rows ahead and the first 32 entries one row ahead, so a row costs one
// dependent L2 round trip (its blocks).  MODE 0 (PCG direction): also writes v to pnew and
// the row's v.out to row_pq.  MODE 1 (residual reset): only out.
template <int MODE>
__device__ __forceinline__ void bsr_rows(int n_cam, int gw, int nw, int lane, const int32_t *__restrict__ order,
                                         const int32_t *__restrict__ ent_ptr, const int2 *__restrict__ ent,
                                         const double *__restrict__ S, const double *__restrict__ dsq, const double *za,
                                         const double *pb, double beta, bool use_pb, double *pnew, double *out,
                                         double *row_pq) {
  // rows order[gw], order[gw + nw], ...: `order` lists the rows by decreasing entry count, so the
  // round-robin deal gives every warp nearly the same number of blocks
  const int2 none = make_int2(0, 0);
  int idx = gw;
  if (idx >= n_cam) return;
  int row = __ldg(order + idx);
  int row1 = idx + nw < n_cam ? __ldg(order + idx + nw) : -1;
  int b0 = __ldg(ent_ptr + row), e0 = __ldg(ent_ptr + row + 1);
  int b1 = 0, e1 = 0;
  if (row1 >= 0) {
    b1 = __ldg(ent_ptr + row1);
    e1 = __ldg(ent_ptr + row1 + 1);
  }
  int2 en0 = b0 + lane < e0 ? __ldg(ent + b0 + lane) : none;
  int2 en0b = b0 + lane + 32 < e0 ? __ldg(ent + b0 + lane + 32) : none;
  for (; idx < n_cam; idx += nw) {
    // prefetch: first 64 entries of the next row, pointers of the one after
    const int2 en1 = b1 + lane < e1 ? __ldg(ent + b1 + lane) : none;
    const int2 en1b = b1 + lane + 32 < e1 ? __ldg(ent + b1 + lane + 32) : none;
    int b2 = 0, e2 = 0, row2 = -1;
    if (idx + 2 * nw < n_cam) {
      row2 = __ldg(order + idx + 2 * nw);
      b2 = __ldg(ent_ptr + row2);
      e2 = __ldg(ent_ptr + row2 + 1);
    }
    double zk = 0.0, pk = 0.0, dk = 0.0;
    if (lane < 6) {
      zk = __ldcg(za + 6 * (size_t)row + lane);
      if (use_pb) pk = __ldcg(pb + 6 * (size_t)row + lane);
      dk = __ldg(dsq + 6 * (size_t)row + lane);
    }
    double acc[6] = {0, 0, 0, 0, 0, 0};
    if (b0 + lane < e0) bsr_entry(en0, S, za, pb, beta, use_pb, acc);
    if (b0 + lane + 32 < e0) bsr_entry(en0b, S, za, pb, beta, use_pb, acc);
    for (int e = b0 + lane + 64; e < e0; e += 32) bsr_entry(__ldg(ent + e), S, za, pb, beta, use_pb, acc);
#pragma unroll
    for (int k = 0; k < 6; ++k) acc[k] = warp_sum(acc[k]);
    const double pv = use_pb ? zk + beta * pk : zk;
    const double qv = pick6(acc, lane) + dk * pv;
    if (lane < 6) {
      if (MODE == 0) pnew[6 * (size_t)row + lane] = pv;
      out[6 * (size_t)row + lane] = qv;
    }
    if (MODE == 0) {
      // v.out of the row, components added in order 0..5 (as k_pcg_q)
      const double t = pv * qv;
      double s = __shfl_sync(BA_FULL, t, 0);
#pragma unroll
      for (int k = 1; k < 6; ++k) s += __shfl_sync(BA_FULL, t, k);
      if (lane == 0) row_pq[row] = s;
    }
    row = row1; row1 = row2;
    b0 = b1; e0 = e1; en0 = en1; en0b = en1b;
    b1 = b2; e1 = e2;
  }
}

// The structure is constant over the PCG solve and a warp owns the same rows in every iteration:
// the entries of its first rows live in a per-warp shared-memory cache (BA_PCG_ENT_SLOTS trips of 32
// entries, BA_PCG_ROWS row records), so a cached row costs ONE dependent L2 round trip (its blocks).
#define BA_PCG_ENT_SLOTS 16
#define BA_PCG_ROWS 16
#define BA_PCG_SMEM_PER_WARP (36 * 32 * 8 + BA_PCG_ENT_SLOTS * 32 * 8 + BA_PCG_ROWS * 16)
template <int MODE>
__device__ __forceinline__ void bsr_rows_cached(int n_cam, int gw, int nw, int lane, int n_cached, const int4 *rowinfo,
                                                const int2 *ecache, const double *__restrict__ S,
                                                const double *__restrict__ dsq, const double *za, const double *pb, double beta,
                                                bool use_pb, double *pnew, double *out, double *row_pq) {
  int slot = 0;
  for (int i = 0; i < n_cached; ++i) {
    const int4 be = rowinfo[i];  // (first entry, end, row, -)
    const int row = be.z;
    double zk = 0.0, pk = 0.0, dk = 0.0;
    if (lane < 6) {
      zk = __ldcg(za + 6 * (size_t)row + lane);
      if (use_pb) pk = __ldcg(pb + 6 * (size_t)row + lane);
      dk = __ldg(dsq + 6 * (size_t)row + lane);
    }
    double acc[6] = {0, 0, 0, 0, 0, 0};
    for (int e = be.x; e < be.y; e += 32, ++slot) {
      const int2 en = ecache[slot * 32 + lane];
      if (e + lane < be.y) bsr_entry(en, S, za, pb, beta, use_pb, acc);
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) acc[k] = warp_sum(acc[k]);
    const double pv = use_pb ? zk + beta * pk : zk;
    const double qv = pick6(acc, lane) + dk * pv;
    if (lane < 6) {
      if (MODE == 0) pnew[6 * (size_t)row + lane] = pv;
      out[6 * (size_t)row + lane] = qv;
    }
    if (MODE == 0) {
      const double t = pv * qv;
      double sum = __shfl_sync(BA_FULL, t, 0);
#pragma unroll
      for (int k = 1; k < 6; ++k) sum += __shfl_sync(BA_FULL, t, k);
      if (lane == 0) row_pq[row] = sum;
    }
  }
}

// sum of n doubles written by other CTAs; every thread of the CTA gets it.  Fixed order:
// thread t adds elements t, t + 256, ... into 4 interleaved accumulators (loads in flight),
// then the usual butterfly / warp order.
__device__ __forceinline__ double block_sum_wide_cg(const double *part, int n, double *smem /*>=BA_WARPS+1*/) {
  // 16-byte loads, 4 in flight per thread; element order per thread is fixed (pairs t, t + 256, ...)
  const double2 *p2 = reinterpret_cast<const double2 *>(part);
  const int n2 = n >> 1;
  double v0 = 0.0, v1 = 0.0, v2 = 0.0, v3 = 0.0;
  int i = threadIdx.x;
  for (; i + 3 * BA_THREADS < n2; i += 4 * BA_THREADS) {
    const double2 a = __ldcg(p2 + i), b = __ldcg(p2 + i + BA_THREADS), c = __ldcg(p2 + i + 2 * BA_THREADS),
                  d = __ldcg(p2 + i + 3 * BA_THREADS);
    v0 += a.x + a.y;
    v1 += b.x + b.y;
    v2 += c.x + c.y;
    v3 += d.x + d.y;
  }
  for (; i < n2; i += BA_THREADS) {
    const double2 a = __ldcg(p2 + i);
    v0 += a.x + a.y;
  }
  if ((n & 1) && threadIdx.x == 0) v1 += __ldcg(part + n - 1);
  double v = (v0 + v1) + (v2 + v3);
  v = warp_sum(v);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) smem[w] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int k = 0; k < BA_WARPS; ++k) s += smem[k];
    smem[BA_WARPS] = s;
  }
  __syncthreads();
  return smem[BA_WARPS];
}

// two sums in one pass (the controller's r.z and x.(b + r)); red >= 2 * BA_WARPS + 2
__device__ __forceinline__ void block_sum2_cg(const double *pa, const double *pb, int n, double *red, double &sa, double &sb) {
  double v = 0.0, w = 0.0;
  for (int i = threadIdx.x; i < n; i += BA_THREADS) {
    v += __ldcg(pa + i);
    w += __ldcg(pb + i);
  }
  v = warp_sum(v);
  w = warp_sum(w);
  const int wid = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) {
    red[wid] = v;
    red[BA_WARPS + wid] = w;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0, t = 0.0;
    for (int k = 0; k < BA_WARPS; ++k) {
      s += red[k];
      t += red[BA_WARPS + k];
    }
    red[2 * BA_WARPS] = s;
    red[2 * BA_WARPS + 1] = t;
  }
  __syncthreads();
  sa = red[2 * BA_WARPS];
  sb = red[2 * BA_WARPS + 1];
}

// phase II for one warp-block of 32 cameras (lane = camera): no CTA barrier.  CACHED: M^-1 of the
// camera comes from the warp's shared-memory copy ([36][32] doubles, conflict-free) and b from registers
// (both constant during the solve, and a warp owns the same cameras in every iteration).
template <int RESET, int CACHED>
__device__ __forceinline__ void pcg_update_warp(int n_cam, int wb, int lane, double alpha, bool skip_r,
                                                const double *__restrict__ b, const double *__restrict__ Minv,
                                                const double *minv_s, const double breg[6], double *x, double *r, double *z,
                                                const double *pnew, const double *q, double *part_rho, double *part_Q) {
  const int c = wb * 32 + lane;
  double rz = 0.0, xq = 0.0;
  if (c < n_cam) {
    double xv[6], rv[6], qv[6], bv[6], zv[6];
    load6cg(x + 6 * (size_t)c, xv);
    if (!RESET) {
      double pv[6];
      load6cg(pnew + 6 * (size_t)c, pv);
#pragma unroll
      for (int k = 0; k < 6; ++k) xv[k] = xv[k] + alpha * pv[k];
      store6(x + 6 * (size_t)c, xv);
    }
    if (!skip_r) {
      load6cg(q + 6 * (size_t)c, qv);
      if (CACHED) {
#pragma unroll
        for (int k = 0; k < 6; ++k) bv[k] = breg[k];
      } else
        load6(b + 6 * (size_t)c, bv);
      if (RESET) {
#pragma unroll
        for (int k = 0; k < 6; ++k) rv[k] = bv[k] - qv[k];
      } else {
        load6cg(r + 6 * (size_t)c, rv);
#pragma unroll
        for (int k = 0; k < 6; ++k) rv[k] = rv[k] - alpha * qv[k];
      }
      store6(r + 6 * (size_t)c, rv);
      if (CACHED) {
#pragma unroll
        for (int a = 0; a < 6; ++a) {
          double sacc = 0.0;
#pragma unroll
          for (int k = 0; k < 6; ++k) sacc += minv_s[(a * 6 + k) * 32 + lane] * rv[k];
          zv[a] = sacc;
        }
      } else
        minv_mul(Minv, c, rv, zv);
      store6(z + 6 * (size_t)c, zv);
#pragma unroll
      for (int k = 0; k < 6; ++k) {
        rz += rv[k] * zv[k];
        xq += xv[k] * (bv[k] + rv[k]);
      }
    }
  }
  if (!skip_r) {
    rz = warp_sum(rz);
    xq = warp_sum(xq);
    if (lane == 0) {
      part_rho[wb] = rz;
      part_Q[wb] = xq;
    }
  }
}

__global__ void __launch_bounds__(BA_THREADS, 1)
k_pcg_sparse_persistent(int n_cam, const int32_t *__restrict__ row_order, const int32_t *__restrict__ ent_ptr,
                        const int2 *__restrict__ ent,
                        const double *__restrict__ S, const double *__restrict__ dsq, const double *__restrict__ b,
                        const double *__restrict__ Minv, double *x, double *r, double *z, double *pbuf0, double *pbuf1,
                        double *q, double *row_pq, double *part_rho, double *part_Q, unsigned int *bar, LmOptions lo,
                        LmState *st, unsigned long long *prof /* nullable: ns per phase, CTA 0 */) {
  if (st->done || st->pcg_done) return;  // identical on every CTA: the state is only written back after the last barrier
  __shared__ double red[2 * BA_WARPS + 4];
  extern __shared__ double minv_all[];  // per warp: M^-1 [36][32] doubles, entry cache [SLOTS][32] int2, row records [ROWS] int2
  const int tid = threadIdx.x, lane = tid & 31;
  const int gw = (blockIdx.x * BA_THREADS + tid) >> 5, nw = (gridDim.x * BA_THREADS) >> 5;
  const int n_wb = (n_cam + 31) / 32;
  // the warp's first camera block: M^-1 into shared memory, b into registers
  char *wsm = reinterpret_cast<char *>(minv_all) + (size_t)(tid >> 5) * BA_PCG_SMEM_PER_WARP;
  double *minv_s = reinterpret_cast<double *>(wsm);
  int2 *ecache = reinterpret_cast<int2 *>(wsm + 36 * 32 * 8);
  int4 *rowinfo = reinterpret_cast<int4 *>(ecache + BA_PCG_ENT_SLOTS * 32);
  // the warp's first rows: entries into the shared-memory cache
  int n_cached = 0;
  {
    int slot = 0;
    for (int idx = gw; idx < n_cam && n_cached < BA_PCG_ROWS; idx += nw) {
      const int row = row_order[idx];
      const int b0 = ent_ptr[row], e0 = ent_ptr[row + 1];
      const int trips = (e0 - b0 + 31) >> 5;
      if (slot + trips > BA_PCG_ENT_SLOTS) break;
      if (lane == 0) rowinfo[n_cached] = make_int4(b0, e0, row, 0);
      for (int e = b0; e < e0; e += 32, ++slot) ecache[slot * 32 + lane] = e + lane < e0 ? ent[e + lane] : make_int2(0, 0);
      ++n_cached;
    }
  }
  double breg[6] = {0, 0, 0, 0, 0, 0};
  if (gw < n_wb) {
    const int c = gw * 32 + lane;
    if (c < n_cam) {
#pragma unroll
      for (int k = 0; k < 36; ++k) minv_s[k * 32 + lane] = Minv[36 * (size_t)c + k];
      load6(b + 6 * (size_t)c, breg);
    }
  }
  __syncwarp();
  int it = st->pcg_it;
  double rho = st->pcg_rho, beta = st->pcg_beta, Q0 = st->pcg_Q0;
  int fail = 0, brk = 0, iters_last = 0;
  unsigned int epoch = 0;
  double *pold = pbuf0, *pnew = pbuf1;
  unsigned long long t0 = 0, tacc[6] = {0, 0, 0, 0, 0, 0};
#define PROF_TICK(slot)                                             \
  if (prof && blockIdx.x == 0 && tid == 0) {                        \
    unsigned long long t1_;                                         \
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t1_));          \
    tacc[slot] += t1_ - t0;                                         \
    t0 = t1_;                                                       \
  }
  if (prof && blockIdx.x == 0 && tid == 0) asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t0));

  for (;;) {
    // ---- phase I: p = z (+ beta p_old), q = S p + D^2 p, per-row p.q
    bsr_rows_cached<0>(n_cam, gw, nw, lane, n_cached, rowinfo, ecache, S, dsq, z, pold, beta, it > 1, pnew, q, row_pq);
    bsr_rows<0>(n_cam, gw + n_cached * nw, nw, lane, row_order, ent_ptr, ent, S, dsq, z, pold, beta, it > 1, pnew, q, row_pq);
    PROF_TICK(0)
    grid_barrier(bar, epoch);
    PROF_TICK(1)

    // ---- phase II: alpha; x += alpha p; r -= alpha q; z = M^-1 r; warp-block partials
    const double pq = block_sum_wide_cg(row_pq, n_cam, red);
    if (pq <= 0.0 || isinf(pq) || isnan(pq)) {  // NO_CONVERGENCE: keep x, stop
      iters_last = it;
      brk = 1;
      break;
    }
    const double alpha = rho / pq;
    if (isinf(alpha)) {
      iters_last = it;
      fail = 1;
      break;
    }
    const bool reset = lo.reset_period > 0 && (it % lo.reset_period) == 0;
    PROF_TICK(2)
    if (gw < n_wb) pcg_update_warp<0, 1>(n_cam, gw, lane, alpha, reset, b, Minv, minv_s, breg, x, r, z, pnew, q, part_rho, part_Q);
    for (int wb = gw + nw; wb < n_wb; wb += nw)
      pcg_update_warp<0, 0>(n_cam, wb, lane, alpha, reset, b, Minv, minv_s, breg, x, r, z, pnew, q, part_rho, part_Q);
    PROF_TICK(3)
    grid_barrier(bar, epoch);
    PROF_TICK(4)
    if (reset) {
      // ---- residual reset: q = S x + D^2 x, then r = b - q, z = M^-1 r
      bsr_rows_cached<1>(n_cam, gw, nw, lane, n_cached, rowinfo, ecache, S, dsq, x, x, 0.0, false, nullptr, q, nullptr);
      bsr_rows<1>(n_cam, gw + n_cached * nw, nw, lane, row_order, ent_ptr, ent, S, dsq, x, x, 0.0, false, nullptr, q, nullptr);
      grid_barrier(bar, epoch);
      if (gw < n_wb) pcg_update_warp<1, 1>(n_cam, gw, lane, 0.0, false, b, Minv, minv_s, breg, x, r, z, pnew, q, part_rho, part_Q);
      for (int wb = gw + nw; wb < n_wb; wb += nw)
        pcg_update_warp<1, 0>(n_cam, wb, lane, 0.0, false, b, Minv, minv_s, breg, x, r, z, pnew, q, part_rho, part_Q);
      grid_barrier(bar, epoch);
    }

    // ---- controller (every CTA, identical inputs, identical order)
    double rho_new, xq;
    block_sum2_cg(part_rho, part_Q, n_wb, red, rho_new, xq);
    iters_last = it;
    const double Q1 = -1.0 * xq;
    const double zeta = it * (Q1 - Q0) / Q1;
    if (zeta < lo.eta && it >= lo.min_pcg) break;
    Q0 = Q1;
    if (it >= lo.max_pcg) break;
    const double beta_new = rho_new / rho;
    if (rho_new == 0.0 || !isfinite(rho_new) || beta_new == 0.0 || !isfinite(beta_new)) {
      iters_last = it + 1;
      fail = 1;
      break;
    }
    rho = rho_new;
    beta = beta_new;
    ++it;
    double *t = pold;
    pold = pnew;
    pnew = t;
    PROF_TICK(5)
  }
  if (prof && blockIdx.x == 0 && tid == 0)
    for (int k = 0; k < 6; ++k) prof[k] += tacc[k];
  if (blockIdx.x == 0 && tid == 0) {
    st->pcg_it = it;
    st->pcg_rho = rho;
    st->pcg_beta = beta;
    st->pcg_Q0 = Q0;
    st->pcg_iters_last = iters_last;
    st->pcg_break = brk;
    if (fail) st->lin_fail = 1;
    st->pcg_done = 1;
  }
}
