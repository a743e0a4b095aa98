// ba_sparse_symbolic.h -- SYMBOLIC phase of the exact sparse Cholesky of the reduced camera system
// (BA_SOLVER_SPARSE_SCHUR_CHOLESKY).  Plain host C++ (no CUDA): integer structure only, run once per upload.
//
// What it replaces: the reference asks Ceres for linear_solver_type = SPARSE_SCHUR
// (headers/BundleAdjustmentConfig.h:62, used by ceres::Solve at src/OptimizationUtils.cpp:300): the reduced camera
// matrix S (6x6 blocks, one per pair of cameras that share a landmark) is factorised by a sparse Cholesky.  Ceres hands
// that to CHOLMOD / Eigen (ordering + supernodal or simplicial factorisation on one CPU thread).  Here the structure work
// is done on the host at BLOCK (camera) granularity and the numeric work by the kernels of ba_kernels_spchol.cuh:
//
//   1. ordering: nested dissection of the camera sequence.  Landmark tracks of a SLAM front end are runs of neighbouring
//      keyframes (src/Map3D.cpp:7-74), so S is block-banded along the trajectory; a range [lo, hi) is cut at a camera c
//      near its middle where the band is narrowest; the separator is the run of cameras [c, r] that the left part
//      reaches, the two remaining parts are ordered recursively, separators are eliminated last.  A sequential banded
//      elimination is a chain of n_cam dependent steps; this ordering turns it into a tree of depth O(log n_cam)
//      whose nodes of one level are independent -- one thread block each.
//   2. symbolic factorisation (elimination tree + column structures of L) in that order;
//   3. supernodes: runs of consecutive columns along a tree path, sized so that a node's front panel
//      ((own + border) x own blocks of 6x6 doubles) fits in one SM's shared memory;
//   4. per node: border list, child -> parent index maps (extend-add), the stored blocks of S that land in its
//      front, its level (children before parents).
#pragma once
#include <stdint.h>

#include <algorithm>
#include <initializer_list>
#include <vector>

#define SPSYM_NODE_INTS 16
enum {
  SPN_K0 = 0,       // first own position (elimination order)
  SPN_M = 1,        // own cameras
  SPN_NB = 2,       // border cameras
  SPN_BORD = 3,     // offset of the border list (positions, ascending)
  SPN_PARENT = 4,   // parent node or -1
  SPN_LEVEL = 5,
  SPN_CHILD = 6,    // offset into the child list
  SPN_NCHILD = 7,
  SPN_AENT = 8,     // offset of the entries of S assembled into this front (4 ints each)
  SPN_NAENT = 9,
  SPN_REL = 10,     // as a child: nb ints, border index -> local index in the parent's (own, border) list
  SPN_INV = 11,     // as a child: parent's nb ints, parent's border index -> own border index or -1
  SPN_PANEL_LO = 12,  // panel offset in 6x6 blocks (low / high 31 bits)
  SPN_PANEL_HI = 13,
  SPN_U_LO = 14,      // update-matrix offset in 6x6 blocks
  SPN_U_HI = 15
};

#ifndef SPSYM_STAMP
#define SPSYM_STAMP(name)  // (profiling hook of the symbolic phase: a harness defines it before including this header)
#endif

struct SpSymbolic {
  int n_cam = 0, n_nodes = 0, n_levels = 0;
  std::vector<int32_t> perm, pos;  // position -> camera, camera -> position
  std::vector<int32_t> node;       // SPSYM_NODE_INTS per node, nodes in ascending first position
  std::vector<int32_t> bord, children, rel, inv, aent, level_ptr, level_nodes;
  int64_t panel_blocks = 0, u_blocks = 0;
  int max_front_blocks = 0, max_m = 0, max_nb = 0, max_children = 0;
  double flops = 0.0;       // multiply-adds x 2 of the numeric factorisation
  double crit_blocks = 0.0; // sum over levels of the largest node's block operations (the dependent chain)
  int error = 0;            // 1: a column's front does not fit the capacity, 2: internal inconsistency
};

namespace spsym {

struct Graph {
  int n;
  std::vector<int32_t> up_ptr, up;  // upper neighbours (j > i) of every camera, ascending
};

inline Graph build_graph(int n_cam, int n_blk, const int32_t *bi, const int32_t *bj) {
  Graph g;
  g.n = n_cam;
  g.up_ptr.assign((size_t)n_cam + 1, 0);
  for (int b = 0; b < n_blk; ++b)
    if (bi[b] < bj[b]) g.up_ptr[bi[b] + 1]++;
  for (int i = 0; i < n_cam; ++i) g.up_ptr[i + 1] += g.up_ptr[i];
  g.up.resize((size_t)g.up_ptr[n_cam]);
  std::vector<int32_t> cur(g.up_ptr.begin(), g.up_ptr.end() - 1);
  for (int b = 0; b < n_blk; ++b)
    if (bi[b] < bj[b]) g.up[cur[bi[b]]++] = bj[b];
  // (the device hands the blocks over sorted by (row, column): the rows are then ascending already)
  for (int i = 0; i < n_cam; ++i) {
    int32_t *rb = g.up.data() + g.up_ptr[i], *re = g.up.data() + g.up_ptr[i + 1];
    if (!std::is_sorted(rb, re)) std::sort(rb, re);
  }
  return g;
}

// largest neighbour of camera i that is < hi (i itself if none)
inline int reach_below(const Graph &g, int i, int hi) {
  const int32_t *b = g.up.data() + g.up_ptr[i], *e = g.up.data() + g.up_ptr[i + 1];
  const int32_t *it = std::lower_bound(b, e, hi);
  return it == b ? i : *(it - 1);
}

// nested dissection of the camera range [lo, hi): appends the elimination order to `order`
inline void nd_order(const Graph &g, int lo, int hi, int leaf, std::vector<int32_t> &order, std::vector<int32_t> &pm) {
  const int len = hi - lo;
  if (len <= 0) return;
  if (len > leaf) {
    // pm[c - lo] = furthest camera (< hi) coupled to [lo, c)
    pm[0] = lo - 1;
    int run = lo - 1;
    for (int c = lo + 1; c <= hi; ++c) {
      run = std::max(run, reach_below(g, c - 1, hi));
      pm[c - lo] = run;
    }
    const int mid = lo + len / 2, delta = std::max(1, len / 8);
    int best_c = -1, best_w = 1 << 30;
    for (int c = std::max(lo + 1, mid - delta); c <= std::min(hi - 1, mid + delta); ++c) {
      const int r = pm[c - lo];
      const int w = r >= c ? r - c + 1 : 0;
      if (r + 1 >= hi && w > 0) continue;  // nothing left on the right
      if (w < best_w || (w == best_w && std::abs(c - mid) < std::abs(best_c - mid))) {
        best_w = w;
        best_c = c;
      }
    }
    if (best_c >= 0 && 2 * best_w < len) {
      const int c = best_c, r = best_w > 0 ? pm[c - lo] : c - 1;
      nd_order(g, lo, c, leaf, order, pm);
      nd_order(g, r + 1, hi, leaf, order, pm);
      for (int k = c; k <= r; ++k) order.push_back(k);
      return;
    }
  }
  for (int k = lo; k < hi; ++k) order.push_back(k);
}

}  // namespace spsym

// n_cam cameras; n_blk stored upper blocks (bi <= bj) of S, any order; leaf = cameras per dissection leaf;
// cap_blocks = 6x6 blocks of shared memory one front may take: (own + border) x (own + 1); max_own = cameras per supernode at most
inline SpSymbolic spsym_build(int n_cam, int n_blk, const int32_t *bi, const int32_t *bj, int leaf, int cap_blocks, int max_own) {
  SpSymbolic S;
  S.n_cam = n_cam;
  const int n = n_cam;
  if (n <= 0) return S;
  const spsym::Graph g = spsym::build_graph(n, n_blk, bi, bj);
  SPSYM_STAMP("graph");
  // ---- 1. ordering
  {
    std::vector<int32_t> pm((size_t)n + 2);
    S.perm.reserve(n);
    spsym::nd_order(g, 0, n, std::max(2, leaf), S.perm, pm);
    if ((int)S.perm.size() != n) {
      S.error = 2;
      return S;
    }
    S.pos.assign(n, -1);
    for (int k = 0; k < n; ++k) S.pos[S.perm[k]] = k;
  }
  SPSYM_STAMP("ordering");
  // ---- 2. symbolic factorisation in elimination order
  // adjacency in elimination positions, CSR: adj_ptr[k] .. adj_ptr[k + 1] = later-eliminated neighbours of position k
  // column structures live in one arena (st_off / st_len); a column's structure is the sorted union of its adjacency and its
  // children's structures without the column itself -- sorted merges (a child's first entry IS its parent), no per-column vectors
  std::vector<int32_t> adj_ptr((size_t)n + 1, 0), adj((size_t)g.up.size());
  for (int i = 0; i < n; ++i)
    for (int e = g.up_ptr[i]; e < g.up_ptr[i + 1]; ++e) adj_ptr[std::min(S.pos[i], S.pos[g.up[e]]) + 1]++;
  for (int k = 0; k < n; ++k) adj_ptr[k + 1] += adj_ptr[k];
  {
    std::vector<int32_t> cur(adj_ptr.begin(), adj_ptr.end() - 1);
    for (int i = 0; i < n; ++i)
      for (int e = g.up_ptr[i]; e < g.up_ptr[i + 1]; ++e) {
        const int a = S.pos[i], b = S.pos[g.up[e]];
        adj[cur[std::min(a, b)]++] = std::max(a, b);
      }
  }
  std::vector<int32_t> parent(n, -1), nchild(n, 0), child_head(n, -1), child_next(n, -1), st_len(n, 0);
  std::vector<int64_t> st_off(n, 0);
  std::vector<int32_t> arena, ta, tb;
  arena.reserve((size_t)n * 48 + 64);
  for (int k = 0; k < n; ++k) {
    ta.assign(adj.begin() + adj_ptr[k], adj.begin() + adj_ptr[k + 1]);
    std::sort(ta.begin(), ta.end());
    for (int c = child_head[k]; c >= 0; c = child_next[c]) {
      const int32_t *cb = arena.data() + st_off[c] + 1, *ce = arena.data() + st_off[c] + st_len[c];  // (skips k itself)
      tb.resize(ta.size() + (size_t)(ce - cb));
      tb.resize((size_t)(std::set_union(ta.begin(), ta.end(), cb, ce, tb.begin()) - tb.begin()));
      ta.swap(tb);
    }
    st_off[k] = (int64_t)arena.size();
    st_len[k] = (int32_t)ta.size();
    arena.insert(arena.end(), ta.begin(), ta.end());
    if (!ta.empty()) {
      parent[k] = ta[0];
      nchild[ta[0]]++;
      child_next[k] = child_head[ta[0]];
      child_head[ta[0]] = k;
    }
  }
  SPSYM_STAMP("column structures");
  // ---- 3. supernodes
  // shared memory of a front: the panel (m + nb) x m blocks plus one more block column (the pivot column kept row-major)
  auto fits = [&](int m, int nb) { return (long long)(m + nb) * (m + 1) <= (long long)cap_blocks && m <= max_own; };
  std::vector<int32_t> node_of(n, -1);
  std::vector<int32_t> k0s, ms;
  for (int k = 0; k < n;) {
    const int start = k;
    int m = 1;
    if (!fits(1, st_len[k])) {
      S.error = 1;
      return S;
    }
    while (k + 1 < n && parent[k] == k + 1 && nchild[k + 1] == 1 && fits(m + 1, st_len[k + 1])) {
      ++k;
      ++m;
    }
    const int id = (int)k0s.size();
    for (int q = start; q <= k; ++q) node_of[q] = id;
    k0s.push_back(start);
    ms.push_back(m);
    ++k;
  }
  const int nn = (int)k0s.size();
  S.n_nodes = nn;
  S.node.assign((size_t)nn * SPSYM_NODE_INTS, 0);
  std::vector<int32_t> level(nn, 0);
  std::vector<std::vector<int32_t>> kids(nn);
  for (int id = 0; id < nn; ++id) {
    int32_t *N = S.node.data() + (size_t)id * SPSYM_NODE_INTS;
    const int k1 = k0s[id] + ms[id] - 1;
    const std::vector<int32_t> b(arena.begin() + st_off[k1], arena.begin() + st_off[k1] + st_len[k1]);
    N[SPN_K0] = k0s[id];
    N[SPN_M] = ms[id];
    N[SPN_NB] = (int)b.size();
    N[SPN_BORD] = (int)S.bord.size();
    S.bord.insert(S.bord.end(), b.begin(), b.end());
    N[SPN_PARENT] = b.empty() ? -1 : node_of[b[0]];
    if (N[SPN_PARENT] >= 0) {
      if (N[SPN_PARENT] <= id) {
        S.error = 2;
        return S;
      }
      kids[N[SPN_PARENT]].push_back(id);
    }
    N[SPN_PANEL_LO] = (int32_t)(S.panel_blocks & 0x7fffffff);
    N[SPN_PANEL_HI] = (int32_t)(S.panel_blocks >> 31);
    N[SPN_U_LO] = (int32_t)(S.u_blocks & 0x7fffffff);
    N[SPN_U_HI] = (int32_t)(S.u_blocks >> 31);
    S.panel_blocks += (int64_t)(ms[id] + (int)b.size()) * ms[id];
    S.u_blocks += (int64_t)b.size() * (int64_t)b.size();
    S.max_front_blocks = std::max(S.max_front_blocks, (ms[id] + (int)b.size()) * (ms[id] + 1));
    S.max_m = std::max(S.max_m, ms[id]);
    S.max_nb = std::max(S.max_nb, (int)b.size());
  }
  SPSYM_STAMP("supernodes");
  // levels: children have smaller ids than parents
  for (int id = 0; id < nn; ++id) {
    const int p = S.node[(size_t)id * SPSYM_NODE_INTS + SPN_PARENT];
    if (p >= 0) level[p] = std::max(level[p], level[id] + 1);
  }
  int nlev = 0;
  for (int id = 0; id < nn; ++id) nlev = std::max(nlev, level[id] + 1);
  S.n_levels = nlev;
  S.level_ptr.assign((size_t)nlev + 1, 0);
  for (int id = 0; id < nn; ++id) S.level_ptr[level[id] + 1]++;
  for (int l = 0; l < nlev; ++l) S.level_ptr[l + 1] += S.level_ptr[l];
  S.level_nodes.resize(nn);
  {
    std::vector<int32_t> cur(S.level_ptr.begin(), S.level_ptr.end() - 1);
    for (int id = 0; id < nn; ++id) S.level_nodes[cur[level[id]]++] = id;
  }
  SPSYM_STAMP("levels");
  // ---- 4. children, extend-add maps
  for (int id = 0; id < nn; ++id) {
    int32_t *N = S.node.data() + (size_t)id * SPSYM_NODE_INTS;
    N[SPN_LEVEL] = level[id];
    N[SPN_CHILD] = (int)S.children.size();
    N[SPN_NCHILD] = (int)kids[id].size();
    S.max_children = std::max(S.max_children, (int)kids[id].size());
    S.children.insert(S.children.end(), kids[id].begin(), kids[id].end());
  }
  for (int id = 0; id < nn; ++id) {
    int32_t *N = S.node.data() + (size_t)id * SPSYM_NODE_INTS;
    const int p = N[SPN_PARENT];
    N[SPN_REL] = (int)S.rel.size();
    N[SPN_INV] = (int)S.inv.size();
    if (p < 0) continue;
    const int32_t *Pn = S.node.data() + (size_t)p * SPSYM_NODE_INTS;
    const int pk0 = Pn[SPN_K0], pm_ = Pn[SPN_M], pnb = Pn[SPN_NB];
    const int32_t *pb = S.bord.data() + Pn[SPN_BORD];
    const int32_t *cb = S.bord.data() + N[SPN_BORD];
    const int nb = N[SPN_NB];
    for (int i = 0; i < nb; ++i) {
      const int q = cb[i];
      if (q < pk0) {
        S.error = 2;
        return S;
      }
      if (q < pk0 + pm_) {
        S.rel.push_back(q - pk0);
      } else {
        const int32_t *it = std::lower_bound(pb, pb + pnb, q);
        if (it == pb + pnb || *it != q) {
          S.error = 2;
          return S;
        }
        S.rel.push_back(pm_ + (int)(it - pb));
      }
    }
    for (int i = 0; i < pnb; ++i) {
      const int32_t *it = std::lower_bound(cb, cb + nb, pb[i]);
      S.inv.push_back((it != cb + nb && *it == pb[i]) ? (int)(it - cb) : -1);
    }
  }
  SPSYM_STAMP("children, extend-add maps");
  // ---- 5. entries of S per front: (block | flags, local row, local column, camera of the column)
  //         flags: bit 31 = use the stored block transposed, bit 30 = diagonal block; block 0x3fffffff = no stored block
  {
    // pass 1 over the blocks: owning node, local row / column, flags (the searches) and the per-node counts; pass 2 only
    // places the finished records into the flat table, in block order within a node
    std::vector<char> has_diag(n, 0);
    std::vector<int32_t> cnt((size_t)nn + 1, 0), t_id((size_t)n_blk), t_rec((size_t)n_blk * 4);
    auto search = [&](int b0, int b1, int32_t *counts, int *err) {
      for (int b = b0; b < b1; ++b) {
        const int i = bi[b], j = bj[b];
        const int pi = S.pos[i], pj = S.pos[j];
        const int c = std::min(pi, pj), r = std::max(pi, pj);
        const int id = node_of[c];
        const int32_t *N = S.node.data() + (size_t)id * SPSYM_NODE_INTS;
        const int k0 = N[SPN_K0], m = N[SPN_M], nb = N[SPN_NB];
        int lr;
        if (r < k0 + m) {
          lr = r - k0;
        } else {
          const int32_t *bb = S.bord.data() + N[SPN_BORD];
          const int32_t *it = std::lower_bound(bb, bb + nb, r);
          if (it == bb + nb || *it != r) {
            *err = 2;
            return;
          }
          lr = m + (int)(it - bb);
        }
        uint32_t code = (uint32_t)b;
        if (i == j) {
          code |= 0x40000000u;
          has_diag[i] = 1;
        } else if (S.perm[r] == j) {
          code |= 0x80000000u;  // F(r, c) = A(cam r, cam c) = S(i, j)^T when cam r is the stored block's column camera
        }
        t_id[b] = id;
        int32_t *e = t_rec.data() + 4 * (size_t)b;
        e[0] = (int32_t)code;
        e[1] = lr;
        e[2] = c - k0;
        e[3] = S.perm[c];
        counts[id + 1]++;
      }
    };
    {
      // (threading this pass over block ranges was tried: 3.4 -> 2.9 ms on 4 threads of an 8-core host -- not worth the threads)
      int err = 0;
      search(0, n_blk, cnt.data(), &err);
      if (err) {
        S.error = err;
        return S;
      }
    }
    SPSYM_STAMP("entries: search pass");
    for (int cam = 0; cam < n; ++cam)
      if (!has_diag[cam]) cnt[node_of[S.pos[cam]] + 1]++;
    for (int id = 0; id < nn; ++id) cnt[id + 1] += cnt[id];
    S.aent.assign((size_t)cnt[nn] * 4, 0);
    for (int id = 0; id < nn; ++id) {
      int32_t *N = S.node.data() + (size_t)id * SPSYM_NODE_INTS;
      N[SPN_AENT] = cnt[id];
      N[SPN_NAENT] = cnt[id + 1] - cnt[id];
    }
    std::vector<int32_t> cur(cnt.begin(), cnt.end() - 1);
    for (int b = 0; b < n_blk; ++b) {
      int32_t *e = S.aent.data() + 4 * (size_t)cur[t_id[b]]++;
      const int32_t *t = t_rec.data() + 4 * (size_t)b;
      e[0] = t[0];
      e[1] = t[1];
      e[2] = t[2];
      e[3] = t[3];
    }
    for (int cam = 0; cam < n; ++cam)
      if (!has_diag[cam]) {  // damping only (fixed camera, camera without observations)
        const int c = S.pos[cam], id = node_of[c];
        const int k0 = S.node[(size_t)id * SPSYM_NODE_INTS + SPN_K0];
        int32_t *e = S.aent.data() + 4 * (size_t)cur[id]++;
        e[0] = (int32_t)(0x3fffffffu | 0x40000000u);
        e[1] = c - k0;
        e[2] = c - k0;
        e[3] = cam;
      }
  }
  SPSYM_STAMP("entries");
  // ---- cost model (block operations of 216 multiply-adds)
  {
    std::vector<double> lev_max(nlev, 0.0);
    for (int id = 0; id < nn; ++id) {
      const int32_t *N = S.node.data() + (size_t)id * SPSYM_NODE_INTS;
      const double m = N[SPN_M], nb = N[SPN_NB];
      double ops = 0.0;
      for (int k = 0; k < (int)m; ++k) {
        const double below = m - k - 1 + nb;
        ops += below + (m - k - 1) * (nb + (m - k) * 0.5);
      }
      ops += m * nb * (nb + 1) * 0.5;
      S.flops += ops * 432.0;
      lev_max[level[id]] = std::max(lev_max[level[id]], ops);
    }
    for (int l = 0; l < nlev; ++l) S.crit_blocks += lev_max[l];
  }
  return S;
}

// ---------------------------------------------------------------------------------------------
// Subtree-to-rank partition of the supernodal tree (multi-GPU factorisation): a CUT through the tree leaves disjoint
// subtrees below it, each factorised by one rank, and a small TOP part above it that every rank factorises redundantly
// from the update matrices of the subtree roots (exchanged once per solve).  The cut starts at the roots and the heaviest
// subtree is opened (its root moves to the top, its children enter the cut) until the subtrees, taken in the order of the
// camera sequence, split into `parts` consecutive groups of about equal work.  Consecutive, because the ranks' point
// shards are consecutive too (landmarks are numbered along the trajectory): a rank then forms most of the blocks of S it
// factorises itself, and only the blocks near the shard borders and those of the top part have to be summed over ranks.
// ---------------------------------------------------------------------------------------------
struct SpPartition {
  int parts = 1;
  std::vector<int32_t> part;  // per node: owning part, -1 = top (replicated)
  std::vector<int32_t> cut;   // roots of the subtrees below the cut, in sequence order
  double total = 0.0, top = 0.0, heaviest = 0.0;  // work in block operations: all, top part, the most loaded part
};

inline double spsym_node_ops(const int32_t *N) {
  const double m = N[SPN_M], nb = N[SPN_NB];
  double ops = 0.0;
  for (int k = 0; k < (int)m; ++k) {
    const double below = m - k - 1 + nb;
    ops += below + (m - k - 1) * (nb + (m - k) * 0.5);
  }
  return ops + m * nb * (nb + 1) * 0.5 + 4.0;
}

inline SpPartition spsym_partition(const SpSymbolic &S, int parts) {
  SpPartition R;
  const int nn = S.n_nodes;
  R.part.assign((size_t)nn, 0);
  if (parts <= 1 || nn == 0) return R;
  auto node = [&](int id) { return S.node.data() + (size_t)id * SPSYM_NODE_INTS; };
  // subtree work and first position (children have smaller ids than parents)
  std::vector<double> sub((size_t)nn);
  std::vector<int32_t> first((size_t)nn);
  for (int id = 0; id < nn; ++id) {
    sub[id] = spsym_node_ops(node(id));
    first[id] = node(id)[SPN_K0];
    R.total += sub[id];
  }
  for (int id = 0; id < nn; ++id) {
    const int p = node(id)[SPN_PARENT];
    if (p >= 0) {
      sub[p] += sub[id];
      first[p] = std::min(first[p], first[id]);
    }
  }
  std::vector<int32_t> cut;
  std::vector<char> top((size_t)nn, 0);
  for (int id = 0; id < nn; ++id)
    if (node(id)[SPN_PARENT] < 0) cut.push_back(id);
  // consecutive groups of the cut (sorted along the camera sequence) with about equal work; returns the largest group
  std::vector<int32_t> group;
  auto split = [&]() -> double {
    std::sort(cut.begin(), cut.end(), [&](int a, int b) { return S.perm[first[a]] < S.perm[first[b]]; });
    double below = 0.0;
    for (int id : cut) below += sub[id];
    group.assign(cut.size(), 0);
    double acc = 0.0, worst = 0.0, cur = 0.0;
    int g = 0;
    for (size_t i = 0; i < cut.size(); ++i) {
      // close the group when the middle of this subtree lies beyond the group's share (and enough subtrees remain)
      const double mid = acc + 0.5 * sub[cut[i]];
      while (g + 1 < parts && mid > below * (g + 1) / parts && cur > 0.0) {
        worst = std::max(worst, cur);
        cur = 0.0;
        ++g;
      }
      group[i] = g;
      cur += sub[cut[i]];
      acc += sub[cut[i]];
    }
    return std::max(worst, cur);
  };
  double top_w = 0.0, heaviest = 0.0;
  for (int iter = 0; iter < 2 * nn; ++iter) {
    heaviest = split();
    double below = R.total - top_w;
    if ((int)cut.size() >= parts && heaviest <= 1.30 * below / parts) break;
    if ((int)cut.size() >= 6 * parts || top_w > 0.3 * R.total) break;  // accept the imbalance rather than a large top part
    int h = -1;
    for (int id : cut)
      if (node(id)[SPN_NCHILD] > 0 && (h < 0 || sub[id] > sub[h])) h = id;
    if (h < 0) break;
    top[h] = 1;
    top_w += spsym_node_ops(node(h));
    cut.erase(std::find(cut.begin(), cut.end(), h));
    const int32_t *ch = S.children.data() + node(h)[SPN_CHILD];
    for (int c = 0; c < node(h)[SPN_NCHILD]; ++c) cut.push_back(ch[c]);
  }
  heaviest = split();
  if ((int)cut.size() < parts) return R;  // (tree too small: one part, replicated)
  R.parts = parts;
  R.cut = cut;
  R.top = top_w;
  R.heaviest = heaviest;
  // parents before children (descending ids): a node inherits its parent's part
  std::vector<int32_t> grp_of((size_t)nn, -2);
  for (size_t i = 0; i < cut.size(); ++i) grp_of[cut[i]] = group[i];
  for (int id = nn - 1; id >= 0; --id) {
    if (top[id]) {
      R.part[id] = -1;
    } else if (grp_of[id] >= 0) {
      R.part[id] = grp_of[id];
    } else {
      R.part[id] = R.part[node(id)[SPN_PARENT]];
    }
  }
  return R;
}

// ---------------------------------------------------------------------------------------------
// Work queues of the persistent tree kernels (k_spchol_tree, k_selinv_tree): items (node, kind), kind >= 0 a tile of the
// node, SPQ_HEAD its factor / prepare item, SPQ_SOLVE, SPQ_FINISH.  The kernels wait on completion counters and cannot
// deadlock only because every item an item waits for is earlier in the same launch or was done by an earlier launch over the
// same counters (tests/test_tree_queue_order.py restates the waits and checks this).
// ---------------------------------------------------------------------------------------------
enum { SPQ_HEAD = -1, SPQ_SOLVE = -2, SPQ_FINISH = -3 };

struct SpQueue {
  std::vector<int32_t> q;      // (node, kind) per item
  std::vector<int32_t> tiles;  // tiles per node (0: no border, or no head item in this queue)
  int n_items() const { return (int)(q.size() / 2); }
};

// tiles of the nodes of a level with `nodes` nodes: more where the level has fewer nodes than the GPU has SMs
inline int spq_level_tiles(int n_sm, int nodes) { return std::max(1, std::min(8, n_sm / std::max(1, nodes))); }

// Appends the levels of the tree, bottom-up or top-down, restricted to the nodes `keep` accepts (levels without such nodes
// are skipped).  Per level one pass over its nodes per entry of `kinds`: SPQ_HEAD items (they fix the node's tiles), 0 for
// the tiles 0 .. tiles - 1 of every node, SPQ_SOLVE or SPQ_FINISH items.
template <class Keep>
inline void spq_push_levels(const SpSymbolic &S, int n_sm, bool top_down, Keep keep, std::initializer_list<int> kinds, SpQueue &Q) {
  for (int k = 0; k < S.n_levels; ++k) {
    const int l = top_down ? S.n_levels - 1 - k : k;
    const int32_t *b = S.level_nodes.data() + S.level_ptr[l], *e = S.level_nodes.data() + S.level_ptr[l + 1];
    const int nodes = (int)std::count_if(b, e, keep);
    if (!nodes) continue;
    const int t_lvl = spq_level_tiles(n_sm, nodes);
    for (const int kind : kinds)
      for (const int32_t *p = b; p < e; ++p) {
        const int id = *p;
        if (!keep(id)) continue;
        if (kind == SPQ_HEAD) Q.tiles[id] = S.node[(size_t)id * SPSYM_NODE_INTS + SPN_NB] > 0 ? t_lvl : 0;
        for (int t = 0; t < (kind == 0 ? Q.tiles[id] : 1); ++t) {
          Q.q.push_back(id);
          Q.q.push_back(kind == 0 ? t : kind);
        }
      }
  }
}

// Queue of k_spchol_tree for the items rank `me` runs (me < 0: one GPU runs every part).  Phase A, one launch per part p, is
// [qA[p], qA[p + 1]): the part's factor levels bottom-up, per level the factor items, then their update tiles.  Phase B,
// [qB, qB + qB_n): the same for the top part, then the backward substitution levels top-down (top part first, then the
// subtrees this GPU holds).  One part: phase A is the whole factorisation, phase B the backward substitution.
struct SpCholQueue : SpQueue {
  std::vector<int32_t> qA;        // parts + 1
  int qB = 0, qB_n = 0;
  std::vector<int32_t> cnt_init;  // completion counters before a solve: 16 tickets, then fdone, udone, sdone per node
  std::vector<int32_t> topcams;   // cameras of the top part
};
inline SpCholQueue spq_cholesky(const SpSymbolic &S, const SpPartition &part, int me, int n_sm) {
  SpCholQueue Q;
  const int nn = S.n_nodes;
  Q.tiles.assign((size_t)nn, 0);
  for (int p = 0; p < part.parts; ++p) {
    Q.qA.push_back(Q.n_items());
    if (me < 0 || p == me) spq_push_levels(S, n_sm, false, [&](int id) { return part.part[id] == p; }, {SPQ_HEAD, 0}, Q);
  }
  Q.qB = Q.n_items();
  Q.qA.push_back(Q.qB);
  if (part.parts > 1) {
    spq_push_levels(S, n_sm, false, [&](int id) { return part.part[id] < 0; }, {SPQ_HEAD, 0}, Q);
    spq_push_levels(S, n_sm, true, [&](int id) { return part.part[id] < 0; }, {SPQ_SOLVE}, Q);
  }
  spq_push_levels(S, n_sm, true, [&](int id) { return part.part[id] >= 0 && (me < 0 || part.part[id] == me); }, {SPQ_SOLVE}, Q);
  Q.qB_n = Q.n_items() - Q.qB;
  // zero, except "all update tiles done" for the subtree roots other ranks factorise (their update matrices arrive with the
  // exchange)
  Q.cnt_init.assign((size_t)3 * nn + 16, 0);
  for (int id = 0; id < nn; ++id) {
    const int32_t *N = S.node.data() + (size_t)id * SPSYM_NODE_INTS;
    if (part.part[id] < 0)
      for (int k = 0; k < N[SPN_M]; ++k) Q.topcams.push_back(S.perm[N[SPN_K0] + k]);
    else if (me >= 0 && part.part[id] != me)
      Q.cnt_init[16 + (size_t)nn + id] = 1 << 20;
  }
  return Q;
}

// Queue of k_selinv_tree: the levels top-down, per level the prepare items, the product tiles, the finish items
inline SpQueue spq_selinv(const SpSymbolic &S, int n_sm) {
  SpQueue Q;
  Q.tiles.assign((size_t)S.n_nodes, 0);
  spq_push_levels(S, n_sm, true, [](int) { return true; }, {SPQ_HEAD, 0, SPQ_FINISH}, Q);
  return Q;
}
