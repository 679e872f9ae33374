// Host-only symbolic phase of the mu-batched reduced solve (no CUDA calls in this file).
//
// The reduced LRBMS operator is block sparse: one N_i x N_j block per subdomain pair that shares a face
// (reference discretize_elliptic_block_swipdg.py:475-507).  The reference unblocks it into one dense matrix and
// calls numpy.linalg.solve (SURVEY.md 8a a10/a12).  Here the scalar index space is cut into 8x8 tiles -- the
// accumulator shape of DMMA.8x8x4 -- irrespective of subdomain boundaries, a symbolic Cholesky is run on the
// tile graph, and the numeric kernel gets a left-looking schedule: for every tile (I, J) of L the list of
// (L_IK, L_JK) pairs, K < J, whose product it has to subtract.  Ragged N_i need no padding except at the very
// end of the matrix.
#include "symbolic.h"

#include <algorithm>
#include <set>
#include <string>

#include "../../include/lrbms_sm100.h"

int lrbms_symbolic_basics(lrbms_symbolic& S, int32_t n_sub, const int32_t* sizes, int32_t n_blocks, const int32_t* bi,
                          const int32_t* bj, std::string* err) {
  auto fail = [&](const char* m) { if (err) *err = m; return (int)LRBMS_ERR_INVALID; };
  if (n_sub <= 0 || !sizes || n_blocks < 0 || (n_blocks && (!bi || !bj))) return fail("symbolic: bad arguments");
  S.n_sub = n_sub;
  S.sizes.assign(sizes, sizes + n_sub);
  S.offsets.assign(n_sub + 1, 0);
  for (int i = 0; i < n_sub; ++i) {
    if (sizes[i] < 0) return fail("symbolic: negative basis size");
    S.offsets[i + 1] = S.offsets[i] + sizes[i];
  }
  S.n_red = S.offsets[n_sub];
  if (S.n_red == 0) return fail("symbolic: empty reduced space");
  S.n_pad = (S.n_red + 7) & ~7;
  S.ntc = S.n_pad / 8;
  S.block_i.assign(bi, bi + n_blocks);
  S.block_j.assign(bj, bj + n_blocks);
  std::vector<char> has_diag(n_sub, 0);
  S.half_bandwidth = 0;
  for (int b = 0; b < n_blocks; ++b) {
    const int i = bi[b], j = bj[b];
    if (i < 0 || i >= n_sub || j < 0 || j >= n_sub) return fail("symbolic: block index out of range");
    if (i == j) has_diag[i] = 1;
    if (i >= j && sizes[i] > 0 && sizes[j] > 0) S.half_bandwidth = std::max(S.half_bandwidth, S.offsets[i + 1] - 1 - S.offsets[j]);
  }
  for (int i = 0; i < n_sub; ++i)
    if (sizes[i] > 0 && !has_diag[i]) return fail("symbolic: every subdomain needs its diagonal block");
  return 0;
}

int lrbms_symbolic_build(lrbms_symbolic& S, int32_t n_sub, const int32_t* sizes, int32_t n_blocks, const int32_t* bi,
                         const int32_t* bj, std::string* err) {
  auto fail = [&](const char* m) { if (err) *err = m; return (int)LRBMS_ERR_INVALID; };
  if (int rc = lrbms_symbolic_basics(S, n_sub, sizes, n_blocks, bi, bj, err)) return rc;

  // ---- tile pattern of the lower triangle of A
  std::vector<std::vector<int32_t>> cols(S.ntc);   // cols[J] = tile rows I >= J with A_IJ != 0
  for (int b = 0; b < n_blocks; ++b) {
    const int i = bi[b], j = bj[b];
    if (i < j) continue;   // symmetric operator: the upper blocks are transposes of the lower ones
    if (sizes[i] == 0 || sizes[j] == 0) continue;
    const int I0 = S.offsets[i] / 8, I1 = (S.offsets[i + 1] - 1) / 8;
    const int J0 = S.offsets[j] / 8, J1 = (S.offsets[j + 1] - 1) / 8;
    for (int J = J0; J <= J1; ++J)
      for (int I = std::max(I0, J); I <= I1; ++I) cols[J].push_back(I);
  }
  for (int J = 0; J < S.ntc; ++J) {
    cols[J].push_back(J);
    std::sort(cols[J].begin(), cols[J].end());
    cols[J].erase(std::unique(cols[J].begin(), cols[J].end()), cols[J].end());
  }
  std::vector<std::vector<int32_t>> a_cols = cols;

  // ---- symbolic Cholesky on the tile graph (elimination-tree merge)
  std::vector<std::vector<int32_t>> children(S.ntc);
  for (int J = 0; J < S.ntc; ++J) {
    std::vector<int32_t>& sj = cols[J];
    for (int K : children[J]) {
      // merge struct(K) \ {K} into struct(J)
      std::vector<int32_t> merged;
      const std::vector<int32_t>& sk = cols[K];
      merged.reserve(sj.size() + sk.size());
      std::set_union(sj.begin(), sj.end(), sk.begin() + 1, sk.end(), std::back_inserter(merged));
      sj.swap(merged);
    }
    // everything merged in is >= J by construction (parent = first off-diagonal row)
    if (sj.size() > 1) children[sj[1]].push_back(J);
  }
  S.col_ptr.assign(S.ntc + 1, 0);
  for (int J = 0; J < S.ntc; ++J) S.col_ptr[J + 1] = S.col_ptr[J] + (int32_t)cols[J].size();
  S.row_idx.clear();
  S.row_idx.reserve(S.col_ptr[S.ntc]);
  S.max_targets = 0;
  for (int J = 0; J < S.ntc; ++J) {
    S.row_idx.insert(S.row_idx.end(), cols[J].begin(), cols[J].end());
    S.max_targets = std::max<int32_t>(S.max_targets, (int32_t)cols[J].size() + 1);
  }
  const int64_t n_tiles = S.n_tiles();

  // ---- operator tiles
  S.a_map.assign(n_tiles, -1);
  S.n_a_tiles = 0;
  for (int J = 0; J < S.ntc; ++J) {
    size_t pa = 0;
    for (int32_t p = S.col_ptr[J]; p < S.col_ptr[J + 1]; ++p) {
      while (pa < a_cols[J].size() && a_cols[J][pa] < S.row_idx[p]) ++pa;
      if (pa < a_cols[J].size() && a_cols[J][pa] == S.row_idx[p]) S.a_map[p] = S.n_a_tiles++;
    }
  }

  // ---- left-looking update pairs.  Right-looking enumeration: column K contributes L_IK L_JK^T to every target
  //      (I, J) with J <= I both in struct(K) \ {K}; visiting K ascending yields each target's list sorted by K.
  const int64_t n_targets = n_tiles + S.ntc;
  std::vector<int64_t> count(n_targets, 0);
  // slot lookup inside a column: position by binary search
  auto slot_of = [&](int I, int J) -> int32_t {
    const int32_t* b = S.row_idx.data() + S.col_ptr[J];
    const int32_t* e = S.row_idx.data() + S.col_ptr[J + 1];
    const int32_t* it = std::lower_bound(b, e, I);
    return (int32_t)(it - S.row_idx.data());
  };
  int64_t total = 0;
  for (int K = 0; K < S.ntc; ++K) {
    const int32_t b = S.col_ptr[K] + 1, e = S.col_ptr[K + 1];
    for (int32_t pj = b; pj < e; ++pj) {
      const int J = S.row_idx[pj];
      for (int32_t pi = pj; pi < e; ++pi) { ++count[slot_of(S.row_idx[pi], J)]; ++total; }
      ++count[n_tiles + J]; ++total;     // forward-solve row: y_J -= y_K L_JK^T
    }
  }
  if (total > (int64_t)1 << 30) return fail("symbolic: reduced system too large for the CTA-per-parameter schedule");
  S.pair_ptr.assign(n_targets + 1, 0);
  for (int64_t tgt = 0; tgt < n_targets; ++tgt) S.pair_ptr[tgt + 1] = S.pair_ptr[tgt] + (int32_t)count[tgt];
  S.pair_a.assign(total, 0);
  S.pair_b.assign(total, 0);
  std::vector<int32_t> fill(S.pair_ptr.begin(), S.pair_ptr.end() - 1);
  for (int K = 0; K < S.ntc; ++K) {
    const int32_t b = S.col_ptr[K] + 1, e = S.col_ptr[K + 1];
    for (int32_t pj = b; pj < e; ++pj) {
      const int J = S.row_idx[pj];
      for (int32_t pi = pj; pi < e; ++pi) {
        const int32_t tgt = slot_of(S.row_idx[pi], J);
        S.pair_a[fill[tgt]] = pi;
        S.pair_b[fill[tgt]] = pj;
        ++fill[tgt];
      }
      const int64_t tgt = n_tiles + J;
      S.pair_a[fill[tgt]] = (int32_t)(n_tiles + K);
      S.pair_b[fill[tgt]] = pj;
      ++fill[tgt];
    }
  }
  // ---- shared-memory window schedule (solve_kernel_v2)
  {
    S.win_slot.assign(n_tiles, -1);
    std::vector<std::vector<int32_t>> by_row(S.ntc);
    for (int J = 0; J < S.ntc; ++J)
      for (int32_t p = S.col_ptr[J] + 1; p < S.col_ptr[J + 1]; ++p) by_row[S.row_idx[p]].push_back(p);
    std::vector<int32_t> free_slots;
    S.n_win_slots = 0;
    for (int J = 0; J < S.ntc; ++J) {
      // tiles (J, K) were last read while column J was formed; column J's own tiles are written after that
      for (int32_t p : by_row[J]) free_slots.push_back(S.win_slot[p]);
      for (int32_t p = S.col_ptr[J] + 1; p < S.col_ptr[J + 1]; ++p) {
        if (!free_slots.empty()) { S.win_slot[p] = free_slots.back(); free_slots.pop_back(); }
        else S.win_slot[p] = S.n_win_slots++;
      }
    }
    S.late_ptr.assign(n_targets, 0);
    // Pairs of a target in tile column J are sorted by source column.  In the staggered schedule "early" pairs have source
    // columns <= J - 3: their operands are final two pipeline iterations before the target is, so the pair loop of the early
    // updates never waits for the triangular solve that runs beside it.  The (at most two) remaining pairs, source columns
    // J - 2 and J - 1, are applied by the warp that has just formed the tile of column J - 1 in the target's row
    // (solve_column).  That needs a carrier: tile (I, J - 1) and tile (J, J - 1) must exist for every target (I, J) that has a
    // source-(J - 2) pair -- always true for a band, not for every sparsity pattern.  Without carriers the schedule falls
    // back to early = source columns <= J - 2 and the kernel puts a barrier between solve and early updates (staggered = 0).
    auto sub_exists = [&](int J) {     // tile (J + 1, J)
      return J >= 0 && J + 1 < S.ntc && S.col_ptr[J + 1] - S.col_ptr[J] >= 2 && S.row_idx[S.col_ptr[J] + 1] == J + 1;
    };
    auto tile_exists = [&](int I, int J) {
      const int32_t* b = S.row_idx.data() + S.col_ptr[J];
      const int32_t* e = S.row_idx.data() + S.col_ptr[J + 1];
      const int32_t* it = std::lower_bound(b, e, I);
      return it != e && *it == I;
    };
    auto set_late = [&](int64_t tgt, int J, int back) {
      int32_t lp = S.pair_ptr[tgt + 1];
      if (J >= 1) {
        const int32_t lim = S.col_ptr[std::max(J - back, 0)];
        lp = S.pair_ptr[tgt];
        while (lp < S.pair_ptr[tgt + 1] && S.pair_b[lp] < lim) ++lp;
      }
      S.late_ptr[tgt] = lp;
    };
    // the target has a pair with source column J - 2 that is not an early pair (it is the first pair after the early ones)
    auto has_late2 = [&](int64_t tgt, int J) {
      const int32_t lp = S.late_ptr[tgt];
      return J >= 2 && lp < S.pair_ptr[tgt + 1] && S.pair_b[lp] < S.col_ptr[J - 1];
    };
    S.staggered = 1;
    for (int J = 0; J < S.ntc && S.staggered; ++J) {
      for (int32_t p = S.col_ptr[J]; p <= S.col_ptr[J + 1] && S.staggered; ++p) {
        const int64_t tgt = (p < S.col_ptr[J + 1]) ? p : n_tiles + J;
        set_late(tgt, J, 2);
        if (!has_late2(tgt, J) || tgt == S.col_ptr[J]) continue;          // (the diagonal target needs no carrier)
        const bool carrier = sub_exists(J - 1) && (tgt >= n_tiles || tile_exists(S.row_idx[tgt], J - 1));
        if (!carrier) S.staggered = 0;
      }
    }
    const int late_back = S.staggered ? 2 : 1;
    S.xo_ptr.assign(S.ntc + 1, 0);
    S.xo_idx.clear();
    for (int J = 0; J < S.ntc; ++J) {
      std::vector<int32_t> items;
      for (int32_t p = S.col_ptr[J]; p < S.col_ptr[J + 1]; ++p) { set_late(p, J, late_back); items.push_back(p); }
      set_late(n_tiles + J, J, late_back);
      items.push_back((int32_t)(n_tiles + J));
      std::stable_sort(items.begin(), items.end(), [&](int32_t a, int32_t b) {
        return (S.late_ptr[a] - S.pair_ptr[a]) > (S.late_ptr[b] - S.pair_ptr[b]);
      });
      S.xo_idx.insert(S.xo_idx.end(), items.begin(), items.end());
      S.xo_ptr[J + 1] = (int32_t)S.xo_idx.size();
    }
    S.win_a.assign(total, 0);
    S.win_b.assign(total, 0);
    S.win_ab.assign(2 * total, 0);
    for (int64_t p = 0; p < total; ++p) {
      const int32_t a = S.pair_a[p];
      S.win_a[p] = (a < n_tiles) ? S.win_slot[a] : -(int32_t)(a - n_tiles + 1);
      S.win_b[p] = S.win_slot[S.pair_b[p]];
      S.win_ab[2 * p] = S.win_a[p];
      S.win_ab[2 * p + 1] = S.win_b[p];
    }
    const int64_t n_items_total = S.xo_ptr[S.ntc];
    S.cdesc.assign(4 * n_items_total, 0);
    S.cslot.assign(n_items_total, -1);
    S.cord.assign(n_items_total, 0);
    S.cinfo.assign(4 * (int64_t)S.ntc, 0);
    S.max_col_pairs = 0;
    for (int J = 0; J < S.ntc; ++J) {
      const int32_t cp0 = S.col_ptr[J], ncol = S.col_ptr[J + 1] - cp0, xo0 = S.xo_ptr[J];
      const int32_t tp0 = S.pair_ptr[cp0], tpn = S.pair_ptr[cp0 + ncol] - tp0;
      const int64_t rt = n_tiles + J;
      const int32_t rp0 = S.pair_ptr[rt], rpn = S.pair_ptr[rt + 1] - rp0;
      S.cinfo[4 * J] = tp0; S.cinfo[4 * J + 1] = tpn; S.cinfo[4 * J + 2] = rp0; S.cinfo[4 * J + 3] = rpn;
      S.max_col_pairs = std::max(S.max_col_pairs, tpn + rpn);
      for (int li = 0; li <= ncol; ++li) {
        const int64_t tgt = (li < ncol) ? (cp0 + li) : rt;
        const int32_t shift = (li < ncol) ? tp0 : (rp0 - tpn);
        int32_t* d = &S.cdesc[4 * (int64_t)(xo0 + li)];
        d[0] = S.pair_ptr[tgt] - shift;
        d[1] = S.late_ptr[tgt] - shift;
        d[2] = S.pair_ptr[tgt + 1] - shift;
        d[3] = (li < ncol) ? S.a_map[tgt] : -1;
        // window slot + 1 (0: diagonal tile / rhs row) in the low bits, bit 20: the target has a source-(J - 2) pair
        S.cslot[xo0 + li] = (((li < ncol) ? S.win_slot[tgt] : -1) + 1) | ((S.staggered && has_late2(tgt, J)) ? (1 << 20) : 0);
      }
      // hand-out order of the early updates: longest item first (the kernel deals them to its 15 update warps in
      // snake order: 1..15, 15..1, ...)
      for (int it = 0; it <= ncol; ++it) {
        const int32_t tgt = S.xo_idx[xo0 + it];
        S.cord[xo0 + it] = (tgt < n_tiles) ? (tgt - cp0) : ncol;
      }
    }
    // operator tiles staged per column (only the items that carry one)
    S.ccol3.assign(4 * (int64_t)S.ntc, 0);
    S.ca_tile.clear();
    S.max_a_col = 0;
    for (int J = 0; J < S.ntc; ++J) {
      const int32_t cp0 = S.col_ptr[J], ncol = S.col_ptr[J + 1] - cp0, xo0 = S.xo_ptr[J];
      S.ccol3[4 * J] = (int32_t)S.ca_tile.size();
      int32_t na = 0;
      for (int li = 0; li < ncol; ++li) {
        int32_t& w = S.cdesc[4 * (int64_t)(xo0 + li) + 3];
        if (w >= 0) { S.ca_tile.push_back(w); w = na++; }
      }
      S.ccol3[4 * J + 1] = na;
      S.max_a_col = std::max(S.max_a_col, na);
    }
    // the staged tiles of kABufs consecutive columns are alive at the same time; they sit in a ring of operator-tile slots
    // (tile k of column J in slot (ccol3[J].x + k) mod a_ring)
    S.a_ring = 1;
    for (int J = 0; J < S.ntc; ++J) {
      int32_t live = 0;
      for (int d = 0; d < kABufs && J + d < S.ntc; ++d) live += S.ccol3[4 * (J + d) + 1];
      S.a_ring = std::max(S.a_ring, live);
    }
    // consumers of the "late" update: tile (I, J) feeds target (I, J + 1) together with tile (J + 1, J)
    S.cnext.assign(n_items_total, -1);
    S.chas.assign(S.ntc, 0);
    for (int J = 0; J + 1 < S.ntc; ++J) {
      const int32_t cp0 = S.col_ptr[J], ncol = S.col_ptr[J + 1] - cp0, xo0 = S.xo_ptr[J];
      if (ncol < 2 || S.row_idx[cp0 + 1] != J + 1) continue;
      S.chas[J] = 1;
      const int32_t np0 = S.col_ptr[J + 1], nncol = S.col_ptr[J + 2] - np0;
      for (int li = 1; li < ncol; ++li) {
        const int I = S.row_idx[cp0 + li];
        const int32_t* b = S.row_idx.data() + np0;
        const int32_t* e = b + nncol;
        const int32_t* it = std::lower_bound(b, e, I);
        if (it != e && *it == I) S.cnext[xo0 + li] = (int32_t)(it - b);
      }
      S.cnext[xo0 + ncol] = nncol;     // rhs row feeds the rhs row of the next column
    }
    S.ccol.assign(4 * (int64_t)(S.ntc + 1), 0);
    for (int J = 0; J <= S.ntc; ++J) {
      S.ccol[4 * J] = S.col_ptr[J];
      S.ccol[4 * J + 1] = (J < S.ntc) ? S.col_ptr[J + 1] - S.col_ptr[J] : 0;
      S.ccol[4 * J + 2] = S.xo_ptr[J];
      S.ccol[4 * J + 3] = (J < S.ntc) ? S.chas[J] : 0;
    }
  }
  // flops per mu: 2 * 512 per pair on L targets (8x8x8 multiply-add), plus potrf / trsm ~ 2 * 512 per tile
  S.flops = 0;
  for (int64_t tgt = 0; tgt < n_tiles; ++tgt) S.flops += (int64_t)count[tgt] * 1024;
  S.flops += n_tiles * 1024;
  // given order
  S.order = LRBMS_ORDER_GIVEN;
  S.perm.resize(n_sub);
  for (int i = 0; i < n_sub; ++i) S.perm[i] = i;
  S.iperm = S.perm;
  S.perm_offsets.assign(S.offsets.begin(), S.offsets.end() - 1);
  S.row_map.resize(S.n_red);
  for (int r = 0; r < S.n_red; ++r) S.row_map[r] = r;
  return LRBMS_OK;
}

size_t lrbms_window_smem_bytes(const lrbms_symbolic& S, int Q) {
  const int maxcol = std::max(1, S.max_targets - 1);
  const size_t MT = (size_t)S.max_targets;
  const size_t region = (size_t)std::max<int64_t>((int64_t)S.n_win_slots * 64, (int64_t)kBackStages * maxcol * 64);
  const size_t mcp = (size_t)std::max(1, S.max_col_pairs);
  return sizeof(double) * (region + 3 * MT * 64 + S.n_pad + 4 * 64 + 2 * kV2Warps * 8 + 32 + (size_t)S.a_ring * Q * 64) +
         16 * ((size_t)kMetaBufs * MT + (size_t)(S.ntc + 1) + 2 * (size_t)S.ntc) + 8 * (size_t)kMetaBufs * mcp +
         4 * (3 * (size_t)kMetaBufs * MT + S.ca_tile.size()) + 64;
}

namespace {

// Cuthill-McKee level-set order of the subdomain graph: per connected component (taken in order of their lowest subdomain)
// a breadth-first search from a pseudo-peripheral subdomain; the unvisited neighbours of each subdomain are appended by
// increasing degree (then index), so within a level subdomains follow their parent's position, then their degree.  On a
// grid of subdomains started in a corner the levels are the anti-diagonals.
std::vector<int32_t> cuthill_mckee(int n, const std::vector<std::vector<int32_t>>& adj) {
  std::vector<int32_t> order, dist(n, -1);
  order.reserve(n);
  std::vector<char> placed(n, 0);
  auto deg = [&](int v) { return (int)adj[v].size(); };
  // breadth-first levels from r over r's component; returns the eccentricity of r, dist holds the levels
  std::vector<int32_t> touched;
  auto bfs = [&](int r) {
    for (int v : touched) dist[v] = -1;
    touched.assign(1, r);
    dist[r] = 0;
    int ecc = 0;
    for (size_t h = 0; h < touched.size(); ++h) {
      const int v = touched[h];
      ecc = std::max(ecc, dist[v]);
      for (int w : adj[v])
        if (dist[w] < 0) { dist[w] = dist[v] + 1; touched.push_back(w); }
    }
    return ecc;
  };
  for (int s = 0; s < n; ++s) {
    if (placed[s]) continue;
    // pseudo-peripheral start (George and Liu): move to the lowest-degree subdomain of the last level while that
    // increases the eccentricity
    int root = s, ecc = bfs(s);
    for (;;) {
      int cand = -1;
      for (int v : touched)
        if (dist[v] == ecc && (cand < 0 || deg(v) < deg(cand) || (deg(v) == deg(cand) && v < cand))) cand = v;
      const int e2 = bfs(cand);
      if (e2 <= ecc) break;
      root = cand;
      ecc = e2;
    }
    const size_t head0 = order.size();
    order.push_back(root);
    placed[root] = 1;
    for (size_t h = head0; h < order.size(); ++h) {
      std::vector<int32_t> next;
      for (int w : adj[order[h]])
        if (!placed[w]) { placed[w] = 1; next.push_back(w); }
      std::sort(next.begin(), next.end(), [&](int a, int b) { return deg(a) != deg(b) ? deg(a) < deg(b) : a < b; });
      order.insert(order.end(), next.begin(), next.end());
    }
  }
  return order;
}

// Column-period model of solve_kernel_v2 in SM cycles per parameter, fitted to the per-warp cycle counters of the C2 system
// (8 x 8 subdomains, N = 20, lexicographic order; profiles/r02_timing_solve_v2.txt): a tile column takes at least the
// critical chain of warp 0 (8 x 8 potrf + inverse and the hand-off to the update warps), else the update warps' work --
// one round of triangular solves per 2 x 14 targets plus the column's update pairs spread over 14 warps, or the longest
// single target if that is longer; the backward substitution streams every L tile once.
double window_cost(const lrbms_symbolic& S) {
  constexpr double kChain = 5000.0, kSolveRound = 1600.0, kPair = 300.0, kBackTile = 60.0;
  constexpr int kUpdWarps = kV2Warps - 2;
  const int64_t n_tiles = S.n_tiles();
  double cost = kBackTile * (double)n_tiles;
  for (int J = 0; J < S.ntc; ++J) {
    const int ncol = S.col_ptr[J + 1] - S.col_ptr[J];
    int64_t pairs = 0, longest = 0;
    for (int32_t p = S.col_ptr[J]; p <= S.col_ptr[J + 1]; ++p) {
      const int64_t tgt = (p < S.col_ptr[J + 1]) ? p : n_tiles + J;
      const int64_t np = S.pair_ptr[tgt + 1] - S.pair_ptr[tgt];
      pairs += np;
      longest = std::max(longest, np);
    }
    const double rounds = (double)((ncol + 2 * kUpdWarps) / (2 * kUpdWarps));
    const double upd = kSolveRound * rounds + kPair * std::max((double)((pairs + kUpdWarps - 1) / kUpdWarps), (double)longest);
    cost += std::max(kChain, upd);
  }
  return cost;
}

}  // namespace

int lrbms_symbolic_choose_order(lrbms_symbolic& S, int Q, int64_t smem_budget, std::string* err) {
  auto fail = [&](const char* m) { if (err) *err = m; return (int)LRBMS_ERR_INVALID; };
  if (S.order != LRBMS_ORDER_GIVEN || S.ntc == 0 || (int)S.perm.size() != S.n_sub)
    return fail("symbolic_reorder: needs a schedule built in the given order");
  const int n = S.n_sub;
  std::vector<std::vector<int32_t>> adj(n);
  for (size_t b = 0; b < S.block_i.size(); ++b) {
    const int i = S.block_i[b], j = S.block_j[b];
    if (i == j) continue;
    adj[i].push_back(j);
    adj[j].push_back(i);
  }
  for (auto& a : adj) {
    std::sort(a.begin(), a.end());
    a.erase(std::unique(a.begin(), a.end()), a.end());
  }
  std::vector<int32_t> cand[3];
  cand[LRBMS_ORDER_GIVEN] = S.perm;
  cand[LRBMS_ORDER_CM] = cuthill_mckee(n, adj);
  cand[LRBMS_ORDER_RCM].assign(cand[LRBMS_ORDER_CM].rbegin(), cand[LRBMS_ORDER_CM].rend());
  S.order_cost[LRBMS_ORDER_GIVEN] = window_cost(S);
  int best = LRBMS_ORDER_GIVEN;
  double best_cost = S.order_cost[LRBMS_ORDER_GIVEN];
  lrbms_symbolic best_T;
  for (int k = LRBMS_ORDER_CM; k <= LRBMS_ORDER_RCM; ++k) {
    S.order_cost[k] = 0.0;
    if (cand[k] == cand[LRBMS_ORDER_GIVEN]) continue;
    // the permuted pattern: subdomain perm[k] in position k; every stored block (i >= j) lands in the lower triangle
    std::vector<int32_t> ip(n), sizes_p(n), bi_p, bj_p;
    for (int p = 0; p < n; ++p) { ip[cand[k][p]] = p; sizes_p[p] = S.sizes[cand[k][p]]; }
    for (size_t b = 0; b < S.block_i.size(); ++b) {
      const int i = S.block_i[b], j = S.block_j[b];
      if (i < j) continue;
      bi_p.push_back(std::max(ip[i], ip[j]));
      bj_p.push_back(std::min(ip[i], ip[j]));
    }
    lrbms_symbolic T;
    if (int rc = lrbms_symbolic_build(T, n, sizes_p.data(), (int32_t)bi_p.size(), bi_p.data(), bj_p.data(), err)) return rc;
    S.order_cost[k] = window_cost(T);
    if (T.staggered < S.staggered || (int64_t)lrbms_window_smem_bytes(T, Q) > smem_budget) continue;
    if (S.order_cost[k] < best_cost) {
      best = k;
      best_cost = S.order_cost[k];
      T.perm = cand[k];
      T.iperm = ip;
      best_T = std::move(T);
    }
  }
  if (best == LRBMS_ORDER_GIVEN) return LRBMS_OK;
  // keep the given-order description of the system (estimator, band solver, the caller's layout), take the schedule
  lrbms_symbolic& T = best_T;
  T.order = best;
  for (int k = 0; k < 3; ++k) T.order_cost[k] = S.order_cost[k];
  T.perm_offsets.resize(n);
  T.row_map.resize(S.n_red);
  for (int i = 0; i < n; ++i) {
    T.perm_offsets[i] = T.offsets[T.iperm[i]];
    for (int a = 0; a < S.sizes[i]; ++a) T.row_map[T.perm_offsets[i] + a] = S.offsets[i] + a;
  }
  T.sizes = std::move(S.sizes);
  T.offsets = std::move(S.offsets);
  T.block_i = std::move(S.block_i);
  T.block_j = std::move(S.block_j);
  T.half_bandwidth = S.half_bandwidth;
  S = std::move(T);
  return LRBMS_OK;
}

extern "C" {

int lrbms_symbolic_create(int32_t n_sub, const int32_t* basis_sizes, int32_t n_blocks, const int32_t* block_i,
                          const int32_t* block_j, lrbms_symbolic_t* out) {
  if (!out) return LRBMS_ERR_INVALID;
  *out = nullptr;
  lrbms_symbolic* S = new lrbms_symbolic();
  std::string err;
  int rc = lrbms_symbolic_build(*S, n_sub, basis_sizes, n_blocks, block_i, block_j, &err);
  if (rc) { delete S; return rc; }
  *out = S;
  return LRBMS_OK;
}

int lrbms_symbolic_reorder(lrbms_symbolic_t s, int32_t Q, int64_t smem_budget) {
  if (!s || Q < 1) return LRBMS_ERR_INVALID;
  return lrbms_symbolic_choose_order(*s, Q, smem_budget, nullptr);
}

int lrbms_symbolic_destroy(lrbms_symbolic_t s) {
  delete s;
  return LRBMS_OK;
}

int lrbms_symbolic_info(lrbms_symbolic_t s, int32_t what, int64_t* out) {
  if (!s || !out) return LRBMS_ERR_INVALID;
  switch (what) {
    case 0: *out = s->n_red; break;
    case 1: *out = s->n_pad; break;
    case 2: *out = s->ntc; break;
    case 3: *out = s->n_tiles(); break;
    case 4: *out = s->n_a_tiles; break;
    case 5: *out = s->n_pairs(); break;
    case 6: *out = s->flops; break;
    case 7: *out = s->max_targets; break;
    case 8: *out = s->n_win_slots; break;
    case 9: *out = s->max_col_pairs; break;
    case 10: *out = s->max_a_col; break;
    case 11: *out = s->staggered; break;
    case 12: *out = s->order; break;
    case 13: case 14: case 15: *out = (int64_t)s->order_cost[what - 13]; break;
    default: return LRBMS_ERR_INVALID;
  }
  return LRBMS_OK;
}

int64_t lrbms_symbolic_get(lrbms_symbolic_t s, int32_t which, int32_t* out, int64_t cap) {
  if (!s || !out) return LRBMS_ERR_INVALID;
  const std::vector<int32_t>* v = nullptr;
  switch (which) {
    case 0: v = &s->col_ptr; break;
    case 1: v = &s->row_idx; break;
    case 2: v = &s->pair_ptr; break;
    case 3: v = &s->pair_a; break;
    case 4: v = &s->pair_b; break;
    case 5: v = &s->a_map; break;
    case 6: v = &s->win_slot; break;
    case 7: v = &s->late_ptr; break;
    case 8: v = &s->win_a; break;
    case 9: v = &s->win_b; break;
    case 10: v = &s->xo_ptr; break;
    case 11: v = &s->xo_idx; break;
    case 12: v = &s->cnext; break;
    case 13: v = &s->chas; break;
    case 14: v = &s->cord; break;
    case 15: v = &s->perm; break;
    case 16: v = &s->iperm; break;
    case 17: v = &s->row_map; break;
    default: return LRBMS_ERR_INVALID;
  }
  const int64_t n = std::min<int64_t>(cap, (int64_t)v->size());
  std::copy(v->begin(), v->begin() + n, out);
  return n;
}

}  // extern "C"
