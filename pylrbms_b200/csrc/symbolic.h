// Host-only symbolic phase of the mu-batched reduced solve: 8x8-tile sparse Cholesky schedule.
#pragma once
#include <cstddef>
#include <cstdint>
#include <string>
#include <vector>

// Shape of solve_kernel_v2 (online.cu) that its shared-memory footprint depends on
constexpr int kV2Warps = 16;
constexpr int kBackStages = 6;   // backward-substitution ring; columns are prefetched kBackStages - 2 ahead
constexpr int kMetaBufs = 5;     // column metadata: columns J-1 .. J+3 are alive at the same time (staged by cp.async)
constexpr int kABufs = 3;        // staged operator tiles: only needed while a column's early updates run

// Elimination order of the subdomains (lrbms_symbolic::order)
enum { LRBMS_ORDER_GIVEN = 0, LRBMS_ORDER_CM = 1, LRBMS_ORDER_RCM = 2 };

struct lrbms_symbolic {
  int32_t n_sub = 0;
  std::vector<int32_t> sizes, offsets;   // N_i, prefix sums (n_sub + 1), in the given subdomain order
  // Elimination order.  The tile schedule below is that of the symmetrically permuted operator P A P^T in which
  // subdomain perm[k] comes k-th; iperm[i] is the position of subdomain i.  perm_offsets[i] = first row of subdomain i in
  // the permuted scalar numbering, row_map[r] = given row of permuted row r (n_red entries).  Given order: identities.
  int32_t order = LRBMS_ORDER_GIVEN;
  std::vector<int32_t> perm, iperm, perm_offsets, row_map;
  double order_cost[3] = {0.0, 0.0, 0.0};   // window-kernel cost model of the given, CM and RCM order (0: not evaluated)
  int32_t n_red = 0;                     // sum N_i
  int32_t n_pad = 0;                     // n_red rounded up to a multiple of 8
  int32_t ntc = 0;                       // tile columns
  int32_t half_bandwidth = 0;            // scalar half bandwidth of the stored lower blocks (max row - column)
  // L tile pattern, compressed by tile column; rows ascending, the diagonal tile first
  std::vector<int32_t> col_ptr, row_idx;
  // update pairs per target: targets are the L tiles (slot order) followed by one rhs target per tile column.
  // pair (a, b): target -= tile[a] * tile[b]^T with a, b slots (slots >= n_tiles address the forward-solve row y_K)
  std::vector<int32_t> pair_ptr, pair_a, pair_b;
  // a_map[slot] = index of the tile in the assembled-operator tile list, or -1 for pure fill
  std::vector<int32_t> a_map;
  int32_t n_a_tiles = 0;
  // scatter list to build operator tiles from reduced blocks: for every stored block (i >= j) entry
  // (block index b, a, c) -> (a-tile index, position in tile); generated on demand by the plan
  std::vector<int32_t> block_i, block_j;
  int64_t flops = 0;
  int32_t max_targets = 0;
  // ---- schedule of the shared-memory-window kernel (solve_kernel_v2)
  // An off-diagonal tile (I, K) of L is live from the step that creates it (column K) until column I has been
  // formed; live tiles are kept in a shared-memory window.  win_slot[tile] is its window slot (-1: diagonal tile).
  std::vector<int32_t> win_slot;
  int32_t n_win_slots = 0;
  // pairs of every target are sorted by source column K; the "late" pairs (K == J - 1, operands produced by the
  // immediately preceding column) start at late_ptr[target]
  std::vector<int32_t> late_ptr;
  // 1: early pairs stop at source column J - 3 and the source-(J - 2) pair rides with the late update (see symbolic.cpp);
  // 0: early pairs include source column J - 2 (patterns without a carrier tile for every such pair)
  int32_t staggered = 1;
  // pair operands as window slots: win_a[p] (or -(K + 1) for the forward-solve row y_K), win_b[p]
  std::vector<int32_t> win_a, win_b;
  // targets of each tile column (tiles of the column, then its rhs target) ordered by decreasing early work
  std::vector<int32_t> xo_ptr, xo_idx;
  // per-column staging tables of the kernel (indexed xo_ptr[J] + li, li = position of the target in its column,
  // the rhs target last):  cdesc = {pair begin, late begin, pair end (all relative to the column's staged pair
  // list), a_map};  cslot = (window slot + 1) | (target has a source-(J - 2) pair) << 20;  cord = li in hand-out order;  cinfo[J] = {first tile pair, tile pairs,
  // first rhs pair, rhs pairs};  win_ab = interleaved (win_a, win_b)
  //   cord = li in hand-out order (longest early update first);  cnext = li of the target (I, J + 1) fed by tile (I, J) (-1: none);
  //   chas[J] = 1 if tile (J + 1, J) exists (then every tile of column J has exactly one "late" consumer in column J + 1)
  std::vector<int32_t> cdesc, cslot, cord, cinfo, win_ab, cnext, chas;
  // per-column table kept in shared memory for the whole kernel: ccol[J] = {first tile, tiles, first item, chas[J]}
  // (one extra entry at J = ntc with the end offsets);  ccol2[J] = {first tile pair, tile pairs, first rhs pair, rhs pairs};
  // ccol3[J] = {first staged operator tile (index into ca_tile), staged operator tiles, 0, 0};  ca_tile = operator tile
  // indices (a_map values) in staging order; cdesc[.].w is the staged position of the item's operator tile or -1
  std::vector<int32_t> ccol, ccol3, ca_tile;
  int32_t max_a_col = 0;
  int32_t a_ring = 1;          // operator-tile slots of the staging ring: most staged tiles of kABufs consecutive columns
  int32_t max_col_pairs = 0;

  int64_t n_tiles() const { return (int64_t)row_idx.size(); }
  int64_t n_pairs() const { return (int64_t)pair_a.size(); }
};

// sizes, offsets, validation and the half bandwidth only (what the band solver needs); lrbms_symbolic_build starts with it
int lrbms_symbolic_basics(lrbms_symbolic& S, int32_t n_sub, const int32_t* sizes, int32_t n_blocks, const int32_t* bi,
                          const int32_t* bj, std::string* err);
int lrbms_symbolic_build(lrbms_symbolic& S, int32_t n_sub, const int32_t* sizes, int32_t n_blocks, const int32_t* bi,
                         const int32_t* bj, std::string* err);
// dynamic shared memory (bytes) solve_kernel_v2 needs for the schedule S and Q affine operator terms
size_t lrbms_window_smem_bytes(const lrbms_symbolic& S, int Q);
// Re-plan S (built by lrbms_symbolic_build in the given order) in the cheapest of the given, Cuthill-McKee and reverse
// Cuthill-McKee subdomain orders by the window kernel's cost model.  A candidate must keep the staggered schedule if the
// given order has it and its footprint for Q terms must stay within smem_budget bytes; the given order wins ties.
int lrbms_symbolic_choose_order(lrbms_symbolic& S, int Q, int64_t smem_budget, std::string* err);
