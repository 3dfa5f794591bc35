// K device-resident CSR relationship matrices (the `mats` / `mat_list` arguments of HE / REML / compute_gradients,
// reference scilmm/SparseCholesky.py:62,177,192) and the per-pattern structures built on them.
#pragma once
#include <cstdint>
#include <map>
#include <stdexcept>
#include <utility>
#include <vector>

#include "common.h"

namespace slmm {

constexpr int MAXK = 8;

struct CsrDev {
  // views: the owned buffers below, the pattern leader's arrays, or device arrays bound by the caller
  const int32_t* indptr = nullptr;
  const int32_t* indices = nullptr;
  const double* data = nullptr;
  DevPtr<int32_t> own_indptr, own_indices;
  DevPtr<double> own_data;
  int64_t nnz = 0;
  int pattern = -1;       // index of the first matrix with this pattern
  std::vector<int32_t> h_indptr;   // kept for pattern comparison (uploaded matrices only)
  uint64_t idx_hash = 0;
  int symmetric = -1;      // -1 unknown, 0 no, 1 yes (checked on the device on first use)
  int32_t* rend = nullptr; // per row: one past the last entry with col <= row (pattern leaders only, built lazily)
  DevPtr<int32_t> rend_base;   // allocation behind rend (rend is shifted by -r0 for row-block shards)
};


struct RedDesc { int64_t off; int32_t stride, nblocks, dst, pad; };

// Tiled lower triangle of one symmetric pattern in the factor's fill-reducing order (quadform_tiled.cu)
struct QuadTiles {
  int ntiles = 0, nrb = 0, ncta = 0;
  int64_t nentries = 0, ndistinct = 0;
  DevPtr<int64_t> tile_ptr;         // [ntiles+1] entry range of every tile
  DevPtr<int32_t> tile_rb;          // [ntiles] row block (64 permuted rows) of the tile
  DevPtr<int32_t> tile_dc0;         // [ntiles] first entry of the tile's column list in dcols
  DevPtr<int32_t> tile_nc;          // [ntiles] columns in the tile (<= 64)
  DevPtr<uint16_t> rowptr;          // [ntiles*65] row starts inside the tile
  DevPtr<uint16_t> rc;              // [nentries] local column << 1 | diagonal flag
  DevPtr<uint8_t> roword;           // [ntiles*64] rows of a tile by decreasing length, dealt to the 8 warps in snake order (0xFF: none)
  DevPtr<uint32_t> pos;             // [nentries] position of the entry in the matrix' own CSR arrays
  DevPtr<int32_t> dcols;            // [ndistinct] ORIGINAL row id of the gathered block for every tile column
  DevPtr<int32_t> rowid;            // [nrb*64] original row id of every permuted row (-1 past n)
  DevPtr<int32_t> cta_begin;        // [ncta+1] contiguous tile ranges of equal cost
  DevPtr<int32_t> pair_base;        // [ncta+1] first (CTA, row block) pair of every CTA
  DevPtr<int32_t> pair_rb;          // [npairs] row block of every pair
  DevPtr<double> hpairs;            // [npairs][64][2][16] narrow-block row products, one block per pair
  int npairs = 0;
  std::vector<int64_t> cta_stats;    // [ncta][3] tiles, non-empty rows, entries of every CTA's range (host copy)
  DevPtr<long long> cta_cycles;      // [ncta] clock64 span of every CTA in the last pass (developer profile)
  std::vector<DevPtr<double>> vals;  // per matrix of the set sharing this pattern: weighted values in tile order
  std::vector<int> vals_of;         // which matrix each vals[] belongs to
};

}  // namespace slmm

struct slmm_matset {
  int n = 0, K = 0;
  int r0 = 0, r1 = 0;      // rows held by this set (a row-block shard of the HE path holds [r0, r1) only)
  bool sharded() const { return r0 != 0 || r1 != n; }
  std::vector<slmm::CsrDev> m;
  std::map<std::pair<int, int>, slmm::DevPtr<int64_t>> cross_maps;   // (probe pattern, target pattern) -> position map (device)
  std::map<int, slmm::QuadTiles> tiles;                  // pattern leader -> tiled lower triangle (built on request)
  slmm::DevPtr<double> d_partial;
  size_t partial_cap = 0;
  slmm::DevPtr<double> d_y;
  slmm::DevPtr<double> d_out;
  slmm::DevPtr<int32_t> d_dst;
  // HE calls: one partial arena for all passes + the cached reduction table
  slmm::DevPtr<double> he_arena;
  size_t he_used = 0;
  static constexpr size_t HE_ARENA = (size_t)148 * 8 * 1024;
  std::vector<slmm::RedDesc> he_desc, he_desc_cached;
  slmm::DevPtr<slmm::RedDesc> d_he_desc;
  double* he_part(size_t count) {
    if (!he_arena) he_arena = slmm::dev_alloc<double>(HE_ARENA);
    if (he_used + count > HE_ARENA) throw std::runtime_error("HE partial arena exhausted");
    double* p = he_arena.get() + he_used;
    he_used += count;
    return p;
  }
  void he_add(const double* part, int nblocks, int nv, const int32_t* dst) {
    for (int k = 0; k < nv; k++) he_desc.push_back({(int64_t)(part - he_arena.get()) + k, nv, nblocks, dst[k], 0});
  }
  double* partial(size_t count) {
    if (count > partial_cap) {
      // free before allocating: the old and the new buffer are never held together
      d_partial.reset();
      partial_cap = 0;
      d_partial = slmm::dev_alloc<double>(count);
      partial_cap = count;
    }
    return d_partial.get();
  }
};

