// tile_stream.cuh -- the nnz-balanced "tile stream" multiply shared by CRS, SS and CSS.
//
// The non-zero stream is cut into fixed tiles of TS_TILE entries, one CTA per tile, so every
// CTA moves the same number of bytes whatever the row-length distribution (R-MAT rows span
// 0 ... 10^5+).  A CTA
//   1. streams its col/val slice with 128-bit loads (L1 no-allocate, L2 evict-first), gathers x
//      and parks the products in shared memory -- never in HBM (the reference's SS plugin
//      materialises them in val_buf, src/opt_ss.cpp:226-238, costing +16 B/nnz);
//   2. reduces the rows it OWNS (rows whose first entry lies in the tile) with an in-tile row-bin
//      scheduler: short rows one thread each, sequentially in ascending column order with
//      unfused mul/add (bit-identical to reference src/opt_crs.cpp:61-67); long rows one warp
//      each (lanes stride, shuffle tree); the piece of a row carried in from the previous tile
//      is reduced by a warp into carry[tile].
// A second, tiny kernel finishes rows that cross tile boundaries: short ones are recomputed
// sequentially (so EVERY row up to TS_LONG entries is bit-exact), long ones get their carries
// added in tile order (deterministic).
//
// Variants measured and rejected on B200 (profiles/r1_call8_9_summary.md): scalar lane-contiguous loads (-20 %:
// 24 instead of 14 load instructions per thread), row_ptr staged in shared memory + warp-local long rows
// (-15 %: 40 registers -> 6 instead of 8 resident CTAs), cp.async.bulk.prefetch.L2 of the tile a later wave will
// stream (-4 % to -27 % with distance), 8-lane sub-warps for rows of 17-256 entries (c4: -26 %), CTA widths 64 / 128 / 512 (c5: -9 / -4 / -3 %), a persistent
// cp.async double-buffered loop at 4 CTAs/SM (c5: -17 %, gather-bound c2/c3: -55 %: the x gathers need the threads).
// Resident CTAs x 24 KB in flight is what feeds HBM.
#pragma once
#include <map>

#include "common.cuh"

namespace b2 {

constexpr int TS_THREADS = 256;
constexpr int TS_IPT = 8;
constexpr int TS_TILE = TS_THREADS * TS_IPT;   // 2048 non-zeros = 24 KB of matrix per CTA
constexpr int TS_LONG = 64;                    // rows longer than this are reduced by a warp
constexpr int TS_MAXLONG = TS_TILE / TS_LONG + 2;

struct TileStream {
    // borrowed
    const int *row_ptr = nullptr;   // [nRow+1]
    const int *col = nullptr;       // [nnz] (may be padded beyond nnz; padding is never read)
    const void *val = nullptr;      // double[nnz], or float[nnz] when f32 (fp32 storage, fp64 arithmetic)
    bool f32 = false;
    int nRow = 0, nnz = 0;
    // owned
    int nTiles = 0;
    DevBuf<int> tile_row;           // [nTiles+1]: first row whose first entry is >= tile start
    DevBuf<double> carry;           // [nTiles], [2 nTiles] when f32 (tile_stream.cu ts_slots)

    int build(const int *row_ptr_d, const int *col_d, const void *val_d, bool val_is_f32, int nRow_, int nnz_,
              cudaStream_t s);
    // y[rowLo..rowHi) = (accumulate ? y : 0) + A x, restricted to tiles [tileLo, tileHi)
    // accumulate: CS_OVERWRITE / CS_CONTINUE / CS_ADD (common.cuh)
    int run(const double *x, double *y, int accumulate, int rowLo, int rowHi, int tileLo, int tileHi,
            cudaStream_t s) const;
    int run_all(const double *x, double *y, int accumulate, cudaStream_t s) const
    {
        return run(x, y, accumulate, 0, nRow, 0, nTiles, s);
    }
    // rows [rb, re) only: looks up (and caches) the tiles that hold their entries
    int run_rows(const double *x, double *y, int accumulate, int rb, int re, cudaStream_t s);
    int prepare(int rb, int re);
    int run_rows_f32(const float *x, float *y, int accumulate, int rb, int re, bool acc64, cudaStream_t s);
    size_t meta_bytes() const { return tile_row.bytes(); }
    std::map<std::pair<int, int>, std::pair<int, int>> range_cache;
};

}  // namespace b2
