// entry_stream.cuh -- the CRS "entry stream": the row-length-agnostic multiply for rows too long for the row-chunk stream
// (BASELINE.json: "warp- and vector-per-row CRS with an adaptive row-bin scheduler" -- here the scheduler disappears: every
// warp moves the same number of entries whatever the rows look like, 27 entries per row (config 4) or 0 ... 10^5 (R-MAT)).
//
// It is the COO entry stream (coo.cu) without the 4 B/entry row ids.  At conversion the row pointers are turned into
//   bits[]     one bit per entry: set where a (non-empty) row begins                        (nnz / 8 bytes)
//   grpRun[g]  number of row starts in front of entry 128 g                                 (4 bytes per 128 entries)
//   nzrow[k]   the k-th non-empty row -- only when the matrix has empty rows (else the identity)
//   empty[]    the empty rows (zero-filled by a tiny kernel: beta = 0)
// and the multiply never reads row_ptr: a lane takes 4 consecutive entries (idx, val: 12 B/entry, by TMA bulk copies on banded
// matrices, by its own 128-bit loads on gather-bound ones), its 4 start bits, sums its runs in registers; a segmented warp
// scan per 128 entries closes the runs that cross lanes; ballots over the start bits give every lane the index of the run it
// continues.  Chunk pieces are stitched per tile, tile pieces by a fix-up kernel in tile order: deterministic, no atomics.
// Sums are re-associated across lanes: within the 1e-12 tolerance, not the bits of the sequential order (options.crs_path = 1
// keeps the tile-stream, which preserves them for rows of up to 64 entries).
#pragma once
#include <map>

#include "common.cuh"

namespace b2 {

// entries per tile: c4 (TMA-fed) 659 against 620 GFLOP/s with 1024; c3 (load-fed) 418 against 411
constexpr int ES_E = 2048;
constexpr int ES_KMAX = 8;         // vectors of one multi-vector multiply

// Y[r, j] = 0 for r < nRow, j < k (row-major Y): the multi-vector multiply of a matrix without entries
int zero_rows_multi(int nRow, int k, double *Y, long long ldy, cudaStream_t s);
int zero_rows_multi(int nRow, int k, float *Y, long long ldy, cudaStream_t s);

struct EntryStream {
    // borrowed
    const int *ptr = nullptr, *idx = nullptr;
    const void *val = nullptr;         // fp64, or fp32 when f32 (the multi-vector multiply with fp32 vectors only)
    bool f32 = false;
    int nRow = 0, nnz = 0;
    // owned
    bool ok = false, tma = false;
    int nTiles = 0, nEmpty = 0;
    DevBuf<unsigned> bits;
    DevBuf<int> grpRun, nzrow, empty;
    DevBuf<double> carry;
    DevBuf<double> carryK;             // nTiles x ES_KMAX carries of run_multi (f32: twice that), allocated by its first call
    std::map<std::pair<int, int>, std::pair<int, int>> range_cache;

    // gather_bound: the x gathers need L2 residency (primitives.cu gathers_need_l2) -> load-fed, else TMA-fed
    // val_is_f32: fp32 values, for run_multi_f32 only (the metadata does not depend on the value type)
    int build(const int *ptr_d, const int *idx_d, const void *val_d, bool val_is_f32, int nRow_, int nnz_, bool gather_bound,
              cudaStream_t s);
    // back to the state of a new EntryStream: ok = false, borrowed pointers and shape cleared, metadata, carries and
    // cached row ranges released.  build() starts with it; a conversion that does not build the entry stream calls it,
    // so nothing of an earlier matrix survives.
    void reset();
    int prepare(int rb, int re);
    int run_rows(const double *x, double *y, int rb, int re, cudaStream_t s);
    // Y[:, 0..k) := A X[:, 0..k) over all rows (k <= ES_KMAX, row-major); each column is summed as run_rows sums it.
    // The first call allocates the carries: refused with B200SPMV_ERR_STATE inside a stream capture.
    int run_multi(int k, const double *X, long long ldx, double *Y, long long ldy, cudaStream_t s);
    // the same with fp32 values and vectors, products and sums in fp32 or (acc64) fp64.  A row that runs past a tile has its
    // partial kept in AT until the fix-up adds the later tiles' carries: Y is rounded to fp32 once per row.
    int run_multi_f32(int k, const float *X, long long ldx, float *Y, long long ldy, bool acc64, cudaStream_t s);
};

}  // namespace b2
