// chunk_stream.cuh -- the TMA-fed "row-chunk stream": the multiply for CRS-shaped data whose rows are short
// (longest row <= CS_MAXLEN): CRS and SS as they are, every column block of CSS, and the column-blocked layout the
// row-wise formats switch to on gather-bound matrices (colblocks.cuh).
//
// A persistent CTA walks chunks of TH consecutive rows (chunk boundaries are multiples of TH, so the largest chunk --
// known at conversion -- bounds the shared-memory stage).  The idx/val run of a chunk is contiguous: ONE elected thread
// brings it into shared memory with two 1-D bulk copies (cp.async.bulk + mbarrier transaction count, SASS UBLKCP) while
// all threads are still busy with the previous chunk.  The matrix stream therefore never touches the threads' load
// pipeline or L1 (measured on B200: an SM sustains about one L1-missing sector per clock, profiles/r2_gather_ceiling.md
// -- the x gathers need all of it); the threads spend their own loads on the row pointers (prefetched one chunk ahead
// in registers) and on the gathers.  One thread per row, ascending column order, unfused mul/add -> bit-identical to
// the reference's CRS loop (src/opt_crs.cpp:61-67) for every row.
// Measured on config 5 (lap3d7 512^3): 920 GFLOP/s = 1.04 of the measured copy peak, against 728 for round 1's
// warp-per-32-rows row-block stream and 702 for the tile-stream kernel (profiles/r2_experiments.md).
#pragma once
#include "common.cuh"

namespace b2 {

constexpr int CS_MAXLEN = 16;      // longest row the row-chunk stream takes (longer: tile-stream kernel; measured on c4's 27-entry
                                   // rows: a looped variant for rows up to 32 was no faster than the tile-stream, 627 vs 645 GFLOP/s)
constexpr int CS_SLACK = 8;        // entries of allocation slack the caller keeps behind idx / val (copies end on 16 bytes)
constexpr int CS_MAXSTAGES = 4;

// Column feed "offset dictionary" (multiply-only metadata, built at conversion): on stencils and other banded matrices a
// row's columns are the row number plus a few offsets that repeat from row to row.  Each chunk stores its distinct
// col - row offsets once (ascending, at most CS_DICT), and each row a bitmask of the offsets it uses; bit j of row r
// stands for column r + dict[j].  Walking the set bits from low to high visits a row's entries in idx order, so the
// sums are the same as with the idx feed, bit for bit.  A chunk's record, CS_META_INTS(TH) ints:
//   dict[CS_DICT] | wbase[TH / 32]: ptr of the first row of every warp | mask[TH]: uint16 per row (0 past nRow)
// It replaces 4 B/entry of idx and 4 B/row of ptr with (64 + TH / 8 + 2 TH) B per chunk: on c5 0.32 GB instead of 4.29 GB.
constexpr int CS_DICT = 16;
__host__ __device__ constexpr int CS_META_INTS(int th) { return CS_DICT + th / 32 + th / 2; }
enum { CS_FEED_IDX = 0, CS_FEED_DICT = 1 };

struct ChunkStream {
    const int *ptr = nullptr, *idx = nullptr;
    const void *val = nullptr;
    bool f32 = false, ok = false;
    int nRow = 0, maxLen = 0, th = 0, cap = 0;
    int feed = CS_FEED_IDX;            // CS_FEED_DICT when every chunk fits CS_DICT offsets (and B200SPMV_CS_FEED != idx)
    DevBuf<int> meta;                  // CS_FEED_DICT: nChunks records of CS_META_INTS(th) ints, then CS_SLACK zeroed ints

    // ok = the matrix qualifies (0 < longest row <= CS_MAXLEN); also picks the feed; synchronises s (once)
    int build(const int *ptr_d, const int *idx_d, const void *val_d, bool val_is_f32, int nRow_, int nnz, int maxLen_,
              cudaStream_t s);
    int run(const double *x, double *y, int rb, int re, int acc, cudaStream_t s) const;
    int run_f32(const float *x, float *y, int rb, int re, int acc, bool acc64, cudaStream_t s) const;
};

}  // namespace b2
