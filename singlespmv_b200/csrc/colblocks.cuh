// colblocks.cuh -- column-blocked multiply engine for the row-wise formats (ELL, JDS, SS) on gather-bound matrices.
//
// Config 2 (uniform random, x = 134 MB) misses L2 on every x[col]: 5.6x DRAM over-fetch (profiles/r1_ncu_kernels.md).
// The reference's remedy is column blocking (CSS, src/opt_css.cpp:33-45): process one column block for ALL rows before
// the next, so that the block's slice of x stays L2-resident.  UNLIKE CSS, block b CONTINUES each row's running sum where
// block b-1 left it (acc = y[r]; acc += ...; y[r] = acc): a row is still summed strictly in ascending column order with
// unfused mul/add.  Two engines:
//  * one sliced ELL per column block (ell.cu, EllColBlocks): one lane per row, padded to the longest piece of a row inside
//    the block per 32-row slice -- the default while the padding stays below 2 slots per entry (config 2: 1.58); same bits
//    as the format's own kernel and the reference for every row;
//  * the CSS partition (stable by column block, one row_ptr per block) with W = 1 and without the chain metadata, every
//    block multiplied by the tile-stream kernel (ss.cu, CrsColBlocks): skewed matrices; rows of up to 64 entries per block
//    give the same bits.
// Block width: slices of x of at most 45 MB (round 1 measured 2 / 3 / 4 / 8 blocks on config 2: 3 is the optimum).
// Measured alternatives for the per-block kernel (profiles/r2_experiments.md): the TMA-fed row-chunk stream (4.43 ms
// on c2 against 2.92 ms: with one thread per row and two shared-memory stages an SM holds ~800 threads, too few gathers
// in flight) and a padding-free "compressed slices" layout with ballot/popc addressing (4.90 ms).
#pragma once
#include <memory>

#include "common.cuh"

namespace b2 {

constexpr long long COLBLOCK_SLICE_BYTES = 45LL << 20;
constexpr int COLBLOCK_MAX = 32;

struct ColBlockEngine {
    virtual ~ColBlockEngine() {}
    virtual int run(const double *x, double *y, int rb, int re, cudaStream_t s) = 0;
    virtual int run_block(int, const double *, double *, int, int, cudaStream_t) { return B200SPMV_ERR_UNSUPPORTED; }   // one block only
    // host-side bookkeeping of rows [rb, re) (may synchronise): afterwards run() on them never does (graph capture)
    virtual int prepare(int, int) { return B200SPMV_OK; }
    virtual int n_blocks() const = 0;
    virtual const char *name() const = 0;
};

// Decides whether the matrix wants column blocking (x larger than 64 MB and rows spread over >= 1.5 blocks on average)
// and builds the engine; *out stays empty otherwise.
// want: 0 = decide, n > 0 = n blocks whatever the statistics say (tests, experiments), < 0 = never.
int make_col_block_engine(const CooView &A, const int *row_ptr, int want, cudaStream_t s,
                          std::unique_ptr<ColBlockEngine> *out);
// one sliced ELL per column block (ell.cu); *out stays empty when the blocks would need more than maxRatio slots per entry
// B: block width (0 = ceil(nCol / nb)); later: what the blocks after the first do with y (CS_CONTINUE, or CS_ADD for CSS)
int make_ell_col_blocks(const CooView &A, const int *row_ptr, int nb, int B, int later, double maxRatio, cudaStream_t s,
                        std::unique_ptr<ColBlockEngine> *out);

}  // namespace b2
