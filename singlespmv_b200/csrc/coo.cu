// coo.cu -- COO plugin (/root/reference/src/opt_coo.{h,cpp}): the converted matrix IS the sorted
// triplet list (the reference aliases the input arrays, opt_coo.cpp:14-19); multiply is y = 0 followed
// by an `omp atomic` scatter-add per entry (:34-46).
//
// B200 multiply: no atomics, no zero-fill pass, two kernels in this file:
//  * coo_stream_kernel (default, options.coo_path = 0): the "entry stream" -- TMA-fed tiles, per-lane runs in registers,
//    one segmented warp scan per 128 entries, deterministic stitching of the pieces (described at the kernel);
//  * coo_tile_kernel (coo_path = 1, and the COO tail of HYB): the order-preserving kernel of round 1.  The entry stream is
//    cut into tiles of COO_TILE entries (one CTA each).  A CTA streams row/col/val with 128-bit loads, parks the products
//    and the row ids in shared memory and reduces every run of equal row ids that STARTS in the tile: short runs one thread
//    each, sequentially in storage order with unfused mul/add (bit-identical to opt_crs.cpp:61-67), long runs one warp each
//    (shuffle tree).  The thread that finds a run start also zero-fills the empty rows in front of it (beta = 0).  Runs
//    crossing a tile boundary are finished by a second tiny kernel (short: recomputed sequentially; long: per-tile carries
//    added in tile order -> deterministic).
#include <algorithm>
#include <map>

#include "common.cuh"

namespace b2 {

constexpr int COO_THREADS = 256;
constexpr int COO_IPT = 8;
constexpr int COO_TILE = COO_THREADS * COO_IPT;
constexpr int COO_LONG = 64;
constexpr int COO_MAXLONG = COO_TILE / COO_LONG + 2;

// ACC (the COO tail of HYB, hyb.cu): y already holds the first part of every row's sum; the runs CONTINUE it
// (acc = y[r]; acc += ...; y[r] = acc), nothing is zero-filled, and a short run that crosses into the next tile is left
// entirely to the fix-up kernel (it restarts from the untouched y[r]).
template <bool ACC>
__global__ void __launch_bounds__(COO_THREADS)
coo_tile_kernel(const int *__restrict__ row, const int *__restrict__ col, const double *__restrict__ val,
                const double *__restrict__ x, double *__restrict__ y, double *__restrict__ carry, int nnz, int nRow,
                int vec_ok)
{
    __shared__ __align__(16) double prod[COO_TILE];
    __shared__ __align__(16) int srow[COO_TILE];
    __shared__ unsigned head[COO_TILE / 32 + 1];     // bit i = entry i starts a run of equal row ids
    __shared__ int long_start[COO_MAXLONG];
    __shared__ int n_long;

    const int tid = threadIdx.x, lane = tid & 31;
    const int t = blockIdx.x;
    const int t0 = t * COO_TILE;
    const int n = min(COO_TILE, nnz - t0);
    const uint64_t pol_stream = policy_evict_first(), pol_x = policy_evict_last();
    if (tid == 0) n_long = 0;
    const bool fast = n == COO_TILE && vec_ok;

    if (fast) {
#pragma unroll
        for (int k = 0; k < COO_IPT / 4; k++) {
            const int o = 4 * (tid + k * COO_THREADS);
            const int4 r = ld_stream_i4(row + t0 + o, pol_stream);
            const int4 c = ld_stream_i4(col + t0 + o, pol_stream);
            const double2 v0 = ld_stream_d2(val + t0 + o, pol_stream), v1 = ld_stream_d2(val + t0 + o + 2, pol_stream);
            const double x0 = ld_x(x + c.x, pol_x), x1 = ld_x(x + c.y, pol_x), x2 = ld_x(x + c.z, pol_x), x3 = ld_x(x + c.w, pol_x);
            *reinterpret_cast<int4 *>(srow + o) = r;
            double2 *dst = reinterpret_cast<double2 *>(prod + o);
            dst[0] = make_double2(__dmul_rn(v0.x, x0), __dmul_rn(v0.y, x1));
            dst[1] = make_double2(__dmul_rn(v1.x, x2), __dmul_rn(v1.y, x3));
            // run starts, in registers: the row id in front of this lane's four entries comes from the lane below
            int prev = __shfl_up_sync(0xffffffffu, r.w, 1);
            if (lane == 0) prev = (t0 + o) > 0 ? row[t0 + o - 1] : -1;
            unsigned bits = (unsigned)(r.x != prev) | ((unsigned)(r.y != r.x) << 1) | ((unsigned)(r.z != r.y) << 2) |
                            ((unsigned)(r.w != r.z) << 3);
            bits <<= 4 * (lane & 7);                           // eight lanes share one 32-entry word
            bits |= __shfl_xor_sync(0xffffffffu, bits, 1);
            bits |= __shfl_xor_sync(0xffffffffu, bits, 2);
            bits |= __shfl_xor_sync(0xffffffffu, bits, 4);
            if ((lane & 7) == 0) head[o >> 5] = bits;
        }
    } else {
        for (int i = tid; i < COO_TILE / 32 + 1; i += COO_THREADS) head[i] = 0u;
        for (int i = tid; i < n; i += COO_THREADS) {
            srow[i] = ld_stream_i1(row + t0 + i, pol_stream);
            prod[i] = __dmul_rn(ld_stream_d1(val + t0 + i, pol_stream), ld_x(x + ld_stream_i1(col + t0 + i, pol_stream), pol_x));
        }
    }
    const int prev_row = t0 > 0 ? row[t0 - 1] : -1;
    const bool last_tile = t0 + n == nnz;
    const int next_row = (ACC && !last_tile) ? row[t0 + n] : -1;
    __syncthreads();
    if (!fast) {
        for (int i = tid; i < n; i += COO_THREADS)
            if (srow[i] != (i ? srow[i - 1] : prev_row)) atomicOr(&head[i >> 5], 1u << (i & 31));
        __syncthreads();
    }

    // ---- one thread per run start among its eight consecutive entries (bits come from one shared word)
    const int base = tid * COO_IPT;
    if (base < n) {
        unsigned mine = (head[base >> 5] >> (base & 31)) & 0xFFu;
        while (mine) {
            const int i = base + __ffs(mine) - 1;
            mine &= mine - 1;
            // end of the run = next run start (or the end of the tile)
            int end;
            {
                int w = i >> 5;
                unsigned rest = head[w] & ~((2u << (i & 31)) - 1u);      // bits above i in its word
                while (!rest && (w + 1) * 32 < n) rest = head[++w];
                end = rest ? min(n, w * 32 + __ffs(rest) - 1) : n;
            }
            const int r = srow[i];
            if (!ACC) {
                const int before = i ? srow[i - 1] : prev_row;
                for (int e = before + 1; e < r; e++) y[e] = 0.0;    // empty rows in front of this run (beta = 0)
            }
            if (end - i > COO_LONG) {
                long_start[atomicAdd(&n_long, 1)] = i;
                continue;
            }
            if (ACC && end == n && next_row == r) {
                // the run goes on in the next tile.  At most COO_LONG entries in all: the fix-up recomputes it from the
                // untouched y[r]; longer: this piece is added now and the fix-up adds the carries of the other tiles
                const int probe = t0 + n + (COO_LONG - (n - i));
                if (!(probe < nnz && row[probe] == r)) continue;
            }
            double acc = ACC ? y[r] : 0.0;
            for (int j = i; j < end; j++) acc = __dadd_rn(acc, prod[j]);
            y[r] = acc;       // complete unless the run continues in the next tile (then the fix-up finishes it)
        }
    }
    if (tid == 0 && n > 0 && srow[0] == prev_row) long_start[atomicAdd(&n_long, 1)] = -1;   // carried-in piece
    if (!ACC && last_tile && n > 0)
        for (int e = srow[n - 1] + 1 + tid; e < nRow; e += COO_THREADS) y[e] = 0.0;          // trailing empty rows
    __syncthreads();

    // ---- one warp per long run / carried-in piece
    const int warp = tid >> 5;
    for (int q = warp; q < n_long; q += COO_THREADS / 32) {
        const int s = long_start[q];
        const int b = s < 0 ? 0 : s;
        const int r = srow[b];
        double acc = 0.0;
        for (int k = b + lane; k < n && srow[k] == r; k += 32) acc += prod[k];
        acc = warp_sum(acc);
        if (lane == 0) {
            if (s < 0) carry[t] = acc;
            else y[r] = ACC ? y[r] + acc : acc;
        }
    }
}

// one thread per tile: finishes the row whose entries continue from the previous tile (first carrying tile only)
template <bool ACC>
__global__ void coo_fixup_kernel(const int *__restrict__ row, const int *__restrict__ col, const double *__restrict__ val,
                                 const double *__restrict__ x, double *__restrict__ y, const double *__restrict__ carry,
                                 int nnz, int nTiles)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < 1 || t >= nTiles) return;
    const int t0 = t * COO_TILE;
    const int rc = row[t0];
    if (row[t0 - 1] != rc) return;                              // a run starts exactly at the tile start
    const int p0 = t0 - COO_TILE;                               // previous tile: does the run merely pass through it?
    if (row[p0] == rc && (p0 == 0 ? false : row[p0 - 1] == rc)) return;
    int b = t0, e = t0;
    while (b > 0 && t0 - b <= COO_LONG && row[b - 1] == rc) b--;
    while (e < nnz && e - t0 <= COO_LONG && row[e] == rc) e++;
    const bool whole = (b == 0 || row[b - 1] != rc) && (e == nnz || row[e] != rc);
    if (whole && e - b <= COO_LONG) {
        double acc = ACC ? y[rc] : 0.0;
        for (int j = b; j < e; j++) acc = __dadd_rn(acc, __dmul_rn(val[j], x[col[j]]));
        y[rc] = acc;
    } else {
        double sum = 0.0;
        for (int u = t; u < nTiles && row[u * COO_TILE] == rc; u++) sum += carry[u];
        y[rc] += sum;
    }
}


// ---------------------------------------------------------------------------------------------------------------------
// The entry stream ("coo_stream"): the default COO multiply.  BASELINE.json asks for "COO ... tile segmented reductions
// using warp shuffles"; the tile kernel above parks every product in shared memory and reads it back (MIO-bound, 0.51
// of the roofline on c5).  Here:
//   * persistent CTAs; the 16 B/entry stream (row, col, val) of tile k+1 is brought into shared memory by three 1-D TMA
//     bulk copies while tile k is reduced -- no thread ever waits for matrix data;
//   * a warp owns CS_CHUNK consecutive entries of the tile, 128 at a time: a lane multiplies 4 consecutive entries,
//     reduces the runs of equal row ids that start AND end inside them in registers, and one segmented warp scan
//     (5 shuffle steps) finishes the runs that cross lanes; the open run is carried in a register to the next 128;
//   * a warp writes y for every run that starts AND ends in its chunk (and zero-fills the empty rows in front of each
//     run: beta = 0); after the tile's barrier one thread stitches the chunks -- the leading piece of a chunk belongs to
//     the run open at the end of the chunk before it -- and the tile's own leading piece goes to carry[tile]: the fix-up
//     kernel adds the carries in tile order (deterministic; no atomics, unlike the reference's `omp atomic`,
//     opt_coo.cpp:34-46).
// Sums are re-associated across lanes: y is within the 1e-12 tolerance, not bit-identical to the CRS order (the
// reference's own COO order is not defined either).  options.coo_path = 1 keeps the order-preserving tile kernel.
constexpr int CS_THREADS = 256;
constexpr int CS_WARPS = CS_THREADS / 32;

struct CooChunkRec {            // what a warp reports about its chunk; combined by one thread after the tile's barrier
    double piece;               // sum of the entries in front of the chunk's first run start (the whole chunk if it has none)
    double tail;                // sum of the run still open at the end of the chunk (started here)
    int tailRow;                // its row, -1 if no run starts in the chunk
    int pad;
};

// TMA = true: persistent CTAs, tiles brought in by bulk copies (above).  TMA = false: one tile per CTA, the lanes load their
// entries straight from global memory with 128-bit streaming loads -- for matrices whose x gathers depend on L2 residency
// (R-MAT, uniform random): with bulk copies in flight x does not stay in L2 (profiles/r2_experiments.md), with LDG + evict_first
// it does.
template <int E, bool TMA>
__global__ void __launch_bounds__(CS_THREADS)
coo_stream_kernel(const int *__restrict__ row, const int *__restrict__ col, const double *__restrict__ val,
                  const double *__restrict__ x, double *__restrict__ y, double *__restrict__ carry, int nnz, int nRow,
                  int nTiles)
{
    constexpr int CHUNK = E / CS_WARPS;                       // entries per warp and tile
    constexpr int GROUPS = CHUNK / 128;
    static_assert(GROUPS >= 1, "a warp pass covers 128 entries");
    extern __shared__ __align__(128) unsigned char cs_smem[];
    // full[s]: the bulk copies of stage s have landed.  One CTA barrier per tile hands the stage back to the copy engine; a
    // variant without it (per-warp release through a second mbarrier, the last warp stitching) let the warps drift apart and
    // was 20 % slower on c5 (0.645 against 0.804 of the roofline, profiles/r2_experiments.md)
    __shared__ __align__(8) uint64_t full[2];
    __shared__ CooChunkRec rec[2][CS_WARPS];
    int *srow = reinterpret_cast<int *>(cs_smem);             // [2][E]
    int *scol = srow + 2 * E;                                 // [2][E]
    double *sval = reinterpret_cast<double *>(scol + 2 * E);  // [2][E]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint64_t pol_stream = policy_evict_first(), pol_x = policy_evict_last();

    auto issue = [&](int s, int t) {                          // thread 0 only
        const long long t0 = (long long)t * E;
        const int n = (int)min((long long)E, (long long)nnz - t0);
        const uint32_t b4 = (uint32_t)((n * 4 + 15) & ~15), b8 = (uint32_t)(n * 8 + 15) & ~15u;   // allocations carry slack
        mbar_expect_tx(&full[s], 2 * b4 + b8);
        tma_load_1d(srow + s * E, row + t0, b4, &full[s], pol_stream);
        tma_load_1d(scol + s * E, col + t0, b4, &full[s], pol_stream);
        tma_load_1d(sval + s * E, val + t0, b8, &full[s], pol_stream);
    };
    if (TMA) {
        if (tid == 0) { mbar_init(&full[0], 1); mbar_init(&full[1], 1); }
        __syncthreads();
        if (tid == 0) {
            if ((int)blockIdx.x < nTiles) issue(0, blockIdx.x);
            if ((int)(blockIdx.x + gridDim.x) < nTiles) issue(1, blockIdx.x + gridDim.x);
        }
    }
    // row id in front of a tile (thread 0 keeps it; fetched one tile ahead so that nobody waits for it)
    int tileBefore = -1;
    if (tid == 0 && (int)blockIdx.x < nTiles && blockIdx.x > 0) tileBefore = row[(long long)blockIdx.x * E - 1];
    int k = 0;
    for (int t = blockIdx.x; t < nTiles; t += gridDim.x, k++) {
        const int s = k & 1;
        const long long t0 = (long long)t * E;
        const int n = (int)min((long long)E, (long long)nnz - t0);
        const int c0 = warp * CHUNK;                          // this warp's chunk inside the tile
        const int nGroups = c0 < n ? min(GROUPS, (n - c0 + 127) >> 7) : 0;
        const int nw = min(CS_WARPS, (n + CHUNK - 1) / CHUNK);                      // warps with entries in this tile
        const int tNext = t + gridDim.x;
        int nextBefore = -1;
        if (tid == 0 && tNext < nTiles) nextBefore = row[(long long)tNext * E - 1];
        if (TMA) mbar_wait(&full[s], (uint32_t)(k >> 1) & 1u);
        const int *R = TMA ? srow + s * E : row + t0, *Cc = TMA ? scol + s * E : col + t0;
        const double *V = TMA ? sval + s * E : val + t0;
        if (nGroups > 0) {
            int before = tileBefore;
            if (lane == 0 && warp > 0) before = R[c0 - 1];
            before = __shfl_sync(0xffffffffu, before, 0);
            bool started = false;                             // a run has started in this chunk (else: still the carried-in piece)
            double cin = 0.0;                                 // sum of the open run so far (or of the carried-in piece)
            double piece = 0.0;
            int lastRow = before;
#pragma unroll
            for (int g = 0; g < GROUPS; g++) {
                if (g >= nGroups) break;
                const int e = c0 + g * 128 + 4 * lane;
                int4 r, c;
                double2 v0, v1;
                const bool fullGroup = c0 + g * 128 + 128 <= n;
                if (fullGroup && TMA) {
                    r = *reinterpret_cast<const int4 *>(R + e);
                    c = *reinterpret_cast<const int4 *>(Cc + e);
                    v0 = *reinterpret_cast<const double2 *>(V + e);
                    v1 = *reinterpret_cast<const double2 *>(V + e + 2);
                } else if (fullGroup) {
                    r = ld_stream_i4(R + e, pol_stream);
                    c = ld_stream_i4(Cc + e, pol_stream);
                    v0 = ld_stream_d2(V + e, pol_stream);
                    v1 = ld_stream_d2(V + e + 2, pol_stream);
                } else {                                      // ragged end of the last tile: missing entries repeat the last row with value 0
                    const int last = R[n - 1];
                    r.x = e < n ? R[e] : last; r.y = e + 1 < n ? R[e + 1] : last; r.z = e + 2 < n ? R[e + 2] : last; r.w = e + 3 < n ? R[e + 3] : last;
                    c.x = e < n ? Cc[e] : 0; c.y = e + 1 < n ? Cc[e + 1] : 0; c.z = e + 2 < n ? Cc[e + 2] : 0; c.w = e + 3 < n ? Cc[e + 3] : 0;
                    v0.x = e < n ? V[e] : 0.0; v0.y = e + 1 < n ? V[e + 1] : 0.0; v1.x = e + 2 < n ? V[e + 2] : 0.0; v1.y = e + 3 < n ? V[e + 3] : 0.0;
                }
                const double x0 = ld_x(x + c.x, pol_x), x1 = ld_x(x + c.y, pol_x), x2 = ld_x(x + c.z, pol_x), x3 = ld_x(x + c.w, pol_x);
                double p0 = __dmul_rn(v0.x, x0), p1 = __dmul_rn(v0.y, x1), p2 = __dmul_rn(v1.x, x2), p3 = __dmul_rn(v1.y, x3);
                if (!fullGroup) {                             // a missing entry adds +0.0, not 0 * x[0] (NaN if x[0] is)
                    p0 = e < n ? p0 : 0.0; p1 = e + 1 < n ? p1 : 0.0; p2 = e + 2 < n ? p2 : 0.0; p3 = e + 3 < n ? p3 : 0.0;
                }
                int rprev = __shfl_up_sync(0xffffffffu, r.w, 1);
                if (lane == 0) rprev = lastRow;
                const bool b0 = r.x != rprev, b1 = r.y != r.x, b2 = r.z != r.y, b3 = r.w != r.z;
                const bool has = b0 | b1 | b2 | b3;
                const int nStarts = (int)b0 + (int)b1 + (int)b2 + (int)b3;
                // head = sum of the entries before the lane's first start, acc = sum from its last start on (all four
                // entries if it has none).  Usual case -- at most one start per lane and no empty rows in between (rows are
                // sorted: r.w - rprev counts the rows that begin here) -- without branches; the rest out of line.
                double head, acc;
                if (__any_sync(0xffffffffu, nStarts > 1 || r.w - rprev != nStarts)) {
                    head = 0.0; acc = 0.0;
                    bool seen = false;
                    auto step = [&](bool b, int rp, int rc, double p) {
                        if (b) {
                            if (!seen) head = acc;
                            else y[rp] = __dadd_rn(acc, 0.0); // a run that started and ended in this lane (+ 0.0: see below)
#pragma unroll 1
                            for (int z = rp + 1; z < rc; z++) y[z] = 0.0;  // empty rows in front of the new run (beta = 0)
                            seen = true;
                            acc = p;
                        } else acc = __dadd_rn(acc, p);
                    };
                    step(b0, rprev, r.x, p0); step(b1, r.x, r.y, p1); step(b2, r.y, r.z, p2); step(b3, r.z, r.w, p3);
                } else {
                    // entries in front of the start go to head, the others to acc; adding 0.0 changes nothing
                    const bool f0 = b0, f1 = f0 | b1, f2 = f1 | b2;                 // "a start at or before this entry"
                    head = __dadd_rn(__dadd_rn((has && !f0) ? p0 : 0.0, (has && !f1) ? p1 : 0.0), (has && !f2) ? p2 : 0.0);
                    acc = __dadd_rn(__dadd_rn(__dadd_rn((!has || f0) ? p0 : 0.0, (!has || f1) ? p1 : 0.0), (!has || f2) ? p2 : 0.0), p3);
                }
                // segmented inclusive scan over the lanes: segments begin at lanes that hold a run start
                const unsigned m = __ballot_sync(0xffffffffu, has);
                const unsigned below = m & (0xffffffffu >> (31 - lane));           // starts at or below this lane
                const int seg = below ? 31 - __clz(below) : 0;
                double v = acc;
                // a segment of k lanes needs the steps d < k only: find the longest gap between starts (with a virtual start at
                // lane 0) from the warp-uniform mask -- 7-entry rows (c5) need ONE step, 27-entry rows (c4) three
                unsigned cov = m | 1u;
                cov |= cov << 1;
                int steps = 1;
                if (cov != 0xffffffffu) {
                    cov |= cov << 2; steps = 2;
                    if (cov != 0xffffffffu) {
                        cov |= cov << 4; steps = 3;
                        if (cov != 0xffffffffu) { cov |= cov << 8; steps = cov != 0xffffffffu ? 5 : 4; }
                    }
                }
#pragma unroll
                for (int i = 0; i < 5; i++) {
                    if (i < steps) {
                        const int d = 1 << i;
                        const double u = __shfl_up_sync(0xffffffffu, v, d);
                        if (lane - d >= seg) v = __dadd_rn(v, u);
                    }
                }
                if (!below) v = __dadd_rn(v, cin);                                  // still the run that was open when the group began
                double excl = __shfl_up_sync(0xffffffffu, v, 1);
                if (lane == 0) excl = cin;
                if (has) {
                    // this lane's first start closes the run that was open in front of it
                    const double total = __dadd_rn(excl, head);
                    const bool firstInChunk = !started && !(m & ((1u << lane) - 1u));
                    if (!firstInChunk) y[rprev] = __dadd_rn(total, 0.0);   // + 0.0: a run of -0.0 products (acc = p) gives +0.0
                    else piece = total;                       // continues a run of an earlier chunk (0 if the chunk begins with a start)
                }
                if (!started && m) piece = __shfl_sync(0xffffffffu, piece, __ffs(m) - 1);
                cin = __shfl_sync(0xffffffffu, v, 31);
                lastRow = __shfl_sync(0xffffffffu, r.w, 31);
                started = started || m != 0u;
            }
            // trailing empty rows after the very last entry
            if (t0 + n == nnz && c0 + CHUNK >= n)
                for (int z = lastRow + 1 + lane; z < nRow; z += 32) y[z] = 0.0;
            if (lane == 0) {
                CooChunkRec q;
                q.piece = started ? piece : cin;
                q.tail = cin;
                q.tailRow = started ? lastRow : -1;
                q.pad = 0;
                rec[s][warp] = q;
            }
        }
        // one thread stitches the chunks of the tile: a chunk's leading piece belongs to the run open at the end of the chunk in
        // front of it; the tile's own leading piece goes to carry[t] (fix-up kernel), runs that end inside the tile get their y
        __syncthreads();                                      // every warp is done with stage s, the chunk records are in place
        if (tid == 32) {
            double tilePiece = 0.0, a2 = 0.0;
            int accRow = -1;
            for (int w = 0; w < nw; w++) {
                const CooChunkRec *o = &rec[s][w];
                const double oPiece = o->piece, oTail = o->tail;
                const int oRow = o->tailRow;
                if (accRow >= 0) a2 = __dadd_rn(a2, oPiece);
                else tilePiece = __dadd_rn(tilePiece, oPiece);
                if (oRow >= 0) {
                    if (accRow >= 0) y[accRow] = __dadd_rn(a2, 0.0);
                    accRow = oRow;
                    a2 = oTail;
                }
            }
            if (accRow >= 0) y[accRow] = __dadd_rn(a2, 0.0);
            carry[t] = tilePiece;
        }
        if (TMA && tid == 0 && t + 2 * (int)gridDim.x < nTiles) issue(s, t + 2 * gridDim.x);
        tileBefore = nextBefore;
    }
}

// one thread per tile: adds the leading pieces of the tiles a run passes through to the y of the tile it started in, in tile order
__global__ void coo_stream_fixup_kernel(const int *__restrict__ row, double *__restrict__ y, const double *__restrict__ carry,
                                        int nnz, int tile, int nTiles)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < 1 || c >= nTiles) return;
    const long long c0 = (long long)c * tile;
    const int rc = row[c0];
    if (row[c0 - 1] != rc) return;                            // a run starts exactly at the tile start
    const long long p0 = c0 - tile;                           // the tile in front merely passes the run through: not the first piece
    if (row[p0] == rc && p0 > 0 && row[p0 - 1] == rc) return;
    double sum = 0.0;
    for (int u = c; u < nTiles && row[(long long)u * tile] == rc; u++) sum = __dadd_rn(sum, carry[u]);
    y[rc] = __dadd_rn(y[rc], sum);
}

// entry-stream tiles: 1024 entries TMA-fed (6 CTAs per SM against 3 with 2048; c5 0.85 against 0.74 of the roofline); load-fed,
// a warp's 256 consecutive entries of a 2048 tile (c3 410 against 385 GFLOP/s)
constexpr int COO_E_TMA = 1024, COO_E_LDG = 2048;

struct CooFormat : Format {
    DevBuf<int> row, col;
    DevBuf<double> val, carry;
    int nTiles = 0;
    int path = 0;                                             // 0 = entry stream fed by TMA, 1 = order-preserving tile kernel, 2 = entry stream fed by LDG
    int want = 0;                                             // options.coo_path (0 = choose the feed from the matrix)
    explicit CooFormat(int path_) : want(path_) {}

    int convert(const CooView &A, cudaStream_t s) override
    {
        nRow = A.nRow; nCol = A.nCol; nnz = A.nnz;
        B2_TRY(validate_sorted_coo(A, s));
        // 8 entries of slack: the bulk copies of the last tile are rounded up to 16 bytes
        B2_TRY(row.alloc((size_t)nnz + 8));
        B2_TRY(col.alloc((size_t)nnz + 8));
        B2_TRY(val.alloc((size_t)nnz + 8));
        B2_CUDA(cudaMemsetAsync(row.p + nnz, 0, 8 * sizeof(int), s));
        B2_CUDA(cudaMemsetAsync(col.p + nnz, 0, 8 * sizeof(int), s));
        B2_CUDA(cudaMemsetAsync(val.p + nnz, 0, 8 * sizeof(double), s));
        B2_CUDA(cudaMemcpyAsync(row.p, A.row, sizeof(int) * (size_t)nnz, cudaMemcpyDeviceToDevice, s));   // opt_coo.cpp:14-19
        B2_CUDA(cudaMemcpyAsync(col.p, A.col, sizeof(int) * (size_t)nnz, cudaMemcpyDeviceToDevice, s));
        B2_CUDA(cudaMemcpyAsync(val.p, A.val, sizeof(double) * (size_t)nnz, cudaMemcpyDeviceToDevice, s));
        path = want;
        if (path == 0 || path == 3) {
            // Entry stream: who feeds it?  Banded matrices (stencils: the x entries a tile touches are a few MB that L1 / L2 hold
            // whatever else streams by) take the TMA-fed persistent kernel: c5 607 GFLOP/s against 530 with loads.  Matrices whose
            // gathers range over tens of MB live on x staying in L2, which it does not with bulk copies in flight: c3 (R-MAT) 211
            // GFLOP/s TMA-fed against 410 with the lanes' own evict-first loads (profiles/r2_experiments.md).
            int band = 0;
            if (path == 0) B2_TRY(max_band(A.row, A.col, nnz, A.rowOffset, &band, s));
            path = (path == 0 && gathers_need_l2(band)) ? 2 : 0;
        }
        nTiles = ceil_div(nnz, path == 1 ? COO_TILE : path == 2 ? COO_E_LDG : COO_E_TMA);
        B2_TRY(carry.alloc((size_t)nTiles));
        B2_CUDA(cudaStreamSynchronize(s));
        return B200SPMV_OK;
    }

    int multiply(const double *x, double *y, cudaStream_t s) override
    {
        if (nRow == 0) return B200SPMV_OK;
        if (nTiles == 0) {
            B2_CUDA(cudaMemsetAsync(y, 0, sizeof(double) * (size_t)nRow, s));
            return B200SPMV_OK;
        }
        if (path == 2) return stream_multiply<COO_E_LDG, false>(x, y, s);
        if (path != 1) return stream_multiply<COO_E_TMA, true>(x, y, s);
        coo_tile_kernel<false><<<nTiles, COO_THREADS, 0, s>>>(row.p, col.p, val.p, x, y, carry.p, nnz, nRow, 1);
        B2_KERNEL_CHECK();
        if (nTiles > 1) {
            coo_fixup_kernel<false><<<ceil_div(nTiles, 256), 256, 0, s>>>(row.p, col.p, val.p, x, y, carry.p, nnz, nTiles);
            B2_KERNEL_CHECK();
        }
        return B200SPMV_OK;
    }

    template <int TE, bool TMA> int stream_multiply(const double *x, double *y, cudaStream_t s)
    {
        constexpr size_t smem = TMA ? 32 * (size_t)TE : 0;
        auto kern = coo_stream_kernel<TE, TMA>;
        static std::map<int, int> per_sm;                      // resident CTAs per SM of this instantiation, by device
        static int sms = 0;
        int dev = 0;
        B2_CUDA(cudaGetDevice(&dev));
        if (!sms) B2_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        auto it = per_sm.find(dev);
        if (it == per_sm.end()) {
            B2_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            int n = 0;
            B2_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kern, CS_THREADS, smem));
            if (n < 1) { set_error("COO entry stream: %zu bytes of shared memory do not fit", smem); return B200SPMV_ERR_UNSUPPORTED; }
            it = per_sm.emplace(dev, n).first;
        }
        const int perSm = std::min(it->second, 6);
        const int grid = TMA ? std::min(nTiles, sms * perSm) : nTiles;
        kern<<<grid, CS_THREADS, smem, s>>>(row.p, col.p, val.p, x, y, carry.p, nnz, nRow, nTiles);
        B2_KERNEL_CHECK();
        if (nTiles > 1) {
            coo_stream_fixup_kernel<<<ceil_div(nTiles, 256), 256, 0, s>>>(row.p, y, carry.p, nnz, TE, nTiles);
            B2_KERNEL_CHECK();
        }
        return B200SPMV_OK;
    }

    bool scalar(const std::string &n, long long *out) override
    {
        if (n == "alg_bytes") {   // SURVEY.md 8d: 16 nnz + 8 nCol + 8 nRow
            *out = 16LL * nnz + 8LL * nCol + 8LL * nRow;
            return true;
        }
        if (n == "launches") { *out = nTiles > 1 ? 2 : 1; return true; }
        if (n == "nTiles") { *out = nTiles; return true; }
        if (n == "coo_path") { *out = path; return true; }
        return false;
    }

    long long array(const std::string &n, void *dst, long long cap) override
    {
        if (n == "row_idx") return export_device(row.p, sizeof(int) * (size_t)nnz, dst, cap);
        if (n == "col_idx") return export_device(col.p, sizeof(int) * (size_t)nnz, dst, cap);
        if (n == "val") return export_device(val.p, sizeof(double) * (size_t)nnz, dst, cap);
        return -1000;
    }
};

Format *make_coo(const b200spmv_options &o) { return new CooFormat(o.coo_path); }

// y[r] continues with the sorted triplets' products, run by run (HYB's COO tail, hyb.cu); carry: ceil(nnz / COO_TILE) doubles
int coo_accumulate(const int *row, const int *col, const double *val, int nnz, int nRow, const double *x, double *y,
                   double *carry, cudaStream_t s)
{
    if (nnz == 0) return B200SPMV_OK;
    const int nTiles = ceil_div(nnz, COO_TILE);
    const int vec_ok = ((reinterpret_cast<uintptr_t>(row) | reinterpret_cast<uintptr_t>(col) | reinterpret_cast<uintptr_t>(val)) & 15) == 0;
    coo_tile_kernel<true><<<nTiles, COO_THREADS, 0, s>>>(row, col, val, x, y, carry, nnz, nRow, vec_ok);
    B2_KERNEL_CHECK();
    if (nTiles > 1) {
        coo_fixup_kernel<true><<<ceil_div(nTiles, 256), 256, 0, s>>>(row, col, val, x, y, carry, nnz, nTiles);
        B2_KERNEL_CHECK();
    }
    return B200SPMV_OK;
}
int coo_tile_entries() { return COO_TILE; }

}  // namespace b2
