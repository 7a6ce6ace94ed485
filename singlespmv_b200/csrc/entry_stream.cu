// entry_stream.cu -- kernels and launcher of the CRS entry stream (see entry_stream.cuh).
#include <algorithm>

#include "entry_stream.cuh"

namespace b2 {

constexpr int ES_THREADS = 256;
constexpr int ES_WARPS = ES_THREADS / 32;

// ---------------------------------------------------------------- conversion: row_ptr -> start bits, run counts, row lists
__global__ void es_bits_kernel(const int *__restrict__ ptr, int nRow, unsigned *__restrict__ bits, int *__restrict__ empty,
                               int *__restrict__ nEmpty)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nRow) return;
    const int b = ptr[r], e = ptr[r + 1];
    if (e > b) atomicOr(&bits[b >> 5], 1u << (b & 31));
    else if (empty) empty[atomicAdd(nEmpty, 1)] = r;
}
__global__ void es_empty_count_kernel(const int *__restrict__ ptr, int nRow, int *__restrict__ nEmpty)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    int c = (r < nRow && ptr[r + 1] == ptr[r]) ? 1 : 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(nEmpty, c);
}
// cnt[g] = row starts among entries [128 g, 128 g + 128); cnt[nGroups] = 0 (scan sentinel)
__global__ void es_group_count_kernel(const unsigned *__restrict__ bits, int nGroups, int *__restrict__ cnt)
{
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g > nGroups) return;
    int c = 0;
    if (g < nGroups) {
        const uint4 w = *reinterpret_cast<const uint4 *>(bits + 4 * (size_t)g);
        c = __popc(w.x) + __popc(w.y) + __popc(w.z) + __popc(w.w);
    }
    cnt[g] = c;
}
// nzrow[k] = the k-th non-empty row (k = number of row starts in front of its first entry)
__global__ void es_nzrow_kernel(const int *__restrict__ ptr, int nRow, const unsigned *__restrict__ bits,
                                const int *__restrict__ grpRun, int *__restrict__ nzrow)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nRow) return;
    const int p = ptr[r];
    if (ptr[r + 1] == p) return;
    const int g = p >> 7;
    int k = grpRun[g];
    for (int w = 4 * g; w < (p >> 5); w++) k += __popc(bits[w]);
    k += __popc(bits[p >> 5] & ((1u << (p & 31)) - 1u));
    nzrow[k] = r;
}
__global__ void es_zero_rows_kernel(const int *__restrict__ rows, int n, int rowLo, int rowHi, double *__restrict__ y)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int r = rows[i];
    if (r >= rowLo && r < rowHi) y[r] = 0.0;
}

// ---------------------------------------------------------------- multiply
struct EsChunkRec {
    double piece, tail;         // sum in front of the chunk's first row start (whole chunk if none); sum of the run open at its end
    int tailRun, pad;           // that run's index, -1 if no row starts in the chunk
};

// TMA = true: persistent CTAs, (idx, val) of tile k+1 arriving by two bulk copies while tile k is reduced.
// TMA = false: one tile per CTA, the lanes load their entries themselves (gather-bound matrices: x must stay in L2).
template <bool TMA>
__global__ void __launch_bounds__(ES_THREADS)
entry_stream_kernel(const int *__restrict__ idx, const double *__restrict__ val, const unsigned *__restrict__ bits,
                    const int *__restrict__ grpRun, const int *__restrict__ nzrow, const double *__restrict__ x,
                    double *__restrict__ y, double *__restrict__ carry, int nnz, int tileLo, int tileHi, int rowLo, int rowHi)
{
    constexpr int E = ES_E;
    constexpr int CHUNK = E / ES_WARPS;
    constexpr int GROUPS = CHUNK / 128;
    static_assert(GROUPS >= 1, "a warp pass covers 128 entries");
    extern __shared__ __align__(128) unsigned char es_smem[];
    __shared__ __align__(8) uint64_t full[2];
    __shared__ EsChunkRec rec[2][ES_WARPS];
    int *scol = reinterpret_cast<int *>(es_smem);                       // [2][E]
    double *sval = reinterpret_cast<double *>(es_smem + 2 * E * sizeof(int));   // [2][E]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint64_t pol_stream = policy_evict_first(), pol_x = policy_evict_last();
    const unsigned lt = (1u << lane) - 1u;

    // y of the run-th non-empty row, if the caller asked for that row.  + 0.0 turns a sum of -0.0 products (a run that
    // starts with acc = p) into +0.0, as the reference's sum from +0.0 gives; it changes no other value
    auto store = [&](int run, double v) {
        const int r = nzrow ? nzrow[run] : run;
        if (r >= rowLo && r < rowHi) y[r] = __dadd_rn(v, 0.0);
    };
    auto issue = [&](int s, int t) {                        // thread 0 only
        const long long t0 = (long long)t * E;
        const int n = (int)min((long long)E, (long long)nnz - t0);
        const uint32_t b4 = (uint32_t)((n * 4 + 15) & ~15), b8 = (uint32_t)(n * 8 + 15) & ~15u;   // the arrays carry slack
        mbar_expect_tx(&full[s], b4 + b8);
        tma_load_1d(scol + s * E, idx + t0, b4, &full[s], pol_stream);
        tma_load_1d(sval + s * E, val + t0, b8, &full[s], pol_stream);
    };
    const int first = tileLo + blockIdx.x;
    if (TMA) {
        if (tid == 0) { mbar_init(&full[0], 1); mbar_init(&full[1], 1); }
        __syncthreads();
        if (tid == 0) {
            if (first < tileHi) issue(0, first);
            if (first + (int)gridDim.x < tileHi) issue(1, first + gridDim.x);
        }
    }
    int k = 0;
    for (int t = first; t < tileHi; t += gridDim.x, k++) {
        const int s = k & 1;
        const long long t0 = (long long)t * E;
        const int n = (int)min((long long)E, (long long)nnz - t0);
        const int c0 = warp * CHUNK;
        const int nGroups = c0 < n ? min(GROUPS, (n - c0 + 127) >> 7) : 0;
        const int nw = min(ES_WARPS, (n + CHUNK - 1) / CHUNK);
        if (TMA) mbar_wait(&full[s], (uint32_t)(k >> 1) & 1u);
        const int *Cc = TMA ? scol + s * E : idx + t0;
        const double *V = TMA ? sval + s * E : val + t0;
        if (nGroups > 0) {
            bool started = false;                           // a row has started in this chunk
            double cin = 0.0, piece = 0.0;
            int lastRun = -1;
#pragma unroll
            for (int g = 0; g < GROUPS; g++) {
                if (g >= nGroups) break;
                const int e = c0 + g * 128 + 4 * lane;
                const long long ge = t0 + e;                // global entry index of the lane's first entry
                int4 c;
                double2 v0, v1;
                const bool full = c0 + g * 128 + 128 <= n;
                if (full) {
                    if (TMA) {
                        c = *reinterpret_cast<const int4 *>(Cc + e);
                        v0 = *reinterpret_cast<const double2 *>(V + e);
                        v1 = *reinterpret_cast<const double2 *>(V + e + 2);
                    } else {
                        c = ld_stream_i4(Cc + e, pol_stream);
                        v0 = ld_stream_d2(V + e, pol_stream);
                        v1 = ld_stream_d2(V + e + 2, pol_stream);
                    }
                } else {                                    // ragged end of the last tile: missing entries are zeros of the open row
                    c.x = e < n ? Cc[e] : 0; c.y = e + 1 < n ? Cc[e + 1] : 0; c.z = e + 2 < n ? Cc[e + 2] : 0; c.w = e + 3 < n ? Cc[e + 3] : 0;
                    v0.x = e < n ? V[e] : 0.0; v0.y = e + 1 < n ? V[e + 1] : 0.0; v1.x = e + 2 < n ? V[e + 2] : 0.0; v1.y = e + 3 < n ? V[e + 3] : 0.0;
                }
                const unsigned word = __ldg(bits + (ge >> 5));                  // beyond nnz the bits are zero
                const unsigned b = (word >> (unsigned)(ge & 31)) & 0xFu;
                const int base = __ldg(grpRun + (ge >> 7));                     // row starts in front of the group
                const double x0 = ld_x(x + c.x, pol_x), x1 = ld_x(x + c.y, pol_x), x2 = ld_x(x + c.z, pol_x), x3 = ld_x(x + c.w, pol_x);
                double p0 = __dmul_rn(v0.x, x0), p1 = __dmul_rn(v0.y, x1), p2 = __dmul_rn(v1.x, x2), p3 = __dmul_rn(v1.y, x3);
                if (!full) {                                // a missing entry adds +0.0, not 0 * x[0] (NaN if x[0] is)
                    p0 = e < n ? p0 : 0.0; p1 = e + 1 < n ? p1 : 0.0; p2 = e + 2 < n ? p2 : 0.0; p3 = e + 3 < n ? p3 : 0.0;
                }
                const bool b0 = b & 1u, b1 = b & 2u, b2 = b & 4u, b3 = b & 8u;
                const bool has = b != 0u;
                const int nStarts = __popc(b);
                // starts in the lower lanes of the group -> index of the run that is open in front of this lane's entries
                const unsigned m = __ballot_sync(0xffffffffu, has);             // lanes that hold a start
                int runOpen = base - 1 + __popc(m & lt);                        // right when no lane holds two starts
                // head = sum of the entries before the lane's first start, acc = sum from its last start on
                double head, acc;
                if (__any_sync(0xffffffffu, nStarts > 1)) {
                    const unsigned m0 = __ballot_sync(0xffffffffu, b0), m1 = __ballot_sync(0xffffffffu, b1),
                                   m2 = __ballot_sync(0xffffffffu, b2), m3 = __ballot_sync(0xffffffffu, b3);
                    runOpen = base - 1 + __popc(m0 & lt) + __popc(m1 & lt) + __popc(m2 & lt) + __popc(m3 & lt);
                    head = 0.0; acc = 0.0;
                    bool seen = false;
                    int run = runOpen;
                    auto step = [&](bool st, double p) {
                        if (st) {
                            if (!seen) head = acc;
                            else store(run, acc);           // a row that begins and ends inside this lane
                            seen = true;
                            run++;
                            acc = p;
                        } else acc = __dadd_rn(acc, p);
                    };
                    step(b0, p0); step(b1, p1); step(b2, p2); step(b3, p3);
                } else {
                    const bool f0 = b0, f1 = f0 | b1, f2 = f1 | b2;             // "a start at or before this entry"
                    head = __dadd_rn(__dadd_rn((has && !f0) ? p0 : 0.0, (has && !f1) ? p1 : 0.0), (has && !f2) ? p2 : 0.0);
                    acc = __dadd_rn(__dadd_rn(__dadd_rn((!has || f0) ? p0 : 0.0, (!has || f1) ? p1 : 0.0), (!has || f2) ? p2 : 0.0), p3);
                }
                // segmented inclusive scan over the lanes: segments begin at lanes that hold a start
                const unsigned below = m & (0xffffffffu >> (31 - lane));
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
                if (!below) v = __dadd_rn(v, cin);
                double excl = __shfl_up_sync(0xffffffffu, v, 1);
                if (lane == 0) excl = cin;
                if (has) {
                    const double total = __dadd_rn(excl, head);                 // the run that was open in front of this lane ends here
                    const bool firstInChunk = !started && !(m & lt);
                    if (!firstInChunk) store(runOpen, total);
                    else piece = total;                     // continues a row of an earlier chunk (0 if the chunk begins with a start)
                }
                if (!started && m) piece = __shfl_sync(0xffffffffu, piece, __ffs(m) - 1);
                cin = __shfl_sync(0xffffffffu, v, 31);
                lastRun = __shfl_sync(0xffffffffu, runOpen + nStarts, 31);
                started = started || m != 0u;
            }
            if (lane == 0) {
                EsChunkRec q;
                q.piece = started ? piece : cin;
                q.tail = cin;
                q.tailRun = started ? lastRun : -1;
                q.pad = 0;
                rec[s][warp] = q;
            }
        }
        __syncthreads();                                    // every warp is done with stage s, the chunk records are in place
        if (tid == 32) {
            double tilePiece = 0.0, a2 = 0.0;
            int accRun = -1;
            for (int w = 0; w < nw; w++) {
                const EsChunkRec *o = &rec[s][w];
                const double oPiece = o->piece, oTail = o->tail;
                const int oRun = o->tailRun;
                if (accRun >= 0) a2 = __dadd_rn(a2, oPiece);
                else tilePiece = __dadd_rn(tilePiece, oPiece);
                if (oRun >= 0) {
                    if (accRun >= 0) store(accRun, a2);
                    accRun = oRun;
                    a2 = oTail;
                }
            }
            if (accRun >= 0) store(accRun, a2);
            carry[t] = tilePiece;
        }
        if (TMA && tid == 0 && t + 2 * (int)gridDim.x < tileHi) issue(s, t + 2 * gridDim.x);
    }
}

// one thread per tile: a row that runs through several tiles gets their leading pieces added, in tile order
__global__ void entry_stream_fixup_kernel(const unsigned *__restrict__ bits, const int *__restrict__ grpRun,
                                          const int *__restrict__ nzrow, double *__restrict__ y, const double *__restrict__ carry,
                                          int E, int tileLo, int tileHi, int rowLo, int rowHi)
{
    const int t = tileLo + 1 + blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= tileHi) return;
    auto first_bit = [&](int u) { const long long e = (long long)u * E; return (bits[e >> 5] >> (unsigned)(e & 31)) & 1u; };
    auto run_at = [&](int u) { return grpRun[((long long)u * E) >> 7] - 1 + (int)first_bit(u); };   // run of the tile's first entry
    if (first_bit(t)) return;                               // a row begins exactly at the tile start
    const int run = run_at(t);
    if (!first_bit(t - 1) && run_at(t - 1) == run) return;  // the tile in front merely passes the row through: not the first piece
    double sum = 0.0;
    for (int u = t; u < tileHi && !first_bit(u) && run_at(u) == run; u++) sum = __dadd_rn(sum, carry[u]);
    const int r = nzrow ? nzrow[run] : run;
    if (r >= rowLo && r < rowHi) y[r] = __dadd_rn(y[r], sum);
}

// the values of a lane's 4 entries of a full group: from the stage (TMA) or by streaming loads
template <bool TMA>
__device__ __forceinline__ void es_vals4(double (&a)[4], const double *V, uint64_t pol)
{
    double2 v0, v1;
    if (TMA) {
        v0 = *reinterpret_cast<const double2 *>(V);
        v1 = *reinterpret_cast<const double2 *>(V + 2);
    } else {
        v0 = ld_stream_d2(V, pol);
        v1 = ld_stream_d2(V + 2, pol);
    }
    a[0] = v0.x; a[1] = v0.y; a[2] = v1.x; a[3] = v1.y;
}
template <bool TMA>
__device__ __forceinline__ void es_vals4(float (&a)[4], const float *V, uint64_t pol)
{
    const float4 v = TMA ? *reinterpret_cast<const float4 *>(V) : ld_stream_f4(V, pol);
    a[0] = v.x; a[1] = v.y; a[2] = v.z; a[3] = v.w;
}

// ---------------------------------------------------------------- multiply of k <= ES_KMAX vectors (X, Y row-major)
// The kernel above with every sum carried for KP vectors at once: the entry stream, start bits, ballots and scans are
// shared, the lane gathers the KP values of a column in one row of X (ld_xrow).  k > KP: the tile is reduced once per
// group of KP vectors (TMA-fed from the same stage, load-fed from L2).  Carries: carry[t * k + j].
// VT = stored value type, XT = type of X and Y, AT = type of products and sums (fp32 vectors: fp32 or fp64).  With fp32 Y
// (TAIL) the row still open at the end of a tile is not stored: its partial goes to the tile's tail slot carry[(nT + t) * k
// + j] in AT, and the fix-up writes that row once -- so a precision-2 row is rounded to fp32 once, after every carry.
template <typename VT, typename XT, typename AT, bool TMA, int KP, bool VEC>
__global__ void __launch_bounds__(ES_THREADS)
entry_stream_multi_kernel(const int *__restrict__ idx, const VT *__restrict__ val, const unsigned *__restrict__ bits,
                          const int *__restrict__ grpRun, const int *__restrict__ nzrow, const XT *__restrict__ X,
                          long long ldx, XT *__restrict__ Y, long long ldy, int kv, AT *__restrict__ carry, int nnz,
                          int tileLo, int tileHi, int rowLo, int rowHi)
{
    constexpr bool TAIL = sizeof(XT) == 4;
    constexpr int E = ES_E;
    constexpr int CHUNK = E / ES_WARPS;
    constexpr int GROUPS = CHUNK / 128;
    extern __shared__ __align__(128) unsigned char es_smem[];
    __shared__ __align__(8) uint64_t full[2];
    __shared__ AT rPiece[ES_WARPS][ES_KMAX], rTail[ES_WARPS][ES_KMAX];
    __shared__ int rRun[ES_WARPS];
    int *scol = reinterpret_cast<int *>(es_smem);
    VT *sval = reinterpret_cast<VT *>(es_smem + 2 * E * sizeof(int));
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint64_t pol_stream = policy_evict_first(), pol_x = policy_evict_last();
    const unsigned lt = (1u << lane) - 1u;

    auto row_of = [&](int run) { return nzrow ? nzrow[run] : run; };
    auto store = [&](int run, int j0, const AT (&a)[KP]) {
        const int r = row_of(run);
        if (r >= rowLo && r < rowHi) {
            XT *yr = Y + (long long)r * ldy + j0;
#pragma unroll
            for (int v = 0; v < KP; v++)
                if (j0 + v < kv) yr[v] = (XT)Arith<AT>::add(a[v], (AT)0);   // + 0: a sum of -0.0 products is +0.0 (store above)
        }
    };
    auto issue = [&](int s, int t) {
        const long long t0 = (long long)t * E;
        const int n = (int)min((long long)E, (long long)nnz - t0);
        const uint32_t b4 = (uint32_t)((n * 4 + 15) & ~15), b8 = (uint32_t)(n * (int)sizeof(VT) + 15) & ~15u;
        mbar_expect_tx(&full[s], b4 + b8);
        tma_load_1d(scol + s * E, idx + t0, b4, &full[s], pol_stream);
        tma_load_1d(sval + s * E, val + t0, b8, &full[s], pol_stream);
    };
    const int first = tileLo + blockIdx.x;
    if (TMA) {
        if (tid == 0) { mbar_init(&full[0], 1); mbar_init(&full[1], 1); }
        __syncthreads();
        if (tid == 0) {
            if (first < tileHi) issue(0, first);
            if (first + (int)gridDim.x < tileHi) issue(1, first + gridDim.x);
        }
    }
    int k = 0;
    for (int t = first; t < tileHi; t += gridDim.x, k++) {
        const int s = k & 1;
        const long long t0 = (long long)t * E;
        const int n = (int)min((long long)E, (long long)nnz - t0);
        const int c0 = warp * CHUNK;
        const int nGroups = c0 < n ? min(GROUPS, (n - c0 + 127) >> 7) : 0;
        const int nw = min(ES_WARPS, (n + CHUNK - 1) / CHUNK);
        if (TMA) mbar_wait(&full[s], (uint32_t)(k >> 1) & 1u);
        const int *Cc = TMA ? scol + s * E : idx + t0;
        const VT *V = TMA ? sval + s * E : val + t0;
        for (int j0 = 0; j0 < kv && nGroups > 0; j0 += KP) {
            bool started = false;
            AT cin[KP], piece[KP];
#pragma unroll
            for (int v = 0; v < KP; v++) cin[v] = piece[v] = (AT)0;
            int lastRun = -1;
#pragma unroll
            for (int g = 0; g < GROUPS; g++) {
                if (g >= nGroups) break;
                const int e = c0 + g * 128 + 4 * lane;
                const long long ge = t0 + e;
                int4 c;
                VT a[4];
                const bool full = c0 + g * 128 + 128 <= n;
                if (full) {
                    if (TMA) c = *reinterpret_cast<const int4 *>(Cc + e);
                    else c = ld_stream_i4(Cc + e, pol_stream);
                    es_vals4<TMA>(a, V + e, pol_stream);
                } else {
                    c.x = e < n ? Cc[e] : 0; c.y = e + 1 < n ? Cc[e + 1] : 0; c.z = e + 2 < n ? Cc[e + 2] : 0; c.w = e + 3 < n ? Cc[e + 3] : 0;
                    a[0] = e < n ? V[e] : (VT)0; a[1] = e + 1 < n ? V[e + 1] : (VT)0; a[2] = e + 2 < n ? V[e + 2] : (VT)0; a[3] = e + 3 < n ? V[e + 3] : (VT)0;
                }
                const unsigned word = __ldg(bits + (ge >> 5));
                const unsigned b = (word >> (unsigned)(ge & 31)) & 0xFu;
                const int base = __ldg(grpRun + (ge >> 7));
                XT x0[KP], x1[KP], x2[KP], x3[KP];
                ld_xrow<KP, VEC>(x0, X + (long long)c.x * ldx + j0, kv - j0, pol_x);
                ld_xrow<KP, VEC>(x1, X + (long long)c.y * ldx + j0, kv - j0, pol_x);
                ld_xrow<KP, VEC>(x2, X + (long long)c.z * ldx + j0, kv - j0, pol_x);
                ld_xrow<KP, VEC>(x3, X + (long long)c.w * ldx + j0, kv - j0, pol_x);
                AT p0[KP], p1[KP], p2[KP], p3[KP];
#pragma unroll
                for (int v = 0; v < KP; v++) {
                    p0[v] = Arith<AT>::mul((AT)a[0], (AT)x0[v]); p1[v] = Arith<AT>::mul((AT)a[1], (AT)x1[v]);
                    p2[v] = Arith<AT>::mul((AT)a[2], (AT)x2[v]); p3[v] = Arith<AT>::mul((AT)a[3], (AT)x3[v]);
                }
                if (!full) {                                    // a missing entry adds +0.0, not 0 * X[0, j]
#pragma unroll
                    for (int v = 0; v < KP; v++) {
                        p0[v] = e < n ? p0[v] : (AT)0; p1[v] = e + 1 < n ? p1[v] : (AT)0;
                        p2[v] = e + 2 < n ? p2[v] : (AT)0; p3[v] = e + 3 < n ? p3[v] : (AT)0;
                    }
                }
                const bool b0 = b & 1u, b1 = b & 2u, b2 = b & 4u, b3 = b & 8u;
                const bool has = b != 0u;
                const int nStarts = __popc(b);
                const unsigned m = __ballot_sync(0xffffffffu, has);
                int runOpen = base - 1 + __popc(m & lt);
                AT head[KP], acc[KP];
                if (__any_sync(0xffffffffu, nStarts > 1)) {
                    const unsigned m0 = __ballot_sync(0xffffffffu, b0), m1 = __ballot_sync(0xffffffffu, b1),
                                   m2 = __ballot_sync(0xffffffffu, b2), m3 = __ballot_sync(0xffffffffu, b3);
                    runOpen = base - 1 + __popc(m0 & lt) + __popc(m1 & lt) + __popc(m2 & lt) + __popc(m3 & lt);
#pragma unroll
                    for (int v = 0; v < KP; v++) head[v] = acc[v] = (AT)0;
                    bool seen = false;
                    int run = runOpen;
                    auto step = [&](bool st, const AT (&p)[KP]) {
                        if (st) {
                            if (!seen) {
#pragma unroll
                                for (int v = 0; v < KP; v++) head[v] = acc[v];
                            } else {
                                store(run, j0, acc);
                            }
                            seen = true;
                            run++;
#pragma unroll
                            for (int v = 0; v < KP; v++) acc[v] = p[v];
                        } else {
#pragma unroll
                            for (int v = 0; v < KP; v++) acc[v] = Arith<AT>::add(acc[v], p[v]);
                        }
                    };
                    step(b0, p0); step(b1, p1); step(b2, p2); step(b3, p3);
                } else {
                    const bool f0 = b0, f1 = f0 | b1, f2 = f1 | b2;
#pragma unroll
                    for (int v = 0; v < KP; v++) {
                        head[v] = Arith<AT>::add(Arith<AT>::add((has && !f0) ? p0[v] : (AT)0, (has && !f1) ? p1[v] : (AT)0), (has && !f2) ? p2[v] : (AT)0);
                        acc[v] = Arith<AT>::add(Arith<AT>::add(Arith<AT>::add((!has || f0) ? p0[v] : (AT)0, (!has || f1) ? p1[v] : (AT)0), (!has || f2) ? p2[v] : (AT)0), p3[v]);
                    }
                }
                const unsigned below = m & (0xffffffffu >> (31 - lane));
                const int seg = below ? 31 - __clz(below) : 0;
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
                AT sc[KP];                                      // the segmented scan, per vector
#pragma unroll
                for (int v = 0; v < KP; v++) sc[v] = acc[v];
#pragma unroll
                for (int i = 0; i < 5; i++) {
                    if (i < steps) {
                        const int d = 1 << i;
#pragma unroll
                        for (int v = 0; v < KP; v++) {
                            const AT u = __shfl_up_sync(0xffffffffu, sc[v], d);
                            if (lane - d >= seg) sc[v] = Arith<AT>::add(sc[v], u);
                        }
                    }
                }
                const bool firstInChunk = !started && !(m & lt);
                AT tot[KP];
#pragma unroll
                for (int v = 0; v < KP; v++) {
                    if (!below) sc[v] = Arith<AT>::add(sc[v], cin[v]);
                    AT excl = __shfl_up_sync(0xffffffffu, sc[v], 1);
                    if (lane == 0) excl = cin[v];
                    tot[v] = Arith<AT>::add(excl, head[v]);
                    if (has && firstInChunk) piece[v] = tot[v];
                }
                if (has && !firstInChunk) store(runOpen, j0, tot);
#pragma unroll
                for (int v = 0; v < KP; v++) {
                    if (!started && m) piece[v] = __shfl_sync(0xffffffffu, piece[v], __ffs(m) - 1);
                    cin[v] = __shfl_sync(0xffffffffu, sc[v], 31);
                }
                lastRun = __shfl_sync(0xffffffffu, runOpen + nStarts, 31);
                started = started || m != 0u;
            }
            if (lane == 0) {
#pragma unroll
                for (int v = 0; v < KP; v++)
                    if (j0 + v < kv) {
                        rPiece[warp][j0 + v] = started ? piece[v] : cin[v];
                        rTail[warp][j0 + v] = cin[v];
                    }
                rRun[warp] = started ? lastRun : -1;
            }
        }
        __syncthreads();                                    // every warp is done with stage s, the chunk records are in place
        if (tid >= 32 && tid < 32 + kv) {                   // one thread per vector stitches the chunks of the tile
            const int j = tid - 32;
            AT tilePiece = (AT)0, a2 = (AT)0;
            int accRun = -1;
            auto put = [&](int run, AT v) {
                const int r = row_of(run);
                if (r >= rowLo && r < rowHi) Y[(long long)r * ldy + j] = (XT)Arith<AT>::add(v, (AT)0);
            };
            for (int w = 0; w < nw; w++) {
                const AT oPiece = rPiece[w][j], oTail = rTail[w][j];
                const int oRun = rRun[w];
                if (accRun >= 0) a2 = Arith<AT>::add(a2, oPiece);
                else tilePiece = Arith<AT>::add(tilePiece, oPiece);
                if (oRun >= 0) {
                    if (accRun >= 0) put(accRun, a2);
                    accRun = oRun;
                    a2 = oTail;
                }
            }
            if (TAIL && accRun >= 0 && t + 1 < tileHi && !((bits[((long long)(t + 1) * E) >> 5] >> (unsigned)(((long long)(t + 1) * E) & 31)) & 1u))
                carry[((long long)tileHi + t) * kv + j] = a2;       // the row goes on in tile t + 1: the fix-up stores it
            else if (accRun >= 0) put(accRun, a2);
            carry[(long long)t * kv + j] = tilePiece;
        }
        __syncthreads();                                    // the records are read before the next tile's warps rewrite them
        if (TMA && tid == 0 && t + 2 * (int)gridDim.x < tileHi) issue(s, t + 2 * gridDim.x);
    }
}

// one thread per (tile, vector): entry_stream_fixup_kernel on column j of Y.  TAIL (fp32 Y): the row's partial from the
// tile in front comes from that tile's tail slot, and Y is written once.
template <typename XT, typename AT>
__global__ void entry_stream_multi_fixup_kernel(const unsigned *__restrict__ bits, const int *__restrict__ grpRun,
                                                const int *__restrict__ nzrow, XT *__restrict__ Y, long long ldy, int kv,
                                                const AT *__restrict__ carry, int E, int tileLo, int tileHi)
{
    constexpr bool TAIL = sizeof(XT) == 4;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int t = tileLo + 1 + (int)(i / kv), j = (int)(i % kv);
    if (t >= tileHi) return;
    auto first_bit = [&](int u) { const long long e = (long long)u * E; return (bits[e >> 5] >> (unsigned)(e & 31)) & 1u; };
    auto run_at = [&](int u) { return grpRun[((long long)u * E) >> 7] - 1 + (int)first_bit(u); };
    if (first_bit(t)) return;
    const int run = run_at(t);
    if (!first_bit(t - 1) && run_at(t - 1) == run) return;
    AT sum = (AT)0;
    for (int u = t; u < tileHi && !first_bit(u) && run_at(u) == run; u++) sum = Arith<AT>::add(sum, carry[(long long)u * kv + j]);
    XT *yr = Y + (long long)(nzrow ? nzrow[run] : run) * ldy + j;
    if (TAIL) *yr = (XT)Arith<AT>::add(carry[((long long)tileHi + t - 1) * kv + j], sum);
    else *yr = Arith<AT>::add(*yr, sum);
}

// Y[r, j] = 0 for the listed rows (all rows [0, n) when rows == NULL) and j < k
template <typename XT>
__global__ void es_zero_rows_multi_kernel(const int *__restrict__ rows, int n, int kv, XT *__restrict__ Y, long long ldy)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)n * kv) return;
    const int q = (int)(i / kv);
    Y[(long long)(rows ? rows[q] : q) * ldy + (int)(i % kv)] = (XT)0;
}

template <typename XT>
static int zero_rows_multi_t(int nRow, int k, XT *Y, long long ldy, cudaStream_t s)
{
    if (nRow <= 0) return B200SPMV_OK;
    es_zero_rows_multi_kernel<<<ceil_div((long long)nRow * k, 256), 256, 0, s>>>(nullptr, nRow, k, Y, ldy);
    B2_KERNEL_CHECK();
    return B200SPMV_OK;
}
int zero_rows_multi(int nRow, int k, double *Y, long long ldy, cudaStream_t s) { return zero_rows_multi_t(nRow, k, Y, ldy, s); }
int zero_rows_multi(int nRow, int k, float *Y, long long ldy, cudaStream_t s) { return zero_rows_multi_t(nRow, k, Y, ldy, s); }

void EntryStream::reset()
{
    ptr = idx = nullptr;
    val = nullptr;
    f32 = false;
    nRow = nnz = 0;
    ok = tma = false;
    nTiles = nEmpty = 0;
    bits.release();
    grpRun.release();
    nzrow.release();
    empty.release();
    carry.release();
    carryK.release();
    range_cache.clear();
}

int EntryStream::build(const int *ptr_d, const int *idx_d, const void *val_d, bool val_is_f32, int nRow_, int nnz_,
                       bool gather_bound, cudaStream_t s)
{
    reset();
    ptr = ptr_d; idx = idx_d; val = val_d; f32 = val_is_f32; nRow = nRow_; nnz = nnz_;
    if (nnz <= 0 || nRow <= 0) return B200SPMV_OK;
    tma = !gather_bound;
    nTiles = ceil_div(nnz, ES_E);
    const int nGroups = ceil_div((long long)nTiles * ES_E, 128);
    B2_TRY(bits.alloc((size_t)nGroups * 4 + 4));
    B2_TRY(grpRun.alloc((size_t)nGroups + 1));
    if (!f32) B2_TRY(carry.alloc((size_t)nTiles));         // run_rows (fp64 only) owns these; run_multi* use carryK
    B2_CUDA(cudaMemsetAsync(bits.p, 0, bits.bytes(), s));
    DevBuf<int> cnt;
    B2_TRY(cnt.alloc(1));
    B2_CUDA(cudaMemsetAsync(cnt.p, 0, sizeof(int), s));
    es_empty_count_kernel<<<ceil_div(nRow, 256), 256, 0, s>>>(ptr, nRow, cnt.p);
    B2_KERNEL_CHECK();
    B2_CUDA(cudaMemcpyAsync(&nEmpty, cnt.p, sizeof(int), cudaMemcpyDeviceToHost, s));
    B2_CUDA(cudaStreamSynchronize(s));
    B2_TRY(empty.alloc((size_t)nEmpty));
    B2_CUDA(cudaMemsetAsync(cnt.p, 0, sizeof(int), s));
    es_bits_kernel<<<ceil_div(nRow, 256), 256, 0, s>>>(ptr, nRow, bits.p, nEmpty ? empty.p : nullptr, cnt.p);
    B2_KERNEL_CHECK();
    es_group_count_kernel<<<ceil_div(nGroups + 1, 256), 256, 0, s>>>(bits.p, nGroups, grpRun.p);
    B2_KERNEL_CHECK();
    B2_TRY(exclusive_scan_i32(grpRun.p, grpRun.p, nGroups + 1, s));
    if (nEmpty) {
        B2_TRY(nzrow.alloc((size_t)(nRow - nEmpty)));
        es_nzrow_kernel<<<ceil_div(nRow, 256), 256, 0, s>>>(ptr, nRow, bits.p, grpRun.p, nzrow.p);
        B2_KERNEL_CHECK();
    }
    B2_CUDA(cudaStreamSynchronize(s));
    ok = true;
    return B200SPMV_OK;
}

int EntryStream::prepare(int rb, int re)
{
    if (rb < 0 || re > nRow || rb > re) { set_error("prepare_rows: bad row range [%d,%d) for %d rows", rb, re, nRow); return B200SPMV_ERR_INVALID; }
    const auto key = std::make_pair(rb, re);
    if (range_cache.count(key)) return B200SPMV_OK;
    int pb = 0, pe = 0;
    B2_CUDA(cudaMemcpy(&pb, ptr + rb, sizeof(int), cudaMemcpyDeviceToHost));
    B2_CUDA(cudaMemcpy(&pe, ptr + re, sizeof(int), cudaMemcpyDeviceToHost));
    const int lo = pb / ES_E, hi = pe > pb ? (pe - 1) / ES_E + 1 : lo;           // tiles that hold an entry of the rows
    range_cache.emplace(key, std::make_pair(lo, hi));
    return B200SPMV_OK;
}

template <bool TMA>
static int es_launch(EntryStream &T, const double *x, double *y, int tileLo, int tileHi, int rb, int re, cudaStream_t s)
{
    constexpr size_t smem = TMA ? 24 * (size_t)ES_E : 0;
    auto kern = entry_stream_kernel<TMA>;
    static std::map<int, int> per_sm;
    static int sms = 0;
    int dev = 0;
    B2_CUDA(cudaGetDevice(&dev));
    if (!sms) B2_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    auto it = per_sm.find(dev);
    if (it == per_sm.end()) {
        if (smem) B2_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int n = 0;
        B2_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kern, ES_THREADS, smem));
        if (n < 1) { set_error("entry stream: %zu bytes of shared memory do not fit", smem); return B200SPMV_ERR_UNSUPPORTED; }
        it = per_sm.emplace(dev, n).first;
    }
    const int nT = tileHi - tileLo;
    const int perSm = std::min(it->second, 6);
    const int grid = TMA ? std::min(nT, sms * perSm) : nT;
    kern<<<grid, ES_THREADS, smem, s>>>(T.idx, static_cast<const double *>(T.val), T.bits.p, T.grpRun.p, T.nEmpty ? T.nzrow.p : nullptr, x, y, T.carry.p, T.nnz, tileLo,
                                        tileHi, rb, re);
    B2_KERNEL_CHECK();
    if (nT > 1) {
        entry_stream_fixup_kernel<<<ceil_div(nT - 1, 256), 256, 0, s>>>(T.bits.p, T.grpRun.p, T.nEmpty ? T.nzrow.p : nullptr, y, T.carry.p, ES_E,
                                                                       tileLo, tileHi, rb, re);
        B2_KERNEL_CHECK();
    }
    return B200SPMV_OK;
}

int EntryStream::run_rows(const double *x, double *y, int rb, int re, cudaStream_t s)
{
    if (rb < 0 || re > nRow || rb > re) { set_error("multiply_rows: bad row range [%d,%d) for %d rows", rb, re, nRow); return B200SPMV_ERR_INVALID; }
    if (rb == re) return B200SPMV_OK;
    int lo = 0, hi = nTiles;
    if (!(rb == 0 && re == nRow)) {
        auto it = range_cache.find(std::make_pair(rb, re));
        if (it == range_cache.end()) {
            cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
            if (cudaStreamIsCapturing(s, &cap) == cudaSuccess && cap != cudaStreamCaptureStatusNone) {
                set_error("multiply_rows: row range [%d,%d) is used for the first time inside a stream capture; call b200spmv_prepare_rows() first", rb, re);
                return B200SPMV_ERR_STATE;
            }
            B2_TRY(prepare(rb, re));
            it = range_cache.find(std::make_pair(rb, re));
        }
        lo = it->second.first;
        hi = it->second.second;
    }
    if (nEmpty) {
        es_zero_rows_kernel<<<ceil_div(nEmpty, 256), 256, 0, s>>>(empty.p, nEmpty, rb, re, y);
        B2_KERNEL_CHECK();
    }
    if (hi <= lo) return B200SPMV_OK;
    if (tma) return es_launch<true>(*this, x, y, lo, hi, rb, re, s);
    return es_launch<false>(*this, x, y, lo, hi, rb, re, s);
}

template <typename VT, typename XT, typename AT, bool TMA, int KP, bool VEC>
static int es_multi_launch(EntryStream &T, int k, const XT *X, long long ldx, XT *Y, long long ldy, cudaStream_t s)
{
    constexpr size_t smem = TMA ? (4 + sizeof(VT)) * 2 * (size_t)ES_E : 0;
    auto kern = entry_stream_multi_kernel<VT, XT, AT, TMA, KP, VEC>;
    static std::map<int, int> per_sm;
    static int sms = 0;
    int dev = 0;
    B2_CUDA(cudaGetDevice(&dev));
    if (!sms) B2_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    auto it = per_sm.find(dev);
    if (it == per_sm.end()) {
        if (smem) B2_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int n = 0;
        B2_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kern, ES_THREADS, smem));
        if (n < 1) { set_error("entry stream: %zu bytes of shared memory do not fit", smem); return B200SPMV_ERR_UNSUPPORTED; }
        it = per_sm.emplace(dev, n).first;
    }
    const int nT = T.nTiles;
    const int grid = TMA ? std::min(nT, sms * std::min(it->second, 6)) : nT;
    AT *carry = reinterpret_cast<AT *>(T.carryK.p);
    kern<<<grid, ES_THREADS, smem, s>>>(T.idx, static_cast<const VT *>(T.val), T.bits.p, T.grpRun.p, T.nEmpty ? T.nzrow.p : nullptr,
                                        X, ldx, Y, ldy, k, carry, T.nnz, 0, nT, 0, T.nRow);
    B2_KERNEL_CHECK();
    if (nT > 1) {
        entry_stream_multi_fixup_kernel<<<ceil_div((long long)(nT - 1) * k, 256), 256, 0, s>>>(
            T.bits.p, T.grpRun.p, T.nEmpty ? T.nzrow.p : nullptr, Y, ldy, k, carry, ES_E, 0, nT);
        B2_KERNEL_CHECK();
    }
    return B200SPMV_OK;
}

template <typename VT, typename XT, typename AT, bool TMA>
static int es_multi_k(EntryStream &T, int k, const XT *X, long long ldx, XT *Y, long long ldy, cudaStream_t s)
{
    if (k == 1) return es_multi_launch<VT, XT, AT, TMA, 1, false>(T, k, X, ldx, Y, ldy, s);
    if (k == 2) {
        return ld_xrow_vec(X, ldx, 2) ? es_multi_launch<VT, XT, AT, TMA, 2, true>(T, k, X, ldx, Y, ldy, s)
                                      : es_multi_launch<VT, XT, AT, TMA, 2, false>(T, k, X, ldx, Y, ldy, s);
    }
    return ld_xrow_vec(X, ldx, 4) ? es_multi_launch<VT, XT, AT, TMA, 4, true>(T, k, X, ldx, Y, ldy, s)
                                  : es_multi_launch<VT, XT, AT, TMA, 4, false>(T, k, X, ldx, Y, ldy, s);
}

// the part shared by both precisions: zero the empty rows, allocate the carries on the first call
template <typename XT>
static int es_multi_prologue(EntryStream &T, int k, XT *Y, long long ldy, const char *entry, cudaStream_t s)
{
    if (!T.carryK.p) {
        cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(s, &cap) == cudaSuccess && cap != cudaStreamCaptureStatusNone) {
            set_error("%s: first call on this handle inside a stream capture; call it once outside the capture first", entry);
            return B200SPMV_ERR_STATE;
        }
        // fp32 vectors: the head carries, then the tail slots of entry_stream_multi_kernel (fp64 or fp32, in fp64 room)
        B2_TRY(T.carryK.alloc((size_t)T.nTiles * ES_KMAX * (T.f32 ? 2 : 1)));
    }
    if (T.nEmpty) {
        es_zero_rows_multi_kernel<<<ceil_div((long long)T.nEmpty * k, 256), 256, 0, s>>>(T.empty.p, T.nEmpty, k, Y, ldy);
        B2_KERNEL_CHECK();
    }
    return B200SPMV_OK;
}

int EntryStream::run_multi(int k, const double *X, long long ldx, double *Y, long long ldy, cudaStream_t s)
{
    if (k < 1 || k > ES_KMAX) { set_error("multiply_multi: k=%d outside 1..%d", k, ES_KMAX); return B200SPMV_ERR_INVALID; }
    if (f32) { set_error("multiply_multi: the entry stream holds fp32 values"); return B200SPMV_ERR_UNSUPPORTED; }
    if (!ok) return zero_rows_multi(nRow, k, Y, ldy, s);      // no entries
    B2_TRY(es_multi_prologue(*this, k, Y, ldy, "multiply_multi", s));
    if (tma) return es_multi_k<double, double, double, true>(*this, k, X, ldx, Y, ldy, s);
    return es_multi_k<double, double, double, false>(*this, k, X, ldx, Y, ldy, s);
}

int EntryStream::run_multi_f32(int k, const float *X, long long ldx, float *Y, long long ldy, bool acc64, cudaStream_t s)
{
    if (k < 1 || k > ES_KMAX) { set_error("multiply_multi_f32: k=%d outside 1..%d", k, ES_KMAX); return B200SPMV_ERR_INVALID; }
    if (!f32) { set_error("multiply_multi_f32: the entry stream holds fp64 values"); return B200SPMV_ERR_STATE; }
    if (!ok) return zero_rows_multi(nRow, k, Y, ldy, s);
    B2_TRY(es_multi_prologue(*this, k, Y, ldy, "multiply_multi_f32", s));
    if (acc64) {
        if (tma) return es_multi_k<float, float, double, true>(*this, k, X, ldx, Y, ldy, s);
        return es_multi_k<float, float, double, false>(*this, k, X, ldx, Y, ldy, s);
    }
    if (tma) return es_multi_k<float, float, float, true>(*this, k, X, ldx, Y, ldy, s);
    return es_multi_k<float, float, float, false>(*this, k, X, ldx, Y, ldy, s);
}

}  // namespace b2
