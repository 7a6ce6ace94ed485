// tile_stream.cu -- kernels of the tile-stream multiply (see tile_stream.cuh).
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <type_traits>

#include "tile_stream.cuh"

namespace b2 {

// fp64 slots per tile in `carry` (s = ts_slots): carry[s t] holds the piece of a row carried in from earlier tiles; with
// fp32 vectors carry[2 t + 1] also holds the partial of the row that runs on past the tile's end.  That partial stays in
// fp64 until the fix-up kernel has added the carries, so a row of fp64 sums (precision 2) is rounded to fp32 once.  fp64
// vectors keep the partial in y.
template <typename XT> __host__ __device__ constexpr int ts_slots() { return std::is_same<XT, float>::value ? 2 : 1; }

// tile_row[t] = first row r with row_ptr[r] >= t*TS_TILE (lower bound over row_ptr[0..nRow]).
// Rows [tile_row[t], tile_row[t+1]) are OWNED by tile t: their first entry lies in it.  Empty
// rows are owned by the tile that contains their (shared) position; trailing rows by the last.
__global__ void tile_row_kernel(const int *__restrict__ ptr, int nRow, int nTiles, int tile, int *__restrict__ tile_row)
{
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t > nTiles) return;
    if (t == nTiles) {
        tile_row[t] = nRow;
        return;
    }
    int key = t * tile, lo = 0, hi = nRow + 1;
    while (lo < hi) {
        int mid = (lo + hi) >> 1;
        if (ptr[mid] < key) lo = mid + 1;
        else hi = mid;
    }
    tile_row[t] = lo;
}

// four consecutive matrix values as doubles: fp64 storage = two 128-bit loads, fp32 storage = one
__device__ __forceinline__ void ld_val4(const double *p, uint64_t pol, double &a, double &b, double &c, double &d)
{
    const double2 lo = ld_stream_d2(p, pol), hi = ld_stream_d2(p + 2, pol);
    a = lo.x; b = lo.y; c = hi.x; d = hi.y;
}
__device__ __forceinline__ void ld_val4(const float *p, uint64_t pol, double &a, double &b, double &c, double &d)
{
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p), "l"(pol));
    a = r.x; b = r.y; c = r.z; d = r.w;                 // fp32 -> fp64 is exact
}
__device__ __forceinline__ double ld_val1(const double *p, uint64_t pol) { return ld_stream_d1(p, pol); }
__device__ __forceinline__ double ld_val1(const float *p, uint64_t pol)
{
    float r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(r) : "l"(p), "l"(pol));
    return (double)r;
}

// four consecutive products to shared memory with 128-bit stores (p is 16-byte aligned for float, 32 for double)
__device__ __forceinline__ void st_prod4(double *p, double a, double b, double c, double d)
{
    reinterpret_cast<double2 *>(p)[0] = make_double2(a, b);
    reinterpret_cast<double2 *>(p)[1] = make_double2(c, d);
}
__device__ __forceinline__ void st_prod4(float *p, float a, float b, float c, float d)
{
    *reinterpret_cast<float4 *>(p) = make_float4(a, b, c, d);
}

// A variant that brought the tile's col / val slices in by TMA bulk copies (to take the matrix stream off the SM's L1 miss
// path, which the x gathers saturate on gather-bound matrices) was measured and removed: with bulk copies in flight the
// x slice no longer stays L2-resident, whatever cache policy the copies carry (c2 4.4-7.4 ms against 2.9, profiles/r2_experiments.md).
// VT = stored value type, XT = type of x and y, AT = type of the products and sums.
template <typename VT, typename XT, typename AT, int TH>
__global__ void __launch_bounds__(TH)
tile_stream_kernel(const int *__restrict__ row_ptr, const int *__restrict__ col,
                   const VT *__restrict__ val, const int *__restrict__ tile_row,
                   const XT *__restrict__ x, XT *__restrict__ y, double *__restrict__ carry,
                   int nnz, int tileLo, int rowLo, int rowHi, int accumulate, int vec_ok)
{
    constexpr int TILE = TH * TS_IPT;
    __shared__ __align__(16) AT prod[TILE];
    __shared__ int long_row[TILE / TS_LONG + 2];
    __shared__ int n_long;

    const int tid = threadIdx.x;
    const int t = tileLo + blockIdx.x;
    const int t0 = t * TILE;
    const int t1 = min(t0 + TILE, nnz);
    const uint64_t pol_stream = policy_evict_first();
    const uint64_t pol_x = policy_evict_last();
    if (tid == 0) n_long = 0;

    // ---- phase 1: stream the tile, gather x, park products in shared memory
    if (t1 - t0 == TILE && vec_ok) {
        int4 c[TS_IPT / 4];
        double2 v[TS_IPT / 2];
#pragma unroll
        for (int k = 0; k < TS_IPT / 4; k++) {
            const int e = t0 + 4 * (tid + k * TH);
            c[k] = ld_stream_i4(col + e, pol_stream);
            ld_val4(val + e, pol_stream, v[2 * k].x, v[2 * k].y, v[2 * k + 1].x, v[2 * k + 1].y);
        }
        XT xs[TS_IPT];
#pragma unroll
        for (int k = 0; k < TS_IPT / 4; k++) {
            xs[4 * k + 0] = ld_x(x + c[k].x, pol_x);
            xs[4 * k + 1] = ld_x(x + c[k].y, pol_x);
            xs[4 * k + 2] = ld_x(x + c[k].z, pol_x);
            xs[4 * k + 3] = ld_x(x + c[k].w, pol_x);
        }
#pragma unroll
        for (int k = 0; k < TS_IPT / 4; k++) {
            const int o = 4 * (tid + k * TH);
            st_prod4(prod + o, Arith<AT>::mul((AT)v[2 * k].x, (AT)xs[4 * k]), Arith<AT>::mul((AT)v[2 * k].y, (AT)xs[4 * k + 1]),
                     Arith<AT>::mul((AT)v[2 * k + 1].x, (AT)xs[4 * k + 2]), Arith<AT>::mul((AT)v[2 * k + 1].y, (AT)xs[4 * k + 3]));
        }
    } else {
        for (int i = tid; i < t1 - t0; i += TH)
            prod[i] = Arith<AT>::mul((AT)ld_val1(val + t0 + i, pol_stream),
                                     (AT)ld_x(x + ld_stream_i1(col + t0 + i, pol_stream), pol_x));
    }

    const int r_lo = tile_row[t], r_hi = tile_row[t + 1];
    const int first = row_ptr[r_lo];          // r_lo <= nRow, row_ptr[nRow] = nnz
    const int cin_end = min(first, t1);       // [t0, cin_end) belongs to row r_lo-1
    __syncthreads();

    // ---- phase 2a: one thread per owned row, in-tile row-bin scheduler
    for (int r = r_lo + tid; r < r_hi; r += TH) {
        if (r < rowLo || r >= rowHi) continue;
        const int b = row_ptr[r], e_full = row_ptr[r + 1];
        const int e = min(e_full, t1);
        if (e_full > t1 && e_full - b <= TS_LONG) continue;   // short row crossing: fix-up recomputes it
        if (e - b > TS_LONG) {
            long_row[atomicAdd(&n_long, 1)] = r;
            continue;
        }
        AT acc = accumulate == CS_CONTINUE ? (AT)y[r] : (AT)0;    // CONTINUE: the running sum of the earlier column blocks
        for (int j = b; j < e; j++) acc = Arith<AT>::add(acc, prod[j - t0]);
        if constexpr (ts_slots<XT>() == 2) {
            if (e_full > t1) {
                carry[2 * t + 1] = (double)(accumulate == CS_ADD ? Arith<AT>::add((AT)y[r], acc) : acc);
                continue;
            }
        }
        y[r] = (XT)(accumulate == CS_ADD ? Arith<AT>::add((AT)y[r], acc) : acc);
    }
    if (tid == 0 && cin_end > t0) {
        const int rc = r_lo - 1;
        if (first - row_ptr[rc] > TS_LONG && rc >= rowLo && rc < rowHi)
            long_row[atomicAdd(&n_long, 1)] = -1;
    }
    __syncthreads();

    // ---- phase 2b: one warp per long row / carried-in piece (fp64 tree whatever AT is: a handful of adds per row)
    const int lane = tid & 31, warp = tid >> 5;
    const int nl = n_long;
    for (int i = warp; i < nl; i += TH / 32) {
        const int r = long_row[i];
        int b, e;
        if (r < 0) {
            b = t0;
            e = cin_end;
        } else {
            b = row_ptr[r];
            e = min(row_ptr[r + 1], t1);
        }
        double acc = 0.0;
        for (int j = b + lane; j < e; j += 32) acc += (double)prod[j - t0];
        acc = warp_sum(acc);
        if (lane == 0) {
            if (r < 0) carry[ts_slots<XT>() * t] = acc;
            else if (ts_slots<XT>() == 2 && row_ptr[r + 1] > t1) carry[2 * t + 1] = accumulate ? (double)y[r] + acc : acc;
            else y[r] = (XT)(accumulate ? (double)y[r] + acc : acc);
        }
    }
}

// Finishes the rows that cross tile boundaries; one thread per tile, only the FIRST carrying
// tile of a row acts.  Short rows are recomputed from global memory in the reference's order.
template <typename VT, typename XT, typename AT>
__global__ void tile_fixup_kernel(const int *__restrict__ row_ptr, const int *__restrict__ col,
                                  const VT *__restrict__ val, const int *__restrict__ tile_row,
                                  const XT *__restrict__ x, XT *__restrict__ y,
                                  const double *__restrict__ carry, int tileLo, int tileHi, int rowLo,
                                  int rowHi, int accumulate, int tile)
{
    const int t = tileLo + blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= tileHi || t == 0) return;
    const int t0 = t * tile;
    const int r0 = tile_row[t];
    const int e = row_ptr[r0];
    if (e <= t0) return;                       // a row starts exactly at the tile start
    const int rc = r0 - 1;
    if (rc < rowLo || rc >= rowHi) return;
    const int b = row_ptr[rc];
    if (t != b / tile + 1) return;
    if (e - b <= TS_LONG) {
        AT acc = accumulate == CS_CONTINUE ? (AT)y[rc] : (AT)0;
        for (int j = b; j < e; j++) acc = Arith<AT>::add(acc, Arith<AT>::mul((AT)val[j], (AT)x[col[j]]));
        y[rc] = (XT)(accumulate == CS_ADD ? Arith<AT>::add((AT)y[rc], acc) : acc);
    } else {
        const int last = (e - 1) / tile;
        double sum = 0.0;
        for (int u = t; u <= last; u++) sum += carry[ts_slots<XT>() * u];
        if constexpr (ts_slots<XT>() == 2) y[rc] = (XT)(carry[2 * (t - 1) + 1] + sum);     // rc starts in tile t - 1
        else y[rc] = (XT)((double)y[rc] + sum);
    }
}

int TileStream::build(const int *row_ptr_d, const int *col_d, const void *val_d, bool val_is_f32, int nRow_, int nnz_,
                      cudaStream_t s)
{
    f32 = val_is_f32;
    row_ptr = row_ptr_d;
    col = col_d;
    val = val_d;
    nRow = nRow_;
    nnz = nnz_;
    static const int env_threads = getenv("B200SPMV_TS_THREADS") ? atoi(getenv("B200SPMV_TS_THREADS")) : 256;
    threads = (env_threads == 128 || env_threads == 512) ? env_threads : 256;
    tile = threads * TS_IPT;
    nTiles = ceil_div(nnz, tile);
    B2_TRY(tile_row.alloc((size_t)nTiles + 1));
    B2_TRY(carry.alloc((size_t)nTiles * (f32 ? 2 : 1)));   // fp32 values: the fp32-vector kernels may run (ts_slots)
    tile_row_kernel<<<ceil_div(nTiles + 1, 256), 256, 0, s>>>(row_ptr, nRow, nTiles, tile, tile_row.p);
    B2_KERNEL_CHECK();
    range_cache.clear();
    return B200SPMV_OK;
}

int TileStream::run_rows(const double *x, double *y, int accumulate, int rb, int re, cudaStream_t s)
{
    if (rb < 0 || re > nRow || rb > re) {
        set_error("multiply_rows: bad row range [%d,%d) for %d rows", rb, re, nRow);
        return B200SPMV_ERR_INVALID;
    }
    if (rb == re) return B200SPMV_OK;
    if (rb == 0 && re == nRow) return run_all(x, y, accumulate, s);
    const auto key = std::make_pair(rb, re);
    auto it = range_cache.find(key);
    if (it == range_cache.end()) {
        // first use of this row range: two row pointers have to be read back.  b200spmv_prepare_rows() does this ahead
        // of time; here it is refused during stream capture (a synchronous copy would invalidate the capture)
        cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(s, &cap) == cudaSuccess && cap != cudaStreamCaptureStatusNone) {
            set_error("multiply_rows: row range [%d,%d) is used for the first time inside a stream capture; call "
                      "b200spmv_prepare_rows() (or run one eager multiply_rows) first", rb, re);
            return B200SPMV_ERR_STATE;
        }
        B2_TRY(prepare(rb, re));
        it = range_cache.find(key);
    }
    return run(x, y, accumulate, rb, re, it->second.first, it->second.second, s);
}

// tiles that hold any entry (or the shared position of empty rows) of rows [rb, re); synchronous, cached
int TileStream::prepare(int rb, int re)
{
    if (rb < 0 || re > nRow || rb > re) {
        set_error("prepare_rows: bad row range [%d,%d) for %d rows", rb, re, nRow);
        return B200SPMV_ERR_INVALID;
    }
    const auto key = std::make_pair(rb, re);
    if (range_cache.count(key)) return B200SPMV_OK;
    int pb = 0, pe = 0;
    B2_CUDA(cudaMemcpy(&pb, row_ptr + rb, sizeof(int), cudaMemcpyDeviceToHost));
    B2_CUDA(cudaMemcpy(&pe, row_ptr + re, sizeof(int), cudaMemcpyDeviceToHost));
    const int lo = nTiles ? std::min(pb / tile, nTiles - 1) : 0;
    const int hi = std::min(nTiles, pe / tile + 1);
    range_cache.emplace(key, std::make_pair(lo, hi));
    return B200SPMV_OK;
}

template <typename VT, typename XT, typename AT>
static int ts_launch(const TileStream &T, const XT *x, XT *y, int acc, int rowLo, int rowHi, int tileLo, int tileHi, cudaStream_t s)
{
    const VT *v = static_cast<const VT *>(T.val);
    const int vec_ok = ((reinterpret_cast<uintptr_t>(T.col) | reinterpret_cast<uintptr_t>(T.val)) & 15) == 0;
    const int nT = tileHi - tileLo;
    const bool fix = nT > 1 || tileLo > 0;
#define TS_ARGS T.row_ptr, T.col, v, T.tile_row.p, x, y, T.carry.p, T.nnz, tileLo, rowLo, rowHi, acc, vec_ok
    if (T.threads == 128) tile_stream_kernel<VT, XT, AT, 128><<<nT, 128, 0, s>>>(TS_ARGS);
    else if (T.threads == 512) tile_stream_kernel<VT, XT, AT, 512><<<nT, 512, 0, s>>>(TS_ARGS);
    else tile_stream_kernel<VT, XT, AT, 256><<<nT, 256, 0, s>>>(TS_ARGS);
#undef TS_ARGS
    if (fix)
        tile_fixup_kernel<VT, XT, AT><<<ceil_div(nT, 256), 256, 0, s>>>(T.row_ptr, T.col, v, T.tile_row.p, x, y, T.carry.p, tileLo,
                                                                        tileHi, rowLo, rowHi, acc, T.tile);
    B2_KERNEL_CHECK();
    return B200SPMV_OK;
}

int TileStream::run(const double *x, double *y, int accumulate, int rowLo, int rowHi, int tileLo,
                    int tileHi, cudaStream_t s) const
{
    if (rowHi <= rowLo) return B200SPMV_OK;
    if (nTiles == 0) {   // no non-zeros at all: y = 0 (beta = 0)
        if (!accumulate) B2_CUDA(cudaMemsetAsync(y + rowLo, 0, sizeof(double) * (size_t)(rowHi - rowLo), s));
        return B200SPMV_OK;
    }
    if (f32) return ts_launch<float, double, double>(*this, x, y, accumulate, rowLo, rowHi, tileLo, tileHi, s);
    return ts_launch<double, double, double>(*this, x, y, accumulate, rowLo, rowHi, tileLo, tileHi, s);
}

// fp32 vectors over fp32 values; acc64: products and sums in fp64
int TileStream::run_rows_f32(const float *x, float *y, int accumulate, int rb, int re, bool acc64, cudaStream_t s)
{
    if (!f32) { set_error("tile-stream: fp32 vectors need fp32 value storage"); return B200SPMV_ERR_STATE; }
    if (rb < 0 || re > nRow || rb > re) { set_error("multiply_rows: bad row range [%d,%d) for %d rows", rb, re, nRow); return B200SPMV_ERR_INVALID; }
    if (rb == re) return B200SPMV_OK;
    int lo = 0, hi = nTiles;
    if (!(rb == 0 && re == nRow)) {
        B2_TRY(prepare(rb, re));
        const auto it = range_cache.find(std::make_pair(rb, re));
        lo = it->second.first;
        hi = it->second.second;
    }
    if (nTiles == 0) {
        if (!accumulate) B2_CUDA(cudaMemsetAsync(y + rb, 0, sizeof(float) * (size_t)(re - rb), s));
        return B200SPMV_OK;
    }
    if (acc64) return ts_launch<float, float, double>(*this, x, y, accumulate, rb, re, lo, hi, s);
    return ts_launch<float, float, float>(*this, x, y, accumulate, rb, re, lo, hi, s);
}

}  // namespace b2
