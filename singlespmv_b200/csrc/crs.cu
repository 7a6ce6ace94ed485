// crs.cu -- CRS plugin: device conversion + adaptive multiply (row-block stream for short rows, tile-stream otherwise).
// Reference: /root/reference/src/opt_crs.{h,cpp} (SpMatOpt{ptr,idx,val}; OptimizeProblem :10-42; SpMV :44-70).
#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "chunk_stream.cuh"
#include "entry_stream.cuh"
#include "tile_stream.cuh"

namespace b2 {

// fp32 storage of the matrix values (options.value_f32): val is rounded to nearest once, at conversion, and
// widened back (exactly) in the kernel -- x, y and every product and sum stay fp64.  Cuts the stream from
// 12 to 8 B/nnz; y equals the fp64 path run on the rounded matrix bit for bit.
__global__ void crs_to_f32_kernel(const double *__restrict__ in, int n, float *__restrict__ out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = __double2float_rn(in[i]);
}
__global__ void crs_to_f64_kernel(const float *__restrict__ in, int n, double *__restrict__ out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (double)in[i];
}

// ---- short-row path ("row-block stream"): used when the longest row has at most RBS_MAXLEN entries.
// A warp owns 32 consecutive rows at a time.  Their entries are one contiguous run of the idx/val streams, so the
// warp reads them lane-contiguously (a request = 128 B of idx / 256 B of val), gathers x, parks the products in
// its PRIVATE slice of shared memory (__syncwarp only: no block barrier, no tiles, no carries, one launch), and
// then every lane sums its own row in ascending column order with unfused mul/add -> bit-identical to the
// reference for every row.  The tile-stream kernel stays the path for everything with longer or skewed rows.
constexpr int RBS_MAXLEN = 16;
constexpr int RBS_WARPS = 8;
constexpr int RBS_ITERS = 8;      // row blocks per warp

__device__ __forceinline__ double rbs_ld(const double *p, uint64_t pol) { return ld_stream_d1(p, pol); }
__device__ __forceinline__ double rbs_ld(const float *p, uint64_t) { return (double)__ldg(p); }

template <typename VT, int U, int MINB>
__global__ void __launch_bounds__(RBS_WARPS * 32, MINB)
crs_rowblock_kernel(const int *__restrict__ ptr, const int *__restrict__ idx, const VT *__restrict__ val,
                    const double *__restrict__ x, double *__restrict__ y, int rowBegin, int rowEnd, int cap, int iters)
{
    extern __shared__ __align__(16) double rbs_prod[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double *prod = rbs_prod + (size_t)warp * cap;
    const uint64_t pol_stream = policy_evict_first(), pol_x = policy_evict_last();
    const long long gw = (long long)blockIdx.x * RBS_WARPS + warp;
    // a warp walks RBS_ITERS consecutive row blocks.  Measured alternatives (profiles/r1_experiments.md): dealing the
    // blocks round-robin to the warps of a CTA, prefetching the next block's row pointers, 16 blocks per warp and
    // batches of 4 instead of 8 loads per lane were all slower on c5 (682-702 vs 748 GFLOP/s)
    for (int it = 0; it < iters; it++) {
        const long long r0l = (long long)rowBegin + (gw * iters + it) * 32;
        if (r0l >= rowEnd) break;                                // warp-uniform
        const int r0 = (int)r0l, r = r0 + lane;
        const int p = ptr[min(r, rowEnd)], q = ptr[min(r + 1, rowEnd)];
        const int base = __shfl_sync(0xffffffffu, p, 0), end = __shfl_sync(0xffffffffu, q, 31);
        const int n = end - base;                                // <= 32 * RBS_MAXLEN <= cap
        for (int k0 = 0; k0 < n; k0 += 32 * U) {
            int c[U];
            double v[U];
#pragma unroll
            for (int u = 0; u < U; u++) {
                const int k = k0 + u * 32 + lane;
                if (k < n) {
                    c[u] = ld_stream_i1(idx + base + k, pol_stream);
                    v[u] = rbs_ld(val + base + k, pol_stream);
                }
            }
#pragma unroll
            for (int u = 0; u < U; u++) {
                const int k = k0 + u * 32 + lane;
                if (k < n) prod[k] = __dmul_rn(v[u], ld_x(x + c[u], pol_x));
            }
        }
        __syncwarp();
        if (r < rowEnd) {
            double acc = 0.0;
            for (int j = p - base; j < q - base; j++) acc = __dadd_rn(acc, prod[j]);
            y[r] = acc;
        }
        __syncwarp();
    }
}

// y[rb..re) = A x for matrices whose longest row has at most RBS_MAXLEN entries (CRS and SS share it)
int rowblock_spmv(const int *ptr, const int *idx, const void *val, bool f32, int maxLen, int rb, int re, const double *x,
                  double *y, cudaStream_t s)
{
    if (rb >= re) return B200SPMV_OK;
    const int cap = 32 * ((maxLen + 1) & ~1);                               // doubles per warp, 16-byte multiple
    const int iters = RBS_ITERS;
    const int grid = ceil_div(re - rb, RBS_WARPS * iters * 32);
    const size_t smem = (size_t)RBS_WARPS * cap * sizeof(double);
    if (smem > 48 * 1024) {
        B2_CUDA(cudaFuncSetAttribute(crs_rowblock_kernel<float, 8, 5>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        B2_CUDA(cudaFuncSetAttribute(crs_rowblock_kernel<double, 8, 5>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    if (f32) crs_rowblock_kernel<float, 8, 5><<<grid, RBS_WARPS * 32, smem, s>>>(ptr, idx, static_cast<const float *>(val), x, y, rb, re, cap, iters);
    else crs_rowblock_kernel<double, 8, 5><<<grid, RBS_WARPS * 32, smem, s>>>(ptr, idx, static_cast<const double *>(val), x, y, rb, re, cap, iters);
    B2_KERNEL_CHECK();
    return B200SPMV_OK;
}
bool rowblock_applies(int maxLen, long long nnz)
{
    static const char *force = getenv("B200SPMV_CRS_PATH");                 // "tile" forces the tile-stream (experiments)
    if (force && !strcmp(force, "tile")) return false;
    static const int lim = getenv("B200SPMV_RBS_MAXLEN") ? atoi(getenv("B200SPMV_RBS_MAXLEN")) : RBS_MAXLEN;
    return nnz > 0 && maxLen <= lim;
}

struct CrsFormat : Format {
    int maxLen = 0;
    bool short_rows = false, use_rbs = false;
    DevBuf<int> ptr, idx;
    DevBuf<double> val;
    DevBuf<float> val32;
    bool f32;
    TileStream ts;
    ChunkStream cs;
    EntryStream es;
    bool use_es = false;
    int path_opt;
    int prec;                             // options.precision: 0 fp64 vectors, 1 fp32 vectors + sums, 2 fp32 vectors, fp64 sums
    explicit CrsFormat(const b200spmv_options &o) : f32(o.value_f32 != 0 || o.precision != 0), path_opt(o.crs_path), prec(o.precision) {}

    int convert(const CooView &A, cudaStream_t s) override
    {
        nRow = A.nRow; nCol = A.nCol; nnz = A.nnz;
        B2_TRY(validate_sorted_coo(A, s));
        B2_TRY(ptr.alloc((size_t)nRow + 1));
        B2_TRY(idx.alloc((size_t)nnz + CS_SLACK));
        B2_TRY(build_row_ptr(A.row, nnz, nRow, ptr.p, s));                      // opt_crs.cpp:27-33
        B2_CUDA(cudaMemcpyAsync(idx.p, A.col, sizeof(int) * (size_t)nnz, cudaMemcpyDeviceToDevice, s));   // :29
        if (f32) {
            val.release();
            B2_TRY(val32.alloc((size_t)nnz + CS_SLACK));
            if (nnz) crs_to_f32_kernel<<<ceil_div(nnz, 256), 256, 0, s>>>(A.val, nnz, val32.p);
            B2_KERNEL_CHECK();
            B2_TRY(ts.build(ptr.p, idx.p, val32.p, true, nRow, nnz, s));
        } else {
            B2_TRY(val.alloc((size_t)nnz + CS_SLACK));
            B2_CUDA(cudaMemcpyAsync(val.p, A.val, sizeof(double) * (size_t)nnz, cudaMemcpyDeviceToDevice, s));   // :30
            B2_TRY(ts.build(ptr.p, idx.p, val.p, false, nRow, nnz, s));
        }
        B2_TRY(max_row_length(ptr.p, nRow, &maxLen, s));
        B2_TRY(cs.build(ptr.p, idx.p, f32 ? (const void *)val32.p : (const void *)val.p, f32, nRow, nnz, maxLen, s));
        // path: 1 = tile-stream always; 2 = round 1's row-block stream where it applies (longest row <= 16);
        // otherwise the TMA-fed row-chunk stream when the rows are short enough, else the tile-stream
        // ... unless the gathers range over tens of MB (uniform random, R-MAT): x must stay in L2, which it does with the
        // tile-stream's evict-first loads and does not with bulk copies in flight (uniform 2^24 x 11: 40 G entries/s TMA-fed)
        use_rbs = path_opt == 2 && !prec && rowblock_applies(maxLen, nnz);
        int band = 0;
        if (path_opt == 0 || path_opt == 4) B2_TRY(max_band(A.row, A.col, nnz, A.rowOffset, &band, s));
        short_rows = path_opt != 1 && path_opt != 4 && (use_rbs || (cs.ok && !gathers_need_l2(band)));
        // gather-bound matrices (fp64): the load-fed entry stream (entry_stream.cuh) -- c3 441 GFLOP/s against 365 for the tile-stream
        // (cuSPARSE CSR: 405).  Banded matrices with medium rows keep the tile-stream: the TMA-fed entry stream is level with it
        // (c4: 659 against 642) and the tile-stream sums rows of up to 64 entries in the reference's order.  crs_path = 4 forces the
        // entry stream, crs_path = 1 / B200SPMV_CRS_PATH=tile the tile-stream.
        static const char *force = getenv("B200SPMV_CRS_PATH");
        use_es = false;
        const bool force_es = force && !strcmp(force, "es") && path_opt == 0;          // experiments: entry stream wherever the rows are not short
        if (!short_rows && !f32 && !prec && (path_opt == 4 || force_es || (path_opt == 0 && gathers_need_l2(band))) && !(force && !strcmp(force, "tile"))) {
            B2_TRY(es.build(ptr.p, idx.p, val.p, nRow, nnz, gathers_need_l2(band), s));
            use_es = es.ok;
        }
        B2_CUDA(cudaStreamSynchronize(s));
        return B200SPMV_OK;
    }

    int multiply(const double *x, double *y, cudaStream_t s) override { return multiply_rows(0, nRow, x, y, s); }
    int multiply_f32(const float *x, float *y, cudaStream_t s) override
    {
        if (!prec) { set_error("multiply_f32: the handle was created with precision = 0 (fp64 vectors)"); return B200SPMV_ERR_STATE; }
        if (short_rows && !use_rbs) return cs.run_f32(x, y, 0, nRow, CS_OVERWRITE, prec == 2, s);
        return ts.run_rows_f32(x, y, CS_OVERWRITE, 0, nRow, prec == 2, s);
    }

    int multiply_rows(int rb, int re, const double *x, double *y, cudaStream_t s) override
    {
        if (prec) { set_error("multiply: the handle was created with precision = %d, use b200spmv_multiply_f32", prec); return B200SPMV_ERR_STATE; }
        if (!short_rows && use_es) return es.run_rows(x, y, rb, re, s);
        if (!short_rows) return ts.run_rows(x, y, CS_OVERWRITE, rb, re, s);
        if (rb < 0 || re > nRow || rb > re) { set_error("multiply_rows: bad row range [%d,%d)", rb, re); return B200SPMV_ERR_INVALID; }
        if (rb == re) return B200SPMV_OK;
        if (use_rbs) return rowblock_spmv(ptr.p, idx.p, f32 ? (const void *)val32.p : (const void *)val.p, f32, maxLen, rb, re, x, y, s);
        return cs.run(x, y, rb, re, CS_OVERWRITE, s);
    }
    bool has_rows() const override { return !prec; }   // multiply_rows has no fp32-vector variant
    int prepare_rows(int rb, int re) override { return short_rows ? B200SPMV_OK : use_es ? es.prepare(rb, re) : ts.prepare(rb, re); }
    int col_extent(int rb, int re, int *cmin, int *cmax) override
    {
        if (rb < 0 || re > nRow || rb > re) { set_error("col_extent: bad row range [%d,%d)", rb, re); return B200SPMV_ERR_INVALID; }
        int pb = 0, pe = 0;
        B2_CUDA(cudaMemcpy(&pb, ptr.p + rb, sizeof(int), cudaMemcpyDeviceToHost));
        B2_CUDA(cudaMemcpy(&pe, ptr.p + re, sizeof(int), cudaMemcpyDeviceToHost));
        if (pe <= pb) { *cmin = 0; *cmax = -1; return B200SPMV_OK; }       // no entries: needs nothing of x
        return minmax_i32(idx.p, pb, pe, cmin, cmax);
    }

    bool scalar(const std::string &n, long long *out) override
    {
        if (n == "alg_bytes") {   // SURVEY.md 8d: 12 nnz + 4 (nRow+1) + 8 nCol + 8 nRow
            *out = (f32 ? 8LL : 12LL) * nnz + 4LL * (nRow + 1) + (prec ? 4LL : 8LL) * ((long long)nCol + nRow);
            return true;
        }
        if (n == "launches") { *out = short_rows ? 1 : use_es ? (es.nTiles > 1 ? 2 : 1) + (es.nEmpty ? 1 : 0) : (ts.nTiles > 1 ? 2 : 1); return true; }
        if (n == "crs_kernel") { *out = short_rows ? 1 : use_es ? (es.tma ? 2 : 3) : 0; return true; }   // 0 tile-stream, 1 row-chunk stream, 2 / 3 entry stream (TMA- / load-fed)
        if (n == "maxLength") { *out = maxLen; return true; }
        if (n == "short_row_path") { *out = short_rows ? 1 : 0; return true; }
        if (n == "chunk_feed") { *out = short_rows && !use_rbs ? cs.feed : CS_FEED_IDX; return true; }   // row-chunk stream: 0 idx / ptr, 1 offset dictionary
        if (n == "nTiles") { *out = ts.nTiles; return true; }
        if (n == "value_f32") { *out = f32 ? 1 : 0; return true; }
        if (n == "precision") { *out = prec; return true; }
        return false;
    }

    long long array(const std::string &n, void *dst, long long cap) override
    {
        if (n == "ptr") return export_device(ptr.p, ptr.bytes(), dst, cap);
        if (n == "idx") return export_device(idx.p, sizeof(int) * (size_t)nnz, dst, cap);
        if (n == "val") {
            if (!f32) return export_device(val.p, sizeof(double) * (size_t)nnz, dst, cap);
            if (!dst) return (long long)(sizeof(double) * (size_t)nnz);
            DevBuf<double> w;
            if (w.alloc((size_t)nnz)) return B200SPMV_ERR_NOMEM;
            if (nnz) crs_to_f64_kernel<<<ceil_div(nnz, 256), 256>>>(val32.p, nnz, w.p);
            return export_device(w.p, w.bytes(), dst, cap);
        }
        return -1000;
    }
};

Format *make_crs(const b200spmv_options &o) { return new CrsFormat(o); }

}  // namespace b2
