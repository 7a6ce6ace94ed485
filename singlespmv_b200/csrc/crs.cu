// crs.cu -- CRS plugin: device conversion + adaptive multiply (row-chunk stream for short rows, entry stream for
// gather-bound matrices, tile-stream otherwise).
// Reference: /root/reference/src/opt_crs.{h,cpp} (SpMatOpt{ptr,idx,val}; OptimizeProblem :10-42; SpMV :44-70).
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

struct CrsFormat : Format {
    int maxLen = 0;
    bool short_rows = false;
    DevBuf<int> ptr, idx;
    DevBuf<double> val;
    DevBuf<float> val32;
    bool f32;
    TileStream ts;
    ChunkStream cs;
    EntryStream es;
    bool use_es = false;
    int path_opt;
    int band = 0, rowOffset = 0;
    bool band_known = false;              // conversion computes the band for crs_path 0 and 4 only
    int prec;                             // options.precision: 0 fp64 vectors, 1 fp32 vectors + sums, 2 fp32 vectors, fp64 sums
    explicit CrsFormat(const b200spmv_options &o) : f32(o.value_f32 != 0 || o.precision != 0), path_opt(o.crs_path), prec(o.precision) {}

    int convert(const CooView &A, cudaStream_t s) override
    {
        nRow = A.nRow; nCol = A.nCol; nnz = A.nnz;
        rowOffset = A.rowOffset;
        // the entry stream borrows ptr / idx / val, which are reallocated below; the multi-vector multiplies build it
        // lazily on tile-stream handles and must find nothing of an earlier matrix
        es.reset();
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
        // path: 1 = tile-stream always; otherwise the TMA-fed row-chunk stream when the rows are short enough, else the tile-stream
        // ... unless the gathers range over tens of MB (uniform random, R-MAT): x must stay in L2, which it does with the
        // tile-stream's evict-first loads and does not with bulk copies in flight (uniform 2^24 x 11: 40 G entries/s TMA-fed)
        band = 0;
        band_known = path_opt == 0 || path_opt == 4;
        if (band_known) B2_TRY(max_band(A.row, A.col, nnz, A.rowOffset, &band, s));
        short_rows = path_opt != 1 && path_opt != 4 && cs.ok && !gathers_need_l2(band);
        // gather-bound matrices (fp64): the load-fed entry stream (entry_stream.cuh) -- c3 441 GFLOP/s against 365 for the tile-stream
        // (cuSPARSE CSR: 405).  Banded matrices with medium rows keep the tile-stream: the TMA-fed entry stream is level with it
        // (c4: 659 against 642) and the tile-stream sums rows of up to 64 entries in the reference's order.  crs_path = 4 forces the
        // entry stream, crs_path = 1 the tile-stream.
        use_es = false;
        if (!short_rows && !f32 && !prec && (path_opt == 4 || (path_opt == 0 && gathers_need_l2(band)))) {
            B2_TRY(es.build(ptr.p, idx.p, val.p, false, nRow, nnz, gathers_need_l2(band), s));
            use_es = es.ok;
        }
        B2_CUDA(cudaStreamSynchronize(s));
        return B200SPMV_OK;
    }

    int multiply(const double *x, double *y, cudaStream_t s) override { return multiply_rows(0, nRow, x, y, s); }
    int multiply_f32(const float *x, float *y, cudaStream_t s) override
    {
        if (!prec) { set_error("multiply_f32: the handle was created with precision = 0 (fp64 vectors)"); return B200SPMV_ERR_STATE; }
        if (short_rows) return cs.run_f32(x, y, 0, nRow, CS_OVERWRITE, prec == 2, s);
        return ts.run_rows_f32(x, y, CS_OVERWRITE, 0, nRow, prec == 2, s);
    }

    int multiply_rows(int rb, int re, const double *x, double *y, cudaStream_t s) override
    {
        if (prec) { set_error("multiply: the handle was created with precision = %d, use b200spmv_multiply_f32", prec); return B200SPMV_ERR_STATE; }
        if (!short_rows && use_es) return es.run_rows(x, y, rb, re, s);
        if (!short_rows) return ts.run_rows(x, y, CS_OVERWRITE, rb, re, s);
        if (rb < 0 || re > nRow || rb > re) { set_error("multiply_rows: bad row range [%d,%d)", rb, re); return B200SPMV_ERR_INVALID; }
        if (rb == re) return B200SPMV_OK;
        return cs.run(x, y, rb, re, CS_OVERWRITE, s);
    }
    // Row-chunk stream and entry stream handles run their own kernel's K-vector form.  Tile-stream handles (rows longer
    // than the row-chunk stream takes, crs_path = 1) run the entry stream's, whose metadata the first call builds.
    int multiply_multi(int k, const double *X, long long ldx, double *Y, long long ldy, cudaStream_t s) override
    {
        if (f32) { set_error("multiply_multi: fp64 values and vectors only (value_f32 = 0, precision = 0)"); return B200SPMV_ERR_UNSUPPORTED; }
        if (short_rows) return cs.run_multi(k, X, ldx, Y, ldy, s);
        if (nnz == 0) return zero_rows_multi(nRow, k, Y, ldy, s);
        if (!use_es && !es.ok) {
            cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
            if (cudaStreamIsCapturing(s, &cap) == cudaSuccess && cap != cudaStreamCaptureStatusNone) {
                set_error("multiply_multi: first call on a tile-stream handle inside a stream capture; call it once outside the capture first");
                return B200SPMV_ERR_STATE;
            }
            B2_TRY(ensure_band(s));
            B2_TRY(es.build(ptr.p, idx.p, val.p, false, nRow, nnz, gathers_need_l2(band), s));
        }
        return es.run_multi(k, X, ldx, Y, ldy, s);
    }
    // The fp32-vector form (precision 1 / 2): row-chunk stream handles run its K-vector form, every other handle (the
    // single multiply runs the tile-stream there) the entry stream on val32, whose metadata the first call builds.
    int multiply_multi_f32(int k, const float *X, long long ldx, float *Y, long long ldy, cudaStream_t s) override
    {
        if (!prec) { set_error("multiply_multi_f32: the handle was created with precision = 0 (fp64 vectors), use b200spmv_multiply_multi"); return B200SPMV_ERR_STATE; }
        if (short_rows) return cs.run_multi_f32(k, X, ldx, Y, ldy, prec == 2, s);
        if (nnz == 0) return zero_rows_multi(nRow, k, Y, ldy, s);
        if (!es.ok) {
            cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
            if (cudaStreamIsCapturing(s, &cap) == cudaSuccess && cap != cudaStreamCaptureStatusNone) {
                set_error("multiply_multi_f32: first call on this handle inside a stream capture; call it once outside the capture first");
                return B200SPMV_ERR_STATE;
            }
            B2_TRY(ensure_band(s));
            B2_TRY(es.build(ptr.p, idx.p, val32.p, true, nRow, nnz, gathers_need_l2(band), s));
        }
        return es.run_multi_f32(k, X, ldx, Y, ldy, prec == 2, s);
    }
    int ensure_band(cudaStream_t s)
    {
        if (!band_known) B2_TRY(max_band_crs(ptr.p, idx.p, nRow, rowOffset, &band, s));
        band_known = true;
        return B200SPMV_OK;
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
        if (n == "multi_kernel") {   // b200spmv_multiply_multi: 1 row-chunk stream, 2 / 3 entry stream TMA- / load-fed, 0 none
            if (f32) *out = 0;
            else if (short_rows) *out = 1;
            else if (use_es) *out = es.tma ? 2 : 3;
            else {
                if (ensure_band(nullptr) != B200SPMV_OK) return false;
                *out = gathers_need_l2(band) ? 3 : 2;
            }
            return true;
        }
        if (n == "multi_kernel_f32") {   // b200spmv_multiply_multi_f32: the same numbering, 0 on precision-0 handles and
            if (!prec || nnz == 0) *out = 0;                     // without entries (Y is only zero-filled)
            else if (short_rows) *out = 1;
            else {
                if (ensure_band(nullptr) != B200SPMV_OK) return false;
                *out = gathers_need_l2(band) ? 3 : 2;
            }
            return true;
        }
        if (n == "maxLength") { *out = maxLen; return true; }
        if (n == "short_row_path") { *out = short_rows ? 1 : 0; return true; }
        if (n == "chunk_feed") { *out = short_rows ? cs.feed : CS_FEED_IDX; return true; }   // row-chunk stream: 0 idx / ptr, 1 offset dictionary
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
