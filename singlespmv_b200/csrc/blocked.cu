// blocked.cu -- matrices with more than 2^31-1 non-zeros on ONE GPU (SURVEY.md 8f: the 64-bit index variant).
// The reference is int32 throughout (SpMat::nNnz is an int, src/util.h:8); its INDEX_64 switch (src/param.h:1-7) only
// widens the SS / CSS col_idx arrays.  A B200 holds 180 GB, i.e. ~10^10 CRS entries, so the limit that matters here is
// the 32-bit entry offset, not memory.  Instead of 64-bit offsets in every kernel (half the row-pointer bandwidth, and
// 64-bit address arithmetic in the inner loops), the matrix is cut into contiguous ROW BLOCKS of fewer than 2^31 entries
// each; every block is an ordinary matrix of the requested format over the full column range, with its own 32-bit
// offsets, multiplied into its slice of y.  Rows are never split, so every row is summed exactly as without blocks.
#include <algorithm>
#include <cstdlib>

#include "common.cuh"

namespace b2 {

Format *make_format(int format, const b200spmv_options &o);   // api.cu

namespace {

__global__ void shift_rows_kernel(const int *__restrict__ row, long long n, int by, int *__restrict__ out)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = row[i] - by;
}

// first entry e with row[e] >= r (row sorted), one thread per query
__global__ void row_lower_bound_kernel(const int *__restrict__ row, long long nnz, const int *__restrict__ q, int nq,
                                       long long *__restrict__ out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nq) return;
    long long lo = 0, hi = nnz;
    while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        if (row[mid] < q[i]) lo = mid + 1;
        else hi = mid;
    }
    out[i] = lo;
}

struct RowBlocked : Format {
    int format;
    b200spmv_options opt;
    long long nnz64 = 0;
    std::vector<std::unique_ptr<Format>> blk;
    std::vector<int> rb;                                      // nBlocks + 1 row bounds

    RowBlocked(int f, const b200spmv_options &o) : format(f), opt(o) {}
    int convert(const CooView &, cudaStream_t) override
    {
        set_error("row-blocked matrix: use convert64");
        return B200SPMV_ERR_STATE;
    }

    int convert64(int nRow_, int nCol_, long long nnzAll, const int *row_d, const int *col_d, const double *val_d,
                  long long limit, cudaStream_t s)
    {
        nRow = nRow_; nCol = nCol_; nnz64 = nnzAll;
        nnz = (int)std::min<long long>(nnzAll, 0x7fffffffLL);
        const int parts = (int)std::max<long long>(1, (nnzAll + limit - 1) / limit);
        std::vector<int> bounds((size_t)parts + 1);
        B2_TRY(b200spmv_partition_rows(row_d, nnzAll, nRow, parts, bounds.data()));
        // entry range of every block
        DevBuf<int> q;
        DevBuf<long long> pos;
        B2_TRY(q.alloc((size_t)parts + 1));
        B2_TRY(pos.alloc((size_t)parts + 1));
        B2_CUDA(cudaMemcpyAsync(q.p, bounds.data(), sizeof(int) * ((size_t)parts + 1), cudaMemcpyHostToDevice, s));
        row_lower_bound_kernel<<<ceil_div(parts + 1, 64), 64, 0, s>>>(row_d, nnzAll, q.p, parts + 1, pos.p);
        B2_KERNEL_CHECK();
        std::vector<long long> e((size_t)parts + 1);
        B2_CUDA(cudaMemcpyAsync(e.data(), pos.p, sizeof(long long) * ((size_t)parts + 1), cudaMemcpyDeviceToHost, s));
        B2_CUDA(cudaStreamSynchronize(s));
        e[(size_t)parts] = nnzAll;
        blk.clear();
        rb.assign(1, 0);
        for (int g = 0; g < parts; g++) {
            const int r0 = bounds[(size_t)g], r1 = bounds[(size_t)g + 1];
            if (r1 <= r0) continue;
            const long long n = e[(size_t)g + 1] - e[(size_t)g];
            if (n > 0x7fffffffLL) { set_error("row-blocked matrix: rows [%d,%d) hold %lld entries (a single row block must stay below 2^31)", r0, r1, n); return B200SPMV_ERR_UNSUPPORTED; }
            DevBuf<int> local;
            B2_TRY(local.alloc((size_t)n));
            if (n) shift_rows_kernel<<<ceil_div(n, 256), 256, 0, s>>>(row_d + e[(size_t)g], n, r0, local.p);
            B2_KERNEL_CHECK();
            std::unique_ptr<Format> f(make_format(format, opt));
            CooView A{r1 - r0, nCol, (int)n, local.p, col_d + e[(size_t)g], val_d + e[(size_t)g], r0};
            B2_TRY(f->convert(A, s));
            B2_CUDA(cudaStreamSynchronize(s));
            blk.push_back(std::move(f));
            rb.push_back(r1);
        }
        if (rb.back() != nRow) { set_error("row-blocked matrix: partition does not cover the rows"); return B200SPMV_ERR_STATE; }
        return B200SPMV_OK;
    }

    int multiply(const double *x, double *y, cudaStream_t s) override
    {
        for (size_t g = 0; g < blk.size(); g++) B2_TRY(blk[g]->multiply(x, y + rb[g], s));
        return B200SPMV_OK;
    }
    int multiply_f32(const float *x, float *y, cudaStream_t s) override
    {
        for (size_t g = 0; g < blk.size(); g++) B2_TRY(blk[g]->multiply_f32(x, y + rb[g], s));
        return B200SPMV_OK;
    }
    int multiply_multi(int k, const double *X, long long ldx, double *Y, long long ldy, cudaStream_t s) override
    {
        for (size_t g = 0; g < blk.size(); g++) B2_TRY(blk[g]->multiply_multi(k, X, ldx, Y + (long long)rb[g] * ldy, ldy, s));
        return B200SPMV_OK;
    }
    int multiply_multi_f32(int k, const float *X, long long ldx, float *Y, long long ldy, cudaStream_t s) override
    {
        for (size_t g = 0; g < blk.size(); g++) B2_TRY(blk[g]->multiply_multi_f32(k, X, ldx, Y + (long long)rb[g] * ldy, ldy, s));
        return B200SPMV_OK;
    }
    bool has_rows() const override
    {
        for (auto &b : blk) if (!b->has_rows()) return false;
        return !blk.empty();
    }
    template <typename F> int for_range(int r0, int r1, F fn)
    {
        if (r0 < 0 || r1 > nRow || r0 > r1) { set_error("row range [%d,%d) outside the %d rows", r0, r1, nRow); return B200SPMV_ERR_INVALID; }
        for (size_t g = 0; g < blk.size(); g++) {
            const int lo = std::max(r0, rb[g]), hi = std::min(r1, rb[g + 1]);
            if (hi > lo) B2_TRY(fn(g, lo - rb[g], hi - rb[g]));
        }
        return B200SPMV_OK;
    }
    int multiply_rows(int r0, int r1, const double *x, double *y, cudaStream_t s) override
    {
        return for_range(r0, r1, [&](size_t g, int lo, int hi) { return blk[g]->multiply_rows(lo, hi, x, y + rb[g], s); });
    }
    int prepare_rows(int r0, int r1) override
    {
        return for_range(r0, r1, [&](size_t g, int lo, int hi) { return blk[g]->prepare_rows(lo, hi); });
    }
    int col_extent(int r0, int r1, int *cmin, int *cmax) override
    {
        int mn = nCol, mx = -1;
        B2_TRY(for_range(r0, r1, [&](size_t g, int lo, int hi) {
            int a = 0, b = -1;
            B2_TRY(blk[g]->col_extent(lo, hi, &a, &b));
            if (b >= a) { mn = std::min(mn, a); mx = std::max(mx, b); }
            return (int)B200SPMV_OK;
        }));
        *cmin = mn; *cmax = mx;
        return B200SPMV_OK;
    }
    bool scalar(const std::string &n, long long *out) override
    {
        if (n == "nNnz") { *out = nnz64; return true; }
        if (n == "row_blocks") { *out = (long long)blk.size(); return true; }
        if (n == "alg_bytes" || n == "launches") {            // x is read once however many blocks there are
            long long sum = 0;
            for (auto &b : blk) {
                long long v = 0;
                if (!b->scalar(n, &v)) return false;
                sum += v;
            }
            if (n == "alg_bytes" && !blk.empty()) sum -= 8LL * nCol * (long long)(blk.size() - 1) / (opt.precision ? 2 : 1);
            *out = sum;
            return true;
        }
        return blk.empty() ? false : blk[0]->scalar(n, out);   // per-block quantities: those of the first block
    }
    long long array(const std::string &, void *, long long) override
    {
        set_error("get_array: a row-blocked matrix (more than 2^31-1 entries) exports no arrays");
        return B200SPMV_ERR_UNSUPPORTED;
    }
};

}  // namespace

// limit: entries per row block; 0 = the default (B200SPMV_BLOCK_NNZ, else 0x70000000: room for the rounding of a split
// to whole rows)
int convert_row_blocked(int format, const b200spmv_options &opt, int nRow, int nCol, long long nnz, const int *row_d,
                        const int *col_d, const double *val_d, cudaStream_t s, std::unique_ptr<Format> &out)
{
    const long long env = getenv("B200SPMV_BLOCK_NNZ") ? atoll(getenv("B200SPMV_BLOCK_NNZ")) : 0;   // read per call: tests switch it
    const long long limit = env > 0 ? std::min<long long>(env, 0x70000000LL) : 0x70000000LL;
    std::unique_ptr<RowBlocked> f(new RowBlocked(format, opt));
    B2_TRY(f->convert64(nRow, nCol, nnz, row_d, col_d, val_d, limit, s));
    out = std::move(f);
    return B200SPMV_OK;
}

long long row_block_limit()
{
    const long long env = getenv("B200SPMV_BLOCK_NNZ") ? atoll(getenv("B200SPMV_BLOCK_NNZ")) : 0;
    return env > 0 ? std::min<long long>(env, 0x70000000LL) : 0x7fffffffLL;
}

}  // namespace b2
