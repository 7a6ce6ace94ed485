// primitives.cu -- error state and the device passes every conversion is composed of.
#include <algorithm>
#include <cub/cub.cuh>

#include "common.cuh"

namespace b2 {

static thread_local std::string g_error;

void set_error(const char *fmt, ...)
{
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_error = buf;
}
void clear_error() { g_error.clear(); }
const char *last_error_cstr() { return g_error.c_str(); }

long long export_device(const void *src_d, size_t bytes, void *dst_h, long long dst_bytes)
{
    if (!dst_h) return (long long)bytes;
    if (dst_bytes < (long long)bytes) {
        set_error("get_array: destination holds %lld bytes, %zu needed", dst_bytes, bytes);
        return B200SPMV_ERR_INVALID;
    }
    if (bytes) {
        cudaError_t e = cudaMemcpy(dst_h, src_d, bytes, cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) {
            set_error("get_array: cudaMemcpy D2H: %s", cudaGetErrorString(e));
            return B200SPMV_ERR_CUDA;
        }
    }
    return (long long)bytes;
}

long long export_host(const void *src_h, size_t bytes, void *dst_h, long long dst_bytes)
{
    if (!dst_h) return (long long)bytes;
    if (dst_bytes < (long long)bytes) {
        set_error("get_array: destination holds %lld bytes, %zu needed", dst_bytes, bytes);
        return B200SPMV_ERR_INVALID;
    }
    if (bytes) memcpy(dst_h, src_h, bytes);
    return (long long)bytes;
}

// ---------------------------------------------------------------- row pointer
// Each ptr entry is written exactly once: entry i fills the rows in (row[i-1], row[i]], the
// virtual entry i == nnz fills (row[nnz-1], nRow].  Same result as the serial sweep of
// reference src/opt_crs.cpp:27-33.
__global__ void row_ptr_kernel(const int *__restrict__ row, int nnz, int nRow, int *__restrict__ ptr)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > nnz) return;
    int prev = i == 0 ? -1 : row[i - 1];
    int cur = i == nnz ? nRow : row[i];
    for (int r = prev + 1; r <= cur; r++) ptr[r] = i;
}

int build_row_ptr(const int *row_d, int nnz, int nRow, int *ptr_d, cudaStream_t s)
{
    row_ptr_kernel<<<ceil_div((long long)nnz + 1, 256), 256, 0, s>>>(row_d, nnz, nRow, ptr_d);
    B2_KERNEL_CHECK();
    return B200SPMV_OK;
}

__global__ void max_len_kernel(const int *__restrict__ ptr, int nRow, int *out)
{
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    int len = r < nRow ? ptr[r + 1] - ptr[r] : 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) len = max(len, __shfl_xor_sync(0xffffffffu, len, o));
    if ((threadIdx.x & 31) == 0 && len > 0) atomicMax(out, len);
}

int max_row_length(const int *ptr_d, int nRow, int *out_h, cudaStream_t s)
{
    DevBuf<int> m;
    B2_TRY(m.alloc(1));
    B2_CUDA(cudaMemsetAsync(m.p, 0, sizeof(int), s));
    if (nRow > 0) {
        max_len_kernel<<<ceil_div(nRow, 256), 256, 0, s>>>(ptr_d, nRow, m.p);
        B2_KERNEL_CHECK();
    }
    B2_CUDA(cudaMemcpyAsync(out_h, m.p, sizeof(int), cudaMemcpyDeviceToHost, s));
    B2_CUDA(cudaStreamSynchronize(s));
    return B200SPMV_OK;
}

template <typename T> static int exclusive_scan_t(const T *in_d, T *out_d, int n, cudaStream_t s)
{
    if (n <= 0) return B200SPMV_OK;
    size_t tmp = 0;
    B2_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp, in_d, out_d, n, s));
    DevBuf<char> t;
    B2_TRY(t.alloc(tmp));
    B2_CUDA(cub::DeviceScan::ExclusiveSum(t.p, tmp, in_d, out_d, n, s));
    B2_CUDA(cudaStreamSynchronize(s));   // temp storage dies with this frame
    return B200SPMV_OK;
}
int exclusive_scan_i32(const int *in_d, int *out_d, int n, cudaStream_t s) { return exclusive_scan_t(in_d, out_d, n, s); }
int exclusive_scan_i64(const long long *in_d, long long *out_d, int n, cudaStream_t s) { return exclusive_scan_t(in_d, out_d, n, s); }

// 64-bit sum of an int32 array (sizes that may pass 2^31); synchronises the stream
__global__ void sum_i64_kernel(const int *__restrict__ in, int n, unsigned long long *out)
{
    long long v = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) v += in[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(out, (unsigned long long)v);
}
int sum_i32_as_i64(const int *in_d, int n, long long *out_h, cudaStream_t s)
{
    DevBuf<unsigned long long> acc;
    B2_TRY(acc.alloc(1));
    B2_CUDA(cudaMemsetAsync(acc.p, 0, sizeof(unsigned long long), s));
    if (n > 0) {
        sum_i64_kernel<<<std::min(ceil_div(n, 256), 148 * 8), 256, 0, s>>>(in_d, n, acc.p);
        B2_KERNEL_CHECK();
    }
    B2_CUDA(cudaMemcpyAsync(out_h, acc.p, sizeof(long long), cudaMemcpyDeviceToHost, s));
    B2_CUDA(cudaStreamSynchronize(s));
    return B200SPMV_OK;
}

__global__ void minmax_kernel(const int *__restrict__ in, long long b, long long e, int *out)
{
    int mn = 0x7fffffff, mx = -0x7fffffff - 1;
    for (long long i = b + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < e; i += (long long)gridDim.x * blockDim.x) {
        const int v = in[i];
        if (v < 0) continue;                                   // ELL padding (ELL_PAD): references no column
        mn = min(mn, v);
        mx = max(mx, v);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    if ((threadIdx.x & 31) == 0) {
        atomicMin(&out[0], mn);
        atomicMax(&out[1], mx);
    }
}
int minmax_i32(const int *in_d, long long b, long long e, int *mn_h, int *mx_h)
{
    DevBuf<int> o;
    B2_TRY(o.alloc(2));
    int init[2] = {0x7fffffff, -0x7fffffff - 1};
    B2_CUDA(cudaMemcpy(o.p, init, sizeof init, cudaMemcpyHostToDevice));
    if (e > b) {
        minmax_kernel<<<(int)std::min<long long>((e - b + 255) / 256, 148 * 8), 256>>>(in_d, b, e, o.p);
        B2_KERNEL_CHECK();
    }
    B2_CUDA(cudaMemcpy(init, o.p, sizeof init, cudaMemcpyDeviceToHost));
    *mn_h = init[0];
    *mx_h = init[1];
    return B200SPMV_OK;
}

// largest |col - row| of a COO: how far apart the x entries of neighbouring rows lie.  Matrices whose gathers range over
// tens of MB depend on x staying in L2, which it does not while TMA bulk copies stream the matrix (profiles/r2_experiments.md):
// the formats use this to choose between their TMA-fed and their load-fed kernels.
__global__ void band_kernel(const int *__restrict__ row, const int *__restrict__ col, int nnz, int rowOffset, int *__restrict__ out)
{
    int m = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (long long)gridDim.x * blockDim.x)
        m = max(m, abs(col[i] - (row[i] + rowOffset)));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0 && m > 0) atomicMax(out, m);
}
int max_band(const int *row_d, const int *col_d, int nnz, int rowOffset, int *band_h, cudaStream_t s)
{
    *band_h = 0;
    if (nnz <= 0) return B200SPMV_OK;
    DevBuf<int> b;
    B2_TRY(b.alloc(1));
    B2_CUDA(cudaMemsetAsync(b.p, 0, sizeof(int), s));
    band_kernel<<<std::min(ceil_div(nnz, 256), 4096), 256, 0, s>>>(row_d, col_d, nnz, rowOffset, b.p);
    B2_KERNEL_CHECK();
    B2_CUDA(cudaMemcpyAsync(band_h, b.p, sizeof(int), cudaMemcpyDeviceToHost, s));
    B2_CUDA(cudaStreamSynchronize(s));
    return B200SPMV_OK;
}
__global__ void band_crs_kernel(const int *__restrict__ ptr, const int *__restrict__ idx, int nRow, int rowOffset,
                                int *__restrict__ out)
{
    int m = 0;
    for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < nRow; r += gridDim.x * blockDim.x) {
        const int b = ptr[r], e = ptr[r + 1];
        if (e > b) m = max(m, max(abs(idx[b] - (r + rowOffset)), abs(idx[e - 1] - (r + rowOffset))));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0 && m > 0) atomicMax(out, m);
}
int max_band_crs(const int *ptr_d, const int *idx_d, int nRow, int rowOffset, int *band_h, cudaStream_t s)
{
    *band_h = 0;
    if (nRow <= 0) return B200SPMV_OK;
    DevBuf<int> b;
    B2_TRY(b.alloc(1));
    B2_CUDA(cudaMemsetAsync(b.p, 0, sizeof(int), s));
    band_crs_kernel<<<std::min(ceil_div(nRow, 256), 4096), 256, 0, s>>>(ptr_d, idx_d, nRow, rowOffset, b.p);
    B2_KERNEL_CHECK();
    B2_CUDA(cudaMemcpyAsync(band_h, b.p, sizeof(int), cudaMemcpyDeviceToHost, s));
    B2_CUDA(cudaStreamSynchronize(s));
    return B200SPMV_OK;
}
bool gathers_need_l2(int band) { return 8LL * band > (32LL << 20); }

// ---------------------------------------------------------------- input contract
__global__ void validate_kernel(const int *__restrict__ row, const int *__restrict__ col, int nnz,
                                int nRow, int nCol, int *bad)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nnz) return;
    int r = row[i], c = col[i];
    bool wrong = r < 0 || r >= nRow || c < 0 || c >= nCol;
    if (i > 0 && !wrong) {
        int pr = row[i - 1], pc = col[i - 1];
        wrong = pr > r || (pr == r && pc >= c);
    }
    if (wrong) atomicMin(bad, i);
}

int validate_sorted_coo(const CooView &A, cudaStream_t s)
{
    if (A.nnz == 0) return B200SPMV_OK;
    DevBuf<int> bad;
    B2_TRY(bad.alloc(1));
    int init = 0x7fffffff, got = 0;
    B2_CUDA(cudaMemcpyAsync(bad.p, &init, sizeof(int), cudaMemcpyHostToDevice, s));
    validate_kernel<<<ceil_div(A.nnz, 256), 256, 0, s>>>(A.row, A.col, A.nnz, A.nRow, A.nCol, bad.p);
    B2_KERNEL_CHECK();
    B2_CUDA(cudaMemcpyAsync(&got, bad.p, sizeof(int), cudaMemcpyDeviceToHost, s));
    B2_CUDA(cudaStreamSynchronize(s));
    if (got != init) {
        set_error("convert: COO entry %d breaks the input contract (sorted by (row,col), no "
                  "duplicates, 0 <= row < nRow, 0 <= col < nCol; reference src/util.cpp:51)", got);
        return B200SPMV_ERR_INVALID;
    }
    return B200SPMV_OK;
}

}  // namespace b2
