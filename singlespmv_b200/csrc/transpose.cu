// transpose.cu -- the COO of A^T from the sorted COO of A (options.transpose = 1, b200spmv_convert_coo_device).
// A^T's triplets are A's with row and column swapped, sorted by (new row, new col) = (col, row).  The input is sorted by
// (row, col) without duplicates, so a STABLE sort on the column alone yields exactly that order: within one column the
// entries keep their ascending rows.  CUB's LSD radix sort is stable and deterministic (no atomics decide an order), so
// the result has the same bits on every run -- the host's np.lexsort((row, col)).  Entry counts and the payload (the
// entry's position in A) are 64-bit, so matrices beyond 2^31-1 entries transpose too; A^T is then converted in row
// blocks like any other matrix of that size (blocked.cu).
#include <cub/cub.cuh>

#include <algorithm>

#include "common.cuh"

namespace b2 {

// kernels outside an anonymous namespace keep their names stable for profiles
__global__ void transpose_iota_kernel(long long n, long long *__restrict__ out)
{
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        out[i] = i;
}

// A^T's column = A's row, A^T's value = A's value, taken at the entry's position in A
__global__ void transpose_gather_kernel(const long long *__restrict__ src, long long n, const int *__restrict__ row,
                                        const double *__restrict__ val, int *__restrict__ colT,
                                        double *__restrict__ valT)
{
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const long long e = src[i];
        colT[i] = row[e];
        valT[i] = val[e];
    }
}

static int grid_for(long long n) { return (int)std::min<long long>(std::max<long long>(ceil_div(n, 256), 1), 148LL * 16); }

// rowT / colT / valT receive nnz entries (A^T has nCol rows and nRow columns).  Scratch is freed before the return; the
// outputs are complete when the stream reaches them.
int transpose_coo(int nCol, long long nnz, const int *row_d, const int *col_d, const double *val_d, cudaStream_t s,
                  DevBuf<int> &rowT, DevBuf<int> &colT, DevBuf<double> &valT)
{
    B2_TRY(rowT.alloc((size_t)nnz));
    if (nnz == 0) {
        B2_TRY(colT.alloc(0));
        return valT.alloc(0);
    }
    DevBuf<long long> pos;
    {
        DevBuf<int> keyAlt;
        DevBuf<long long> posAlt;
        B2_TRY(keyAlt.alloc((size_t)nnz));
        B2_TRY(pos.alloc((size_t)nnz));
        B2_TRY(posAlt.alloc((size_t)nnz));
        B2_CUDA(cudaMemcpyAsync(rowT.p, col_d, sizeof(int) * (size_t)nnz, cudaMemcpyDeviceToDevice, s));
        transpose_iota_kernel<<<grid_for(nnz), 256, 0, s>>>(nnz, pos.p);
        B2_KERNEL_CHECK();
        int bits = 1;                                             // columns are in [0, nCol): sort only their bits
        while (bits < 31 && (1LL << bits) < nCol) bits++;
        // keys as unsigned: every column is >= 0, and no sign-bit twiddling is wanted on a partial bit range
        cub::DoubleBuffer<unsigned> keys(reinterpret_cast<unsigned *>(rowT.p), reinterpret_cast<unsigned *>(keyAlt.p));
        cub::DoubleBuffer<long long> vals(pos.p, posAlt.p);
        size_t tmp = 0;
        B2_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp, keys, vals, nnz, 0, bits, s));
        DevBuf<char> t;
        B2_TRY(t.alloc(tmp));
        B2_CUDA(cub::DeviceRadixSort::SortPairs(t.p, tmp, keys, vals, nnz, 0, bits, s));
        // the sorted halves may have ended in the alternate buffers: keep those, free the others
        if (keys.Current() != reinterpret_cast<unsigned *>(rowT.p)) std::swap(rowT.p, keyAlt.p);
        if (vals.Current() != pos.p) std::swap(pos.p, posAlt.p);
        B2_CUDA(cudaStreamSynchronize(s));                        // the scratch is freed below
    }
    B2_TRY(colT.alloc((size_t)nnz));
    B2_TRY(valT.alloc((size_t)nnz));
    transpose_gather_kernel<<<grid_for(nnz), 256, 0, s>>>(pos.p, nnz, row_d, val_d, colT.p, valT.p);
    B2_KERNEL_CHECK();
    B2_CUDA(cudaStreamSynchronize(s));
    return B200SPMV_OK;
}

}  // namespace b2
