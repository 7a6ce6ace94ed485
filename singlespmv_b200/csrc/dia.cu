// dia.cu -- DIA plugin.  Logical content = the reference's DIA (/root/reference/src/opt_dia.cpp:
// diagonal id d = col - row + (nRow-1) :21-28, ioff = ascending non-empty ids :35-45, diag[p][col]
// dense and zero-filled :47-56, multiply accumulating diagonal by diagonal :83-92).
//
// Device layout: diag_r[p][row] (indexed by ROW, leading dimension padded to 32 doubles), so that a
// CTA's slice of every diagonal starts on a 256-byte boundary whatever the offset; the export maps it
// back to the reference's [nDiag][nCol] column-indexed arrays.
//
// Multiply: one CTA per block of DIA_R rows, one thread per row (DIA_RPT rows per thread, strided by
// the CTA width -> every warp request is a contiguous 256-byte run).  Consecutive diagonals (ioff
// runs) read overlapping windows of x: each run's window is staged ONCE per CTA in shared memory by a
// 1-D TMA bulk copy (cp.async.bulk + mbarrier transaction count), so a 27-point stencil pulls 9
// windows from L2 instead of 27.  Per row the diagonals are accumulated in ascending order with
// unfused mul/add = the reference's order (and, padding zeros aside, opt_crs.cpp's) -> bit-identical y.
#include <algorithm>
#include <set>

#include "common.cuh"

namespace b2 {

constexpr int DIA_THREADS = 256;
constexpr int DIA_RPT = 2;
constexpr int DIA_R = DIA_THREADS * DIA_RPT;
constexpr int DIA_MAX_DIAG = 64;     // TMA variant: per-diagonal window bases live in shared memory
constexpr int DIA_MAX_RUNS = 16;
constexpr int DIA_MAX_SMEM = 200 * 1024;   // TMA variant: largest x-window staging a handle may ask for

struct DiaRuns {
    int n;
    int off[DIA_MAX_RUNS];    // col - row of the run's first diagonal
    int p0[DIA_MAX_RUNS];     // first diagonal of the run
    int cnt[DIA_MAX_RUNS];    // diagonals in the run
    int soff[DIA_MAX_RUNS];   // start of the run's window in shared memory (doubles, even)
};

// ---------------------------------------------------------------- conversion kernels
__global__ void dia_flag_kernel(const int *__restrict__ row, const int *__restrict__ col, int nnz, int shift,
                                int *__restrict__ flag)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nnz) flag[col[i] - row[i] + shift] = 1;           // opt_dia.cpp:26 (benign same-value race)
}

__global__ void dia_ioff_kernel(const int *__restrict__ flag, const int *__restrict__ slot, int N,
                                int *__restrict__ ioff)
{
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d < N && flag[d]) ioff[slot[d]] = d;                  // opt_dia.cpp:38-44
}

template <typename VT>
__global__ void dia_scatter_kernel(const int *__restrict__ row, const int *__restrict__ col,
                                   const double *__restrict__ val, int nnz, int shift,
                                   const int *__restrict__ slot, size_t ld, VT *__restrict__ diag)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nnz) diag[(size_t)slot[col[i] - row[i] + shift] * ld + row[i]] = (VT)val[i];   // opt_dia.cpp:52-54 (fp32 storage: rounded once)
}

// reference layout diag[p][col]: the entry of row col - off_p, zero where that row does not exist
template <typename VT>
__global__ void dia_logical_kernel(const VT *__restrict__ diag, size_t ld, const int *__restrict__ ioff,
                                   int nDiag, int nRow, int nCol, double *__restrict__ out)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)nDiag * nCol) return;
    const int p = (int)(i / nCol), c = (int)(i % nCol);
    const int r = c + (nRow - 1) - ioff[p];
    out[i] = (r >= 0 && r < nRow) ? (double)diag[(size_t)p * ld + r] : 0.0;
}

// window of run g for the CTA starting at row0: columns [c_lo, c_hi), smem index = col - w0
struct DiaWindow {
    int w0, s_begin, s_end, a_begin, a_end, len;
};
__device__ __forceinline__ DiaWindow dia_window(int row0, int off, int cnt, int nCol)
{
    DiaWindow w;
    const int c_lo = row0 + off, c_hi = row0 + off + DIA_R + cnt - 1;
    w.w0 = c_lo & ~1;                                   // floor to even (two's complement, negatives too)
    w.len = c_hi - w.w0;
    w.s_begin = max(c_lo, 0);
    w.s_end = min(c_hi, nCol);
    if (w.s_begin >= w.s_end) { w.s_begin = w.s_end = w.a_begin = w.a_end = w.w0; return w; }
    w.a_begin = (w.s_begin + 1) & ~1;
    w.a_end = w.s_end & ~1;
    if (w.a_begin >= w.a_end) w.a_begin = w.a_end = w.s_begin;   // nothing for the TMA unit
    return w;
}

// ---------------------------------------------------------------- multiply, TMA-staged x
template <int DU, int MINB>
__global__ void __launch_bounds__(DIA_THREADS, MINB)
dia_spmv_tma_kernel(const double *__restrict__ diag, size_t ld, int nDiag, const DiaRuns runs,
                    const double *__restrict__ x, double *__restrict__ y, int rowBegin, int rowEnd, int nCol)
{
    extern __shared__ __align__(16) double xs[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ int dbase[DIA_MAX_DIAG];

    const int tid = threadIdx.x;
    const int row0 = rowBegin + blockIdx.x * DIA_R;
    const uint64_t pol_x = policy_evict_last(), pol_stream = policy_evict_first();

    if (tid == 0) mbar_init(&bar, 1);
    __syncthreads();
    if (tid == 0) {
        uint32_t total = 0;
        for (int g = 0; g < runs.n; g++) {
            const DiaWindow w = dia_window(row0, runs.off[g], runs.cnt[g], nCol);
            total += (uint32_t)(w.a_end - w.a_begin) * 8u;
        }
        mbar_expect_tx(&bar, total);
        for (int g = 0; g < runs.n; g++) {
            const DiaWindow w = dia_window(row0, runs.off[g], runs.cnt[g], nCol);
            if (w.a_end > w.a_begin)
                tma_load_1d(xs + runs.soff[g] + (w.a_begin - w.w0), x + w.a_begin,
                            (uint32_t)(w.a_end - w.a_begin) * 8u, &bar, pol_x);
        }
    }
    // the few window slots the 16-byte-granular bulk copy cannot cover: unaligned edge elements are
    // loaded by threads, slots outside [0, nCol) (matrix border) are zero
    for (int g = 0; g < runs.n; g++) {
        const DiaWindow w = dia_window(row0, runs.off[g], runs.cnt[g], nCol);
        const int head = w.a_begin - w.w0, tail0 = w.a_end - w.w0;
        const int extra = head + (w.len - tail0);
        for (int i = tid; i < extra; i += DIA_THREADS) {
            const int pos = i < head ? i : tail0 + (i - head);
            const int c = w.w0 + pos;
            xs[runs.soff[g] + pos] = (c >= w.s_begin && c < w.s_end) ? x[c] : 0.0;
        }
    }
    for (int p = tid; p < nDiag; p += DIA_THREADS) {
        int g = 0;
        while (g + 1 < runs.n && runs.p0[g + 1] <= p) g++;
        const int c_lo = row0 + runs.off[g];
        dbase[p] = runs.soff[g] + (c_lo - (c_lo & ~1)) + (p - runs.p0[g]);
    }
    __syncthreads();

    const int rows = min(DIA_R, rowEnd - row0);
    const double *dp = diag + row0 + tid;
    double acc[DIA_RPT];
#pragma unroll
    for (int k = 0; k < DIA_RPT; k++) acc[k] = 0.0;

    if (rows == DIA_R) {
        // DIA_U x DIA_RPT independent 8-byte loads per thread per round; enough CTAs stay resident
        // (launch bounds below) that no software double buffer is needed
        constexpr int U = DU;
        double d[U][DIA_RPT];
        int p = 0;
#pragma unroll
        for (int u = 0; u < U; u++)
#pragma unroll
            for (int k = 0; k < DIA_RPT; k++)
                d[u][k] = (u < nDiag) ? ld_stream_d1(dp + (size_t)u * ld + k * DIA_THREADS, pol_stream) : 0.0;
        mbar_wait(&bar, 0);                 // the first round of diagonal values is in flight while the x windows land
        for (;;) {
            const int m = min(U, nDiag - p);
#pragma unroll
            for (int u = 0; u < U; u++)
                if (u < m) {
                    const double *xw = xs + dbase[p + u] + tid;
#pragma unroll
                    for (int k = 0; k < DIA_RPT; k++)
                        acc[k] = __dadd_rn(acc[k], __dmul_rn(d[u][k], xw[k * DIA_THREADS]));
                }
            p += U;
            if (p >= nDiag) break;
#pragma unroll
            for (int u = 0; u < U; u++)
#pragma unroll
                for (int k = 0; k < DIA_RPT; k++)
                    d[u][k] = (p + u < nDiag) ? ld_stream_d1(dp + (size_t)(p + u) * ld + k * DIA_THREADS, pol_stream) : 0.0;
        }
#pragma unroll
        for (int k = 0; k < DIA_RPT; k++) y[row0 + tid + k * DIA_THREADS] = acc[k];
    } else {
        mbar_wait(&bar, 0);
        for (int p = 0; p < nDiag; p++) {
            const double *xw = xs + dbase[p] + tid;
#pragma unroll
            for (int k = 0; k < DIA_RPT; k++)
                if (tid + k * DIA_THREADS < rows)
                    acc[k] = __dadd_rn(acc[k], __dmul_rn(ld_stream_d1(dp + (size_t)p * ld + k * DIA_THREADS, pol_stream),
                                                         xw[k * DIA_THREADS]));
        }
#pragma unroll
        for (int k = 0; k < DIA_RPT; k++)
            if (tid + k * DIA_THREADS < rows) y[row0 + tid + k * DIA_THREADS] = acc[k];
    }
}

// ---------------------------------------------------------------- multiply, x through L1/L2 (any number of diagonals)
__global__ void __launch_bounds__(DIA_THREADS)
dia_spmv_direct_kernel(const double *__restrict__ diag, size_t ld, int nDiag, const int *__restrict__ ioff,
                       const double *__restrict__ x, double *__restrict__ y, int rowBegin, int rowEnd, int nRow, int nCol)
{
    const int r = rowBegin + blockIdx.x * DIA_THREADS + threadIdx.x;
    if (r >= rowEnd) return;
    const uint64_t pol_x = policy_evict_last(), pol_stream = policy_evict_first();
    const int shift = nRow - 1;
    double acc = 0.0;
    int p = 0;
    for (; p + 4 <= nDiag; p += 4) {
        double d[4], xv[4];
#pragma unroll
        for (int u = 0; u < 4; u++) d[u] = ld_stream_d1(diag + (size_t)(p + u) * ld + r, pol_stream);
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int c = r + ioff[p + u] - shift;
            xv[u] = (c >= 0 && c < nCol) ? ld_x(x + c, pol_x) : 0.0;
        }
#pragma unroll
        for (int u = 0; u < 4; u++) acc = __dadd_rn(acc, __dmul_rn(d[u], xv[u]));
    }
    for (; p < nDiag; p++) {
        const int c = r + ioff[p] - shift;
        const double xv = (c >= 0 && c < nCol) ? ld_x(x + c, pol_x) : 0.0;
        acc = __dadd_rn(acc, __dmul_rn(ld_stream_d1(diag + (size_t)p * ld + r, pol_stream), xv));
    }
    y[r] = acc;
}

// fp32 variant (options.precision): fp32 diagonals and vectors, x through L1 / L2 (coalesced: lane = row), sums in AT
template <typename AT>
__global__ void __launch_bounds__(DIA_THREADS)
dia_spmv_f32_kernel(const float *__restrict__ diag, size_t ld, int nDiag, const int *__restrict__ ioff,
                    const float *__restrict__ x, float *__restrict__ y, int nRow, int nCol)
{
    const int r = blockIdx.x * DIA_THREADS + threadIdx.x;
    if (r >= nRow) return;
    const uint64_t pol_x = policy_evict_last();
    const int shift = nRow - 1;
    AT acc = (AT)0;
    int p = 0;
    for (; p + 4 <= nDiag; p += 4) {
        float d[4], xv[4];
#pragma unroll
        for (int u = 0; u < 4; u++) d[u] = __ldcs(diag + (size_t)(p + u) * ld + r);
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int c = r + ioff[p + u] - shift;
            xv[u] = (c >= 0 && c < nCol) ? ld_x(x + c, pol_x) : 0.0f;
        }
#pragma unroll
        for (int u = 0; u < 4; u++) acc = Arith<AT>::add(acc, Arith<AT>::mul((AT)d[u], (AT)xv[u]));
    }
    for (; p < nDiag; p++) {
        const int c = r + ioff[p] - shift;
        const float xv = (c >= 0 && c < nCol) ? ld_x(x + c, pol_x) : 0.0f;
        acc = Arith<AT>::add(acc, Arith<AT>::mul((AT)__ldcs(diag + (size_t)p * ld + r), (AT)xv));
    }
    y[r] = (float)acc;
}

// Windows beyond the default 48 KB of dynamic shared memory need the kernels' opt-in limit raised.  That limit belongs
// to the kernel on a device, not to a handle, so it is raised once per device to the largest size any handle may ask
// for: a handle converted later can never lower it below what a live handle launches with.
static int dia_tma_allow_max_smem()
{
    static std::set<int> raised;
    int dev = 0;
    B2_CUDA(cudaGetDevice(&dev));
    if (raised.count(dev)) return B200SPMV_OK;
    for (auto kern : {dia_spmv_tma_kernel<5, 6>, dia_spmv_tma_kernel<7, 5>, dia_spmv_tma_kernel<3, 8>})
        B2_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, DIA_MAX_SMEM));
    raised.insert(dev);
    return B200SPMV_OK;
}

struct DiaFormat : Format {
    int nDiag = 0;
    size_t ld = 0;
    DevBuf<int> ioff;
    DevBuf<double> diag;
    DevBuf<float> diag32;                 // options.precision = 1 / 2
    int prec = 0;
    explicit DiaFormat(const b200spmv_options &o) : prec(o.precision) {}
    DiaRuns runs{};
    int offMin = 0, offMax = 0;           // smallest / largest col - row over the stored diagonals
    bool tma_ok = false;
    size_t smem_bytes = 0;

    int convert(const CooView &A, cudaStream_t s) override
    {
        nRow = A.nRow; nCol = A.nCol; nnz = A.nnz;
        B2_TRY(validate_sorted_coo(A, s));
        const long long Nll = (long long)nRow + nCol - 1;
        if (Nll > 0x7ffffff0LL) { set_error("DIA: nRow+nCol-1 exceeds int32"); return B200SPMV_ERR_INVALID; }
        const int N = Nll > 0 ? (int)Nll : 0, shift = nRow - 1;
        DevBuf<int> flag, slot;
        B2_TRY(flag.alloc((size_t)N + 1));
        B2_TRY(slot.alloc((size_t)N + 1));
        B2_CUDA(cudaMemsetAsync(flag.p, 0, flag.bytes(), s));
        if (nnz) {
            dia_flag_kernel<<<ceil_div(nnz, 256), 256, 0, s>>>(A.row, A.col, nnz, shift, flag.p);
            B2_KERNEL_CHECK();
        }
        B2_TRY(exclusive_scan_i32(flag.p, slot.p, N + 1, s));
        B2_CUDA(cudaMemcpy(&nDiag, slot.p + N, sizeof(int), cudaMemcpyDeviceToHost));
        ld = ((size_t)nRow + 31) & ~(size_t)31;
        size_t freeB = 0, totalB = 0;
        B2_CUDA(cudaMemGetInfo(&freeB, &totalB));
        if ((double)nDiag * (double)ld * (prec ? 4.0 : 8.0) > (double)freeB * 0.95) {
            set_error("DIA: %d diagonals x %d rows = %.1f GB do not fit the free %.1f GB of HBM (the reference "
                      "allocates the same dense slab, src/opt_dia.cpp:47-51)", nDiag, nRow, nDiag * (double)ld * 8e-9, freeB * 1e-9);
            return B200SPMV_ERR_NOMEM;
        }
        B2_TRY(ioff.alloc((size_t)nDiag));
        if (prec) {
            B2_TRY(diag32.alloc((size_t)nDiag * ld));
            B2_CUDA(cudaMemsetAsync(diag32.p, 0, diag32.bytes(), s));
        } else {
            B2_TRY(diag.alloc((size_t)nDiag * ld));
            B2_CUDA(cudaMemsetAsync(diag.p, 0, diag.bytes(), s));
        }
        if (N) {
            dia_ioff_kernel<<<ceil_div(N, 256), 256, 0, s>>>(flag.p, slot.p, N, ioff.p);
            B2_KERNEL_CHECK();
        }
        if (nnz) {
            if (prec) dia_scatter_kernel<float><<<ceil_div(nnz, 256), 256, 0, s>>>(A.row, A.col, A.val, nnz, shift, slot.p, ld, diag32.p);
            else dia_scatter_kernel<double><<<ceil_div(nnz, 256), 256, 0, s>>>(A.row, A.col, A.val, nnz, shift, slot.p, ld, diag.p);
            B2_KERNEL_CHECK();
        }
        // runs of consecutive diagonals share one x window
        std::vector<int> h((size_t)nDiag);
        B2_CUDA(cudaStreamSynchronize(s));
        if (nDiag) B2_CUDA(cudaMemcpy(h.data(), ioff.p, sizeof(int) * (size_t)nDiag, cudaMemcpyDeviceToHost));
        offMin = nDiag ? h[0] - shift : 0;
        offMax = nDiag ? h[(size_t)nDiag - 1] - shift : 0;
        memset(&runs, 0, sizeof runs);
        tma_ok = nDiag > 0 && nDiag <= DIA_MAX_DIAG;
        int soff = 0;
        for (int p = 0; p < nDiag && tma_ok; p++) {
            if (p > 0 && h[p] == h[p - 1] + 1) {
                runs.cnt[runs.n - 1]++;
                continue;
            }
            if (runs.n == DIA_MAX_RUNS) { tma_ok = false; break; }
            runs.off[runs.n] = h[p] - shift;
            runs.p0[runs.n] = p;
            runs.cnt[runs.n] = 1;
            runs.n++;
        }
        if (tma_ok) {
            for (int g = 0; g < runs.n; g++) {
                runs.soff[g] = soff;
                soff += (DIA_R + runs.cnt[g] + 1 + 1) & ~1;       // window + alignment slack, kept even
            }
            smem_bytes = (size_t)soff * sizeof(double);
            if (smem_bytes > DIA_MAX_SMEM) tma_ok = false;
            else if (smem_bytes > 48 * 1024) B2_TRY(dia_tma_allow_max_smem());
        }
        return B200SPMV_OK;
    }

    int multiply(const double *x, double *y, cudaStream_t s) override { return multiply_rows(0, nRow, x, y, s); }
    int multiply_f32(const float *x, float *y, cudaStream_t s) override
    {
        if (!prec) { set_error("multiply_f32: the handle was created with precision = 0 (fp64 vectors)"); return B200SPMV_ERR_STATE; }
        if (nRow == 0) return B200SPMV_OK;
        if (nDiag == 0) { B2_CUDA(cudaMemsetAsync(y, 0, sizeof(float) * (size_t)nRow, s)); return B200SPMV_OK; }
        const int grid = ceil_div(nRow, DIA_THREADS);
        if (prec == 2) dia_spmv_f32_kernel<double><<<grid, DIA_THREADS, 0, s>>>(diag32.p, ld, nDiag, ioff.p, x, y, nRow, nCol);
        else dia_spmv_f32_kernel<float><<<grid, DIA_THREADS, 0, s>>>(diag32.p, ld, nDiag, ioff.p, x, y, nRow, nCol);
        B2_KERNEL_CHECK();
        return B200SPMV_OK;
    }
    bool has_rows() const override { return !prec; }
    int col_extent(int rb, int re, int *cmin, int *cmax) override
    {
        if (rb < 0 || re > nRow || rb > re) { set_error("col_extent: bad row range [%d,%d)", rb, re); return B200SPMV_ERR_INVALID; }
        if (rb == re || nDiag == 0) { *cmin = 0; *cmax = -1; return B200SPMV_OK; }
        *cmin = std::max(0, rb + offMin);
        *cmax = std::min(nCol - 1, re - 1 + offMax);
        return B200SPMV_OK;
    }

    int multiply_rows(int rb, int re, const double *x, double *y, cudaStream_t s) override
    {
        if (rb < 0 || re > nRow || rb > re) { set_error("multiply_rows: bad row range [%d,%d)", rb, re); return B200SPMV_ERR_INVALID; }
        if (prec) { set_error("multiply: the handle was created with precision = %d, use b200spmv_multiply_f32", prec); return B200SPMV_ERR_STATE; }
        if (rb == re) return B200SPMV_OK;
        if (nDiag == 0) {
            B2_CUDA(cudaMemsetAsync(y + rb, 0, sizeof(double) * (size_t)(re - rb), s));
            return B200SPMV_OK;
        }
        // diagonals per load round, measured (profiles/r1_experiments.md): 27 diagonals want 7 (c4: 0.99 of the copy
        // peak, 5 gives 0.88), 7 diagonals want 3 (c5: 1.06 vs 0.99), up to 5 diagonals go in one round
        const int du = nDiag >= 16 ? 7 : nDiag <= 5 ? 5 : 3;
        if (tma_ok && (reinterpret_cast<uintptr_t>(x) & 15) == 0) {
            const int grid = ceil_div(re - rb, DIA_R);
            if (du == 7) dia_spmv_tma_kernel<7, 5><<<grid, DIA_THREADS, smem_bytes, s>>>(diag.p, ld, nDiag, runs, x, y, rb, re, nCol);
            else if (du == 3) dia_spmv_tma_kernel<3, 8><<<grid, DIA_THREADS, smem_bytes, s>>>(diag.p, ld, nDiag, runs, x, y, rb, re, nCol);
            else dia_spmv_tma_kernel<5, 6><<<grid, DIA_THREADS, smem_bytes, s>>>(diag.p, ld, nDiag, runs, x, y, rb, re, nCol);
        }
        else
            dia_spmv_direct_kernel<<<ceil_div(re - rb, DIA_THREADS), DIA_THREADS, 0, s>>>(diag.p, ld, nDiag, ioff.p, x, y, rb, re, nRow, nCol);
        B2_KERNEL_CHECK();
        return B200SPMV_OK;
    }

    bool scalar(const std::string &n, long long *out) override
    {
        if (n == "nDiag") { *out = nDiag; return true; }
        if (n == "nRuns") { *out = runs.n; return true; }
        if (n == "tma") { *out = tma_ok ? 1 : 0; return true; }
        if (n == "alg_bytes") {   // SURVEY.md 8d: 8 nDiag nCol + 4 nDiag + 8 nCol + 8 nRow
            *out = (prec ? 4LL : 8LL) * ((long long)nDiag * nCol + nCol + nRow) + 4LL * nDiag;
            return true;
        }
        if (n == "launches") { *out = 1; return true; }
        if (n == "precision") { *out = prec; return true; }
        return false;
    }

    long long array(const std::string &n, void *dst, long long cap) override
    {
        if (n == "ioff") return export_device(ioff.p, ioff.bytes(), dst, cap);
        if (n == "diag") {
            const size_t cnt = (size_t)nDiag * nCol;
            if (!dst) return (long long)(cnt * sizeof(double));
            DevBuf<double> out;
            if (out.alloc(cnt)) return B200SPMV_ERR_NOMEM;
            if (cnt && prec) dia_logical_kernel<float><<<ceil_div((long long)cnt, 256), 256>>>(diag32.p, ld, ioff.p, nDiag, nRow, nCol, out.p);
            else if (cnt) dia_logical_kernel<double><<<ceil_div((long long)cnt, 256), 256>>>(diag.p, ld, ioff.p, nDiag, nRow, nCol, out.p);
            return export_device(out.p, cnt * sizeof(double), dst, cap);
        }
        return -1000;
    }
};

Format *make_dia(const b200spmv_options &o) { return new DiaFormat(o); }

}  // namespace b2
