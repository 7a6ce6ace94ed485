// ell.cu -- ELL plugin.  Logical content = the reference's ELLPACK (/root/reference/src/opt_ell.cpp:
// K = longest row :28-31, slot k >= len padded with col = k, val = 0 :46-52, multiply over all K
// slots :75-89).  Device layout = sliced ELL: slices of 32 rows (one warp), slice-local width
// rounded to V slots, stored [slice][k/V][lane][V] so that a lane reads V column ids and V
// values with 128-bit loads and a warp request is one contiguous 512 B / 1 KB run.
#include "colblocks.cuh"
#include "common.cuh"

namespace b2 {

// groups[s] = ceil(max row length in slice s / V)
// Row r holds the entries [beg[r], end[r]) of col / val: the whole row (beg = ptr, end = ptr + 1) or its part inside one
// column block (EllColBlocks below).
template <int V>
__global__ void ell_slice_groups_kernel(const int *__restrict__ beg, const int *__restrict__ end, int nRow, int nSlices,
                                        long long *__restrict__ groups)
{
    const int s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (s > nSlices) return;                       // s == nSlices: sentinel entry for the scan
    const int r = s * 32 + lane;
    int len = (s < nSlices && r < nRow) ? end[r] - beg[r] : 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) len = max(len, __shfl_xor_sync(0xffffffffu, len, o));
    if (lane == 0) groups[s] = (len + V - 1) / V;
}

// padCol: column of the slots beyond K (0 for the format's own layout; the first column of the block for a column block)
template <int V, typename VT>
__global__ void ell_fill_kernel(const int *__restrict__ beg, const int *__restrict__ end, const int *__restrict__ col,
                                const double *__restrict__ val, int nRow, int nSlices,
                                const long long *__restrict__ slice_off, int K, int padCol, int *__restrict__ ecol,
                                VT *__restrict__ eval)
{
    const int s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (s >= nSlices) return;
    const int r = s * 32 + lane;
    const long long g0 = slice_off[s], g1 = slice_off[s + 1];
    const int b = r < nRow ? beg[r] : 0, len = r < nRow ? end[r] - b : 0;
    for (long long g = g0; g < g1; g++)
#pragma unroll
        for (int j = 0; j < V; j++) {
            const int k = (int)(g - g0) * V + j;
            const size_t at = ((size_t)g * 32 + lane) * V + j;
            const bool real = k < len;
            // padding: col = slot index (opt_ell.cpp:48) for the reference's K slots; the extra slots that round a
            // slice up to V (k >= K, never exported) point at column 0 so that no gather leaves x when K is close to nCol
            ecol[at] = real ? col[b + k] : ((r < nRow && k < K) ? k : padCol);
            eval[at] = real ? (VT)val[b + k] : (VT)0;      // fp32 storage: rounded to nearest once, here
        }
}

template <int V, typename VT> struct EllGroup {
    int c[V];
    VT v[V];
};

template <int V>
__device__ __forceinline__ void ell_load(EllGroup<V, double> &g, const int *ecol, const double *eval, size_t at,
                                         uint64_t pol)
{
    if (V == 4) {
        int4 c = ld_stream_i4(ecol + at, pol);
        double2 a = ld_stream_d2(eval + at, pol), b = ld_stream_d2(eval + at + 2, pol);
        g.c[0] = c.x; g.c[1] = c.y; g.c[V - 2] = c.z; g.c[V - 1] = c.w;
        g.v[0] = a.x; g.v[1] = a.y; g.v[V - 2] = b.x; g.v[V - 1] = b.y;
    } else {
        int2 c = ld_stream_i2(ecol + at, pol);
        double2 a = ld_stream_d2(eval + at, pol);
        g.c[0] = c.x; g.c[1] = c.y;
        g.v[0] = a.x; g.v[1] = a.y;
    }
}
template <int V>
__device__ __forceinline__ void ell_load(EllGroup<V, float> &g, const int *ecol, const float *eval, size_t at,
                                         uint64_t pol)
{
    if (V == 4) {
        int4 c = ld_stream_i4(ecol + at, pol);
        float4 a;
        asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
                     : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w) : "l"(eval + at), "l"(pol));
        g.c[0] = c.x; g.c[1] = c.y; g.c[V - 2] = c.z; g.c[V - 1] = c.w;
        g.v[0] = a.x; g.v[1] = a.y; g.v[V - 2] = a.z; g.v[V - 1] = a.w;
    } else {
        int2 c = ld_stream_i2(ecol + at, pol);
        float2 a;
        asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v2.f32 {%0,%1}, [%2], %3;"
                     : "=f"(a.x), "=f"(a.y) : "l"(eval + at), "l"(pol));
        g.c[0] = c.x; g.c[1] = c.y;
        g.v[0] = a.x; g.v[1] = a.y;
    }
}


// One lane per row; the K-loop runs in ascending slot order with unfused mul/add, i.e. the
// reference's own order -> y is bit-identical to opt_ell.cpp / opt_crs.cpp (fp64).
// VT = stored value type, XT = type of x and y, AT = type of the products and the row sum.
__device__ __forceinline__ double ell_gather(const double *p, uint64_t pol, int xm)
{
    switch (xm) {
    case 1: return ld_x_mode<1>(p, pol);
    case 2: return ld_x_mode<2>(p, pol);
    case 3: return ld_x_mode<3>(p, pol);
    case 4: return ld_x_mode<4>(p, pol);
    case 5: return ld_x_mode<5>(p, pol);
    default: return ld_x_mode<0>(p, pol);
    }
}
__device__ __forceinline__ float ell_gather(const float *p, uint64_t pol, int) { return ld_x(p, pol); }

// ACC = CS_CONTINUE: the row sums continue what y holds (acc = y[r]; ...; y[r] = acc): the next column block of the same
// running sum.  ACC = CS_ADD: y[r] = y[r] + sum (CSS adds its block sums, src/opt_css.cpp:298).
template <int V, int XM, typename VT, typename XT, typename AT, int ACC = CS_OVERWRITE>
__global__ void __launch_bounds__(256)
ell_spmv_kernel(const long long *__restrict__ slice_off, const int *__restrict__ ecol,
                const VT *__restrict__ eval, const XT *__restrict__ x, XT *__restrict__ y,
                int rowBegin, int rowEnd, int sliceBegin, int sliceEnd)
{
    const int s = sliceBegin + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (s >= sliceEnd) return;
    const uint64_t pol_stream = policy_evict_first(), pol_x = policy_evict_last();
    const long long g0 = slice_off[s], g1 = slice_off[s + 1];
    const int r = s * 32 + lane;
    const bool mine = r >= rowBegin && r < rowEnd;
    const AT y0 = (ACC != CS_OVERWRITE && mine) ? (AT)y[r] : (AT)0;
    AT acc = ACC == CS_CONTINUE ? y0 : (AT)0;
    long long g = g0;
    for (; g + 2 <= g1; g += 2) {
        EllGroup<V, VT> a, b;
        ell_load<V>(a, ecol, eval, ((size_t)g * 32 + lane) * V, pol_stream);
        ell_load<V>(b, ecol, eval, ((size_t)(g + 1) * 32 + lane) * V, pol_stream);
        XT xa[V], xb[V];
#pragma unroll
        for (int j = 0; j < V; j++) xa[j] = ell_gather(x + a.c[j], pol_x, XM);
#pragma unroll
        for (int j = 0; j < V; j++) xb[j] = ell_gather(x + b.c[j], pol_x, XM);
#pragma unroll
        for (int j = 0; j < V; j++) acc = Arith<AT>::add(acc, Arith<AT>::mul((AT)xa[j], (AT)a.v[j]));
#pragma unroll
        for (int j = 0; j < V; j++) acc = Arith<AT>::add(acc, Arith<AT>::mul((AT)xb[j], (AT)b.v[j]));
    }
    if (g < g1) {
        EllGroup<V, VT> a;
        ell_load<V>(a, ecol, eval, ((size_t)g * 32 + lane) * V, pol_stream);
        XT xa[V];
#pragma unroll
        for (int j = 0; j < V; j++) xa[j] = ell_gather(x + a.c[j], pol_x, XM);
#pragma unroll
        for (int j = 0; j < V; j++) acc = Arith<AT>::add(acc, Arith<AT>::mul((AT)xa[j], (AT)a.v[j]));
    }
    if (mine) y[r] = (XT)(ACC == CS_ADD ? Arith<AT>::add(y0, acc) : acc);
}

// Logical [nRow][K] view for parity checks (slots beyond the slice width are padding).
template <int V, typename VT>
__global__ void ell_logical_kernel(const long long *__restrict__ slice_off, const int *__restrict__ ecol,
                                   const VT *__restrict__ eval, int nRow, int K, int *__restrict__ lcol,
                                   double *__restrict__ lval)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)nRow * K) return;
    const int r = (int)(i / K), k = (int)(i % K);
    const int s = r >> 5, lane = r & 31;
    const long long g0 = slice_off[s], g1 = slice_off[s + 1];
    if (k < (int)(g1 - g0) * V) {
        const size_t at = ((size_t)(g0 + k / V) * 32 + lane) * V + k % V;
        lcol[i] = ecol[at];
        lval[i] = (double)eval[at];
    } else {
        lcol[i] = k;
        lval[i] = 0.0;
    }
}

struct EllFormat : Format {
    int K = 0, V = 4, nSlices = 0;
    long long slots = 0;
    DevBuf<long long> slice_off;
    DevBuf<int> ecol;
    DevBuf<double> eval;
    DevBuf<float> eval32;             // options.precision = 1 / 2: fp32 value storage
    int prec = 0;
    std::unique_ptr<ColBlockEngine> cb;   // column-blocked multiply layout when x does not fit L2 (colblocks.cuh)
    int cbs_want = 0;
    explicit EllFormat(const b200spmv_options &o) : prec(o.precision), cbs_want(o.col_blocks) {}

    template <int VV> int convert_t(const CooView &A, const int *ptr, cudaStream_t s)
    {
        DevBuf<long long> groups;
        B2_TRY(groups.alloc((size_t)nSlices + 1));
        B2_TRY(slice_off.alloc((size_t)nSlices + 1));
        ell_slice_groups_kernel<VV><<<ceil_div(((long long)nSlices + 1) * 32, 256), 256, 0, s>>>(ptr, ptr + 1, nRow, nSlices, groups.p);
        B2_KERNEL_CHECK();
        B2_TRY(exclusive_scan_i64(groups.p, slice_off.p, nSlices + 1, s));
        long long totalGroups = 0;
        B2_CUDA(cudaMemcpy(&totalGroups, slice_off.p + nSlices, sizeof(long long), cudaMemcpyDeviceToHost));
        slots = totalGroups * 32 * VV;
        B2_TRY(ecol.alloc((size_t)slots));
        if (prec) B2_TRY(eval32.alloc((size_t)slots));
        else B2_TRY(eval.alloc((size_t)slots));
        if (nSlices) {
            const int grid = ceil_div((long long)nSlices * 32, 256);
            if (prec) ell_fill_kernel<VV, float><<<grid, 256, 0, s>>>(ptr, ptr + 1, A.col, A.val, nRow, nSlices, slice_off.p, K, 0, ecol.p, eval32.p);
            else ell_fill_kernel<VV, double><<<grid, 256, 0, s>>>(ptr, ptr + 1, A.col, A.val, nRow, nSlices, slice_off.p, K, 0, ecol.p, eval.p);
            B2_KERNEL_CHECK();
        }
        return B200SPMV_OK;
    }

    int convert(const CooView &A, cudaStream_t s) override
    {
        nRow = A.nRow; nCol = A.nCol; nnz = A.nnz;
        B2_TRY(validate_sorted_coo(A, s));
        DevBuf<int> ptr;
        B2_TRY(ptr.alloc((size_t)nRow + 1));
        B2_TRY(build_row_ptr(A.row, nnz, nRow, ptr.p, s));
        B2_TRY(max_row_length(ptr.p, nRow, &K, s));                 // opt_ell.cpp:28-31
        if (K > nCol) {
            set_error("ELL: K=%d exceeds nCol=%d; the reference's padding rule col=k (opt_ell.cpp:48) is undefined", K, nCol);
            return B200SPMV_ERR_INVALID;
        }
        V = (K % 4 == 0 || K >= 32) ? 4 : 2;
        nSlices = ceil_div(nRow, 32);
        int st = V == 4 ? convert_t<4>(A, ptr.p, s) : convert_t<2>(A, ptr.p, s);
        B2_TRY(st);
        cb.reset();
        if (!prec) B2_TRY(make_col_block_engine(A, ptr.p, cbs_want, s, &cb));
        B2_CUDA(cudaStreamSynchronize(s));
        return B200SPMV_OK;
    }

    int multiply(const double *x, double *y, cudaStream_t s) override { return multiply_rows(0, nRow, x, y, s); }
    int multiply_f32(const float *x, float *y, cudaStream_t s) override
    {
        if (!prec) { set_error("multiply_f32: the handle was created with precision = 0 (fp64 vectors)"); return B200SPMV_ERR_STATE; }
        if (nRow == 0) return B200SPMV_OK;
        const int blocks = ceil_div((long long)nSlices * 32, 256);
        if (V == 4 && prec == 1) ell_spmv_kernel<4, 0, float, float, float><<<blocks, 256, 0, s>>>(slice_off.p, ecol.p, eval32.p, x, y, 0, nRow, 0, nSlices);
        else if (V == 4) ell_spmv_kernel<4, 0, float, float, double><<<blocks, 256, 0, s>>>(slice_off.p, ecol.p, eval32.p, x, y, 0, nRow, 0, nSlices);
        else if (prec == 1) ell_spmv_kernel<2, 0, float, float, float><<<blocks, 256, 0, s>>>(slice_off.p, ecol.p, eval32.p, x, y, 0, nRow, 0, nSlices);
        else ell_spmv_kernel<2, 0, float, float, double><<<blocks, 256, 0, s>>>(slice_off.p, ecol.p, eval32.p, x, y, 0, nRow, 0, nSlices);
        B2_KERNEL_CHECK();
        return B200SPMV_OK;
    }
    bool has_rows() const override { return !(cb != nullptr) && !prec; }   // a row chunk would pay every column-block switch again
    int prepare_rows(int rb, int re) override { return cb != nullptr ? cb->prepare(rb, re) : B200SPMV_OK; }
    int col_extent(int rb, int re, int *cmin, int *cmax) override
    {
        if (rb < 0 || re > nRow || rb > re) { set_error("col_extent: bad row range [%d,%d)", rb, re); return B200SPMV_ERR_INVALID; }
        if (rb == re) { *cmin = 0; *cmax = -1; return B200SPMV_OK; }
        if ((cb != nullptr)) return Format::col_extent(rb, re, cmin, cmax);
        long long g[2] = {0, 0};                        // whole slices: padding columns (slot numbers) included
        B2_CUDA(cudaMemcpy(&g[0], slice_off.p + rb / 32, sizeof(long long), cudaMemcpyDeviceToHost));
        B2_CUDA(cudaMemcpy(&g[1], slice_off.p + ceil_div(re, 32), sizeof(long long), cudaMemcpyDeviceToHost));
        if (g[1] <= g[0]) { *cmin = 0; *cmax = -1; return B200SPMV_OK; }
        return minmax_i32(ecol.p, g[0] * 32 * V, g[1] * 32 * V, cmin, cmax);
    }

    int multiply_rows(int rb, int re, const double *x, double *y, cudaStream_t s) override
    {
        if (rb < 0 || re > nRow || rb > re) { set_error("multiply_rows: bad row range [%d,%d)", rb, re); return B200SPMV_ERR_INVALID; }
        if (prec) { set_error("multiply: the handle was created with precision = %d, use b200spmv_multiply_f32", prec); return B200SPMV_ERR_STATE; }
        if (rb == re) return B200SPMV_OK;
        if ((cb != nullptr)) return cb->run(x, y, rb, re, s);
        const int sb = rb / 32, se = ceil_div(re, 32);
        const int blocks = ceil_div((long long)(se - sb) * 32, 256);
#define ELL_LAUNCH(VV, XM) ell_spmv_kernel<VV, XM, double, double, double><<<blocks, 256, 0, s>>>(slice_off.p, ecol.p, eval.p, x, y, rb, re, sb, se)
#define ELL_LAUNCH_V(VV)                                   \
    switch (xload_mode()) {                                \
    case 1: ELL_LAUNCH(VV, 1); break;                      \
    case 2: ELL_LAUNCH(VV, 2); break;                      \
    case 3: ELL_LAUNCH(VV, 3); break;                      \
    case 4: ELL_LAUNCH(VV, 4); break;                      \
    case 5: ELL_LAUNCH(VV, 5); break;                      \
    default: ELL_LAUNCH(VV, 0); break;                     \
    }
        if (V == 4) { ELL_LAUNCH_V(4) } else { ELL_LAUNCH_V(2) }
        B2_KERNEL_CHECK();
        return B200SPMV_OK;
    }

    bool scalar(const std::string &n, long long *out) override
    {
        if (n == "K") { *out = K; return true; }
        if (n == "slots") { *out = slots; return true; }
        if (n == "slice_vec") { *out = V; return true; }
        if (n == "alg_bytes") {   // 12 B per stored slot + slice offsets + x + y
            *out = (prec ? 8LL : 12LL) * slots + 8LL * (nSlices + 1) + (prec ? 4LL : 8LL) * ((long long)nCol + nRow);
            return true;
        }
        if (n == "launches") { *out = (cb != nullptr) ? cb->n_blocks() : 1; return true; }
        if (n == "col_blocks") { *out = (cb != nullptr) ? cb->n_blocks() : 0; return true; }
        if (n == "col_block_engine") { *out = (cb == nullptr) ? 0 : (cb->name()[0] == 'e' ? 1 : 2); return true; }   // 1 = sliced ELL per block, 2 = tile-stream
        if (n == "precision") { *out = prec; return true; }
        return false;
    }

    long long array(const std::string &n, void *dst, long long cap) override
    {
        if (n != "col_idx" && n != "val") return -1000;
        const bool isCol = n == "col_idx";
        const size_t cnt = (size_t)nRow * K, bytes = cnt * (isCol ? sizeof(int) : sizeof(double));
        if (!dst) return (long long)bytes;
        DevBuf<int> lcol;
        DevBuf<double> lval;
        if (lcol.alloc(cnt) || lval.alloc(cnt)) return B200SPMV_ERR_NOMEM;
        if (cnt) {
            const int grid = ceil_div((long long)cnt, 256);
            if (V == 4 && prec) ell_logical_kernel<4, float><<<grid, 256>>>(slice_off.p, ecol.p, eval32.p, nRow, K, lcol.p, lval.p);
            else if (V == 4) ell_logical_kernel<4, double><<<grid, 256>>>(slice_off.p, ecol.p, eval.p, nRow, K, lcol.p, lval.p);
            else if (prec) ell_logical_kernel<2, float><<<grid, 256>>>(slice_off.p, ecol.p, eval32.p, nRow, K, lcol.p, lval.p);
            else ell_logical_kernel<2, double><<<grid, 256>>>(slice_off.p, ecol.p, eval.p, nRow, K, lcol.p, lval.p);
        }
        return export_device(isCol ? (const void *)lcol.p : (const void *)lval.p, bytes, dst, cap);
    }
};

Format *make_ell(const b200spmv_options &o) { return new EllFormat(o); }

// ---------------------------------------------------------------------------------------------------------------------
// Column-block engine as one sliced ELL per column block (colblocks.cuh).  A row's columns ascend, so its entries inside
// column block b are a contiguous piece [start_b[r], start_b+1[r]) of the row: every block gets its own slices of 32 rows,
// padded to the longest piece INSIDE the block (V = 2 slots at a time), and is multiplied by the ELL kernel -- one lane per
// row, ascending slots, block b continuing the sum block b-1 left in y.  Same bits as the format's own kernel and as the
// reference CRS result, whatever the row lengths.  On config 2 the pieces are Binomial(32, 1/3): 1.58 slots per entry;
// the padding costs stream bytes but no gather wavefronts (a padded lane re-reads one hot x entry), and the gathers are
// what bounds the kernel: 2.25 ms against 2.94 ms for the tile-stream per block (profiles/r2_experiments.md).
__global__ void cb_starts_kernel(const int *__restrict__ ptr, const int *__restrict__ col, int nRow, int B, int nb,
                                 int *__restrict__ start /* [nb + 1][nRow] */)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nRow) return;
    const int b0 = ptr[r], e0 = ptr[r + 1];
    int at = b0;
    for (int b = 0; b <= nb; b++) {
        const long long bound = (long long)b * B;              // first column of block b
        while (at < e0 && col[at] < bound) at++;
        start[(size_t)b * nRow + r] = b == nb ? e0 : at;
    }
}

struct EllColBlocks : ColBlockEngine {
    struct Blk {
        DevBuf<long long> slice_off;
        DevBuf<int> ecol;
        DevBuf<double> eval;
        long long slots = 0;
    };
    int nRow = 0, nSlices = 0;
    std::vector<std::unique_ptr<Blk>> blk;
    long long slots = 0;

    int later = CS_CONTINUE;                                  // what blocks after the first do with y: CS_CONTINUE or CS_ADD (CSS)

    int build(const CooView &A, const int *row_ptr, int nb, int Bwant, double maxRatio, bool *ok, cudaStream_t s)
    {
        *ok = false;
        nRow = A.nRow;
        nSlices = ceil_div(nRow, 32);
        const int B = Bwant > 0 ? Bwant : (A.nCol + nb - 1) / nb;
        DevBuf<int> start;
        DevBuf<long long> groups;
        B2_TRY(start.alloc((size_t)(nb + 1) * nRow));
        B2_TRY(groups.alloc((size_t)nSlices + 1));
        cb_starts_kernel<<<ceil_div(nRow, 256), 256, 0, s>>>(row_ptr, A.col, nRow, B, nb, start.p);
        B2_KERNEL_CHECK();
        slots = 0;
        for (int b = 0; b < nb; b++) {
            std::unique_ptr<Blk> k(new Blk());
            const int *beg = start.p + (size_t)b * nRow, *end = start.p + (size_t)(b + 1) * nRow;
            B2_TRY(k->slice_off.alloc((size_t)nSlices + 1));
            ell_slice_groups_kernel<2><<<ceil_div(((long long)nSlices + 1) * 32, 256), 256, 0, s>>>(beg, end, nRow, nSlices, groups.p);
            B2_KERNEL_CHECK();
            B2_TRY(exclusive_scan_i64(groups.p, k->slice_off.p, nSlices + 1, s));
            long long totalGroups = 0;
            B2_CUDA(cudaMemcpyAsync(&totalGroups, k->slice_off.p + nSlices, sizeof(long long), cudaMemcpyDeviceToHost, s));
            B2_CUDA(cudaStreamSynchronize(s));
            k->slots = totalGroups * 32 * 2;
            slots += k->slots;
            if ((double)slots > maxRatio * (double)std::max(A.nnz, 1)) return B200SPMV_OK;      // too much padding: not this engine
            B2_TRY(k->ecol.alloc((size_t)k->slots));
            B2_TRY(k->eval.alloc((size_t)k->slots));
            if (nSlices) {
                ell_fill_kernel<2, double><<<ceil_div((long long)nSlices * 32, 256), 256, 0, s>>>(beg, end, A.col, A.val, nRow, nSlices, k->slice_off.p, 0,
                                                                                                 (int)std::min<long long>((long long)b * B, A.nCol - 1), k->ecol.p, k->eval.p);
                B2_KERNEL_CHECK();
            }
            blk.push_back(std::move(k));
        }
        B2_CUDA(cudaStreamSynchronize(s));
        *ok = true;
        return B200SPMV_OK;
    }

    int run_block(int b, const double *x, double *y, int rb, int re, cudaStream_t s) override
    {
        if (rb >= re) return B200SPMV_OK;
        const int sb = rb / 32, se = ceil_div(re, 32);
        const int blocks = ceil_div((long long)(se - sb) * 32, 256);
        const Blk &k = *blk[(size_t)b];
        if (b == 0) ell_spmv_kernel<2, 0, double, double, double, CS_OVERWRITE><<<blocks, 256, 0, s>>>(k.slice_off.p, k.ecol.p, k.eval.p, x, y, rb, re, sb, se);
        else if (later == CS_ADD) ell_spmv_kernel<2, 0, double, double, double, CS_ADD><<<blocks, 256, 0, s>>>(k.slice_off.p, k.ecol.p, k.eval.p, x, y, rb, re, sb, se);
        else ell_spmv_kernel<2, 0, double, double, double, CS_CONTINUE><<<blocks, 256, 0, s>>>(k.slice_off.p, k.ecol.p, k.eval.p, x, y, rb, re, sb, se);
        B2_KERNEL_CHECK();
        return B200SPMV_OK;
    }
    int run(const double *x, double *y, int rb, int re, cudaStream_t s) override
    {
        for (size_t b = 0; b < blk.size(); b++) B2_TRY(run_block((int)b, x, y, rb, re, s));
        return B200SPMV_OK;
    }
    int n_blocks() const override { return (int)blk.size(); }
    const char *name() const override { return "ell"; }
};

int make_ell_col_blocks(const CooView &A, const int *row_ptr, int nb, int B, int later, double maxRatio, cudaStream_t s,
                        std::unique_ptr<ColBlockEngine> *out)
{
    std::unique_ptr<EllColBlocks> e(new EllColBlocks());
    e->later = later;
    bool ok = false;
    B2_TRY(e->build(A, row_ptr, nb, B, maxRatio, &ok, s));
    if (ok) *out = std::move(e);
    return B200SPMV_OK;
}

}  // namespace b2
