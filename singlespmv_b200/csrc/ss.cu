// ss.cu -- SS ("segmented sum", /root/reference/src/opt_ss.{h,cpp}) and CSS (column-blocked SS,
// /root/reference/src/opt_css.{h,cpp}) plugins.
//
// Conversion reproduces every array of the reference bit-exactly, on the device:
//   slabs row_idx/col_idx/val [H][W] with padding (SS: row=nRow, CSS: row=0; col=0, val=0)
//                                                         opt_ss.cpp:64-85, opt_css.cpp:60-111
//   row_ptr (CRS-style; CSS: one per column block)       opt_ss.cpp:64-85, opt_css.cpp:88-110
//   segment_index = position of a whole-row segment in its chain     opt_ss.cpp:91-107
//   nStep, sum_segs[s], sum_segs_count[s] = log-step fold schedule   opt_ss.cpp:121-142
//
// Multiply, default: ONE fused pass -- the tile-stream kernel (tile_stream.cuh) multiplies and
// reduces in shared memory, never writing the products to HBM.  The reference materialises them in
// val_buf, folds whole-row segments level by level and gathers per row (opt_ss.cpp:222-303): three
// sweeps, +16 B/nnz.  With options.ss_faithful = 1 that three-phase schedule is executed instead,
// in the reference's operation order, so y is bit-identical to the reference's SS/CSS result (this
// is how the schedule arrays are proven to be functionally right, not just equal).
// CSS runs one tile-stream pass per column block, accumulating into y in block order; with the
// block's slice of x resident in L2 (that is the point of the format, opt_css.cpp:33-45).  x is protected by the
// per-load evict_last policy; a persisting-L2 stream access-policy window instead was measured 8 % slower
// (profiles/r1_experiments.md).
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <cub/cub.cuh>

#include "chunk_stream.cuh"
#include "colblocks.cuh"
#include "tile_stream.cuh"

namespace b2 {

// ---------------------------------------------------------------- slabs
__global__ void ss_slab_kernel(const int *__restrict__ row, const int *__restrict__ col, const double *__restrict__ val,
                               long long nnz, long long slots, int padRow, int *__restrict__ row2d,
                               int *__restrict__ col2d, double *__restrict__ val2d)
{
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= slots) return;
    const bool real = p < nnz;
    row2d[p] = real ? row[p] : padRow;
    col2d[p] = real ? col[p] : 0;
    val2d[p] = real ? val[p] : 0.0;
}

// ---------------------------------------------------------------- whole-row segment chains (shared by SS and CSS)
// mixed[s] = 1 if the W row ids of segment s are not all equal
__global__ void chain_mixed_kernel(const int *__restrict__ row2d, long long slots, int W, int *__restrict__ mixed)
{
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= slots || (p % W) == 0) return;
    if (row2d[p] != row2d[p - 1]) mixed[p / W] = 1;
}
// head[s] = s for segments that start a chain (or belong to none), 0 otherwise; an inclusive max-scan
// then gives, for every segment, the head of its chain: segment_index = s - head.
__global__ void chain_head_kernel(const int *__restrict__ row2d, const int *__restrict__ mixed, int H, int W,
                                  int *__restrict__ head)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= H) return;
    const bool chained = s > 0 && !mixed[s] && row2d[(size_t)(s - 1) * W] == row2d[(size_t)s * W];
    head[s] = chained ? 0 : s;
}
__global__ void chain_index_kernel(const int *__restrict__ headscan, int H, int *__restrict__ segment_index,
                                   int *__restrict__ deepest)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    int idx = 0;
    if (s < H) {
        idx = s - headscan[s];
        segment_index[s] = idx;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) idx = max(idx, __shfl_xor_sync(0xffffffffu, idx, o));
    if ((threadIdx.x & 31) == 0 && idx > 0) atomicMax(deepest, idx);
}
// level of a chained segment: s such that 2^(nStep-1-s) <= index < 2^(nStep-s)
__global__ void chain_level_kernel(const int *__restrict__ segment_index, int H, int nStep, int *__restrict__ level,
                                   int *__restrict__ counts)
{
    __shared__ int local[32];
    if (threadIdx.x < 32) local[threadIdx.x] = 0;
    __syncthreads();
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < H) {
        const int idx = segment_index[s];
        int lv = 31;                                       // "not in any list" sorts last
        if (idx > 0) {
            lv = nStep - 1 - (31 - __clz(idx));
            atomicAdd(&local[lv], 1);
        }
        level[s] = lv;
    }
    __syncthreads();
    if (threadIdx.x < 32 && local[threadIdx.x]) atomicAdd(&counts[threadIdx.x], local[threadIdx.x]);
}
__global__ void iota_kernel(int *a, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] = i;
}

struct MaxOp {
    __host__ __device__ int operator()(int a, int b) const { return a > b ? a : b; }
};

// Builds segment_index (device, H ints at seg_index_out), nStep, per-level counts (host) and the
// concatenated level lists (device) for one slab of H segments.
static int build_chain(const int *row2d, int H, int W, int *seg_index_out, int *nStep_out, std::vector<int> &counts_out,
                       DevBuf<int> &segs_out, cudaStream_t s)
{
    *nStep_out = 0;
    counts_out.clear();
    B2_TRY(segs_out.alloc(0));
    if (H <= 0) return B200SPMV_OK;
    const long long slots = (long long)H * W;
    DevBuf<int> mixed, head, misc;
    B2_TRY(mixed.alloc((size_t)H));
    B2_TRY(head.alloc((size_t)H));
    B2_TRY(misc.alloc(1 + 32));                          // [0] deepest index, [1..32] level counts
    B2_CUDA(cudaMemsetAsync(mixed.p, 0, mixed.bytes(), s));
    B2_CUDA(cudaMemsetAsync(misc.p, 0, misc.bytes(), s));
    chain_mixed_kernel<<<ceil_div(slots, 256), 256, 0, s>>>(row2d, slots, W, mixed.p);
    chain_head_kernel<<<ceil_div(H, 256), 256, 0, s>>>(row2d, mixed.p, H, W, head.p);
    B2_KERNEL_CHECK();
    {
        size_t tmp = 0;
        B2_CUDA(cub::DeviceScan::InclusiveScan(nullptr, tmp, head.p, head.p, MaxOp(), H, s));
        DevBuf<char> t;
        B2_TRY(t.alloc(tmp));
        B2_CUDA(cub::DeviceScan::InclusiveScan(t.p, tmp, head.p, head.p, MaxOp(), H, s));
        B2_CUDA(cudaStreamSynchronize(s));
    }
    chain_index_kernel<<<ceil_div(H, 256), 256, 0, s>>>(head.p, H, seg_index_out, misc.p);
    B2_KERNEL_CHECK();
    int deepest = 0;
    B2_CUDA(cudaMemcpyAsync(&deepest, misc.p, sizeof(int), cudaMemcpyDeviceToHost, s));
    B2_CUDA(cudaStreamSynchronize(s));
    int nStep = 0;
    while ((1LL << nStep) < (long long)deepest + 1) nStep++;          // ceil(log2(max_index+1)), opt_ss.cpp:121
    *nStep_out = nStep;
    if (nStep == 0) return B200SPMV_OK;
    DevBuf<int> level, ids, level_sorted, ids_sorted;
    B2_TRY(level.alloc((size_t)H));
    B2_TRY(ids.alloc((size_t)H));
    B2_TRY(level_sorted.alloc((size_t)H));
    B2_TRY(ids_sorted.alloc((size_t)H));
    chain_level_kernel<<<ceil_div(H, 256), 256, 0, s>>>(seg_index_out, H, nStep, level.p, misc.p + 1);
    iota_kernel<<<ceil_div(H, 256), 256, 0, s>>>(ids.p, H);
    B2_KERNEL_CHECK();
    {
        // stable sort by level keeps ascending segment order inside each list (opt_ss.cpp:134-139)
        size_t tmp = 0;
        B2_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp, level.p, level_sorted.p, ids.p, ids_sorted.p, H, 0, 5, s));
        DevBuf<char> t;
        B2_TRY(t.alloc(tmp));
        B2_CUDA(cub::DeviceRadixSort::SortPairs(t.p, tmp, level.p, level_sorted.p, ids.p, ids_sorted.p, H, 0, 5, s));
        B2_CUDA(cudaStreamSynchronize(s));
    }
    int counts[32];
    B2_CUDA(cudaMemcpy(counts, misc.p + 1, sizeof counts, cudaMemcpyDeviceToHost));
    long long total = 0;
    for (int l = 0; l < nStep; l++) {
        counts_out.push_back(counts[l]);
        total += counts[l];
    }
    B2_TRY(segs_out.alloc((size_t)total));
    if (total) B2_CUDA(cudaMemcpy(segs_out.p, ids_sorted.p, sizeof(int) * (size_t)total, cudaMemcpyDeviceToDevice));
    return B200SPMV_OK;
}

// ---------------------------------------------------------------- faithful three-phase multiply
__global__ void ss_mul_kernel(const int *__restrict__ col2d, const double *__restrict__ val2d, const double *__restrict__ x,
                              long long slots, double *__restrict__ val_buf)
{
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < slots) val_buf[p] = __dmul_rn(val2d[p], x[col2d[p]]);          // opt_ss.cpp:226-238
}
__global__ void ss_fold_kernel(const int *__restrict__ segs, long long count, int W, int dist, double *__restrict__ val_buf)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count * W) return;
    const int h = segs[i / W], j = (int)(i % W);
    double *dst = val_buf + (size_t)(h - dist) * W + j;
    *dst = __dadd_rn(*dst, val_buf[(size_t)h * W + j]);                     // opt_ss.cpp:242-260
}
__global__ void ss_gather_kernel(const int *__restrict__ row_ptr, const double *__restrict__ val_buf, int nRow, int W,
                                 int accumulate, double *__restrict__ y)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nRow) return;
    int begin = row_ptr[r], end = row_ptr[r + 1];
    double acc = 0.0;
    if (begin / W == end / W) {                                            // opt_ss.cpp:264-303
        for (int j = begin; j < end; j++) acc = __dadd_rn(acc, val_buf[j]);
    } else {
        if (begin & (W - 1)) {
            const int stop = (begin & ~(W - 1)) + W;
            for (int j = begin; j < stop; j++) acc = __dadd_rn(acc, val_buf[j]);
            begin = stop;
        }
        if (end & (W - 1)) {
            const int stop = end & ~(W - 1);
            for (int j = end; j > stop; j--) acc = __dadd_rn(acc, val_buf[j - 1]);
            end = stop;
        }
        if (begin != end)
            for (int j = 0; j < W; j++) acc = __dadd_rn(acc, val_buf[begin + j]);
    }
    y[r] = accumulate ? __dadd_rn(y[r], acc) : acc;
}

static int faithful_fold(const DevBuf<int> &segs, const std::vector<int> &counts, int W, double *val_buf, cudaStream_t s)
{
    long long base = 0;
    const int nStep = (int)counts.size();
    for (int l = 0; l < nStep; l++) {
        const long long n = counts[(size_t)l];
        if (n) {
            ss_fold_kernel<<<ceil_div(n * W, 256), 256, 0, s>>>(segs.p + base, n, W, 1 << (nStep - 1 - l), val_buf);
            B2_KERNEL_CHECK();
        }
        base += n;
    }
    return B200SPMV_OK;
}

// options.profile (faithful mode): the reference's PROF_BEGIN/PROF_END pairs around the Mul and the Sum phase
// (src/util.h:59-65, opt_ss.cpp:225-304) become CUDA events; the multiply then synchronises and the last call's
// phase times are readable as scalars MulTime_ns / SumTime_ns.
struct PhaseTimer {
    cudaEvent_t e[3] = {nullptr, nullptr, nullptr};
    long long mul_ns = 0, sum_ns = 0;
    bool on = false;
    ~PhaseTimer() { for (auto &x : e) if (x) cudaEventDestroy(x); }
    int mark(int i, cudaStream_t s)
    {
        if (!on) return B200SPMV_OK;
        if (!e[i]) B2_CUDA(cudaEventCreate(&e[i]));
        B2_CUDA(cudaEventRecord(e[i], s));
        return B200SPMV_OK;
    }
    int finish()
    {
        if (!on) return B200SPMV_OK;
        B2_CUDA(cudaEventSynchronize(e[2]));
        float a = 0, b = 0;
        B2_CUDA(cudaEventElapsedTime(&a, e[0], e[1]));
        B2_CUDA(cudaEventElapsedTime(&b, e[1], e[2]));
        mul_ns = (long long)(a * 1e6);
        sum_ns = (long long)(b * 1e6);
        return B200SPMV_OK;
    }
    bool scalar(const std::string &n, long long *out) const
    {
        if (n == "MulTime_ns") { *out = mul_ns; return true; }
        if (n == "SumTime_ns") { *out = sum_ns; return true; }
        return false;
    }
};

// ================================================================= SS
struct SsFormat : Format {
    int W, H = 0, nStep = 0, faithful, maxLen = 0;
    bool short_rows = false;
    DevBuf<int> row_ptr, row2d, col2d, seg_index, segs;
    DevBuf<double> val2d, val_buf;
    std::vector<int> counts;
    TileStream ts;
    ChunkStream cs;
    bool use_rbs = false;
    PhaseTimer prof;
    std::unique_ptr<ColBlockEngine> cb;   // column-blocked multiply layout when x does not fit L2 (colblocks.cuh)
    int cbs_want;

    int path_opt;
    explicit SsFormat(const b200spmv_options &o) : W(o.segment_width), faithful(o.ss_faithful), cbs_want(o.col_blocks), path_opt(o.crs_path) { prof.on = o.profile != 0 && o.ss_faithful != 0; }

    int convert(const CooView &A, cudaStream_t s) override
    {
        nRow = A.nRow; nCol = A.nCol; nnz = A.nnz;
        B2_TRY(validate_sorted_coo(A, s));
        H = nnz / W + (nnz % W != 0);                                       // opt_ss.cpp:33
        const long long slots = (long long)H * W;
        B2_TRY(row_ptr.alloc((size_t)nRow + 1));
        B2_TRY(row2d.alloc((size_t)slots));
        B2_TRY(col2d.alloc((size_t)slots + CS_SLACK));       // slack: bulk copies of the row-chunk stream end on 16 bytes
        B2_TRY(val2d.alloc((size_t)slots + CS_SLACK));
        B2_TRY(seg_index.alloc((size_t)H));
        B2_TRY(build_row_ptr(A.row, nnz, nRow, row_ptr.p, s));
        if (slots) {
            ss_slab_kernel<<<ceil_div(slots, 256), 256, 0, s>>>(A.row, A.col, A.val, nnz, slots, nRow, row2d.p, col2d.p, val2d.p);
            B2_KERNEL_CHECK();
        }
        B2_TRY(build_chain(row2d.p, H, W, seg_index.p, &nStep, counts, segs, s));
        B2_TRY(ts.build(row_ptr.p, col2d.p, val2d.p, false, nRow, nnz, s));
        B2_TRY(max_row_length(row_ptr.p, nRow, &maxLen, s));
        B2_TRY(cs.build(row_ptr.p, col2d.p, val2d.p, false, nRow, nnz, maxLen, s));
        use_rbs = path_opt == 2 && rowblock_applies(maxLen, nnz);
        int band = 0;
        if (path_opt == 0 && cs.ok) B2_TRY(max_band(A.row, A.col, nnz, A.rowOffset, &band, s));
        short_rows = path_opt != 1 && (use_rbs || (cs.ok && !gathers_need_l2(band)));   // see crs.cu
        cb.reset();
        if (!faithful) B2_TRY(make_col_block_engine(A, row_ptr.p, cbs_want, s, &cb));
        if (faithful) B2_TRY(val_buf.alloc((size_t)slots));
        B2_CUDA(cudaStreamSynchronize(s));
        return B200SPMV_OK;
    }

    int multiply(const double *x, double *y, cudaStream_t s) override
    {
        if (!faithful) return multiply_rows(0, nRow, x, y, s);
        if (nRow == 0) return B200SPMV_OK;
        const long long slots = (long long)H * W;
        B2_TRY(prof.mark(0, s));
        if (slots) {
            ss_mul_kernel<<<ceil_div(slots, 256), 256, 0, s>>>(col2d.p, val2d.p, x, slots, val_buf.p);
            B2_KERNEL_CHECK();
        }
        B2_TRY(prof.mark(1, s));
        B2_TRY(faithful_fold(segs, counts, W, val_buf.p, s));
        ss_gather_kernel<<<ceil_div(nRow, 256), 256, 0, s>>>(row_ptr.p, val_buf.p, nRow, W, 0, y);
        B2_KERNEL_CHECK();
        B2_TRY(prof.mark(2, s));
        return prof.finish();
    }

    bool has_rows() const override { return !faithful && !(cb != nullptr); }
    int prepare_rows(int rb, int re) override
    {
        if (faithful) return B200SPMV_OK;
        if (cb != nullptr) return cb->prepare(rb, re);
        return short_rows ? B200SPMV_OK : ts.prepare(rb, re);
    }
    int col_extent(int rb, int re, int *cmin, int *cmax) override
    {
        if (rb < 0 || re > nRow || rb > re) { set_error("col_extent: bad row range [%d,%d)", rb, re); return B200SPMV_ERR_INVALID; }
        int pb = 0, pe = 0;
        B2_CUDA(cudaMemcpy(&pb, row_ptr.p + rb, sizeof(int), cudaMemcpyDeviceToHost));
        B2_CUDA(cudaMemcpy(&pe, row_ptr.p + re, sizeof(int), cudaMemcpyDeviceToHost));
        if (pe <= pb) { *cmin = 0; *cmax = -1; return B200SPMV_OK; }
        return minmax_i32(col2d.p, pb, pe, cmin, cmax);
    }
    int multiply_rows(int rb, int re, const double *x, double *y, cudaStream_t s) override
    {
        if (faithful) return Format::multiply_rows(rb, re, x, y, s);
        if ((cb != nullptr)) return cb->run(x, y, rb, re, s);
        if (short_rows) {        // same fused product+sum, warp-per-32-rows stream (crs.cu)
            if (rb < 0 || re > nRow || rb > re) { set_error("multiply_rows: bad row range [%d,%d)", rb, re); return B200SPMV_ERR_INVALID; }
            if (use_rbs) return rowblock_spmv(row_ptr.p, col2d.p, val2d.p, false, maxLen, rb, re, x, y, s);
            return cs.run(x, y, rb, re, CS_OVERWRITE, s);
        }
        return ts.run_rows(x, y, CS_OVERWRITE, rb, re, s);
    }

    bool scalar(const std::string &n, long long *out) override
    {
        if (prof.scalar(n, out)) return true;
        if (n == "col_blocks") { *out = (cb != nullptr) ? cb->n_blocks() : 0; return true; }
        if (n == "col_block_engine") { *out = (cb == nullptr) ? 0 : (cb->name()[0] == 'e' ? 1 : 2); return true; }   // 1 = sliced ELL per block, 2 = tile-stream
        if (n == "short_row_path") { *out = short_rows ? 1 : 0; return true; }   // 1 = row-chunk / row-block stream, 0 = tile-stream
        if (n == "chunk_feed") { *out = !faithful && cb == nullptr && short_rows && !use_rbs ? cs.feed : CS_FEED_IDX; return true; }   // see crs.cu
        if (n == "H") { *out = H; return true; }
        if (n == "nStep") { *out = nStep; return true; }
        if (n == "W") { *out = W; return true; }
        if (n == "alg_bytes") {   // SURVEY.md 8d: 12 nnz + 4 (nRow+1) + 8 nCol + 8 nRow (no val_buf)
            *out = 12LL * nnz + 4LL * (nRow + 1) + 8LL * nCol + 8LL * nRow;
            return true;
        }
        if (n == "launches") {
            if (!faithful) { *out = (cb != nullptr) ? cb->n_blocks() : short_rows ? 1 : (ts.nTiles > 1 ? 2 : 1); return true; }
            int l = 2;
            for (int c : counts) l += c > 0;
            *out = l;
            return true;
        }
        return false;
    }

    long long array(const std::string &n, void *dst, long long cap) override
    {
        if (n == "row_ptr") return export_device(row_ptr.p, row_ptr.bytes(), dst, cap);
        if (n == "row_idx") return export_device(row2d.p, row2d.bytes(), dst, cap);
        if (n == "col_idx") return export_device(col2d.p, sizeof(int) * (size_t)H * W, dst, cap);
        if (n == "val") return export_device(val2d.p, sizeof(double) * (size_t)H * W, dst, cap);
        if (n == "segment_index") return export_device(seg_index.p, seg_index.bytes(), dst, cap);
        if (n == "sum_segs") return export_device(segs.p, segs.bytes(), dst, cap);
        if (n == "sum_segs_count") return export_host(counts.data(), counts.size() * sizeof(int), dst, cap);
        return -1000;
    }
};

Format *make_ss(const b200spmv_options &o) { return new SsFormat(o); }

// ================================================================= CSS
constexpr int CSS_HIST = 1024;     // column blocks counted in shared memory (more: global atomics)
__global__ void css_block_key_kernel(const int *__restrict__ col, int nnz, int B, int nBlock, int *__restrict__ key,
                                     int *__restrict__ id, int *__restrict__ blockNnz)
{
    __shared__ int hist[CSS_HIST];
    const bool local = nBlock <= CSS_HIST;
    if (local)
        for (int k = threadIdx.x; k < nBlock; k += blockDim.x) hist[k] = 0;
    __syncthreads();
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += gridDim.x * blockDim.x) {
        const int b = col[i] / B;                                          // opt_css.cpp:40
        key[i] = b;
        id[i] = i;
        atomicAdd(local ? &hist[b] : &blockNnz[b], 1);
    }
    __syncthreads();
    if (local)
        for (int k = threadIdx.x; k < nBlock; k += blockDim.x)
            if (hist[k]) atomicAdd(&blockNnz[k], hist[k]);
}
// entry k of the block-sorted order goes to slab position base[b] + (k - start[b])
__global__ void css_scatter_kernel(const int *__restrict__ row, const int *__restrict__ col, const double *__restrict__ val,
                                   const int *__restrict__ key_sorted, const int *__restrict__ id_sorted, int nnz,
                                   const long long *__restrict__ slabBase, const int *__restrict__ blockStart,
                                   int *__restrict__ row2d, int *__restrict__ col2d, double *__restrict__ val2d)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nnz) return;
    const int b = key_sorted[k], i = id_sorted[k];
    const long long p = slabBase[b] + (k - blockStart[b]);
    row2d[p] = row[i];
    col2d[p] = col[i];
    val2d[p] = val[i];
}

__global__ void colblock_spread_kernel(const int *__restrict__ ptr, const int *__restrict__ col, int nRow, int B,
                                       unsigned long long *__restrict__ stats)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    int touched = 0, nonEmpty = 0;
    if (r < nRow) {
        int last = -1;
        for (int j = ptr[r]; j < ptr[r + 1]; j++) {
            const int b = col[j] / B;
            touched += b != last;
            last = b;
        }
        nonEmpty = touched > 0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        touched += __shfl_xor_sync(0xffffffffu, touched, o);
        nonEmpty += __shfl_xor_sync(0xffffffffu, nonEmpty, o);
    }
    if ((threadIdx.x & 31) == 0 && touched) {
        atomicAdd(&stats[0], (unsigned long long)touched);
        atomicAdd(&stats[1], (unsigned long long)nonEmpty);
    }
}

struct CssBlock {
    int H = 0, nStep = 0, cnt = 0, maxLen = 0;
    long long base = 0;                  // first slab slot of the block
    std::vector<int> counts;
    DevBuf<int> segs;
    TileStream ts;
    ChunkStream cs;                      // TMA-fed row-chunk stream when the block's rows are short enough
    // acc: CS_OVERWRITE / CS_CONTINUE / CS_ADD.  gather_bound: the blocks exist because x does not fit L2 -- there the
    // tile-stream kernel wins (2048 threads per SM keep more gathers in flight: c2, 2.92 ms against 4.43 ms for the
    // row-chunk stream, profiles/r2_experiments.md); on short-row blocks of local matrices the row-chunk stream does
    int run(const double *x, double *y, int rb, int re, bool gather_bound, int acc, cudaStream_t s)
    {
        if (cs.ok && !gather_bound) return cs.run(x, y, rb, re, acc, s);
        return ts.run_rows(x, y, acc, rb, re, s);
    }
};

struct CssFormat : Format {
    int W, nBlockWanted, faithful;
    bool lean = false;                   // column-block engine of another format: W = 1, no chain metadata, no row slab
    bool gather_bound = false;           // rows spread over the column blocks (decided at conversion): tile-stream per block
    int B = 0, nBlock = 0, totalH = 0;
    DevBuf<int> row_ptr, row2d, col2d, seg_index;      // row_ptr: [nBlock][nRow+1]
    DevBuf<double> val2d, val_buf;
    std::vector<std::unique_ptr<CssBlock>> blocks;
    std::unique_ptr<ColBlockEngine> ellb;   // gather-bound matrices: the blocks as sliced ELL (multiply only; the CSS arrays stay)
    PhaseTimer prof;

    explicit CssFormat(const b200spmv_options &o) : W(o.segment_width), nBlockWanted(o.n_block), faithful(o.ss_faithful) { prof.on = o.profile != 0 && o.ss_faithful != 0; }
    bool input_checked = false;          // lean: the owning format validated the COO already

    int convert(const CooView &A, cudaStream_t s) override
    {
        nRow = A.nRow; nCol = A.nCol; nnz = A.nnz;
        if (!input_checked) B2_TRY(validate_sorted_coo(A, s));
        blocks.clear();
        ellb.reset();
        gather_bound = lean ? gather_bound : false;
        B = nCol > 0 ? (nCol + nBlockWanted - 1) / nBlockWanted : 1;       // ceil(nCol / N_BLOCK), opt_css.cpp:34
        if (B < 1) B = 1;
        nBlock = nCol / B + (nCol % B ? 1 : 0);                            // opt_css.cpp:35
        if ((long long)nBlock * ((long long)nRow + 1) > 0x7fffffffLL * 8LL) { set_error("CSS: nBlock x (nRow+1) too large"); return B200SPMV_ERR_INVALID; }
        DevBuf<int> key, id, key_sorted, id_sorted, blockNnz, blockStart;
        DevBuf<long long> slabBase;
        B2_TRY(key.alloc((size_t)nnz));
        B2_TRY(id.alloc((size_t)nnz));
        B2_TRY(key_sorted.alloc((size_t)nnz));
        B2_TRY(id_sorted.alloc((size_t)nnz));
        B2_TRY(blockNnz.alloc((size_t)nBlock + 1));
        B2_TRY(blockStart.alloc((size_t)nBlock + 1));
        B2_TRY(slabBase.alloc((size_t)nBlock + 1));
        B2_CUDA(cudaMemsetAsync(blockNnz.p, 0, blockNnz.bytes(), s));
        if (nnz) {
            css_block_key_kernel<<<std::min(ceil_div(nnz, 256), 148 * 16), 256, 0, s>>>(A.col, nnz, B, nBlock, key.p, id.p, blockNnz.p);
            B2_KERNEL_CHECK();
            int bits = 1;
            while ((1 << bits) < nBlock) bits++;
            size_t tmp = 0;                                                 // stable: COO order kept inside a block
            B2_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp, key.p, key_sorted.p, id.p, id_sorted.p, nnz, 0, bits, s));
            DevBuf<char> t;
            B2_TRY(t.alloc(tmp));
            B2_CUDA(cub::DeviceRadixSort::SortPairs(t.p, tmp, key.p, key_sorted.p, id.p, id_sorted.p, nnz, 0, bits, s));
            B2_CUDA(cudaStreamSynchronize(s));
        }
        std::vector<int> cnt((size_t)nBlock + 1, 0), start((size_t)nBlock + 1, 0);
        std::vector<long long> base((size_t)nBlock + 1, 0);
        if (nBlock) B2_CUDA(cudaMemcpy(cnt.data(), blockNnz.p, sizeof(int) * (size_t)nBlock, cudaMemcpyDeviceToHost));
        totalH = 0;
        for (int b = 0; b < nBlock; b++) {
            std::unique_ptr<CssBlock> blk(new CssBlock());
            blk->cnt = cnt[(size_t)b];
            blk->H = blk->cnt / W + (blk->cnt % W ? 1 : 0);                // opt_css.cpp:52-56
            blk->base = base[(size_t)b];
            start[(size_t)b + 1] = start[(size_t)b] + blk->cnt;
            base[(size_t)b + 1] = base[(size_t)b] + (long long)blk->H * W;
            if (lean) base[(size_t)b + 1] = (base[(size_t)b + 1] + 3) & ~3LL;      // 16-byte aligned block starts (vector / bulk loads)
            totalH += blk->H;
            blocks.push_back(std::move(blk));
        }
        const long long slots = lean ? base[(size_t)nBlock] : (long long)totalH * W;
        B2_CUDA(cudaMemcpyAsync(blockStart.p, start.data(), sizeof(int) * ((size_t)nBlock + 1), cudaMemcpyHostToDevice, s));
        B2_CUDA(cudaMemcpyAsync(slabBase.p, base.data(), sizeof(long long) * ((size_t)nBlock + 1), cudaMemcpyHostToDevice, s));
        B2_TRY(row2d.alloc((size_t)slots));
        B2_TRY(col2d.alloc((size_t)slots + CS_SLACK));                      // slack: the row-chunk stream's copies end on 16 bytes
        B2_TRY(val2d.alloc((size_t)slots + CS_SLACK));
        B2_TRY(seg_index.alloc(lean ? 0 : (size_t)totalH));
        B2_TRY(row_ptr.alloc((size_t)nBlock * ((size_t)nRow + 1)));
        B2_CUDA(cudaMemsetAsync(row2d.p, 0, row2d.bytes(), s));             // padding: row = 0, col = 0, val = 0 (opt_css.cpp:103)
        B2_CUDA(cudaMemsetAsync(col2d.p, 0, col2d.bytes(), s));
        B2_CUDA(cudaMemsetAsync(val2d.p, 0, val2d.bytes(), s));
        if (nnz) {
            css_scatter_kernel<<<ceil_div(nnz, 256), 256, 0, s>>>(A.row, A.col, A.val, key_sorted.p, id_sorted.p, nnz, slabBase.p,
                                                                 blockStart.p, row2d.p, col2d.p, val2d.p);
            B2_KERNEL_CHECK();
        }
        int seg0 = 0;
        for (int b = 0; b < nBlock; b++) {
            CssBlock &k = *blocks[(size_t)b];
            int *rp = row_ptr.p + (size_t)b * ((size_t)nRow + 1);
            B2_TRY(build_row_ptr(row2d.p + k.base, k.cnt, nRow, rp, s));
            if (!lean) B2_TRY(build_chain(row2d.p + k.base, k.H, W, seg_index.p + seg0, &k.nStep, k.counts, k.segs, s));
            B2_TRY(k.ts.build(rp, col2d.p + k.base, val2d.p + k.base, false, nRow, k.cnt, s));
            B2_TRY(max_row_length(rp, nRow, &k.maxLen, s));
            B2_TRY(k.cs.build(rp, col2d.p + k.base, val2d.p + k.base, false, nRow, k.cnt, k.maxLen, s));
            seg0 += k.H;
        }
        if (lean) { B2_CUDA(cudaStreamSynchronize(s)); row2d.release(); }
        if (!lean && nBlock > 1 && nnz > 0) {
            // several column blocks: do the rows really spread over them (x gathers from everywhere), or is the matrix local?
            DevBuf<int> ptr;
            DevBuf<unsigned long long> stats;
            B2_TRY(ptr.alloc((size_t)nRow + 1));
            B2_TRY(stats.alloc(2));
            B2_TRY(build_row_ptr(A.row, nnz, nRow, ptr.p, s));
            B2_CUDA(cudaMemsetAsync(stats.p, 0, stats.bytes(), s));
            colblock_spread_kernel<<<ceil_div(nRow, 256), 256, 0, s>>>(ptr.p, A.col, nRow, B, stats.p);
            B2_KERNEL_CHECK();
            unsigned long long st[2] = {0, 0};
            B2_CUDA(cudaMemcpyAsync(st, stats.p, sizeof st, cudaMemcpyDeviceToHost, s));
            B2_CUDA(cudaStreamSynchronize(s));
            gather_bound = (double)st[0] >= 1.5 * (double)st[1];
            // gather-bound: one sliced ELL per column block, block sums ADDED like the tile-stream path does (colblocks.cuh)
            const char *env_e = getenv("B200SPMV_COL_BLOCK_ENGINE");
            if (gather_bound && !faithful && !(env_e && !strcmp(env_e, "crs")))
                B2_TRY(make_ell_col_blocks(A, ptr.p, nBlock, B, CS_ADD, 2.0, s, &ellb));
        }
        if (faithful) B2_TRY(val_buf.alloc((size_t)slots));
        B2_CUDA(cudaStreamSynchronize(s));
        return B200SPMV_OK;
    }

    int multiply(const double *x, double *y, cudaStream_t s) override
    {
        if (nRow == 0) return B200SPMV_OK;
        if (nBlock == 0) {
            B2_CUDA(cudaMemsetAsync(y, 0, sizeof(double) * (size_t)nRow, s));
            return B200SPMV_OK;
        }
        if (!faithful) {
            if (ellb) return ellb->run(x, y, 0, nRow, s);
            for (int b = 0; b < nBlock; b++) B2_TRY(blocks[(size_t)b]->run(x, y, 0, nRow, gather_bound, b > 0 ? CS_ADD : CS_OVERWRITE, s));
            return B200SPMV_OK;
        }
        const long long slots = (long long)totalH * W;
        B2_TRY(prof.mark(0, s));
        if (slots) {
            ss_mul_kernel<<<ceil_div(slots, 256), 256, 0, s>>>(col2d.p, val2d.p, x, slots, val_buf.p);   // opt_css.cpp:226-240
            B2_KERNEL_CHECK();
        }
        B2_TRY(prof.mark(1, s));
        B2_CUDA(cudaMemsetAsync(y, 0, sizeof(double) * (size_t)nRow, s));
        for (int b = 0; b < nBlock; b++) {
            CssBlock &k = *blocks[(size_t)b];
            B2_TRY(faithful_fold(k.segs, k.counts, W, val_buf.p + k.base, s));
            ss_gather_kernel<<<ceil_div(nRow, 256), 256, 0, s>>>(row_ptr.p + (size_t)b * ((size_t)nRow + 1), val_buf.p + k.base,
                                                                nRow, W, 1, y);                           // opt_css.cpp:298
            B2_KERNEL_CHECK();
        }
        B2_TRY(prof.mark(2, s));
        return prof.finish();
    }

    bool has_rows() const override { return !faithful; }
    int prepare_rows(int rb, int re) override
    {
        if (faithful || ellb || (rb == 0 && re == nRow)) return B200SPMV_OK;
        for (auto &k : blocks) if (!k->cs.ok || gather_bound) B2_TRY(k->ts.prepare(rb, re));     // the blocks CssBlock::run gives to the tile-stream
        return B200SPMV_OK;
    }
    int multiply_rows(int rb, int re, const double *x, double *y, cudaStream_t s) override
    {
        if (faithful) return Format::multiply_rows(rb, re, x, y, s);
        if (rb < 0 || re > nRow || rb > re) { set_error("multiply_rows: bad row range [%d,%d)", rb, re); return B200SPMV_ERR_INVALID; }
        if (rb == re) return B200SPMV_OK;
        if (nBlock == 0) {
            B2_CUDA(cudaMemsetAsync(y + rb, 0, sizeof(double) * (size_t)(re - rb), s));
            return B200SPMV_OK;
        }
        if (ellb) return ellb->run(x, y, rb, re, s);
        for (int b = 0; b < nBlock; b++) B2_TRY(blocks[(size_t)b]->run(x, y, rb, re, gather_bound, b > 0 ? CS_ADD : CS_OVERWRITE, s));
        return B200SPMV_OK;
    }
    // the running-sum variant used by the column-block engine of ELL / JDS / SS: block b continues the sums block b-1
    // left in y, so rows of up to TS_LONG entries per block are summed strictly in ascending column order
    int multiply_continue(int rb, int re, const double *x, double *y, cudaStream_t s)
    {
        bool first = true;
        for (auto &k : blocks) {
            if (k->cnt == 0 && !first) continue;
            if (k->cnt == 0) { B2_CUDA(cudaMemsetAsync(y + rb, 0, sizeof(double) * (size_t)(re - rb), s)); first = false; continue; }
            B2_TRY(k->run(x, y, rb, re, gather_bound, first ? CS_OVERWRITE : CS_CONTINUE, s));
            first = false;
        }
        return B200SPMV_OK;
    }

    int n_x_slices() const override { return faithful || nBlock < 1 ? 1 : nBlock; }
    void x_slice(int i, long long *c0, long long *c1) const override
    {
        if (faithful || nBlock < 1) { *c0 = 0; *c1 = nCol; return; }
        *c0 = (long long)i * B;
        *c1 = std::min<long long>(nCol, *c0 + B);
    }
    int multiply_rows_slice(int i, int rb, int re, const double *x, double *y, cudaStream_t s) override
    {
        if (faithful || nBlock < 1) return multiply_rows(rb, re, x, y, s);
        if (ellb) return ellb->run_block(i, x, y, rb, re, s);
        return blocks[(size_t)i]->run(x, y, rb, re, gather_bound, i > 0 ? CS_ADD : CS_OVERWRITE, s);
    }

    bool scalar(const std::string &n, long long *out) override
    {
        if (prof.scalar(n, out)) return true;
        if (n == "B") { *out = B; return true; }
        if (n == "col_block_engine") { *out = ellb ? 1 : (gather_bound ? 2 : 0); return true; }
        if (n == "nBlock") { *out = nBlock; return true; }
        if (n == "chunk_feed") {   // 1: every block on the row-chunk stream reads the offset dictionary (and there is one)
            bool any = false, all = true;
            if (!faithful && !ellb && !gather_bound)
                for (auto &k : blocks) if (k->cs.ok) { any = true; all = all && k->cs.feed == CS_FEED_DICT; }
            *out = any && all ? CS_FEED_DICT : CS_FEED_IDX;
            return true;
        }
        if (n == "totalH") { *out = totalH; return true; }
        if (n == "W") { *out = W; return true; }
        if (n == "alg_bytes") {   // SS bytes with one row_ptr per block
            *out = 12LL * nnz + 4LL * nBlock * ((long long)nRow + 1) + 8LL * nCol + 8LL * nRow;
            return true;
        }
        if (n == "launches") {
            long long l = 0;
            if (!faithful && ellb) l = ellb->n_blocks();
            else if (!faithful) for (auto &k : blocks) l += k->cs.ok ? 1 : (k->ts.nTiles > 1 ? 2 : 1);
            else { l = 2; for (auto &k : blocks) { l += 1; for (int c : k->counts) l += c > 0; } }
            *out = l;
            return true;
        }
        return false;
    }

    long long array(const std::string &n, void *dst, long long cap) override
    {
        if (n == "row_ptr") return export_device(row_ptr.p, row_ptr.bytes(), dst, cap);
        if (n == "row_idx") return export_device(row2d.p, row2d.bytes(), dst, cap);
        if (n == "col_idx") return export_device(col2d.p, sizeof(int) * (size_t)totalH * W, dst, cap);
        if (n == "val") return export_device(val2d.p, sizeof(double) * (size_t)totalH * W, dst, cap);
        if (n == "segment_index") return export_device(seg_index.p, seg_index.bytes(), dst, cap);
        std::vector<int> h;
        if (n == "H") { for (auto &k : blocks) h.push_back(k->H); return export_host(h.data(), h.size() * sizeof(int), dst, cap); }
        if (n == "nStep") { for (auto &k : blocks) h.push_back(k->nStep); return export_host(h.data(), h.size() * sizeof(int), dst, cap); }
        if (n == "sum_segs_count") {
            for (auto &k : blocks) h.insert(h.end(), k->counts.begin(), k->counts.end());
            return export_host(h.data(), h.size() * sizeof(int), dst, cap);
        }
        if (n == "sum_segs") {                  // blocks, then levels, concatenated
            size_t total = 0;
            for (auto &k : blocks) total += k->segs.n;
            if (!dst) return (long long)(total * sizeof(int));
            if (cap < (long long)(total * sizeof(int))) { set_error("get_array: destination too small"); return B200SPMV_ERR_INVALID; }
            size_t at = 0;
            for (auto &k : blocks) {
                if (k->segs.n && cudaMemcpy((int *)dst + at, k->segs.p, k->segs.bytes(), cudaMemcpyDeviceToHost) != cudaSuccess) {
                    set_error("get_array: cudaMemcpy D2H failed");
                    return B200SPMV_ERR_CUDA;
                }
                at += k->segs.n;
            }
            return (long long)(total * sizeof(int));
        }
        return -1000;
    }
};

Format *make_css(const b200spmv_options &o) { return new CssFormat(o); }

// ================================================================= column-block engine for ELL / JDS / SS (colblocks.cuh)
struct CrsColBlocks : ColBlockEngine {
    CssFormat css;
    explicit CrsColBlocks(const b200spmv_options &o) : css(o) { css.lean = true; css.input_checked = true; }
    int run(const double *x, double *y, int rb, int re, cudaStream_t s) override { return css.multiply_continue(rb, re, x, y, s); }
    int prepare(int rb, int re) override { return css.prepare_rows(rb, re); }
    int n_blocks() const override { return css.nBlock; }
    const char *name() const override { return "crs"; }
};
int make_col_block_engine(const CooView &A, const int *row_ptr, int want, cudaStream_t s, std::unique_ptr<ColBlockEngine> *out)
{
    out->reset();
    static const char *env_n = getenv("B200SPMV_COL_BLOCKS");           // experiments: 0 = never, n = n blocks
    if (env_n) want = atoi(env_n) == 0 ? -1 : atoi(env_n);
    if (want < 0 || A.nnz == 0 || A.nRow == 0 || A.nCol == 0) return B200SPMV_OK;
    int nb = want;
    if (want == 0) {
        if ((long long)A.nCol * 8 <= 64LL << 20) return B200SPMV_OK;     // x fits in L2 next to the matrix stream
        nb = (int)(((long long)A.nCol * 8 + COLBLOCK_SLICE_BYTES - 1) / COLBLOCK_SLICE_BYTES);
        if (nb > COLBLOCK_MAX) nb = COLBLOCK_MAX;
        const int B = (A.nCol + nb - 1) / nb;
        DevBuf<unsigned long long> stats;
        B2_TRY(stats.alloc(2));
        B2_CUDA(cudaMemsetAsync(stats.p, 0, stats.bytes(), s));
        colblock_spread_kernel<<<ceil_div(A.nRow, 256), 256, 0, s>>>(row_ptr, A.col, A.nRow, B, stats.p);
        B2_KERNEL_CHECK();
        unsigned long long st[2] = {0, 0};
        B2_CUDA(cudaMemcpyAsync(st, stats.p, sizeof st, cudaMemcpyDeviceToHost, s));
        B2_CUDA(cudaStreamSynchronize(s));
        // rows that each live in one block (stencils, banded matrices) already reuse x through L1 / L2
        if ((double)st[0] < 1.5 * (double)st[1]) return B200SPMV_OK;
    }
    const char *env_e = getenv("B200SPMV_COL_BLOCK_ENGINE");            // "crs" forces the tile-stream engine (tests, experiments)
    if (!(env_e && !strcmp(env_e, "crs"))) {
        B2_TRY(make_ell_col_blocks(A, row_ptr, nb, 0, CS_CONTINUE, 2.0, s, out));
        if (*out) return B200SPMV_OK;
    }
    b200spmv_options o{};
    o.segment_width = 1;
    o.n_block = nb;
    std::unique_ptr<CrsColBlocks> e(new CrsColBlocks(o));
    e->css.gather_bound = true;
    B2_TRY(e->css.convert(A, s));
    *out = std::move(e);
    return B200SPMV_OK;
}

}  // namespace b2
