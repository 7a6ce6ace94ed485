// csr5.cu -- CSR5-style plugin.  Algorithm source: Liu & Vinter's CSR5 as vendored by the reference under
// /root/reference/opt/Benchmark_SpMV_using_CSR5/ (there is no src/opt_csr5.cpp; SURVEY.md 8a a17/a18).
//   conversion: CSR5_cuda/anonymouslib_cuda.h:105-219 + detail/cuda/format_cuda.h, CPU twin
//               CSR5_avx2/detail/avx2/format_avx2.h:8-458 (the executable oracle, omega = 32)
//   multiply  : CSR5_cuda/detail/cuda/csr5_spmv_cuda.h:59-200 (tile), :313-382 (calibrate), :384-419 (tail)
//
// omega = 32 lanes (one warp per tile), sigma entries per lane, tile = omega*sigma consecutive non-zeros.
// Arrays produced on the device, bit-exact against the oracle:
//   tile_ptr[p+1]       row holding the tile's first non-zero; MSB = the tile's row span has an empty row
//   tile_desc[p*32*np]  per lane: y_offset | scansum_offset | sigma bit flags (1 = a row starts here)
//   tile_desc_offset_ptr[p+1], tile_desc_offset[]   y indices of the segments of empty-row tiles
//   col/val             transposed to step-major inside every full, non-fast-track tile
//
// Multiply = two launches, deterministic, true overwrite semantics (upstream needs a pre-zeroed y and
// three launches with CAS-loop atomics):
//   compute  : one warp per full tile.  Each lane walks its sigma entries (a warp request = 32 consecutive
//              entries), closes a segment at every bit flag and stores finished rows straight to y; the
//              partials that belong to a row opened by an earlier lane travel through a warp-shuffle
//              segmented sum (a tree, no subtractive scan); the tile's leading partial goes to carry[t].
//              Lanes of empty-row tiles zero the empty rows of their span.  Extra CTAs finish the tail
//              tile as plain CSR, one thread per row (sequential, reference order).
//   calibrate: one thread per tile; the first tile of each row adds that row's carries in tile order.
#include <cub/cub.cuh>
#include <type_traits>

#include "common.cuh"

namespace b2 {

constexpr int C5_OMEGA = 32;
constexpr int C5_WARPS = 4;               // tiles per CTA
constexpr uint32_t C5_MASK = 0x7FFFFFFFu;

__host__ __device__ __forceinline__ int count_le_dev(const int *a, int key, int size)
{
    int lo = 0, hi = size - 1;            // CSR5_*/detail/*/utils_*.h binary_search_right_boundary_kernel
    while (hi >= lo) {
        const int mid = (hi + lo) / 2;
        if (key >= a[mid]) lo = mid + 1;
        else hi = mid - 1;
    }
    return lo;
}

// ---------------------------------------------------------------- conversion
__global__ void c5_tile_ptr_kernel(const int *__restrict__ row_ptr, int m, int nnz, int T, int p, uint32_t *__restrict__ tile_ptr)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t > p) return;
    const long long b = (long long)t * T;
    const int boundary = b > nnz ? nnz : (int)b;
    tile_ptr[t] = (uint32_t)(count_le_dev(row_ptr, boundary, m + 1) - 1);          // format_avx2.h:16-26
}

__global__ void c5_dirty_kernel(const int *__restrict__ row_ptr, int m, int p, uint32_t *__restrict__ tile_ptr)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= p) return;
    const uint32_t start = tile_ptr[t] & C5_MASK, stop = tile_ptr[t + 1] & C5_MASK;
    if (start == stop) return;
    for (uint32_t r = start; r <= stop && r < (uint32_t)m; r++)                      // format_avx2.h:48-61
        if (row_ptr[r] == row_ptr[r + 1]) {
            tile_ptr[t] = start | 0x80000000u;
            return;
        }
}

__global__ void c5_flag_kernel(const int *__restrict__ row_ptr, int m, int sigma, int p, int bit_all, int num_packet,
                               uint32_t *__restrict__ desc)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r > m) return;
    const int ptr = row_ptr[r], pid = ptr / (C5_OMEGA * sigma);
    if (pid >= p - 1) return;                                                       // format_avx2.h:99-122 (full tiles only)
    const int lx = (ptr / sigma) % C5_OMEGA, glid = ptr % sigma + bit_all;
    atomicOr(&desc[(size_t)pid * C5_OMEGA * num_packet + (size_t)(glid / 32) * C5_OMEGA + lx], 1u << (31 - glid % 32));
}

// the sigma bit flags of a lane, step i at bit (31 - i)
__device__ __forceinline__ uint32_t c5_lane_flags(const uint32_t *__restrict__ dt, int lane, int num_packet, int bit_all, int sigma)
{
    uint64_t w = (uint64_t)dt[lane] << 32;
    if (num_packet > 1) w |= dt[C5_OMEGA + lane];
    w <<= bit_all;
    uint32_t f = (uint32_t)(w >> 32);
    if (sigma < 32) f &= ~((1u << (32 - sigma)) - 1u);
    return f;
}

// warp per full tile: y_offset, scansum_offset, per-tile segment count of empty-row tiles (format_avx2.h:125-233)
__global__ void c5_desc_kernel(const uint32_t *__restrict__ tile_ptr, uint32_t *__restrict__ desc, int *__restrict__ cnt,
                               int sigma, int p, int bit_y, int bit_all, int num_packet)
{
    const int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (t >= p - 1) return;
    const uint32_t ts = tile_ptr[t];
    const uint32_t start = ts & C5_MASK, stop = tile_ptr[t + 1] & C5_MASK;
    if (start == stop) return;
    uint32_t *dt = desc + (size_t)t * C5_OMEGA * num_packet;
    uint32_t f = c5_lane_flags(dt, lane, num_packet, bit_all, sigma);
    if (lane == 0) f |= 0x80000000u;
    const int segn = __popc(f);
    int scan = segn;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, scan, o);
        if (lane >= o) scan += v;
    }
    const int total = __shfl_sync(0xffffffffu, scan, 31);
    const int excl = scan - segn;
    const uint32_t present = __ballot_sync(0xffffffffu, f != 0);
    int sso = 0;
    if (f != 0 && lane < 31) {
        const uint32_t higher = present >> (lane + 1);
        sso = higher ? __ffs(higher) - 1 : 31 - lane;
    }
    const int y_offset = lane ? excl - 1 : 0;
    dt[lane] |= ((uint32_t)y_offset << (32 - bit_y)) | ((uint32_t)sso << (32 - bit_all));
    if (lane == 0 && (ts >> 31)) cnt[t] = total;
}

// warp per empty-row tile: true y index of every segment (format_avx2.h:279-349)
__global__ void c5_offset_kernel(const int *__restrict__ row_ptr, const uint32_t *__restrict__ tile_ptr,
                                 const uint32_t *__restrict__ desc, const int *__restrict__ offset_ptr,
                                 int *__restrict__ offset, int sigma, int p, int bit_y, int bit_all, int num_packet)
{
    const int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (t >= p - 1) return;
    const uint32_t ts = tile_ptr[t];
    if (!(ts >> 31)) return;
    const int start = (int)(ts & C5_MASK), stop = (int)(tile_ptr[t + 1] & C5_MASK);
    const uint32_t *dt = desc + (size_t)t * C5_OMEGA * num_packet;
    int y_offset = (int)(dt[lane] >> (32 - bit_y));
    const uint32_t f = c5_lane_flags(dt, lane, num_packet, bit_all, sigma);
    const int base = offset_ptr[t];
    for (int i = 0; i < sigma; i++) {
        if (!((f >> (31 - i)) & 1u) || (lane == 0 && i == 0)) continue;
        const int idx = t * C5_OMEGA * sigma + lane * sigma + i;
        offset[base + y_offset] = count_le_dev(row_ptr + start + 1, idx, stop - start) - 1;
        y_offset++;
    }
}

// (lane l, step i): l*sigma+i -> i*32+l inside full tiles whose raw tile_ptr differs from the next (format_avx2.h:366-420)
template <typename VT>
__global__ void c5_transpose_kernel(const int *__restrict__ col, const double *__restrict__ val, const uint32_t *__restrict__ tile_ptr,
                                    int nnz, int sigma, int p, int *__restrict__ col_out, VT *__restrict__ val_out)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nnz) return;
    const int T = C5_OMEGA * sigma, t = k / T;
    int src = k;
    if (t < p - 1 && tile_ptr[t] != tile_ptr[t + 1]) {
        const int d = k - t * T, i = d / C5_OMEGA, l = d % C5_OMEGA;
        src = t * T + l * sigma + i;
    }
    col_out[k] = col[src];
    val_out[k] = (VT)val[src];                       // fp32 storage (options.precision): rounded once, here
}

// ---------------------------------------------------------------- multiply
// VT = stored value type, XT = type of x and y, AT = type of the products and segment sums (carries stay fp64)
__device__ __forceinline__ double c5_ld_val(const double *p, uint64_t pol) { return ld_stream_d1(p, pol); }
__device__ __forceinline__ float c5_ld_val(const float *p, uint64_t pol)
{
    float r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(r) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

template <typename VT, typename XT, typename AT>
__global__ void __launch_bounds__(C5_WARPS * 32)
c5_compute_kernel(const int *__restrict__ col, const VT *__restrict__ val, const int *__restrict__ row_ptr,
                  const uint32_t *__restrict__ tile_ptr, const uint32_t *__restrict__ desc,
                  const int *__restrict__ offset_ptr, const int *__restrict__ offset, const XT *__restrict__ x,
                  XT *__restrict__ y, double *__restrict__ carry, int m, int sigma, int p, int bit_y, int bit_all,
                  int num_packet, int nTileBlocks)
{
    const int lane = threadIdx.x & 31;
    const int T = C5_OMEGA * sigma;
    const uint64_t pol_stream = policy_evict_first(), pol_x = policy_evict_last();

    if ((int)blockIdx.x >= nTileBlocks) {
        // ---- tail tile: plain CSR, one thread per row, sequential in the reference's order
        const int r0 = (int)(tile_ptr[p - 1] & C5_MASK);
        const int r = r0 + ((int)blockIdx.x - nTileBlocks) * blockDim.x + threadIdx.x;
        if (r >= m) return;
        const int b = r == r0 ? (p - 1) * T : row_ptr[r], e = row_ptr[r + 1];
        AT acc = (AT)0;
        for (int j = b; j < e; j++) acc = Arith<AT>::add(acc, Arith<AT>::mul((AT)val[j], (AT)ld_x(x + col[j], pol_x)));
        if (r == r0) carry[p - 1] = (double)acc;       // the row may have started in an earlier tile
        else y[r] = (XT)acc;
        return;
    }

    const int t = blockIdx.x * C5_WARPS + (threadIdx.x >> 5);
    if (t >= p - 1) return;
    const uint32_t ts = tile_ptr[t];
    const int start = (int)(ts & C5_MASK), stop = (int)(tile_ptr[t + 1] & C5_MASK);
    const int *c = col + (size_t)t * T + lane;
    const VT *v = val + (size_t)t * T + lane;

    if (start == stop) {                       // fast track: the whole tile lies inside one row
        AT sum = (AT)0;
        for (int i = 0; i < sigma; i++)
            sum += (AT)c5_ld_val(v + i * C5_OMEGA, pol_stream) * (AT)ld_x(x + ld_stream_i1(c + i * C5_OMEGA, pol_stream), pol_x);
        sum = warp_sum(sum);
        if (lane == 0) carry[t] = (double)sum;
        return;
    }

    const bool dirty = ts >> 31;
    const uint32_t *dt = desc + (size_t)t * C5_OMEGA * num_packet;
    int y_offset = (int)(dt[lane] >> (32 - bit_y));
    uint32_t flags = c5_lane_flags(dt, lane, num_packet, bit_all, sigma);
    const bool starts_row = flags >> 31;       // a row starts at this lane's first entry
    if (lane == 0) flags |= 0x80000000u;       // csr5_spmv_cuda.h:138
    XT *yt = y + start + 1;
    const int *off = dirty ? offset + offset_ptr[t] : nullptr;

    if (dirty)                                  // beta = 0: rows without entries inside this tile's span
        for (int r = start + 1 + lane; r <= stop && r < m; r += 32)
            if (row_ptr[r] == row_ptr[r + 1]) y[r] = (XT)0;

    // ---- thread-level segmented sums (csr5_spmv_cuda.h:141-176)
    bool direct = starts_row && lane != 0;
    AT sum = (AT)0, first_sum = (AT)0;
    constexpr int CH = 4;                       // entries per lane in flight (8: 72 registers, 37 % occupancy in ncu)
    for (int i0 = 0; i0 < sigma; i0 += CH) {
        int cc[CH];
        VT vv[CH];
        XT xx[CH];
#pragma unroll
        for (int u = 0; u < CH; u++)
            if (i0 + u < sigma) {
                cc[u] = ld_stream_i1(c + (i0 + u) * C5_OMEGA, pol_stream);
                vv[u] = c5_ld_val(v + (i0 + u) * C5_OMEGA, pol_stream);
            }
#pragma unroll
        for (int u = 0; u < CH; u++)
            if (i0 + u < sigma) xx[u] = ld_x(x + cc[u], pol_x);
#pragma unroll
        for (int u = 0; u < CH; u++) {
            const int i = i0 + u;
            if (i < sigma) {
                if (i > 0 && ((flags >> (31 - i)) & 1u)) {
                    if (direct) {
                        yt[off ? off[y_offset] : y_offset] = (XT)sum;
                        y_offset++;
                    } else {
                        first_sum = sum;
                    }
                    direct = true;
                    sum = (AT)0;
                }
                sum += (AT)vv[u] * (AT)xx[u];
            }
        }
    }
    if (!direct) first_sum = sum;               // no row starts in this lane (lane 0: none after its first entry)
    AT last_sum = sum;

    // ---- partials that belong to a row opened by an earlier lane: segmented sum by warp shuffles.
    // Lane k (k > 0, not starting a row) hands first_sum to the nearest lane j < k that holds a flag.
    const uint32_t present = __ballot_sync(0xffffffffu, flags != 0);
    const bool gives = lane != 0 && !starts_row;
    const int owner = lane ? 31 - __clz(present & ((1u << lane) - 1u)) : -1;     // lane 0 always holds a flag
    AT g = gives ? first_sum : (AT)0;
    const int key = gives ? owner : -2 - lane;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {                                           // suffix sums inside runs of equal key
        const AT gv = __shfl_down_sync(0xffffffffu, g, o);
        const int gk = __shfl_down_sync(0xffffffffu, key, o);
        if (lane + o < 32 && gk == key) g += gv;
    }
    const AT incoming = __shfl_down_sync(0xffffffffu, g, 1);                 // run of lane j starts at lane j + 1
    const int incoming_key = __shfl_down_sync(0xffffffffu, key, 1);
    if (flags != 0 && lane < 31 && incoming_key == lane) last_sum += incoming;

    if (direct) yt[off ? off[y_offset] : y_offset] = (XT)last_sum;                    // csr5_spmv_cuda.h:193-195
    if (lane == 0) carry[t] = (double)(direct ? first_sum : last_sum);                      // :198-199
    // fp32 vectors: the tile's last segment, whose row may go on into the next tile, also in fp64 for the calibration, so
    // that a row of fp64 sums (precision 2) is rounded to fp32 once
    if constexpr (std::is_same<XT, float>::value)
        if (direct && (present >> lane) == 1u) carry[p + t] = (double)last_sum;
}

// one thread per tile; the first tile of row R adds R's carries in tile order.  R's entries before that
// tile were stored by the compute kernel unless R starts exactly on the tile boundary.
template <typename XT>
__global__ void c5_calibrate_kernel(const int *__restrict__ row_ptr, const uint32_t *__restrict__ tile_ptr,
                                    const double *__restrict__ carry, XT *__restrict__ y, int p, int T)
{
    const int gid = blockIdx.x * blockDim.x + threadIdx.x;
    const int first_row = (int)(tile_ptr[0] & C5_MASK);
    for (int r = gid; r < first_row; r += gridDim.x * blockDim.x) y[r] = (XT)0;   // leading empty rows
    const int t = gid;
    if (t >= p) return;
    const uint32_t R = tile_ptr[t] & C5_MASK;
    if (t > 0 && (tile_ptr[t - 1] & C5_MASK) == R) return;
    double sum = 0.0;
    for (int u = t; u < p && (tile_ptr[u] & C5_MASK) == R; u++) sum += carry[u];
    if constexpr (std::is_same<XT, float>::value) y[R] = (XT)(row_ptr[R] == t * T ? sum : carry[p + t - 1] + sum);
    else y[R] = (XT)(row_ptr[R] == t * T ? sum : (double)y[R] + sum);
}

struct Csr5Format : Format {
    int sigma_opt, sigma = 0, p = 0, bit_y = 0, bit_ss = 0, num_packet = 0, num_offsets = 0;
    DevBuf<int> row_ptr, col, offset_ptr, offset;
    DevBuf<uint32_t> tile_ptr, desc;
    DevBuf<double> val, carry;
    DevBuf<float> val32;                  // options.precision = 1 / 2
    int tail_rows = 0, prec = 0;

    explicit Csr5Format(const b200spmv_options &o) : sigma_opt(o.csr5_sigma), prec(o.precision) {}

    int convert(const CooView &A, cudaStream_t s) override
    {
        nRow = A.nRow; nCol = A.nCol; nnz = A.nnz;
        B2_TRY(validate_sorted_coo(A, s));
        sigma = sigma_opt;
        if (sigma <= 0) {                                   // upstream's auto-tuning rule, anonymouslib_cuda.h:293-317
            const int per_row = nRow > 0 ? nnz / nRow : 0;
            sigma = per_row <= 4 ? 4 : per_row <= 32 ? per_row : per_row <= 256 ? 32 : 6;
            // 0 = tuned for B200: a warp needs at least 16 entries per lane in flight (c5, 7 nnz/row: sigma 6 -> 492,
            // sigma 16 -> 690 GFLOP/s); -1 = upstream's rule verbatim
            if (sigma_opt == 0 && sigma < 16) sigma = 16;
        }
        int base = 2;                                       // anonymouslib_cuda.h:121-137
        bit_y = 1;
        while (base < C5_OMEGA * sigma) { base *= 2; bit_y++; }
        bit_ss = 5;
        const int bit_all = bit_y + bit_ss, T = C5_OMEGA * sigma;
        num_packet = (bit_all + sigma + 31) / 32;
        p = (int)(((long long)nnz + T - 1) / T);
        B2_TRY(row_ptr.alloc((size_t)nRow + 1));
        B2_TRY(build_row_ptr(A.row, nnz, nRow, row_ptr.p, s));
        B2_TRY(tile_ptr.alloc((size_t)p + 1));
        B2_TRY(desc.alloc((size_t)p * C5_OMEGA * num_packet));
        B2_TRY(offset_ptr.alloc((size_t)p + 1));
        B2_TRY(col.alloc((size_t)nnz));
        if (prec) B2_TRY(val32.alloc((size_t)nnz));
        else B2_TRY(val.alloc((size_t)nnz));
        B2_TRY(carry.alloc((size_t)p * (prec ? 2 : 1)));   // fp32 vectors: [p + t] = fp64 last segment of tile t
        B2_CUDA(cudaMemsetAsync(desc.p, 0, desc.bytes() ? desc.bytes() : 4, s));
        DevBuf<int> cnt;
        B2_TRY(cnt.alloc((size_t)p + 1));
        B2_CUDA(cudaMemsetAsync(cnt.p, 0, cnt.bytes(), s));
        c5_tile_ptr_kernel<<<ceil_div((long long)p + 1, 256), 256, 0, s>>>(row_ptr.p, nRow, nnz, T, p, tile_ptr.p);
        if (p) c5_dirty_kernel<<<ceil_div(p, 256), 256, 0, s>>>(row_ptr.p, nRow, p, tile_ptr.p);
        c5_flag_kernel<<<ceil_div((long long)nRow + 1, 256), 256, 0, s>>>(row_ptr.p, nRow, sigma, p, bit_all, num_packet, desc.p);
        if (p > 1) c5_desc_kernel<<<ceil_div((long long)(p - 1) * 32, 256), 256, 0, s>>>(tile_ptr.p, desc.p, cnt.p, sigma, p, bit_y, bit_all, num_packet);
        B2_KERNEL_CHECK();
        B2_TRY(exclusive_scan_i32(cnt.p, offset_ptr.p, p + 1, s));                 // format_avx2.h:262-265
        B2_CUDA(cudaMemcpy(&num_offsets, offset_ptr.p + p, sizeof(int), cudaMemcpyDeviceToHost));
        B2_TRY(offset.alloc((size_t)num_offsets));
        // every empty-row tile owns one slot more than it has listed segments (its leading partial is never
        // listed); upstream leaves that slot uninitialised (anonymouslib_avx2.h:178-180), here it is 0
        B2_CUDA(cudaMemsetAsync(offset.p, 0, offset.bytes() ? offset.bytes() : 4, s));
        if (num_offsets) {
            c5_offset_kernel<<<ceil_div((long long)(p - 1) * 32, 256), 256, 0, s>>>(row_ptr.p, tile_ptr.p, desc.p, offset_ptr.p, offset.p,
                                                                                   sigma, p, bit_y, bit_all, num_packet);
            B2_KERNEL_CHECK();
        }
        if (nnz) {
            if (prec) c5_transpose_kernel<float><<<ceil_div(nnz, 256), 256, 0, s>>>(A.col, A.val, tile_ptr.p, nnz, sigma, p, col.p, val32.p);
            else c5_transpose_kernel<double><<<ceil_div(nnz, 256), 256, 0, s>>>(A.col, A.val, tile_ptr.p, nnz, sigma, p, col.p, val.p);
            B2_KERNEL_CHECK();
        }
        tail_rows = 0;
        if (p) {
            uint32_t r0 = 0;
            B2_CUDA(cudaMemcpyAsync(&r0, tile_ptr.p + (p - 1), sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
            B2_CUDA(cudaStreamSynchronize(s));
            tail_rows = nRow - (int)(r0 & C5_MASK);
        }
        B2_CUDA(cudaStreamSynchronize(s));
        return B200SPMV_OK;
    }

    template <typename VT, typename XT, typename AT> int run(const VT *v, const XT *x, XT *y, cudaStream_t s)
    {
        if (nRow == 0) return B200SPMV_OK;
        if (p == 0) {
            B2_CUDA(cudaMemsetAsync(y, 0, sizeof(XT) * (size_t)nRow, s));
            return B200SPMV_OK;
        }
        const int threads = C5_WARPS * 32;
        const int nTileBlocks = ceil_div(p - 1, C5_WARPS), nTailBlocks = ceil_div(tail_rows, threads);
        c5_compute_kernel<VT, XT, AT><<<nTileBlocks + nTailBlocks, threads, 0, s>>>(col.p, v, row_ptr.p, tile_ptr.p, desc.p, offset_ptr.p,
                                                                                  offset.p, x, y, carry.p, nRow, sigma, p, bit_y,
                                                                                  bit_y + bit_ss, num_packet, nTileBlocks);
        c5_calibrate_kernel<XT><<<ceil_div(p, 256), 256, 0, s>>>(row_ptr.p, tile_ptr.p, carry.p, y, p, C5_OMEGA * sigma);
        B2_KERNEL_CHECK();
        return B200SPMV_OK;
    }
    int multiply(const double *x, double *y, cudaStream_t s) override
    {
        if (prec) { set_error("multiply: the handle was created with precision = %d, use b200spmv_multiply_f32", prec); return B200SPMV_ERR_STATE; }
        return run<double, double, double>(val.p, x, y, s);
    }
    int multiply_f32(const float *x, float *y, cudaStream_t s) override
    {
        if (!prec) { set_error("multiply_f32: the handle was created with precision = 0 (fp64 vectors)"); return B200SPMV_ERR_STATE; }
        if (prec == 2) return run<float, float, double>(val32.p, x, y, s);
        return run<float, float, float>(val32.p, x, y, s);
    }

    bool scalar(const std::string &n, long long *out) override
    {
        if (n == "sigma") { *out = sigma; return true; }
        if (n == "p") { *out = p; return true; }
        if (n == "bit_y_offset") { *out = bit_y; return true; }
        if (n == "bit_scansum_offset") { *out = bit_ss; return true; }
        if (n == "num_packet") { *out = num_packet; return true; }
        if (n == "num_offsets") { *out = num_offsets; return true; }
        if (n == "alg_bytes") {   // SURVEY.md 8d: 12 nnz + 4 (nRow+1) + 4 (p+1) + 4 p omega num_packet + 8 nCol + 8 nRow
            *out = (prec ? 8LL : 12LL) * nnz + 4LL * (nRow + 1) + 4LL * (p + 1) + 4LL * p * C5_OMEGA * num_packet +
                   (prec ? 4LL : 8LL) * ((long long)nCol + nRow);
            return true;
        }
        if (n == "launches") { *out = p ? 2 : 1; return true; }
        if (n == "precision") { *out = prec; return true; }
        return false;
    }

    long long array(const std::string &n, void *dst, long long cap) override
    {
        if (n == "row_ptr") return export_device(row_ptr.p, row_ptr.bytes(), dst, cap);
        if (n == "tile_ptr") return export_device(tile_ptr.p, tile_ptr.bytes(), dst, cap);
        if (n == "tile_desc") return export_device(desc.p, desc.bytes(), dst, cap);
        if (n == "tile_desc_offset_ptr") return export_device(offset_ptr.p, offset_ptr.bytes(), dst, cap);
        if (n == "tile_desc_offset") return export_device(offset.p, offset.bytes(), dst, cap);
        if (n == "col_idx") return export_device(col.p, col.bytes(), dst, cap);
        if (n == "val" && !prec) return export_device(val.p, val.bytes(), dst, cap);
        return -1000;
    }
};

Format *make_csr5(const b200spmv_options &o) { return new Csr5Format(o); }

}  // namespace b2
