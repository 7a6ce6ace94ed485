// common.cuh -- shared host/device plumbing of libb200spmv (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "b200spmv.h"

namespace b2 {

// ---------------------------------------------------------------- errors
void set_error(const char *fmt, ...);
void clear_error();

#define B2_CUDA(expr)                                                                         \
    do {                                                                                      \
        cudaError_t e__ = (expr);                                                             \
        if (e__ != cudaSuccess) {                                                             \
            b2::set_error("%s: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
            return B200SPMV_ERR_CUDA;                                                         \
        }                                                                                     \
    } while (0)

#define B2_TRY(expr)                       \
    do {                                   \
        int s__ = (expr);                  \
        if (s__ != B200SPMV_OK) return s__; \
    } while (0)

#define B2_KERNEL_CHECK() B2_CUDA(cudaGetLastError())

// ---------------------------------------------------------------- device memory
template <typename T> struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() { release(); }
    void release()
    {
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
    }
    int alloc(size_t count)
    {
        release();
        n = count;
        if (count == 0) count = 1;   // keep pointers non-null so kernels can take them
        cudaError_t e = cudaMalloc((void **)&p, count * sizeof(T));
        if (e != cudaSuccess) {
            p = nullptr;
            n = 0;
            set_error("cudaMalloc(%zu bytes): %s", count * sizeof(T), cudaGetErrorString(e));
            return e == cudaErrorMemoryAllocation ? B200SPMV_ERR_NOMEM : B200SPMV_ERR_CUDA;
        }
        return B200SPMV_OK;
    }
    size_t bytes() const { return n * sizeof(T); }
};

// Copies a device array to a host destination with the get_array() size protocol.
long long export_device(const void *src_d, size_t bytes, void *dst_h, long long dst_bytes);
long long export_host(const void *src_h, size_t bytes, void *dst_h, long long dst_bytes);

// ---------------------------------------------------------------- input view + format interface
struct CooView {
    int nRow, nCol;
    int nnz;                 // < 2^31 like the reference (src/util.h:8)
    const int *row, *col;    // device
    const double *val;       // device
    int rowOffset = 0;       // global row of local row 0 (row blocks of a larger matrix, blocked.cu): only locality heuristics use it
};

// how a multiply over a row range treats what y already holds (shared by the tile-stream and the row-chunk stream)
enum { CS_OVERWRITE = 0,           // y[r] = sum
       CS_CONTINUE = 1,            // acc = y[r]; acc += a_ij x_j ...; y[r] = acc   (next column block of the SAME running sum)
       CS_ADD = 2 };               // y[r] = y[r] + sum                            (CSS: block sums added, src/opt_css.cpp:298)

struct Format {
    int nRow = 0, nCol = 0, nnz = 0;
    virtual ~Format() {}
    virtual int convert(const CooView &A, cudaStream_t s) = 0;
    virtual int multiply(const double *x, double *y, cudaStream_t s) = 0;
    // options.precision = 1 / 2: fp32 matrix values and vectors (accumulation in fp32 / fp64)
    virtual int multiply_f32(const float *, float *, cudaStream_t)
    {
        set_error("multiply_f32: this format has no fp32 variant (CRS, ELL and DIA do)");
        return B200SPMV_ERR_UNSUPPORTED;
    }
    // Y[:, 0..k) := A X[:, 0..k), X and Y row-major with leading dimensions ldx, ldy (b200spmv_multiply_multi)
    virtual int multiply_multi(int, const double *, long long, double *, long long, cudaStream_t)
    {
        set_error("multiply_multi: this format has no multi-vector multiply (CRS has)");
        return B200SPMV_ERR_UNSUPPORTED;
    }
    // the same with fp32 vectors (b200spmv_multiply_multi_f32, options.precision = 1 / 2)
    virtual int multiply_multi_f32(int, const float *, long long, float *, long long, cudaStream_t)
    {
        set_error("multiply_multi_f32: this format has no multi-vector multiply (CRS has)");
        return B200SPMV_ERR_UNSUPPORTED;
    }
    virtual int multiply_rows(int, int, const double *, double *, cudaStream_t)
    {
        set_error("multiply_rows: this format does not support row ranges (CRS, SS, CSS, ELL, DIA do)");
        return B200SPMV_ERR_UNSUPPORTED;
    }
    // host-side bookkeeping for a row range (may synchronise): afterwards multiply_rows on it never does
    virtual int prepare_rows(int, int) { return B200SPMV_OK; }
    // smallest / largest column referenced by rows [rb, re) (conservative; may synchronise).  The host-semantics
    // pipeline uploads x in ascending pieces and starts a row chunk as soon as the pieces up to its largest column
    // have landed: banded matrices (stencils) multiply while most of x is still crossing PCIe.
    virtual int col_extent(int, int, int *cmin, int *cmax) { *cmin = 0; *cmax = nCol - 1; return B200SPMV_OK; }
    virtual bool has_rows() const { return false; }      // multiply_rows available (host-semantics pipeline uses it)
    // Column slices of x in order of first use (CSS: one per column block; everything else: all of x at once).
    // multiply_rows_slice(i, ...) adds slice i's contribution to rows [rb, re) (slice 0 overwrites), so the host
    // pipeline can start multiplying while later slices of x are still crossing PCIe.
    virtual int n_x_slices() const { return 1; }
    virtual void x_slice(int, long long *c0, long long *c1) const { *c0 = 0; *c1 = nCol; }
    virtual int multiply_rows_slice(int, int rb, int re, const double *x, double *y, cudaStream_t s) { return multiply_rows(rb, re, x, y, s); }
    // format-specific scalars/arrays; return false / -1 when the name is unknown
    virtual bool scalar(const std::string &name, long long *out) = 0;
    virtual long long array(const std::string &name, void *dst_h, long long dst_bytes) = 0;
    virtual int set_perm(const int *, int)
    {
        set_error("set_perm: only the JDS format takes a row permutation");
        return B200SPMV_ERR_UNSUPPORTED;
    }
};

Format *make_crs(const b200spmv_options &);
Format *make_coo(const b200spmv_options &);
Format *make_ell(const b200spmv_options &);
Format *make_jds(const b200spmv_options &);
Format *make_dia(const b200spmv_options &);
Format *make_ss(const b200spmv_options &);
Format *make_css(const b200spmv_options &);
Format *make_csr5(const b200spmv_options &);
Format *make_hyb(const b200spmv_options &);

// ---------------------------------------------------------------- shared device passes (primitives.cu)
// ptr[r] = first index i with row[i] >= r, ptr[nRow] = nnz  (reference src/opt_crs.cpp:27-33)
int build_row_ptr(const int *row_d, int nnz, int nRow, int *ptr_d, cudaStream_t s);
// max over r of ptr[r+1]-ptr[r]; synchronises the stream
int max_row_length(const int *ptr_d, int nRow, int *out_h, cudaStream_t s);
// exclusive prefix sums (CUB); out may alias in; n >= 0
int exclusive_scan_i32(const int *in_d, int *out_d, int n, cudaStream_t s);
int exclusive_scan_i64(const long long *in_d, long long *out_d, int n, cudaStream_t s);
int sum_i32_as_i64(const int *in_d, int n, long long *out_h, cudaStream_t s);
// min and max of the non-negative values of in_d[b..e) (negative ones are ELL padding); synchronous
int minmax_i32(const int *in_d, long long b, long long e, int *mn_h, int *mx_h);
// largest |col - row| (synchronises); gathers_need_l2: the x entries a stretch of rows touches span more than 32 MB
int max_band(const int *row_d, const int *col_d, int nnz, int rowOffset, int *band_h, cudaStream_t s);
// the same from a CRS matrix (columns ascending within a row: a row's first and last entry are its extremes)
int max_band_crs(const int *ptr_d, const int *idx_d, int nRow, int rowOffset, int *band_h, cudaStream_t s);
bool gathers_need_l2(int band);
// checks the input contract: sorted by (row, col), no duplicates, indices in range
int validate_sorted_coo(const CooView &A, cudaStream_t s);

static inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

// ---------------------------------------------------------------- device helpers
#ifdef __CUDACC__
// Matrix arrays are read exactly once per multiply: stream them around L1 and mark the lines
// evict-first in L2 so that they do not push x (the only reused operand) out of the 126 MB L2.
__device__ __forceinline__ uint64_t policy_evict_first()
{
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ uint64_t policy_evict_last()
{
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ int4 ld_stream_i4(const int *p, uint64_t pol)
{
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.s32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ int2 ld_stream_i2(const int *p, uint64_t pol)
{
    int2 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v2.s32 {%0,%1}, [%2], %3;"
                 : "=r"(r.x), "=r"(r.y) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ int ld_stream_i1(const int *p, uint64_t pol)
{
    int r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.s32 %0, [%1], %2;"
                 : "=r"(r) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ double2 ld_stream_d2(const double *p, uint64_t pol)
{
    double2 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v2.f64 {%0,%1}, [%2], %3;"
                 : "=d"(r.x), "=d"(r.y) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ double ld_stream_d1(const double *p, uint64_t pol)
{
    double r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.f64 %0, [%1], %2;"
                 : "=d"(r) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ float4 ld_stream_f4(const float *p, uint64_t pol)
{
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p), "l"(pol));
    return r;
}
// x gathers: cached in L1 (stencil reuse) and kept in L2 with evict-last priority.
__device__ __forceinline__ double ld_x(const double *p, uint64_t pol)
{
    double r;
    asm volatile("ld.global.nc.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(r) : "l"(p), "l"(pol));
    return r;
}
// ---------------------------------------------------------------- mbarrier / TMA (sm_90+ PTX)
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    uint32_t done;
    do {
        asm volatile("{\n\t.reg .pred p;\n\t"
                     "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                     "selp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    } while (!done);
}
// 1-D bulk copy global -> shared through the TMA unit; bytes % 16 == 0, both addresses 16-byte aligned
__device__ __forceinline__ void tma_load_1d(void *dst_smem, const void *src, uint32_t bytes, uint64_t *bar,
                                            uint64_t pol)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint "
                 "[%0], [%1], %2, [%3], %4;"
                 ::"r"(smem_u32(dst_smem)), "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(pol) : "memory");
}

// Arithmetic of one precision: unfused multiply and add (the reference's g++ -O2 build does not contract, and a fixed
// operation order keeps every kernel deterministic), and the x gather with the L2 evict-last hint.
template <typename T> struct Arith;
template <> struct Arith<double> {
    static __device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
    static __device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
};
template <> struct Arith<float> {
    static __device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
    static __device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
};
__device__ __forceinline__ float ld_x(const float *p, uint64_t pol)
{
    float r;
    asm volatile("ld.global.nc.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(r) : "l"(p), "l"(pol));
    return r;
}

// Gathers of the multi-vector multiply (X row-major, X[c*ldx + j]): the hint of ld_x, but not volatile, so that the
// compiler may batch the loads of several entries.  ld_xrow reads X[c*ldx + j0 + v] for v < min(KP, k - j0) (the other
// slots read nothing and hold 0): with W2 (ldx even, X 16-byte aligned, j0 even) pairs of columns come in one 16-byte load.
__device__ __forceinline__ double ld_xm(const double *p, uint64_t pol)
{
    double r;
    asm("ld.global.nc.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(r) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ double2 ld_xm2(const double *p, uint64_t pol)
{
    double2 r;
    asm("ld.global.nc.L2::cache_hint.v2.f64 {%0,%1}, [%2], %3;" : "=d"(r.x), "=d"(r.y) : "l"(p), "l"(pol));
    return r;
}
template <int KP, bool W2>
__device__ __forceinline__ void ld_xrow(double (&xv)[KP], const double *p, int n, uint64_t pol)
{
#pragma unroll
    for (int v = 0; v < KP; v += W2 ? 2 : 1) {
        if (W2 && v + 1 < KP) {
            if (v + 1 < n) {
                const double2 t = ld_xm2(p + v, pol);
                xv[v] = t.x;
                xv[v + 1] = t.y;
            } else {
                xv[v] = v < n ? ld_xm(p + v, pol) : 0.0;
                xv[v + 1] = 0.0;
            }
        } else {
            xv[v] = v < n ? ld_xm(p + v, pol) : 0.0;
        }
    }
}
// fp32 X: with VEC (ldx a multiple of W = min(KP, 4), X aligned to W floats, j0 a multiple of W) groups of W columns come
// in one 8- or 16-byte load; one row of X holds up to 8 columns in a single 32-byte sector.
__device__ __forceinline__ float ld_xm(const float *p, uint64_t pol)
{
    float r;
    asm("ld.global.nc.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(r) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ float2 ld_xm2(const float *p, uint64_t pol)
{
    float2 r;
    asm("ld.global.nc.L2::cache_hint.v2.f32 {%0,%1}, [%2], %3;" : "=f"(r.x), "=f"(r.y) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ float4 ld_xm4(const float *p, uint64_t pol)
{
    float4 r;
    asm("ld.global.nc.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
        : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p), "l"(pol));
    return r;
}
template <int KP, bool VEC>
__device__ __forceinline__ void ld_xrow(float (&xv)[KP], const float *p, int n, uint64_t pol)
{
    constexpr int W = VEC ? (KP < 4 ? KP : 4) : 1;
#pragma unroll
    for (int v = 0; v < KP; v += W) {
        if (W == 4 && v + W - 1 < n) {
            const float4 t = ld_xm4(p + v, pol);
            xv[v] = t.x; xv[v + 1] = t.y; xv[v + 2] = t.z; xv[v + 3] = t.w;
        } else if (W == 2 && v + W - 1 < n) {
            const float2 t = ld_xm2(p + v, pol);
            xv[v] = t.x; xv[v + 1] = t.y;
        } else {
#pragma unroll
            for (int i = 0; i < W; i++) xv[v + i] = v + i < n ? ld_xm(p + v + i, pol) : 0.0f;
        }
    }
}
#endif
// The vector gathers ld_xrow may use for k columns of X (KP = k rounded up): pairs of fp64 columns, W = min(KP, 4) fp32
// columns; ldx and X must be aligned to that width
template <typename XT>
static inline bool ld_xrow_vec(const XT *X, long long ldx, int KP)
{
    const int w = sizeof(XT) == 8 ? 2 : (KP < 4 ? KP : 4);
    return ldx % w == 0 && reinterpret_cast<uintptr_t>(X) % (w * sizeof(XT)) == 0;
}
#ifdef __CUDACC__

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
#endif

}  // namespace b2
