// api.cu -- the extern "C" surface declared in include/b200spmv.h.
#include <algorithm>
#include <cstdlib>

#include "common.cuh"

namespace b2 {
Format *make_format(int format, const b200spmv_options &o);
const char *last_error_cstr();
// blocked.cu: more than 2^31-1 entries (or B200SPMV_BLOCK_NNZ) -> contiguous row blocks of the requested format
int convert_row_blocked(int format, const b200spmv_options &opt, int nRow, int nCol, long long nnz, const int *row_d,
                        const int *col_d, const double *val_d, cudaStream_t s, std::unique_ptr<Format> &out);
long long row_block_limit();
// transpose.cu: A^T's sorted COO (nnz entries) from A's
int transpose_coo(int nCol, long long nnz, const int *row_d, const int *col_d, const double *val_d, cudaStream_t s,
                  DevBuf<int> &rowT, DevBuf<int> &colT, DevBuf<double> &valT);
}
using namespace b2;

constexpr int MAX_HOST_CHUNKS = 32;
constexpr int MAX_HOST_SLICES = 64;

struct b200spmv_matrix {
    int format = 0;
    b200spmv_options opt{};
    std::unique_ptr<Format> impl;
    bool converted = false, blocked = false;
    // options.transpose = 1: A^T, converted from A's transposed COO with the same format and options (row-blocked on its own)
    std::unique_ptr<Format> timpl;
    bool tblocked = false;
    // plan of the host-semantics pipeline (built on first use)
    int plan_chunks = 0, plan_pieces = 0;
    int chunk_rb[MAX_HOST_CHUNKS + 1] = {}, chunk_need[MAX_HOST_CHUNKS] = {};
    long long piece_c0[MAX_HOST_SLICES + 1] = {};
    // staging for host-semantics multiply
    DevBuf<double> x_stage, y_stage;
    DevBuf<float> x_stage32, y_stage32;
    cudaStream_t stream = nullptr, copy_stream = nullptr, in_stream = nullptr;
    cudaEvent_t chunk_done[MAX_HOST_CHUNKS] = {};
    cudaEvent_t slice_in[MAX_HOST_SLICES] = {};
    ~b200spmv_matrix()
    {
        if (stream) cudaStreamDestroy(stream);
        if (copy_stream) cudaStreamDestroy(copy_stream);
        if (in_stream) cudaStreamDestroy(in_stream);
        for (auto e : chunk_done) if (e) cudaEventDestroy(e);
        for (auto e : slice_in) if (e) cudaEventDestroy(e);
    }
};

Format *b2::make_format(int format, const b200spmv_options &o)
{
    switch (format) {
    case B200SPMV_CRS: return make_crs(o);
    case B200SPMV_COO: return make_coo(o);
    case B200SPMV_ELL: return make_ell(o);
    case B200SPMV_JDS: return make_jds(o);
    case B200SPMV_DIA: return make_dia(o);
    case B200SPMV_SS: return make_ss(o);
    case B200SPMV_CSS: return make_css(o);
    case B200SPMV_CSR5: return make_csr5(o);
    case B200SPMV_HYB: return make_hyb(o);
    default: return nullptr;
    }
}

static int require_device()
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        set_error("no CUDA device available (%s); libb200spmv has no CPU fallback",
                  e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
        return B200SPMV_ERR_CUDA;
    }
    return B200SPMV_OK;
}

extern "C" {

int b200spmv_version(void) { return B200SPMV_VERSION; }

const char *b200spmv_last_error(void) { return last_error_cstr(); }

int b200spmv_device_count(int *count)
{
    if (!count) return B200SPMV_ERR_INVALID;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        cudaGetLastError();
        n = 0;
    }
    *count = n;
    return B200SPMV_OK;
}

int b200spmv_create(int format, const b200spmv_options *opts, b200spmv_matrix **out)
{
    clear_error();
    if (!out) {
        set_error("create: out is NULL");
        return B200SPMV_ERR_INVALID;
    }
    *out = nullptr;
    b200spmv_options o{};
    if (opts) o = *opts;
    if (o.segment_width == 0) o.segment_width = 4;     // ALIGNMENT/sizeof(double), param.h:9-11 with ALIGNMENT=32
    if (o.n_block == 0) o.n_block = 1;                 // param.h:18-20
    if (o.segment_width < 1 || (o.segment_width & (o.segment_width - 1))) {
        set_error("create: segment_width=%d must be a power of two (reference src/opt_ss.cpp:272 masks with W-1)", o.segment_width);
        return B200SPMV_ERR_INVALID;
    }
    if (o.n_block < 1 || o.csr5_sigma < -1 || o.csr5_sigma > 32) {
        set_error("create: bad option (n_block=%d csr5_sigma=%d)", o.n_block, o.csr5_sigma);
        return B200SPMV_ERR_INVALID;
    }
    if (o.crs_path == 2) {
        set_error("create: crs_path=2 selected round 1's row-block stream, which was removed; 3 selects the row-chunk stream");
        return B200SPMV_ERR_INVALID;
    }
    if (o.crs_path < 0 || o.crs_path > 4 || o.coo_path < 0 || o.coo_path > 3) {
        set_error("create: bad option (crs_path=%d, 0..4 without 2; coo_path=%d, 0..3)", o.crs_path, o.coo_path);
        return B200SPMV_ERR_INVALID;
    }
    if (o.hyb_k < 0) {
        set_error("create: hyb_k=%d (0 = the width rule, > 0 = that width)", o.hyb_k);
        return B200SPMV_ERR_INVALID;
    }
    if (o.value_f32 && format != B200SPMV_CRS) {
        set_error("create: value_f32 is implemented for the CRS format only");
        return B200SPMV_ERR_UNSUPPORTED;
    }
    if (o.precision < 0 || o.precision > 2) { set_error("create: precision=%d (0 fp64, 1 fp32, 2 fp32 with fp64 sums)", o.precision); return B200SPMV_ERR_INVALID; }
    if (o.transpose != 0 && o.transpose != 1) { set_error("create: transpose=%d (0 or 1)", o.transpose); return B200SPMV_ERR_INVALID; }
    if (o.precision && format != B200SPMV_CRS && format != B200SPMV_ELL && format != B200SPMV_DIA && format != B200SPMV_CSR5) {
        set_error("create: the fp32 variant exists for the CRS, ELL, DIA and CSR5 formats");
        return B200SPMV_ERR_UNSUPPORTED;
    }
    Format *f = make_format(format, o);
    if (!f) {
        set_error("create: unknown format %d", format);
        return B200SPMV_ERR_INVALID;
    }
    b200spmv_matrix *m = new b200spmv_matrix();
    m->format = format;
    m->opt = o;
    m->impl.reset(f);
    *out = m;
    return B200SPMV_OK;
}

int b200spmv_destroy(b200spmv_matrix *m)
{
    delete m;
    return B200SPMV_OK;
}

// Converts a sorted COO into impl: row blocks beyond row_block_limit(), else impl's own convert (a row-blocked impl is
// replaced by a plain one first)
static int convert_impl(int format, const b200spmv_options &opt, int nRow, int nCol, long long nnz, const int *row_d,
                        const int *col_d, const double *val_d, cudaStream_t s, std::unique_ptr<Format> &impl,
                        bool &blocked)
{
    if (nnz > row_block_limit()) {
        // beyond the reference's int32 entry count (src/util.h:8): row blocks with 32-bit offsets each (blocked.cu)
        std::unique_ptr<Format> f;
        B2_TRY(convert_row_blocked(format, opt, nRow, nCol, nnz, row_d, col_d, val_d, s, f));
        impl = std::move(f);
        blocked = true;
        return B200SPMV_OK;
    }
    if (blocked) {
        impl.reset(make_format(format, opt));
        blocked = false;
    }
    CooView A{nRow, nCol, (int)nnz, row_d, col_d, val_d};
    return impl->convert(A, s);
}

// A^T: its COO (transpose.cu), then a fresh matrix of the handle's format and options converted from it like A
static int convert_transpose(b200spmv_matrix *m, int nRow, int nCol, long long nnz, const int *row_d, const int *col_d,
                             const double *val_d, cudaStream_t s)
{
    DevBuf<int> rowT, colT;
    DevBuf<double> valT;
    B2_TRY(transpose_coo(nCol, nnz, row_d, col_d, val_d, s, rowT, colT, valT));
    b200spmv_options o = m->opt;
    o.transpose = 0;
    m->timpl.reset(make_format(m->format, o));
    m->tblocked = false;
    B2_TRY(convert_impl(m->format, o, nCol, nRow, nnz, rowT.p, colT.p, valT.p, s, m->timpl, m->tblocked));
    B2_CUDA(cudaStreamSynchronize(s));                           // A^T's COO is freed on return
    return B200SPMV_OK;
}

int b200spmv_convert_coo_device(b200spmv_matrix *m, int nRow, int nCol, long long nnz, const int *row_d,
                                const int *col_d, const double *val_d, void *stream)
{
    clear_error();
    if (!m) { set_error("convert: NULL handle"); return B200SPMV_ERR_INVALID; }
    if (nRow < 0 || nCol < 0 || nnz < 0) { set_error("convert: negative dimension (nRow=%d nCol=%d nnz=%lld)", nRow, nCol, nnz); return B200SPMV_ERR_INVALID; }
    if (nnz > 0 && (!row_d || !col_d || !val_d)) { set_error("convert: NULL COO array"); return B200SPMV_ERR_INVALID; }
    B2_TRY(require_device());
    m->converted = false;
    m->plan_chunks = m->plan_pieces = 0;
    m->timpl.reset();                                           // the old A^T's memory is free while the new one is built
    B2_TRY(convert_impl(m->format, m->opt, nRow, nCol, nnz, row_d, col_d, val_d, (cudaStream_t)stream, m->impl, m->blocked));
    if (m->opt.transpose) {
        const int st = convert_transpose(m, nRow, nCol, nnz, row_d, col_d, val_d, (cudaStream_t)stream);
        if (st != B200SPMV_OK) {
            m->timpl.reset();
            const std::string why = last_error_cstr();
            set_error("convert: the transposed conversion (A^T, %d x %d) failed: %s", nCol, nRow, why.c_str());
            return st;
        }
    }
    m->converted = true;
    return B200SPMV_OK;
}

int b200spmv_convert_coo_host(b200spmv_matrix *m, int nRow, int nCol, long long nnz, const int *row_h,
                              const int *col_h, const double *val_h)
{
    clear_error();
    if (!m) { set_error("convert: NULL handle"); return B200SPMV_ERR_INVALID; }
    if (nnz < 0) { set_error("convert: nnz=%lld", nnz); return B200SPMV_ERR_INVALID; }
    if (nnz > 0 && (!row_h || !col_h || !val_h)) { set_error("convert: NULL COO array"); return B200SPMV_ERR_INVALID; }
    B2_TRY(require_device());
    DevBuf<int> r, c;
    DevBuf<double> v;
    B2_TRY(r.alloc((size_t)nnz));
    B2_TRY(c.alloc((size_t)nnz));
    B2_TRY(v.alloc((size_t)nnz));
    if (nnz) {
        B2_CUDA(cudaMemcpy(r.p, row_h, r.bytes(), cudaMemcpyHostToDevice));
        B2_CUDA(cudaMemcpy(c.p, col_h, c.bytes(), cudaMemcpyHostToDevice));
        B2_CUDA(cudaMemcpy(v.p, val_h, v.bytes(), cudaMemcpyHostToDevice));
    }
    return b200spmv_convert_coo_device(m, nRow, nCol, nnz, r.p, c.p, v.p, nullptr);
}

int b200spmv_jds_set_perm_host(b200spmv_matrix *m, const int *perm_h, int nRow)
{
    clear_error();
    if (!m || !perm_h) { set_error("jds_set_perm: NULL argument"); return B200SPMV_ERR_INVALID; }
    return m->impl->set_perm(perm_h, nRow);
}

static int check_ready(b200spmv_matrix *m, const void *x, const void *y)
{
    if (!m) { set_error("multiply: NULL handle"); return B200SPMV_ERR_INVALID; }
    if (!m->converted) { set_error("multiply: matrix not converted yet"); return B200SPMV_ERR_STATE; }
    if ((!x && m->impl->nCol > 0) || (!y && m->impl->nRow > 0)) { set_error("multiply: NULL vector"); return B200SPMV_ERR_INVALID; }
    return B200SPMV_OK;
}

int b200spmv_multiply(b200spmv_matrix *m, const double *x_d, double *y_d, void *stream)
{
    B2_TRY(check_ready(m, x_d, y_d));
    return m->impl->multiply(x_d, y_d, (cudaStream_t)stream);
}

// y[0..nCol) := A^T x[0..nRow): A^T's matrix multiplies like any other (x and y swap their lengths)
static int check_transpose_ready(b200spmv_matrix *m, const void *x, const void *y, const char *who)
{
    clear_error();
    if (!m) { set_error("%s: NULL handle", who); return B200SPMV_ERR_INVALID; }
    if (!m->converted) { set_error("%s: matrix not converted yet", who); return B200SPMV_ERR_STATE; }
    if (!m->timpl) { set_error("%s: the handle was created with transpose = 0 (no A^T)", who); return B200SPMV_ERR_STATE; }
    if ((!x && m->timpl->nCol > 0) || (!y && m->timpl->nRow > 0)) { set_error("%s: NULL vector", who); return B200SPMV_ERR_INVALID; }
    return B200SPMV_OK;
}

int b200spmv_multiply_transpose(b200spmv_matrix *m, const double *x_d, double *y_d, void *stream)
{
    B2_TRY(check_transpose_ready(m, x_d, y_d, "multiply_transpose"));
    return m->timpl->multiply(x_d, y_d, (cudaStream_t)stream);
}

int b200spmv_multiply_transpose_f32(b200spmv_matrix *m, const float *x_d, float *y_d, void *stream)
{
    B2_TRY(check_transpose_ready(m, x_d, y_d, "multiply_transpose_f32"));
    return m->timpl->multiply_f32(x_d, y_d, (cudaStream_t)stream);
}

int b200spmv_multiply_multi(b200spmv_matrix *m, int k, const double *X_d, long long ldx, double *Y_d, long long ldy,
                            void *stream)
{
    clear_error();
    if (!m) { set_error("multiply_multi: NULL handle"); return B200SPMV_ERR_INVALID; }
    if (k < 1 || k > 8 || ldx < k || ldy < k) {
        set_error("multiply_multi: k=%d (1..8), ldx=%lld, ldy=%lld (>= k)", k, ldx, ldy);
        return B200SPMV_ERR_INVALID;
    }
    if (m->format != B200SPMV_CRS) { set_error("multiply_multi: CRS handles only (format %d)", m->format); return B200SPMV_ERR_UNSUPPORTED; }
    if (m->opt.value_f32) { set_error("multiply_multi: value_f32 handles are not supported"); return B200SPMV_ERR_UNSUPPORTED; }
    if (m->opt.precision) {
        set_error("multiply_multi: the handle was created with precision = %d (fp32 vectors)", m->opt.precision);
        return B200SPMV_ERR_STATE;
    }
    B2_TRY(check_ready(m, X_d, Y_d));
    return m->impl->multiply_multi(k, X_d, ldx, Y_d, ldy, (cudaStream_t)stream);
}

int b200spmv_multiply_multi_f32(b200spmv_matrix *m, int k, const float *X_d, long long ldx, float *Y_d, long long ldy,
                                void *stream)
{
    clear_error();
    if (!m) { set_error("multiply_multi_f32: NULL handle"); return B200SPMV_ERR_INVALID; }
    if (k < 1 || k > 8 || ldx < k || ldy < k) {
        set_error("multiply_multi_f32: k=%d (1..8), ldx=%lld, ldy=%lld (>= k)", k, ldx, ldy);
        return B200SPMV_ERR_INVALID;
    }
    if (m->format != B200SPMV_CRS) { set_error("multiply_multi_f32: CRS handles only (format %d)", m->format); return B200SPMV_ERR_UNSUPPORTED; }
    if (!m->opt.precision) {
        set_error("multiply_multi_f32: the handle was created with precision = 0 (fp64 vectors), use b200spmv_multiply_multi");
        return B200SPMV_ERR_STATE;
    }
    B2_TRY(check_ready(m, X_d, Y_d));
    return m->impl->multiply_multi_f32(k, X_d, ldx, Y_d, ldy, (cudaStream_t)stream);
}

int b200spmv_multiply_f32(b200spmv_matrix *m, const float *x_d, float *y_d, void *stream)
{
    B2_TRY(check_ready(m, x_d, y_d));
    return m->impl->multiply_f32(x_d, y_d, (cudaStream_t)stream);
}

int b200spmv_multiply_host_f32(b200spmv_matrix *m, const float *x_h, float *y_h)
{
    B2_TRY(check_ready(m, x_h, y_h));
    Format *f = m->impl.get();
    if (m->x_stage32.n != (size_t)f->nCol) B2_TRY(m->x_stage32.alloc((size_t)f->nCol));
    if (m->y_stage32.n != (size_t)f->nRow) B2_TRY(m->y_stage32.alloc((size_t)f->nRow));
    B2_CUDA(cudaMemcpyAsync(m->x_stage32.p, x_h, sizeof(float) * (size_t)f->nCol, cudaMemcpyHostToDevice, nullptr));
    B2_TRY(f->multiply_f32(m->x_stage32.p, m->y_stage32.p, nullptr));
    B2_CUDA(cudaMemcpyAsync(y_h, m->y_stage32.p, sizeof(float) * (size_t)f->nRow, cudaMemcpyDeviceToHost, nullptr));
    B2_CUDA(cudaStreamSynchronize(nullptr));
    return B200SPMV_OK;
}

int b200spmv_multiply_rows(b200spmv_matrix *m, int rowBegin, int rowEnd, const double *x_d, double *y_d,
                           void *stream)
{
    B2_TRY(check_ready(m, x_d, y_d));
    return m->impl->multiply_rows(rowBegin, rowEnd, x_d, y_d, (cudaStream_t)stream);
}

int b200spmv_prepare_rows(b200spmv_matrix *m, int rowBegin, int rowEnd)
{
    clear_error();
    if (!m) { set_error("prepare_rows: NULL handle"); return B200SPMV_ERR_INVALID; }
    if (!m->converted) { set_error("prepare_rows: matrix not converted yet"); return B200SPMV_ERR_STATE; }
    return m->impl->prepare_rows(rowBegin, rowEnd);
}

int b200spmv_rows_col_extent(b200spmv_matrix *m, int rowBegin, int rowEnd, int *colMin, int *colMax)
{
    clear_error();
    if (!m || !colMin || !colMax) { set_error("rows_col_extent: NULL argument"); return B200SPMV_ERR_INVALID; }
    if (!m->converted) { set_error("rows_col_extent: matrix not converted yet"); return B200SPMV_ERR_STATE; }
    return m->impl->col_extent(rowBegin, rowEnd, colMin, colMax);
}

// Page-locks a caller-owned host range so that copies to and from it are true asynchronous DMA (the reference's
// driver allocates x and y with _mm_malloc: pageable).  Already pinned memory is accepted as is.
int b200spmv_host_register(void *p, unsigned long long bytes)
{
    clear_error();
    if (!p || bytes == 0) { set_error("host_register: empty range"); return B200SPMV_ERR_INVALID; }
    B2_TRY(require_device());
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) == cudaSuccess && a.type == cudaMemoryTypeHost) return B200SPMV_OK;
    cudaGetLastError();
    cudaError_t e = cudaHostRegister(p, (size_t)bytes, cudaHostRegisterDefault);
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_error("host_register(%p, %llu bytes): %s", p, bytes, cudaGetErrorString(e));
        return B200SPMV_ERR_CUDA;
    }
    return B200SPMV_OK;
}

int b200spmv_host_unregister(void *p)
{
    clear_error();
    if (!p) return B200SPMV_OK;
    cudaError_t e = cudaHostUnregister(p);
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_error("host_unregister(%p): %s", p, cudaGetErrorString(e));
        return B200SPMV_ERR_CUDA;
    }
    return B200SPMV_OK;
}

static bool host_pinned(const void *p)
{
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

// builds (once per handle and shape) the plan of the host-semantics pipeline: row chunks, the x piece each needs
static int plan_host_pipeline(b200spmv_matrix *m, int nChunks, int nPieces)
{
    Format *f = m->impl.get();
    if (m->plan_chunks == nChunks && m->plan_pieces == nPieces) return B200SPMV_OK;
    const long long pieceLen = ((((long long)f->nCol + nPieces - 1) / nPieces) + 31) & ~31LL;     // 256-byte multiples
    for (int p = 0; p <= nPieces; p++) m->piece_c0[p] = std::min<long long>(f->nCol, pieceLen * p);
    for (int c = 0; c <= nChunks; c++)
        m->chunk_rb[c] = c == nChunks ? f->nRow : (int)((long long)f->nRow * c / nChunks) & ~31;
    for (int c = 0; c < nChunks; c++) {
        B2_TRY(f->prepare_rows(m->chunk_rb[c], m->chunk_rb[c + 1]));
        int cmin = 0, cmax = f->nCol - 1;
        if (nPieces > 1) B2_TRY(f->col_extent(m->chunk_rb[c], m->chunk_rb[c + 1], &cmin, &cmax));
        m->chunk_need[c] = cmax < 0 ? -1 : (int)std::min<long long>(nPieces - 1, cmax / std::max<long long>(pieceLen, 1));
    }
    m->plan_chunks = nChunks;
    m->plan_pieces = nPieces;
    return B200SPMV_OK;
}

int b200spmv_multiply_host(b200spmv_matrix *m, const double *x_h, double *y_h)
{
    B2_TRY(check_ready(m, x_h, y_h));
    Format *f = m->impl.get();
    if (!m->stream) {
        B2_CUDA(cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking));
        B2_CUDA(cudaStreamCreateWithFlags(&m->copy_stream, cudaStreamNonBlocking));
        B2_CUDA(cudaStreamCreateWithFlags(&m->in_stream, cudaStreamNonBlocking));
        for (auto &e : m->chunk_done) B2_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        for (auto &e : m->slice_in) B2_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    if (m->x_stage.n != (size_t)f->nCol) B2_TRY(m->x_stage.alloc((size_t)f->nCol));
    if (m->y_stage.n != (size_t)f->nRow) B2_TRY(m->y_stage.alloc((size_t)f->nRow));
    // The reference's cuSPARSE plugin serialises H2D x, multiply, D2H y (src/opt_cusparse.cpp:72-82).  Here the three
    // overlap where the format and the host memory allow it:
    //   * x goes up in pieces on its own stream (CSS: the column slices the format consumes one after the other;
    //     everything else: ascending pieces, and a row chunk starts as soon as the pieces up to its largest column
    //     have landed -- a banded matrix multiplies while most of x is still crossing PCIe),
    //   * rows are multiplied in chunks, and the D2H copy of a finished chunk of y runs under the next chunk's
    //     multiply on a third stream (PCIe is full duplex).
    // The pipeline needs true asynchronous copies: with pageable vectors every cudaMemcpyAsync is staged and the D2H
    // blocks the host, so the chunks would only add launches -> one H2D, one multiply, one D2H instead.
    const bool big = f->nRow >= (1 << 20) && f->has_rows() && host_pinned(x_h) && host_pinned(y_h);
    if (!big) {
        B2_CUDA(cudaMemcpyAsync(m->x_stage.p, x_h, sizeof(double) * (size_t)f->nCol, cudaMemcpyHostToDevice, m->stream));
        B2_TRY(f->multiply(m->x_stage.p, m->y_stage.p, m->stream));
        B2_CUDA(cudaMemcpyAsync(y_h, m->y_stage.p, sizeof(double) * (size_t)f->nRow, cudaMemcpyDeviceToHost, m->stream));
        B2_CUDA(cudaStreamSynchronize(m->stream));
        return B200SPMV_OK;
    }
    const bool sliced = f->n_x_slices() > 1 && f->n_x_slices() <= MAX_HOST_SLICES;   // CSS
    // chunks of at least 4 MB of y; measured on c2 (profiles/r1_experiments.md): CSS pays for every chunk with another
    // round of x-slice switches in L2 and is best with 2
    const int byBytes = (int)std::max<long long>(2, std::min<long long>(16, (long long)f->nRow * 8 / (4 << 20)));
    const int nChunks = std::min(sliced ? 2 : byBytes, MAX_HOST_CHUNKS);
    const int nPieces = sliced ? f->n_x_slices() : std::min(nChunks, MAX_HOST_SLICES);
    B2_TRY(plan_host_pipeline(m, nChunks, sliced ? 1 : nPieces));
    for (int i = 0; i < nPieces; i++) {
        long long c0 = m->piece_c0[i], c1 = m->piece_c0[i + 1];
        if (sliced) f->x_slice(i, &c0, &c1);
        if (c1 > c0)
            B2_CUDA(cudaMemcpyAsync(m->x_stage.p + c0, x_h + c0, sizeof(double) * (size_t)(c1 - c0), cudaMemcpyHostToDevice, m->in_stream));
        B2_CUDA(cudaEventRecord(m->slice_in[i], m->in_stream));
    }
    for (int c = 0; c < nChunks; c++) {
        const int rb = m->chunk_rb[c], re = m->chunk_rb[c + 1];
        if (!sliced) {
            if (m->chunk_need[c] >= 0) B2_CUDA(cudaStreamWaitEvent(m->stream, m->slice_in[m->chunk_need[c]], 0));
            B2_TRY(f->multiply_rows(rb, re, m->x_stage.p, m->y_stage.p, m->stream));
        } else {
            for (int i = 0; i < nPieces; i++) {
                if (c == 0) B2_CUDA(cudaStreamWaitEvent(m->stream, m->slice_in[i], 0));
                B2_TRY(f->multiply_rows_slice(i, rb, re, m->x_stage.p, m->y_stage.p, m->stream));
            }
        }
        B2_CUDA(cudaEventRecord(m->chunk_done[c], m->stream));
        B2_CUDA(cudaStreamWaitEvent(m->copy_stream, m->chunk_done[c], 0));
        if (re > rb)
            B2_CUDA(cudaMemcpyAsync(y_h + rb, m->y_stage.p + rb, sizeof(double) * (size_t)(re - rb), cudaMemcpyDeviceToHost, m->copy_stream));
    }
    B2_CUDA(cudaStreamSynchronize(m->copy_stream));
    B2_CUDA(cudaStreamSynchronize(m->stream));
    B2_CUDA(cudaStreamSynchronize(m->in_stream));
    return B200SPMV_OK;
}

int b200spmv_get_scalar(b200spmv_matrix *m, const char *name, long long *out)
{
    if (!m || !name || !out) { set_error("get_scalar: NULL argument"); return B200SPMV_ERR_INVALID; }
    if (!m->converted) { set_error("get_scalar: matrix not converted yet"); return B200SPMV_ERR_STATE; }
    std::string n(name);
    Format *f = m->impl.get();
    if (n == "transpose") { *out = m->timpl ? 1 : 0; return B200SPMV_OK; }
    if (n.compare(0, 2, "t.") == 0) {                           // t.<name>: the same scalar of A^T
        if (!m->timpl) { set_error("get_scalar: '%s' names A^T, and the handle was created with transpose = 0", name); return B200SPMV_ERR_STATE; }
        f = m->timpl.get();
        n.erase(0, 2);
    }
    if (n == "nRow") { *out = f->nRow; return B200SPMV_OK; }
    if (n == "nCol") { *out = f->nCol; return B200SPMV_OK; }
    if (n == "nNnz") { if (!f->scalar(n, out)) *out = f->nnz; return B200SPMV_OK; }
    if (n == "format") { *out = m->format; return B200SPMV_OK; }
    if (n == "has_rows") { *out = f->has_rows() ? 1 : 0; return B200SPMV_OK; }
    if (f->scalar(n, out)) return B200SPMV_OK;
    set_error("get_scalar: format %d has no scalar '%s'", m->format, name);
    return B200SPMV_ERR_INVALID;
}

long long b200spmv_get_array(b200spmv_matrix *m, const char *name, void *dst_h, long long dst_bytes)
{
    if (!m || !name) { set_error("get_array: NULL argument"); return B200SPMV_ERR_INVALID; }
    if (!m->converted) { set_error("get_array: matrix not converted yet"); return B200SPMV_ERR_STATE; }
    std::string n(name);
    Format *f = m->impl.get();
    if (n.compare(0, 2, "t.") == 0) {                           // t.<name>: the same array of A^T
        if (!m->timpl) { set_error("get_array: '%s' names A^T, and the handle was created with transpose = 0", name); return B200SPMV_ERR_STATE; }
        f = m->timpl.get();
        n.erase(0, 2);
    }
    long long r = f->array(n, dst_h, dst_bytes);
    if (r == -1000) {
        set_error("get_array: format %d has no array '%s'", m->format, name);
        return B200SPMV_ERR_INVALID;
    }
    return r;
}

int b200spmv_reference_vectors(unsigned seed, int nCol, int nRow, double *x_h, double *y_h)
{
    if (nCol > 0 && !x_h) { set_error("reference_vectors: NULL x"); return B200SPMV_ERR_INVALID; }
    srand(seed);                                                     // src/main.cpp:18
    for (int i = 0; i < nCol; i++) x_h[i] = double(rand()) / RAND_MAX;   // src/util.cpp:97-99
    if (y_h)
        for (int i = 0; i < nRow; i++) y_h[i] = double(rand()) / RAND_MAX;
    return B200SPMV_OK;
}

}  // extern "C"
