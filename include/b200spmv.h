/*
 * b200spmv.h -- C-ABI of the B200-native SpMV engine (libb200spmv.so).
 *
 * This is the drop-in boundary for the hot path of hir0shim/singleSpMV: the per-format
 * plugin pair
 *
 *     void OptimizeProblem(const SpMat &A, const Vec &x, SpMatOpt &A_opt, VecOpt &x_opt);
 *     extern "C" void SpMV(const SpMatOpt &A, const VecOpt &x, Vec &y);
 *
 * declared in /root/reference/src/opt_{crs,coo,ell,jds,dia,ss,css}.h (e.g. opt_crs.h:15-18)
 * and selected at compile time by /root/reference/src/opt.h:1-28 / opt.cpp:5-33.
 * A maintainer of the reference binds these entry points from a plugin file
 * (singlespmv_b200/plugin/opt_b200.{h,cpp}; INTEGRATION.md shows the stub).
 *
 * Conventions
 *   - plain C types only; `_h` = host pointer, `_d` = device pointer on the current device
 *   - indices are int32 and values fp64, like the reference (src/param.h:1-7, src/util.h:7-19)
 *   - input is COO sorted by (row, col) without duplicate coordinates (src/util.cpp:51)
 *   - every function returns 0 on success or a negative b200spmv_status; it never exits
 *     (the reference's plugins assert()/exit(): src/util.h:48-55, src/util.cpp:32-35)
 *   - a handle is used from one host thread at a time, and its multiplies are serialised on ONE stream at a time:
 *     rows that cross tile boundaries are finished through per-handle carry buffers, so two multiplies of the same
 *     handle in flight on different streams would race (b200spmv_multiply_host uses its own private streams: do not
 *     overlap it with b200spmv_multiply on the same handle)
 *   - there is NO CPU fallback: without a CUDA device every compute entry fails with
 *     B200SPMV_ERR_CUDA.
 *   - signed zeros, infinities and NaN (stored-entry semantics; every format and path but DIA and ss_faithful SS / CSS):
 *     y[i] depends only on the stored entries of row i and on x at their columns.  With p = a * x[c] the exact products
 *     of those entries, y[i] is NaN if any p is NaN (a NaN in x or A, a stored 0 times +-Inf) or if the row has both
 *     +Inf and -Inf products; else +-Inf if it has infinite products of one sign; else finite.  This holds whatever
 *     order a kernel sums in, as long as the finite part of the row cannot overflow.  A row whose products are all +-0
 *     (an empty row too) is +0.0.  No kernel reads x for a slot that holds no entry (padding, ragged tile ends).
 *   - DIA and SS / CSS with ss_faithful = 1 have the reference's padding semantics instead: they run the reference's own
 *     operations, 0 * x over its padding included (DIA cannot tell padding from stored zeros), and give its bits.
 *   - results claimed bit-identical to the reference are so on the bits, NaN aside: a NaN's payload is unspecified.
 */
#ifndef B200SPMV_H
#define B200SPMV_H

#ifdef __cplusplus
extern "C" {
#endif

#define B200SPMV_VERSION 100
#if defined(__GNUC__)
#define B200SPMV_API __attribute__((visibility("default")))
#else
#define B200SPMV_API
#endif

typedef struct b200spmv_matrix b200spmv_matrix;      /* opaque converted matrix (SpMatOpt) */

/* Storage formats = the reference's plugins (src/opt.h:1-28) + the vendored CSR5
 * (opt/Benchmark_SpMV_using_CSR5/CSR5_cuda/anonymouslib_cuda.h). */
typedef enum {
    B200SPMV_CRS  = 0,   /* src/opt_crs.cpp  */
    B200SPMV_COO  = 1,   /* src/opt_coo.cpp  */
    B200SPMV_ELL  = 2,   /* src/opt_ell.cpp  (device layout: sliced ELL) */
    B200SPMV_JDS  = 3,   /* src/opt_jds.cpp  */
    B200SPMV_DIA  = 4,   /* src/opt_dia.cpp  */
    B200SPMV_SS   = 5,   /* src/opt_ss.cpp   */
    B200SPMV_CSS  = 6,   /* src/opt_css.cpp  */
    B200SPMV_CSR5 = 7,   /* opt/.../CSR5_cuda */
    B200SPMV_HYB  = 8    /* ELL + COO tail: named, never implemented upstream (CSR5_cuda/detail/common.h:22) */
} b200spmv_format;

typedef enum {
    B200SPMV_OK              =  0,
    B200SPMV_ERR_INVALID     = -1,   /* bad argument / input breaks the contract above   */
    B200SPMV_ERR_CUDA        = -2,   /* CUDA runtime error (see b200spmv_last_error)      */
    B200SPMV_ERR_UNSUPPORTED = -3,   /* format/option combination not available           */
    B200SPMV_ERR_STATE       = -4,   /* call order (multiply before convert, ...)         */
    B200SPMV_ERR_NOMEM       = -5
} b200spmv_status;

/* Tunables.  The reference fixes these at compile time with -D macros
 * (Makefile:10-21, src/param.h:9-20); here they are per-handle.  Zero = default. */
typedef struct {
    int segment_width;   /* SS/CSS: SEGMENT_WIDTH (W), power of two; default 4 (= ALIGNMENT/8, ALIGNMENT=32) */
    int n_block;         /* CSS: N_BLOCK; default 1 */
    int csr5_sigma;      /* CSR5: sigma 1..32; -1 = upstream's auto rule (anonymouslib_cuda.h:293-317);
                            0 = the same rule with a floor of 16 (tuned on B200) */
    int ss_faithful;     /* SS/CSS: 1 = three-phase Mul/fold/gather with val_buf, the reference's
                            operation order (src/opt_ss.cpp:222-303); 0 = fused one-pass kernel */
    int value_f32;       /* CRS: 1 = store the matrix values as fp32 (rounded once at conversion); x, y and all
                            arithmetic stay fp64.  8 instead of 12 B/nnz; tolerance 1e-5 (BASELINE.json north star) */
    int crs_path;        /* CRS / SS: 0 = choose from the matrix (longest row <= 16 and banded: TMA-fed row-chunk stream; CRS on matrices
                            whose gathers range over > 32 MB of x: the entry stream, sums re-associated within 1e-12; else the
                            tile-stream), 1 = always the tile-stream kernel (rows of up to 64 entries summed in the reference's
                            order); 3 = the TMA-fed row-chunk stream wherever it applies; CRS: 4 = always the entry stream.
                            2 (round 1's row-block stream) was removed and is rejected, like any value outside 0..4 */
    int profile;         /* SS/CSS with ss_faithful: time the Mul and the Sum phase of every multiply with CUDA events
                            (the reference's -DPROFILING, src/util.h:59-65); the multiply then synchronises and the
                            scalars MulTime_ns / SumTime_ns hold the last call's phases */
    int col_blocks;      /* ELL / JDS / SS: column-blocked device layout (csrc/colblocks.cuh) for matrices whose
                            gathers do not fit L2.  0 = decide from the matrix (x > 64 MB and rows spread over the column
                            blocks), n > 0 = force n column blocks, -1 = never.  The reference arrays (exports) and y
                            are the same either way: every row is still summed in ascending column order (rows of more
                            than 64 entries per block: within the 1e-12 tolerance) */
    int precision;       /* CRS / ELL / DIA / CSR5: 0 = fp64 (the reference); 1 = fp32: matrix values rounded once to fp32 at conversion,
                            x and y are float arrays, products and sums in fp32; 2 = the same storage and vectors with
                            fp64 products and sums.  Multiply with b200spmv_multiply_f32 / _host_f32; tolerance 1e-5
                            against the reference's (fp64) CRS result.  Halves the bytes of every array but the indices */
    int hyb_k;           /* HYB: width K of the ELL part (the first K entries of every row; the rest form the COO tail).
                            0 = the largest width k <= 4096 that at least min(nRow, max(4096, nRow/3)) rows fill (rows
                            longer than 4096 count as 4096 long, so K never exceeds 4096); K = 1 when no width qualifies,
                            0 for a matrix without entries.  n > 0 = min(n, longest row).  Negative values are rejected */
    int coo_path;        /* COO: 0 = entry stream (segmented warp scans; sums re-associated within 1e-12), fed by TMA bulk copies or
                            by the lanes' own loads, whichever suits the matrix; 1 = the order-preserving tile kernel (rows <= 64
                            entries bit-identical to the CRS result); 2 / 3 = force the load-fed / the TMA-fed entry stream;
                            other values are rejected */
    int transpose;       /* 1 = also build A^T at conversion, for b200spmv_multiply_transpose{,_f32}: A's COO transposed on the
                            device (a stable, deterministic sort on the column: the host's lexsort of (col, row)), then
                            converted like A -- the same format and options, row blocks above 2^31-1 entries -- into a
                            second matrix the handle holds.  Conversion time and device memory grow by about A's; the
                            transposed COO and its sort scratch are freed before the conversion returns.  A JDS permutation
                            (b200spmv_jds_set_perm_host) applies to A only: A^T orders ties by ascending row.  If A^T cannot
                            be built (e.g. B200SPMV_ERR_NOMEM: an ELL of A^T pads to A's longest column), the conversion
                            fails and the handle stays unconverted.  0 = no A^T (default); other values are rejected.
                            Not accepted by b200spmv_mg_create */
    int reserved[4];
} b200spmv_options;

/* ---- library ---- */
B200SPMV_API int b200spmv_version(void);
/* Message of the last failing call on this thread ("" if none). */
B200SPMV_API const char *b200spmv_last_error(void);
B200SPMV_API int b200spmv_device_count(int *count);

/* ---- lifetime (the reference never frees: src/util.h:12-18) ---- */
B200SPMV_API int b200spmv_create(int format, const b200spmv_options *opts /* may be NULL */, b200spmv_matrix **out);
B200SPMV_API int b200spmv_destroy(b200spmv_matrix *m);

/* ---- conversion: replaces OptimizeProblem (src/opt_crs.cpp:10, opt_ell.cpp:7, opt_jds.cpp:8,
 * opt_dia.cpp:6, opt_ss.cpp:14, opt_css.cpp:17, opt_coo.cpp:3).  All format arrays are built on
 * the device from the COO triplets.  _host copies the triplets H2D first. */
B200SPMV_API int b200spmv_convert_coo_host(b200spmv_matrix *m, int nRow, int nCol, long long nnz,
                              const int *row_h, const int *col_h, const double *val_h);
B200SPMV_API int b200spmv_convert_coo_device(b200spmv_matrix *m, int nRow, int nCol, long long nnz,
                                const int *row_d, const int *col_d, const double *val_d,
                                void *stream /* cudaStream_t */);
/* JDS only, optional, before convert: impose the row permutation (e.g. the one libstdc++'s
 * unstable std::sort produced for the reference, src/opt_jds.cpp:41-46).  It must order rows
 * by non-increasing length.  Without it ties are ordered by ascending row. */
B200SPMV_API int b200spmv_jds_set_perm_host(b200spmv_matrix *m, const int *perm_h, int nRow);

/* ---- multiply: replaces SpMV (src/opt_crs.cpp:45 etc.).  y := A*x, every y[0..nRow) is
 * overwritten (beta = 0); the call may be repeated any number of times (src/main.cpp:41-88). */
B200SPMV_API int b200spmv_multiply(b200spmv_matrix *m, const double *x_d, double *y_d, void *stream);
/* Y[:, 0..k) := A * X[:, 0..k) for k = 1..8 vectors; row-major: X[c*ldx + j], Y[r*ldy + j]; ldx, ldy >= k (in doubles).
 * CRS handles with precision = 0 and value_f32 = 0.  Columns k..ld-1 of X are never read into a result; those of Y are
 * never written.  beta = 0 for every Y[r, j], j < k.  Same one-stream-at-a-time rule per handle as b200spmv_multiply.
 * The matrix is streamed once for all k vectors, and one gather fetches the k values of a column from one row of X.
 * The kernel follows the one conversion chose (scalar multi_kernel: 1 row-chunk stream, 2 / 3 entry stream TMA- / load-fed):
 *   - row-chunk stream and entry stream handles: column j of Y has the bits of b200spmv_multiply on column j of X;
 *   - tile-stream handles (rows longer than 16 that are not gather-bound, e.g. 27-point stencils, and crs_path = 1) run
 *     the entry stream, whose metadata the first call builds (it synchronises): rows of up to 64 entries are then summed
 *     in another association than b200spmv_multiply sums them, within the entry stream's 1e-12 tolerance.
 * The first call on an entry-stream or tile-stream handle allocates per-handle buffers: made inside a stream capture it is
 * refused with B200SPMV_ERR_STATE; later calls can be captured.  Errors: B200SPMV_ERR_INVALID (NULL handle or vector,
 * k outside 1..8, ldx or ldy < k), B200SPMV_ERR_UNSUPPORTED (formats other than CRS, value_f32), B200SPMV_ERR_STATE
 * (before convert, precision 1 / 2, first call inside a capture). */
B200SPMV_API int b200spmv_multiply_multi(b200spmv_matrix *m, int k, const double *X_d, long long ldx,
                                         double *Y_d, long long ldy, void *stream);
/* y[0..nCol) := A^T x[0..nRow) for handles created with options.transpose = 1; every y entry is overwritten (beta = 0).
 * A^T is a matrix of the handle's own format converted from A's transposed COO, so these calls run that format's kernels
 * on it and have the bits of b200spmv_multiply / b200spmv_multiply_f32 on a handle of the same format and options
 * converted from the transposed triplets (nCol x nRow, sorted by (col, row)).  The scalars and arrays of A^T are read
 * with the prefix "t." (t.nRow, t.crs_kernel, t.alg_bytes, t.ptr, ...; B200SPMV_ERR_STATE without A^T); the scalar
 * "transpose" is 1 when A^T was built.  A^T has carry buffers of its own, but the one-stream-at-a-time rule covers the
 * handle in both directions: do not overlap b200spmv_multiply and b200spmv_multiply_transpose on different streams.
 * Errors, decided before any CUDA call and in this order: B200SPMV_ERR_INVALID (NULL handle), B200SPMV_ERR_STATE (before
 * convert; handle created with transpose = 0), B200SPMV_ERR_INVALID (NULL x with nRow > 0, NULL y with nCol > 0), then
 * the precision checks of b200spmv_multiply / _f32 (B200SPMV_ERR_STATE). */
B200SPMV_API int b200spmv_multiply_transpose(b200spmv_matrix *m, const double *x_d, double *y_d, void *stream);
B200SPMV_API int b200spmv_multiply_transpose_f32(b200spmv_matrix *m, const float *x_d, float *y_d, void *stream);
/* Host semantics (what SpMV(A_opt, x_opt, y) means to the reference's driver): copies x H2D,
 * multiplies, copies y D2H, synchronises -- like src/opt_cusparse.cpp:72-82. */
B200SPMV_API int b200spmv_multiply_host(b200spmv_matrix *m, const double *x_h, double *y_h);
/* fp32 variant (options.precision = 1 or 2; src/param.h has no value-type switch, the CSR5 benchmark the reference
 * vendors does: CSR5_cuda/Makefile:4 VALUE_TYPE).  The handle must have been created with that precision. */
B200SPMV_API int b200spmv_multiply_f32(b200spmv_matrix *m, const float *x_d, float *y_d, void *stream);
B200SPMV_API int b200spmv_multiply_host_f32(b200spmv_matrix *m, const float *x_h, float *y_h);
/* Y[:, 0..k) := A * X[:, 0..k) for k = 1..8 fp32 vectors: b200spmv_multiply_multi for CRS handles created with precision
 * = 1 or 2 (X[c*ldx + j], Y[r*ldy + j]; ldx, ldy >= k, in floats; the same rules for columns >= k, beta = 0 and streams).
 * The matrix (4 B values) is streamed once, and one row of X -- up to 8 columns in one 32-byte sector -- is gathered once
 * per entry; for one contiguous vector b200spmv_multiply_f32 is faster.  The kernel (scalar multi_kernel_f32: 1 row-chunk
 * stream, 2 / 3 entry stream TMA- / load-fed, 0 on precision-0 handles and on matrices without entries):
 *   - row-chunk stream handles: column j of Y has the bits of b200spmv_multiply_f32 on column j of X (one thread per row,
 *     ascending column order, unfused mul / add in fp32 (precision 1) or fp64 (precision 2), rounded to fp32 once);
 *   - every other handle (b200spmv_multiply_f32 runs the tile-stream there) runs the entry stream, whose metadata the first
 *     call builds (it synchronises).  Sums are re-associated: precision 1 within (n+1) 2^-24 sum|a x| of the exact row sum,
 *     precision 2 (fp64 products and sums, carried in fp64 across tiles, rounded to fp32 once) within 2^-24 |s| +
 *     n 2^-53 sum|a x|.
 * The first call on an entry-stream handle allocates per-handle buffers: made inside a stream capture it is refused with
 * B200SPMV_ERR_STATE; later calls can be captured.  Errors, decided before any CUDA call and in this order:
 * B200SPMV_ERR_INVALID (NULL handle, k outside 1..8, ldx or ldy < k), B200SPMV_ERR_UNSUPPORTED (formats other than CRS),
 * B200SPMV_ERR_STATE (precision = 0, value_f32 handles included: use b200spmv_multiply_multi; before convert),
 * B200SPMV_ERR_INVALID (NULL X or Y with nCol or nRow > 0). */
B200SPMV_API int b200spmv_multiply_multi_f32(b200spmv_matrix *m, int k, const float *X_d, long long ldx,
                                             float *Y_d, long long ldy, void *stream);
/* Rows [rowBegin,rowEnd) only (CRS, SS, CSS, ELL, DIA; others return B200SPMV_ERR_UNSUPPORTED): used by
 * the row-partitioned multi-GPU path to overlap the interior block with the halo exchange, and by
 * b200spmv_multiply_host to overlap the D2H copy of finished rows with the rest of the multiply. */
B200SPMV_API int b200spmv_multiply_rows(b200spmv_matrix *m, int rowBegin, int rowEnd, const double *x_d,
                           double *y_d, void *stream);

/* Host-side bookkeeping for a row range (reads two row pointers back: synchronises).  multiply_rows on a prepared
 * range never synchronises and can be captured in a CUDA graph; an unprepared range is prepared on first use
 * (refused with B200SPMV_ERR_STATE inside a stream capture). */
B200SPMV_API int b200spmv_prepare_rows(b200spmv_matrix *m, int rowBegin, int rowEnd);
/* Smallest and largest column referenced by rows [rowBegin,rowEnd) (conservative: CRS, SS, ELL, DIA look at their
 * arrays, the other formats answer [0, nCol-1]; colMax < colMin = the rows are empty).  Lets a caller that streams x
 * in from the host (or from a peer GPU) start a row range as soon as that part of x is there. */
B200SPMV_API int b200spmv_rows_col_extent(b200spmv_matrix *m, int rowBegin, int rowEnd, int *colMin, int *colMax);
/* Page-lock / release a caller-owned host vector.  b200spmv_multiply_host overlaps H2D x, the multiply and D2H y
 * only when BOTH vectors are page-locked; with pageable vectors (the reference's _mm_malloc'ed x and y,
 * src/util.cpp:92-102) it falls back to copy - multiply - copy.  The plugin layer registers x in OptimizeProblem
 * and y on the first SpMV; the caller must keep a registered range alive until it is unregistered. */
B200SPMV_API int b200spmv_host_register(void *p, unsigned long long bytes);
B200SPMV_API int b200spmv_host_unregister(void *p);

/* ---- read-back for parity checks: the SpMatOpt fields under the reference's names.
 * Scalars: nRow nCol nNnz | K | maxLength | nDiag | H nStep W | B nBlock totalH | sigma p ... and
 *          alg_bytes (compulsory bytes per multiply, SURVEY.md 8d), launches (kernels/multiply).
 * Arrays are returned in the reference's LOGICAL layout (ELL [nRow][K], DIA [nDiag][nCol], ...).
 * get_array: dst_h == NULL returns the size in bytes; otherwise copies and returns the size;
 * negative = error. */
B200SPMV_API int b200spmv_get_scalar(b200spmv_matrix *m, const char *name, long long *out);
B200SPMV_API long long b200spmv_get_array(b200spmv_matrix *m, const char *name, void *dst_h, long long dst_bytes);

/* ---- synthetic inputs on the device (SURVEY.md 8d; same definitions as oracle/synth_oracle.c).
 * The reference loads Matrix-Market text (src/util.cpp:30-66); BASELINE.json's shapes are up to
 * 938 M non-zeros, so they are generated in HBM instead. */
typedef enum {
    B200SPMV_SYNTH_LAP2D5  = 0,  /* p0 = n        : 2-D 5-point Laplacian, n*n rows          */
    B200SPMV_SYNTH_LAP3D7  = 1,  /* p0 = n        : 3-D 7-point Laplacian, n^3 rows          */
    B200SPMV_SYNTH_BOX3D27 = 2,  /* p0 = n        : 3-D 27-point stencil,  n^3 rows          */
    B200SPMV_SYNTH_UNIFORM = 3,  /* p0 = nRow=nCol, p1 = K distinct uniform columns per row  */
    B200SPMV_SYNTH_RMAT    = 4   /* p0 = scale, p1 = edge draws; duplicates removed          */
} b200spmv_synth_kind;

typedef struct {
    int nRow, nCol;          /* GLOBAL dimensions                                             */
    int rowBegin, rowEnd;    /* rows actually generated (row ids in row_d stay global)        */
    long long nnz;           /* entries in the arrays                                         */
    int *row_d, *col_d;
    double *val_d;
} b200spmv_coo;

/* Generates rows [rowBegin,rowEnd) (rowEnd <= 0: all rows) of the named matrix into newly
 * allocated device arrays.  RMAT supports the full range only. */
B200SPMV_API int b200spmv_synth(int kind, long long p0, long long p1, unsigned long long seed,
                   int rowBegin, int rowEnd, b200spmv_coo *out, void *stream);
B200SPMV_API int b200spmv_coo_free(b200spmv_coo *coo);
/* Uploads entries of rows [rowBegin,rowEnd) of a sorted host COO (row ids stay global): the block a rank of the
 * row-partitioned multiply owns when the matrix comes from a file instead of a generator. */
B200SPMV_API int b200spmv_coo_upload(int nRow, int nCol, int rowBegin, int rowEnd, long long nnz, const int *row_h,
                        const int *col_h, const double *val_h, b200spmv_coo *out);
/* Copies the triplets to host arrays of coo->nnz entries (parity checks, CPU baseline input). */
B200SPMV_API int b200spmv_coo_download(const b200spmv_coo *coo, int *row_h, int *col_h, double *val_h);

/* ---- row-partitioned multi-GPU multiply (SURVEY.md 8e).  The reference is single-node OpenMP
 * (its only "distribution" is the static row schedule of src/opt_crs.cpp:57-58); this is the
 * B200 design for BASELINE.json config 5: contiguous row blocks balanced by non-zero count, x
 * distributed like the rows, per multiply only the referenced remote x entries ("halo") move.
 * One process per GPU; the host side (singlespmv_b200/dist.py) carries the exchange over
 * NCCL/NVLink and overlaps it with the interior rows via b200spmv_multiply_rows. */
/* bounds_h[0..nParts]: block g owns rows [bounds[g], bounds[g+1]), split where the running
 * non-zero count passes g*nnz/nParts. */
B200SPMV_API int b200spmv_partition_rows(const int *row_d /* sorted COO row ids */, long long nnz, int nRow,
                            int nParts, int *bounds_h);
/* the same split for a synthetic matrix, from its row lengths alone (nothing is generated) */
B200SPMV_API int b200spmv_partition_synth(int kind, long long p0, long long p1, int nParts, int *bounds_h);

/* ---- the same multiply with ONE process driving all GPUs (csrc/mg.cu): what the C++ plugin uses with -DB200_NGPU=N so
 * that the reference's driver loop (src/main.cpp:58-102) runs over 8 B200s like over one.  Partition and halo
 * renumbering as above; the halo is PULLED by a kernel out of the owners' x slices through NVLink peer mappings, overlapped
 * with the interior rows, and the whole step of all GPUs is one multi-device CUDA graph launch.  Square matrices. */
typedef struct b200spmv_mg b200spmv_mg;
B200SPMV_API int b200spmv_mg_create(int nGPU, int format, const b200spmv_options *opts /* may be NULL */, b200spmv_mg **out);
B200SPMV_API int b200spmv_mg_destroy(b200spmv_mg *m);
/* any sorted COO on the host (e.g. what src/util.cpp:30-66 loads): split by non-zero balance, one block per GPU */
B200SPMV_API int b200spmv_mg_convert_coo_host(b200spmv_mg *m, int nRow, int nCol, long long nnz, const int *row_h,
                                 const int *col_h, const double *val_h);
/* synthetic matrix (b200spmv_synth kinds except RMAT): every GPU generates its own rows in its own HBM */
B200SPMV_API int b200spmv_mg_convert_synth(b200spmv_mg *m, int kind, long long p0, long long p1, unsigned long long seed);
/* host semantics, = SpMV(A_opt, x_opt, y): scatter x to the GPUs, exchange + multiply, gather y, synchronise */
B200SPMV_API int b200spmv_mg_multiply_host(b200spmv_mg *m, const double *x_h, double *y_h);
/* device-resident vectors: upload x once, then each mg_multiply is exchange + multiply only (asynchronous) */
B200SPMV_API int b200spmv_mg_upload_x(b200spmv_mg *m, const double *x_h);
B200SPMV_API int b200spmv_mg_multiply(b200spmv_mg *m);
B200SPMV_API int b200spmv_mg_synchronize(b200spmv_mg *m);
B200SPMV_API int b200spmv_mg_download_y(b200spmv_mg *m, double *y_h);
/* nGPU nRow nCol nNnz | halo_total (x entries crossing NVLink per multiply) | graphed | alg_bytes | launches */
B200SPMV_API int b200spmv_mg_get_scalar(b200spmv_mg *m, const char *name, long long *out);
B200SPMV_API int b200spmv_mg_get_bounds(b200spmv_mg *m, int *bounds_h /* nGPU + 1 */);

typedef struct b200spmv_halo b200spmv_halo;
/* coo holds rows [rowBegin,rowEnd) with GLOBAL ids; the block owns x[colBegin,colEnd).  In place:
 * rows become block-local and columns get the monotone local numbering
 *   [left halo | owned slice | right halo]   (halo = referenced remote columns, ascending),
 * so rows stay sorted and are summed in the single-GPU order.  coo->nRow/nCol become the local
 * dimensions; convert it with any format afterwards. */
B200SPMV_API int b200spmv_halo_plan(b200spmv_coo *coo, int colBegin, int colEnd, b200spmv_halo **out, void *stream);
/* info8 = nLocal, nLeft, nRight, interiorBegin, interiorEnd, nSend, rowBegin, rowEnd.  Local rows
 * [interiorBegin, interiorEnd) reference owned columns only. */
B200SPMV_API int b200spmv_halo_info(const b200spmv_halo *h, long long *info8);
/* the halo's global column ids (get_array size protocol) -- what this block asks its peers for */
B200SPMV_API long long b200spmv_halo_cols(const b200spmv_halo *h, int *cols_h, long long cap_bytes);
/* global ids of OWNED columns the peers asked for, concatenated in peer order */
B200SPMV_API int b200spmv_halo_set_send(b200spmv_halo *h, const int *send_cols_h, long long n);
/* sendbuf[i] = x_owned[send column i]: one gather kernel per multiply */
B200SPMV_API int b200spmv_halo_pack(const b200spmv_halo *h, const double *x_owned_d, double *sendbuf_d, void *stream);
B200SPMV_API int b200spmv_halo_free(b200spmv_halo *h);

/* ---- x windows: the halo exchange of the one-process-per-GPU path as ONE kernel over NVLink peer memory
 * (csrc/xwin.cu; host side singlespmv_b200/dist.py).  Every rank keeps x_ext = [left halo | owned | right halo] in a
 * cudaMalloc'ed window that the other processes of the node map through CUDA IPC; per step one kernel signals "my
 * slice is in place" into the readers' windows, waits for the owners' signals, pulls exactly its halo entries out of the
 * owners' slices and acknowledges -- no pack kernel, no staging buffer, no NCCL kernels.  When the step's kernel has
 * finished, every reader has finished pulling: the owned slice may be overwritten. */
typedef struct b200spmv_xwin b200spmv_xwin;
/* nExt doubles of x_ext on the current device, the owned slice starts at ownedOff (= nLeft) */
B200SPMV_API int b200spmv_xwin_create(int rank, int world, long long nExt, long long ownedOff, b200spmv_xwin **out);
B200SPMV_API void *b200spmv_xwin_x_ext(b200spmv_xwin *w);               /* device pointer of x_ext */
/* 80-byte blob (cudaIpcMemHandle_t + layout) to hand to the other ranks, and its counterpart */
B200SPMV_API int b200spmv_xwin_export(b200spmv_xwin *w, void *blob80);
B200SPMV_API int b200spmv_xwin_import(b200spmv_xwin *w, int peer, const void *blob80);
/* same-process twin of export + import (several blocks driven by one process) */
B200SPMV_API int b200spmv_xwin_attach(b200spmv_xwin *w, int peer, b200spmv_xwin *other);
/* halo_cols_h: b200spmv_halo_cols (global ids, ascending); bounds_h[world+1]: the column split; readers_h: ranks that
 * asked this one for columns */
B200SPMV_API int b200spmv_xwin_plan(b200spmv_xwin *w, const int *halo_cols_h, int nHalo, int nLeft, int nLocal,
                       const long long *bounds_h, const int *readers_h, int nReaders);
/* one step's exchange, asynchronous on `stream` (may be captured in a CUDA graph); every rank calls it once per step */
B200SPMV_API int b200spmv_xwin_exchange(b200spmv_xwin *w, void *stream);
/* steps finished; *timed_out != 0 if a flag wait ever gave up after ~10 s (a peer that did not take part) */
B200SPMV_API int b200spmv_xwin_status(b200spmv_xwin *w, long long *steps, int *timed_out);
B200SPMV_API int b200spmv_xwin_free(b200spmv_xwin *w);

/* ---- Matrix-Market ingest into a device COO (SURVEY.md 8f).  The reference's loader (src/util.cpp:30-66)
 * ignores the banner and keeps duplicates; the CSR5 benchmark it vendors reads the same files through mmio and
 * honours symmetric / pattern banners (opt/Benchmark_SpMV_using_CSR5/CSR5_avx2/main.cpp:145-282). */
typedef enum {
    B200SPMV_MTX_BANNER    = 0,  /* real|integer|pattern x general|symmetric|skew-symmetric; mirrored entries added,
                                    duplicate coordinates summed: the result satisfies the plugins' input contract */
    B200SPMV_MTX_REFERENCE = 1   /* src/util.cpp:30-66 bit for bit: banner ignored, exactly L triples, duplicates kept */
} b200spmv_mtx_mode;
/* Parses on the host, sorts by (row, col) (and reduces duplicates) on the device.  Free with b200spmv_coo_free. */
B200SPMV_API int b200spmv_load_mtx(const char *path, int mode, b200spmv_coo *out, void *stream);

/* ---- matrix statistics and format recommendation (SURVEY.md 8f).  The statistics are those the reference's
 * tooling prints (matrix/script/counter.cpp:19-42: max/min non-zeros per row and per column, variance of the
 * row counts) plus empty rows and the number of non-empty diagonals (src/opt_dia.cpp:29-34). */
typedef struct {
    int nRow, nCol;
    long long nnz;
    int rowMax, rowMin, colMax, colMin;
    double rowMean, rowVar;          /* rowVar = sum (cnt - mean)^2 / nRow, as counter.cpp:31-34 */
    long long nEmptyRows, nDiag;
} b200spmv_stats;
B200SPMV_API int b200spmv_analyze(const b200spmv_coo *coo /* whole matrix */, b200spmv_stats *out, void *stream);
/* Returns a b200spmv_format; opts_out (may be NULL) receives the tunables that go with it (CSS: n_block).
 * Rules and the measurements behind them: singlespmv_b200/csrc/analyze.cu, profiles/. */
B200SPMV_API int b200spmv_recommend_format(const b200spmv_stats *stats, b200spmv_options *opts_out);

/* x = rand()/RAND_MAX stream of src/util.cpp:92-102 after srand(seed) (src/main.cpp:18):
 * writes x_h[0..nCol) (and y_h[0..nRow) if y_h != NULL), host side, glibc rand(). */
B200SPMV_API int b200spmv_reference_vectors(unsigned seed, int nCol, int nRow, double *x_h, double *y_h);

#ifdef __cplusplus
}
#endif
#endif /* B200SPMV_H */
