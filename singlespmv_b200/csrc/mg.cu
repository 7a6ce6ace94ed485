// mg.cu -- row-partitioned multi-GPU multiply behind the C-ABI, ONE process driving all GPUs of the box
// (SURVEY.md 8e / 8b: b200spmv_mg_*).  The reference is single-node OpenMP; its driver loop (src/main.cpp:58-102) calls
// one SpMV per iteration -- here that one call fans out over the GPUs, so the C++ plugin (plugin/opt_b200.cpp with
// -DB200_NGPU=N) drives 8 B200s exactly like it drives one.
//
//   partition   contiguous row blocks where the running non-zero count passes g nnz / G (any sorted COO, host or
//               synthetic); x is distributed like the rows (square matrices)
//   per GPU     b200spmv_halo_plan: columns renumbered [left halo | owned | right halo] monotonically (rows stay
//               sorted -> same summation order as on one GPU -> bit-identical y), then any format's conversion
//   exchange    PULL over NVLink peer memory: every GPU has every other GPU's x slice mapped (cudaDeviceEnablePeerAccess)
//               and one small kernel gathers exactly the halo entries it needs straight out of the owners' slices --
//               no pack kernel, no send/recv pairs, no staging buffer.  A halo that covers most of x (R-MAT) is the
//               same kernel reading the peers' slices almost contiguously: the all-gather case needs no second path.
//   overlap     the pull runs on a communication stream while the interior rows (those that touch owned columns only)
//               run on the compute stream; the boundary rows follow once the halo has landed
//   launch      the whole step of all GPUs is captured once into ONE multi-device CUDA graph (fork / join through
//               events): a step is a single cudaGraphLaunch from the single host thread
// The multi-process twin of this file is singlespmv_b200/dist.py (torchrun, one process per GPU, NCCL send/recv).
#include <algorithm>
#include <chrono>
#include <cstdlib>

#include "common.cuh"

using namespace b2;

namespace {

// x_ext halo slot i <- the owner's x slice: slots [0, nLeft) sit below the owned slice, the rest above it.
// CTAs of 64 threads in a grid-stride loop with four loads in flight: the interior rows run as persistent CTAs that leave ~4096
// registers per SM, so only small CTAs get an SM while they run (measured on the torchrun twin of this kernel, xwin.cu: 256-thread
// CTAs only started once the interior rows had drained)
constexpr int MG_PULL_THREADS = 64;
__global__ void __launch_bounds__(MG_PULL_THREADS)
mg_pull_kernel(const double *const *__restrict__ peer_x, const int *__restrict__ owner, const int *__restrict__ idx, int nHalo,
               int nLeft, int nLocal, double *__restrict__ x_ext)
{
    const int stride = gridDim.x * MG_PULL_THREADS;
    for (int i0 = blockIdx.x * MG_PULL_THREADS + threadIdx.x; i0 < nHalo; i0 += 4 * stride) {
        double v[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int i = i0 + u * stride;
            if (i < nHalo) v[u] = peer_x[owner[i]][idx[i]];        // NVLink peer load (or a local load when owner == self)
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int i = i0 + u * stride;
            if (i < nHalo) x_ext[i < nLeft ? i : nLocal + i] = v[u];
        }
    }
}

struct MgBlock {
    int dev = 0, rowBegin = 0, rowEnd = 0;
    int nLocal = 0, nLeft = 0, nRight = 0, interiorBegin = 0, interiorEnd = 0;
    long long nnz = 0;
    b200spmv_halo *halo = nullptr;
    b200spmv_matrix *A = nullptr;
    double *x_ext = nullptr, *y = nullptr;
    int *pull_owner = nullptr, *pull_idx = nullptr;
    const double **peer_x = nullptr;
    cudaStream_t compute = nullptr, comm = nullptr;
    cudaEvent_t ev_x = nullptr, ev_halo = nullptr, ev_done = nullptr;            // eager steps: cross-stream / cross-step ordering
    cudaEvent_t cev_halo = nullptr, cev_join = nullptr;                          // recorded only inside the graph capture
    double *x_owned() const { return x_ext + nLeft; }
};

}  // namespace

struct b200spmv_mg {
    int nGPU = 0, format = 0;
    b200spmv_options opt{};
    int nRow = 0, nCol = 0;
    long long nnz = 0, haloTotal = 0;
    std::vector<int> bounds;
    std::vector<MgBlock> blk;
    bool converted = false;
    cudaGraphExec_t graph = nullptr;
    bool graph_tried = false;
    cudaEvent_t ev_fork = nullptr;
    int home = 0;                                              // device that was current at create
};

#define MG_CUDA(expr) B2_CUDA(expr)

static void mg_release(b200spmv_mg *m)
{
    if (m->graph) { cudaGraphExecDestroy(m->graph); m->graph = nullptr; }
    m->graph_tried = false;
    for (auto &b : m->blk) {
        cudaSetDevice(b.dev);
        if (b.A) b200spmv_destroy(b.A);
        if (b.halo) b200spmv_halo_free(b.halo);
        if (b.x_ext) cudaFree(b.x_ext);
        if (b.y) cudaFree(b.y);
        if (b.pull_owner) cudaFree(b.pull_owner);
        if (b.pull_idx) cudaFree(b.pull_idx);
        if (b.peer_x) cudaFree((void *)b.peer_x);
        if (b.compute) cudaStreamDestroy(b.compute);
        if (b.comm) cudaStreamDestroy(b.comm);
        for (cudaEvent_t e : {b.ev_x, b.ev_halo, b.ev_done, b.cev_halo, b.cev_join}) if (e) cudaEventDestroy(e);
    }
    m->blk.clear();
    m->converted = false;
    cudaSetDevice(m->home);
}

// after every block's coo is on its device: halo plan, conversion, buffers, pull plan
static int mg_finish_blocks(b200spmv_mg *m, std::vector<b200spmv_coo> &coos)
{
    const int G = m->nGPU;
    std::vector<std::vector<int>> halo_cols((size_t)G);
    for (int g = 0; g < G; g++) {
        MgBlock &b = m->blk[(size_t)g];
        MG_CUDA(cudaSetDevice(b.dev));
        int lo = 0, hi = 0;
        MG_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        MG_CUDA(cudaStreamCreateWithPriority(&b.compute, cudaStreamNonBlocking, lo));
        MG_CUDA(cudaStreamCreateWithPriority(&b.comm, cudaStreamNonBlocking, hi));   // the small pull kernel must not queue behind the interior rows
        for (cudaEvent_t *e : {&b.ev_x, &b.ev_halo, &b.ev_done, &b.cev_halo, &b.cev_join}) MG_CUDA(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
        b200spmv_coo &c = coos[(size_t)g];
        b.nnz = c.nnz;
        B2_TRY(b200spmv_halo_plan(&c, b.rowBegin, b.rowEnd, &b.halo, nullptr));
        long long info[8];
        B2_TRY(b200spmv_halo_info(b.halo, info));
        b.nLocal = (int)info[0]; b.nLeft = (int)info[1]; b.nRight = (int)info[2];
        b.interiorBegin = (int)info[3]; b.interiorEnd = (int)info[4];
        B2_TRY(b200spmv_create(m->format, &m->opt, &b.A));
        B2_TRY(b200spmv_convert_coo_device(b.A, c.nRow, c.nCol, c.nnz, c.row_d, c.col_d, c.val_d, nullptr));
        b200spmv_coo_free(&c);
        const int nRows = b.rowEnd - b.rowBegin;
        // row-range bookkeeping now: the step is captured in a graph and must never synchronise
        long long hasRows = 0;
        if (b200spmv_get_scalar(b.A, "has_rows", &hasRows) != B200SPMV_OK || !hasRows) { b.interiorBegin = 0; b.interiorEnd = 0; }
        if (hasRows) {
            if (b.interiorEnd > b.interiorBegin) B2_TRY(b200spmv_prepare_rows(b.A, b.interiorBegin, b.interiorEnd));
            if (b.interiorBegin > 0) B2_TRY(b200spmv_prepare_rows(b.A, 0, b.interiorBegin));
            if (b.interiorEnd < nRows) B2_TRY(b200spmv_prepare_rows(b.A, b.interiorEnd, nRows));
        }
        const size_t nx = (size_t)b.nLeft + b.nLocal + b.nRight;
        MG_CUDA(cudaMalloc((void **)&b.x_ext, sizeof(double) * std::max<size_t>(nx, 1)));
        MG_CUDA(cudaMalloc((void **)&b.y, sizeof(double) * std::max<size_t>((size_t)nRows, 1)));
        MG_CUDA(cudaMemset(b.x_ext, 0, sizeof(double) * std::max<size_t>(nx, 1)));
        const long long nb = b200spmv_halo_cols(b.halo, nullptr, 0);
        if (nb < 0) return (int)nb;
        halo_cols[(size_t)g].resize((size_t)nb / sizeof(int));
        if (nb) { const long long r = b200spmv_halo_cols(b.halo, halo_cols[(size_t)g].data(), nb); if (r < 0) return (int)r; }
        m->haloTotal += (long long)halo_cols[(size_t)g].size();
    }
    // pull plan: owner and position inside the owner's slice of every halo column; the peers' slice addresses
    std::vector<const double *> slices((size_t)G);
    for (int g = 0; g < G; g++) slices[(size_t)g] = m->blk[(size_t)g].x_owned();
    for (int g = 0; g < G; g++) {
        MgBlock &b = m->blk[(size_t)g];
        MG_CUDA(cudaSetDevice(b.dev));
        const std::vector<int> &hc = halo_cols[(size_t)g];
        std::vector<int> owner(hc.size()), idx(hc.size());
        for (size_t i = 0; i < hc.size(); i++) {
            const int p = (int)(std::upper_bound(m->bounds.begin(), m->bounds.end(), hc[i]) - m->bounds.begin()) - 1;
            if (p < 0 || p >= G || p == g) { set_error("mg: halo column %d of block %d has no remote owner", hc[i], g); return B200SPMV_ERR_STATE; }
            owner[i] = p;
            idx[i] = hc[i] - m->bounds[(size_t)p];
        }
        MG_CUDA(cudaMalloc((void **)&b.pull_owner, sizeof(int) * std::max<size_t>(hc.size(), 1)));
        MG_CUDA(cudaMalloc((void **)&b.pull_idx, sizeof(int) * std::max<size_t>(hc.size(), 1)));
        MG_CUDA(cudaMalloc((void **)&b.peer_x, sizeof(double *) * (size_t)G));
        if (!hc.empty()) {
            MG_CUDA(cudaMemcpy(b.pull_owner, owner.data(), sizeof(int) * hc.size(), cudaMemcpyHostToDevice));
            MG_CUDA(cudaMemcpy(b.pull_idx, idx.data(), sizeof(int) * hc.size(), cudaMemcpyHostToDevice));
        }
        MG_CUDA(cudaMemcpy((void *)b.peer_x, slices.data(), sizeof(double *) * (size_t)G, cudaMemcpyHostToDevice));
    }
    MG_CUDA(cudaSetDevice(m->home));
    m->converted = true;
    return B200SPMV_OK;
}

// enqueue one step on every GPU's streams.  captured = inside the graph capture: consecutive graph launches are
// serialised as a whole, so the cross-step ordering events are not needed; the capture uses its own events (an event
// recorded during capture cannot be waited on by ordinary stream work afterwards)
static int mg_enqueue_step(b200spmv_mg *m, bool captured)
{
    for (auto &b : m->blk) {
        MG_CUDA(cudaSetDevice(b.dev));
        const int nHalo = b.nLeft + b.nRight;
        if (!captured) {
            MG_CUDA(cudaStreamWaitEvent(b.comm, b.ev_done, 0));               // the previous step's boundary rows still read the halo slots
            for (auto &p : m->blk) if (p.dev != b.dev) MG_CUDA(cudaStreamWaitEvent(b.comm, p.ev_x, 0));   // the owners' slices are in place
        }
        if (nHalo) {
            int sms = 148;
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, b.dev);
            mg_pull_kernel<<<std::max(1, std::min(2 * sms, ceil_div(nHalo, 4 * MG_PULL_THREADS))), MG_PULL_THREADS, 0, b.comm>>>(
                b.peer_x, b.pull_owner, b.pull_idx, nHalo, b.nLeft, b.nLocal, b.x_ext);
            B2_KERNEL_CHECK();
        }
        MG_CUDA(cudaEventRecord(captured ? b.cev_halo : b.ev_halo, b.comm));
    }
    for (auto &b : m->blk) {
        MG_CUDA(cudaSetDevice(b.dev));
        const int nRows = b.rowEnd - b.rowBegin;
        if (!captured) MG_CUDA(cudaStreamWaitEvent(b.compute, b.ev_x, 0));
        if (b.interiorEnd > b.interiorBegin) {
            B2_TRY(b200spmv_multiply_rows(b.A, b.interiorBegin, b.interiorEnd, b.x_ext, b.y, b.compute));     // overlaps the pull
            MG_CUDA(cudaStreamWaitEvent(b.compute, captured ? b.cev_halo : b.ev_halo, 0));
            if (b.interiorBegin > 0) B2_TRY(b200spmv_multiply_rows(b.A, 0, b.interiorBegin, b.x_ext, b.y, b.compute));
            if (b.interiorEnd < nRows) B2_TRY(b200spmv_multiply_rows(b.A, b.interiorEnd, nRows, b.x_ext, b.y, b.compute));
        } else {
            MG_CUDA(cudaStreamWaitEvent(b.compute, captured ? b.cev_halo : b.ev_halo, 0));
            B2_TRY(b200spmv_multiply(b.A, b.x_ext, b.y, b.compute));
        }
        if (!captured) MG_CUDA(cudaEventRecord(b.ev_done, b.compute));
    }
    return B200SPMV_OK;
}

static int mg_capture(b200spmv_mg *m)
{
    m->graph_tried = true;
    static const bool off = getenv("B200SPMV_MG_NO_GRAPH") != nullptr;
    if (off) return B200SPMV_OK;
    MgBlock &root = m->blk[0];
    MG_CUDA(cudaSetDevice(root.dev));
    if (!m->ev_fork) MG_CUDA(cudaEventCreateWithFlags(&m->ev_fork, cudaEventDisableTiming));
    cudaGraph_t g = nullptr;
    bool ok = cudaStreamBeginCapture(root.compute, cudaStreamCaptureModeRelaxed) == cudaSuccess;
    if (ok) ok = cudaEventRecord(m->ev_fork, root.compute) == cudaSuccess;
    for (auto &b : m->blk) {                                   // every other stream joins the capture
        if (!ok) break;
        cudaSetDevice(b.dev);
        if (b.compute != root.compute) ok = cudaStreamWaitEvent(b.compute, m->ev_fork, 0) == cudaSuccess;
        if (ok) ok = cudaStreamWaitEvent(b.comm, m->ev_fork, 0) == cudaSuccess;
    }
    if (ok) ok = mg_enqueue_step(m, true) == B200SPMV_OK;
    for (auto &b : m->blk) {                                   // ... and is joined back into the origin stream
        if (!ok) break;
        cudaSetDevice(b.dev);
        ok = cudaEventRecord(b.cev_join, b.compute) == cudaSuccess;         // comm is already joined through cev_halo
        cudaSetDevice(root.dev);
        if (ok && b.compute != root.compute) ok = cudaStreamWaitEvent(root.compute, b.cev_join, 0) == cudaSuccess;
    }
    cudaSetDevice(root.dev);
    const cudaError_t e = cudaStreamEndCapture(root.compute, &g);
    if (!ok || e != cudaSuccess || !g) {
        cudaGetLastError();
        if (g) cudaGraphDestroy(g);
        return B200SPMV_OK;                                    // eager launches instead
    }
    if (cudaGraphInstantiate(&m->graph, g, 0) != cudaSuccess) { cudaGetLastError(); m->graph = nullptr; }
    cudaGraphDestroy(g);
    return B200SPMV_OK;
}

extern "C" {

int b200spmv_mg_create(int nGPU, int format, const b200spmv_options *opts, b200spmv_mg **out)
{
    clear_error();
    if (!out || nGPU < 1) { set_error("mg_create: bad argument"); return B200SPMV_ERR_INVALID; }
    *out = nullptr;
    if (opts && opts->transpose) {                              // a block's local A^T is not a block of the global A^T
        set_error("mg_create: options.transpose is not supported by the multi-GPU handle");
        return B200SPMV_ERR_UNSUPPORTED;
    }
    int have = 0;
    if (cudaGetDeviceCount(&have) != cudaSuccess || have < nGPU) {
        cudaGetLastError();
        set_error("mg_create: %d GPUs requested, %d visible; libb200spmv has no CPU fallback", nGPU, have);
        return B200SPMV_ERR_CUDA;
    }
    std::unique_ptr<b200spmv_mg> m(new b200spmv_mg());
    m->nGPU = nGPU;
    m->format = format;
    if (opts) m->opt = *opts;
    B2_CUDA(cudaGetDevice(&m->home));
    {   // validates format / options once
        b200spmv_matrix *probe = nullptr;
        B2_TRY(b200spmv_create(format, opts, &probe));
        b200spmv_destroy(probe);
    }
    for (int a = 0; a < nGPU; a++) {                           // every GPU maps every other GPU's memory (NVLink / NVSwitch)
        B2_CUDA(cudaSetDevice(a));
        for (int b = 0; b < nGPU; b++) {
            if (a == b) continue;
            int can = 0;
            B2_CUDA(cudaDeviceCanAccessPeer(&can, a, b));
            if (!can) { cudaSetDevice(m->home); set_error("mg_create: GPU %d cannot map GPU %d's memory (no peer access)", a, b); return B200SPMV_ERR_UNSUPPORTED; }
            const cudaError_t e = cudaDeviceEnablePeerAccess(b, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { cudaSetDevice(m->home); set_error("cudaDeviceEnablePeerAccess(%d -> %d): %s", a, b, cudaGetErrorString(e)); return B200SPMV_ERR_CUDA; }
            cudaGetLastError();
        }
    }
    B2_CUDA(cudaSetDevice(m->home));
    *out = m.release();
    return B200SPMV_OK;
}

int b200spmv_mg_destroy(b200spmv_mg *m)
{
    if (!m) return B200SPMV_OK;
    mg_release(m);
    if (m->ev_fork) cudaEventDestroy(m->ev_fork);
    delete m;
    return B200SPMV_OK;
}

int b200spmv_mg_convert_coo_host(b200spmv_mg *m, int nRow, int nCol, long long nnz, const int *row_h, const int *col_h,
                                 const double *val_h)
{
    clear_error();
    if (!m) { set_error("mg_convert: NULL handle"); return B200SPMV_ERR_INVALID; }
    if (nRow != nCol) { set_error("mg_convert: x is distributed like the rows, the matrix must be square (%d x %d)", nRow, nCol); return B200SPMV_ERR_UNSUPPORTED; }
    if (nnz < 0 || (nnz > 0 && (!row_h || !col_h || !val_h))) { set_error("mg_convert: bad COO arrays"); return B200SPMV_ERR_INVALID; }
    mg_release(m);
    const int G = m->nGPU;
    m->nRow = nRow; m->nCol = nCol; m->nnz = nnz; m->haloTotal = 0;
    // split where the running non-zero count passes g nnz / G (the rule of b200spmv_partition_rows)
    m->bounds.assign((size_t)G + 1, 0);
    m->bounds[(size_t)G] = nRow;
    for (int g = 1; g < G; g++) {
        const long long e = nnz * g / G;
        int bnd = nRow;
        if (e < nnz) { const int r = row_h[e]; bnd = (e == 0 || row_h[e - 1] != r) ? r : r + 1; }
        m->bounds[(size_t)g] = std::max(bnd, m->bounds[(size_t)g - 1]);
    }
    m->blk.assign((size_t)G, MgBlock());
    std::vector<b200spmv_coo> coos((size_t)G);
    for (int g = 0; g < G; g++) {
        MgBlock &b = m->blk[(size_t)g];
        b.dev = g;
        b.rowBegin = m->bounds[(size_t)g];
        b.rowEnd = m->bounds[(size_t)g + 1];
        const long long e0 = std::lower_bound(row_h, row_h + nnz, b.rowBegin) - row_h, e1 = std::lower_bound(row_h, row_h + nnz, b.rowEnd) - row_h;
        b200spmv_coo &c = coos[(size_t)g];
        memset(&c, 0, sizeof c);
        c.nRow = nRow; c.nCol = nCol; c.rowBegin = b.rowBegin; c.rowEnd = b.rowEnd; c.nnz = e1 - e0;
        B2_CUDA(cudaSetDevice(g));
        const size_t n = (size_t)std::max<long long>(c.nnz, 1);
        B2_CUDA(cudaMalloc((void **)&c.row_d, n * sizeof(int)));
        B2_CUDA(cudaMalloc((void **)&c.col_d, n * sizeof(int)));
        B2_CUDA(cudaMalloc((void **)&c.val_d, n * sizeof(double)));
        if (c.nnz) {
            B2_CUDA(cudaMemcpy(c.row_d, row_h + e0, (size_t)c.nnz * sizeof(int), cudaMemcpyHostToDevice));
            B2_CUDA(cudaMemcpy(c.col_d, col_h + e0, (size_t)c.nnz * sizeof(int), cudaMemcpyHostToDevice));
            B2_CUDA(cudaMemcpy(c.val_d, val_h + e0, (size_t)c.nnz * sizeof(double), cudaMemcpyHostToDevice));
        }
    }
    const int st = mg_finish_blocks(m, coos);
    if (st != B200SPMV_OK) { for (auto &c : coos) b200spmv_coo_free(&c); mg_release(m); }
    return st;
}

int b200spmv_mg_convert_synth(b200spmv_mg *m, int kind, long long p0, long long p1, unsigned long long seed)
{
    clear_error();
    if (!m) { set_error("mg_convert: NULL handle"); return B200SPMV_ERR_INVALID; }
    mg_release(m);
    const int G = m->nGPU;
    m->bounds.assign((size_t)G + 1, 0);
    B2_CUDA(cudaSetDevice(0));
    B2_TRY(b200spmv_partition_synth(kind, p0, p1, G, m->bounds.data()));
    m->nRow = m->nCol = m->bounds[(size_t)G];
    m->nnz = 0; m->haloTotal = 0;
    m->blk.assign((size_t)G, MgBlock());
    std::vector<b200spmv_coo> coos((size_t)G);
    for (int g = 0; g < G; g++) {                              // every GPU generates its own rows: nothing crosses PCIe
        MgBlock &b = m->blk[(size_t)g];
        b.dev = g;
        b.rowBegin = m->bounds[(size_t)g];
        b.rowEnd = m->bounds[(size_t)g + 1];
        B2_CUDA(cudaSetDevice(g));
        if (b.rowEnd <= b.rowBegin) { mg_release(m); set_error("mg_convert_synth: GPU %d would own no rows", g); return B200SPMV_ERR_INVALID; }
        const int st = b200spmv_synth(kind, p0, p1, seed, b.rowBegin, b.rowEnd, &coos[(size_t)g], nullptr);
        if (st != B200SPMV_OK) { for (auto &c : coos) b200spmv_coo_free(&c); mg_release(m); return st; }
        m->nnz += coos[(size_t)g].nnz;
    }
    const int st = mg_finish_blocks(m, coos);
    if (st != B200SPMV_OK) { for (auto &c : coos) b200spmv_coo_free(&c); mg_release(m); }
    return st;
}

static int mg_ready(b200spmv_mg *m, const char *what)
{
    if (!m) { set_error("%s: NULL handle", what); return B200SPMV_ERR_INVALID; }
    if (!m->converted) { set_error("%s: matrix not converted yet", what); return B200SPMV_ERR_STATE; }
    return B200SPMV_OK;
}

int b200spmv_mg_upload_x(b200spmv_mg *m, const double *x_h)
{
    B2_TRY(mg_ready(m, "mg_upload_x"));
    if (!x_h && m->nCol) { set_error("mg_upload_x: NULL x"); return B200SPMV_ERR_INVALID; }
    if (m->graph) {                                            // every earlier step (graph launches on GPU 0's compute stream) is finished
        B2_CUDA(cudaSetDevice(m->blk[0].dev));
        B2_CUDA(cudaStreamSynchronize(m->blk[0].compute));
    }
    for (auto &b : m->blk) {
        B2_CUDA(cudaSetDevice(b.dev));
        if (!m->graph) {
            B2_CUDA(cudaStreamWaitEvent(b.compute, b.ev_done, 0));
            for (auto &p : m->blk) B2_CUDA(cudaStreamWaitEvent(b.compute, p.ev_halo, 0));   // nobody is still pulling from this slice
        }
        if (b.nLocal) B2_CUDA(cudaMemcpyAsync(b.x_owned(), x_h + b.rowBegin, sizeof(double) * (size_t)b.nLocal, cudaMemcpyHostToDevice, b.compute));
        B2_CUDA(cudaEventRecord(b.ev_x, b.compute));
    }
    if (m->graph) {                                            // graph launches are ordered on GPU 0's compute stream only
        for (auto &b : m->blk) { B2_CUDA(cudaSetDevice(b.dev)); B2_CUDA(cudaStreamSynchronize(b.compute)); }
    }
    B2_CUDA(cudaSetDevice(m->home));
    return B200SPMV_OK;
}

static int mg_sync_all(b200spmv_mg *m)
{
    for (auto &b : m->blk) {
        B2_CUDA(cudaSetDevice(b.dev));
        B2_CUDA(cudaStreamSynchronize(b.compute));
        B2_CUDA(cudaStreamSynchronize(b.comm));
    }
    return B200SPMV_OK;
}

// one step, by graph launch or by eager launches
static int mg_step(b200spmv_mg *m, bool graph)
{
    if (graph) {
        B2_CUDA(cudaSetDevice(m->blk[0].dev));
        B2_CUDA(cudaGraphLaunch(m->graph, m->blk[0].compute));
        return B200SPMV_OK;
    }
    return mg_enqueue_step(m, false);
}

int b200spmv_mg_multiply(b200spmv_mg *m)
{
    B2_TRY(mg_ready(m, "mg_multiply"));
    if (!m->graph_tried) {
        for (auto &b : m->blk) { B2_CUDA(cudaSetDevice(b.dev)); B2_CUDA(cudaDeviceSynchronize()); }
        B2_TRY(mg_enqueue_step(m, false));                     // one eager step first: lazy kernel loading, first-use attributes
        for (auto &b : m->blk) { B2_CUDA(cudaSetDevice(b.dev)); B2_CUDA(cudaDeviceSynchronize()); }
        B2_TRY(mg_capture(m));
        if (m->graph) {
            // graph replay or eager launches, whichever is faster here (plan time, like DistSpmv.choose_launch): the multi-device
            // graph saves the host ~50 API calls per step but its fork / join nodes add latency -- 8 GPUs, c5: 0.320 ms replayed
            // against 0.291 ms eager; B200SPMV_MG_GRAPH=1 / B200SPMV_MG_NO_GRAPH keep one of them unconditionally
            static const bool keep = getenv("B200SPMV_MG_GRAPH") != nullptr;
            double t[2] = {0.0, 0.0};
            for (int mode = 0; mode < 2 && !keep; mode++) {
                for (int i = 0; i < 3; i++) B2_TRY(mg_step(m, mode == 0));
                B2_TRY(mg_sync_all(m));
                const auto t0 = std::chrono::steady_clock::now();
                for (int i = 0; i < 10; i++) B2_TRY(mg_step(m, mode == 0));
                B2_TRY(mg_sync_all(m));
                t[mode] = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
            }
            if (!keep && t[1] < t[0]) {
                cudaGraphExecDestroy(m->graph);
                m->graph = nullptr;
            }
        }
    }
    const int st = mg_step(m, m->graph != nullptr);
    B2_CUDA(cudaSetDevice(m->home));
    return st;
}

int b200spmv_mg_synchronize(b200spmv_mg *m)
{
    B2_TRY(mg_ready(m, "mg_synchronize"));
    for (auto &b : m->blk) {
        B2_CUDA(cudaSetDevice(b.dev));
        B2_CUDA(cudaStreamSynchronize(b.compute));
        B2_CUDA(cudaStreamSynchronize(b.comm));
    }
    B2_CUDA(cudaSetDevice(m->home));
    return B200SPMV_OK;
}

int b200spmv_mg_download_y(b200spmv_mg *m, double *y_h)
{
    B2_TRY(mg_ready(m, "mg_download_y"));
    if (!y_h && m->nRow) { set_error("mg_download_y: NULL y"); return B200SPMV_ERR_INVALID; }
    B2_TRY(b200spmv_mg_synchronize(m));
    for (auto &b : m->blk) {
        B2_CUDA(cudaSetDevice(b.dev));
        const int n = b.rowEnd - b.rowBegin;
        if (n) B2_CUDA(cudaMemcpyAsync(y_h + b.rowBegin, b.y, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, b.compute));
    }
    return b200spmv_mg_synchronize(m);
}

// SpMV(A_opt, x_opt, y) of the reference's driver, over all GPUs: scatter x, exchange + multiply, gather y
int b200spmv_mg_multiply_host(b200spmv_mg *m, const double *x_h, double *y_h)
{
    B2_TRY(b200spmv_mg_upload_x(m, x_h));
    B2_TRY(b200spmv_mg_multiply(m));
    return b200spmv_mg_download_y(m, y_h);
}

int b200spmv_mg_get_scalar(b200spmv_mg *m, const char *name, long long *out)
{
    if (!m || !name || !out) { set_error("mg_get_scalar: NULL argument"); return B200SPMV_ERR_INVALID; }
    const std::string n(name);
    if (n == "nGPU") { *out = m->nGPU; return B200SPMV_OK; }
    B2_TRY(mg_ready(m, "mg_get_scalar"));
    if (n == "nRow") { *out = m->nRow; return B200SPMV_OK; }
    if (n == "nCol") { *out = m->nCol; return B200SPMV_OK; }
    if (n == "nNnz") { *out = m->nnz; return B200SPMV_OK; }
    if (n == "halo_total") { *out = m->haloTotal; return B200SPMV_OK; }
    if (n == "graphed") { *out = m->graph ? 1 : 0; return B200SPMV_OK; }
    if (n == "alg_bytes") {                                    // compulsory bytes of the GLOBAL multiply: the blocks' matrix bytes + x + y once
        long long sum = 0;
        for (auto &b : m->blk) {
            long long v = 0, nr = b.rowEnd - b.rowBegin, nc = (long long)b.nLeft + b.nLocal + b.nRight;
            cudaSetDevice(b.dev);
            B2_TRY(b200spmv_get_scalar(b.A, "alg_bytes", &v));
            sum += v - 8 * nr - 8 * nc;
        }
        cudaSetDevice(m->home);
        *out = sum + 8LL * m->nRow + 8LL * m->nCol;
        return B200SPMV_OK;
    }
    if (n == "launches") {
        long long sum = 0;
        for (auto &b : m->blk) {
            long long v = 0;
            B2_TRY(b200spmv_get_scalar(b.A, "launches", &v));
            const int nRows = b.rowEnd - b.rowBegin;
            const int parts = b.interiorEnd > b.interiorBegin ? 1 + (b.interiorBegin > 0) + (b.interiorEnd < nRows) : 1;
            sum += v * parts + ((b.nLeft + b.nRight) ? 1 : 0);
        }
        *out = sum;
        return B200SPMV_OK;
    }
    set_error("mg_get_scalar: unknown scalar '%s'", name);
    return B200SPMV_ERR_INVALID;
}

int b200spmv_mg_get_bounds(b200spmv_mg *m, int *bounds_h)
{
    B2_TRY(mg_ready(m, "mg_get_bounds"));
    if (!bounds_h) { set_error("mg_get_bounds: NULL argument"); return B200SPMV_ERR_INVALID; }
    for (int g = 0; g <= m->nGPU; g++) bounds_h[g] = m->bounds[(size_t)g];
    return B200SPMV_OK;
}

}  // extern "C"
