// chunk_stream.cu -- kernel and launcher of the TMA-fed row-chunk stream (see chunk_stream.cuh).
#include <algorithm>
#include <climits>
#include <cstdlib>
#include <cstring>
#include <map>

#include "chunk_stream.cuh"

namespace b2 {

// VT = stored value type, XT = type of x and y, AT = type the row sums are accumulated in.  DICT = the column feed:
// false = idx (bulk-copied with the values) and ptr (two loads per row, prefetched a chunk ahead); true = the chunk's
// offset dictionary, row masks and warp bases (one bulk copy of its meta record, chunk_stream.cuh).  In both, capI is
// the ints of a stage's column part: the idx run (rounded to 16 bytes) or the meta record.
template <typename VT, typename XT, typename AT, int MAXL, int TH, bool ACC, bool DICT>
__global__ void __launch_bounds__(TH)
chunk_stream_kernel(const int *__restrict__ ptr, const int *__restrict__ idx, const int *__restrict__ meta,
                    const VT *__restrict__ val, const XT *__restrict__ x, XT *__restrict__ y, int rowBegin, int rowEnd,
                    int chunk0, int nChunks, int capI, int capV, int S, int acc_mode)
{
    constexpr int MI = CS_META_INTS(TH);
    extern __shared__ __align__(128) unsigned char cs_smem[];
    __shared__ __align__(8) uint64_t bar[CS_MAXSTAGES];
    __shared__ int sbaseI[CS_MAXSTAGES], sbaseV[CS_MAXSTAGES];    // entry index that sits at slot 0 of the stage
    int *sidx = reinterpret_cast<int *>(cs_smem);
    VT *sval = reinterpret_cast<VT *>(cs_smem + (size_t)S * capI * sizeof(int));
    const int tid = threadIdx.x;
    const uint64_t pol_stream = policy_evict_first(), pol_x = policy_evict_last();

    // thread 0 only: bulk copies of chunk g's column part and of its entries [b, e) into stage s; the entry copies'
    // sources rounded down / sizes rounded up to 16 bytes (meta records are whole multiples of 16 bytes)
    auto issue = [&](int s, long long g, int b, int e) {
        const int *srcI = idx + b;
        const VT *srcV = val + b;
        const int misI = (int)((reinterpret_cast<uintptr_t>(srcI) & 15) / sizeof(int));
        const int misV = (int)((reinterpret_cast<uintptr_t>(srcV) & 15) / sizeof(VT));
        const int n = e - b;
        const uint32_t bytesI = DICT ? (uint32_t)(MI * sizeof(int)) : n ? (uint32_t)(((n + misI) * (int)sizeof(int) + 15) & ~15) : 0u;
        const uint32_t bytesV = n ? (uint32_t)(((n + misV) * (int)sizeof(VT) + 15) & ~15) : 0u;
        sbaseI[s] = b - misI;
        sbaseV[s] = b - misV;
        mbar_expect_tx(&bar[s], bytesI + bytesV);               // release: sbase*[s] visible to whoever passes the wait
        if (DICT) tma_load_1d(sidx + (size_t)s * capI, meta + g * MI, bytesI, &bar[s], pol_stream);
        if (n) {
            if (!DICT) tma_load_1d(sidx + (size_t)s * capI, srcI - misI, bytesI, &bar[s], pol_stream);
            tma_load_1d(sval + (size_t)s * capV, srcV - misV, bytesV, &bar[s], pol_stream);
        }
    };
    // chunk g covers rows [g TH, (g+1) TH) clipped to [rowBegin, rowEnd)
    auto lo_of = [&](long long g) { return (int)min((long long)rowEnd, max((long long)rowBegin, g * TH)); };

    if (tid == 0)
        for (int s = 0; s < S; s++) mbar_init(&bar[s], 1);
    __syncthreads();
    if (tid == 0) {
        for (int s = 0; s < S; s++) {
            const long long c = (long long)blockIdx.x + (long long)s * gridDim.x;
            if (c < nChunks) issue(s, chunk0 + c, ptr[lo_of(chunk0 + c)], ptr[lo_of(chunk0 + c + 1)]);
        }
    }
    long long g = (long long)chunk0 + blockIdx.x;
    int r = (int)min(g * TH + tid, (long long)0x7fffffff);
    bool valid = r >= rowBegin && r < rowEnd;
    int p = 0, q = 0;
    if (!DICT && valid) {
        p = ptr[r];
        q = ptr[r + 1];
    }
    int k = 0;
    for (long long c = blockIdx.x; c < nChunks; c += gridDim.x, k++) {
        const int s = k % S;
        // prefetches that land while this chunk is being reduced: the bounds of the chunk issued at the end of this
        // iteration (thread 0), this thread's row pointers in the CTA's next chunk (idx feed), and y for the
        // accumulating modes
        const long long cIssue = c + (long long)S * gridDim.x, cNext = c + gridDim.x;
        int nb = 0, ne = 0, pn = 0, qn = 0;
        if (tid == 0 && cIssue < nChunks) {
            nb = ptr[lo_of(chunk0 + cIssue)];
            ne = ptr[lo_of(chunk0 + cIssue + 1)];
        }
        const long long rnl = (chunk0 + cNext) * TH + tid;
        const int rn = (int)min(rnl, (long long)0x7fffffff);
        const bool validn = cNext < nChunks && rn >= rowBegin && rn < rowEnd;
        if (!DICT && validn) {
            pn = ptr[rn];
            qn = ptr[rn + 1];
        }
        const AT y0 = (ACC && valid) ? (AT)y[r] : (AT)0;
        mbar_wait(&bar[s], (uint32_t)(k / S) & 1u);
        AT acc = (ACC && acc_mode == CS_CONTINUE) ? y0 : (AT)0;
        XT xs[MAXL];
        int len, vo;
        if (DICT) {
            const int *rec = sidx + (size_t)s * capI;
            const uint32_t mrow = reinterpret_cast<const uint16_t *>(rec + CS_DICT + TH / 32)[tid];
            // the row's first entry: its warp's base plus the entries of the warp's rows before it (every row of the
            // chunk counts, in range or not: the bases are those of the whole chunk)
            const int lane = tid & 31, cnt = __popc(mrow);
            int inc = cnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= o) inc += t;
            }
            vo = s * capV + (rec[CS_DICT + (tid >> 5)] + inc - cnt - sbaseV[s]);
            uint32_t m = valid ? mrow : 0u;
            len = __popc(m);
#pragma unroll
            for (int j = 0; j < MAXL; j++)
                if (j < len) {                                  // set bits low to high = ascending columns = idx order
                    xs[j] = ld_x(x + (r + rec[__ffs(m) - 1]), pol_x);
                    m &= m - 1;
                }
        } else {
            const int io = s * capI + (p - sbaseI[s]);
            vo = s * capV + (p - sbaseV[s]);
            len = q - p;
#pragma unroll
            for (int j = 0; j < MAXL; j++)
                if (j < len) xs[j] = ld_x(x + sidx[io + j], pol_x);
        }
#pragma unroll
        for (int j = 0; j < MAXL; j++)
            if (j < len) acc = Arith<AT>::add(acc, Arith<AT>::mul((AT)sval[vo + j], (AT)xs[j]));
        if (valid) y[r] = (XT)((ACC && acc_mode == CS_ADD) ? Arith<AT>::add(y0, acc) : acc);
        __syncthreads();                                       // every thread is done with stage s
        if (tid == 0 && cIssue < nChunks) issue(s, chunk0 + cIssue, nb, ne);
        r = rn; p = pn; q = qn; valid = validn;
    }
}

// The multi-vector form (overwrite; VT, XT, AT as in chunk_stream_kernel): chunks arrive exactly as in chunk_stream_kernel,
// and the thread of row r sums KP vectors (columns j < k of X; KP = k rounded up to 1, 2, 4, 8) over the row's entries in
// ascending column order, each with the unfused mul / add of the single multiply.  VEC: X rows gathered in 8- or 16-byte
// pieces (ld_xrow).
template <typename VT, typename XT, typename AT, int MAXL, int TH, bool DICT, int KP, bool VEC>
__global__ void __launch_bounds__(TH, 1)
chunk_stream_multi_kernel(const int *__restrict__ ptr, const int *__restrict__ idx, const int *__restrict__ meta,
                          const VT *__restrict__ val, const XT *__restrict__ X, long long ldx, XT *__restrict__ Y,
                          long long ldy, int kv, int rowBegin, int rowEnd, int chunk0, int nChunks, int capI, int capV, int S)
{
    constexpr int MI = CS_META_INTS(TH);
    extern __shared__ __align__(128) unsigned char cs_smem[];
    __shared__ __align__(8) uint64_t bar[CS_MAXSTAGES];
    __shared__ int sbaseI[CS_MAXSTAGES], sbaseV[CS_MAXSTAGES];
    int *sidx = reinterpret_cast<int *>(cs_smem);
    VT *sval = reinterpret_cast<VT *>(cs_smem + (size_t)S * capI * sizeof(int));
    const int tid = threadIdx.x;
    const uint64_t pol_stream = policy_evict_first(), pol_x = policy_evict_last();

    auto issue = [&](int s, long long g, int b, int e) {
        const int *srcI = idx + b;
        const VT *srcV = val + b;
        const int misI = (int)((reinterpret_cast<uintptr_t>(srcI) & 15) / sizeof(int));
        const int misV = (int)((reinterpret_cast<uintptr_t>(srcV) & 15) / sizeof(VT));
        const int n = e - b;
        const uint32_t bytesI = DICT ? (uint32_t)(MI * sizeof(int)) : n ? (uint32_t)(((n + misI) * (int)sizeof(int) + 15) & ~15) : 0u;
        const uint32_t bytesV = n ? (uint32_t)(((n + misV) * (int)sizeof(VT) + 15) & ~15) : 0u;
        sbaseI[s] = b - misI;
        sbaseV[s] = b - misV;
        mbar_expect_tx(&bar[s], bytesI + bytesV);
        if (DICT) tma_load_1d(sidx + (size_t)s * capI, meta + g * MI, bytesI, &bar[s], pol_stream);
        if (n) {
            if (!DICT) tma_load_1d(sidx + (size_t)s * capI, srcI - misI, bytesI, &bar[s], pol_stream);
            tma_load_1d(sval + (size_t)s * capV, srcV - misV, bytesV, &bar[s], pol_stream);
        }
    };
    auto lo_of = [&](long long g) { return (int)min((long long)rowEnd, max((long long)rowBegin, g * TH)); };

    if (tid == 0)
        for (int s = 0; s < S; s++) mbar_init(&bar[s], 1);
    __syncthreads();
    if (tid == 0) {
        for (int s = 0; s < S; s++) {
            const long long c = (long long)blockIdx.x + (long long)s * gridDim.x;
            if (c < nChunks) issue(s, chunk0 + c, ptr[lo_of(chunk0 + c)], ptr[lo_of(chunk0 + c + 1)]);
        }
    }
    long long g = (long long)chunk0 + blockIdx.x;
    int r = (int)min(g * TH + tid, (long long)0x7fffffff);
    bool valid = r >= rowBegin && r < rowEnd;
    int p = 0, q = 0;
    if (!DICT && valid) {
        p = ptr[r];
        q = ptr[r + 1];
    }
    int k = 0;
    for (long long c = blockIdx.x; c < nChunks; c += gridDim.x, k++) {
        const int s = k % S;
        const long long cIssue = c + (long long)S * gridDim.x, cNext = c + gridDim.x;
        int nb = 0, ne = 0, pn = 0, qn = 0;
        if (tid == 0 && cIssue < nChunks) {
            nb = ptr[lo_of(chunk0 + cIssue)];
            ne = ptr[lo_of(chunk0 + cIssue + 1)];
        }
        const long long rnl = (chunk0 + cNext) * TH + tid;
        const int rn = (int)min(rnl, (long long)0x7fffffff);
        const bool validn = cNext < nChunks && rn >= rowBegin && rn < rowEnd;
        if (!DICT && validn) {
            pn = ptr[rn];
            qn = ptr[rn + 1];
        }
        mbar_wait(&bar[s], (uint32_t)(k / S) & 1u);
        const int *rec = sidx + (size_t)s * capI;
        int len, vo, io = 0;
        uint32_t m = 0;
        if (DICT) {
            const uint32_t mrow = reinterpret_cast<const uint16_t *>(rec + CS_DICT + TH / 32)[tid];
            const int lane = tid & 31, cnt = __popc(mrow);
            int inc = cnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= o) inc += t;
            }
            vo = s * capV + (rec[CS_DICT + (tid >> 5)] + inc - cnt - sbaseV[s]);
            m = valid ? mrow : 0u;
            len = __popc(m);
        } else {
            io = s * capI + (p - sbaseI[s]);
            vo = s * capV + (p - sbaseV[s]);
            len = q - p;
        }
        AT acc[KP];
#pragma unroll
        for (int v = 0; v < KP; v++) acc[v] = (AT)0;
#pragma unroll
        for (int j = 0; j < MAXL; j++)
            if (j < len) {
                int col;
                if (DICT) {                                     // set bits low to high = ascending columns = idx order
                    col = r + rec[__ffs(m) - 1];
                    m &= m - 1;
                } else {
                    col = sidx[io + j];
                }
                XT xv[KP];
                ld_xrow<KP, VEC>(xv, X + (long long)col * ldx, kv, pol_x);
                const AT a = (AT)sval[vo + j];
#pragma unroll
                for (int v = 0; v < KP; v++) acc[v] = Arith<AT>::add(acc[v], Arith<AT>::mul(a, (AT)xv[v]));
            }
        if (valid) {
            XT *yr = Y + (long long)r * ldy;
#pragma unroll
            for (int v = 0; v < KP; v++)
                if (v < kv) yr[v] = (XT)acc[v];
        }
        __syncthreads();
        if (tid == 0 && cIssue < nChunks) issue(s, chunk0 + cIssue, nb, ne);
        r = rn; p = pn; q = qn; valid = validn;
    }
}

__global__ void chunk_cap_kernel(const int *__restrict__ ptr, int nRow, int th, int nChunks, int *__restrict__ out)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    int n = 0;
    if (c < nChunks) n = ptr[(int)min((long long)nRow, ((long long)c + 1) * th)] - ptr[(long long)c * th];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) n = max(n, __shfl_xor_sync(0xffffffffu, n, o));
    if ((threadIdx.x & 31) == 0 && n > 0) atomicMax(out, n);
}

// One CTA per chunk of TH rows, one thread per row (rows have at most CS_MAXLEN entries): the chunk's meta record
// (chunk_stream.cuh).  The distinct col - row offsets come out in ascending order, one block minimum of "the smallest
// offset above the last one" at a time; a (CS_DICT + 1)-th sets *overflow, and so does a row whose columns do not ascend
// (the masks could not keep its order).
template <int TH>
__global__ void __launch_bounds__(TH)
chunk_dict_kernel(const int *__restrict__ ptr, const int *__restrict__ idx, int nRow, int *__restrict__ meta,
                  int *__restrict__ overflow)
{
    __shared__ int red[2][TH / 32];
    __shared__ int dict[CS_DICT];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const long long r = (long long)blockIdx.x * TH + tid;
    int b = 0, n = 0;
    if (r < nRow) {
        b = ptr[r];
        n = ptr[r + 1] - b;
    }
    int off[CS_MAXLEN];                                        // INT_MAX: no entry (a column is below INT_MAX)
#pragma unroll
    for (int j = 0; j < CS_MAXLEN; j++) off[j] = j < n ? idx[b + j] - (int)r : INT_MAX;
    int nd = 0;
    for (int cur = INT_MIN;;) {                               // every offset is above INT_MIN
        int mn = INT_MAX;
#pragma unroll
        for (int j = 0; j < CS_MAXLEN; j++)
            if (off[j] > cur) mn = min(mn, off[j]);
        mn = __reduce_min_sync(0xffffffffu, mn);
        if (lane == 0) red[nd & 1][w] = mn;                   // two buffers: one barrier per round
        __syncthreads();
        mn = INT_MAX;
#pragma unroll
        for (int i = 0; i < TH / 32; i++) mn = min(mn, red[nd & 1][i]);
        if (mn == INT_MAX) break;                              // uniform: no offset above cur
        if (nd == CS_DICT) {                                   // uniform
            if (tid == 0) *overflow = 1;
            return;
        }
        if (tid == 0) dict[nd] = mn;
        cur = mn;
        nd++;
    }
    uint32_t m = 0;
    int last = -1;
    bool bad = false;
#pragma unroll
    for (int j = 0; j < CS_MAXLEN; j++)
        if (j < n) {
            int k = 0;                                         // dict[k] == off[j]
            for (int i = 0; i < nd; i++) k += dict[i] < off[j];
            bad |= k <= last;
            last = k;
            m |= 1u << k;
        }
    if (bad) *overflow = 1;
    int *rec = meta + (size_t)blockIdx.x * CS_META_INTS(TH);
    if (tid < CS_DICT) rec[tid] = tid < nd ? dict[tid] : 0;
    if (lane == 0) rec[CS_DICT + w] = ptr[min(r, (long long)nRow)];
    reinterpret_cast<uint16_t *>(rec + CS_DICT + TH / 32)[tid] = (uint16_t)m;
}

int ChunkStream::build(const int *ptr_d, const int *idx_d, const void *val_d, bool val_is_f32, int nRow_, int nnz,
                       int maxLen_, cudaStream_t s)
{
    ptr = ptr_d; idx = idx_d; val = val_d; f32 = val_is_f32; nRow = nRow_; maxLen = maxLen_;
    feed = CS_FEED_IDX;
    meta.release();
    static const int env_max = getenv("B200SPMV_TMA_MAXLEN") ? atoi(getenv("B200SPMV_TMA_MAXLEN")) : CS_MAXLEN;
    const int env_th = getenv("B200SPMV_TMA_R") ? atoi(getenv("B200SPMV_TMA_R")) : 0;   // read per build: tests switch it
    ok = nnz > 0 && nRow > 0 && maxLen > 0 && maxLen <= std::min(env_max, CS_MAXLEN);
    if (!ok) return B200SPMV_OK;
    // rows per chunk = threads per CTA (c5: 256 and 512 within 1.5 % of each other, 128: -15 %)
    th = env_th == 512 ? 512 : 256;
    const int nChunks = ceil_div(nRow, th);
    // the offset dictionary unless B200SPMV_CS_FEED=idx (experiments)
    const char *env_feed = getenv("B200SPMV_CS_FEED");
    const bool want_dict = !(env_feed && !strcmp(env_feed, "idx"));
    DevBuf<int> m;                                             // [0] largest chunk, [1] dictionary overflow
    B2_TRY(m.alloc(2));
    B2_CUDA(cudaMemsetAsync(m.p, 0, 2 * sizeof(int), s));
    chunk_cap_kernel<<<ceil_div(nChunks, 256), 256, 0, s>>>(ptr, nRow, th, nChunks, m.p);
    B2_KERNEL_CHECK();
    const size_t metaInts = (size_t)nChunks * CS_META_INTS(th);
    if (want_dict) {
        B2_TRY(meta.alloc(metaInts + CS_SLACK));
        B2_CUDA(cudaMemsetAsync(meta.p + metaInts, 0, CS_SLACK * sizeof(int), s));
        if (th == 512) chunk_dict_kernel<512><<<nChunks, 512, 0, s>>>(ptr, idx, nRow, meta.p, m.p + 1);
        else chunk_dict_kernel<256><<<nChunks, 256, 0, s>>>(ptr, idx, nRow, meta.p, m.p + 1);
        B2_KERNEL_CHECK();
    }
    int h[2] = {0, 0};
    B2_CUDA(cudaMemcpyAsync(h, m.p, sizeof h, cudaMemcpyDeviceToHost, s));
    B2_CUDA(cudaStreamSynchronize(s));
    cap = h[0];
    if (want_dict && !h[1]) feed = CS_FEED_DICT;
    else meta.release();
    // a stage must fit twice into one SM's shared memory next to nothing else
    const size_t stage = (size_t)(cap + 16) * (f32 ? 4 : 8) + (feed == CS_FEED_DICT ? CS_META_INTS(th) * 4 : (size_t)(cap + 16) * 4);
    if (2 * stage > 200 * 1024) ok = false;
    return B200SPMV_OK;
}

// CTAs per SM of the single multiply, from the occupancy limit: shed CTAs while their stages take more than
// CS_SMEM_PER_SM of the SM's 256 KB of L1 and shared memory, but never below CS_MIN_THREADS_PER_SM threads.  The stages
// hold the values only, so the L1 the gathers of x hit in is what the stages leave.  Measured on c5 (B200, fp64,
// dictionary feed, profiles/chunk_ctas_ab.md): 6 CTAs of 29.9 KB (180 KB) lost to 5 (150 KB) in every session; 4 CTAs
// (1024 threads) lost to both; fp32 at 8 CTAs of 15.6 KB (125 KB) lost 4 % at 6 and 9 % at 5.
constexpr size_t CS_SMEM_PER_SM = 160 * 1024;
constexpr int CS_MIN_THREADS_PER_SM = 1280;
static int cs_ctas_per_sm(int occupancy, int th, size_t smem)
{
    int n = occupancy;
    while ((n - 1) * th >= CS_MIN_THREADS_PER_SM && (size_t)n * smem > CS_SMEM_PER_SM) n--;
    return n;
}

// the launch of one feed
template <typename VT, typename XT, typename AT, int MAXL, int TH, bool ACC, bool DICT>
static int cs_launch(const ChunkStream &c, const XT *x, XT *y, int rb, int re, int acc, cudaStream_t s)
{
    constexpr int VA = 16 / (int)sizeof(VT);
    static const int env_s = getenv("B200SPMV_TMA_S") ? atoi(getenv("B200SPMV_TMA_S")) : 0;
    static const int env_b = getenv("B200SPMV_TMA_CTAS") ? atoi(getenv("B200SPMV_TMA_CTAS")) : 0;
    const int S = (env_s >= 1 && env_s <= CS_MAXSTAGES) ? env_s : 2;
    const int capI = DICT ? CS_META_INTS(TH) : (c.cap + 8) & ~3, capV = (c.cap + 2 * VA) & ~(VA - 1);
    const size_t smem = (size_t)S * ((size_t)capI * 4 + (size_t)capV * sizeof(VT));
    auto kern = chunk_stream_kernel<VT, XT, AT, MAXL, TH, ACC, DICT>;
    static int sms = 0;
    // occupancy of THIS instantiation by (device, shared-memory size): the opt-in shared-memory attribute is per device
    static std::map<std::pair<int, size_t>, int> per_sm;
    int dev = 0;
    B2_CUDA(cudaGetDevice(&dev));
    if (!sms) B2_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const auto key = std::make_pair(dev, smem);
    auto it = per_sm.find(key);
    if (it == per_sm.end()) {
        B2_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 200 * 1024)));
        int n = 0;
        B2_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kern, TH, smem));
        if (n < 1) { set_error("row-chunk stream: %zu bytes of shared memory do not fit", smem); return B200SPMV_ERR_UNSUPPORTED; }
        it = per_sm.emplace(key, n).first;
    }
    const int perSm = env_b > 0 ? std::min(it->second, env_b) : cs_ctas_per_sm(it->second, TH, smem);
    const int chunk0 = rb / TH, nChunks = ceil_div(re, TH) - chunk0;
    const int grid = std::min(nChunks, sms * perSm);
    kern<<<grid, TH, smem, s>>>(c.ptr, c.idx, c.meta.p, static_cast<const VT *>(c.val), x, y, rb, re, chunk0, nChunks, capI, capV, S, acc);
    B2_KERNEL_CHECK();
    return B200SPMV_OK;
}

template <typename VT, typename XT, typename AT, int MAXL, int TH, bool ACC>
static int cs_feed(const ChunkStream &c, const XT *x, XT *y, int rb, int re, int acc, cudaStream_t s)
{
    if (c.feed == CS_FEED_DICT) return cs_launch<VT, XT, AT, MAXL, TH, ACC, true>(c, x, y, rb, re, acc, s);
    return cs_launch<VT, XT, AT, MAXL, TH, ACC, false>(c, x, y, rb, re, acc, s);
}

template <typename VT, typename XT, typename AT>
static int cs_dispatch(const ChunkStream &c, const XT *x, XT *y, int rb, int re, int acc, cudaStream_t s)
{
#define CS_GO(MAXL)                                                                                       \
    do {                                                                                                  \
        if (c.th == 512 && acc) return cs_feed<VT, XT, AT, MAXL, 512, true>(c, x, y, rb, re, acc, s);   \
        if (c.th == 512) return cs_feed<VT, XT, AT, MAXL, 512, false>(c, x, y, rb, re, acc, s);         \
        if (acc) return cs_feed<VT, XT, AT, MAXL, 256, true>(c, x, y, rb, re, acc, s);                  \
        return cs_feed<VT, XT, AT, MAXL, 256, false>(c, x, y, rb, re, acc, s);                          \
    } while (0)
    if (c.maxLen <= 8) CS_GO(8);
    else CS_GO(16);
#undef CS_GO
}

int ChunkStream::run(const double *x, double *y, int rb, int re, int acc, cudaStream_t s) const
{
    if (rb < 0 || re > nRow || rb > re) { set_error("multiply_rows: bad row range [%d,%d) for %d rows", rb, re, nRow); return B200SPMV_ERR_INVALID; }
    if (rb == re) return B200SPMV_OK;
    if (f32) return cs_dispatch<float, double, double>(*this, x, y, rb, re, acc, s);
    return cs_dispatch<double, double, double>(*this, x, y, rb, re, acc, s);
}

// fp32 vectors (values must be stored as fp32): accumulation in fp32 or fp64
int ChunkStream::run_f32(const float *x, float *y, int rb, int re, int acc, bool acc64, cudaStream_t s) const
{
    if (rb < 0 || re > nRow || rb > re) { set_error("multiply_rows: bad row range [%d,%d) for %d rows", rb, re, nRow); return B200SPMV_ERR_INVALID; }
    if (!f32) { set_error("row-chunk stream: fp32 vectors need fp32 value storage"); return B200SPMV_ERR_STATE; }
    if (rb == re) return B200SPMV_OK;
    if (acc64) return cs_dispatch<float, float, double>(*this, x, y, rb, re, acc, s);
    return cs_dispatch<float, float, float>(*this, x, y, rb, re, acc, s);
}

// the multi-vector launch: stages, grid and occupancy as in cs_launch
template <typename VT, typename XT, typename AT, int MAXL, int TH, bool DICT, int KP, bool VEC>
static int cs_multi_launch(const ChunkStream &c, int k, const XT *X, long long ldx, XT *Y, long long ldy, cudaStream_t s)
{
    constexpr int S = 2, VA = 16 / (int)sizeof(VT);
    const int capI = DICT ? CS_META_INTS(TH) : (c.cap + 8) & ~3, capV = (c.cap + 2 * VA) & ~(VA - 1);
    const size_t smem = (size_t)S * ((size_t)capI * 4 + (size_t)capV * sizeof(VT));
    auto kern = chunk_stream_multi_kernel<VT, XT, AT, MAXL, TH, DICT, KP, VEC>;
    static int sms = 0;
    static std::map<std::pair<int, size_t>, int> per_sm;
    int dev = 0;
    B2_CUDA(cudaGetDevice(&dev));
    if (!sms) B2_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const auto key = std::make_pair(dev, smem);
    auto it = per_sm.find(key);
    if (it == per_sm.end()) {
        B2_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 200 * 1024)));
        int n = 0;
        B2_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kern, TH, smem));
        if (n < 1) { set_error("row-chunk stream: %zu bytes of shared memory do not fit", smem); return B200SPMV_ERR_UNSUPPORTED; }
        it = per_sm.emplace(key, n).first;
    }
    const int nChunks = ceil_div(c.nRow, TH);
    const int grid = std::min(nChunks, sms * it->second);
    kern<<<grid, TH, smem, s>>>(c.ptr, c.idx, c.meta.p, static_cast<const VT *>(c.val), X, ldx, Y, ldy, k, 0, c.nRow, 0,
                                nChunks, capI, capV, S);
    B2_KERNEL_CHECK();
    return B200SPMV_OK;
}

template <typename VT, typename XT, typename AT, int MAXL, int TH, bool DICT>
static int cs_multi_k(const ChunkStream &c, int k, const XT *X, long long ldx, XT *Y, long long ldy, cudaStream_t s)
{
#define CS_MK(KP)                                                                                              \
    return ld_xrow_vec(X, ldx, KP) ? cs_multi_launch<VT, XT, AT, MAXL, TH, DICT, KP, true>(c, k, X, ldx, Y, ldy, s) \
                                   : cs_multi_launch<VT, XT, AT, MAXL, TH, DICT, KP, false>(c, k, X, ldx, Y, ldy, s)
    if (k == 1) return cs_multi_launch<VT, XT, AT, MAXL, TH, DICT, 1, false>(c, k, X, ldx, Y, ldy, s);
    if (k == 2) CS_MK(2);
    if (k <= 4) CS_MK(4);
    CS_MK(8);
#undef CS_MK
}

template <typename VT, typename XT, typename AT>
static int cs_multi_dispatch(const ChunkStream &c, int k, const XT *X, long long ldx, XT *Y, long long ldy, cudaStream_t s)
{
#define CS_MF(MAXL, TH)                                                                                         \
    return c.feed == CS_FEED_DICT ? cs_multi_k<VT, XT, AT, MAXL, TH, true>(c, k, X, ldx, Y, ldy, s)              \
                                  : cs_multi_k<VT, XT, AT, MAXL, TH, false>(c, k, X, ldx, Y, ldy, s)
    if (c.th == 512) {
        if (c.maxLen <= 8) CS_MF(8, 512);
        CS_MF(16, 512);
    }
    if (c.maxLen <= 8) CS_MF(8, 256);
    CS_MF(16, 256);
#undef CS_MF
}

int ChunkStream::run_multi(int k, const double *X, long long ldx, double *Y, long long ldy, cudaStream_t s) const
{
    if (f32) { set_error("multiply_multi: the row-chunk stream holds fp32 values"); return B200SPMV_ERR_UNSUPPORTED; }
    if (nRow == 0) return B200SPMV_OK;
    return cs_multi_dispatch<double, double, double>(*this, k, X, ldx, Y, ldy, s);
}

int ChunkStream::run_multi_f32(int k, const float *X, long long ldx, float *Y, long long ldy, bool acc64, cudaStream_t s) const
{
    if (!f32) { set_error("row-chunk stream: fp32 vectors need fp32 value storage"); return B200SPMV_ERR_STATE; }
    if (nRow == 0) return B200SPMV_OK;
    if (acc64) return cs_multi_dispatch<float, float, double>(*this, k, X, ldx, Y, ldy, s);
    return cs_multi_dispatch<float, float, float>(*this, k, X, ldx, Y, ldy, s);
}

}  // namespace b2
