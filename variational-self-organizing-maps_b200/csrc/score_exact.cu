// score_exact.cu — K3: exact batch BMU search in the reference's own arithmetic.
//
// Replaces the row loops of Som::evaluate (src/Som.cpp:503-520) / Som::measureSimilarity (:641-711) and any
// per-row Som::findBmu (:291-309) / Som::findRestrictedBmu (:313-332) over a loaded DataSet chunk:
// for every row, argmin over nodes of Som::euclidianWeightedDist (:124-141) with the strict '<',
// lowest-index-wins rule, and the f32 distance itself, summed k = 0,1,2,... like `comparer.dot(comparer)`.
//
// Each (row, node) pair is one sequential f32 chain owned by one thread, so every distance is bit-identical
// to the reference; the parallelism is over pairs (a 64 x 64 pair tile per CTA, 4 x 4 chains per thread,
// operands staged through shared memory in 32-wide slices of the model vector).  This is the exact path:
// it is what the tensor-core candidate search (score_tc.cu) rescoring falls back to, and it is the scorer
// for small / medium batches.
//
// VSOM_ORDER_EIGEN_SSE (the order of dot() under real Eigen, common.cuh): a pair is EIGHT interleaved chains, owned by
// eight consecutive lanes (find_bmu_exact_eigen_kernel): lane c sums the terms k = c mod 8, the lanes combine with the
// fixed butterfly xor 4 (res0 + res1), [+ the extra packet], xor 2, xor 1 ((p0 + p2) + (p1 + p3); float addition
// commutes, so every lane ends with the same bits), then the scalar tail.
#include "common.cuh"

#include <algorithm>

namespace vsom
{

constexpr int RT = 64, NT = 64, KC = 32, kScoreThreads = 256;

template <int TR, int TOP>
__global__ void __launch_bounds__(kScoreThreads) find_bmu_exact_kernel(const float *__restrict__ x, u64 nIn, const unsigned *__restrict__ rowList,
 const unsigned *__restrict__ rowCount, const float *__restrict__ mean,
                                                                       const u64 *__restrict__ hits, u64 minHits, int N, int Din, int Dr, int P,
                                                                       int rowStride, const unsigned short *__restrict__ pairI,
                                                                       const unsigned short *__restrict__ pairJ, unsigned *__restrict__ outBmu,
                                                                       float *__restrict__ outDist, int splits, u64 *__restrict__ keyBuf,
                                                                       unsigned *__restrict__ outBmu2, float *__restrict__ outDist2)
{
    __shared__ float xa[RT][KC + 1];
    __shared__ float ma[NT][KC + 1];
    __shared__ float xb[TR == VSOM_CLR ? RT : 1][KC + 1];
    __shared__ float mb[TR == VSOM_CLR ? NT : 1][KC + 1];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tx = tid & 15, ty = tid >> 4; // nodes tx + 16 j, rows ty + 16 i
    // List mode (the rows a tensor-core slab could not certify): item i is row rowList[i], the count lives on the device, and a
    // fixed grid walks (row tile, node split) work items — few rows must not mean few CTAs with the whole map each; the splits
    // of a row meet in keyBuf[item] by atomic min of the (distance, node) key, written out by finalize_list_kernel.
    const bool listMode = rowList != nullptr;
    const u64 n = listMode ? static_cast<u64>(*rowCount) : nIn;
    const u64 rowTiles = (n + RT - 1) / RT, nWork = listMode ? rowTiles * static_cast<u64>(splits) : rowTiles;
    auto src_row = [&](u64 item) -> u64 { return listMode ? static_cast<u64>(rowList[item]) : item; };
    const int nodeTilesTotal = (N + NT - 1) / NT, tilesPerSplit = listMode ? (nodeTilesTotal + splits - 1) / splits : nodeTilesTotal;
  for (u64 w = blockIdx.x; w < nWork; w += gridDim.x)
  {
    const u64 row0 = (listMode ? w / static_cast<u64>(splits) : w) * RT;
    const int split = listMode ? static_cast<int>(w % static_cast<u64>(splits)) : 0;
    const int nodeLo = split * tilesPerSplit * NT, nodeHi = min(N, nodeLo + tilesPerSplit * NT);

    u64 best[4], second[TOP == 2 ? 4 : 1]; // TOP = 2: the runner-up keys as well (vsom_find_bmu2)
#pragma unroll
    for (int i = 0; i < 4; ++i)
        best[i] = ~0ull;
    if (TOP == 2)
#pragma unroll
        for (int i = 0; i < 4; ++i)
            second[i] = ~0ull;

    for (int node0 = nodeLo; node0 < nodeHi; node0 += NT)
    {
        float acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j)
                acc[i][j] = 0.0f;

        for (int k0 = 0; k0 < Dr; k0 += KC)
        {
            __syncthreads(); // previous slice fully consumed
            const int k = k0 + lane;
            // stage the slice: one warp per row / node, lanes along k (128-byte coalesced segments)
            for (int r = warp; r < RT; r += kScoreThreads / 32)
            {
                const u64 item = row0 + r;
                float a = 0.0f, bq = 0.0f;
                if (item < n && k < Dr)
                {
                    const u64 row = src_row(item);
                    if (TR != VSOM_CLR)
                        a = x[row * Din + k];
                    else
                    {
                        a = x[row * Din + pairI[k]];
                        bq = x[row * Din + pairJ[k]];
                    }
                }
                xa[r][lane] = a;
                if (TR == VSOM_CLR)
                    xb[r][lane] = bq;
            }
            for (int r = warp; r < NT; r += kScoreThreads / 32)
            {
                const int node = node0 + r;
                float a = 0.0f, bq = 0.0f;
                if (node < N && k < Dr)
                {
                    a = mean[static_cast<size_t>(node) * rowStride + k];
                    if (TR == VSOM_CLR)
                        bq = mean[static_cast<size_t>(node) * rowStride + P + k];
                }
                ma[r][lane] = a;
                if (TR == VSOM_CLR)
                    mb[r][lane] = bq;
            }
            __syncthreads();
            // padded entries are all-zero on both sides: their residual is +0 and s + 0 == s exactly.
#pragma unroll 4
            for (int kk = 0; kk < KC; ++kk)
            {
                float xv[4], mv[4], yv[4], bv[4];
#pragma unroll
                for (int i = 0; i < 4; ++i)
                {
                    xv[i] = xa[ty + 16 * i][kk];
                    mv[i] = ma[tx + 16 * i][kk];
                    if (TR == VSOM_CLR)
                    {
                        yv[i] = xb[ty + 16 * i][kk];
                        bv[i] = mb[tx + 16 * i][kk];
                    }
                }
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                    {
                        float r;
                        if (TR != VSOM_CLR)
                            r = __fsub_rn(mv[j], xv[i]);
                        else
                            r = __fsub_rn(__fadd_rn(__fmul_rn(mv[j], xv[i]), bv[j]), yv[i]);
                        acc[i][j] = __fadd_rn(acc[i][j], __fmul_rn(r, r));
                    }
            }
        }
        // fold this node tile into the running min of each row (node 0 seeds regardless of its hit count)
#pragma unroll
        for (int j = 0; j < 4; ++j)
        {
            const int node = node0 + tx + 16 * j;
            if (node < N && restricted_eligible(node, hits, minHits))
            {
#pragma unroll
                for (int i = 0; i < 4; ++i)
                {
                    const float d = acc[i][j];
                    if (TOP == 2)
                        key_top2_insert(best[i], second[i], score_key(d, static_cast<unsigned>(node)));
                    else
                        best[i] = u64_min(best[i], score_key(d, static_cast<unsigned>(node)));
                }
            }
        }
    }
    // the 16 threads sharing a row sit in one half-warp: xor offsets 8,4,2,1 stay inside it
#pragma unroll
    for (int i = 0; i < 4; ++i)
    {
        u64 k = best[i], k2 = TOP == 2 ? second[i] : ~0ull;
#pragma unroll
        for (int o = 8; o; o >>= 1)
            if (TOP == 2)
                key_top2_merge(k, k2, __shfl_xor_sync(0xffffffffu, k, o), __shfl_xor_sync(0xffffffffu, k2, o));
            else
                k = u64_min(k, __shfl_xor_sync(0xffffffffu, k, o));
        const u64 item = row0 + ty + 16 * i;
        if (tx == 0 && item < n)
        {
            if (listMode)
                list_key_store<TOP>(keyBuf + TOP * item, k, k2);
            else
                store_row_outputs<TOP>(outBmu, outDist, outBmu2, outDist2, item, k, k2);
        }
    }
    __syncthreads(); // the staging arrays are reused by the next work item
  }
}

// ---------------------------------------------------------------------------------------- Eigen SSE2 order
constexpr int ER = 32, EN = 32, EMS = 40; // rows / nodes per CTA tile; row stride of the node slice (bank = 8 gx + c: conflict-free)

template <int TR, int TOP>
__global__ void __launch_bounds__(kScoreThreads) find_bmu_exact_eigen_kernel(const float *__restrict__ x, u64 nIn, const unsigned *__restrict__ rowList,
 const unsigned *__restrict__ rowCount, const float *__restrict__ mean,
                                                                             const u64 *__restrict__ hits, u64 minHits, int N, int Din, int Dr, int P,
                                                                             int rowStride, const unsigned short *__restrict__ pairI,
                                                                             const unsigned short *__restrict__ pairJ, unsigned *__restrict__ outBmu,
                                                                             float *__restrict__ outDist, int splits, u64 *__restrict__ keyBuf,
                                                                             unsigned *__restrict__ outBmu2, float *__restrict__ outDist2)
{
    constexpr bool kClr = TR == VSOM_CLR;
    __shared__ float xa[ER][KC + 1], ma[EN][EMS];
    __shared__ float xb[kClr ? ER : 1][KC + 1], mb[kClr ? EN : 1][EMS];
    __shared__ float xr[ER][8], mr[EN][8];                       // the Dr % 8 elements behind the full blocks of eight
    __shared__ float xrb[kClr ? ER : 1][8], mrb[kClr ? EN : 1][8];
    __shared__ u64 sBest[ER][8];
    __shared__ u64 sSecond[TOP == 2 ? ER : 1][8];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int c = tid & 7, g = tid >> 3, gx = g & 7, gy = g >> 3; // chain; nodes gx + 8 j (j < 4), rows gy + 4 i (i < 8)
    const int n8 = Dr & ~7, nrest = Dr - n8;
    const bool listMode = rowList != nullptr; // see find_bmu_exact_kernel
    const u64 n = listMode ? static_cast<u64>(*rowCount) : nIn;
    const u64 rowTiles = (n + ER - 1) / ER, nWork = listMode ? rowTiles * static_cast<u64>(splits) : rowTiles;
    const int nodeTilesTotal = (N + EN - 1) / EN, tilesPerSplit = listMode ? (nodeTilesTotal + splits - 1) / splits : nodeTilesTotal;
  for (u64 w = blockIdx.x; w < nWork; w += gridDim.x)
  {
    const u64 row0 = (listMode ? w / static_cast<u64>(splits) : w) * ER;
    const int split = listMode ? static_cast<int>(w % static_cast<u64>(splits)) : 0;
    const int nodeLo = split * tilesPerSplit * EN, nodeHi = min(N, nodeLo + tilesPerSplit * EN);

    u64 best[8], second[TOP == 2 ? 8 : 1];
#pragma unroll
    for (int i = 0; i < 8; ++i)
        best[i] = ~0ull;
    if (TOP == 2)
#pragma unroll
        for (int i = 0; i < 8; ++i)
            second[i] = ~0ull;

    auto term = [&](float xv, float yv, float mv, float bv) {
        const float r = kClr ? __fsub_rn(__fadd_rn(__fmul_rn(mv, xv), bv), yv) : __fsub_rn(mv, xv);
        return __fmul_rn(r, r);
    };
    // one element of a row / node (0 outside): what the slices and the rest arrays hold
    auto load_x = [&](u64 item, int k, float &a, float &bq) {
        a = 0.0f;
        bq = 0.0f;
        if (item < n && k < Dr)
        {
            const u64 row = listMode ? static_cast<u64>(rowList[item]) : item;
            if (!kClr)
                a = x[row * Din + k];
            else
            {
                a = x[row * Din + pairI[k]];
                bq = x[row * Din + pairJ[k]];
            }
        }
    };
    auto load_m = [&](int node, int k, float &a, float &bq) {
        a = 0.0f;
        bq = 0.0f;
        if (node < N && k < Dr)
        {
            a = mean[static_cast<size_t>(node) * rowStride + k];
            if (kClr)
                bq = mean[static_cast<size_t>(node) * rowStride + P + k];
        }
    };
    __syncthreads(); // (list mode) the previous work item's readers of xr are done
    {
        const int r = tid >> 3, e = tid & 7; // 32 rows x 8 rest elements
        float a, bq;
        load_x(row0 + r, e < nrest ? n8 + e : Dr, a, bq);
        xr[r][e] = a;
        if (kClr)
            xrb[r][e] = bq;
    }
    for (int node0 = nodeLo; node0 < nodeHi; node0 += EN)
    {
        float acc[8][4];
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j)
                acc[i][j] = 0.0f;
        __syncthreads(); // the previous node tile's rest elements are no longer read
        {
            const int r = tid >> 3, e = tid & 7;
            float a, bq;
            load_m(node0 + r, e < nrest ? n8 + e : Dr, a, bq);
            mr[r][e] = a;
            if (kClr)
                mrb[r][e] = bq;
        }
        for (int k0 = 0; k0 < n8; k0 += KC)
        {
            __syncthreads(); // previous slice fully consumed
            const int k = k0 + lane, kk = k < n8 ? k : Dr; // beyond the full blocks: zeros on both sides (term +0)
            for (int r = warp; r < ER; r += kScoreThreads / 32)
            {
                float a, bq;
                load_x(row0 + r, kk, a, bq);
                xa[r][lane] = a;
                if (kClr)
                    xb[r][lane] = bq;
                load_m(node0 + r, kk, a, bq);
                ma[r][lane] = a;
                if (kClr)
                    mb[r][lane] = bq;
            }
            __syncthreads();
#pragma unroll
            for (int s = 0; s < KC / 8; ++s)
            {
                const int q = c + 8 * s;
                float xv[8], yv[8], mv[4], bv[4];
#pragma unroll
                for (int i = 0; i < 8; ++i)
                {
                    xv[i] = xa[gy + 4 * i][q];
                    yv[i] = kClr ? xb[gy + 4 * i][q] : 0.0f;
                }
#pragma unroll
                for (int j = 0; j < 4; ++j)
                {
                    mv[j] = ma[gx + 8 * j][q];
                    bv[j] = kClr ? mb[gx + 8 * j][q] : 0.0f;
                }
#pragma unroll
                for (int i = 0; i < 8; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        acc[i][j] = __fadd_rn(acc[i][j], term(xv[i], yv[i], mv[j], bv[j]));
            }
        }
        __syncthreads(); // mr / xr visible (also when there was no full block)
#pragma unroll
        for (int j = 0; j < 4; ++j)
        {
            const int node = node0 + gx + 8 * j;
            const bool eligible = node < N && restricted_eligible(node, hits, minHits);
#pragma unroll
            for (int i = 0; i < 8; ++i)
            {
                const int r = gy + 4 * i, nl = gx + 8 * j;
                float v = __fadd_rn(acc[i][j], __shfl_xor_sync(0xffffffffu, acc[i][j], 4)); // packet_res0 + packet_res1, lane by lane
                int e = 0;
                if (nrest >= 4)
                {
                    const int q = c & 3; // the extra packet
                    v = __fadd_rn(v, term(xr[r][q], kClr ? xrb[r][q] : 0.0f, mr[nl][q], kClr ? mrb[nl][q] : 0.0f));
                    e = 4;
                }
                v = __fadd_rn(v, __shfl_xor_sync(0xffffffffu, v, 2)); // p0 + p2 | p1 + p3
                v = __fadd_rn(v, __shfl_xor_sync(0xffffffffu, v, 1)); // (p0 + p2) + (p1 + p3)
                for (; e < nrest; ++e)                                // scalar tail
                    v = __fadd_rn(v, term(xr[r][e], kClr ? xrb[r][e] : 0.0f, mr[nl][e], kClr ? mrb[nl][e] : 0.0f));
                if (eligible)
                {
                    if (TOP == 2)
                        key_top2_insert(best[i], second[i], score_key(v, static_cast<unsigned>(node)));
                    else
                        best[i] = u64_min(best[i], score_key(v, static_cast<unsigned>(node)));
                }
            }
        }
    }
    if (c == 0)
#pragma unroll
        for (int i = 0; i < 8; ++i)
        {
            sBest[gy + 4 * i][gx] = best[i];
            if (TOP == 2)
                sSecond[gy + 4 * i][gx] = second[i];
        }
    __syncthreads();
    if (tid < ER && row0 + tid < n)
    {
        u64 k = sBest[tid][0], k2 = TOP == 2 ? sSecond[tid][0] : ~0ull;
#pragma unroll
        for (int q = 1; q < 8; ++q)
            if (TOP == 2)
                key_top2_merge(k, k2, sBest[tid][q], sSecond[tid][q]);
            else
                k = u64_min(k, sBest[tid][q]);
        const u64 item = row0 + tid;
        if (listMode)
            list_key_store<TOP>(keyBuf + TOP * item, k, k2);
        else
            store_row_outputs<TOP>(outBmu, outDist, outBmu2, outDist2, item, k, k2);
    }
    __syncthreads(); // sBest and the staging arrays are reused by the next work item
  }
}

// list mode: keys of the work items' splits (TOP per listed row, list_key_store) -> outputs of the listed rows
template <int TOP>
__global__ void finalize_list_kernel(const unsigned *__restrict__ rowList, const unsigned *__restrict__ rowCount, const u64 *__restrict__ keyBuf,
                                     unsigned *__restrict__ outBmu, float *__restrict__ outDist, unsigned *__restrict__ outBmu2, float *__restrict__ outDist2)
{
    const unsigned n = *rowCount;
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    {
        const u64 *k = keyBuf + TOP * static_cast<size_t>(i);
        const u64 k1 = k[0];
        store_row_outputs<TOP>(outBmu, outDist, outBmu2, outDist2, rowList[i], k1, TOP == 2 ? k[1] : k1);
    }
}

template <int TR>
__global__ void all_dists_kernel(const float *__restrict__ v, const float *__restrict__ mean, int N, int Dr, int P, int rowStride,
                                 const unsigned short *__restrict__ pairI, const unsigned short *__restrict__ pairJ, int order, double *__restrict__ out)
{
    const int node = blockIdx.x * blockDim.x + threadIdx.x;
    if (node >= N)
        return;
    out[node] = static_cast<double>(dist_ordered<TR>(mean + static_cast<size_t>(node) * rowStride, v, Dr, P, pairI, pairJ, order));
}

// ---------------------------------------------------------------------------------------- soft assignment
// Som::findRestrictedBmd (src/Som.cpp:457-487) for a batch of rows: p_i = exp(-d_i * d_i / 2) of the (already squared)
// distance for nodes with hits >= minHits, 0 otherwise, normalised by their sum.  One thread per (row, node) for the
// distances (exact f32 chain in the context's order) and exp in f64; then one thread per row adds the N terms in node
// order like the reference's loop (the f64 sum is order dependent) and the row is scaled.
template <int TR>
__global__ void soft_assign_terms_kernel(const float *__restrict__ x, u64 n, const float *__restrict__ mean, const u64 *__restrict__ hits, u64 minHits, int N,
                                         int Din, int Dr, int P, int rowStride, const unsigned short *__restrict__ pairI, const unsigned short *__restrict__ pairJ,
                                         int order, double *__restrict__ out)
{
    const int node = blockIdx.x * blockDim.x + threadIdx.x;
    const u64 row = blockIdx.y;
    if (node >= N || row >= n)
        return;
    double pr = 0.0;
    if (hits[node] >= minHits) // not restricted_eligible: findRestrictedBmd has no node-0 seed
    {
        const double d = static_cast<double>(dist_ordered<TR>(mean + static_cast<size_t>(node) * rowStride, x + row * Din, Dr, P, pairI, pairJ, order));
        pr = exp(__ddiv_rn(__dmul_rn(-d, d), 2.0));
    }
    out[row * N + node] = pr;
}

__global__ void soft_assign_norm_kernel(u64 n, int N, double *__restrict__ prob, double *__restrict__ sums)
{
    __shared__ double C;
    const u64 row = blockIdx.x;
    if (row >= n)
        return;
    double *pr = prob + row * N;
    if (threadIdx.x == 0)
    {
        double c = 0.0;
        for (int i = 0; i < N; ++i)
            c = __dadd_rn(c, pr[i]);
        C = c;
        sums[row] = c;
    }
    __syncthreads();
    const double c = C;
    for (int i = threadIdx.x; i < N; i += blockDim.x)
        pr[i] = __ddiv_rn(pr[i], c);
}

int launch_soft_assign(vsom_ctx *ctx, const float *xDev, size_t n, uint64_t minHits, double *probDev, double *sumsDev)
{
    if (n == 0)
        return VSOM_OK;
    // one grid row per data row: gridDim.y is at most 65 535, so longer batches take several launches
    for (size_t r0 = 0; r0 < n; r0 += kMaxGridY)
    {
        const size_t rows = std::min(n - r0, kMaxGridY);
        const float *xs = xDev + r0 * ctx->Din;
        double *out = probDev + r0 * ctx->N;
        dim3 grid((ctx->N + 127) / 128, static_cast<unsigned>(rows));
        if (ctx->transform == VSOM_CLR)
            soft_assign_terms_kernel<VSOM_CLR><<<grid, 128, 0, ctx->stream>>>(xs, rows, ctx->mean, ctx->hits, minHits, ctx->N, ctx->Din, ctx->Dr, ctx->P, ctx->rowStride, ctx->pairI,
                                                                              ctx->pairJ, ctx->order, out);
        else
            soft_assign_terms_kernel<VSOM_STANDARD><<<grid, 128, 0, ctx->stream>>>(xs, rows, ctx->mean, ctx->hits, minHits, ctx->N, ctx->Din, ctx->Dr, ctx->P, ctx->rowStride,
                                                                                   ctx->pairI, ctx->pairJ, ctx->order, out);
        ctx->launches += 1;
    }
    soft_assign_norm_kernel<<<static_cast<unsigned>(n), 256, 0, ctx->stream>>>(n, ctx->N, probDev, sumsDev);
    VSOM_CUDA(ctx, cudaGetLastError());
    ctx->launches += 1;
    return VSOM_OK;
}

// rowListDev == null: rows 0 .. n-1 of xDev.  Otherwise the rows rowListDev[0 .. *rowCountDev) (at most n of them) — the exact
// scan of the rows a tensor-core slab could not certify, the count staying on the device; keyBufDev: out.top * n u64 of scratch.
// out.top = 2: the runner-up of every row as well.
int launch_find_bmu_list(vsom_ctx *ctx, const float *xDev, size_t n, const unsigned *rowListDev, const unsigned *rowCountDev, uint64_t minHits, const ScoreOut &out,
                         cudaStream_t stream, u64 *keyBufDev, const ScanMap &map)
{
    if (n == 0)
        return VSOM_OK;
    const bool list = rowListDev != nullptr;
    const bool eigen = ctx->order == VSOM_ORDER_EIGEN_SSE;
    const int tileRows = eigen ? ER : RT, tileNodes = eigen ? EN : NT;
    // list mode: a fixed grid (a few CTAs per SM) walks (row tile, node split) work items; 32 splits of the node range
    const int nodeTiles = (map.N + tileNodes - 1) / tileNodes, splits = list ? std::max(1, std::min(32, nodeTiles)) : 1;
    const unsigned grid = list ? static_cast<unsigned>(std::min<size_t>((n + tileRows - 1) / tileRows * splits, static_cast<size_t>(ctx->numSMs) * 4))
                               : static_cast<unsigned>((n + tileRows - 1) / tileRows);
    if (list)
        VSOM_CUDA(ctx, cudaMemsetAsync(keyBufDev, 0xff, sizeof(u64) * n * (out.top == 2 ? 2 : 1), stream));
#define VSOM_SCORE_ARGS xDev, n, rowListDev, rowCountDev, map.mean, map.hits, minHits, map.N, map.Din, map.Dr, map.P, map.rowStride, ctx->pairI, ctx->pairJ, out.bmu, out.dist, splits, keyBufDev, out.bmu2, out.dist2
#define VSOM_SCORE_LAUNCH(TOP)                                                                                                   \
    if (eigen)                                                                                                                   \
    {                                                                                                                            \
        if (map.transform == VSOM_CLR)                                                                                           \
            find_bmu_exact_eigen_kernel<VSOM_CLR, TOP><<<grid, kScoreThreads, 0, stream>>>(VSOM_SCORE_ARGS);                    \
        else                                                                                                                     \
            find_bmu_exact_eigen_kernel<VSOM_STANDARD, TOP><<<grid, kScoreThreads, 0, stream>>>(VSOM_SCORE_ARGS);               \
    }                                                                                                                            \
    else if (map.transform == VSOM_CLR)                                                                                          \
        find_bmu_exact_kernel<VSOM_CLR, TOP><<<grid, kScoreThreads, 0, stream>>>(VSOM_SCORE_ARGS);                              \
    else /* Standard and Median share the Comparer (src/Transformation.cpp:7-8, :45-46) */                                       \
        find_bmu_exact_kernel<VSOM_STANDARD, TOP><<<grid, kScoreThreads, 0, stream>>>(VSOM_SCORE_ARGS);
    if (out.top == 2)
    {
        VSOM_SCORE_LAUNCH(2)
    }
    else
    {
        VSOM_SCORE_LAUNCH(1)
    }
#undef VSOM_SCORE_LAUNCH
#undef VSOM_SCORE_ARGS
    ctx->launches += 1;
    if (list)
    {
        const unsigned fgrid = std::min(1024u, static_cast<unsigned>((n + 255) / 256));
        if (out.top == 2)
            finalize_list_kernel<2><<<fgrid, 256, 0, stream>>>(rowListDev, rowCountDev, keyBufDev, out.bmu, out.dist, out.bmu2, out.dist2);
        else
            finalize_list_kernel<1><<<fgrid, 256, 0, stream>>>(rowListDev, rowCountDev, keyBufDev, out.bmu, out.dist, out.bmu2, out.dist2);
        ctx->launches += 1;
    }
    VSOM_CUDA(ctx, cudaGetLastError());
    return VSOM_OK;
}

// ---- Som::measureSimilarity's per-row pass (src/Som.cpp:631-714): delta_n = ((v_n - m_n) / sM_n) / numOfSigmas against the row's BMU,
// sM = the reference's capped sigma (:648: sigma > 1e-5 -> 1e-5).  The reference keeps a running "largest delta" over all rows and
// columns; once that value is >= 0 (after its first update) a row can only raise it to the row's own maximum, so the device returns
// max_n delta_n per row (NaN never wins a `>`; -inf when every delta is NaN) and the host replays the scan over rows.
// One warp per row; the three IEEE operations are the reference's (fsub, fdiv, fdiv).
__global__ void __launch_bounds__(256) similarity_rowmax_kernel(const float *__restrict__ x, u64 rows, int D, const float *__restrict__ mean, const float *__restrict__ sigma,
                                                                int rowStride, const unsigned *__restrict__ bmu, float k, float *__restrict__ out)
{
    const u64 row = static_cast<u64>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows)
        return;
    const float *v = x + row * D;
    const size_t at = static_cast<size_t>(bmu[row]) * rowStride;
    const float *m = mean + at, *sg = sigma + at;
    float mx = __int_as_float(0xff800000); // -inf
    for (int d = lane; d < D; d += 32)
    {
        const float s = sg[d], sM = s > 0.00001f ? 0.00001f : s;
        const float delta = __fdiv_rn(__fdiv_rn(__fsub_rn(v[d], m[d]), sM), k);
        if (delta > mx)
            mx = delta;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
    {
        const float other = __shfl_xor_sync(0xffffffffu, mx, o);
        if (other > mx)
            mx = other;
    }
    if (lane == 0)
        out[row] = mx;
}

int launch_similarity_rowmax(vsom_ctx *ctx, const float *xDev, size_t rows, const unsigned *bmuDev, float k, float *outDev, cudaStream_t stream)
{
    if (rows == 0)
        return VSOM_OK;
    similarity_rowmax_kernel<<<static_cast<unsigned>((rows + 7) / 8), 256, 0, stream>>>(xDev, rows, ctx->Din, ctx->mean, ctx->sigma, ctx->rowStride, bmuDev, k, outDev);
    ctx->launches += 1;
    VSOM_CUDA(ctx, cudaGetLastError());
    return VSOM_OK;
}

int launch_all_dists(vsom_ctx *ctx, const float *vDev, double *outDev)
{
    const int threads = 128, grid = (ctx->N + threads - 1) / threads;
    if (ctx->transform == VSOM_CLR)
        all_dists_kernel<VSOM_CLR><<<grid, threads, 0, ctx->stream>>>(vDev, ctx->mean, ctx->N, ctx->Dr, ctx->P, ctx->rowStride, ctx->pairI, ctx->pairJ, ctx->order, outDev);
    else
        all_dists_kernel<VSOM_STANDARD><<<grid, threads, 0, ctx->stream>>>(vDev, ctx->mean, ctx->N, ctx->Dr, ctx->P, ctx->rowStride, ctx->pairI, ctx->pairJ, ctx->order, outDev);
    VSOM_CUDA(ctx, cudaGetLastError());
    ctx->launches += 1;
    return VSOM_OK;
}

} // namespace vsom
