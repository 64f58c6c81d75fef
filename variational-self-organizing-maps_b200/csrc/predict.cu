// predict.cu — vsom_predict_columns: the BMU of every row over a subset S of the columns, and that node's mean and sigma at the
// other columns Q as the prediction.
//
// The search is the scoring dispatcher (score_rows: K2's tiers + the exact scan K3) on a compacted operand: the columns S of the mean
// plane, gathered once per call into an N x |S| plane padded to a multiple of 4 like the context's own, and the columns S of the rows.
// Device rows are gathered once into an n x |S| buffer; host rows cross PCIe full width in the dispatcher's slabs and are gathered
// per slab on the device (ScanMap::cols).  So the results are, bit for bit, those of vsom_find_bmu_exact on a Standard context whose
// mean plane is the compacted one.  A fill behind each row's final BMU copies mean / sigma at Q from the context's own planes.
#include "common.cuh"

#include <algorithm>

namespace vsom
{

// dst[r * dstStride + j] = src[r * srcStride + cols[j]] for j < m, 0 for m <= j < dstStride: one warp per row, lanes over the columns
// (the writes coalesce; the reads stay inside the row)
__global__ void gather_columns_kernel(const float *__restrict__ src, long long rows, long long srcStride, const int *__restrict__ cols, int m, int dstStride,
                                      float *__restrict__ dst)
{
    const int lane = threadIdx.x & 31;
    const long long warps = static_cast<long long>(gridDim.x) * (blockDim.x >> 5);
    for (long long r = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5); r < rows; r += warps)
    {
        const float *s = src + r * srcStride;
        float *d = dst + r * dstStride;
        for (int j = lane; j < dstStride; j += 32)
            d[j] = j < m ? s[__ldg(cols + j)] : 0.0f;
    }
}

// mean / sigma (either may be null) of row r's BMU at the columns q[0 .. nq): out[r * nq + j] = plane[bmu[r] * rowStride + q[j]]
__global__ void predict_fill_kernel(const unsigned *__restrict__ bmu, long long rows, const float *__restrict__ mean, const float *__restrict__ sigma, int rowStride,
                                    const int *__restrict__ q, int nq, float *__restrict__ outMean, float *__restrict__ outSigma)
{
    const int lane = threadIdx.x & 31;
    const long long warps = static_cast<long long>(gridDim.x) * (blockDim.x >> 5);
    for (long long r = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5); r < rows; r += warps)
    {
        const size_t node = static_cast<size_t>(__ldg(bmu + r)) * static_cast<size_t>(rowStride);
        for (int j = lane; j < nq; j += 32)
        {
            const int c = __ldg(q + j);
            if (outMean)
                outMean[r * nq + j] = mean[node + c];
            if (outSigma)
                outSigma[r * nq + j] = sigma[node + c];
        }
    }
}

// warps of 256-thread CTAs, one per row, with a grid of at most a few waves (the kernels loop over the rest)
static unsigned row_warp_grid(const vsom_ctx *ctx, size_t rows)
{
    return static_cast<unsigned>(std::min<size_t>((rows + 7) / 8, static_cast<size_t>(ctx->numSMs) * 16));
}

int launch_gather_columns(vsom_ctx *ctx, const float *src, size_t rows, size_t srcStride, const int *colsDev, int m, int outStride, float *outDev, cudaStream_t stream)
{
    if (rows == 0)
        return VSOM_OK;
    gather_columns_kernel<<<row_warp_grid(ctx, rows), 256, 0, stream>>>(src, static_cast<long long>(rows), static_cast<long long>(srcStride), colsDev, m, outStride,
                                                                        outDev);
    ctx->launches += 1;
    VSOM_CUDA(ctx, cudaGetLastError());
    return VSOM_OK;
}

int launch_predict_fill(vsom_ctx *ctx, const unsigned *bmuDev, size_t rows, const ScoreOut &out, bool toStaging, cudaStream_t stream)
{
    if (rows == 0 || out.q == 0)
        return VSOM_OK;
    float *m = toStaging ? (out.mean ? out.meanDev : nullptr) : out.mean;
    float *s = toStaging ? (out.sigma ? out.sigmaDev : nullptr) : out.sigma;
    if (!m && !s)
        return VSOM_OK;
    predict_fill_kernel<<<row_warp_grid(ctx, rows), 256, 0, stream>>>(bmuDev, static_cast<long long>(rows), ctx->mean, ctx->sigma, ctx->rowStride, out.predCols, out.q, m,
                                                                      s);
    ctx->launches += 1;
    VSOM_CUDA(ctx, cudaGetLastError());
    return VSOM_OK;
}

// The call after its argument checks (capi.cu): match[Dm] is 0 / 1 with at least one 1; the context is an unsharded Standard / Median
// one.  `out` holds the caller's bmu / dist / mean / sigma (device memory when !hostRows).  stage slots: 10 = compacted plane and the
// two column lists, 11 = compacted device rows (host rows: the dispatcher's gathered slabs), 12 = BMUs of device rows when the
// caller wants none (host rows: the dispatcher's slab staging of the predicted columns).
int predict_columns(vsom_ctx *ctx, const float *x, bool hostRows, size_t n, const uint8_t *match, uint64_t minHits, const ScoreOut &out)
{
    const int Dm = ctx->Dm, N = ctx->N;
    std::vector<int> cols; // S, then Q
    cols.reserve(Dm);
    for (int j = 0; j < Dm; ++j)
        if (match[j])
            cols.push_back(j);
    const int m = static_cast<int>(cols.size()), q = Dm - m;
    for (int j = 0; j < Dm; ++j)
        if (!match[j])
            cols.push_back(j);
    const int planeStride = (m + 3) & ~3;
    const size_t planeBytes = sizeof(float) * static_cast<size_t>(N) * planeStride;
    int rc = stage_reserve(ctx, 10, planeBytes + sizeof(int) * Dm);
    if (rc)
        return rc;
    float *plane = static_cast<float *>(ctx->stage[10]);
    int *colsDev = reinterpret_cast<int *>(static_cast<unsigned char *>(ctx->stage[10]) + planeBytes);
    VSOM_CUDA(ctx, cudaMemcpyAsync(colsDev, cols.data(), sizeof(int) * Dm, cudaMemcpyHostToDevice, ctx->stream));
    rc = launch_gather_columns(ctx, ctx->mean, N, ctx->rowStride, colsDev, m, planeStride, plane, ctx->stream);
    if (rc)
        return rc;

    // the compacted map: a Standard operand of m columns (Median shares the Comparer), the context's hits
    ScanMap map;
    map.mean = plane;
    map.hits = ctx->hits;
    map.N = N;
    map.rowStride = planeStride;
    map.transform = VSOM_STANDARD;
    map.Din = m;
    map.Dr = m;
    ScoreOut o = out;
    o.predCols = colsDev + m;
    o.q = q;
    const bool fill = q != 0 && (out.mean || out.sigma);
    const float *rows = x;
    if (hostRows)
    {
        map.cols = colsDev;
        map.srcDin = ctx->Din;
    }
    else
    {
        if (n)
        {
            rc = stage_reserve(ctx, 11, sizeof(float) * n * m);
            if (rc)
                return rc;
            float *xc = static_cast<float *>(ctx->stage[11]);
            rc = launch_gather_columns(ctx, x, n, ctx->Din, colsDev, m, m, xc, ctx->stream);
            if (rc)
                return rc;
            rows = xc;
        }
        if (fill && !o.bmu && n)
        {
            rc = stage_reserve(ctx, 12, sizeof(unsigned) * n);
            if (rc)
                return rc;
            o.bmu = static_cast<unsigned *>(ctx->stage[12]);
        }
    }
    rc = score_rows(ctx, rows, hostRows, n, minHits, true, o, nullptr, map);
    if (rc)
        return rc;
    if (hostRows) // the tensor-core path's result copies run on its re-scoring stream; tc_finish joined it to the context's stream
        VSOM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return VSOM_OK;
}

} // namespace vsom
