// batch_map.cu — K6: one chunk-epoch of the batch-map trainer (a "next" row of the scope table, SURVEY.md §8f-1).
//
// Replaces Som::trainBatchSomEpoch (src/Som.cpp:756-879), in the order the reference has when its parallel algorithms
// run on the sequential backend (rows in order, neurons independent):
//   phase A  per row: BMU — global on the first epoch (findBmu, :771), the greedy local walk from the row's lastBMU
//            afterwards (findLocalBmu, :793) — hit count and squared residual;
//   phase B  per neuron: West/Finch incremental weighted mean and variance over ALL rows of the chunk in row order,
//            weights = neighbourhood of the row's BMU evaluated with the reference's SomIndex(map, index) coordinates
//            (which divide by the map HEIGHT, src/SomIndex.cpp:15-18):
//                sumW += w;  delta = Stepper(x, cur);  cur += (w / sumW) * delta;  S += (w * delta) * delta
//            then map = cur, sigmaMap = sqrt(S / sumW), weightMap = sumW  (:871-875).
// Every (neuron, component) pair is a strictly sequential f32 chain over the rows, so the result is bit-identical to
// the reference; the parallelism is over chains: a CTA owns a few neurons, streams the rows through shared memory in
// batches, one warp turns (row, neuron) into the two coefficients w and w / sumW (one IEEE division per pair instead of
// one per chain) a batch ahead, and the other threads advance their chains (4-8 per thread, in registers).
#include "common.cuh"

#include <algorithm>

namespace vsom
{

constexpr int BM_ROWS = 32;   // rows per shared-memory batch at most
constexpr int BM_LUT_SMEM = 4096; // neighbourhood tables up to this many entries are kept in shared memory
constexpr int BM_MAXNB = 8;   // neurons per CTA at most

// reference coordinates of a linear index: SomIndex(const Som&, index), src/SomIndex.cpp:15-18
__host__ __device__ inline void quirky_xy(unsigned index, int W, int H, int &x, int &y)
{
    x = static_cast<int>(index % static_cast<unsigned>(W));
    y = static_cast<int>((index - index % static_cast<unsigned>(W)) / static_cast<unsigned>(H));
}

__global__ void bmu_xy_kernel(const unsigned *__restrict__ bmu, u64 n, int W, int H, int2 *__restrict__ out)
{
    const u64 j = static_cast<u64>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (j >= n)
        return;
    int x, y;
    quirky_xy(bmu[j], W, H, x, y);
    out[j] = make_int2(x, y);
}

__global__ void hits_add_kernel(const unsigned *__restrict__ bmu, u64 n, u64 *__restrict__ hits)
{
    const u64 j = static_cast<u64>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (j < n)
        atomicAdd(hits + bmu[j], 1ull);
}

// ---- phase A for the later epochs: findLocalBmu (src/Som.cpp:335-454) per row, EIGHT lanes per row (four rows per warp).
// The lanes of a group evaluate the candidate cells' distances (each a sequential f32 chain like the reference — one lane per
// distance is all the parallelism a strict summation order leaves, so a whole warp per row kept 24 lanes idle), every lane of
// the group then replays the reference's comparisons on the shuffled values, so the walk state stays group-uniform.
template <int TR>
__global__ void __launch_bounds__(256) local_bmu_rows_kernel(const float *__restrict__ x, u64 n, const float *__restrict__ mean, int W, int H, int Din,
                                                             int Dr, int P, int rowStride, const unsigned short *__restrict__ pairI,
                                                             const unsigned short *__restrict__ pairJ, int order, const u64 *__restrict__ start,
                                                             unsigned *__restrict__ outBmu, float *__restrict__ outDist)
{
    const u64 row = (static_cast<u64>(blockIdx.x) * blockDim.x + threadIdx.x) >> 3;
    const int lane = threadIdx.x & 7;                              // lane inside the group of eight
    const unsigned gmask = 0xffu << (threadIdx.x & 24);            // the group's lanes inside the warp
    if (row >= n)
        return;
    const float *xr = x + row * Din;
    auto dist = [&](u64 node) { return dist_ordered<TR>(mean + node * rowStride, xr, Dr, P, pairI, pairJ, order); };
    const u64 uW = static_cast<u64>(W), uH = static_cast<u64>(H), M1 = ~0ull;
    const u64 fx[8] = {M1, 0, 1, 1, 1, 0, M1, M1}, fy[8] = {1, 1, 1, 0, M1, M1, M1, 0};
    u64 lastBMU = start ? start[row] : 0ull, minIndex = lastBMU, lastMeasured = lastBMU;
    float minDist = __shfl_sync(gmask, lane == 0 ? dist(lastBMU) : 0.0f, 0, 8);
    for (;;)
    {
        const u64 lmX = lastMeasured % uW, lmY = lastMeasured / uW, lbX = lastBMU % uW;
        if (lastMeasured == lastBMU)
        {
            u64 idx[8];
#pragma unroll
            for (int i = 0; i < 8; ++i)
            {
                const u64 cx = lmX + fx[i] < uW - 1 ? lmX + fx[i] : uW - 1, cy = lmY + fy[i] < uH - 1 ? lmY + fy[i] : uH - 1;
                idx[i] = cy * uW + cx;
            }
            float mine = 0.0f;
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if (lane == i)
                    mine = dist(idx[i]);
#pragma unroll
            for (int i = 0; i < 8; ++i)
            {
                const float v = __shfl_sync(gmask, mine, i, 8);
                if (v < minDist)
                {
                    minDist = v;
                    minIndex = idx[i];
                }
            }
            if (minIndex == lastBMU)
                break;
            lastMeasured = minIndex;
        }
        else
        {
            if (lmX - lbX)
            {
                u64 idx[3];
#pragma unroll
                for (int i = 0; i < 3; ++i)
                {
                    const u64 ox = lmX + lmX - lbX, oy = lmY + static_cast<u64>(static_cast<long long>(i - 1));
                    idx[i] = (oy < uH - 1 ? oy : uH - 1) * uW + (ox < uW - 1 ? ox : uW - 1);
                }
                float mine = 0.0f;
#pragma unroll
                for (int i = 0; i < 3; ++i)
                    if (lane == i)
                        mine = dist(idx[i]);
#pragma unroll
                for (int i = 0; i < 3; ++i)
                {
                    const float v = __shfl_sync(gmask, mine, i, 8);
                    if (v < minDist)
                    {
                        minDist = v;
                        minIndex = idx[i];
                    }
                }
            }
            if (minIndex == lastMeasured)
                break;
            lastBMU = lastMeasured;
            lastMeasured = minIndex;
        }
    }
    if (lane == 0)
    {
        outBmu[row] = static_cast<unsigned>(minIndex);
        // the squared residual at the chosen node (src/Som.cpp:803): the same f32 sum as its distance
        outDist[row] = dist(minIndex);
    }
}

// ---- phase B
// A CTA owns G neurons; neuron g's Dq chains belong to T consecutive threads (thread t: components t, t + T, ... — CPT of
// them, all of ONE neuron, so the row's two coefficients are read once per thread and the CPT chains are independent
// instruction streams).  One extra warp prepares, one batch ahead, the coefficients of the next R rows (the sumW chain is
// sequential per neuron; the divisions are not) while the chain threads work; the rows themselves arrive by cp.async into the
// other half of a double buffer.  One __syncthreads per batch.
template <int TR, int CPT>
__global__ void __launch_bounds__(768) batch_update_kernel(const float *__restrict__ x, u64 n, int Din, int Dq, int P, int W, int H, int N, int G, int T,
                                                            int R, int xVec, const int2 *__restrict__ bmuXY, const float *__restrict__ lut, int lutW, int lutN,
                                                            const unsigned short *__restrict__ pairI, const unsigned short *__restrict__ pairJ,
                                                            float *__restrict__ mean, float *__restrict__ sigma, float *__restrict__ weight, int rowStride)
{
    extern __shared__ __align__(16) float bmSmem[];
    const int xsFloats = (R * Din + 3) & ~3;
    float *xs = bmSmem;                  // [2][R * Din]
    float *wS = xs + 2 * xsFloats;       // [2][G * R]  w
    float *cS = wS + 2 * G * R;          // [2][G * R]  w / sumW
    float *sS = cS + 2 * G * R;          // [G * R]     running sumW (scratch of the coefficient warp), then [G] final sumW
    int2 *xyS = reinterpret_cast<int2 *>(sS + G * R + (G * R & 1)); // [3][R] BMU coordinates of the batches' rows
    float *lutS = reinterpret_cast<float *>(xyS + 3 * R);           // [lutN] neighbourhood table (when it fits)

    const int tid = threadIdx.x, nChainThreads = G * T;
    const bool coefWarp = tid >= nChainThreads;
    const int g = coefWarp ? 0 : tid / T, t = tid - g * T;
    const int p0 = blockIdx.x * G;
    const int nb = min(G, N - p0);
    const bool active = !coefWarp && g < nb;

    float cur[CPT], S[CPT], curB[TR == VSOM_CLR ? CPT : 1], SB[TR == VSOM_CLR ? CPT : 1];
    int kk[CPT], kj[TR == VSOM_CLR ? CPT : 1];
#pragma unroll
    for (int s = 0; s < CPT; ++s)
    {
        cur[s] = 0.0f;
        S[s] = 0.0f;
        const int k = t + s * T;
        const int kc = k < Dq ? k : 0; // chains past the end shadow component 0 and are dropped at the end
        if (TR == VSOM_CLR)
        {
            curB[s] = 0.0f;
            SB[s] = 0.0f;
            kk[s] = pairI[kc];
            kj[s] = pairJ[kc];
        }
        else
            kk[s] = kc;
    }
    // coefficient warp: lane p < nb carries sumW of neuron p0 + p over all rows
    const int lane = tid & 31;
    float sumW = 0.0f;
    int cx = 0, cy = 0;
    if (coefWarp && lane < nb)
        quirky_xy(static_cast<unsigned>(p0 + lane), W, H, cx, cy);

    // rows of batch j0 -> row buffer `buf`
    auto stage_rows = [&](u64 j0, int buf) {
        const int rows = static_cast<int>(min(static_cast<u64>(R), n - j0));
        const float *src = x + j0 * Din;
        float *dst = xs + buf * xsFloats;
        const int total = rows * Din;
        if (xVec && ((j0 * Din) & 3) == 0)
        {
            const int vec = total >> 2;
            for (int i = tid; i < vec; i += blockDim.x)
                cp_async16(dst + 4 * i, src + 4 * i);
            for (int i = 4 * vec + tid; i < total; i += blockDim.x)
                cp_async4(dst + i, src + i);
        }
        else
            for (int i = tid; i < total; i += blockDim.x)
                cp_async4(dst + i, src + i);
    };
    // BMU coordinates of batch j0's rows -> slot `slot` of a ring of three (they are needed one batch before the rows)
    auto stage_xy = [&](u64 j0, int slot) {
        const int rows = static_cast<int>(min(static_cast<u64>(R), n - j0));
        if (tid < rows)
            cp_async8(xyS + slot * R + tid, bmuXY + j0 + tid);
    };
    auto coefficients = [&](u64 j0, int slot, int cbuf) {
        if (!coefWarp)
            return;
        const int rows = static_cast<int>(min(static_cast<u64>(R), n - j0));
        float *wB = wS + cbuf * G * R, *cB = cS + cbuf * G * R;
        const int2 *xyB = xyS + slot * R;
        if (lane < nb)
        {
            for (int r0 = 0; r0 < rows; r0 += 8)
            {
                float w[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) // independent loads first, the sequential sum after them
                    if (r0 + i < rows)
                    {
                        const int2 b = xyB[r0 + i];
                        const int dx = cx > b.x ? cx - b.x : b.x - cx, dy = cy > b.y ? cy - b.y : b.y - cy;
                        w[i] = lutN ? lutS[dy * lutW + dx] : __ldg(lut + dy * lutW + dx);
                    }
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    if (r0 + i < rows)
                    {
                        sumW = __fadd_rn(sumW, w[i]); // Eq. 47
                        wB[lane * R + r0 + i] = w[i];
                        sS[lane * R + r0 + i] = sumW;
                    }
            }
        }
        __syncwarp();
        for (int i = lane; i < nb * R; i += 32)
            if (i % R < rows)
                cB[i] = __fdiv_rn(wB[i], sS[i]); // currentWeight / sumOfWeights
    };

    // pipeline, iteration j: rows of batch j + 1 and coordinates of batch j + 2 in flight (cp.async), the coefficient warp on
    // batch j + 1, the chain threads on batch j.  Row buffers and coefficient buffers: two each; coordinates: a ring of three.
    for (int i = tid; i < lutN; i += blockDim.x)
        lutS[i] = lut[i];
    stage_rows(0, 0);
    stage_xy(0, 0);
    if (static_cast<u64>(R) < n)
        stage_xy(R, 1);
    cp_async_wait_all();
    __syncthreads();
    coefficients(0, 0, 0);
    int buf = 0, slot = 0;
    for (u64 j0 = 0; j0 < n; j0 += R, buf ^= 1, slot = slot == 2 ? 0 : slot + 1)
    {
        const int rows = static_cast<int>(min(static_cast<u64>(R), n - j0));
        const int slot1 = slot == 2 ? 0 : slot + 1, slot2 = slot1 == 2 ? 0 : slot1 + 1;
        cp_async_wait_all();
        __syncthreads(); // visible: rows + coefficients of batch j, coordinates of batch j + 1; everybody is done with batch j - 1
        if (j0 + R < n)
        {
            stage_rows(j0 + R, buf ^ 1);
            if (j0 + 2 * static_cast<u64>(R) < n)
                stage_xy(j0 + 2 * static_cast<u64>(R), slot2);
            coefficients(j0 + R, slot1, buf ^ 1);
        }
        if (!active)
            continue;
        const float *xb = xs + buf * xsFloats;
        const float *wp = wS + (buf * G + g) * R, *cp = cS + (buf * G + g) * R;
#pragma unroll 2
        for (int r = 0; r < rows; ++r)
        {
            const float w = wp[r], c = cp[r];
            const float *xr = xb + r * Din;
            if (TR != VSOM_CLR)
            {
#pragma unroll
                for (int s = 0; s < CPT; ++s)
                {
                    float d = __fsub_rn(xr[kk[s]], cur[s]);
                    if (TR == VSOM_MEDIAN)
                    {
                        const float a = fabsf(d);
                        d = a > 0.0f ? __uint_as_float((__float_as_uint(d) & 0x80000000u) | 0x3f800000u) : a;
                    }
                    cur[s] = __fadd_rn(cur[s], __fmul_rn(c, d));             // Eq. 53
                    S[s] = __fadd_rn(S[s], __fmul_rn(__fmul_rn(w, d), d));   // Eq. 68
                }
            }
            else
            {
#pragma unroll
                for (int s = 0; s < CPT; ++s)
                {
                    const float xi = xr[kk[s]], xj = xr[kj[s]];
                    const float inner = __fsub_rn(__fadd_rn(__fmul_rn(cur[s], xi), curB[s]), xj);
                    const float db = __fmul_rn(-2.0f, inner), da = __fmul_rn(db, xi);
                    cur[s] = __fadd_rn(cur[s], __fmul_rn(c, da));
                    curB[s] = __fadd_rn(curB[s], __fmul_rn(c, db));
                    S[s] = __fadd_rn(S[s], __fmul_rn(__fmul_rn(w, da), da));
                    SB[s] = __fadd_rn(SB[s], __fmul_rn(__fmul_rn(w, db), db));
                }
            }
        }
    }
    __syncthreads();
    if (coefWarp && lane < nb)
    {
        sS[lane] = sumW;
        weight[p0 + lane] = sumW; // :875
    }
    __syncthreads();
    if (!active)
        return;
    const size_t at = static_cast<size_t>(p0 + g) * rowStride;
    const float sw = sS[g];
#pragma unroll
    for (int s = 0; s < CPT; ++s)
    {
        const int k = t + s * T;
        if (k >= Dq)
            continue;
        mean[at + k] = cur[s];                                              // :871
        sigma[at + k] = __fsqrt_rn(__fdiv_rn(S[s], sw));                    // :873 (no abs)
        if (TR == VSOM_CLR)
        {
            mean[at + P + k] = curB[s];
            sigma[at + P + k] = __fsqrt_rn(__fdiv_rn(SB[s], sw));
        }
    }
}

// one chunk-epoch; x / bmu / dist on the device.  isFirst selects the global search; otherwise lastDev holds the start
// nodes of the local walks.  On return bmuDev holds every row's BMU and distDev its squared residual.
int launch_batch_epoch(vsom_ctx *ctx, const float *xDev, size_t n, double sigma, int isFirst, const u64 *lastDev, unsigned *bmuDev, float *distDev)
{
    if (ctx->world > 1)
        return set_error(ctx, VSOM_ERR_UNSUPPORTED, "batch-map trainer needs an unsharded context");
    if (n == 0)
        return VSOM_OK;
    // ---- phase B's launch shape, first: a shape it cannot run is refused before anything is enqueued (no hits counted)
    const int Dq = ctx->transform == VSOM_CLR ? ctx->P : ctx->Dm;
    // chains per thread: the value that wastes the fewest lanes once T is rounded up to whole warps (ties: more chains per thread)
    const int cptMax = ctx->transform == VSOM_CLR ? 4 : 8, cptMin = ctx->transform == VSOM_CLR ? 2 : 4;
    int cpt = cptMin, T = 0;
    long bestCost = -1;
    for (int c = cptMin; c <= cptMax; ++c)
    {
        const int t = ((Dq + c - 1) / c + 31) / 32 * 32;
        if (t > 736)
            continue;
        const long cost = static_cast<long>(t) * c;
        if (bestCost < 0 || cost <= bestCost)
        {
            bestCost = cost;
            cpt = c;
            T = t;
        }
    }
    if (bestCost < 0)
        return set_error(ctx, VSOM_ERR_UNSUPPORTED, "batch-map trainer: model vector longer than 5888 components");
    // neurons per CTA: as many as keep every SM busy in the fewest rounds (the rows are streamed once per CTA)
    const int gMax = std::max(1, std::min(BM_MAXNB, 736 / T));
    int G = 1;
    long bestRounds = -1;
    for (int gq = 1; gq <= gMax; ++gq)
    {
        const long ctas = (ctx->N + gq - 1) / gq, rounds = (ctas + ctx->numSMs - 1) / ctx->numSMs * gq;
        if (bestRounds < 0 || rounds <= bestRounds)
        {
            bestRounds = rounds;
            G = gq;
        }
    }
    // rows per batch: two batches of rows in shared memory, at most 96 KB each
    const int R = std::max(4, std::min(BM_ROWS, static_cast<int>((100 * 1024) / (sizeof(float) * ctx->Din)) & ~3));
    if (sizeof(float) * 2 * R * ctx->Din > 208 * 1024)
        return set_error(ctx, VSOM_ERR_UNSUPPORTED, "batch-map trainer: rows longer than 6400 values");
    int rc;
    // ---- phase A; last_score_tc reports which search ran (K2's tier, or 0 for the exact scan and the local walks)
    if (isFirst)
    {
        ScoreOut out;
        out.bmu = bmuDev;
        out.dist = distDev;
        rc = score_rows(ctx, xDev, false, n, 0, true, out, nullptr);
        if (rc)
            return rc;
    }
    else
    {
        ctx->lastScoreTier = 0;
        const unsigned grid = static_cast<unsigned>((n + 31) / 32);
        if (ctx->transform == VSOM_CLR)
            local_bmu_rows_kernel<VSOM_CLR><<<grid, 256, 0, ctx->stream>>>(xDev, n, ctx->mean, ctx->W, ctx->H, ctx->Din, ctx->Dr, ctx->P, ctx->rowStride,
                                                                           ctx->pairI, ctx->pairJ, ctx->order, lastDev, bmuDev, distDev);
        else
            local_bmu_rows_kernel<VSOM_STANDARD><<<grid, 256, 0, ctx->stream>>>(xDev, n, ctx->mean, ctx->W, ctx->H, ctx->Din, ctx->Dr, ctx->P,
                                                                                ctx->rowStride, ctx->pairI, ctx->pairJ, ctx->order, lastDev, bmuDev, distDev);
        ctx->launches += 1;
    }
    hits_add_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, ctx->stream>>>(bmuDev, n, ctx->hits);
    // ---- phase B: neighbourhood table over the reference's (quirky) coordinates, (float)nw
    int mx, my;
    quirky_xy(static_cast<unsigned>(ctx->N - 1), ctx->W, ctx->H, mx, my);
    const int lw = ctx->W, lh = my + 1;
    std::vector<float> lutHost(static_cast<size_t>(lw) * lh);
    for (int dy = 0; dy < lh; ++dy)
        for (int dx = 0; dx < lw; ++dx)
            lutHost[static_cast<size_t>(dy) * lw + dx] = static_cast<float>(neighbourhood_weight(dx, dy, sigma));
    rc = stage_reserve(ctx, 6, sizeof(float) * lutHost.size() + 256);
    if (rc)
        return rc;
    rc = stage_reserve(ctx, 7, sizeof(int2) * n);
    if (rc)
        return rc;
    float *lutDev = static_cast<float *>(ctx->stage[6]);
    int2 *xyDev = static_cast<int2 *>(ctx->stage[7]);
    VSOM_CUDA(ctx, cudaMemcpyAsync(lutDev, lutHost.data(), sizeof(float) * lutHost.size(), cudaMemcpyHostToDevice, ctx->stream));
    VSOM_CUDA(ctx, cudaStreamSynchronize(ctx->stream)); // lutHost is a local
    bmu_xy_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, ctx->stream>>>(bmuDev, n, ctx->W, ctx->H, xyDev);
    const unsigned grid = static_cast<unsigned>((ctx->N + G - 1) / G);
    const unsigned threads = static_cast<unsigned>(G * T + 32);
    const int lutN = lutHost.size() <= static_cast<size_t>(BM_LUT_SMEM) ? static_cast<int>(lutHost.size()) : 0;
    const size_t smem = sizeof(float) * (2 * static_cast<size_t>((R * ctx->Din + 3) & ~3) + 5 * static_cast<size_t>(G) * R + 2 + lutN) + sizeof(int2) * 3 * R;
    const int xVec = (reinterpret_cast<uintptr_t>(xDev) & 15) == 0;
#define VSOM_BM_LAUNCH(TR, C)                                                                                                                        \
    {                                                                                                                                                \
        VSOM_CUDA(ctx, cudaFuncSetAttribute(batch_update_kernel<TR, C>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));        \
        batch_update_kernel<TR, C><<<grid, threads, smem, ctx->stream>>>(xDev, n, ctx->Din, Dq, ctx->P, ctx->W, ctx->H, ctx->N, G, T, R, xVec, xyDev, \
                                                                         lutDev, lw, lutN, ctx->pairI, ctx->pairJ, ctx->mean, ctx->sigma, ctx->weight,     \
                                                                         ctx->rowStride);                                                            \
    }
#define VSOM_BM_CPT(TR)                  \
    switch (cpt)                         \
    {                                    \
    case 4: VSOM_BM_LAUNCH(TR, 4) break; \
    case 5: VSOM_BM_LAUNCH(TR, 5) break; \
    case 6: VSOM_BM_LAUNCH(TR, 6) break; \
    case 7: VSOM_BM_LAUNCH(TR, 7) break; \
    default: VSOM_BM_LAUNCH(TR, 8) break; \
    }
    if (ctx->transform == VSOM_STANDARD)
        VSOM_BM_CPT(VSOM_STANDARD)
    else if (ctx->transform == VSOM_MEDIAN)
        VSOM_BM_CPT(VSOM_MEDIAN)
    else
        switch (cpt)
        {
        case 2: VSOM_BM_LAUNCH(VSOM_CLR, 2) break;
        case 3: VSOM_BM_LAUNCH(VSOM_CLR, 3) break;
        default: VSOM_BM_LAUNCH(VSOM_CLR, 4) break;
        }
#undef VSOM_BM_CPT
#undef VSOM_BM_LAUNCH
    ctx->launches += 3;
    VSOM_CUDA(ctx, cudaGetLastError());
    return VSOM_OK;
}

} // namespace vsom
