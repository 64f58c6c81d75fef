// cluster.cu — vsom_cluster_nodes: k-means over the map's nodes (SOM Toolbox som_kmeans / kmeans_clusters, after Vesanto &
// Alhoniemi (2000), "Clustering of the self-organizing map").  The points are the N rows of the mean plane; the contract, written
// so that numpy can restate every bit of it, is in include/vsom_b200.h.
//
//   check    one pass over the plane: a non-finite element raises a device flag and the call is refused.
//   seeding  k-means++ on draws fixed by the seed.  Per pick: cluster_seed_dist_kernel streams the plane once (D_p = min(D_p,
//            d(p, c_new)); rows are staged through shared memory in slices of 32 components and every node keeps its own chain,
//            dist_ordered's sequential sum or EigenSseSum), cluster_block_sums_kernel forms the f64 block sums T_b, and
//            cluster_pick_kernel (one CTA) walks the blocks and the chosen block's nodes and copies the chosen row into the
//            centroids.  No pick waits for the host.
//   assign   K3 (find_bmu_exact_kernel / find_bmu_exact_eigen_kernel, score_exact.cu): the plane's rows scored against the f32
//            centroids as a Standard map of k nodes — the argmin of (d, j) in the context's order.
//   update   K5's index build (som_index.cu) with k bins lists every cluster's members in ascending node order;
//            cluster_group_sums_kernel sums each group of VSOM_CLUSTER_BLOCK members per component, cluster_update_kernel adds a
//            cluster's group sums in group order and divides.  One flag per iteration comes back: whether a label changed.
#include "common.cuh"

#include <algorithm>

namespace vsom
{

constexpr int kBlock = VSOM_CLUSTER_BLOCK;
constexpr int kSeedNodes = 256, kSeedSlice = 32; // seeding pass: nodes per CTA, components per staged slice
constexpr int kSumThreads = 256;                 // group sums / update: components per CTA
enum ClusterFlag
{
    kFlagNonFinite = 0, // an element of the mean plane is NaN or infinite
    kFlagTotal = 1,     // a seeding total was 0 or not finite
    kFlagChanged = 2,   // a label differs from the previous assignment's
    kFlagCount = 3
};

// w_p: 1 (VSOM_CLUSTER_UNIFORM, hits == null) or the node's hit count (VSOM_CLUSTER_HITS)
static __device__ __forceinline__ double node_weight(const u64 *hits, u64 p) { return hits ? __ull2double_rn(hits[p]) : 1.0; }

__global__ void __launch_bounds__(256) cluster_check_kernel(const float *__restrict__ mean, int N, int Dm, int rowStride, int *__restrict__ flags)
{
    const int lane = threadIdx.x & 31;
    const u64 warps = static_cast<u64>(gridDim.x) * (blockDim.x >> 5);
    bool bad = false;
    for (u64 p = static_cast<u64>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5); p < static_cast<u64>(N); p += warps)
        for (int k = lane; k < Dm; k += 32)
            bad |= !isfinite(mean[p * rowStride + k]);
    if (bad)
        flags[kFlagNonFinite] = 1;
}

// D_p = min(D_p, d(p, c)) for every node (first: D_p = d(p, c)).  Warps stage 32-component slices of 256 rows (128-byte segments):
// every lane holds its 32 elements of the next slice in registers, loaded while the CTA computes on the current one, so the loads of
// a slice are in flight behind the arithmetic of the previous.  Each thread continues its node's chain over the slice:
// dist_sequential's s + r*r, or EigenSseSum's blocks of eight and its finish — the arithmetic of dist_ordered<VSOM_STANDARD>(row, c,
// Dm, ...) with the residual m - c.
template <bool EIGEN>
__global__ void __launch_bounds__(kSeedNodes) cluster_seed_dist_kernel(const float *__restrict__ mean, int N, int Dm, int rowStride, const float *__restrict__ c,
                                                                       int first, float *__restrict__ dmin, const int *__restrict__ flags)
{
    constexpr int kWarps = kSeedNodes / 32, kRowsPerWarp = kSeedNodes / kWarps;
    __shared__ float rows[kSeedNodes][kSeedSlice + 1];
    __shared__ float cs[kSeedSlice];
    if (flags[kFlagNonFinite] | flags[kFlagTotal])
        return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int node0 = blockIdx.x * kSeedNodes;
    float next[kRowsPerWarp]; // rows warp + kWarps i of the next slice, element lane
    auto load = [&](int k0) {
        const int k = k0 + lane;
#pragma unroll
        for (int i = 0; i < kRowsPerWarp; ++i)
        {
            const int p = node0 + warp + kWarps * i;
            next[i] = p < N && k < Dm ? mean[static_cast<size_t>(p) * rowStride + k] : 0.0f;
        }
    };
    float s = 0.0f;
    EigenSseSum acc;
    float rest[8];
#pragma unroll
    for (int j = 0; j < 8; ++j)
        rest[j] = 0.0f;
    load(0);
    for (int k0 = 0; k0 < Dm; k0 += kSeedSlice)
    {
        __syncthreads(); // the previous slice is consumed
#pragma unroll
        for (int i = 0; i < kRowsPerWarp; ++i)
            rows[warp + kWarps * i][lane] = next[i];
        if (warp == 0)
            cs[lane] = k0 + lane < Dm ? c[k0 + lane] : 0.0f;
        __syncthreads();
        if (k0 + kSeedSlice < Dm)
            load(k0 + kSeedSlice);
        const float *m = rows[tid];
        if (!EIGEN)
        {
            const int len = min(kSeedSlice, Dm - k0);
            for (int j = 0; j < len; ++j)
            {
                const float r = residual<VSOM_STANDARD>(m, cs, j, 0, nullptr, nullptr);
                s = __fadd_rn(s, __fmul_rn(r, r));
            }
        }
        else
        {
#pragma unroll
            for (int b = 0; b < kSeedSlice; b += 8)
            {
                float t[8];
#pragma unroll
                for (int j = 0; j < 8; ++j)
                {
                    const float r = residual<VSOM_STANDARD>(m, cs, b + j, 0, nullptr, nullptr);
                    t[j] = __fmul_rn(r, r);
                }
                if (k0 + b + 8 <= Dm) // a full block of eight
                    acc.block(t);
                else if (k0 + b < Dm) // the Dm % 8 terms behind the last full block
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        rest[j] = t[j];
            }
        }
    }
    const int p = node0 + tid;
    if (p >= N)
        return;
    const float d = EIGEN ? acc.finish(rest, Dm & 7) : s;
    dmin[p] = first ? d : (d < dmin[p] ? d : dmin[p]);
}

// T_b = sequential f64 sum, from 0 in node order, of q_p over the nodes of block b: q_p = w_p (d == null), else w_p * (double)d[p]
__global__ void __launch_bounds__(kBlock) cluster_block_sums_kernel(const float *__restrict__ d, const u64 *__restrict__ hits, int N, double *__restrict__ T,
                                                                    const int *__restrict__ flags)
{
    __shared__ double q[kBlock];
    if (flags[kFlagNonFinite] | flags[kFlagTotal])
        return;
    const int p0 = blockIdx.x * kBlock, count = min(kBlock, N - p0), i = threadIdx.x;
    if (i < count)
    {
        const double w = node_weight(hits, p0 + i);
        q[i] = d ? __dmul_rn(w, static_cast<double>(d[p0 + i])) : w;
    }
    __syncthreads();
    if (i == 0)
    {
        double s = 0.0;
        for (int j = 0; j < count; ++j)
            s = __dadd_rn(s, q[j]);
        T[blockIdx.x] = s;
    }
}

// Pick j of the seeding (dynamic shared memory: nb doubles).  Thread 0 takes the total and the target u_j * total, walks the block
// sums to the first block whose running sum exceeds the target (else the last block with T_b > 0), then that block's q_p from the
// sum of the earlier blocks to the first node whose running sum exceeds it (else the last node with q_p > 0).  The CTA copies the
// chosen row into centroid j.  A total of 0 or one that is not finite raises kFlagTotal instead.
__global__ void __launch_bounds__(kBlock) cluster_pick_kernel(const double *__restrict__ T, int nb, const float *__restrict__ dmin, const u64 *__restrict__ hits, int N,
                                                              double u, int j, const float *__restrict__ mean, int Dm, int rowStride, double *__restrict__ cent64,
                                                              float *__restrict__ cent32, int *__restrict__ flags)
{
    extern __shared__ double sT[];
    __shared__ double q[kBlock];
    __shared__ double sRun, sTarget;
    __shared__ int sBlock, sNode;
    if (flags[kFlagNonFinite] | flags[kFlagTotal])
        return;
    const int tid = threadIdx.x;
    for (int b = tid; b < nb; b += kBlock)
        sT[b] = T[b];
    __syncthreads();
    if (tid == 0)
    {
        double total = 0.0;
        for (int b = 0; b < nb; ++b)
            total = __dadd_rn(total, sT[b]);
        int blk = -1, lastPos = -1;
        double run = 0.0, runLastPos = 0.0;
        const double target = __dmul_rn(u, total);
        if (total > 0.0 && isfinite(total))
        {
            for (int b = 0; b < nb; ++b)
            {
                const double next = __dadd_rn(run, sT[b]);
                if (next > target)
                {
                    blk = b;
                    break;
                }
                if (sT[b] > 0.0)
                {
                    lastPos = b;
                    runLastPos = run;
                }
                run = next;
            }
            if (blk < 0)
            {
                blk = lastPos;
                run = runLastPos;
            }
        }
        else
            flags[kFlagTotal] = 1;
        sBlock = blk;
        sRun = run;
        sTarget = target;
    }
    __syncthreads();
    const int blk = sBlock;
    if (blk < 0)
        return;
    const int p0 = blk * kBlock, count = min(kBlock, N - p0);
    if (tid < count)
    {
        const double w = node_weight(hits, p0 + tid);
        q[tid] = dmin ? __dmul_rn(w, static_cast<double>(dmin[p0 + tid])) : w;
    }
    __syncthreads();
    if (tid == 0)
    {
        double run = sRun;
        const double target = sTarget;
        int node = -1, lastPos = -1;
        for (int i = 0; i < count; ++i)
        {
            run = __dadd_rn(run, q[i]);
            if (run > target)
            {
                node = i;
                break;
            }
            if (q[i] > 0.0)
                lastPos = i;
        }
        sNode = p0 + (node >= 0 ? node : lastPos);
    }
    __syncthreads();
    const float *row = mean + static_cast<size_t>(sNode) * rowStride;
    for (int k = tid; k < Dm; k += kBlock)
    {
        const float v = row[k];
        cent32[static_cast<size_t>(j) * rowStride + k] = v;
        cent64[static_cast<size_t>(j) * Dm + k] = static_cast<double>(v);
    }
}

__global__ void cluster_labels_changed_kernel(const unsigned *__restrict__ a, const unsigned *__restrict__ b, int N, int *__restrict__ flags)
{
    bool changed = false;
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < N; p += gridDim.x * blockDim.x)
        changed |= a[p] != b[p];
    if (changed)
        flags[kFlagChanged] = 1;
}

// groups of every cluster: ceil(count_j / VSOM_CLUSTER_BLOCK)
__global__ void cluster_group_counts_kernel(const u64 *__restrict__ counts, int k, u64 *__restrict__ groups)
{
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < k; j += gridDim.x * blockDim.x)
        groups[j] = (counts[j] + kBlock - 1) / kBlock;
}

// One CTA per (group g, 256 columns from col0): column c < Dm sums w_p * (double)m_p[c], column Dm sums w_p, sequentially from 0
// over the group's members in ascending node order.  Group g is group g - goff[j] of the cluster j with goff[j] <= g < goff[j + 1].
__global__ void __launch_bounds__(kSumThreads) cluster_group_sums_kernel(const float *__restrict__ mean, int rowStride, int Dm, int col0, const u64 *__restrict__ hits, int k,
                                                                         const u64 *__restrict__ offsets, const unsigned *__restrict__ members,
                                                                         const u64 *__restrict__ goff, double *__restrict__ gsum)
{
    __shared__ unsigned mem[kBlock];
    __shared__ double w[kBlock];
    const u64 g = blockIdx.x;
    if (g >= goff[k])
        return;
    int lo = 0, hi = k - 1; // the last j with goff[j] <= g: clusters without members own no group
    while (lo < hi)
    {
        const int mid = (lo + hi + 1) >> 1;
        if (goff[mid] <= g)
            lo = mid;
        else
            hi = mid - 1;
    }
    const u64 m0 = offsets[lo] + (g - goff[lo]) * kBlock, m1 = min(offsets[lo + 1], m0 + kBlock);
    const int count = static_cast<int>(m1 - m0);
    for (int i = threadIdx.x; i < count; i += kSumThreads)
    {
        const unsigned p = members[m0 + i];
        mem[i] = p;
        w[i] = node_weight(hits, p);
    }
    __syncthreads();
    const int c = col0 + blockIdx.y * kSumThreads + threadIdx.x;
    if (c > Dm)
        return;
    double s = 0.0;
    if (c < Dm)
    {
#pragma unroll 8
        for (int i = 0; i < count; ++i)
            s = __dadd_rn(s, __dmul_rn(w[i], static_cast<double>(mean[static_cast<size_t>(mem[i]) * rowStride + c])));
    }
    else
        for (int i = 0; i < count; ++i)
            s = __dadd_rn(s, w[i]);
    gsum[g * (Dm + 1) + c] = s;
}

// One CTA per (cluster j, 256 columns from col0): W_j and the numerators are the cluster's group sums added from 0 in group order.
// Column Dm writes W_j (weight, may be null); the others, when W_j != 0, write c_j = numerator / W_j and its f32 rounding.
__global__ void __launch_bounds__(kSumThreads) cluster_update_kernel(const double *__restrict__ gsum, int Dm, int col0, const u64 *__restrict__ goff,
                                                                     double *__restrict__ cent64, float *__restrict__ cent32, int cStride, double *__restrict__ weight)
{
    const int j = blockIdx.x, c = col0 + blockIdx.y * kSumThreads + threadIdx.x;
    if (c > Dm)
        return;
    const u64 g0 = goff[j], g1 = goff[j + 1];
    double W = 0.0;
    for (u64 g = g0; g < g1; ++g)
        W = __dadd_rn(W, gsum[g * (Dm + 1) + Dm]);
    if (c == Dm)
    {
        if (weight)
            weight[j] = W;
        return;
    }
    if (W == 0.0) // a cluster without weight keeps its centroid
        return;
    double s = 0.0;
    for (u64 g = g0; g < g1; ++g)
        s = __dadd_rn(s, gsum[g * (Dm + 1) + c]);
    const double v = __ddiv_rn(s, W);
    cent64[static_cast<size_t>(j) * Dm + c] = v;
    cent32[static_cast<size_t>(j) * cStride + c] = __double2float_rn(v);
}

// The call's scratch is carved from the context's grow-only staging slot kClusterStage, every buffer on a 256-byte boundary: a call
// that fits what an earlier one reserved allocates nothing.  (The index build it calls stages in slots 3 and 4; the exact scan in none.)
constexpr int kClusterStage = 5;
template <class T>
static void carve(unsigned char *base, size_t &off, T *&p, size_t count)
{
    p = reinterpret_cast<T *>(base + off);
    off += (sizeof(T) * std::max<size_t>(count, 1) + 255) & ~static_cast<size_t>(255);
}

// CUDA events around the phases of one call, read once the stream has drained: ms[0] seeding (check included), ms[1] the
// assignments, ms[2] the updates, ms[3] the outputs (weights of the final labels, inertia)
struct PhaseEvents
{
    std::vector<cudaEvent_t> ev;
    std::vector<int> phase; // of every (start, end) pair
    ~PhaseEvents()
    {
        for (cudaEvent_t e : ev)
            cudaEventDestroy(e);
    }
    cudaError_t mark(cudaStream_t st, int ph, bool start)
    {
        cudaEvent_t e;
        cudaError_t rc = cudaEventCreate(&e);
        if (rc != cudaSuccess)
            return rc;
        ev.push_back(e);
        if (start)
            phase.push_back(ph);
        return cudaEventRecord(e, st);
    }
    void read(double ms[4]) const
    {
        ms[0] = ms[1] = ms[2] = ms[3] = 0.0;
        for (size_t i = 0; i + 1 < ev.size(); i += 2)
        {
            float t = 0.0f;
            if (cudaEventElapsedTime(&t, ev[i], ev[i + 1]) == cudaSuccess)
                ms[phase[i / 2]] += t;
        }
    }
};

#define CLUSTER_TRY(expr)       \
    do                          \
    {                           \
        const int _rc = (expr); \
        if (_rc)                \
            return _rc;         \
    } while (0)

// splitmix64 (state += golden gamma; two xor-shift-multiply rounds; a final xor-shift), one draw per pick: (z >> 11) * 2^-53
static std::vector<double> seeding_draws(uint64_t seed, int k)
{
    std::vector<double> u(k);
    uint64_t state = seed;
    for (int j = 0; j < k; ++j)
    {
        state += 0x9E3779B97F4A7C15ull;
        uint64_t z = state;
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        z ^= z >> 31;
        u[j] = static_cast<double>(z >> 11) * 0x1.0p-53;
    }
    return u;
}

int cluster_nodes(vsom_ctx *ctx, int k, uint64_t seed, int weighting, int maxIter, ClusterResult &res)
{
    const int N = ctx->N, Dm = ctx->Dm, rs = ctx->rowStride, nb = (N + kBlock - 1) / kBlock;
    const size_t groupsMax = static_cast<size_t>(nb) + k; // sum over clusters of ceil(count_j / kBlock)
    const u64 *hits = weighting == VSOM_CLUSTER_HITS ? ctx->hits : nullptr;
    const bool eigen = ctx->order == VSOM_ORDER_EIGEN_SSE;
    cudaStream_t st = ctx->stream;

    int *flags;
    double *T, *cent64, *gsum, *weight;
    float *dmin, *cent32, *dist;
    unsigned *labels[2], *members;
    u64 *counts, *offsets, *groups, *goff;
    auto layout = [&](unsigned char *base) {
        size_t off = 0;
        carve(base, off, flags, kFlagCount);
        carve(base, off, T, nb);
        carve(base, off, dmin, N);
        carve(base, off, cent64, static_cast<size_t>(k) * Dm);
        carve(base, off, cent32, static_cast<size_t>(k) * rs);
        carve(base, off, labels[0], N);
        carve(base, off, labels[1], N);
        carve(base, off, dist, N);
        carve(base, off, members, N);
        carve(base, off, counts, k);
        carve(base, off, offsets, static_cast<size_t>(k) + 1);
        carve(base, off, groups, k);
        carve(base, off, goff, static_cast<size_t>(k) + 1);
        carve(base, off, gsum, groupsMax * (Dm + 1));
        carve(base, off, weight, k);
        return off;
    };
    CLUSTER_TRY(stage_reserve(ctx, kClusterStage, layout(nullptr)));
    layout(static_cast<unsigned char *>(ctx->stage[kClusterStage]));
    PhaseEvents events;
    VSOM_CUDA(ctx, events.mark(st, 0, true));
    VSOM_CUDA(ctx, cudaMemsetAsync(flags, 0, sizeof(int) * kFlagCount, st));
    VSOM_CUDA(ctx, cudaMemsetAsync(cent32, 0, sizeof(float) * k * rs, st)); // row padding of the Standard map K3 reads

    // ---- check and seeding
    cluster_check_kernel<<<ctx->numSMs * 4, 256, 0, st>>>(ctx->mean, N, Dm, rs, flags);
    ctx->launches += 1;
    const std::vector<double> u = seeding_draws(seed, k);
    // the block sums in shared memory: nb <= 16 384 (N < 2^24) is at most 128 KiB beside the kernel's 8 KiB of static arrays; the
    // opt-in is set on every call, as static and dynamic memory together may pass the 48 KiB default from nb = 5 117 on
    const size_t pickSmem = sizeof(double) * nb;
    VSOM_CUDA(ctx, cudaFuncSetAttribute(cluster_pick_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(pickSmem)));
    const unsigned seedGrid = static_cast<unsigned>((N + kSeedNodes - 1) / kSeedNodes);
    for (int j = 0; j < k; ++j)
    {
        const float *dj = nullptr;
        if (j > 0)
        {
            const float *c = cent32 + static_cast<size_t>(j - 1) * rs;
            if (eigen)
                cluster_seed_dist_kernel<true><<<seedGrid, kSeedNodes, 0, st>>>(ctx->mean, N, Dm, rs, c, j == 1, dmin, flags);
            else
                cluster_seed_dist_kernel<false><<<seedGrid, kSeedNodes, 0, st>>>(ctx->mean, N, Dm, rs, c, j == 1, dmin, flags);
            dj = dmin;
        }
        cluster_block_sums_kernel<<<nb, kBlock, 0, st>>>(dj, hits, N, T, flags);
        cluster_pick_kernel<<<1, kBlock, pickSmem, st>>>(T, nb, dj, hits, N, u[j], j, ctx->mean, Dm, rs, cent64, cent32, flags);
        ctx->launches += j > 0 ? 3 : 2;
    }
    VSOM_CUDA(ctx, cudaGetLastError());
    VSOM_CUDA(ctx, events.mark(st, 0, false));
    int hFlags[kFlagCount];
    VSOM_CUDA(ctx, cudaMemcpyAsync(hFlags, flags, sizeof(hFlags), cudaMemcpyDeviceToHost, st));
    VSOM_CUDA(ctx, cudaStreamSynchronize(st));
    if (hFlags[kFlagNonFinite])
        return set_error(ctx, VSOM_ERR_INVALID, "vsom_cluster_nodes: the mean plane has a NaN or infinite element");
    if (hFlags[kFlagTotal])
        return set_error(ctx, VSOM_ERR_INVALID, "vsom_cluster_nodes: a seeding total is 0 or not finite (fewer than k distinct nodes carry weight, "
                                                "a map without hits under VSOM_CLUSTER_HITS, or distances that overflow f32)");

    // ---- Lloyd iterations: the plane's rows scored against the f32 centroids, a Standard map of k nodes
    ScanMap map;
    map.mean = cent32;
    map.N = k;
    map.rowStride = rs;
    map.transform = VSOM_STANDARD;
    map.Din = rs;
    map.Dr = Dm;
    const unsigned sumCols = static_cast<unsigned>((Dm + 1 + kSumThreads - 1) / kSumThreads);
    // members grouped by label; the group sums of columns col0 .. Dm; then centroids (update) and W_j
    auto sums = [&](const unsigned *lab, int col0, bool update) -> int {
        CLUSTER_TRY(launch_build_index(ctx, lab, N, k, counts, offsets, members));
        cluster_group_counts_kernel<<<std::min((k + 255) / 256, 1024), 256, 0, st>>>(counts, k, groups);
        ctx->launches += 1;
        CLUSTER_TRY(launch_offsets_scan(ctx, groups, k, goff));
        const unsigned cols = update ? sumCols : 1u;
        cluster_group_sums_kernel<<<dim3(static_cast<unsigned>(groupsMax), cols), kSumThreads, 0, st>>>(ctx->mean, rs, Dm, col0, hits, k, offsets, members, goff, gsum);
        cluster_update_kernel<<<dim3(static_cast<unsigned>(k), cols), kSumThreads, 0, st>>>(gsum, Dm, col0, goff, cent64, cent32, rs, weight);
        ctx->launches += 2;
        VSOM_CUDA(ctx, cudaGetLastError());
        return VSOM_OK;
    };
    int cur = 0;
    for (int it = 1;; ++it)
    {
        cur = it & 1;
        VSOM_CUDA(ctx, events.mark(st, 1, true));
        CLUSTER_TRY(launch_find_bmu_list(ctx, ctx->mean, N, nullptr, nullptr, 0, ScoreOut{labels[cur], dist}, st, nullptr, map));
        VSOM_CUDA(ctx, events.mark(st, 1, false));
        res.iterations = it;
        if (it > 1)
        {
            VSOM_CUDA(ctx, cudaMemsetAsync(flags + kFlagChanged, 0, sizeof(int), st));
            cluster_labels_changed_kernel<<<std::min((N + 255) / 256, ctx->numSMs * 8), 256, 0, st>>>(labels[cur], labels[cur ^ 1], N, flags);
            ctx->launches += 1;
            int changed = 0;
            VSOM_CUDA(ctx, cudaMemcpyAsync(&changed, flags + kFlagChanged, sizeof(int), cudaMemcpyDeviceToHost, st));
            VSOM_CUDA(ctx, cudaStreamSynchronize(st));
            if (!changed)
            {
                res.converged = 1;
                break;
            }
        }
        if (it == maxIter)
        {
            res.converged = 0;
            break;
        }
        VSOM_CUDA(ctx, events.mark(st, 2, true));
        CLUSTER_TRY(sums(labels[cur], 0, true));
        VSOM_CUDA(ctx, events.mark(st, 2, false));
    }

    // ---- outputs: W_j of the final labels, the inertia in the seeding's block order, labels and centroids
    VSOM_CUDA(ctx, events.mark(st, 3, true));
    CLUSTER_TRY(sums(labels[cur], Dm, false));
    cluster_block_sums_kernel<<<nb, kBlock, 0, st>>>(dist, hits, N, T, flags);
    ctx->launches += 1;
    VSOM_CUDA(ctx, cudaGetLastError());
    VSOM_CUDA(ctx, events.mark(st, 3, false));
    std::vector<double> hT(nb);
    std::vector<unsigned> lab(N);
    res.centroids.resize(static_cast<size_t>(k) * Dm);
    res.weight.resize(k);
    VSOM_CUDA(ctx, cudaMemcpyAsync(hT.data(), T, sizeof(double) * nb, cudaMemcpyDeviceToHost, st));
    VSOM_CUDA(ctx, cudaMemcpyAsync(lab.data(), labels[cur], sizeof(unsigned) * N, cudaMemcpyDeviceToHost, st));
    VSOM_CUDA(ctx, cudaMemcpyAsync(res.centroids.data(), cent64, sizeof(double) * k * Dm, cudaMemcpyDeviceToHost, st));
    VSOM_CUDA(ctx, cudaMemcpyAsync(res.weight.data(), weight, sizeof(double) * k, cudaMemcpyDeviceToHost, st));
    VSOM_CUDA(ctx, cudaStreamSynchronize(st));
    res.inertia = 0.0;
    for (double t : hT)
        res.inertia += t;
    res.label.assign(lab.begin(), lab.end());
    events.read(res.phaseMs);
    return VSOM_OK;
}

} // namespace vsom
