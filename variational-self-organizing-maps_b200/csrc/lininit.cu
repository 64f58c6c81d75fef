// lininit.cu — linear initialisation along the data's two principal components (vsom_linear_init, include/vsom_b200.h; not in
// the reference: SOM_PAK lininit, SOM Toolbox som_lininit).
//
//   co-moment pass   host rows stream through two device buffers in slabs of VSOM_LINEAR_INIT_SLAB_ROWS rows (the copy of slab
//                    s + 1 overlaps the pass over slab s).  Work items are (upper-triangle 64 x 64 tile, block of rows); each
//                    accumulates S2 = sum (x - x0)(x - x0)^T (and, on diagonal tiles, S1 = sum (x - x0)) of its rows in f64 and
//                    writes one partial tile; a second kernel adds the partial tiles in row-block order.  The partition follows
//                    D only, so the bits depend on the rows alone (never on the device).
//   eigen step       subspace iteration in f64 on p = min(D, 8) vectors: C V and the orthonormalisation on the device, the p x p
//                    Rayleigh-Ritz step on the host.
//   fill             the mean plane of the context's grid rows, and zero S, sigma, weight and hits.
//
// No reference parity constrains this path: products are fused on purpose (__fma_rn), every other operation is an explicit
// round-to-nearest intrinsic, so -fmad=false changes nothing here.
#include "common.cuh"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdint>
#include <numeric>

namespace vsom
{
namespace
{

constexpr int kTile = 64;                        // co-moment tile: 64 x 64 columns
constexpr int kTileSlot = kTile * kTile + kTile; // one tile's S2 block, then its 64 S1 entries (diagonal tiles; 0 elsewhere)
constexpr int kPassThreads = 256;                // 16 x 16 threads, 4 x 4 outputs each
constexpr int kRowChunk = 32;                    // rows staged in shared memory per step
constexpr int kPartialTiles = 2048;              // partial tiles per slab: row blocks per slab = clamp(2048 / tiles, 1, 64)
constexpr int kP = 8;                            // subspace block size (p = min(D, kP))
constexpr int kMaxIter = 300;                    // cap of the subspace iteration
constexpr double kTol = 1e-11;                   // stop when |C v_i - lambda_i v_i| <= kTol * lambda_1 for i = 1, 2
constexpr int kBlockThreads = 512;               // single-CTA kernels of the eigen step
constexpr int kRotateThreads = 256;              // ... the rotation (more registers per thread)

__host__ __device__ __forceinline__ int tile_index(int ti, int tj, int nt) { return ti * nt - ti * (ti - 1) / 2 + (tj - ti); }

// ---------------------------------------------------------------------------------------------------- co-moment pass

// partial[blockIdx.y][blockIdx.x]: S2 of tile blockIdx.x (upper triangle, row-major) and S1 of its columns, over the rows
// [blockIdx.y * blockRows, +blockRows) of this slab, each sum sequential in row order
__global__ void __launch_bounds__(kPassThreads) lininit_comoment_kernel(const float *__restrict__ x, int rows, int D, int nt, int blockRows,
                                                                        const double *__restrict__ x0, double *__restrict__ partial, int *flag)
{
    int t = blockIdx.x, ti = 0;
    while (t >= nt - ti)
    {
        t -= nt - ti;
        ++ti;
    }
    const int tj = ti + t;
    const bool diag = ti == tj;
    const int r0 = blockIdx.y * blockRows, r1 = min(rows, r0 + blockRows);
    __shared__ double As[kRowChunk][kTile], Bs[kRowChunk][kTile];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    double acc[4][4], s1[4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
    {
        s1[i] = 0.0;
#pragma unroll
        for (int j = 0; j < 4; ++j)
            acc[i][j] = 0.0;
    }
    bool bad = false;
    for (int rc = r0; rc < r1; rc += kRowChunk)
    {
        const int nr = min(kRowChunk, r1 - rc);
        for (int e = threadIdx.x; e < kRowChunk * kTile; e += kPassThreads)
        {
            const int r = e / kTile, c = e % kTile, ca = ti * kTile + c, cb = tj * kTile + c;
            double a = 0.0, b = 0.0;
            if (r < nr)
            {
                const float *row = x + static_cast<size_t>(rc + r) * D;
                if (ca < D)
                    a = __dsub_rn(static_cast<double>(row[ca]), x0[ca]);
                if (cb < D)
                {
                    const float v = row[cb];
                    bad |= !isfinite(v); // every column is some tile's j side
                    b = __dsub_rn(static_cast<double>(v), x0[cb]);
                }
            }
            As[r][c] = a;
            Bs[r][c] = b;
        }
        __syncthreads();
        for (int r = 0; r < nr; ++r)
        {
            double a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
            {
                a[i] = As[r][ty + 16 * i];
                b[i] = Bs[r][tx + 16 * i];
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    acc[i][j] = __fma_rn(a[i], b[j], acc[i][j]);
            if (diag && ty == 0)
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    s1[j] = __dadd_rn(s1[j], b[j]);
        }
        __syncthreads();
    }
    if (bad)
        *flag = 1;
    double *out = partial + (static_cast<size_t>(blockIdx.y) * gridDim.x + blockIdx.x) * kTileSlot;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j)
            out[(ty + 16 * i) * kTile + tx + 16 * j] = acc[i][j];
    if (ty == 0)
#pragma unroll
        for (int j = 0; j < 4; ++j)
            out[kTile * kTile + tx + 16 * j] = s1[j];
}

// acc += the nb partial tiles of one slab, added in row-block order
__global__ void lininit_reduce_kernel(const double *__restrict__ partial, int nb, size_t slots, double *__restrict__ acc)
{
    for (size_t e = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; e < slots; e += static_cast<size_t>(gridDim.x) * blockDim.x)
    {
        double s = partial[e];
        for (int b = 1; b < nb; ++b)
            s = __dadd_rn(s, partial[static_cast<size_t>(b) * slots + e]);
        acc[e] = __dadd_rn(acc[e], s);
    }
}

// mu = x0 + S1 / n and the full symmetric C = (S2 - S1 S1^T / n) / (n - 1) (element (i, j) from the upper-triangle entry)
__global__ void lininit_finish_kernel(const double *__restrict__ acc, int D, int nt, double n, const double *__restrict__ x0, double *__restrict__ mean,
                                      double *__restrict__ C)
{
    const size_t total = static_cast<size_t>(D) * D;
    for (size_t e = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; e < total; e += static_cast<size_t>(gridDim.x) * blockDim.x)
    {
        const int i = static_cast<int>(e / D), j = static_cast<int>(e % D), a = min(i, j), b = max(i, j);
        const double s2 = acc[static_cast<size_t>(tile_index(a / kTile, b / kTile, nt)) * kTileSlot + (a % kTile) * kTile + b % kTile];
        const double s1a = acc[static_cast<size_t>(tile_index(a / kTile, a / kTile, nt)) * kTileSlot + kTile * kTile + a % kTile];
        const double s1b = acc[static_cast<size_t>(tile_index(b / kTile, b / kTile, nt)) * kTileSlot + kTile * kTile + b % kTile];
        C[e] = __ddiv_rn(__dsub_rn(s2, __ddiv_rn(__dmul_rn(s1a, s1b), n)), __dsub_rn(n, 1.0));
        if (i == j)
            mean[i] = __dadd_rn(x0[i], __ddiv_rn(s1a, n));
    }
}

// ---------------------------------------------------------------------------------------------------- eigen step
// Blocks of vectors are D x kP, row-major (row i holds component i of the kP vectors); columns >= p are zero.

// W = C Q: one warp per row of C, lanes stride over k, partial sums combined by a fixed xor butterfly
__global__ void lininit_sym_times_kernel(const double *__restrict__ C, int D, const double *__restrict__ Q, double *__restrict__ W)
{
    const int row = static_cast<int>((static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (row >= D)
        return;
    double acc[kP];
#pragma unroll
    for (int j = 0; j < kP; ++j)
        acc[j] = 0.0;
    const double *c = C + static_cast<size_t>(row) * D;
    for (int k = lane; k < D; k += 32)
    {
        const double ck = c[k];
#pragma unroll
        for (int j = 0; j < kP; ++j)
            acc[j] = __fma_rn(ck, Q[static_cast<size_t>(k) * kP + j], acc[j]);
    }
#pragma unroll
    for (int j = 0; j < kP; ++j)
#pragma unroll
        for (int o = 16; o; o >>= 1)
            acc[j] = __dadd_rn(acc[j], __shfl_xor_sync(0xffffffffu, acc[j], o));
    if (lane == 0)
#pragma unroll
        for (int j = 0; j < kP; ++j)
            W[static_cast<size_t>(row) * kP + j] = acc[j];
}

// sums of K per-thread values over the CTA in a fixed order; every thread gets the K sums.  sm: 32 * K doubles.
template <int K>
__device__ __forceinline__ void block_sum(double (&v)[K], double *sm)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
#pragma unroll
    for (int j = 0; j < K; ++j)
#pragma unroll
        for (int o = 16; o; o >>= 1)
            v[j] = __dadd_rn(v[j], __shfl_xor_sync(0xffffffffu, v[j], o));
    if (lane == 0)
#pragma unroll
        for (int j = 0; j < K; ++j)
            sm[warp * K + j] = v[j];
    __syncthreads();
#pragma unroll
    for (int j = 0; j < K; ++j)
    {
        double s = sm[j];
        for (int w = 1; w < warps; ++w)
            s = __dadd_rn(s, sm[w * K + j]);
        v[j] = s;
    }
    __syncthreads();
}

// Q = an orthonormal basis of the p columns of Z: classical Gram-Schmidt applied twice per column.  A column that loses all but
// 1e-10 of its norm to the earlier ones (C of rank < p) is replaced by the first unit vector e_j, e_j+1, ... that does not.
__global__ void __launch_bounds__(kBlockThreads) lininit_orthonormalize_kernel(const double *__restrict__ Z, int D, int p, double *__restrict__ Q)
{
    __shared__ double sm[32 * kP];
    for (int e = threadIdx.x; e < D * kP; e += blockDim.x)
        Q[e] = e % kP < p ? Z[e] : 0.0;
    __syncthreads();
    for (int j = 0; j < p; ++j)
        for (int attempt = 0; attempt <= D; ++attempt)
        {
            if (attempt > 0)
            {
                const int unit = (j + attempt - 1) % D;
                for (int i = threadIdx.x; i < D; i += blockDim.x)
                    Q[i * kP + j] = i == unit ? 1.0 : 0.0;
                __syncthreads();
            }
            double before[1] = {0.0};
            for (int i = threadIdx.x; i < D; i += blockDim.x)
                before[0] = __fma_rn(Q[i * kP + j], Q[i * kP + j], before[0]);
            block_sum(before, sm);
            for (int pass = 0; pass < 2 && j > 0; ++pass)
            {
                double d[kP];
#pragma unroll
                for (int l = 0; l < kP; ++l)
                    d[l] = 0.0;
                for (int i = threadIdx.x; i < D; i += blockDim.x)
#pragma unroll
                    for (int l = 0; l < kP; ++l)
                        if (l < j)
                            d[l] = __fma_rn(Q[i * kP + l], Q[i * kP + j], d[l]);
                block_sum(d, sm);
                for (int i = threadIdx.x; i < D; i += blockDim.x)
                {
                    double q = Q[i * kP + j];
#pragma unroll
                    for (int l = 0; l < kP; ++l)
                        if (l < j)
                            q = __fma_rn(-d[l], Q[i * kP + l], q);
                    Q[i * kP + j] = q;
                }
                __syncthreads();
            }
            double after[1] = {0.0};
            for (int i = threadIdx.x; i < D; i += blockDim.x)
                after[0] = __fma_rn(Q[i * kP + j], Q[i * kP + j], after[0]);
            block_sum(after, sm);
            if (after[0] > 0.0 && after[0] > 1e-20 * before[0])
            {
                const double nrm = __dsqrt_rn(after[0]);
                for (int i = threadIdx.x; i < D; i += blockDim.x)
                    Q[i * kP + j] = __ddiv_rn(Q[i * kP + j], nrm);
                __syncthreads();
                break;
            }
        }
}

// H = Q^T W (kP x kP)
__global__ void __launch_bounds__(kBlockThreads) lininit_gram_kernel(const double *__restrict__ Q, const double *__restrict__ W, int D, double *__restrict__ H)
{
    __shared__ double sm[32 * kP];
    for (int l = 0; l < kP; ++l)
    {
        double h[kP];
#pragma unroll
        for (int m = 0; m < kP; ++m)
            h[m] = 0.0;
        for (int i = threadIdx.x; i < D; i += blockDim.x)
        {
            const double q = Q[i * kP + l];
#pragma unroll
            for (int m = 0; m < kP; ++m)
                h[m] = __fma_rn(q, W[i * kP + m], h[m]);
        }
        block_sum(h, sm);
        if (threadIdx.x == 0)
#pragma unroll
            for (int m = 0; m < kP; ++m)
                H[l * kP + m] = h[m];
    }
}

// Ritz vectors V = Q Y, Z = W Y (= C V, the next iteration's block) and res[m] = |Z_m - theta_m V_m|^2 for m = 0, 1
__global__ void __launch_bounds__(kRotateThreads) lininit_rotate_kernel(const double *__restrict__ Q, const double *__restrict__ W, int D,
                                                                       const double *__restrict__ Y, const double *__restrict__ theta, double *__restrict__ V,
                                                                       double *__restrict__ Z, double *__restrict__ res)
{
    __shared__ double sm[32 * 2];
    __shared__ double y[kP * kP];
    for (int e = threadIdx.x; e < kP * kP; e += blockDim.x)
        y[e] = Y[e];
    __syncthreads();
    const double t0 = theta[0], t1 = theta[1];
    double r[2] = {0.0, 0.0};
    for (int i = threadIdx.x; i < D; i += blockDim.x)
    {
        double q[kP], w[kP];
#pragma unroll
        for (int l = 0; l < kP; ++l)
        {
            q[l] = Q[i * kP + l];
            w[l] = W[i * kP + l];
        }
#pragma unroll
        for (int m = 0; m < kP; ++m)
        {
            double v = 0.0, z = 0.0;
#pragma unroll
            for (int l = 0; l < kP; ++l)
            {
                v = __fma_rn(q[l], y[l * kP + m], v);
                z = __fma_rn(w[l], y[l * kP + m], z);
            }
            V[i * kP + m] = v;
            Z[i * kP + m] = z;
            if (m < 2)
            {
                const double d = __fma_rn(-(m == 0 ? t0 : t1), v, z);
                r[m] = __fma_rn(d, d, r[m]);
            }
        }
    }
    block_sum(r, sm);
    if (threadIdx.x == 0)
    {
        res[0] = r[0];
        res[1] = r[1];
    }
}

// ---------------------------------------------------------------------------------------------------- fill

__global__ void lininit_fill_kernel(float *__restrict__ mean, float *__restrict__ S, float *__restrict__ sigma, float *__restrict__ weight, u64 *__restrict__ hits,
                                    int W, int H, int localRows, int shardBlock, int rank, int world, int Dm, int rowStride, const double *__restrict__ mu,
                                    const double *__restrict__ vx, const double *__restrict__ vy, double sx, double sy)
{
    const size_t total = static_cast<size_t>(localRows) * W * rowStride;
    for (size_t e = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; e < total; e += static_cast<size_t>(gridDim.x) * blockDim.x)
    {
        const size_t node = e / rowStride;
        const int k = static_cast<int>(e - node * rowStride), ly = static_cast<int>(node / W), gx = static_cast<int>(node - static_cast<size_t>(ly) * W);
        const int gy = shard_global_row(ly, shardBlock, rank, world);
        float m = 0.0f;
        if (k < Dm)
        {
            const double cx = W > 1 ? __ddiv_rn(static_cast<double>(2 * gx - (W - 1)), static_cast<double>(W - 1)) : 0.0;
            const double cy = H > 1 ? __ddiv_rn(static_cast<double>(2 * gy - (H - 1)), static_cast<double>(H - 1)) : 0.0;
            m = __double2float_rn(__dadd_rn(__dadd_rn(mu[k], __dmul_rn(__dmul_rn(cx, sx), vx[k])), __dmul_rn(__dmul_rn(cy, sy), vy[k])));
        }
        mean[e] = m;
        S[e] = 0.0f;
        sigma[e] = 0.0f;
        if (k == 0)
        {
            weight[node] = 0.0f;
            hits[node] = 0ull;
        }
    }
}

// ---------------------------------------------------------------------------------------------------- host side

// device buffers, the copy stream and its events of one call
struct Scratch
{
    vsom_ctx *ctx;
    std::vector<void *> bufs;
    cudaStream_t copy = nullptr;
    cudaEvent_t copied[2] = {}, consumed[2] = {};
    explicit Scratch(vsom_ctx *c) : ctx{c} {}
    ~Scratch()
    {
        cudaStreamSynchronize(ctx->stream);
        if (copy)
        {
            cudaStreamSynchronize(copy);
            cudaStreamDestroy(copy);
        }
        for (int i = 0; i < 2; ++i)
        {
            if (copied[i])
                cudaEventDestroy(copied[i]);
            if (consumed[i])
                cudaEventDestroy(consumed[i]);
        }
        for (void *p : bufs)
            cudaFree(p);
    }
    template <class T>
    int alloc(T *&p, size_t count)
    {
        void *q = nullptr;
        VSOM_CUDA(ctx, cudaMalloc(&q, sizeof(T) * std::max<size_t>(count, 1)));
        bufs.push_back(q);
        p = static_cast<T *>(q);
        return VSOM_OK;
    }
};

#define LININIT_TRY(expr)      \
    do                         \
    {                          \
        const int _rc = (expr); \
        if (_rc)               \
            return _rc;        \
    } while (0)

// eigenpairs of the symmetric p x p matrix A (cyclic Jacobi): theta in descending order (ties: lower index first), Y[l][m] the
// m-th eigenvector
void small_symmetric_eigen(int p, const double (&Ain)[kP][kP], double (&theta)[kP], double (&Y)[kP][kP])
{
    double A[kP][kP], V[kP][kP];
    double total = 0.0;
    for (int i = 0; i < kP; ++i)
        for (int j = 0; j < kP; ++j)
        {
            A[i][j] = i < p && j < p ? 0.5 * (Ain[i][j] + Ain[j][i]) : 0.0;
            V[i][j] = i == j ? 1.0 : 0.0;
            total += A[i][j] * A[i][j];
        }
    for (int sweep = 0; sweep < 100; ++sweep)
    {
        double off = 0.0;
        for (int i = 0; i < p; ++i)
            for (int j = i + 1; j < p; ++j)
                off += A[i][j] * A[i][j];
        if (off <= 1e-34 * total)
            break;
        for (int a = 0; a < p; ++a)
            for (int b = a + 1; b < p; ++b)
            {
                if (A[a][b] == 0.0)
                    continue;
                const double th = (A[b][b] - A[a][a]) / (2.0 * A[a][b]);
                const double t = (th >= 0 ? 1.0 : -1.0) / (std::fabs(th) + std::sqrt(th * th + 1.0));
                const double c = 1.0 / std::sqrt(t * t + 1.0), s = t * c;
                for (int k = 0; k < p; ++k)
                {
                    const double ka = A[k][a], kb = A[k][b];
                    A[k][a] = c * ka - s * kb;
                    A[k][b] = s * ka + c * kb;
                }
                for (int k = 0; k < p; ++k)
                {
                    const double ak = A[a][k], bk = A[b][k];
                    A[a][k] = c * ak - s * bk;
                    A[b][k] = s * ak + c * bk;
                }
                for (int k = 0; k < p; ++k)
                {
                    const double ka = V[k][a], kb = V[k][b];
                    V[k][a] = c * ka - s * kb;
                    V[k][b] = s * ka + c * kb;
                }
            }
    }
    int idx[kP];
    std::iota(idx, idx + kP, 0);
    std::stable_sort(idx, idx + p, [&](int a, int b) { return A[a][a] > A[b][b]; });
    for (int m = 0; m < kP; ++m)
    {
        theta[m] = m < p ? A[idx[m]][idx[m]] : 0.0;
        for (int l = 0; l < kP; ++l)
            Y[l][m] = m < p ? V[l][idx[m]] : 0.0;
    }
}

// the sign rule: the component of largest magnitude is positive (lowest index among equal magnitudes)
void orient(std::vector<double> &v)
{
    size_t best = 0;
    for (size_t k = 1; k < v.size(); ++k)
        if (std::fabs(v[k]) > std::fabs(v[best]))
            best = k;
    if (v[best] < 0.0)
        for (double &c : v)
            c = -c;
}

// the pseudo-random but fixed start block: a hash of (row, column), values in [-1, 1)
double start_value(int i, int j)
{
    uint64_t z = static_cast<uint64_t>(i) * kP + static_cast<uint64_t>(j) + 0x9e3779b97f4a7c15ull;
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    z ^= z >> 31;
    return static_cast<double>(z >> 11) * 0x1.0p-52 - 1.0;
}

double ms_since(std::chrono::steady_clock::time_point t0)
{
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
}

} // namespace

int linear_init_fit(vsom_ctx *ctx, const float *x, size_t n, LinearFit &fit)
{
    const auto t0 = std::chrono::steady_clock::now();
    const int D = ctx->Din;
    const int nt = (D + kTile - 1) / kTile, tiles = nt * (nt + 1) / 2;
    const size_t slots = static_cast<size_t>(tiles) * kTileSlot;
    const int blocksPerSlab = std::max(1, std::min(64, kPartialTiles / tiles));
    const size_t slabRows = VSOM_LINEAR_INIT_SLAB_ROWS;
    const size_t perBlock = (slabRows + blocksPerSlab - 1) / blocksPerSlab; // a slab never needs more than blocksPerSlab blocks
    const int blockRows = static_cast<int>((perBlock + kRowChunk - 1) / kRowChunk * kRowChunk);
    const int p = std::min(D, kP);
    cudaStream_t st = ctx->stream;

    Scratch sc(ctx);
    float *stage[2];
    double *partial, *acc, *x0, *mean, *C, *blk[5], *H, *Y, *theta, *res;
    int *flag;
    for (float *&s : stage)
        LININIT_TRY(sc.alloc(s, slabRows * D));
    LININIT_TRY(sc.alloc(partial, slots * blocksPerSlab));
    LININIT_TRY(sc.alloc(acc, slots));
    LININIT_TRY(sc.alloc(x0, D));
    LININIT_TRY(sc.alloc(mean, D));
    LININIT_TRY(sc.alloc(C, static_cast<size_t>(D) * D));
    for (double *&b : blk)
        LININIT_TRY(sc.alloc(b, static_cast<size_t>(D) * kP));
    LININIT_TRY(sc.alloc(H, kP * kP));
    LININIT_TRY(sc.alloc(Y, kP * kP));
    LININIT_TRY(sc.alloc(theta, kP));
    LININIT_TRY(sc.alloc(res, 2));
    LININIT_TRY(sc.alloc(flag, 1));
    VSOM_CUDA(ctx, cudaStreamCreateWithFlags(&sc.copy, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i)
    {
        VSOM_CUDA(ctx, cudaEventCreateWithFlags(&sc.copied[i], cudaEventDisableTiming));
        VSOM_CUDA(ctx, cudaEventCreateWithFlags(&sc.consumed[i], cudaEventDisableTiming));
    }

    // ---- co-moment pass, shifted by the first row
    std::vector<double> hx0(x, x + D);
    VSOM_CUDA(ctx, cudaMemcpyAsync(x0, hx0.data(), sizeof(double) * D, cudaMemcpyHostToDevice, st));
    VSOM_CUDA(ctx, cudaMemsetAsync(acc, 0, sizeof(double) * slots, st));
    VSOM_CUDA(ctx, cudaMemsetAsync(flag, 0, sizeof(int), st));
    VSOM_CUDA(ctx, cudaStreamSynchronize(st)); // the copy stream starts after these
    const size_t slabs = (n + slabRows - 1) / slabRows;
    for (size_t s = 0; s < slabs; ++s)
    {
        const int b = static_cast<int>(s & 1);
        const size_t rows = std::min(slabRows, n - s * slabRows);
        if (s >= 2)
            VSOM_CUDA(ctx, cudaStreamWaitEvent(sc.copy, sc.consumed[b], 0));
        VSOM_CUDA(ctx, cudaMemcpyAsync(stage[b], x + s * slabRows * D, sizeof(float) * rows * D, cudaMemcpyHostToDevice, sc.copy));
        VSOM_CUDA(ctx, cudaEventRecord(sc.copied[b], sc.copy));
        VSOM_CUDA(ctx, cudaStreamWaitEvent(st, sc.copied[b], 0));
        const int nb = static_cast<int>((rows + blockRows - 1) / blockRows);
        lininit_comoment_kernel<<<dim3(tiles, nb), kPassThreads, 0, st>>>(stage[b], static_cast<int>(rows), D, nt, blockRows, x0, partial, flag);
        VSOM_CUDA(ctx, cudaGetLastError());
        const int rg = static_cast<int>(std::min<size_t>((slots + 255) / 256, 4096));
        lininit_reduce_kernel<<<rg, 256, 0, st>>>(partial, nb, slots, acc);
        VSOM_CUDA(ctx, cudaGetLastError());
        VSOM_CUDA(ctx, cudaEventRecord(sc.consumed[b], st));
        ctx->launches += 2;
    }
    {
        const size_t total = static_cast<size_t>(D) * D;
        const int fg = static_cast<int>(std::min<size_t>((total + 255) / 256, 8192));
        lininit_finish_kernel<<<fg, 256, 0, st>>>(acc, D, nt, static_cast<double>(n), x0, mean, C);
        VSOM_CUDA(ctx, cudaGetLastError());
        ++ctx->launches;
    }
    int hflag = 0;
    fit.mean.assign(D, 0.0);
    VSOM_CUDA(ctx, cudaMemcpyAsync(&hflag, flag, sizeof(int), cudaMemcpyDeviceToHost, st));
    VSOM_CUDA(ctx, cudaMemcpyAsync(fit.mean.data(), mean, sizeof(double) * D, cudaMemcpyDeviceToHost, st));
    VSOM_CUDA(ctx, cudaStreamSynchronize(st));
    if (hflag)
        return set_error(ctx, VSOM_ERR_INVALID, "vsom_linear_init: the rows hold a non-finite value");
    ctx->linInitPhase[0] = ms_since(t0);

    // ---- top two eigenpairs
    const auto t1 = std::chrono::steady_clock::now();
    fit.axis1.assign(D, 0.0);
    fit.axis2.assign(D, 0.0);
    int iterations = 0;
    if (D == 1)
    {
        double c00 = 0.0;
        VSOM_CUDA(ctx, cudaMemcpyAsync(&c00, C, sizeof(double), cudaMemcpyDeviceToHost, st));
        VSOM_CUDA(ctx, cudaStreamSynchronize(st));
        fit.lambda[0] = std::max(c00, 0.0);
        fit.lambda[1] = 0.0;
        fit.axis1[0] = 1.0;
    }
    else
    {
        double *Qd = blk[0], *Wd = blk[1], *Vd = blk[2], *Zd = blk[3], *V0 = blk[4];
        std::vector<double> hv(static_cast<size_t>(D) * kP, 0.0);
        for (int i = 0; i < D; ++i)
            for (int j = 0; j < p; ++j)
                hv[static_cast<size_t>(i) * kP + j] = start_value(i, j);
        VSOM_CUDA(ctx, cudaMemcpyAsync(V0, hv.data(), sizeof(double) * hv.size(), cudaMemcpyHostToDevice, st));
        const int mg = (D * 32 + 255) / 256;
        lininit_sym_times_kernel<<<mg, 256, 0, st>>>(C, D, V0, Zd);
        VSOM_CUDA(ctx, cudaGetLastError());
        ++ctx->launches;
        double hH[kP][kP], th[kP], hY[kP][kP], hres[2];
        for (;;)
        {
            ++iterations;
            lininit_orthonormalize_kernel<<<1, kBlockThreads, 0, st>>>(Zd, D, p, Qd);
            lininit_sym_times_kernel<<<mg, 256, 0, st>>>(C, D, Qd, Wd);
            lininit_gram_kernel<<<1, kBlockThreads, 0, st>>>(Qd, Wd, D, H);
            VSOM_CUDA(ctx, cudaGetLastError());
            VSOM_CUDA(ctx, cudaMemcpyAsync(hH, H, sizeof(hH), cudaMemcpyDeviceToHost, st));
            VSOM_CUDA(ctx, cudaStreamSynchronize(st));
            small_symmetric_eigen(p, hH, th, hY);
            VSOM_CUDA(ctx, cudaMemcpyAsync(Y, hY, sizeof(hY), cudaMemcpyHostToDevice, st));
            VSOM_CUDA(ctx, cudaMemcpyAsync(theta, th, sizeof(th), cudaMemcpyHostToDevice, st));
            lininit_rotate_kernel<<<1, kRotateThreads, 0, st>>>(Qd, Wd, D, Y, theta, Vd, Zd, res);
            VSOM_CUDA(ctx, cudaGetLastError());
            ctx->launches += 4;
            VSOM_CUDA(ctx, cudaMemcpyAsync(hres, res, sizeof(hres), cudaMemcpyDeviceToHost, st));
            VSOM_CUDA(ctx, cudaStreamSynchronize(st));
            const double bound = kTol * std::max(th[0], 0.0);
            if ((std::sqrt(hres[0]) <= bound && std::sqrt(hres[1]) <= bound) || iterations >= kMaxIter)
                break;
        }
        std::vector<double> hV(static_cast<size_t>(D) * kP);
        VSOM_CUDA(ctx, cudaMemcpyAsync(hV.data(), Vd, sizeof(double) * hV.size(), cudaMemcpyDeviceToHost, st));
        VSOM_CUDA(ctx, cudaStreamSynchronize(st));
        for (int i = 0; i < D; ++i)
        {
            fit.axis1[i] = hV[static_cast<size_t>(i) * kP];
            fit.axis2[i] = hV[static_cast<size_t>(i) * kP + 1];
        }
        fit.lambda[0] = std::max(th[0], 0.0);
        fit.lambda[1] = std::max(th[1], 0.0);
        orient(fit.axis1);
        orient(fit.axis2);
    }
    ctx->linInitPhase[1] = ms_since(t1);
    ctx->linInitPhase[3] = iterations;
    return VSOM_OK;
}

int launch_linear_fill(vsom_ctx *ctx, const LinearFit &fit)
{
    const auto t0 = std::chrono::steady_clock::now();
    const int D = ctx->Din;
    // the first axis runs along the longer side of the grid
    const bool wide = ctx->W >= ctx->H;
    const std::vector<double> &vx = wide ? fit.axis1 : fit.axis2, &vy = wide ? fit.axis2 : fit.axis1;
    const double sx = std::sqrt(fit.lambda[wide ? 0 : 1]), sy = std::sqrt(fit.lambda[wide ? 1 : 0]);
    Scratch sc(ctx);
    double *dev;
    LININIT_TRY(sc.alloc(dev, 3 * static_cast<size_t>(D)));
    std::vector<double> h(fit.mean);
    h.insert(h.end(), vx.begin(), vx.end());
    h.insert(h.end(), vy.begin(), vy.end());
    VSOM_CUDA(ctx, cudaMemcpyAsync(dev, h.data(), sizeof(double) * h.size(), cudaMemcpyHostToDevice, ctx->stream));
    const size_t total = static_cast<size_t>(ctx->localN) * ctx->rowStride;
    const int grid = static_cast<int>(std::min<size_t>((total + 255) / 256, 16384));
    lininit_fill_kernel<<<grid, 256, 0, ctx->stream>>>(ctx->mean, ctx->S, ctx->sigma, ctx->weight, ctx->hits, ctx->W, ctx->H, ctx->localRows, ctx->shardBlock,
                                                       ctx->rank, ctx->world, ctx->Dm, ctx->rowStride, dev, dev + D, dev + 2 * D, sx, sy);
    VSOM_CUDA(ctx, cudaGetLastError());
    ++ctx->launches;
    VSOM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->linInitPhase[2] = ms_since(t0);
    return VSOM_OK;
}

} // namespace vsom
