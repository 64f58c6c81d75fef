// som_index.cu — K5: the "SomIndex build": histogram of BMU ids and rows grouped by BMU.
//
// Replaces what Som::addBmu accumulates over a pass (src/Som.cpp:1189-1192: bmuHits[y*W+x]++) and the
// per-neuron row sets the batch trainer scans (src/Som.cpp:845-868): counts[N], offsets[N+1] (exclusive
// prefix sum) and row_ids[n] = the rows of each BMU in ascending row order.
//
// Integer work, bit-exact by construction: a stable least-significant-digit radix sort of (bmu, row) on
// 8-bit digits — per-CTA digit histograms, one exclusive scan over the (digit, CTA) table, and a stable
// scatter that ranks equal digits inside a warp with __match_any_sync — so that equal BMUs keep row order.
#include "common.cuh"
#include <algorithm>

namespace vsom
{

constexpr int kSortThreads = 256;
constexpr int kSortItems = 8;                          // rounds of 256 consecutive items per CTA
constexpr int kSortChunk = kSortThreads * kSortItems;  // 2048 rows per CTA

__global__ void index_hist_kernel(const unsigned *__restrict__ bmu, u64 n, int N, u64 *__restrict__ counts, int *__restrict__ bad)
{
    const u64 stride = static_cast<u64>(gridDim.x) * blockDim.x;
    for (u64 r = static_cast<u64>(blockIdx.x) * blockDim.x + threadIdx.x; r < n; r += stride)
    {
        const unsigned k = bmu[r];
        if (k < static_cast<unsigned>(N))
            atomicAdd(counts + k, 1ull);
        else
            *bad = 1;
    }
}

// the same histogram with a CTA-private copy in shared memory (maps of up to 24 576 nodes): 16.8 M global 64-bit atomics on 16 384
// addresses took 313 us (L2 atomic throughput); shared-memory atomics + one flush per CTA and bin do not
__global__ void __launch_bounds__(1024) index_hist_smem_kernel(const unsigned *__restrict__ bmu, u64 n, int N, u64 *__restrict__ counts, int *__restrict__ bad)
{
    extern __shared__ unsigned histS[];
    for (int k = threadIdx.x; k < N; k += blockDim.x)
        histS[k] = 0u;
    __syncthreads();
    const u64 stride = static_cast<u64>(gridDim.x) * blockDim.x;
    bool anyBad = false;
    for (u64 r = static_cast<u64>(blockIdx.x) * blockDim.x + threadIdx.x; r < n; r += stride)
    {
        const unsigned k = bmu[r];
        if (k < static_cast<unsigned>(N))
            atomicAdd(histS + k, 1u);
        else
            anyBad = true;
    }
    if (anyBad)
        *bad = 1;
    __syncthreads();
    for (int k = threadIdx.x; k < N; k += blockDim.x)
    {
        const unsigned c = histS[k];
        if (c)
            atomicAdd(counts + k, static_cast<u64>(c));
    }
}

// exclusive scan of counts[N] into offsets[N+1]; one CTA, each thread owns a contiguous run
__global__ void __launch_bounds__(1024) index_scan_kernel(const u64 *__restrict__ counts, int N, u64 *__restrict__ offsets)
{
    __shared__ u64 part[1024];
    const int tid = threadIdx.x;
    const int per = (N + 1023) / 1024;
    const int lo = tid * per, hi = lo + per < N ? lo + per : N;
    u64 s = 0;
    for (int k = lo; k < hi; ++k)
        s += counts[k];
    part[tid] = s;
    __syncthreads();
    if (tid == 0)
    {
        u64 run = 0;
        for (int q = 0; q < 1024; ++q)
        {
            const u64 v = part[q];
            part[q] = run;
            run += v;
        }
        offsets[N] = run;
    }
    __syncthreads();
    u64 run = part[tid];
    for (int k = lo; k < hi; ++k)
    {
        offsets[k] = run;
        run += counts[k];
    }
}

// pass 1 of a radix pass: digit histogram of each CTA's chunk -> table[digit * nblocks + block]
__global__ void __launch_bounds__(kSortThreads) radix_hist_kernel(const unsigned *__restrict__ keys, u64 n, int shift, unsigned *__restrict__ table, unsigned nblocks)
{
    __shared__ unsigned h[256];
    h[threadIdx.x] = 0;
    __syncthreads();
    const u64 base = static_cast<u64>(blockIdx.x) * kSortChunk;
    for (int it = 0; it < kSortItems; ++it)
    {
        const u64 r = base + static_cast<u64>(it) * kSortThreads + threadIdx.x;
        if (r < n)
            atomicAdd(&h[(keys[r] >> shift) & 0xff], 1u);
    }
    __syncthreads();
    table[static_cast<size_t>(threadIdx.x) * nblocks + blockIdx.x] = h[threadIdx.x];
}

// Exclusive scan over the whole (digit-major) table in three coalesced steps (one CTA walking 2M entries with a stride of
// 2048 between its threads took 3.5 ms per pass): chunk sums, a one-CTA scan of the chunk sums, chunk-local scans.
constexpr int kScanChunk = 4096; // entries per CTA: 256 threads x 16

__global__ void __launch_bounds__(256) scan_chunk_sums_kernel(const unsigned *__restrict__ table, u64 len, unsigned *__restrict__ sums)
{
    __shared__ unsigned w[8];
    const u64 base = static_cast<u64>(blockIdx.x) * kScanChunk;
    unsigned s = 0;
    for (int i = threadIdx.x; i < kScanChunk; i += 256)
        if (base + i < len)
            s += table[base + i];
    for (int o = 16; o; o >>= 1)
        s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0)
        w[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0)
        sums[blockIdx.x] = w[0] + w[1] + w[2] + w[3] + w[4] + w[5] + w[6] + w[7];
}

// one CTA: exclusive scan of the chunk sums in place (each thread a contiguous run, then the 1024 partials serially)
__global__ void __launch_bounds__(1024) scan_sums_kernel(unsigned *__restrict__ sums, unsigned count)
{
    __shared__ unsigned part[1024];
    const int tid = threadIdx.x;
    const unsigned per = (count + 1023) / 1024, lo = tid * per, hi = lo + per < count ? lo + per : count;
    unsigned s = 0;
    for (unsigned q = lo; q < hi; ++q)
        s += sums[q];
    part[tid] = s;
    __syncthreads();
    if (tid == 0)
    {
        unsigned run = 0;
        for (int q = 0; q < 1024; ++q)
        {
            const unsigned v = part[q];
            part[q] = run;
            run += v;
        }
    }
    __syncthreads();
    unsigned run = part[tid];
    for (unsigned q = lo; q < hi; ++q)
    {
        const unsigned v = sums[q];
        sums[q] = run;
        run += v;
    }
}

// every CTA scans its chunk (thread t owns the 16 consecutive entries 16 t .. 16 t + 15) and adds the chunk's offset
__global__ void __launch_bounds__(256) scan_chunks_kernel(unsigned *__restrict__ table, u64 len, const unsigned *__restrict__ sums)
{
    __shared__ unsigned w[8];
    const u64 base = static_cast<u64>(blockIdx.x) * kScanChunk + static_cast<u64>(threadIdx.x) * 16;
    unsigned v[16], s = 0;
#pragma unroll
    for (int i = 0; i < 16; ++i)
    {
        v[i] = base + i < len ? table[base + i] : 0u;
        s += v[i];
    }
    unsigned inc = s; // inclusive scan of the threads' sums inside the warp
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
    {
        const unsigned u = __shfl_up_sync(0xffffffffu, inc, o);
        if ((threadIdx.x & 31) >= o)
            inc += u;
    }
    if ((threadIdx.x & 31) == 31)
        w[threadIdx.x >> 5] = inc;
    __syncthreads();
    unsigned run = sums[blockIdx.x] + inc - s;
    for (int q = 0; q < (threadIdx.x >> 5); ++q)
        run += w[q];
#pragma unroll
    for (int i = 0; i < 16; ++i)
        if (base + i < len)
        {
            table[base + i] = run;
            run += v[i];
        }
}

// pass 2: stable scatter.  Items are taken in rounds of 256 consecutive rows; inside a round the rank of an
// item among equal digits is (items of that digit in lower warps) + (lower lanes of its own warp).
__global__ void __launch_bounds__(kSortThreads) radix_scatter_kernel(const unsigned *__restrict__ keysIn, const unsigned *__restrict__ valsIn, u64 n,
                                                                      int shift, const unsigned *__restrict__ table, unsigned nblocks,
                                                                      unsigned *__restrict__ keysOut, unsigned *__restrict__ valsOut, int firstPass)
{
    __shared__ unsigned base[256];                       // running output position per digit
    __shared__ unsigned warpCnt[kSortThreads / 32][256]; // per round: items of each digit in each warp
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    base[tid] = table[static_cast<size_t>(tid) * nblocks + blockIdx.x];
    const u64 chunk0 = static_cast<u64>(blockIdx.x) * kSortChunk;
    for (int it = 0; it < kSortItems; ++it)
    {
        for (int w = 0; w < kSortThreads / 32; ++w)
            warpCnt[w][tid] = 0;
        __syncthreads();
        const u64 r = chunk0 + static_cast<u64>(it) * kSortThreads + tid;
        const bool valid = r < n;
        unsigned key = 0, val = 0, digit = 0, rankInWarp = 0;
        if (valid)
        {
            key = keysIn[r];
            val = firstPass ? static_cast<unsigned>(r) : valsIn[r];
            digit = (key >> shift) & 0xff;
        }
        // invalid lanes use a digit outside 0..255 so they never match a valid lane
        const unsigned peers = __match_any_sync(0xffffffffu, valid ? digit : 0x100u + lane);
        if (valid)
        {
            rankInWarp = __popc(peers & ((1u << lane) - 1u));
            if (rankInWarp == 0)
                warpCnt[warp][digit] = __popc(peers);
        }
        __syncthreads();
        // thread d turns the per-warp counts of digit d into exclusive prefixes and advances base[d]
        {
            unsigned run = base[tid];
            for (int w = 0; w < kSortThreads / 32; ++w)
            {
                const unsigned c = warpCnt[w][tid];
                warpCnt[w][tid] = run;
                run += c;
            }
            base[tid] = run;
        }
        __syncthreads();
        if (valid)
        {
            const unsigned pos = warpCnt[warp][digit] + rankInWarp;
            if (keysOut)
                keysOut[pos] = key;
            valsOut[pos] = val;
        }
        __syncthreads();
    }
}

int launch_offsets_scan(vsom_ctx *ctx, const u64 *countsDev, int count, u64 *offsetsDev)
{
    index_scan_kernel<<<1, 1024, 0, ctx->stream>>>(countsDev, count, offsetsDev);
    ctx->launches += 1;
    VSOM_CUDA(ctx, cudaGetLastError());
    return VSOM_OK;
}

int launch_build_index(vsom_ctx *ctx, const unsigned *bmuDev, size_t n, int bins, u64 *countsDev, u64 *offsetsDev, unsigned *rowIdsDev)
{
    const int N = bins;
    if (n >= (1ull << 32))
        return set_error(ctx, VSOM_ERR_INVALID, "build_index: row ids are 32-bit; split the pass");
    // counts + offsets
    VSOM_CUDA(ctx, cudaMemsetAsync(countsDev, 0, sizeof(u64) * N, ctx->stream));
    VSOM_CUDA(ctx, cudaMemsetAsync(ctx->errFlag, 0, sizeof(int), ctx->stream));
    if (n > 0)
    {
        const size_t histBytes = sizeof(unsigned) * static_cast<size_t>(N);
        if (histBytes <= 96 * 1024 && n >= (1u << 16))
        {
            // one CTA per SM, each with its own shared-memory histogram (a CTA sees at most n / numSMs + 1024 rows: 32-bit counts)
            VSOM_CUDA(ctx, cudaFuncSetAttribute(index_hist_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(histBytes)));
            index_hist_smem_kernel<<<static_cast<unsigned>(ctx->numSMs), 1024, histBytes, ctx->stream>>>(bmuDev, n, N, countsDev, ctx->errFlag);
        }
        else
        {
            const unsigned grid = static_cast<unsigned>(std::min<size_t>((n + 255) / 256, static_cast<size_t>(ctx->numSMs) * 8));
            index_hist_kernel<<<grid, 256, 0, ctx->stream>>>(bmuDev, n, N, countsDev, ctx->errFlag);
        }
        ctx->launches += 1;
    }
    int rc = launch_offsets_scan(ctx, countsDev, N, offsetsDev);
    if (rc)
        return rc;
    if (n == 0 || !rowIdsDev)
        return VSOM_OK;

    // stable LSD radix sort of (bmu, row)
    int bits = 1;
    while ((1ll << bits) < N)
        ++bits;
    const int passes = (bits + 7) / 8;
    const unsigned nblocks = static_cast<unsigned>((n + kSortChunk - 1) / kSortChunk);
    const size_t tableLen = static_cast<size_t>(256) * nblocks;
    const unsigned scanChunks = static_cast<unsigned>((tableLen + kScanChunk - 1) / kScanChunk);
    rc = stage_reserve(ctx, 3, sizeof(unsigned) * (tableLen + scanChunks + 64));
    if (rc)
        return rc;
    rc = stage_reserve(ctx, 4, sizeof(unsigned) * n * 3); // keys ping, keys pong, vals pong
    if (rc)
        return rc;
    unsigned *table = static_cast<unsigned *>(ctx->stage[3]);
    unsigned *keysA = static_cast<unsigned *>(ctx->stage[4]);
    unsigned *keysB = keysA + n;
    unsigned *valsB = keysB + n;
    // the final pass must land in rowIdsDev: passes alternate (valsB, rowIdsDev) so that the last one does
    const unsigned *kin = bmuDev;
    const unsigned *vin = nullptr;
    for (int pass = 0; pass < passes; ++pass)
    {
        const bool last = pass == passes - 1;
        const bool toRow = ((passes - 1 - pass) % 2) == 0;
        unsigned *vout = toRow ? rowIdsDev : valsB;
        unsigned *kout = last ? nullptr : ((pass % 2) == 0 ? keysA : keysB);
        radix_hist_kernel<<<nblocks, kSortThreads, 0, ctx->stream>>>(kin, n, 8 * pass, table, nblocks);
        scan_chunk_sums_kernel<<<scanChunks, 256, 0, ctx->stream>>>(table, tableLen, table + tableLen);
        scan_sums_kernel<<<1, 1024, 0, ctx->stream>>>(table + tableLen, scanChunks);
        scan_chunks_kernel<<<scanChunks, 256, 0, ctx->stream>>>(table, tableLen, table + tableLen);
        radix_scatter_kernel<<<nblocks, kSortThreads, 0, ctx->stream>>>(kin, vin, n, 8 * pass, table, nblocks, kout, vout, pass == 0 ? 1 : 0);
        ctx->launches += 5;
        kin = kout;
        vin = vout;
    }
    VSOM_CUDA(ctx, cudaGetLastError());
    return VSOM_OK;
}

} // namespace vsom
