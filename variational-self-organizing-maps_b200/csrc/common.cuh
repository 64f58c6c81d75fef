// common.cuh — context, error plumbing and device helpers shared by the sm_100a kernels of libvsom_b200.so.
//
// Arithmetic rule for every kernel in this library: the reference CPU build has no FMA (build/Makefile:18,
// -msse2 only), so each float/double operation on a parity path is written with an explicit round-to-nearest
// intrinsic (__fadd_rn, __fmul_rn, __fsub_rn, __fdiv_rn, __fsqrt_rn, __dadd_rn, ...) that nvcc never
// contracts or reassociates; the library is additionally compiled with -fmad=false.
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <cmath>
#include <string>
#include <vector>

#include "vsom_b200.h"

namespace vsom
{

typedef unsigned long long u64;

// CUDA's limit on gridDim.y (and z): launchers that put rows or tiles on y launch longer ranges in pieces of this size
constexpr size_t kMaxGridY = 65535;

// One neighbourhood-table entry per (|dy|, |dx|): Som::calculateNeighbourhoodWeight (src/Som.cpp:949-975)
// evaluated on the host with the same libm exp() the reference calls, then pre-rounded the way
// Som::trainSingle uses it (src/Som.cpp:922-941).
struct LutEntry
{
    double nw;  // neighbourhood weight (f64)
    float cexp; // (float)(nw * eta)  — Exponential decay: added to weightMap and multiplies the step
    float nwf;  // (float)nw          — multiplies the Welford term; added to weightMap in InverseProportional
};

// Som::calculateNeighbourhoodWeight (src/Som.cpp:949-975) of a node (dx, dy) cells from the BMU, with the division order of
// :962-963 and the host libm exp() the reference calls (the host code is compiled with -ffp-contract=off)
inline double neighbourhood_weight(int dx, int dy, double sigma)
{
    if (sigma > 1.0)
    {
        const double ddx = static_cast<double>(dx), ddy = static_cast<double>(dy);
        return std::exp(-(ddx * ddx / 2.0 / sigma / sigma + ddy * ddy / 2.0 / sigma / sigma));
    }
    return (dx == 0 && dy == 0) ? 1.0 : 0.0;
}

struct StepParams
{
    int W, H;                 // full grid
    int node0, nodeCount;     // nodes held by this device (node0 is 0; sharded contexts map local <-> global with shard_*_node below)
    int shardBlock;           // node-sharded contexts: grid rows are dealt to the ranks round-robin in blocks of this many rows
    int Din, Dm, Dr, P;       // sample length, model length, residual length (Dm or P), CLR pair count
    int rowStride;            // floats between rows of the global planes
    float *mean, *S, *sigma, *weight;
    u64 *hits;
    const float *x;           // n x Din samples (device)
    u64 n;
    int decay;
    double radius;            // 2.5 * sigma (src/Som.cpp:899-903)
    const LutEntry *lut;
    int lutW;
    const unsigned short *pairI, *pairJ; // CLR pair tables (src/Transformation.cpp:94-101)
    u64 *slots;               // [2][G][pitch] min-loc exchange: slots[buffer][destination CTA][source CTA]
    int *err;                 // set to 1 when a CTA gave up waiting
    unsigned *outBmu;         // per sample, may be null
    float *outDist;           // per sample, may be null
    int resident;             // planes of the owned nodes live in shared memory for the whole chunk
    int smStride;             // row stride (floats) of the resident copy
    long long timeoutCycles, peerTimeoutCycles; // waiting for a CTA of this launch / for another rank's launch
    int lutSmem, lutCount;    // copy the table into shared memory (it fits behind the resident rows)
    int xVec;                 // sample rows are 16-byte aligned: 16-byte cp.async
    int order;                // vsom_reduction_order of the distances
    int lanesPerNode;         // K1F: lanes that share one node's distance chain (1, or 8 in the Eigen order)
    int world, rank;          // node-sharded training across GPUs (world == 1: single GPU)
    u64 *rankSlots;           // [2][world] keys pushed into THIS GPU's memory by every rank (peer stores over NVLink)
    u64 *peerSlots[8];        // rankSlots of every rank (index = rank), peer-mapped; peerSlots[rank] == rankSlots
    u64 stepBase;             // samples trained before this launch: the cross-GPU exchange is indexed by the global step
    int localSearch;          // sigma <= 1: BMU by the reference's greedy local walk (findLocalBmu) instead of the global argmin
    float *distBuf;           // [2][nodeCount] per-step distances of every node (local search only)
    const u64 *lastIn;        // per-sample start node of the walk (DataSet::lastBMU), null = 0
    long long *prof;          // optional [gridDim.x][5] per-phase cycle sums of thread 0 (diagnostics), else null
    const unsigned *winTab;   // K1F: [W + H] update window per BMU column / row, start | end << 16 (src/Som.cpp:899-903)
    // K1F exchange rows, placed by L2 die (online_step_fast.cu, "L2 die calibration")
    const int *dieOfSm;       // [256] die of an SM id
    const int *rowBlocks;     // [2 dies][160 slots][2 buffers] 2 KB block of the row pool
    int *rowOf;               // [G] row (die * 160 + slot) every CTA claimed in this launch
    unsigned *rowCtr;         // [0..1] rows claimed per die, [2] arrivals at the one-off grid barrier
    u64 *rowPool;
    int pollDelay;            // cycles between the pushes and the first poll: 0 in every launch (without the wait, ptxas gives K1F's PROF builds a register more)
    u64 *distTag;             // K1F, sigma <= 1: [2][N] (distance bits << 32 | step + 1) of every node, self-validating words
    int scanBufs, scanSeg, scanNSeg; // K1 on HBM-resident rows: streamed scan (ring of scanBufs buffers of 32 row segments of scanSeg floats)
    const void *scanMap;      // ... its TMA descriptor of the mean plane (device memory)
};

// How one online-step kernel is launched on a context: K1 (online_step.cu) is always configured, K1F (online_step_fast.cu)
// only where it is eligible.  Both are fixed at vsom_create; launch_online_step picks one per chunk.
struct StepPlan
{
    void (*kernel[2])(const StepParams) = {}; // [profiling]: K1F has a profiled instantiation, K1 tests p.prof at run time
    int grid = 0;                             // CTAs; 0: the kernel is not configured on this context
    int threads = 0;
    size_t smem = 0;                          // dynamic shared memory without the neighbourhood table
    size_t smemCap = 0;                       // dynamic shared memory the kernel may use: the table rides behind smem if it fits
    int resident = 0;                         // StepParams::resident, smStride, lanesPerNode
    int smStride = 0;
    int lanesPerNode = 0;
    int profStride = 0;                       // profiling slots per CTA (StepParams::prof)
    unsigned char profFold[5] = {};           // vsom_debug_phase_cycles: phase i is the sum of the slots in bit mask profFold[i]
};

} // namespace vsom

struct vsom_ctx
{
    int device = 0;
    int W = 0, H = 0, N = 0, Din = 0, Dm = 0, Dr = 0, P = 0;
    int rank = 0, world = 1;      // node sharding: grid rows are dealt to the ranks round-robin in blocks of shardBlock rows
    int localN = 0;               // localRows * W
    int shardBlock = 0, localRows = 0;
    std::vector<int> localRowY;   // global grid row of every local row
    float *peerMean[8] = {};      // mean planes of the ranks (U-matrix halo rows), peer-mapped; peerMean[rank] == mean
    bool peerMeanOpened[8] = {};
    vsom::u64 *rankSlots = nullptr;
    vsom::u64 *peerSlots[8] = {};
    bool peerOpened[8] = {};
    vsom::u64 stepBase = 0;
    float *distBuf = nullptr; // local-search regime scratch
    int transform = 0, order = 0;
    int rowStride = 0;
    int numSMs = 0, smemOptin = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t auxStream = nullptr;           // K2: re-scoring of slab i overlaps the search of slab i + 1
    cudaStream_t copyStream = nullptr;          // host-buffer scoring: H2D of slab i + 1 overlaps the search of slab i
    cudaStream_t outStream = nullptr;           // vsom_predict_columns, host rows: the fill and D2H of slab i's predictions overlap the
    cudaEvent_t evOut = nullptr;                // re-scoring of slab i + 1 and the H2D copies (created on first use)
    cudaEvent_t evScore[2] = {}, evDone[2] = {}, evCopied[3] = {}, evSlabDone[3] = {}; // evCopied / evSlabDone: per host staging buffer (three)
    int tcAttrSet = 0;                          // K2's dynamic shared-memory opt-in was set on this context's device
    int tcPairOk = 0;                           // ... and the device can co-schedule a cluster of two K2 CTAs (cta_group::2 kernel)
    int lastScorePair = 0;                      // the last K2 search ran the CTA-pair kernel (reported while lastScoreTier != 0)
    float *mean = nullptr, *S = nullptr, *sigma = nullptr, *weight = nullptr;
    vsom::u64 *hits = nullptr;
    double *umatrix = nullptr;
    unsigned short *pairI = nullptr, *pairJ = nullptr;
    // online-step scratch
    vsom::u64 *slots = nullptr;
    int *errFlag = nullptr;
    vsom::LutEntry *lut = nullptr;
    size_t lutCap = 0;
    std::vector<vsom::LutEntry> lutHost;
    double lutEta = -1, lutSigma = -1;
    int lutW = 0, lutH = 0;
    // grow-only device staging for the host entry points (10..12: vsom_predict_columns, predict.cu)
    void *stage[13] = {};
    size_t stageCap[13] = {};
    bool trainEnqueued = false;              // vsom_train_chunk_device work not yet checked for an abort
    bool poisoned = false;                   // an online-step chunk aborted: the context refuses further chunks
    unsigned long long tcStats[3] = {0, 0, 0}; // K2 fallback causes since creation: list overflow, NaN / nothing eligible, certificate
    int lastScoreTier = 0;                   // path of the last scoring call (score_rows): 0 the exact scan, else K2's tier (1: one half
                                             // per operand, 2: hi / lo pairs, 3: the probes sent the rest to the exact scan)
    uint64_t launches = 0;
    vsom::StepPlan k1, k1f;                  // online step: the generic kernel, and K1F (k1f.grid == 0: not eligible)
    const vsom::StepPlan *lastPlan = nullptr; // the plan of the last online-step launch
    // K1F (online_step_fast.cu): window table of the current sigma
    unsigned *winTab = nullptr;
    double winSigma = -1;
    vsom::u64 *rowPool = nullptr; // K1F exchange rows: 1024 blocks of 2 KB
    int *rowMeta = nullptr;       // dieOfSm[256] | rowBlocks[640] | rowOf[160] | counters[4]
    int dieAware = 0;             // the row pool was classified by L2 die
    vsom::u64 *distTag = nullptr; // K1F local-walk regime: tagged per-step distances
    int scanBufs = 0, scanSeg = 0, scanNSeg = 0; // K1: HBM-resident rows are streamed through a ring of segment buffers
    void *scanMapDev = nullptr;                   // TMA descriptor of the mean plane for that scan
    void *umTab = nullptr;        // K4: per-grid-row pointer tables (mean rows, sigma rows) + the tiles this context computes
    int umTiles = 0;
    long long *profDev = nullptr; // diagnostics: per-phase cycle sums of the last online-step launch
    size_t profSamples = 0;
    double linInitPhase[4] = {};  // vsom_debug_linear_init_phases: pass, eigen step and fill (ms), iterations of the last call
    double clusterPhase[5] = {};  // vsom_debug_cluster_phases: seeding, assignments, updates, outputs (device ms), assignments of the last call
    std::string err;
};

namespace vsom
{

int set_error(vsom_ctx *ctx, int code, const std::string &msg);
int cuda_fail(vsom_ctx *ctx, cudaError_t e, const char *what, const char *file, int line);
// grow-only device buffer `slot` of at least `bytes`
int stage_reserve(vsom_ctx *ctx, int slot, size_t bytes);

#define VSOM_CUDA(ctx, call)                                                   \
    do                                                                         \
    {                                                                          \
        cudaError_t _e = (call);                                               \
        if (_e != cudaSuccess)                                                 \
            return ::vsom::cuda_fail((ctx), _e, #call, __FILE__, __LINE__);    \
    } while (0)

// The per-row results of one scoring call; every pointer may be null.  All of them are in the memory of the call's rows: device
// memory for device rows, host memory for host rows (rowMaxDev is always device memory).
struct ScoreOut
{
    unsigned *bmu = nullptr;
    float *dist = nullptr;
    unsigned *bmu2 = nullptr; // top == 2 (vsom_find_bmu2): every row's runner-up and its distance
    float *dist2 = nullptr;
    int top = 1;
    // vsom_measure_similarity (k != 0, host rows only): each row's largest normalised deviation from its BMU, computed into
    // rowMaxDev behind the row's final BMU and copied to rowMax
    float *rowMax = nullptr;
    float *rowMaxDev = nullptr;
    float k = 0.0f;
    // vsom_predict_columns (q != 0): the mean and sigma of each row's final BMU at the columns predCols[0 .. q) (device), q values per
    // row.  Device rows: written to mean / sigma after the search; host rows: computed into meanDev / sigmaDev behind each slab's BMUs
    // and copied to mean / sigma.  meanDev / sigmaDev are slab staging that the host paths point at per slab (at() leaves them)
    const int *predCols = nullptr;
    int q = 0;
    float *mean = nullptr, *sigma = nullptr;
    float *meanDev = nullptr, *sigmaDev = nullptr;

    // the same outputs from row r on
    ScoreOut at(size_t r) const
    {
        ScoreOut o = *this;
        auto shift = [](auto *&p, size_t by) {
            if (p)
                p += by;
        };
        shift(o.bmu, r);
        shift(o.dist, r);
        shift(o.bmu2, r);
        shift(o.dist2, r);
        shift(o.rowMax, r);
        shift(o.rowMaxDev, r);
        const size_t rq = r * static_cast<size_t>(q);
        shift(o.mean, rq);
        shift(o.sigma, rq);
        return o;
    }
};

// kernels' host launchers (each returns a vsom_status)
int launch_online_step(vsom_ctx *ctx, const float *xDev, size_t n, double eta, double sigma, int decay, unsigned *outBmuDev, float *outDistDev,
                       const u64 *lastInDev = nullptr);
int configure_online_step(vsom_ctx *ctx);
void configure_online_step_fast(vsom_ctx *ctx);
int prepare_online_step_fast(vsom_ctx *ctx, StepParams &p, double sigma); // K1F's per-chunk buffers and StepParams fields
// cuTensorMapEncodeTiled of the driver, null when the driver does not have it
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                  const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn tensor_map_encoder();
// The map operand of the exact scan (K3): the nodes every row is scored against, and how the rows are read.  scan_map(ctx) is the
// context's own mean plane; vsom_cluster_nodes scores the plane's rows against its f32 centroids as a Standard map (cluster.cu).
struct ScanMap
{
    const float *mean = nullptr; // N rows, rowStride floats apart
    const u64 *hits = nullptr;   // per-node hit counts for min_hits > 0; null: every node competes (min_hits must be 0)
    int N = 0, rowStride = 0;
    int transform = VSOM_STANDARD; // the kernel's Comparer: CLR, or Standard (Standard and Median)
    int Din = 0;                   // floats between consecutive rows of x
    int Dr = 0, P = 0;             // residual length, CLR pair count
    // host rows of vsom_predict_columns: the caller's rows are srcDin floats apart, and each host slab is gathered on the device to its
    // columns cols[0 .. Din) (device memory) before the search reads it.  Null: the rows are read as they are (device rows always are).
    const int *cols = nullptr;
    int srcDin = 0;
};
inline ScanMap scan_map(const vsom_ctx *ctx)
{
    ScanMap m;
    m.mean = ctx->mean;
    m.hits = ctx->hits;
    m.N = ctx->N;
    m.rowStride = ctx->rowStride;
    m.transform = ctx->transform == VSOM_CLR ? VSOM_CLR : VSOM_STANDARD;
    m.Din = ctx->Din;
    m.Dr = ctx->Dr;
    m.P = ctx->P;
    return m;
}
// Every scoring call: x holds n rows (host memory when hostRows), results go to `out`, the nodes are those of `map` (scan_map(ctx),
// or the compacted plane of vsom_predict_columns).  Chooses K2 or the exact scan, runs K2's tiers and the exact scan of the rows K2
// leaves, and records the path for vsom_debug_last_score_tc (score_tc.cu).
int score_rows(vsom_ctx *ctx, const float *x, bool hostRows, size_t n, uint64_t minHits, bool allowTc, const ScoreOut &out, uint64_t *fallbackRows,
               const ScanMap &map);
// The exact scan (K3) of rows 0 .. n-1 of xDev, or (rowListDev != null) of the rows rowListDev[0 .. *rowCountDev), against `map`
int launch_find_bmu_list(vsom_ctx *ctx, const float *xDev, size_t n, const unsigned *rowListDev, const unsigned *rowCountDev, uint64_t minHits, const ScoreOut &out,
                         cudaStream_t stream, u64 *keyBufDev, const ScanMap &map);
int launch_batch_epoch(vsom_ctx *ctx, const float *xDev, size_t n, double sigma, int isFirst, const u64 *lastDev, unsigned *bmuDev, float *distDev);
int launch_all_dists(vsom_ctx *ctx, const float *vDev, double *outDev);
int launch_soft_assign(vsom_ctx *ctx, const float *xDev, size_t n, uint64_t minHits, double *probDev, double *sumsDev);
int launch_similarity_rowmax(vsom_ctx *ctx, const float *xDev, size_t rows, const unsigned *bmuDev, float k, float *outDev, cudaStream_t stream);
int launch_umatrix_tiles(vsom_ctx *ctx, const float *const *meanRowDev, const float *const *sigmaRowDev, const int2 *tilesDev, int nTiles);
int umatrix_tile_rows();
// ids are bins 0 .. bins-1: the context's nodes (vsom_build_index), or the clusters of vsom_cluster_nodes
int launch_build_index(vsom_ctx *ctx, const unsigned *bmuDev, size_t n, int bins, u64 *countsDev, u64 *offsetsDev, unsigned *rowIdsDev);
// exclusive scan of countsDev[count] into offsetsDev[count + 1] (one CTA, som_index.cu)
int launch_offsets_scan(vsom_ctx *ctx, const u64 *countsDev, int count, u64 *offsetsDev);
// vsom_linear_init (lininit.cu): the mean and the two leading principal axes of n host rows (sign rule applied), then the planes
struct LinearFit
{
    std::vector<double> mean, axis1, axis2;
    double lambda[2] = {0.0, 0.0};
};
int linear_init_fit(vsom_ctx *ctx, const float *x, size_t n, LinearFit &fit);
int launch_linear_fill(vsom_ctx *ctx, const LinearFit &fit);
// vsom_cluster_nodes (cluster.cu): k-means++ seeding and Lloyd iterations over the mean plane; the outputs are host arrays
struct ClusterResult
{
    std::vector<int32_t> label;
    std::vector<double> centroids, weight;
    double inertia = 0.0;
    int iterations = 0, converged = 0;
    double phaseMs[4] = {}; // device time of the seeding, the assignments, the updates and the outputs (vsom_debug_cluster_phases)
};
int cluster_nodes(vsom_ctx *ctx, int k, uint64_t seed, int weighting, int maxIter, ClusterResult &res);
// vsom_predict_columns (predict.cu): rows[r][cols[j]] -> out[r * outStride + j] for j < m, zeros up to outStride; and the BMU's mean
// and sigma at out.predCols behind each row's BMU (into out.meanDev / sigmaDev when toStaging, else out.mean / sigma)
int launch_gather_columns(vsom_ctx *ctx, const float *src, size_t rows, size_t srcStride, const int *colsDev, int m, int outStride, float *outDev, cudaStream_t stream);
int launch_predict_fill(vsom_ctx *ctx, const unsigned *bmuDev, size_t rows, const ScoreOut &out, bool toStaging, cudaStream_t stream);
int predict_columns(vsom_ctx *ctx, const float *x, bool hostRows, size_t n, const uint8_t *match, uint64_t minHits, const ScoreOut &out);

// ------------------------------------------------------------------------------------------ device helpers
#ifdef __CUDACC__

__device__ __forceinline__ u64 ld_relaxed_gpu(const u64 *p)
{
    u64 v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ float ld_relaxed_gpu_f32(const float *p)
{
    float v;
    asm volatile("ld.relaxed.gpu.global.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_gpu(u64 *p, u64 v)
{
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ u64 ld_relaxed_sys(const u64 *p)
{
    u64 v;
    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_sys(u64 *p, u64 v)
{
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// ---- packed f32x2 arithmetic (sm_100: FADD2 / FMUL2 / FFMA2 — one issue slot for two IEEE-rounded f32 operations; each half
// rounds exactly like the scalar .rn instruction, so packed code stays bit-identical to the scalar chains it replaces)
__device__ __forceinline__ u64 f2_pack(float lo, float hi)
{
    u64 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void f2_unpack(u64 v, float &lo, float &hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ u64 f2_add(u64 a, u64 b)
{
    u64 d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ u64 f2_sub(u64 a, u64 b)
{
    u64 d;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ u64 f2_mul(u64 a, u64 b)
{
    u64 d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
// CAUTION (ptxas 12.9, seen in SASS): a mul.rn.f32x2 whose only consumer is an add.rn.f32x2 IS contracted into one FFMA2 — with
// -fmad=false, with the explicit .rn forms that are never fused for scalars, even when the product is written as fma(a, b, -0).
// That changes the rounding.  Whenever a product feeds an addition, multiply the halves with scalar __fmul_rn (f2_mul_halves) and
// add packed: one more issue slot per pair, bits identical to the scalar chain.
__device__ __forceinline__ u64 f2_mul_halves(u64 a, u64 b)
{
    float al, ah, bl, bh;
    f2_unpack(a, al, ah);
    f2_unpack(b, bl, bh);
    return f2_pack(__fmul_rn(al, bl), __fmul_rn(ah, bh));
}
__device__ __forceinline__ u64 f2_fma(u64 a, u64 b, u64 c)
{
    u64 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}

__device__ __forceinline__ void cp_async4(void *smemDst, const void *gmemSrc)
{
    unsigned d = static_cast<unsigned>(__cvta_generic_to_shared(smemDst));
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(gmemSrc) : "memory");
}
__device__ __forceinline__ void cp_async8(void *smemDst, const void *gmemSrc)
{
    const unsigned d = static_cast<unsigned>(__cvta_generic_to_shared(smemDst));
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(gmemSrc) : "memory");
}
__device__ __forceinline__ void cp_async16(void *smemDst, const void *gmemSrc)
{
    unsigned d = static_cast<unsigned>(__cvta_generic_to_shared(smemDst));
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gmemSrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

__device__ __forceinline__ u64 u64_min(u64 a, u64 b) { return a < b ? a : b; }
__device__ __forceinline__ u64 warp_min_u64(u64 v)
{
#pragma unroll
    for (int o = 16; o; o >>= 1)
        v = u64_min(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// min over the warp of a 64-bit key with two REDUX instead of ten shuffles: min of the high words, then min of
// the low words among the lanes that hold that high word.  All lanes get the result.
__device__ __forceinline__ u64 warp_min_key(u64 k)
{
    const unsigned hi = static_cast<unsigned>(k >> 32), lo = static_cast<unsigned>(k);
    const unsigned mhi = __reduce_min_sync(0xffffffffu, hi);
    const unsigned mlo = __reduce_min_sync(0xffffffffu, hi == mhi ? lo : 0xffffffffu);
    return (static_cast<u64>(mhi) << 32) | mlo;
}

// (distance, node) -> sortable key.  Distances are sums of squares (>= +0), so their IEEE bit patterns order
// like the values; the node index in the low word reproduces findBmu's strict '<' / lowest-index-wins rule
// (src/Som.cpp:296-304).  A NaN distance never wins, except at node 0 which seeds the search (:293).  `seed` is the
// index node 0 has in the key's numbering: 0, or ~0u (no node) on a node-sharded rank that does not hold global node 0.
// Layout: [63:32] distance bits, [31:8] node, [7:0] tag (exchange sequence number; equal for all keys of a step).
__device__ __forceinline__ u64 make_key(float d, unsigned node, unsigned tag, unsigned seed = 0u)
{
    unsigned bits = __float_as_uint(d);
    if (d != d)
        bits = node == seed ? 0u : 0x7fffffffu;
    return (static_cast<u64>(bits) << 32) | (static_cast<u64>(node) << 8) | tag;
}
__device__ __forceinline__ unsigned key_node(u64 k) { return static_cast<unsigned>((k >> 8) & 0xffffffu); }

// ---- best and second-best keys (vsom_find_bmu2).  Keys of distinct nodes are distinct, so the pair (k1 < k2) is simply the two
// smallest keys: k1 is the BMU of findBmu's rule (a NaN at node 0 wins, key 0), k2 the runner-up with NaN distances after every
// number (0x7fffffff), lower index first.  ~0ull: no key.
__device__ __forceinline__ u64 u64_max(u64 a, u64 b) { return a > b ? a : b; }
__device__ __forceinline__ void key_top2_insert(u64 &k1, u64 &k2, u64 k)
{
    k2 = u64_min(k2, u64_max(k1, k));
    k1 = u64_min(k1, k);
}
__device__ __forceinline__ void key_top2_merge(u64 &k1, u64 &k2, u64 o1, u64 o2)
{
    k2 = u64_min(u64_min(k2, o2), u64_max(k1, o1));
    k1 = u64_min(k1, o1);
}
// (k1, k2) of several producers meeting in global memory (two words per row): whichever of the new k1 and the old one loses
// the first atomic min is a candidate for the second word, and so is the producer's own k2.  Once every producer has passed,
// word 0 holds the smallest key and word 1 the smallest of all the others.
__device__ __forceinline__ void key_top2_atomic(u64 *slot, u64 k1, u64 k2)
{
    const u64 old = atomicMin(slot, k1);
    atomicMin(slot + 1, u64_min(k2, u64_max(old, k1)));
}
// distance of a key as the scoring calls return it (a canonical NaN for NaN distances)
__device__ __forceinline__ float key_dist(u64 k) { return (k & 1ull) ? __uint_as_float(0x7fc00000u) : __uint_as_float(static_cast<unsigned>(k >> 32)); }
// the second-best outputs of a row: 0xFFFFFFFF and NaN when the row has no runner-up (fewer than two eligible nodes)
__device__ __forceinline__ void store_second(unsigned *outBmu2, float *outDist2, u64 row, u64 k2)
{
    if (outBmu2)
        outBmu2[row] = k2 == ~0ull ? 0xffffffffu : key_node(k2);
    if (outDist2)
        outDist2[row] = k2 == ~0ull ? __uint_as_float(0x7fc00000u) : key_dist(k2);
}

// ---- Som::findRestrictedBmu (src/Som.cpp:313-332), the rules of the scoring kernels K3 (score_exact.cu) and K2's rescore (score_tc.cu)
// a node competes when it has at least minHits hits; node 0 seeds the search whatever its hits (:316-322)
template <class I>
__device__ __forceinline__ bool restricted_eligible(I node, const u64 *hits, u64 minHits)
{
    return node == 0 || minHits == 0 || hits[node] >= minHits;
}
// scoring key of a (distance, node) pair in findBmu's order (make_key); the tag bit marks a NaN distance for key_dist
__device__ __forceinline__ u64 score_key(float d, unsigned node) { return make_key(d, node, d != d ? 1u : 0u); }
// a row's outputs from its key(s): BMU and distance (a canonical NaN), and with TOP = 2 the runner-up (k2, read only then)
template <int TOP>
__device__ __forceinline__ void store_row_outputs(unsigned *outBmu, float *outDist, unsigned *outBmu2, float *outDist2, u64 row, u64 k1, const u64 &k2)
{
    if (outBmu)
        outBmu[row] = key_node(k1);
    if (outDist)
        outDist[row] = key_dist(k1);
    if (TOP == 2)
        store_second(outBmu2, outDist2, row, k2);
}
// a producer's key(s) of one row in list mode, where several producers meet in global memory: TOP words at `slot`
template <int TOP>
__device__ __forceinline__ void list_key_store(u64 *slot, u64 k1, u64 k2)
{
    if (TOP == 2)
        key_top2_atomic(slot, k1, k2);
    else
        atomicMin(slot, k1);
}

// ---- node-sharded contexts (BASELINE config 5): block b of `shardBlock` grid rows lives on rank b % world as that rank's
// local block b / world.  Local node order is global node order restricted to the rank (monotone), so keys compare the same
// way inside a rank whichever index they carry.
__host__ __device__ __forceinline__ int shard_local_row(int y, int block, int rank, int world)
{
    const int b = y / block;
    if (b % world != rank)
        return -1;
    return (b / world) * block + (y - b * block);
}
__host__ __device__ __forceinline__ int shard_global_row(int ly, int block, int rank, int world)
{
    const int lb = ly / block;
    return (lb * world + rank) * block + (ly - lb * block);
}
__device__ __forceinline__ unsigned shard_global_node(const StepParams &p, unsigned q)
{
    if (p.world == 1)
        return q;
    const unsigned ly = q / static_cast<unsigned>(p.W);
    return static_cast<unsigned>(shard_global_row(static_cast<int>(ly), p.shardBlock, p.rank, p.world)) * static_cast<unsigned>(p.W) + (q - ly * static_cast<unsigned>(p.W));
}
// local linear index of grid cell (x, y), -1 when another rank holds that row
__device__ __forceinline__ int shard_local_node(const StepParams &p, int x, int y)
{
    if (p.world == 1)
        return y * p.W + x;
    const int ly = shard_local_row(y, p.shardBlock, p.rank, p.world);
    return ly < 0 ? -1 : ly * p.W + x;
}

// ---- Som::trainSingle's per-node arithmetic (src/Som.cpp:912-942), shared by the online-step kernels K1 (online_step.cu) and
// K1F (online_step_fast.cu)

// the Median Stepper (src/Transformation.cpp:49-50): sign(d) in {-1, +0, +1}, NaN stays NaN.  |d| > 0 ? copysign(1, d) : |d| gives
// +0 for a zero like the reference's (0<d)-(d<0); NaN fails the comparison and |NaN| is NaN.
__device__ __forceinline__ float median_sign(float d)
{
    const float a = fabsf(d);
    const float one = __uint_as_float((__float_as_uint(d) & 0x80000000u) | 0x3f800000u); // copysign(1, d)
    return a > 0.0f ? one : a;
}

// residual of one CLR pair: (A x' + B) - y' (src/Transformation.cpp:104), scalar round-to-nearest operations: a * x + b must never
// contract
__device__ __forceinline__ float clr_residual(float a, float b, float xi, float xj) { return __fsub_rn(__fadd_rn(__fmul_rn(a, xi), b), xj); }

// one pair of the window update (src/Som.cpp:912-941 with the CLR Stepper, src/Transformation.cpp:107-142):
//   inner = (A x' + B) - y';  delta = [(-2 inner) x' || -2 inner];  model += c * delta;  S += nwf * (delta0 * delta1)
// pend = squared residual of this sample against the UPDATED model (trainSingle's return value, :946).  A caller may pass references
// into memory: the model pair is read first and written before S is read.
__device__ __forceinline__ void clr_update_pair(float xi, float xj, float c, float nwf, float &a, float &b, float &sa, float &sb, float &pend)
{
    const float a0 = a, b0 = b;
    const float in0 = clr_residual(a0, b0, xi, xj);
    const float db0 = __fmul_rn(-2.0f, in0);
    const float da0 = __fmul_rn(db0, xi);
    const float a1 = __fadd_rn(a0, __fmul_rn(c, da0));
    const float b1 = __fadd_rn(b0, __fmul_rn(c, db0));
    const float in1 = clr_residual(a1, b1, xi, xj);
    const float db1 = __fmul_rn(-2.0f, in1);
    const float da1 = __fmul_rn(db1, xi);
    a = a1;
    b = b1;
    sa = __fadd_rn(sa, __fmul_rn(nwf, __fmul_rn(da0, da1)));
    sb = __fadd_rn(sb, __fmul_rn(nwf, __fmul_rn(db0, db1)));
    pend = __fmul_rn(in1, in1);
}

// the neighbourhood-table entry (LutEntry as a float4) of a node dx, dy cells from the BMU, from the shared-memory copy when the
// launch made one
__device__ __forceinline__ float4 neighbourhood_entry(int lutSmem, const LutEntry *lutS, const LutEntry *lut, int lutW, int dx, int dy)
{
    const int li = dy * lutW + dx;
    if (lutSmem)
        return *reinterpret_cast<const float4 *>(lutS + li);
    return __ldg(reinterpret_cast<const float4 *>(lut + li));
}

// weightMap update and step coefficient of a window node (src/Som.cpp:922-935) from its table entry: w is updated in place,
// the result is {step coefficient c, (float)nw}
__device__ __forceinline__ float2 step_coefficient(const float4 entry, bool exponential, float &w)
{
    if (exponential)
    {
        w = __fadd_rn(w, entry.z);           // :924
        return make_float2(entry.z, entry.w); // :925
    }
    w = __fadd_rn(w, entry.w); // :930
    const double nw = __hiloint2double(__float_as_int(entry.y), __float_as_int(entry.x));
    const double tw = (w == 0.0f) ? 1.0 : __ddiv_rn(nw, static_cast<double>(w)); // :933
    return make_float2(static_cast<float>(tw), entry.w);                         // :935
}

// sigmaMap of a visited node: sqrt(|S / (float)(W == 0 ? 1e-6 : W)|) with its final S and W (src/Som.cpp:939-942)
__device__ __forceinline__ float lazy_sigma(float S, float w)
{
    const float twf = static_cast<float>((w == 0.0f) ? 0.000001 : static_cast<double>(w));
    return __fsqrt_rn(fabsf(__fdiv_rn(S, twf)));
}

// One residual of the Comparer, and its square accumulated in f32 (src/Som.cpp:136-140).
//   Standard / Median: r = m - v           (src/Transformation.cpp:7-8, :45-46)
//   CLR:               r = (A*x' + B) - y' (src/Transformation.cpp:104), clr_residual's expression written out: calling it with
//                      the four elements reorders their loads, and soft_assign_terms_kernel<CLR> then needs ten more registers
template <int TR>
__device__ __forceinline__ float residual(const float *m, const float *xs, int k, int P, const unsigned short *pi, const unsigned short *pj)
{
    if (TR != VSOM_CLR)
        return __fsub_rn(m[k], xs[k]);
    return __fsub_rn(__fadd_rn(__fmul_rn(m[k], xs[pi[k]]), m[P + k]), xs[pj[k]]);
}

// Squared distance in the reference's order: k = 0..Dr-1 sequentially (one thread).
template <int TR>
__device__ __forceinline__ float dist_sequential(const float *m, const float *xs, int Dr, int P, const unsigned short *pi, const unsigned short *pj)
{
    float s = 0.0f;
#pragma unroll 8
    for (int k = 0; k < Dr; ++k)
    {
        const float r = residual<TR>(m, xs, k, P, pi, pj);
        s = __fadd_rn(s, __fmul_rn(r, r));
    }
    return s;
}

// ---- summation orders of one squared distance (vsom_reduction_order, include/vsom_b200.h)
// EIGEN_SSE restates what `a.dot(b)` / `squaredNorm()` compile to in the reference when it is built against real Eigen
// (3.3 / 3.4, README.md:64-69) with its release flags (-msse2 only, build/Makefile:18): Eigen's redux_impl<...,
// LinearVectorizedTraversal, NoUnrolling> over Packet4f — two packet accumulators over strides of 8 elements, the sum of
// the two, one more packet if 4..7 elements remain, predux = (p0 + p2) + (p1 + p3), then the scalar tail in order.  The
// reduced expression has no direct access, so the aligned start is element 0.
struct EigenSseSum
{
    float a[8];
    __device__ __forceinline__ EigenSseSum()
    {
#pragma unroll
        for (int j = 0; j < 8; ++j)
            a[j] = 0.0f; // 0 + t == t exactly for the terms of this library (squares: never -0)
    }
    // terms t[8 b + j] of a full block of eight
    __device__ __forceinline__ void block(const float (&t)[8])
    {
#pragma unroll
        for (int j = 0; j < 8; ++j)
            a[j] = __fadd_rn(a[j], t[j]);
    }
    // after n / 8 blocks: `rest` = the n % 8 remaining terms in order
    __device__ __forceinline__ float finish(const float *rest, int nrest) const
    {
        float r0 = __fadd_rn(a[0], a[4]), r1 = __fadd_rn(a[1], a[5]), r2 = __fadd_rn(a[2], a[6]), r3 = __fadd_rn(a[3], a[7]);
        int k = 0;
        if (nrest >= 4)
        {
            r0 = __fadd_rn(r0, rest[0]);
            r1 = __fadd_rn(r1, rest[1]);
            r2 = __fadd_rn(r2, rest[2]);
            r3 = __fadd_rn(r3, rest[3]);
            k = 4;
        }
        float s = __fadd_rn(__fadd_rn(r0, r2), __fadd_rn(r1, r3));
#pragma unroll
        for (int j = 0; j < 7; ++j) // static indices: `rest` stays in registers
            if (j >= k && j < nrest)
                s = __fadd_rn(s, rest[j]);
        return s;
    }
};

// |m - x|^2 of two plain rows (Standard / Median Comparer, src/Transformation.cpp:7-8, :45-46) by ONE thread, in the given
// order.  m is a row of a plane (16-byte aligned); x may be unaligned.
__device__ __forceinline__ float dist_rows_f32(const float *__restrict__ m, const float *__restrict__ x, int D, int order)
{
    if (order == VSOM_ORDER_EIGEN_SSE)
    {
        EigenSseSum acc;
        int k = 0;
        for (; k + 8 <= D; k += 8)
        {
            const float4 m0 = *reinterpret_cast<const float4 *>(m + k), m1 = *reinterpret_cast<const float4 *>(m + k + 4);
            float t[8];
            const float mm[8] = {m0.x, m0.y, m0.z, m0.w, m1.x, m1.y, m1.z, m1.w};
#pragma unroll
            for (int j = 0; j < 8; ++j)
            {
                const float d = __fsub_rn(mm[j], x[k + j]);
                t[j] = __fmul_rn(d, d);
            }
            acc.block(t);
        }
        float rest[8];
        const int nrest = D - k;
        for (int j = 0; j < nrest; ++j)
        {
            const float d = __fsub_rn(m[k + j], x[k + j]);
            rest[j] = __fmul_rn(d, d);
        }
        return acc.finish(rest, nrest);
    }
    float s = 0.0f;
    int k = 0;
    for (; k + 4 <= D; k += 4)
    {
        const float4 a = *reinterpret_cast<const float4 *>(m + k);
        float q = __fsub_rn(a.x, x[k]);
        s = __fadd_rn(s, __fmul_rn(q, q));
        q = __fsub_rn(a.y, x[k + 1]);
        s = __fadd_rn(s, __fmul_rn(q, q));
        q = __fsub_rn(a.z, x[k + 2]);
        s = __fadd_rn(s, __fmul_rn(q, q));
        q = __fsub_rn(a.w, x[k + 3]);
        s = __fadd_rn(s, __fmul_rn(q, q));
    }
    for (; k < D; ++k)
    {
        const float q = __fsub_rn(m[k], x[k]);
        s = __fadd_rn(s, __fmul_rn(q, q));
    }
    return s;
}

// Squared distance of one node by ONE thread in the given order (any transformation).
template <int TR>
__device__ __forceinline__ float dist_ordered(const float *m, const float *xs, int Dr, int P, const unsigned short *pi, const unsigned short *pj, int order)
{
    if (order != VSOM_ORDER_EIGEN_SSE)
        return dist_sequential<TR>(m, xs, Dr, P, pi, pj);
    EigenSseSum acc;
    int k = 0;
    for (; k + 8 <= Dr; k += 8)
    {
        float t[8];
#pragma unroll
        for (int j = 0; j < 8; ++j)
        {
            const float r = residual<TR>(m, xs, k + j, P, pi, pj);
            t[j] = __fmul_rn(r, r);
        }
        acc.block(t);
    }
    float rest[8];
    const int nrest = Dr - k;
    for (int j = 0; j < nrest; ++j)
    {
        const float r = residual<TR>(m, xs, k + j, P, pi, pj);
        rest[j] = __fmul_rn(r, r);
    }
    return acc.finish(rest, nrest);
}

// Squared distance with 32 interleaved partial sums and a fixed xor butterfly (all 32 lanes call; all get the value).
template <int TR>
__device__ __forceinline__ float dist_lanes(const float *m, const float *xs, int Dr, int P, const unsigned short *pi, const unsigned short *pj, int lane)
{
    float s = 0.0f;
#pragma unroll 4
    for (int k = lane; k < Dr; k += 32)
    {
        const float r = residual<TR>(m, xs, k, P, pi, pj);
        s = __fadd_rn(s, __fmul_rn(r, r));
    }
#pragma unroll
    for (int o = 16; o; o >>= 1)
        s = __fadd_rn(s, __shfl_xor_sync(0xffffffffu, s, o));
    return s;
}

// Som::findLocalBmu (src/Som.cpp:335-454) on the per-step distances (read through `load(node)`): greedy walk from `start` over the
// 8-neighbourhood, then three cells one step further in the X direction of travel, until the best node stops moving.
// The reference's size_t arithmetic is kept: the "-1" offsets are 2^64-1, min(x + off, W-1) therefore wraps the left / up
// neighbour of column / row 0 to the last column / row, and its Y-direction continuation loop never runs (it starts at
// size_t(-1)).  Distances are compared as the reference does (strict '<', first candidate in its order wins).
template <class Load>
__device__ __forceinline__ unsigned local_bmu_walk(Load load, u64 W, u64 H, u64 start)
{
    const u64 M1 = ~0ull;
    const u64 fx[8] = {M1, 0, 1, 1, 1, 0, M1, M1};
    const u64 fy[8] = {1, 1, 1, 0, M1, M1, M1, 0};
    u64 lastBMU = start, minIndex = start, lastMeasured = start;
    float minDist = load(start);
    for (;;)
    {
        const u64 lmX = lastMeasured % W, lmY = lastMeasured / W, lbX = lastBMU % W;
        if (lastMeasured == lastBMU)
        {
            u64 idx[8];
            float v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i)
            {
                const u64 cx = lmX + fx[i] < W - 1 ? lmX + fx[i] : W - 1; // min(x + off, W-1) in size_t
                const u64 cy = lmY + fy[i] < H - 1 ? lmY + fy[i] : H - 1;
                idx[i] = cy * W + cx;
                v[i] = load(idx[i]);
            }
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if (v[i] < minDist)
                {
                    minDist = v[i];
                    minIndex = idx[i];
                }
            if (minIndex == lastBMU)
                return static_cast<unsigned>(minIndex);
            lastMeasured = minIndex;
        }
        else
        {
            if (lmX - lbX) // moving in X
            {
                u64 idx[3];
                float v[3];
#pragma unroll
                for (int i = 0; i < 3; ++i)
                {
                    const u64 ox = lmX + lmX - lbX, oy = lmY + static_cast<u64>(static_cast<long long>(i - 1));
                    const u64 cx = ox < W - 1 ? ox : W - 1, cy = oy < H - 1 ? oy : H - 1;
                    idx[i] = cy * W + cx;
                    v[i] = load(idx[i]);
                }
#pragma unroll
                for (int i = 0; i < 3; ++i)
                    if (v[i] < minDist)
                    {
                        minDist = v[i];
                        minIndex = idx[i];
                    }
            }
            if (minIndex == lastMeasured)
                return static_cast<unsigned>(minIndex);
            lastBMU = lastMeasured;
            lastMeasured = minIndex;
        }
    }
}


#endif // __CUDACC__

} // namespace vsom
