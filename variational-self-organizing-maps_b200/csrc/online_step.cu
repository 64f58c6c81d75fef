// online_step.cu — K1: the online VSOM training step as ONE persistent sm_100a kernel per sample chunk.
//
// Replaces, per sample and in sample order: Som::trainSingle (src/Som.cpp:885-947) = Som::findBmu (:291-309)
// over Som::euclidianWeightedDist (:124-141) + the Gaussian-neighbourhood update of map / weightMap / SMap /
// sigmaMap (:899-944, Som::calculateNeighbourhoodWeight :949-975) + Som::addBmu (:1189-1192).
//
// Design (see DESIGN.md §K1)
//   * grid = one CTA per SM, launched cooperatively so that all CTAs are co-resident.  Grid nodes are dealt
//     round-robin: CTA b owns shard-local nodes b, b+G, b+2G, ...  Ownership never changes, so a node's rows
//     are read and written by exactly one CTA: when the owned rows of the mean and S planes fit in shared
//     memory they are loaded once, stay there for the whole chunk and are written back at the end
//     (configs 1-3); otherwise they are addressed in global memory (large maps).
//   * per sample there is exactly ONE grid-wide exchange: every CTA pushes the min (distance,node) key of its
//     nodes, tagged with the step number, into a private row of every other CTA (slots[dest][src]); each CTA
//     then polls only its own row (G words, lines nobody else reads) and takes the min itself.  Pushing keeps
//     the polling traffic off shared cache lines: with a single shared row, 148 pollers hammering the same
//     ten L2 lines cost ~4000 cycles per sample (profiles/r01_bench_k1_v1.json).  No second barrier is needed
//     because the window update of a node is done by its owner, which is also the only CTA that scans it for
//     the next sample.  Round-robin ownership spreads any update window evenly over the SMs.
//   * sigmaMap is a pure function of the node's SMap and weightMap at its LAST visit
//     (sigma = sqrt(|S / (W==0 ? 1e-6 : W)|), src/Som.cpp:939-942, overwritten at every visit), and nothing on
//     this path reads it (all shipped Comparers ignore `dispersion`).  The kernel therefore only marks the
//     visited nodes and evaluates that expression once per visited node at the end of the chunk — the stored
//     plane is bit-identical, and the IEEE divide + square root leave the per-sample loop.
//   * reduction order is a template parameter (vsom_reduction_order): REFERENCE sums the squared residuals
//     sequentially like the reference's dot product (one thread per node), so BMUs and every plane stay
//     bit-identical to it; LANES uses a warp per node.
//   * the distance of the sample to its UPDATED BMU (trainSingle's return value, :946) is computed by an
//     otherwise idle thread / warp of the owner CTA during the next sample's scan, off the critical path.
#include "common.cuh"

#include <cmath>
#include <cstdlib>
#include <string>

namespace vsom
{

constexpr int kThreads = 1024;
constexpr int kWarps = kThreads / 32;
constexpr int kMaxSlotsPerLane = 5;   // the exchange row of a CTA is read by one warp: at most 160 CTAs
constexpr size_t kStaticSmem = 1024; // static __shared__ of the kernel, rounded up

// One element of the window update (src/Som.cpp:912-941) for Standard / Median; sigma is evaluated lazily.
template <int TR>
__device__ __forceinline__ void update_element(float xv, float c, float nwf, float &m, float &S)
{
    // Transformation::Stepper for Standard (src/Transformation.cpp:11-12) and Median (:49-50)
    auto stepper = [](float d) { return TR == VSOM_MEDIAN ? median_sign(d) : d; };
    const float d0 = stepper(__fsub_rn(xv, m));                  // :912 (and :935, same value)
    const float m1 = __fadd_rn(m, __fmul_rn(c, d0));             // :925 / :935
    const float d1 = stepper(__fsub_rn(xv, m1));                 // :941 Stepper on the new mean
    S = __fadd_rn(S, __fmul_rn(nwf, __fmul_rn(d0, d1)));         // :941
    m = m1;
}

// Squared distance, reference order, over zero-padded rows with 128-bit loads (Standard / Median).
// The chain s += r*r is 4 cycles per element and cannot be shortened without changing the order; the loads of
// the next group are issued before the current group's adds so that their latency stays off the chain.
__device__ __forceinline__ void acc4(float &s, const float4 a, const float4 b)
{
    float r = __fsub_rn(a.x, b.x);
    s = __fadd_rn(s, __fmul_rn(r, r));
    r = __fsub_rn(a.y, b.y);
    s = __fadd_rn(s, __fmul_rn(r, r));
    r = __fsub_rn(a.z, b.z);
    s = __fadd_rn(s, __fmul_rn(r, r));
    r = __fsub_rn(a.w, b.w);
    s = __fadd_rn(s, __fmul_rn(r, r));
}
__device__ __forceinline__ float dist_sequential_v4(const float *m, const float *xs, int n4)
{
    const float4 *m4 = reinterpret_cast<const float4 *>(m);
    const float4 *x4 = reinterpret_cast<const float4 *>(xs);
    float s = 0.0f;
    const int pairs = n4 >> 1;
    if (pairs > 0)
    {
        float4 a0 = m4[0], b0 = x4[0], a1 = m4[1], b1 = x4[1];
        for (int g = 1; g < pairs; ++g)
        {
            const float4 c0 = m4[2 * g], d0 = x4[2 * g], c1 = m4[2 * g + 1], d1 = x4[2 * g + 1];
            acc4(s, a0, b0);
            acc4(s, a1, b1);
            a0 = c0;
            b0 = d0;
            a1 = c1;
            b1 = d1;
        }
        acc4(s, a0, b0);
        acc4(s, a1, b1);
    }
    if (n4 & 1)
        acc4(s, m4[n4 - 1], x4[n4 - 1]);
    return s;
}

// Eigen SSE2 order over zero-padded rows (Standard / Median): full blocks of eight with two 128-bit loads each, then the
// Dm % 8 remaining elements (common.cuh, EigenSseSum)
__device__ __forceinline__ float dist_eigen_v4(const float *m, const float *xs, int Dm)
{
    const float4 *m4 = reinterpret_cast<const float4 *>(m);
    const float4 *x4 = reinterpret_cast<const float4 *>(xs);
    EigenSseSum acc;
    const int n8 = Dm >> 3;
#pragma unroll 2
    for (int b = 0; b < n8; ++b)
    {
        const float4 a0 = m4[2 * b], b0 = x4[2 * b], a1 = m4[2 * b + 1], b1 = x4[2 * b + 1];
        float t[8];
        float r = __fsub_rn(a0.x, b0.x);
        t[0] = __fmul_rn(r, r);
        r = __fsub_rn(a0.y, b0.y);
        t[1] = __fmul_rn(r, r);
        r = __fsub_rn(a0.z, b0.z);
        t[2] = __fmul_rn(r, r);
        r = __fsub_rn(a0.w, b0.w);
        t[3] = __fmul_rn(r, r);
        r = __fsub_rn(a1.x, b1.x);
        t[4] = __fmul_rn(r, r);
        r = __fsub_rn(a1.y, b1.y);
        t[5] = __fmul_rn(r, r);
        r = __fsub_rn(a1.z, b1.z);
        t[6] = __fmul_rn(r, r);
        r = __fsub_rn(a1.w, b1.w);
        t[7] = __fmul_rn(r, r);
        acc.block(t);
    }
    float rest[8];
    const int k0 = n8 << 3, nrest = Dm - k0;
    for (int j = 0; j < nrest; ++j)
    {
        const float r = __fsub_rn(m[k0 + j], xs[k0 + j]);
        rest[j] = __fmul_rn(r, r);
    }
    return acc.finish(rest, nrest);
}

// distance of one node by one thread, in the reference's sequential order or in Eigen's SSE2 order
template <int TR, int ORDER>
__device__ __forceinline__ float node_dist_reference(const float *m, const float *xs, const StepParams &p, int n4, const unsigned short *pi,
                                                     const unsigned short *pj)
{
    if (ORDER == VSOM_ORDER_EIGEN_SSE)
    {
        if (TR != VSOM_CLR)
            return dist_eigen_v4(m, xs, p.Dm);
        return dist_ordered<TR>(m, xs, p.Dr, p.P, pi, pj, VSOM_ORDER_EIGEN_SSE);
    }
    if (TR != VSOM_CLR)
        return dist_sequential_v4(m, xs, n4); // the zero padding adds +0 terms: s + 0 == s exactly
    return dist_sequential<TR>(m, xs, p.Dr, p.P, pi, pj);
}

constexpr int kScanSegMax = 132; // floats of a row per streamed segment at most; a segment is (odd number) x 4 floats long
constexpr int kScanMaxBufs = 6;  // buffers per scan warp
constexpr int kListThreshold = 96; // owned nodes per CTA above which the update window is enumerated cell by cell
constexpr int kScanWarps = 4;    // warps that stream and scan (each its own ring)

__device__ __forceinline__ unsigned smem_addr(const void *p) { return static_cast<unsigned>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void scan_bar_init(u64 *bar, unsigned count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory"); }
__device__ __forceinline__ void scan_bar_expect(u64 *bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool scan_bar_try_wait(u64 *bar, unsigned parity)
{
    unsigned ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(smem_addr(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// one TMA box of the mean plane -> shared memory, completion counted in bytes on an mbarrier.  The plane is described as
// the 3-D tensor (column, owner CTA, owned-row index): row = index * G + cta, so a box {scanSeg, 1, 32} is a segment of 32
// consecutive OWNED rows of one CTA although they lie G rows apart in memory.
__device__ __forceinline__ void scan_tma_load(void *dst, const void *map, u64 *bar, int col, int cta, int row)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(smem_addr(dst)), "l"(map),
                 "r"(smem_addr(bar)), "r"(col), "r"(cta), "r"(row)
                 : "memory");
}

template <int TR, int ORDER, bool RES>
__global__ void __launch_bounds__(kThreads, 1) online_step_kernel(const StepParams p)
{
    extern __shared__ __align__(16) unsigned char smemRaw[];
    __shared__ u64 sWarpKey[kWarps];
    __shared__ int sWin[8]; // local index of the BMU (-1: another rank's), bx, by, startX, endX, startY, endY of the current sample
    __shared__ int sAbort;
    __shared__ int sPendL; // local node whose post-update distance is still owed (-1: none)
    __shared__ u64 sPendT; // ... for this sample
    __shared__ long long sClk[6], sProf[5]; // diagnostics (thread 0 only)

    const int G = gridDim.x, b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int Lmax = (p.nodeCount + G - 1) / G;
    const int L = (p.nodeCount > b) ? (p.nodeCount - b + G - 1) / G : 0;
    const int DinPad = (p.Din + 3) & ~3;
    const int DmPad = (p.Dm + 3) & ~3;
    const int n4 = DmPad >> 2;
    const int Gp = (G + 15) & ~15; // pitch of one destination row of the exchange (whole 128-byte lines)

    // ---- carve shared memory (every region 16-byte aligned)
    float *xs = reinterpret_cast<float *>(smemRaw);                          // [3][DinPad] sample ring
    float *wbuf = xs + 3 * DinPad;                                           // [Lpad] weightMap of the owned nodes
    const int Lpad = (Lmax + 3) & ~3;
    float2 *coef = reinterpret_cast<float2 *>(wbuf + Lpad);                  // [Lpad] per owned node in the window: {step coefficient, (float)nw}
    const bool useList = Lmax > kListThreshold; // many owned nodes: enumerate the window's cells instead of testing every owned node
    int2 *nodeXY = reinterpret_cast<int2 *>(coef + Lpad);                    // [Lpad] grid position of the owned nodes (not with the list)
    unsigned *touched = reinterpret_cast<unsigned *>(nodeXY + (useList ? 0 : Lpad)); // [Lpad] visited in this chunk
    unsigned *inWin = touched + Lpad;                                        // [Lpad] inside the window of the current sample
    unsigned short *pi = reinterpret_cast<unsigned short *>(inWin + Lpad);   // [Ppad] CLR pair tables
    const int Ppad = (p.P + 7) & ~7;
    unsigned short *pj = pi + Ppad;
    float *planes = reinterpret_cast<float *>(pj + Ppad);                    // resident rows: 2 x Lmax x smStride
    // !RES with p.scanBufs: ring of streamed row segments [warps][bufs][32][scanSeg], 128-byte aligned for the TMA engine
    // (pointer arithmetic on a shared-memory pointer, not an integer round trip: the loads must stay LDS, not generic LD)
    float *sbuf = planes + (((128u - (smem_addr(planes) & 127u)) & 127u) >> 2);
    LutEntry *lutS = reinterpret_cast<LutEntry *>(RES ? planes + 2 * static_cast<size_t>(Lmax) * p.smStride
                                                      : (p.scanBufs > 0 ? sbuf + static_cast<size_t>(kScanWarps) * p.scanBufs * 32 * p.scanSeg : planes)); // optional copy of the table
    __shared__ __align__(8) u64 sScanBar[kScanWarps * kScanMaxBufs];
    __shared__ int sListN;                                                   // owned nodes inside the window of the current sample

    float *mBase, *sBase;
    size_t stride;
    if (RES)
    {
        stride = static_cast<size_t>(p.smStride);
        mBase = planes;
        sBase = planes + static_cast<size_t>(Lmax) * stride;
    }
    else
    {
        stride = static_cast<size_t>(G) * p.rowStride;
        mBase = p.mean + static_cast<size_t>(b) * p.rowStride;
        sBase = p.S + static_cast<size_t>(b) * p.rowStride;
    }

    // slices of 128 elements of the model vector (CLR: of the pair index): one warp per (window node, slice)
    const int nq = TR == VSOM_CLR ? p.P : DmPad;
    const int nCh = (nq + 127) >> 7;

    // ---- prologue: pair tables, neighbourhood table, owned weights / positions, resident rows, first sample
    if (TR == VSOM_CLR)
        for (int q = tid; q < p.P; q += kThreads)
        {
            pi[q] = p.pairI[q];
            pj[q] = p.pairJ[q];
        }
    if (p.lutSmem)
        for (int i = tid; i < p.lutCount; i += kThreads)
            lutS[i] = p.lut[i];
    for (int l = tid; l < L; l += kThreads)
    {
        const unsigned node = shard_global_node(p, static_cast<unsigned>(l * G + b));
        wbuf[l] = p.weight[static_cast<size_t>(l) * G + b];
        if (!useList)
            nodeXY[l] = make_int2(static_cast<int>(node % static_cast<unsigned>(p.W)), static_cast<int>(node / static_cast<unsigned>(p.W)));
        touched[l] = 0;
    }
    for (int k = tid; k < 3 * DinPad; k += kThreads)
        xs[k] = 0.0f; // keeps the pad lanes of the 128-bit paths at zero
    if (RES)
        for (int l = warp; l < L; l += kWarps)
        {
            const size_t g = (static_cast<size_t>(l) * G + b) * p.rowStride;
            for (int k = lane; k < static_cast<int>(stride); k += 32)
            {
                const bool in = k < p.Dm;
                mBase[l * stride + k] = in ? p.mean[g + k] : 0.0f;
                sBase[l * stride + k] = in ? p.S[g + k] : 0.0f;
            }
        }
    if (tid == 0)
    {
        sAbort = 0;
        sPendL = -1;
        sPendT = 0;
        for (int i = 0; i < kScanWarps * kScanMaxBufs; ++i)
            scan_bar_init(&sScanBar[i], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    int scanBuf = 0;      // streamed scan: next buffer of this warp's ring to consume ...
    unsigned scanPar = 0; // ... and the phase its mbarrier completes next
    __syncthreads();

    // sample prefetch: 16-byte cp.async.cg (L2 only — a streamed sample must not evict the L1-resident table)
    // when rows are 16-byte aligned, else 4-byte cp.async.ca
    auto prefetch = [&](u64 t, int slot) {
        float *dst = xs + slot * DinPad;
        const float *src = p.x + t * static_cast<u64>(p.Din);
        if (p.xVec)
        {
            for (int k = tid * 4; k < p.Din; k += kThreads * 4)
                cp_async16(dst + k, src + k);
        }
        else
        {
            for (int k = tid; k < p.Din; k += kThreads)
                cp_async4(dst + k, src + k);
        }
    };
    if (p.n > 0)
        prefetch(0, 0);

    const double dW = static_cast<double>(p.W), dH = static_cast<double>(p.H);
    if (tid == 0)
        for (int i = 0; i < 5; ++i)
            sProf[i] = 0;
    // the owed output of sample pendT, whose BMU is owned node pendL: distance d to its updated BMU (src/Som.cpp:946) + addBmu
    // (:1189-1192)
    auto write_owed = [&](int pendL, u64 pendT, float d) {
        const size_t q = static_cast<size_t>(pendL) * G + b;
        if (p.outBmu)
            p.outBmu[pendT] = shard_global_node(p, static_cast<unsigned>(q));
        if (p.outDist)
            p.outDist[pendT] = d;
        p.hits[q] += 1;
    };

    // keys carry local node indices (see the exchange below): only the rank holding global node 0 (rank 0, block 0) lets a
    // NaN distance at its local node 0 win, like findBmu's seed; on other ranks local node 0 is an ordinary node
    const unsigned nanSeed = p.rank == 0 ? 0u : ~0u;
    int ring = 0; // t % 3
    for (u64 t = 0; t < p.n; ++t, ring = ring == 2 ? 0 : ring + 1)
    {
        if (p.prof && tid == 0)
            sClk[0] = clock64();
        const float *xt = xs + ring * DinPad;
        cp_async_wait_all();
        __syncthreads(); // sample t landed; update of sample t-1 is complete; sPend* of t-1 visible
        if (t + 1 < p.n)
            prefetch(t + 1, ring == 2 ? 0 : ring + 1);
        if (p.prof && tid == 0)
            sClk[1] = clock64();
        const unsigned tag = static_cast<unsigned>((t >> 1) & 0xff);

        // ---- owed output of sample t-1: distance to its updated BMU (src/Som.cpp:946) + addBmu (:1189-1192)
        const int pendL = sPendL;
        const u64 pendT = sPendT;
        const float *xprev = xs + (ring == 0 ? 2 : ring - 1) * DinPad; // sample t-1

        // ---- scan: distance of sample t to every owned node, min key per thread
        u64 best = ~0ull;
        // distance d of owned node l: kept for the local walk (by the thread that writes it), folded into this thread's key
        auto record = [&](int l, float d, bool writer) {
            if (p.localSearch && writer)
                p.distBuf[(t & 1) * static_cast<u64>(p.nodeCount) + static_cast<u64>(l) * G + b] = d;
            best = u64_min(best, make_key(d, static_cast<unsigned>(l * G + b), tag, nanSeed));
        };
        if (ORDER != VSOM_ORDER_LANES)
        {
            if (tid == kThreads - 1 && pendL >= 0)
                write_owed(pendL, pendT, node_dist_reference<TR, ORDER>(mBase + pendL * stride, xprev, p, n4, pi, pj));
            if (!RES && TR != VSOM_CLR && p.scanBufs > 0)
            {
                // HBM-resident map.  A thread-per-node scan reads 16 bytes per row and instruction and reaches 49 % of the HBM
                // roofline; coalescing through warp tiles of 128-byte row chunks was slower still (many small scattered
                // requests, little in flight).  Here the rows are STREAMED: each of the first kScanWarps warps keeps its own
                // ring of buffers in flight, a buffer being filled by 32 bulk copies (cp.async.bulk: one contiguous row
                // segment of ~0.5 KB per lane, completion counted in bytes on an mbarrier); lane r then walks row r's
                // segment in order — the reference's sequential sum, one row per lane, fed by contiguous DRAM bursts with
                // ~100 KB in flight per SM.  The other warps wait at the barrier below.
                if (warp < kScanWarps)
                {
                    const int nSeg = p.scanNSeg, Kseg = p.scanSeg, segStride = Kseg, NB = p.scanBufs;
                    const int nGroups = (L + 31) >> 5;
                    const int myGroups = nGroups > warp ? (nGroups - warp + kScanWarps - 1) / kScanWarps : 0, steps = myGroups * nSeg;
                    float *ring = sbuf + static_cast<size_t>(warp) * NB * 32 * segStride;
                    u64 *bars = sScanBar + warp * kScanMaxBufs;
                    // issue and consume cursors advance incrementally (no divisions on this path): segment within the group,
                    // group, buffer of the ring; the ring position and the mbarrier phase carry over from sample to sample
                    int sgI = 0, gI = warp, bufI = scanBuf;
                    auto issue = [&]() {
                        if (lane == 0)
                        {
                            scan_bar_expect(&bars[bufI], static_cast<unsigned>(32 * Kseg * 4)); // a box always delivers all its bytes (zero fill outside)
                            scan_tma_load(ring + static_cast<size_t>(bufI) * 32 * segStride, p.scanMap, &bars[bufI], sgI * Kseg, b, 32 * gI);
                        }
                        if (++sgI == nSeg)
                        {
                            sgI = 0;
                            gI += kScanWarps;
                        }
                        if (++bufI == NB)
                            bufI = 0;
                    };
                    int issued = 0;
                    for (; issued < NB && issued < steps; ++issued)
                        issue();
                    float sacc = 0.0f;
                    EigenSseSum eacc;   // ORDER == EIGEN_SSE: the eight chains of this lane's row, carried across its segments
                    float erest[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                    const int nFull4 = (p.Dm >> 3) << 1; // 128-bit words of a row that belong to full blocks of eight
                    int sg = 0, g = warp;
                    for (int i = 0; i < steps; ++i)
                    {
                        unsigned spins = 0;
                        while (!scan_bar_try_wait(&bars[scanBuf], scanPar))
                            if (++spins > (1u << 24))
                            {
                                sAbort = 1; // a box that never lands is a bug, not a wait
                                *p.err = 1;
                                break;
                            }
                        const int n4s = min(Kseg, DmPad - sg * Kseg) >> 2;
                        if (sg == 0)
                        {
                            sacc = 0.0f;
                            if (ORDER == VSOM_ORDER_EIGEN_SSE)
                                eacc = EigenSseSum();
                        }
                        const int l = 32 * g + lane;
                        if (l < L && ORDER == VSOM_ORDER_EIGEN_SSE)
                        {
                            // word Q of the row goes to lanes 0..3 (Q even) or 4..7 (Q odd) of the packet accumulators; the words
                            // behind the full blocks (at most two, zero padded) are kept for the extra packet / scalar tail
                            const float4 *m4 = reinterpret_cast<const float4 *>(ring + (static_cast<size_t>(scanBuf) * 32 + lane) * segStride);
                            const float4 *x4 = reinterpret_cast<const float4 *>(xt + sg * Kseg);
                            const int q0 = sg * (Kseg >> 2);
                            const int qFull = max(0, min(n4s, nFull4 - q0)); // words of this segment inside full blocks of eight
                            auto sq4 = [](const float4 a, const float4 bq, float &t0, float &t1, float &t2, float &t3) {
                                float r = __fsub_rn(a.x, bq.x);
                                t0 = __fmul_rn(r, r);
                                r = __fsub_rn(a.y, bq.y);
                                t1 = __fmul_rn(r, r);
                                r = __fsub_rn(a.z, bq.z);
                                t2 = __fmul_rn(r, r);
                                r = __fsub_rn(a.w, bq.w);
                                t3 = __fmul_rn(r, r);
                            };
                            auto add_lo = [&](const float4 a, const float4 bq) {
                                float t0, t1, t2, t3;
                                sq4(a, bq, t0, t1, t2, t3);
                                eacc.a[0] = __fadd_rn(eacc.a[0], t0);
                                eacc.a[1] = __fadd_rn(eacc.a[1], t1);
                                eacc.a[2] = __fadd_rn(eacc.a[2], t2);
                                eacc.a[3] = __fadd_rn(eacc.a[3], t3);
                            };
                            auto add_hi = [&](const float4 a, const float4 bq) {
                                float t0, t1, t2, t3;
                                sq4(a, bq, t0, t1, t2, t3);
                                eacc.a[4] = __fadd_rn(eacc.a[4], t0);
                                eacc.a[5] = __fadd_rn(eacc.a[5], t1);
                                eacc.a[6] = __fadd_rn(eacc.a[6], t2);
                                eacc.a[7] = __fadd_rn(eacc.a[7], t3);
                            };
                            int q = 0;
                            if ((q0 & 1) && q < qFull) // the segment starts in the middle of a block of eight
                            {
                                add_hi(m4[0], x4[0]);
                                q = 1;
                            }
                            // (even, odd) word pairs: no branches, the next pair's loads in flight during the adds
                            if (q + 2 <= qFull)
                            {
                                float4 a0 = m4[q], b0 = x4[q], a1 = m4[q + 1], b1 = x4[q + 1];
                                for (q += 2; q + 2 <= qFull; q += 2)
                                {
                                    const float4 c0 = m4[q], d0 = x4[q], c1 = m4[q + 1], d1 = x4[q + 1];
                                    add_lo(a0, b0);
                                    add_hi(a1, b1);
                                    a0 = c0;
                                    b0 = d0;
                                    a1 = c1;
                                    b1 = d1;
                                }
                                add_lo(a0, b0);
                                add_hi(a1, b1);
                            }
                            if (q < qFull)
                            {
                                add_lo(m4[q], x4[q]);
                                ++q;
                            }
                            for (; q < n4s; ++q) // behind the full blocks: the extra packet and / or the scalar tail (zero padded)
                            {
                                float t0, t1, t2, t3;
                                sq4(m4[q], x4[q], t0, t1, t2, t3);
                                if (q0 + q == nFull4)
                                {
                                    erest[0] = t0;
                                    erest[1] = t1;
                                    erest[2] = t2;
                                    erest[3] = t3;
                                }
                                else
                                {
                                    erest[4] = t0;
                                    erest[5] = t1;
                                    erest[6] = t2;
                                    erest[7] = t3;
                                }
                            }
                            if (sg == nSeg - 1)
                            {
                                sacc = eacc.finish(erest, p.Dm & 7);
                                record(l, sacc, true);
                            }
                        }
                        else if (l < L)
                        {
                            // s += (m_k - x_k)^2 in order, loads a pair of 128-bit words ahead of the adds
                            const float4 *m4 = reinterpret_cast<const float4 *>(ring + (static_cast<size_t>(scanBuf) * 32 + lane) * segStride);
                            const float4 *x4 = reinterpret_cast<const float4 *>(xt + sg * Kseg);
                            const int pairs = n4s >> 1;
                            if (pairs > 0)
                            {
                                float4 a0 = m4[0], b0 = x4[0], a1 = m4[1], b1 = x4[1];
                                for (int k = 1; k < pairs; ++k)
                                {
                                    const float4 c0 = m4[2 * k], d0 = x4[2 * k], c1 = m4[2 * k + 1], d1 = x4[2 * k + 1];
                                    acc4(sacc, a0, b0);
                                    acc4(sacc, a1, b1);
                                    a0 = c0;
                                    b0 = d0;
                                    a1 = c1;
                                    b1 = d1;
                                }
                                acc4(sacc, a0, b0);
                                acc4(sacc, a1, b1);
                            }
                            if (n4s & 1)
                                acc4(sacc, m4[n4s - 1], x4[n4s - 1]);
                            if (sg == nSeg - 1)
                                record(l, sacc, true);
                        }
                        __syncwarp(); // every lane is done with this buffer before it is refilled
                        if (issued < steps)
                        {
                            issue();
                            ++issued;
                        }
                        if (++sg == nSeg)
                        {
                            sg = 0;
                            g += kScanWarps;
                        }
                        if (++scanBuf == NB)
                        {
                            scanBuf = 0;
                            scanPar ^= 1u;
                        }
                    }
                }
            }
            else
                for (int l = tid; l < L; l += kThreads)
                    record(l, node_dist_reference<TR, ORDER>(mBase + l * stride, xt, p, n4, pi, pj), true);
        }
        else
        {
            if (warp == kWarps - 1 && pendL >= 0)
            {
                const float d = dist_lanes<TR>(mBase + pendL * stride, xprev, p.Dr, p.P, pi, pj, lane);
                if (lane == 0)
                    write_owed(pendL, pendT, d);
            }
            for (int l = warp; l < L; l += kWarps)
                record(l, dist_lanes<TR>(mBase + l * stride, xt, p.Dr, p.P, pi, pj, lane), lane == 0);
        }
        if (p.localSearch)
            __threadfence(); // the distances written above must be visible before this CTA's key is
        // REFERENCE order with at most 32 owned nodes: every key already sits in warp 0 — no CTA barrier
        const bool crossWarp = ORDER == VSOM_ORDER_LANES || L > 32;
        if (crossWarp)
        {
            best = warp_min_key(best);
            if (lane == 0)
                sWarpKey[warp] = best;
            __syncthreads();
        }

        // ---- grid-wide min-loc: push the key into every CTA's row, then poll the own row
        if (warp == 0)
        {
            u64 k = crossWarp ? (lane < kWarps ? sWarpKey[lane] : ~0ull) : best;
            k = warp_min_key(k);
            if (k == ~0ull) // CTA without nodes (cannot happen: G <= nodeCount) — still publish a tagged key
                k = (~0ull << 8) | tag;
            u64 *buf = p.slots + static_cast<size_t>(t & 1) * G * Gp;
            if (p.prof && tid == 0)
                sClk[2] = clock64();
            for (int d = lane; d < G; d += 32)
                st_relaxed_gpu(buf + static_cast<size_t>(d) * Gp + b, k);
            const u64 *row = buf + static_cast<size_t>(b) * Gp;
            const long long t0 = clock64();
            u64 m;
            bool abort = false;
            const u64 filler = (~0ull << 8) | tag;
            for (;;)
            {
                // all loads of a round are issued before any is consumed: one L2 round trip per round, not G/32
                u64 v[kMaxSlotsPerLane];
#pragma unroll
                for (int j = 0; j < kMaxSlotsPerLane; ++j)
                {
                    const int i = lane + 32 * j;
                    v[j] = i < G ? ld_relaxed_gpu(row + i) : filler;
                }
                m = ~0ull;
                int ok = 1;
#pragma unroll
                for (int j = 0; j < kMaxSlotsPerLane; ++j)
                {
                    ok &= (static_cast<unsigned>(v[j] & 0xff) == tag);
                    m = u64_min(m, v[j]);
                }
                if (__all_sync(0xffffffffu, ok))
                    break;
                if (__any_sync(0xffffffffu, clock64() - t0 > p.timeoutCycles))
                {
                    abort = true;
                    break;
                }
            }
            m = warp_min_key(m);
            if (p.world > 1 && !abort)
            {
                // ---- node-sharded map: the GPU-local winner is pushed into every rank's memory over NVLink by CTA 0
                // (system-scope stores to peer-mapped pointers); every CTA then polls ITS OWN GPU's row of `world`
                // tagged keys.  Indexed by the global step, so it needs neither a reset nor a host barrier between
                // launches; ranks can never be more than one step apart.
                const u64 gs = p.stepBase + t;
                const unsigned gtag = static_cast<unsigned>((gs >> 1) & 0xff);
                const int gbuf = static_cast<int>(gs & 1);
                // keys carry LOCAL node indices inside a GPU (they order like the global ones there); across GPUs the global index
                const u64 mine = (m & 0xffffffff00000000ull) | (static_cast<u64>(shard_global_node(p, key_node(m))) << 8) | gtag;
                if (b == 0 && lane < p.world)
                    st_relaxed_sys(p.peerSlots[lane] + gbuf * p.world + p.rank, mine);
                const u64 *grow = p.rankSlots + gbuf * p.world;
                const long long g0 = clock64();
                u64 gv;
                for (;;)
                {
                    gv = lane < p.world ? ld_relaxed_sys(grow + lane) : ((~0ull << 8) | gtag);
                    if (__all_sync(0xffffffffu, static_cast<unsigned>(gv & 0xff) == gtag))
                        break;
                    if (__any_sync(0xffffffffu, clock64() - g0 > p.peerTimeoutCycles)) // ranks start their chunks at different times
                    {
                        abort = true;
                        break;
                    }
                }
                m = warp_min_key(gv);
                if (b == 0 && lane == 0 && p.outBmu && !abort)
                    p.outBmu[t] = key_node(m); // every rank records the global BMU of every sample
            }
            if (p.localSearch && !abort)
            {
                // every CTA has seen every CTA's key of this step, hence (fence above) every distance of this step
                __threadfence();
                __syncwarp();
            }
            // window of the update (src/Som.cpp:899-903): [startX,endX) x [startY,endY), asymmetric.  Lane 0 computes it
            // (f64, exactly the reference's expressions) and broadcasts it to the warp.
            int wbmu = 0, wbx = 0, wby = 0, wsx = 0, wex = 0, wsy = 0, wey = 0;
            if (lane == 0)
            {
                unsigned bmu = key_node(m);
                if (p.localSearch && !abort)
                {
                    const float *dist = p.distBuf + (t & 1) * static_cast<u64>(p.nodeCount);
                    bmu = local_bmu_walk([&](u64 i) { return ld_relaxed_gpu_f32(dist + i); }, static_cast<u64>(p.W), static_cast<u64>(p.H),
                                         p.lastIn ? p.lastIn[t] : 0ull);
                    if (b == 0 && p.outBmu)
                        p.outBmu[t] = bmu;
                }
                wbx = static_cast<int>(bmu % static_cast<unsigned>(p.W));
                wby = static_cast<int>(bmu / static_cast<unsigned>(p.W));
                wbmu = shard_local_node(p, wbx, wby); // local index of the BMU, -1 when another rank holds it
                double lo = __dsub_rn(static_cast<double>(wbx), p.radius);
                wsx = static_cast<int>(static_cast<u64>(lo > 0. ? lo : 0.));
                lo = __dsub_rn(static_cast<double>(wby), p.radius);
                wsy = static_cast<int>(static_cast<u64>(lo > 0. ? lo : 0.));
                double hi = __dadd_rn(static_cast<double>(wbx), p.radius);
                wex = static_cast<int>(static_cast<u64>(hi < dW ? hi : dW));
                hi = __dadd_rn(static_cast<double>(wby), p.radius);
                wey = static_cast<int>(static_cast<u64>(hi < dH ? hi : dH));
                sPendL = -1;
                if (abort)
                {
                    sAbort = 1;
                    *p.err = 1;
                }
            }
            wbmu = __shfl_sync(0xffffffffu, wbmu, 0);
            wbx = __shfl_sync(0xffffffffu, wbx, 0);
            wby = __shfl_sync(0xffffffffu, wby, 0);
            wsx = __shfl_sync(0xffffffffu, wsx, 0);
            wex = __shfl_sync(0xffffffffu, wex, 0);
            wsy = __shfl_sync(0xffffffffu, wsy, 0);
            wey = __shfl_sync(0xffffffffu, wey, 0);
            if (lane == 0)
            {
                sWin[0] = wbmu;
                sWin[1] = wbx;
                sWin[2] = wby;
                sWin[3] = wsx;
                sWin[4] = wex;
                sWin[5] = wsy;
                sWin[6] = wey;
            }
            // ---- per owned node (lanes = nodes): neighbourhood entry, weightMap update and the step coefficient
            //      (src/Som.cpp:915-939).  When a node's vector spans several warps (nCh > 1) this is done once here;
            //      with one warp per node (nCh == 1) each update warp does it for its own node after the barrier,
            //      which keeps it off this warp's critical path.
            if (lane == 0)
                sListN = 0;
            for (int l = lane; nCh > 1 && !useList && l < L; l += 32)
            {
                const int2 xy = nodeXY[l];
                float2 cf = make_float2(-1.0f, 0.0f);
                if (xy.x >= wsx && xy.x < wex && xy.y >= wsy && xy.y < wey)
                {
                    const int dx = xy.x > wbx ? xy.x - wbx : wbx - xy.x, dy = xy.y > wby ? xy.y - wby : wby - xy.y;
                    const float4 entry = neighbourhood_entry(p.lutSmem, lutS, p.lut, p.lutW, dx, dy);
                    float w = wbuf[l];
                    cf = step_coefficient(entry, p.decay == VSOM_EXPONENTIAL, w);
                    wbuf[l] = w;
                    touched[l] = 1;
                    if (l * G + b == wbmu)
                    {
                        sPendL = l;
                        sPendT = t;
                    }
                    inWin[l] = 1;
                }
                else
                    inWin[l] = 0;
                coef[l] = cf;
            }
            if (p.prof && tid == 0)
                sClk[3] = clock64();
        }
        __syncthreads();
        if (sAbort)
            break;
        if (useList)
        {
            // every thread walks cells of the window; an owned node is appended to the list (kept in inWin[]) together with
            // its neighbourhood entry, new weightMap value and step coefficient (src/Som.cpp:915-939).  Nodes are
            // independent, so the order of the list does not matter.
            const int wbmu = sWin[0], wbx = sWin[1], wby = sWin[2], wsx = sWin[3], wex = sWin[4], wsy = sWin[5], wey = sWin[6];
            const int ww = wex - wsx, cells = ww * (wey - wsy);
            for (int cidx = tid; cidx < cells; cidx += kThreads)
            {
                const int cy = cidx / ww, cx = cidx - cy * ww;
                const int x = wsx + cx, y = wsy + cy;
                const int rel = shard_local_node(p, x, y);
                if (rel < 0)
                    continue;
                const int l = rel / G;
                if (rel - l * G != b)
                    continue;
                const int dx = x > wbx ? x - wbx : wbx - x, dy = y > wby ? y - wby : wby - y;
                const float4 entry = neighbourhood_entry(p.lutSmem, lutS, p.lut, p.lutW, dx, dy);
                float w = wbuf[l];
                const float2 cf = step_coefficient(entry, p.decay == VSOM_EXPONENTIAL, w);
                wbuf[l] = w;
                touched[l] = 1;
                coef[l] = cf;
                if (rel == wbmu)
                {
                    sPendL = l;
                    sPendT = t;
                }
                inWin[atomicAdd(&sListN, 1)] = static_cast<unsigned>(l);
            }
            __syncthreads();
        }
        if (p.prof && tid == 0)
            sClk[4] = clock64();
        // ---- update: one warp per (window node, 128-element slice) of the model vector (src/Som.cpp:912-941)
        {
            const int items = (useList ? sListN : L) * nCh;
            for (int it = warp; it < items; it += kWarps)
            {
                int l = nCh > 1 ? it / nCh : it;
                const int ch = nCh > 1 ? it - l * nCh : 0;
                float c, nwf;
                if (useList)
                {
                    l = static_cast<int>(inWin[l]);
                    const float2 cf = coef[l];
                    c = cf.x;
                    nwf = cf.y;
                }
                else if (nCh > 1)
                {
                    if (!inWin[l])
                        continue;
                    const float2 cf = coef[l];
                    c = cf.x;
                    nwf = cf.y;
                }
                else
                {
                    // one warp owns the whole node: every lane derives the coefficient (redundantly, no traffic),
                    // lane 0 records the new weight
                    const int2 xy = nodeXY[l];
                    const int bx = sWin[1], by = sWin[2];
                    if (!(xy.x >= sWin[3] && xy.x < sWin[4] && xy.y >= sWin[5] && xy.y < sWin[6]))
                        continue;
                    const int dx = xy.x > bx ? xy.x - bx : bx - xy.x, dy = xy.y > by ? xy.y - by : by - xy.y;
                    const float4 entry = neighbourhood_entry(p.lutSmem, lutS, p.lut, p.lutW, dx, dy);
                    float w = wbuf[l];
                    const float2 cf = step_coefficient(entry, p.decay == VSOM_EXPONENTIAL, w);
                    c = cf.x;
                    nwf = cf.y;
                    __syncwarp(); // every lane has read the old weight
                    if (lane == 0)
                    {
                        wbuf[l] = w;
                        touched[l] = 1;
                        if (l * G + b == sWin[0])
                        {
                            sPendL = l;
                            sPendT = t;
                        }
                    }
                }
                float *m = mBase + l * stride, *S = sBase + l * stride;
                if (TR != VSOM_CLR)
                {
                    const int k = (ch << 7) + (lane << 2);
                    if (k < DmPad)
                    {
                        float4 mv = *reinterpret_cast<float4 *>(m + k);
                        float4 sv = *reinterpret_cast<float4 *>(S + k);
                        const float4 xv = *reinterpret_cast<const float4 *>(xt + k);
                        update_element<TR>(xv.x, c, nwf, mv.x, sv.x);
                        update_element<TR>(xv.y, c, nwf, mv.y, sv.y);
                        update_element<TR>(xv.z, c, nwf, mv.z, sv.z);
                        update_element<TR>(xv.w, c, nwf, mv.w, sv.w);
                        *reinterpret_cast<float4 *>(m + k) = mv;
                        *reinterpret_cast<float4 *>(S + k) = sv;
                    }
                }
                else
                {
                    // Stepper of CLR (src/Transformation.cpp:107-142), pair by pair in place
                    const int P = p.P;
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                    {
                        const int q = (ch << 7) + (j << 5) + lane;
                        if (q < P)
                        {
                            float unused;
                            clr_update_pair(xt[pi[q]], xt[pj[q]], c, nwf, m[q], m[P + q], S[q], S[P + q], unused);
                        }
                    }
                }
            }
        }
        if (!RES && p.scanBufs > 0)
            asm volatile("fence.proxy.async.global;" ::: "memory"); // this sample's stores to the mean plane before the next scan's TMA reads
        if (p.prof && tid == 0)
        {
            sClk[5] = clock64();
            for (int i = 0; i < 5; ++i)
                sProf[i] += sClk[i + 1] - sClk[i];
        }
        // the __syncthreads at the top of the next iteration orders these writes before the next scan
    }

    // ---- epilogue: last owed output, lazy sigma, then write the owned rows back
    __syncthreads();
    if (sPendL >= 0)
    {
        const int pendL = sPendL;
        const u64 pendT = sPendT;
        const float *xprev = xs + static_cast<int>(pendT % 3) * DinPad;
        float d = 0.0f;
        bool writer = false;
        if (ORDER != VSOM_ORDER_LANES)
        {
            if (tid == 0)
            {
                d = node_dist_reference<TR, ORDER>(mBase + pendL * stride, xprev, p, n4, pi, pj);
                writer = true;
            }
        }
        else if (warp == 0)
        {
            d = dist_lanes<TR>(mBase + pendL * stride, xprev, p.Dr, p.P, pi, pj, lane);
            writer = lane == 0;
        }
        if (writer)
            write_owed(pendL, pendT, d);
    }
    const float *wfin = wbuf;
    for (int l = tid; l < L; l += kThreads)
        p.weight[static_cast<size_t>(l) * G + b] = wfin[l];
    for (int l = warp; l < L; l += kWarps)
    {
        const size_t g = (static_cast<size_t>(l) * G + b) * p.rowStride;
        const bool vis = touched[l] != 0;
        const float w = wfin[l]; // sigmaMap of a visited node (lazy_sigma)
        for (int k = lane; k < p.Dm; k += 32)
        {
            const float sv = sBase[l * stride + k];
            if (RES)
            {
                p.mean[g + k] = mBase[l * stride + k];
                p.S[g + k] = sv;
            }
            if (vis)
                p.sigma[g + k] = lazy_sigma(sv, w);
        }
    }
    if (p.prof && tid == 0)
        for (int i = 0; i < 5; ++i)
            p.prof[static_cast<size_t>(b) * 5 + i] = sProf[i];
}

// --------------------------------------------------------------------------------------------- host side

static int resident_stride(const vsom_ctx *ctx)
{
    // rows start 16-byte aligned and (stride / 4) is odd: the thread-per-node scan (lanes = nodes, 128-bit
    // loads) and the warp-per-node update (lanes = consecutive words) are both bank-conflict free.
    const int n4 = (ctx->Dm + 3) / 4;
    return 4 * (n4 | 1);
}

static size_t online_step_smem(const vsom_ctx *ctx, int G, bool resident, int smStride)
{
    const int Lmax = (ctx->localN + G - 1) / G;
    const int Lpad = (Lmax + 3) & ~3;
    const int DinPad = (ctx->Din + 3) & ~3;
    const int Ppad = (ctx->P + 7) & ~7;
    size_t bytes = sizeof(float) * (3 * static_cast<size_t>(DinPad) + 3 * static_cast<size_t>(Lpad));
    bytes += ((Lmax > kListThreshold ? 0 : sizeof(int2)) + 2 * sizeof(unsigned)) * static_cast<size_t>(Lpad);
    bytes += 2 * sizeof(unsigned short) * static_cast<size_t>(Ppad);
    if (resident)
        bytes += sizeof(float) * 2 * static_cast<size_t>(Lmax) * smStride;
    return bytes;
}

typedef void (*StepKernel)(const StepParams);
static StepKernel pick_kernel(int transform, int order, int resident)
{
#define VSOM_K(TR, ORD) {online_step_kernel<TR, ORD, false>, online_step_kernel<TR, ORD, true>}
#define VSOM_KO(TR) {VSOM_K(TR, VSOM_ORDER_REFERENCE), VSOM_K(TR, VSOM_ORDER_LANES), VSOM_K(TR, VSOM_ORDER_EIGEN_SSE)}
    static const StepKernel table[3][3][2] = {VSOM_KO(VSOM_STANDARD), VSOM_KO(VSOM_MEDIAN), VSOM_KO(VSOM_CLR)};
#undef VSOM_KO
#undef VSOM_K
    return table[transform][order][resident ? 1 : 0];
}

// mean plane as (column, owner CTA, owned-row index), box {seg, 1, 32}; the descriptor lives in device memory
static int make_scan_map(vsom_ctx *ctx, int G, int seg)
{
    const EncodeTiledFn enc = tensor_map_encoder();
    if (!enc)
        return set_error(ctx, VSOM_ERR_CUDA, "online step: cuTensorMapEncodeTiled entry point not available");
    const int Lmax = (ctx->localN + G - 1) / G;
    CUtensorMap map;
    const cuuint64_t dims[3] = {static_cast<cuuint64_t>(ctx->rowStride), static_cast<cuuint64_t>(G), static_cast<cuuint64_t>(Lmax)};
    const cuuint64_t strides[2] = {static_cast<cuuint64_t>(ctx->rowStride) * 4, static_cast<cuuint64_t>(ctx->rowStride) * 4 * G};
    const cuuint32_t box[3] = {static_cast<cuuint32_t>(seg), 1, 32};
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = enc(&map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, ctx->mean, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
        return set_error(ctx, VSOM_ERR_CUDA, "online step: cuTensorMapEncodeTiled failed (" + std::to_string(static_cast<int>(r)) + ")");
    if (!ctx->scanMapDev)
        VSOM_CUDA(ctx, cudaMalloc(&ctx->scanMapDev, 256));
    VSOM_CUDA(ctx, cudaMemcpyAsync(ctx->scanMapDev, &map, sizeof(map), cudaMemcpyHostToDevice, ctx->stream));
    VSOM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return VSOM_OK;
}

// K1's plan, which every context has (an error when the map's bookkeeping does not fit), then K1F's where it is eligible
int configure_online_step(vsom_ctx *ctx)
{
    int G = ctx->localN < ctx->numSMs ? ctx->localN : ctx->numSMs;
    if (G > 32 * kMaxSlotsPerLane)
        G = 32 * kMaxSlotsPerLane;
    const int smStride = resident_stride(ctx);
    const size_t statics = kStaticSmem;
    size_t bytes = online_step_smem(ctx, G, true, smStride);
    int resident = 1;
    ctx->scanBufs = 0;
    if (bytes + statics > static_cast<size_t>(ctx->smemOptin))
    {
        resident = 0;
        bytes = online_step_smem(ctx, G, false, smStride);
        if (bytes + statics > static_cast<size_t>(ctx->smemOptin))
            return set_error(ctx, VSOM_ERR_UNSUPPORTED, "online step: per-CTA bookkeeping does not fit in shared memory for this map");
        // streamed scan of the HBM-resident rows (Standard / Median, reference order): as many segment buffers as fit
        if (ctx->transform != VSOM_CLR && ctx->order != VSOM_ORDER_LANES)
        {
            const int DmPad = (ctx->Dm + 3) & ~3;
            int seg = DmPad < kScanSegMax ? DmPad : kScanSegMax;
            if (((seg >> 2) & 1) == 0)
                seg -= 4; // (seg / 4) odd: lanes = rows read the dense box without bank conflicts
            if (seg >= 4)
                for (int bufs = kScanMaxBufs; bufs >= 2; --bufs)
                {
                    const size_t ring = sizeof(float) * kScanWarps * bufs * 32 * seg;
                    if (bytes + ring + statics + 1024 <= static_cast<size_t>(ctx->smemOptin))
                    {
                        int rc = make_scan_map(ctx, G, seg);
                        if (rc)
                            return rc;
                        ctx->scanBufs = bufs;
                        ctx->scanSeg = seg;
                        ctx->scanNSeg = (DmPad + seg - 1) / seg;
                        bytes += ring + 1024; // room to start the ring on a 1 KB boundary
                        break;
                    }
                }
        }
    }
    StepKernel k = pick_kernel(ctx->transform, ctx->order, resident);
    VSOM_CUDA(ctx, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, ctx->smemOptin - static_cast<int>(kStaticSmem)));
    int perSm = 0;
    VSOM_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSm, k, kThreads, bytes));
    if (perSm < 1)
        return set_error(ctx, VSOM_ERR_UNSUPPORTED, "online step: kernel does not fit on an SM");
    StepPlan &pl = ctx->k1;
    pl.kernel[0] = pl.kernel[1] = k;
    pl.grid = G;
    pl.threads = kThreads;
    pl.smem = bytes;
    pl.smemCap = static_cast<size_t>(ctx->smemOptin) - kStaticSmem;
    pl.resident = resident;
    pl.smStride = smStride;
    pl.profStride = 5;
    for (int i = 0; i < 5; ++i)
        pl.profFold[i] = static_cast<unsigned char>(1u << i); // the five phases of the kernel's profile
    configure_online_step_fast(ctx);
    return VSOM_OK;
}

// Neighbourhood table for one (eta, sigma), rounded the way LutEntry describes.
static int build_lut(vsom_ctx *ctx, double eta, double sigma)
{
    if (ctx->lutEta == eta && ctx->lutSigma == sigma && ctx->lut)
        return VSOM_OK;
    const double radius = 2.5 * sigma;
    const int reach = static_cast<int>(std::ceil(radius));
    const int lw = (ctx->W - 1 < reach ? ctx->W - 1 : reach) + 1;
    const int lh = (ctx->H - 1 < reach ? ctx->H - 1 : reach) + 1;
    ctx->lutHost.resize(static_cast<size_t>(lw) * lh);
    for (int dy = 0; dy < lh; ++dy)
        for (int dx = 0; dx < lw; ++dx)
        {
            const double nw = neighbourhood_weight(dx, dy, sigma);
            LutEntry e;
            e.nw = nw;
            e.cexp = static_cast<float>(nw * eta);
            e.nwf = static_cast<float>(nw);
            ctx->lutHost[static_cast<size_t>(dy) * lw + dx] = e;
        }
    const size_t bytes = ctx->lutHost.size() * sizeof(LutEntry);
    if (bytes > ctx->lutCap)
    {
        if (ctx->lut)
            VSOM_CUDA(ctx, cudaFree(ctx->lut));
        ctx->lut = nullptr;
        VSOM_CUDA(ctx, cudaMalloc(&ctx->lut, bytes));
        ctx->lutCap = bytes;
    }
    // the previous chunk's kernel may still be reading the old table: the copy is stream-ordered behind it, and
    // a copy from pageable memory is staged by the runtime before the call returns, so lutHost can be reused.
    VSOM_CUDA(ctx, cudaMemcpyAsync(ctx->lut, ctx->lutHost.data(), bytes, cudaMemcpyHostToDevice, ctx->stream));
    ctx->lutEta = eta;
    ctx->lutSigma = sigma;
    ctx->lutW = lw;
    ctx->lutH = lh;
    return VSOM_OK;
}

// K1's per-chunk state: the exchange slots, the local walk's distance buffer, the streamed scan of HBM-resident rows
static int prepare_online_step(vsom_ctx *ctx, StepParams &p)
{
    const int G = ctx->k1.grid;
    const int Gp = (G + 15) & ~15;
    VSOM_CUDA(ctx, cudaMemsetAsync(ctx->slots, 0xff, sizeof(u64) * 2 * static_cast<size_t>(G) * Gp, ctx->stream));
    p.slots = ctx->slots;
    if (p.localSearch && !ctx->distBuf)
        VSOM_CUDA(ctx, cudaMalloc(&ctx->distBuf, sizeof(float) * 2 * static_cast<size_t>(ctx->N)));
    p.distBuf = ctx->distBuf;
    p.scanBufs = ctx->scanBufs;
    p.scanSeg = ctx->scanSeg;
    p.scanNSeg = ctx->scanNSeg;
    p.scanMap = ctx->scanMapDev;
    return VSOM_OK;
}

// One chunk of online steps.  K1F runs it when configure_online_step_fast gave the context a plan and the chunk has fewer
// than 2^32 - 1 samples (K1F counts steps in 32 bits).  That plan exists for one GPU, VSOM_ONLINE_KERNEL not "generic" at
// vsom_create, the reference or Eigen order, grid sides <= 4096, at most 512 owned nodes per CTA, planes (CLR: [A || B] rows
// and pair tables) that fit in shared memory; every transformation, sigma > 1 and the local walk (sigma <= 1) alike.
// Everything else (LANES order, HBM-resident and node-sharded maps) runs K1.
int launch_online_step(vsom_ctx *ctx, const float *xDev, size_t n, double eta, double sigma, int decay, unsigned *outBmuDev, float *outDistDev,
                       const u64 *lastInDev)
{
    const bool localSearch = !(sigma > 1.0); // SIGMA_SWITCH_TO_LOCAL (include/SOM.hpp:37, src/Som.cpp:889-892)
    if (localSearch && ctx->world > 1)
        return set_error(ctx, VSOM_ERR_UNSUPPORTED, "online step: the findLocalBmu regime (sigma <= 1) is not available on node-sharded contexts");
    if (decay != VSOM_EXPONENTIAL && decay != VSOM_INVERSE_PROPORTIONAL)
        return set_error(ctx, VSOM_ERR_INVALID, "online step: decay must be Exponential or InverseProportional");
    if (n == 0)
        return VSOM_OK;
    if (ctx->world > 1)
        for (int r = 0; r < ctx->world; ++r)
            if (!ctx->peerSlots[r])
                return set_error(ctx, VSOM_ERR_INVALID, "online step: sharded context without vsom_peer_import for every rank");
    if (ctx->poisoned)
        return set_error(ctx, VSOM_ERR_TIMEOUT, "online step: an earlier chunk of this context aborted (a CTA or a rank never published its key); "
                                                "the map and the cross-rank step counter are no longer consistent — re-create the context");
    int rc = build_lut(ctx, eta, sigma);
    if (rc)
        return rc;
    const bool fast = ctx->k1f.grid && n < (1ull << 32) - 1;
    const StepPlan &plan = fast ? ctx->k1f : ctx->k1;
    VSOM_CUDA(ctx, cudaMemsetAsync(ctx->errFlag, 0, sizeof(int), ctx->stream));

    StepParams p{};
    p.W = ctx->W;
    p.H = ctx->H;
    p.shardBlock = ctx->shardBlock;
    p.nodeCount = ctx->localN;
    p.order = ctx->order;
    p.world = ctx->world;
    p.rank = ctx->rank;
    p.rankSlots = ctx->rankSlots;
    for (int r = 0; r < 8; ++r)
        p.peerSlots[r] = ctx->peerSlots[r];
    p.stepBase = ctx->stepBase;
    p.Din = ctx->Din;
    p.Dm = ctx->Dm;
    p.Dr = ctx->Dr;
    p.P = ctx->P;
    p.rowStride = ctx->rowStride;
    p.mean = ctx->mean;
    p.S = ctx->S;
    p.sigma = ctx->sigma;
    p.weight = ctx->weight;
    p.hits = ctx->hits;
    p.x = xDev;
    p.n = n;
    p.decay = decay;
    p.radius = 2.5 * sigma;
    p.lut = ctx->lut;
    p.lutW = ctx->lutW;
    p.pairI = ctx->pairI;
    p.pairJ = ctx->pairJ;
    p.err = ctx->errFlag;
    p.outBmu = outBmuDev;
    p.outDist = outDistDev;
    p.timeoutCycles = 4000000000ll; // ~2 s at 1.9 GHz: a peer CTA of the same launch that never publishes is a bug, not a wait
    {
        // other RANKS launch their chunk from their own process: a pageable H2D copy, a buffer re-allocation or a scheduler
        // stall on one of them delays its first key by far more than a CTA ever lags.  Default 60 s, VSOM_PEER_TIMEOUT_S overrides.
        const char *e = getenv("VSOM_PEER_TIMEOUT_S");
        const double secs = e && atof(e) > 0 ? atof(e) : 60.0;
        p.peerTimeoutCycles = static_cast<long long>(secs * 2.0e9);
    }
    p.localSearch = localSearch ? 1 : 0;
    p.lastIn = lastInDev;
    p.prof = ctx->profDev;
    p.xVec = (ctx->Din % 4 == 0 && (reinterpret_cast<uintptr_t>(xDev) & 15) == 0) ? 1 : 0;
    p.resident = plan.resident;
    p.smStride = plan.smStride;
    p.lanesPerNode = plan.lanesPerNode;
    // the neighbourhood table rides in shared memory behind the kernel's own data when it fits
    p.lutCount = ctx->lutW * ctx->lutH;
    const size_t lutBytes = sizeof(LutEntry) * static_cast<size_t>(p.lutCount);
    p.lutSmem = plan.smem + lutBytes <= plan.smemCap ? 1 : 0;
    rc = fast ? prepare_online_step_fast(ctx, p, sigma) : prepare_online_step(ctx, p);
    if (rc)
        return rc;

    void *args[] = {&p};
    VSOM_CUDA(ctx, cudaLaunchCooperativeKernel(reinterpret_cast<void *>(plan.kernel[p.prof ? 1 : 0]), dim3(plan.grid), dim3(plan.threads), args,
                                               plan.smem + (p.lutSmem ? lutBytes : 0), ctx->stream));
    ctx->lastPlan = &plan;
    ctx->profSamples = n;
    ctx->launches += 1;
    ctx->stepBase += n;
    return VSOM_OK;
}

} // namespace vsom
