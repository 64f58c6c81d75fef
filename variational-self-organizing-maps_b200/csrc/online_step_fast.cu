// online_step_fast.cu — K1F: the online VSOM training step for the common regime, one persistent sm_100a kernel
// per sample chunk with the shortest per-sample dependency chain this library has.
//
// Same contract and the same bits as online_step.cu's generic kernel (Som::trainSingle src/Som.cpp:885-947 =
// findBmu :291-309 / findLocalBmu :335-454 over euclidianWeightedDist :124-141, window update :899-944,
// calculateNeighbourhoodWeight :949-975, addBmu :1189-1192), for maps whose planes fit on chip, on one GPU.  Which chunks
// it runs is decided in one place, launch_online_step (online_step.cu).
//
// Why a second kernel: the generic one measures (profiles/r01_bench_default_final_candidate.json, cycles per sample
// at 64x64x128) wait 593 + scan 1535 + exchange 3323 + broadcast 248 + update 1643.  The strict per-sample dependency
// makes these ADD, so each phase is rebuilt here for latency (now: chain 896 + CTA min 135 + exchange 1560 +
// coefficients 438 + barrier 114 + update 768 + barrier 61):
//   * update and scan are fused where the work is parallel and split where it is sequential.  The warp that updates
//     a node slice (lanes = 4 consecutive elements each, 128-bit accesses) also squares the residuals of the NEXT
//     sample against the fresh means and leaves them in a `terms` row.  What remains of the scan is the part the
//     reference order forces to be sequential: one lane per node adds its row's terms k = 0,1,2,... with a chain of
//     FADDs (4 cycles each) fed by 128-bit shared-memory loads.  The f32 values added, and their order, are exactly
//     the reference's `comparer.dot(comparer)` (src/Som.cpp:140).
//   * with at most four (node, slice) items per warp their mean and S values live in registers for the whole chunk;
//     512 threads: the critical path is one warp's serial code, so registers count for more than warps.
//   * packed f32x2 arithmetic where a contraction cannot change a bit (see the note at sub2 / add2 / mul2 below).
//   * the lanes of the scan warps keep their node's grid position and weightMap entry in registers; after the exchange
//     the same lanes turn the BMU into per-node update coefficients (window test against a host-built table of
//     [start,end) per BMU column / row, neighbourhood table lookup), 32 nodes per instruction.
//   * the (distance, y, x) key carries the BMU's grid position, so nobody divides by the map width.
//   * trainSingle's return value (distance of the sample to its UPDATED BMU, :946) is produced the same way: the
//     updating warp leaves the squared residuals in a `pend` row and an otherwise idle lane adds them up during the
//     next sample's scan.  bmuHits are counted in shared memory and flushed once per chunk.
//   * samples are prefetched two ahead with cp.async into a ring of four, by one warp.
//   * the rows of the grid-wide exchange are placed by measured L2 die ("L2 die calibration" below,
//     profiles/r01_exchange_micro.md): exchange 2975 -> 1545 cycles.
//   * CLR: rows [A || B] in shared memory, pairs gathered once per sample; sigma <= 1: self-validating tagged distances
//     in global memory and the reference's greedy walk after the exchange.
#include "common.cuh"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <mutex>

namespace vsom
{

constexpr int kFThreads = 512;
constexpr int kFWarps = kFThreads / 32;
constexpr int kFMaxSlotsPerLane = 5; // the exchange row of a CTA is read by one warp: at most 160 CTAs
constexpr int kFMaxCtas = 32 * kFMaxSlotsPerLane;
constexpr size_t kFStaticSmem = 4096;
constexpr int kFPoolBlocks = 1024; // 2 KB blocks of the exchange row pool (2 MB per context)
constexpr int kWalkReplicas = 1;   // copies of the per-step distance array of the local-walk regime (8 copies measured slower:
                                   // the walk is bound by L2 round trips per step, not by readers queueing on a line)

__device__ __forceinline__ void named_bar_sync(int id, int threads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory"); }
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }

// ---- packed f32x2 arithmetic (sm_100 FADD2 / FMUL2): two IEEE round-to-nearest operations per issue slot.
// CAUTION: ptxas contracts mul.rn.f32x2 + add.rn.f32x2 into FFMA2 even under --fmad=false (it never does that to the
// scalar .rn forms).  The packed forms are therefore used only where a contraction cannot change a bit: subtractions,
// products that are not followed by an addition in registers, and the Median update, whose products are exact
// (one factor is -1, 0 or +1), so that fma(a, b, c) == a * b + c with separate roundings.
__device__ __forceinline__ u64 pk(float2 v) { return (static_cast<u64>(__float_as_uint(v.y)) << 32) | __float_as_uint(v.x); }
__device__ __forceinline__ float2 unpk(u64 v) { return make_float2(__uint_as_float(static_cast<unsigned>(v)), __uint_as_float(static_cast<unsigned>(v >> 32))); }
__device__ __forceinline__ float2 sub2(float2 a, float2 b)
{
    u64 d;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(pk(a)), "l"(pk(b)));
    return unpk(d);
}
__device__ __forceinline__ float2 add2(float2 a, float2 b)
{
    u64 d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(pk(a)), "l"(pk(b)));
    return unpk(d);
}
__device__ __forceinline__ float2 mul2(float2 a, float2 b)
{
    u64 d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(pk(a)), "l"(pk(b)));
    return unpk(d);
}

// two elements of src/Som.cpp:912-941 (sigma is evaluated lazily at the end of the chunk):
//   d0 = Stepper(x, m); m' = m + c * d0; d1 = Stepper(x, m'); S += nwf * (d0 * d1)
// the packed form of K1's scalar update_element<TR> (online_step.cu), whose bits it must reproduce element by element
template <int TR>
__device__ __forceinline__ void fast_update_pair(float2 x, float c, float nwf, float2 &m, float2 &S)
{
    if (TR == VSOM_MEDIAN)
    {
        float2 d0 = sub2(x, m);
        d0 = make_float2(median_sign(d0.x), median_sign(d0.y));
        const float2 m1 = add2(m, mul2(make_float2(c, c), d0)); // exact product: contraction-proof (see above)
        float2 d1 = sub2(x, m1);
        d1 = make_float2(median_sign(d1.x), median_sign(d1.y));
        S = add2(S, mul2(make_float2(nwf, nwf), mul2(d0, d1))); // exact products again
        m = m1;
    }
    else
    {
        const float2 d0 = sub2(x, m);
        const float2 m1 = make_float2(__fadd_rn(m.x, __fmul_rn(c, d0.x)), __fadd_rn(m.y, __fmul_rn(c, d0.y))); // scalar: never contracted
        const float2 d1 = sub2(x, m1);
        const float2 q = mul2(d0, d1);
        S = make_float2(__fadd_rn(S.x, __fmul_rn(nwf, q.x)), __fadd_rn(S.y, __fmul_rn(nwf, q.y)));
        m = m1;
    }
}

template <int TR>
__device__ __forceinline__ void fast_update4(const float4 xv, float c, float nwf, float4 &mv, float4 &sv)
{
    float2 m0 = make_float2(mv.x, mv.y), m1 = make_float2(mv.z, mv.w), s0 = make_float2(sv.x, sv.y), s1 = make_float2(sv.z, sv.w);
    fast_update_pair<TR>(make_float2(xv.x, xv.y), c, nwf, m0, s0);
    fast_update_pair<TR>(make_float2(xv.z, xv.w), c, nwf, m1, s1);
    mv = make_float4(m0.x, m0.y, m1.x, m1.y);
    sv = make_float4(s0.x, s0.y, s1.x, s1.y);
}

// squared residuals of four elements: r = model - value (Comparer, src/Transformation.cpp:7-8, :45-46), r * r
__device__ __forceinline__ float4 sq_res4(const float4 m, const float4 x)
{
    const float2 r0 = sub2(make_float2(m.x, m.y), make_float2(x.x, x.y)), r1 = sub2(make_float2(m.z, m.w), make_float2(x.z, x.w));
    const float2 q0 = mul2(r0, r0), q1 = mul2(r1, r1);
    return make_float4(q0.x, q0.y, q1.x, q1.y);
}

__device__ __forceinline__ void add4(float &s, const float4 a)
{
    s = __fadd_rn(s, a.x);
    s = __fadd_rn(s, a.y);
    s = __fadd_rn(s, a.z);
    s = __fadd_rn(s, a.w);
}

// s = ((t0 + t1) + t2) + ... over a row of n16 blocks of 16 terms (zero padded; + 0 terms do not change a sum of squares).
// 128 dependent FADDs cost 4 cycles each; the next block's four 128-bit loads are issued before the current block's adds.
__device__ __forceinline__ float chain_terms(const float *row, int n16)
{
    const float4 *r4 = reinterpret_cast<const float4 *>(row);
    float s = 0.0f;
    float4 a0 = r4[0], a1 = r4[1], a2 = r4[2], a3 = r4[3];
#pragma unroll 2
    for (int g = 1; g < n16; ++g)
    {
        r4 += 4;
        const float4 b0 = r4[0], b1 = r4[1], b2 = r4[2], b3 = r4[3];
        add4(s, a0);
        add4(s, a1);
        add4(s, a2);
        add4(s, a3);
        a0 = b0;
        a1 = b1;
        a2 = b2;
        a3 = b3;
    }
    add4(s, a0);
    add4(s, a1);
    add4(s, a2);
    add4(s, a3);
    return s;
}

// The same row of terms in Eigen's SSE2 packet order (VSOM_ORDER_EIGEN_SSE, common.cuh): eight interleaved chains over the
// first Dr / 8 * 8 terms, res0 + res1, the extra packet, (p0 + p2) + (p1 + p3), the scalar tail.  Eight independent chains:
// the adds issue back to back (one per cycle) instead of waiting 4 cycles each.
__device__ __forceinline__ float chain_terms_eigen(const float *row, int Dr)
{
    const float4 *r4 = reinterpret_cast<const float4 *>(row);
    EigenSseSum acc;
    const int n8 = Dr >> 3;
    // two blocks of eight per turn, the next turn's four 128-bit loads issued before this turn's adds (the loads' latency
    // must stay off the chains, exactly like in chain_terms)
    int b = 0;
    if (n8 >= 2)
    {
        float4 u0 = r4[0], v0 = r4[1], u1 = r4[2], v1 = r4[3];
        for (b = 2; b + 2 <= n8; b += 2)
        {
            const float4 nu0 = r4[2 * b], nv0 = r4[2 * b + 1], nu1 = r4[2 * b + 2], nv1 = r4[2 * b + 3];
            const float t0[8] = {u0.x, u0.y, u0.z, u0.w, v0.x, v0.y, v0.z, v0.w}, t1[8] = {u1.x, u1.y, u1.z, u1.w, v1.x, v1.y, v1.z, v1.w};
            acc.block(t0);
            acc.block(t1);
            u0 = nu0;
            v0 = nv0;
            u1 = nu1;
            v1 = nv1;
        }
        const float t0[8] = {u0.x, u0.y, u0.z, u0.w, v0.x, v0.y, v0.z, v0.w}, t1[8] = {u1.x, u1.y, u1.z, u1.w, v1.x, v1.y, v1.z, v1.w};
        acc.block(t0);
        acc.block(t1);
    }
    else
        b = 0;
    for (; b < n8; ++b) // an odd block count (or a single block)
    {
        const float4 u = r4[2 * b], v = r4[2 * b + 1];
        const float t[8] = {u.x, u.y, u.z, u.w, v.x, v.y, v.z, v.w};
        acc.block(t);
    }
    const int nrest = Dr & 7;
    float rest[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (nrest) // the row is at least 4 floats longer than its padded length: these reads stay inside it
    {
        const float4 u = r4[2 * n8], v = r4[2 * n8 + 1];
        rest[0] = u.x;
        rest[1] = u.y;
        rest[2] = u.z;
        rest[3] = u.w;
        rest[4] = v.x;
        rest[5] = v.y;
        rest[6] = v.z;
        rest[7] = v.w;
    }
    return acc.finish(rest, nrest);
}
// The eight chains of the Eigen SSE2 order on EIGHT consecutive lanes (lane c sums the terms k = c mod 8), combined with the
// fixed butterfly xor 4 (res0 + res1), [+ the extra packet], xor 2, xor 1 ((p0 + p2) + (p1 + p3): float addition commutes, so
// every lane ends with the same bits), then the scalar tail — Dr / 8 dependent adds instead of Dr (or Dr / 8 turns of eight).
// All 32 lanes of the warp call it (shuffles).
__device__ __forceinline__ float chain_lanes8(const float *row, int Dr, int c)
{
    const int n8 = Dr >> 3;
    float a = 0.0f;
    const float *q = row + c;
    // groups of eight terms of this lane's chain (one term per block of eight): the next group's eight loads are issued before
    // the current group's eight dependent adds — left to itself the compiler puts all loads of a turn in front of its adds
    // and the chain waits for them every turn (ncu: 110 cycles per turn instead of ~40)
    int b = 0;
    if (n8 >= 8)
    {
        float v[8], w[8];
#pragma unroll
        for (int j = 0; j < 8; ++j)
            v[j] = q[8 * j];
#pragma unroll 1
        for (b = 8; b + 8 <= n8; b += 8)
        {
#pragma unroll
            for (int j = 0; j < 8; ++j)
                w[j] = q[8 * (b + j)];
#pragma unroll
            for (int j = 0; j < 8; ++j)
                a = __fadd_rn(a, v[j]);
#pragma unroll
            for (int j = 0; j < 8; ++j)
                v[j] = w[j];
        }
#pragma unroll
        for (int j = 0; j < 8; ++j)
            a = __fadd_rn(a, v[j]);
    }
#pragma unroll 1
    for (; b < n8; ++b)
        a = __fadd_rn(a, q[8 * b]);
    float r = __fadd_rn(a, __shfl_xor_sync(0xffffffffu, a, 4));
    const int nrest = Dr & 7;
    const float *rest = row + (n8 << 3);
    int k = 0;
    if (nrest >= 4)
    {
        r = __fadd_rn(r, rest[c & 3]);
        k = 4;
    }
    r = __fadd_rn(r, __shfl_xor_sync(0xffffffffu, r, 2));
    r = __fadd_rn(r, __shfl_xor_sync(0xffffffffu, r, 1));
    for (; k < nrest; ++k)
        r = __fadd_rn(r, rest[k]);
    return r;
}
__device__ __forceinline__ float chain_any(const float *row, int n16, int Dr, int eigen) { return eigen ? chain_terms_eigen(row, Dr) : chain_terms(row, n16); }

// ---- CLR (src/Transformation.cpp:79-167): squared residuals of four pairs against a node (clr_residual, common.cuh).
// xi / xj: the sample's elements already gathered per pair (x' = x[pi_q], y' = x[pj_q] are the same for every node)
__device__ __forceinline__ float4 clr_terms4(const float4 a, const float4 b, const float4 xi, const float4 xj)
{
    float4 t;
    float r = clr_residual(a.x, b.x, xi.x, xj.x);
    t.x = __fmul_rn(r, r);
    r = clr_residual(a.y, b.y, xi.y, xj.y);
    t.y = __fmul_rn(r, r);
    r = clr_residual(a.z, b.z, xi.z, xj.z);
    t.z = __fmul_rn(r, r);
    r = clr_residual(a.w, b.w, xi.w, xj.w);
    t.w = __fmul_rn(r, r);
    return t;
}

// key layout: [63:32] distance bits | [31:20] y | [19:8] x | [7:0] tag.  (y, x) orders like the node index y*W + x.
__device__ __forceinline__ u64 make_key_xy(float d, unsigned x, unsigned y, unsigned tag)
{
    unsigned bits = __float_as_uint(d);
    if (d != d)
        bits = (x | y) == 0 ? 0u : 0x7fffffffu; // NaN never wins, except at node 0 which seeds findBmu (src/Som.cpp:293)
    return (static_cast<u64>(bits) << 32) | (static_cast<u64>(y) << 20) | (static_cast<u64>(x) << 8) | tag;
}

__device__ __forceinline__ unsigned ld_relaxed_gpu_u32(const unsigned *p)
{
    unsigned v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// IPW > 0: every warp owns at most IPW (node, 128-element slice) items, whose mean and S values then live in REGISTERS
// for the whole chunk (configs 1 and 2); IPW == 0: the owned rows live in shared memory and the warps loop over the items.
// 256 threads: the per-sample critical path is one warp's serial code, so registers (no rematerialised addresses) matter
// more than warps; the update phase is issue-bound either way.
template <int TR, int IPW, bool PROF>
__global__ void __launch_bounds__(kFThreads, 1) online_step_fast_kernel(const StepParams p)
{
    constexpr int NI = IPW > 0 ? IPW : 1;
    extern __shared__ __align__(16) unsigned char smemRaw[];
    __shared__ u64 *sRowPtr[2][kFMaxCtas]; // exchange row of every CTA (two buffers), homed on that CTA's L2 die
    __shared__ u64 sWarpKey[kFWarps];
    __shared__ int sPend[2];  // owned node that was the BMU of sample t (slot t & 1), -1: not ours
    __shared__ unsigned sBmu; // y << 12 | x of the current sample's BMU
    __shared__ int sAbort;
    __shared__ long long sProf[8];

    const int G = gridDim.x, b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int Lmax = (p.nodeCount + G - 1) / G;
    const int L = (p.nodeCount - b + G - 1) / G; // G <= nodeCount: every CTA owns at least one node; L <= kFThreads
    const int Lpad = (Lmax + 3) & ~3;
    // CLR (combinatorial linear regression, src/Transformation.cpp:79-167): the model of a node is [A(P) || B(P)], the
    // residual has one element per pair q: r_q = (A_q x[pi_q] + B_q) - x[pj_q].  Items, terms rows and the chain run over
    // the P pairs; the shared-memory rows hold [A(Ppad) || B(Ppad)].  CLR always takes the shared-memory-row mode.
    constexpr bool kClr = TR == VSOM_CLR;
    const int Ppad = (p.P + 3) & ~3;
    const int DmPad = kClr ? Ppad : (p.Dm + 3) & ~3; // length of the residual / terms row (padded)
    const int XS = kClr ? ((p.Din + 3) & ~3) + 4 : DmPad; // ring slot of a sample; CLR keeps four zeros behind it for the pad pairs
    const int stride = p.smStride;     // terms rows: 16 q + 4 floats, 16 q >= DmPad
    const int rstride = kClr ? 2 * Ppad : stride; // mean / S rows (shared-memory-row mode)
    const int n16 = (stride - 4) >> 4; // blocks of 16 terms the chain walks
    // lanes per owned node in the scan: 1, or 8 in the Eigen order when the host chose so (long rows, or all nodes still fit one warp)
    const int LPN = p.lanesPerNode;
    const int nSW = (L * LPN + 31) >> 5; // warps whose lanes own a node (or an eighth of one) each
    const int nCh = (DmPad + 127) >> 7;
    const int items = L * nCh;
    const unsigned n = static_cast<unsigned>(p.n); // the host keeps chunks below 2^32 samples on this path

    // ---- carve shared memory (every region 16-byte aligned)
    float *xs = reinterpret_cast<float *>(smemRaw);                        // [4][XS] sample ring
    float2 *coef = reinterpret_cast<float2 *>(xs + 4 * XS);                // [Lpad] {step coefficient, (float)nw}; nw < 0: outside the window
    unsigned *hitsS = reinterpret_cast<unsigned *>(coef + Lpad);           // [Lpad] bmuHits of this chunk
    unsigned *touchedS = hitsS + Lpad;                                     // [Lpad] node visited in this chunk (epilogue only)
    float *wS = reinterpret_cast<float *>(touchedS + Lpad);                // [Lpad] final weightMap entries (epilogue only)
    unsigned *winX = reinterpret_cast<unsigned *>(wS + Lpad);              // [Wpad] startX | endX << 16 per BMU column
    const int Wpad = (p.W + 3) & ~3, Hpad = (p.H + 3) & ~3;
    unsigned *winY = winX + Wpad;                                          // [Hpad]
    float *tBase = reinterpret_cast<float *>(winY + Hpad);                 // [Lmax][stride] squared residuals of the next sample
    float *pendRow = tBase + static_cast<size_t>(Lmax) * stride;           // [stride] squared residuals of the sample against its updated BMU
    float *mBase = pendRow + stride;                                       // [Lmax][rstride] means      (IPW == 0 only)
    float *sBase = mBase + (IPW > 0 ? 0 : static_cast<size_t>(Lmax) * rstride); // [Lmax][rstride] Welford S  (IPW == 0 only)
    ushort4 *pairS = reinterpret_cast<ushort4 *>(sBase + (IPW > 0 ? 0 : static_cast<size_t>(Lmax) * rstride)); // CLR: [2][Ppad / 4] pair tables pi, pj
    float *gS = reinterpret_cast<float *>(pairS + (kClr ? 2 * (Ppad >> 2) : 0));   // CLR: [3][2][Ppad] x' = x[pi], y' = x[pj] of samples t, t+1, t+2
    LutEntry *lutS = reinterpret_cast<LutEntry *>(gS + (kClr ? 6 * Ppad : 0));     // optional copy of the neighbourhood table
    if (kClr)
    {
        unsigned short *pt = reinterpret_cast<unsigned short *>(pairS);
        const unsigned short zeroAt = static_cast<unsigned short>(XS - 4); // pad pairs read the zeros behind the sample
        for (int q = tid; q < Ppad; q += kFThreads)
        {
            pt[q] = q < p.P ? p.pairI[q] : zeroAt;
            pt[Ppad + q] = q < p.P ? p.pairJ[q] : zeroAt;
        }
    }

    // ---- prologue
    // exchange rows: this CTA claims a row pair homed on the L2 die of the SM it runs on, publishes the choice, and after
    // a one-off grid barrier (cooperative launch: all CTAs are resident) everybody knows everybody's rows.
    if (tid == 0)
    {
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        const int die = p.dieOfSm[smid & 255];
        const unsigned idx = atomicAdd(p.rowCtr + die, 1u);
        p.rowOf[b] = die * kFMaxCtas + static_cast<int>(idx);
        __threadfence();
        atomicAdd(p.rowCtr + 2, 1u);
        const long long b0 = clock64();
        while (ld_relaxed_gpu_u32(p.rowCtr + 2) < static_cast<unsigned>(G))
            if (clock64() - b0 > p.timeoutCycles) // cooperative launch: all CTAs are resident, so this is a bug, not a wait
            {
                *p.err = 1;
                break;
            }
        __threadfence();
    }
    if (p.lutSmem)
        for (int i = tid; i < p.lutCount; i += kFThreads)
            lutS[i] = p.lut[i];
    for (int i = tid; i < p.W; i += kFThreads)
        winX[i] = p.winTab[i];
    for (int i = tid; i < p.H; i += kFThreads)
        winY[i] = p.winTab[p.W + i];
    for (int l = tid; l < Lpad; l += kFThreads)
    {
        hitsS[l] = 0;
        touchedS[l] = 0;
    }
    for (int k = tid; k < 4 * XS; k += kFThreads)
        xs[k] = 0.0f; // pad lanes of the 128-bit paths stay zero
    for (int k = tid; k < stride; k += kFThreads)
        pendRow[k] = 0.0f;
    for (int l = warp; l < L; l += kFWarps)
    {
        const size_t g = (static_cast<size_t>(l) * G + b) * p.rowStride;
        for (int k = lane; k < stride; k += 32)
        {
            tBase[l * stride + k] = 0.0f;
            if (IPW == 0 && !kClr)
            {
                const bool in = k < p.Dm;
                mBase[l * stride + k] = in ? p.mean[g + k] : 0.0f;
                sBase[l * stride + k] = in ? p.S[g + k] : 0.0f;
            }
        }
        if (kClr)
            for (int k = lane; k < rstride; k += 32)
            {
                const int half = k >= Ppad ? 1 : 0, q = k - half * Ppad;
                const bool in = q < p.P;
                mBase[l * rstride + k] = in ? p.mean[g + half * p.P + q] : 0.0f;
                sBase[l * rstride + k] = in ? p.S[g + half * p.P + q] : 0.0f;
            }
    }
    if (tid == 0)
    {
        sAbort = 0;
        sPend[0] = sPend[1] = -1;
        for (int i = 0; i < 8; ++i)
            sProf[i] = 0;
    }
    // IPW > 0: this warp's items it = warp + kFWarps * j, four mean / S values per lane and item
    int rl[NI], rk[NI];
    bool ract[NI];
    float4 rm[NI], rs[NI];
#pragma unroll
    for (int j = 0; j < NI; ++j)
    {
        const int it = warp + kFWarps * j;
        rl[j] = it / nCh;
        rk[j] = ((it - rl[j] * nCh) << 7) + (lane << 2);
        ract[j] = IPW > 0 && it < items && rk[j] < DmPad;
        if (!ract[j])
        {
            rl[j] = 0; // inactive: loads of the update phase stay in bounds, nothing is stored
            rk[j] = 0;
        }
        rm[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        rs[j] = rm[j];
        if (ract[j])
        {
            const size_t g = (static_cast<size_t>(rl[j]) * G + b) * p.rowStride + rk[j];
            float *m = reinterpret_cast<float *>(&rm[j]), *s = reinterpret_cast<float *>(&rs[j]);
#pragma unroll
            for (int e = 0; e < 4; ++e)
                if (rk[j] + e < p.Dm)
                {
                    m[e] = p.mean[g + e];
                    s[e] = p.S[g + e];
                }
        }
    }
    // per-lane state of the scan warps: thread <-> owned node
    const int myL = LPN == 8 ? tid >> 3 : tid, mySub = LPN == 8 ? tid & 7 : 0;
    const bool inScan = myL < L;               // this lane takes part in its node's chain
    const bool hasNode = inScan && mySub == 0; // ... and keeps the node's state (position, weightMap entry, coefficients)
    unsigned myX = 0, myY = 0;
    float myW = 0.0f;
    unsigned myTouched = 0;
    if (hasNode)
    {
        const unsigned node = static_cast<unsigned>(p.node0 + myL * G + b);
        myX = node % static_cast<unsigned>(p.W);
        myY = node / static_cast<unsigned>(p.W);
        myW = p.weight[static_cast<size_t>(myL) * G + b];
    }
    const float *myTerms = tBase + (inScan ? myL : 0) * stride;
    __syncthreads();
    for (int i = tid; i < 2 * G; i += kFThreads)
    {
        const int d = i >> 1, buf = i & 1;
        const int r = p.rowOf[d]; // written before the grid barrier above
        sRowPtr[buf][d] = p.rowPool + static_cast<size_t>(p.rowBlocks[2 * r + buf]) * 256;
    }

    // sample prefetch by ONE warp that is not the first scan warp (everything the other warps execute at the top of a
    // step competes with the scan warp's FADD chain for issue slots); loops kept rolled to stay small
    constexpr int kPrefetchWarp = kFWarps - 2;
    const float *xsrc = p.x; // next sample to fetch (prefetch warp only)
    int xdst = 0;            // its ring slot offset
    auto prefetch = [&]() {
        float *dst = xs + xdst;
        if (p.xVec)
        {
#pragma unroll 1
            for (int k = lane * 4; k < p.Din; k += 128)
                cp_async16(dst + k, xsrc + k);
        }
        else
        {
#pragma unroll 1
            for (int k = lane; k < p.Din; k += 32)
                cp_async4(dst + k, xsrc + k);
        }
        cp_async_commit();
        xsrc += p.Din;
        xdst = xdst + XS == 4 * XS ? 0 : xdst + XS;
    };
    if (warp == kPrefetchWarp)
    {
        if (n > 0)
            prefetch();
        if (n > 1)
            prefetch();
        cp_async_wait_all();
    }
    __syncthreads();
    // CLR: every thread below Ppad owns one pair for the gathers
    int gpi = 0, gpj = 0;
    if (kClr && tid < Ppad)
    {
        const unsigned short *pt = reinterpret_cast<const unsigned short *>(pairS);
        gpi = pt[tid];
        gpj = pt[Ppad + tid];
    }
    auto gather = [&](int slot, const float *x) { // x' and y' of one sample for every pair
        for (int q = tid; q < Ppad; q += kFThreads)
        {
            const unsigned short *pt = reinterpret_cast<const unsigned short *>(pairS);
            const int qi = q == tid ? gpi : pt[q], qj = q == tid ? gpj : pt[Ppad + q];
            gS[(slot * 2) * Ppad + q] = x[qi];
            gS[(slot * 2 + 1) * Ppad + q] = x[qj];
        }
    };
    if (kClr)
    {
        gather(0, xs);
        if (n > 1)
            gather(1, xs + XS);
        __syncthreads();
    }
    // terms of sample 0 against the initial means
    if (IPW > 0)
    {
#pragma unroll
        for (int j = 0; j < NI; ++j)
            if (ract[j])
                *reinterpret_cast<float4 *>(tBase + rl[j] * stride + rk[j]) = sq_res4(rm[j], *reinterpret_cast<const float4 *>(xs + rk[j]));
    }
    else
        for (int it = warp; it < items; it += kFWarps)
        {
            const int l = nCh > 1 ? it / nCh : it, ch = nCh > 1 ? it - l * nCh : 0;
            const int k = (ch << 7) + (lane << 2);
            if (k < DmPad)
            {
                if (kClr)
                {
                    const float4 av = *reinterpret_cast<const float4 *>(mBase + l * rstride + k), bv = *reinterpret_cast<const float4 *>(mBase + l * rstride + Ppad + k);
                    *reinterpret_cast<float4 *>(tBase + l * stride + k) =
                        clr_terms4(av, bv, *reinterpret_cast<const float4 *>(gS + k), *reinterpret_cast<const float4 *>(gS + Ppad + k));
                }
                else
                    *reinterpret_cast<float4 *>(tBase + l * stride + k) =
                        sq_res4(*reinterpret_cast<const float4 *>(mBase + l * stride + k), *reinterpret_cast<const float4 *>(xs + k));
            }
        }
    __syncthreads();

    long long c0 = 0, c1 = 0, c2 = 0, c3 = 0, c4 = 0, c5 = 0, c6 = 0;
    int curOff = 0, nextOff = XS; // ring offsets of samples t and t+1
    int gSlot = 0;                // CLR: gather slot of sample t (t mod 3)
    // the scan warp's serial code is the critical path: keep what it reads from the parameter block in registers
    int lutW = p.lutW, lutInSmem = p.lutSmem, expDecay = p.decay == VSOM_EXPONENTIAL ? 1 : 0, eigenOrder = p.order == VSOM_ORDER_EIGEN_SSE ? 1 : 0;
    asm volatile("" : "+r"(lutW), "+r"(lutInSmem), "+r"(expDecay), "+r"(eigenOrder));
    for (unsigned t = 0; t < n; ++t)
    {
        if (PROF && tid == 0)
            c0 = clock64();
        const unsigned tag = (t >> 1) & 0xffu;
        const int par = static_cast<int>(t & 1u);

        if (warp == kPrefetchWarp && t + 2 < n)
            prefetch(); // sample t+2 on its way while this step runs (its slot held sample t-2)

        // ---- owed output of sample t-1: distance to its updated BMU (src/Som.cpp:946) + addBmu (:1189-1192)
        if (tid == kFThreads - 1 && t > 0)
        {
            const int pl = sPend[par ^ 1];
            if (pl >= 0)
            {
                const float d = chain_any(pendRow, n16, p.Dr, eigenOrder);
                if (p.outBmu)
                    p.outBmu[t - 1] = static_cast<unsigned>(p.node0 + pl * G + b);
                if (p.outDist)
                    p.outDist[t - 1] = d;
                hitsS[pl] += 1;
            }
        }

        // ---- scan: the sequential part of the distance, one lane per owned node
        if (warp < nSW)
        {
            u64 key = ~0ull;
            float dScan = 0.0f;
            if (LPN == 8)
                dScan = chain_lanes8(myTerms, p.Dr, mySub); // every lane of the scan warps (shuffles); lanes without a node read row 0
            else if (hasNode)
                dScan = chain_any(myTerms, n16, p.Dr, eigenOrder);
            if (hasNode)
            {
                const float d = dScan;
                key = make_key_xy(d, myX, myY, tag);
                if (p.localSearch) // sigma <= 1: the walk below reads distances of arbitrary nodes; the word validates itself.
                {                  // (kWalkReplicas copies, CTA b reads copy b % kWalkReplicas)
                    const u64 w = (static_cast<u64>(__float_as_uint(d)) << 32) | (t + 1u);
                    u64 *dst = p.distTag + static_cast<size_t>(par) * kWalkReplicas * p.nodeCount + (myY * static_cast<unsigned>(p.W) + myX);
#pragma unroll
                    for (int r = 0; r < kWalkReplicas; ++r)
                        st_relaxed_gpu(dst + static_cast<size_t>(r) * p.nodeCount, w);
                }
            }
            if (PROF && tid == 0)
                c1 = clock64();
            key = warp_min_key(key);
            if (nSW > 1)
            {
                if (lane == 0)
                    sWarpKey[warp] = key;
                named_bar_sync(1, nSW * 32);
            }
            unsigned bxy = 0;
            bool abort = false;
            if (warp == 0)
            {
                if (nSW > 1)
                    key = warp_min_key(lane < nSW ? sWarpKey[lane] : ~0ull);
                if (PROF && tid == 0)
                    c2 = clock64();
                // ---- grid-wide min-loc: push the key into every CTA's row, then poll the own row
                u64 *const *rp = sRowPtr[par];
#pragma unroll
                for (int j = 0; j < kFMaxSlotsPerLane; ++j)
                    if (lane + 32 * j < G)
                        st_relaxed_gpu(rp[lane + 32 * j] + b, key);
                const u64 *row = rp[b];
                const u64 filler = (~0ull << 8) | tag;
                u64 m;
                long long t0 = 0;
                // one batch of loads per round, all in flight together.  (Two batches in flight were measured twice and
                // lose: exchange 1529 -> 1855 cycles; more polling traffic on the lines the keys arrive in delays them.)
                if (p.pollDelay > 0)
                {
                    const long long w0 = clock64();
                    while (clock64() - w0 < p.pollDelay)
                        ;
                }
                for (unsigned round = 0;; ++round)
                {
                    u64 v[kFMaxSlotsPerLane];
#pragma unroll
                    for (int j = 0; j < kFMaxSlotsPerLane; ++j)
                    {
                        const int i = lane + 32 * j;
                        v[j] = i < G ? ld_relaxed_gpu(row + i) : filler;
                    }
                    m = ~0ull;
                    int ok = 1;
#pragma unroll
                    for (int j = 0; j < kFMaxSlotsPerLane; ++j)
                    {
                        ok &= (static_cast<unsigned>(v[j] & 0xff) == tag);
                        m = u64_min(m, v[j]);
                    }
                    if (__all_sync(0xffffffffu, ok))
                        break;
                    if ((round & 63) == 63)
                    {
                        if (t0 == 0)
                            t0 = clock64();
                        else if (__any_sync(0xffffffffu, clock64() - t0 > p.timeoutCycles))
                        {
                            abort = true;
                            break;
                        }
                    }
                }
                m = warp_min_key(m);
                bxy = static_cast<unsigned>(m >> 8) & 0xffffffu;
                if (p.localSearch && !abort)
                {
                    // findLocalBmu regime (src/Som.cpp:889-892, :335-454): every CTA has seen every CTA's key of this step, so
                    // every distance of this step has been stored; a word whose tag is not yet this step's is re-read.
                    // Every CTA walks the same path (lane 0), like every CTA takes the same global minimum.
                    if (lane == 0)
                    {
                        const u64 *dt = p.distTag + (static_cast<size_t>(par) * kWalkReplicas + (b % kWalkReplicas)) * p.nodeCount;
                        const unsigned want = t + 1u;
                        const unsigned bmu = local_bmu_walk(
                            [&](u64 i) {
                                u64 w = ld_relaxed_gpu(dt + i);
                                if (static_cast<unsigned>(w) != want) // written by a CTA whose key this CTA has already seen: a re-read or two
                                {
                                    const long long w0 = clock64();
                                    do
                                        w = ld_relaxed_gpu(dt + i);
                                    while (static_cast<unsigned>(w) != want && clock64() - w0 < p.timeoutCycles);
                                    if (static_cast<unsigned>(w) != want)
                                        *p.err = 1;
                                }
                                return __uint_as_float(static_cast<unsigned>(w >> 32));
                            },
                            static_cast<u64>(p.W), static_cast<u64>(p.H), p.lastIn ? p.lastIn[t] : 0ull);
                        bxy = ((bmu / static_cast<unsigned>(p.W)) << 12) | (bmu % static_cast<unsigned>(p.W));
                    }
                    bxy = __shfl_sync(0xffffffffu, bxy, 0);
                }
                if (lane == 0)
                {
                    sBmu = bxy;
                    sPend[par] = -1;
                    if (abort)
                    {
                        sAbort = 1;
                        *p.err = 1;
                    }
                }
                if (PROF && tid == 0)
                    c3 = clock64();
                if (nSW > 1)
                    named_bar_sync(2, nSW * 32);
                else
                    __syncwarp();
            }
            else
            {
                named_bar_sync(2, nSW * 32);
                bxy = sBmu;
                abort = sAbort != 0;
            }
            // ---- per owned node: window test, neighbourhood entry, weightMap and step coefficient (src/Som.cpp:899-939)
            if (hasNode && !abort)
            {
                const unsigned bx = bxy & 0xfffu, by = bxy >> 12;
                const unsigned wx = winX[bx], wy = winY[by];
                float2 cf = make_float2(0.0f, -1.0f);
                if (myX >= (wx & 0xffffu) && myX < (wx >> 16) && myY >= (wy & 0xffffu) && myY < (wy >> 16))
                {
                    const int dx = myX > bx ? myX - bx : bx - myX, dy = myY > by ? myY - by : by - myY;
                    cf = step_coefficient(neighbourhood_entry(lutInSmem, lutS, p.lut, lutW, dx, dy), expDecay, myW);
                    myTouched = 1;
                    if (dx == 0 && dy == 0)
                        sPend[par] = myL;
                }
                coef[myL] = cf;
            }
        }
        if (warp == kPrefetchWarp)
            cp_async_wait_all(); // samples t+1 (and t+2) have landed; the barrier publishes them
        if (PROF && tid == 0)
            c4 = clock64();
        __syncthreads(); // B1: coefficients, BMU owner and sample t+1 visible
        if (sAbort)
            break;
        if (PROF && tid == 0)
            c5 = clock64();

        // ---- update of the owned nodes inside the window (src/Som.cpp:912-941) fused with the squared residuals of
        //      sample t+1 against the new means; one warp per (node, 128-element slice)
        {
            const float *xt = xs + curOff;
            const float *xn = xs + nextOff;
            const int pl = sPend[par];
            const float *gCur = gS + gSlot * 2 * Ppad, *gNext = gS + (gSlot == 2 ? 0 : gSlot + 1) * 2 * Ppad;
            if (kClr && t + 2 < n) // sample t+2 landed with barrier B1: its x', y' are needed from the next step on
                gather(gSlot == 0 ? 2 : gSlot - 1, xs + (nextOff + XS == 4 * XS ? 0 : nextOff + XS));
            if (IPW > 0)
            {
                // all loads first; when every item of the warp is inside the window (warp-uniform, the usual case while the
                // neighbourhood is wide) the items are updated in one straight-line block so that their dependency chains
                // interleave; otherwise item by item
                float2 cf[NI];
                float4 nv[NI], xv[NI];
                bool allIn = true;
#pragma unroll
                for (int j = 0; j < NI; ++j)
                {
                    cf[j] = coef[rl[j]];
                    nv[j] = *reinterpret_cast<const float4 *>(xn + rk[j]);
                    xv[j] = *reinterpret_cast<const float4 *>(xt + rk[j]);
                    allIn = allIn && ract[j] && cf[j].y >= 0.0f;
                }
                if (allIn)
                {
#pragma unroll
                    for (int j = 0; j < NI; ++j)
                        fast_update4<TR>(xv[j], cf[j].x, cf[j].y, rm[j], rs[j]);
#pragma unroll
                    for (int j = 0; j < NI; ++j)
                    {
                        if (rl[j] == pl)
                            *reinterpret_cast<float4 *>(pendRow + rk[j]) = sq_res4(rm[j], xv[j]);
                        *reinterpret_cast<float4 *>(tBase + rl[j] * stride + rk[j]) = sq_res4(rm[j], nv[j]);
                    }
                }
                else
                {
#pragma unroll
                    for (int j = 0; j < NI; ++j)
                        if (ract[j])
                        {
                            if (cf[j].y >= 0.0f)
                            {
                                fast_update4<TR>(xv[j], cf[j].x, cf[j].y, rm[j], rs[j]);
                                if (rl[j] == pl)
                                    *reinterpret_cast<float4 *>(pendRow + rk[j]) = sq_res4(rm[j], xv[j]);
                            }
                            *reinterpret_cast<float4 *>(tBase + rl[j] * stride + rk[j]) = sq_res4(rm[j], nv[j]);
                        }
                }
            }
            else
                for (int it = warp; it < items; it += kFWarps)
                {
                    const int l = nCh > 1 ? it / nCh : it, ch = nCh > 1 ? it - l * nCh : 0;
                    const int k = (ch << 7) + (lane << 2);
                    if (kClr)
                    {
                        if (k < DmPad)
                        {
                            const float2 cf = coef[l];
                            float *ap = mBase + l * rstride + k, *bp = ap + Ppad;
                            float4 av = *reinterpret_cast<float4 *>(ap), bv = *reinterpret_cast<float4 *>(bp);
                            if (cf.y >= 0.0f)
                            {
                                float *sap = sBase + l * rstride + k, *sbp = sap + Ppad;
                                float4 sav = *reinterpret_cast<float4 *>(sap), sbv = *reinterpret_cast<float4 *>(sbp);
                                const float4 xi = *reinterpret_cast<const float4 *>(gCur + k), xj = *reinterpret_cast<const float4 *>(gCur + Ppad + k);
                                float4 pendv;
                                clr_update_pair(xi.x, xj.x, cf.x, cf.y, av.x, bv.x, sav.x, sbv.x, pendv.x);
                                clr_update_pair(xi.y, xj.y, cf.x, cf.y, av.y, bv.y, sav.y, sbv.y, pendv.y);
                                clr_update_pair(xi.z, xj.z, cf.x, cf.y, av.z, bv.z, sav.z, sbv.z, pendv.z);
                                clr_update_pair(xi.w, xj.w, cf.x, cf.y, av.w, bv.w, sav.w, sbv.w, pendv.w);
                                *reinterpret_cast<float4 *>(ap) = av;
                                *reinterpret_cast<float4 *>(bp) = bv;
                                *reinterpret_cast<float4 *>(sap) = sav;
                                *reinterpret_cast<float4 *>(sbp) = sbv;
                                if (l == pl)
                                    *reinterpret_cast<float4 *>(pendRow + k) = pendv;
                            }
                            *reinterpret_cast<float4 *>(tBase + l * stride + k) =
                                clr_terms4(av, bv, *reinterpret_cast<const float4 *>(gNext + k), *reinterpret_cast<const float4 *>(gNext + Ppad + k));
                        }
                    }
                    else if (k < DmPad)
                    {
                        const float2 cf = coef[l];
                        float *mp = mBase + l * stride + k;
                        float4 mv = *reinterpret_cast<float4 *>(mp);
                        const float4 nv = *reinterpret_cast<const float4 *>(xn + k);
                        if (cf.y >= 0.0f)
                        {
                            float *sp = sBase + l * stride + k;
                            float4 sv = *reinterpret_cast<float4 *>(sp);
                            const float4 xv = *reinterpret_cast<const float4 *>(xt + k);
                            fast_update4<TR>(xv, cf.x, cf.y, mv, sv);
                            *reinterpret_cast<float4 *>(mp) = mv;
                            *reinterpret_cast<float4 *>(sp) = sv;
                            if (l == pl)
                                *reinterpret_cast<float4 *>(pendRow + k) = sq_res4(mv, xv);
                        }
                        *reinterpret_cast<float4 *>(tBase + l * stride + k) = sq_res4(mv, nv);
                    }
                }
        }
        curOff = nextOff;
        nextOff = nextOff + XS == 4 * XS ? 0 : nextOff + XS;
        gSlot = gSlot == 2 ? 0 : gSlot + 1;
        if (PROF && tid == 0)
            c6 = clock64();
        __syncthreads(); // B2: terms of sample t+1 and the pend row are complete
        if (PROF && tid == 0)
        {
            const long long c7 = clock64();
            sProf[0] += c1 - c0; // the FADD chain
            sProf[1] += c2 - c1; // CTA min
            sProf[2] += c3 - c2; // grid-wide exchange
            sProf[3] += c4 - c3; // coefficients
            sProf[4] += c5 - c4; // barrier B1
            sProf[5] += c6 - c5; // update + next sample's squared residuals (this warp)
            sProf[6] += c7 - c6; // barrier B2 (slowest warp's update)
        }
    }

    // ---- epilogue: last owed output, lazy sigma, write the owned rows back
    if (!sAbort && n > 0 && tid == kFThreads - 1)
    {
        const int pl = sPend[(n - 1) & 1];
        if (pl >= 0)
        {
            const float d = chain_any(pendRow, n16, p.Dr, eigenOrder);
            if (p.outBmu)
                p.outBmu[n - 1] = static_cast<unsigned>(p.node0 + pl * G + b);
            if (p.outDist)
                p.outDist[n - 1] = d;
            hitsS[pl] += 1;
        }
    }
    if (hasNode)
    {
        wS[myL] = myW;
        touchedS[myL] = myTouched;
    }
    __syncthreads();
    for (int l = tid; l < L; l += kFThreads)
    {
        const size_t q = static_cast<size_t>(l) * G + b;
        p.weight[q] = wS[l];
        if (hitsS[l])
            p.hits[q] += hitsS[l];
    }
    // sigmaMap of the visited nodes (lazy_sigma)
    if (IPW > 0)
    {
#pragma unroll
        for (int j = 0; j < NI; ++j)
            if (ract[j])
            {
                const size_t g = (static_cast<size_t>(rl[j]) * G + b) * p.rowStride + rk[j];
                const bool vis = touchedS[rl[j]] != 0;
                const float w = wS[rl[j]];
                const float *m = reinterpret_cast<const float *>(&rm[j]), *s = reinterpret_cast<const float *>(&rs[j]);
#pragma unroll
                for (int e = 0; e < 4; ++e)
                    if (rk[j] + e < p.Dm)
                    {
                        p.mean[g + e] = m[e];
                        p.S[g + e] = s[e];
                        if (vis)
                            p.sigma[g + e] = lazy_sigma(s[e], w);
                    }
            }
    }
    else
        for (int l = warp; l < L; l += kFWarps)
        {
            const size_t g = (static_cast<size_t>(l) * G + b) * p.rowStride;
            const bool vis = touchedS[l] != 0;
            const float w = wS[l];
            for (int k = lane; k < p.Dm; k += 32)
            {
                // CLR rows are [A(Ppad) || B(Ppad)] in shared memory, [A(P) || B(P)] in the plane
                const int ks = kClr ? (k < p.P ? k : Ppad + (k - p.P)) : k;
                const float sv = sBase[l * rstride + ks];
                p.mean[g + k] = mBase[l * rstride + ks];
                p.S[g + k] = sv;
                if (vis)
                    p.sigma[g + k] = lazy_sigma(sv, w);
            }
        }
    if (PROF && p.prof && tid == 0)
        for (int i = 0; i < 8; ++i)
            p.prof[static_cast<size_t>(b) * 8 + i] = sProf[i];
}

// ------------------------------------------------------------------------------------ L2 die calibration
// B200's L2 is split over two dies.  A strong (gpu-scope) store -> poll signal between two SMs costs ~480 cycles one way
// when writer, poller and the line's home partition share a die, ~735 when only the POLLER is on the line's die, and
// ~1000 and more when the poller is on the other die (tests/micro/die_bench2.cu, profiles/r01_exchange_micro.md).  The
// exchange therefore gives every CTA rows homed on the die of the SM it runs on.  Neither map is documented, so both
// are measured: (1) SM -> die, once per device and process, from the ping-pong round trip of SM pairs through one
// flag block (two clean modes, ~950 vs ~1750 cycles); (2) 2 KB block -> die, per context, from ping-pongs of same-die
// SM pairs on each block of the context's row pool.
__global__ void die_pingpong_kernel(u64 *f1, u64 *f2, int ctaA, int ctaB, int iters, u64 base, long long *out, int *smids)
{
    if (threadIdx.x != 0)
        return;
    const int b = blockIdx.x;
    if (b != ctaA && b != ctaB)
        return;
    unsigned smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    smids[b == ctaA ? 0 : 1] = static_cast<int>(smid);
    const long long t0 = clock64();
    const long long limit = 400000000ll;
    for (int t = 1; t <= iters; ++t)
    {
        const u64 v = base + t;
        if (b == ctaA)
        {
            st_relaxed_gpu(f1, v);
            while (ld_relaxed_gpu(f2) != v)
                if (clock64() - t0 > limit)
                    return;
        }
        else
        {
            while (ld_relaxed_gpu(f1) != v)
                if (clock64() - t0 > limit)
                    return;
            st_relaxed_gpu(f2, v);
        }
    }
    if (b == ctaA)
        out[0] = clock64() - t0;
}

// every pair of same-die SMs (pairOfSm / roleOfSm, indexed by %smid) ping-pongs on the blocks k = pair, pair + nPairs, ...
__global__ void die_classify_blocks_kernel(u64 *pool, int nBlocks, const int *pairOfSm, const int *roleOfSm, int nPairs, int iters, float *rtOut)
{
    if (threadIdx.x != 0)
        return;
    unsigned smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    const int pr = pairOfSm[smid & 255], role = roleOfSm[smid & 255];
    if (pr < 0)
        return;
    const long long start = clock64();
    const long long limit = 2000000000ll;
    for (int k = pr; k < nBlocks; k += nPairs)
    {
        u64 *f1 = pool + static_cast<size_t>(k) * 256, *f2 = f1 + 16;
        const long long t0 = clock64();
        for (int t = 1; t <= iters; ++t)
        {
            const u64 v = static_cast<u64>(t);
            if (role == 0)
            {
                st_relaxed_gpu(f1, v);
                while (ld_relaxed_gpu(f2) != v)
                    if (clock64() - start > limit)
                        return;
            }
            else
            {
                while (ld_relaxed_gpu(f1) != v)
                    if (clock64() - start > limit)
                        return;
                st_relaxed_gpu(f2, v);
            }
        }
        if (role == 0)
            rtOut[k] = static_cast<float>(clock64() - t0) / static_cast<float>(iters);
    }
}

// --------------------------------------------------------------------------------------------- host side

static int fast_stride(const vsom_ctx *ctx)
{
    const int DmPad = ctx->transform == VSOM_CLR ? (ctx->P + 3) & ~3 : (ctx->Dm + 3) & ~3; // residual length
    return ((DmPad + 15) & ~15) + 4; // 16 q + 4: rows 16-byte aligned, stride / 4 odd (conflict-free 128-bit access both ways)
}

// items per warp kept in registers (1, 2 or 4), 0 when the CTA owns more items than that: rows in shared memory
static int fast_ipw(const vsom_ctx *ctx, int G)
{
    if (ctx->transform == VSOM_CLR)
        return 0; // [A || B] rows stay in shared memory
    const int Lmax = (ctx->localN + G - 1) / G;
    const int nCh = (((ctx->Dm + 3) & ~3) + 127) >> 7;
    const int items = Lmax * nCh;
    for (int ipw = 1; ipw <= 4; ipw *= 2)
        if (items <= kFWarps * ipw)
            return ipw;
    return 0;
}

static size_t fast_smem(const vsom_ctx *ctx, int G, int stride)
{
    const int Lmax = (ctx->localN + G - 1) / G;
    const int Lpad = (Lmax + 3) & ~3;
    const bool clr = ctx->transform == VSOM_CLR;
    const int Ppad = (ctx->P + 3) & ~3;
    const int XS = clr ? ((ctx->Din + 3) & ~3) + 4 : (ctx->Dm + 3) & ~3;
    const int Wpad = (ctx->W + 3) & ~3, Hpad = (ctx->H + 3) & ~3;
    size_t bytes = sizeof(float) * 4 * static_cast<size_t>(XS);
    bytes += (sizeof(float2) + 2 * sizeof(unsigned) + sizeof(float)) * static_cast<size_t>(Lpad);
    bytes += sizeof(unsigned) * (static_cast<size_t>(Wpad) + Hpad);
    bytes += sizeof(float) * (static_cast<size_t>(Lmax) + 1) * stride; // terms rows + pend row
    if (fast_ipw(ctx, G) == 0)
        bytes += sizeof(float) * 2 * static_cast<size_t>(Lmax) * (clr ? 2 * Ppad : stride); // mean and S rows
    if (clr)
        bytes += sizeof(unsigned short) * 2 * static_cast<size_t>(Ppad) + sizeof(float) * 6 * static_cast<size_t>(Ppad);
    return bytes;
}

typedef void (*FastKernel)(const StepParams);
static FastKernel pick_fast(int transform, int ipw, bool prof)
{
    if (transform == VSOM_CLR)
        return prof ? online_step_fast_kernel<VSOM_CLR, 0, true> : online_step_fast_kernel<VSOM_CLR, 0, false>;
#define VSOM_FK(TR, I) {online_step_fast_kernel<TR, I, false>, online_step_fast_kernel<TR, I, true>}
#define VSOM_FKS(TR) {VSOM_FK(TR, 0), VSOM_FK(TR, 1), VSOM_FK(TR, 2), VSOM_FK(TR, 4)}
    static const FastKernel table[2][4][2] = {VSOM_FKS(VSOM_STANDARD), VSOM_FKS(VSOM_MEDIAN)};
#undef VSOM_FKS
#undef VSOM_FK
    const int slot = ipw == 4 ? 3 : ipw;
    return table[transform == VSOM_MEDIAN ? 1 : 0][slot][prof ? 1 : 0];
}

// ---- SM -> die map, measured once per device and process
struct DieMap
{
    bool tried = false, valid = false;
    int dieOfSm[256] = {};
    int count[2] = {0, 0};
};
static DieMap g_dieMap[64];
static std::mutex g_dieMapMutex; // contexts of several host threads may reach their first K1F launch together

// Two-mode split of round-trip times: threshold halfway between the lower and the upper quartile (both maps are close
// to half / half), accepted when the quartiles are clearly apart and few values sit near the threshold.
static bool split_bimodal(std::vector<float> v, float &thr)
{
    if (v.size() < 8)
        return false;
    std::sort(v.begin(), v.end());
    const float q1 = v[v.size() / 4], q3 = v[(3 * v.size()) / 4];
    thr = 0.5f * (q1 + q3);
    if (q3 < 1.3f * q1)
        return false;
    const float band = 0.15f * (q3 - q1);
    size_t near = 0, low = 0;
    for (float x : v)
    {
        near += (x > thr - band && x < thr + band) ? 1 : 0;
        low += x <= thr ? 1 : 0;
    }
    return near * 20 <= v.size() && low * 10 >= 3 * v.size() && low * 10 <= 7 * v.size();
}

static int calibrate_die_map(vsom_ctx *ctx)
{
    std::lock_guard<std::mutex> lock(g_dieMapMutex);
    DieMap &dm = g_dieMap[ctx->device & 63];
    if (dm.tried)
        return VSOM_OK;
    dm.tried = true;
    const int n = ctx->numSMs;
    if (n > 256)
        return VSOM_OK;
    u64 *flags = nullptr;
    long long *out = nullptr;
    int *smids = nullptr;
    const int kCand = 16; // candidate flag blocks (2 KB apart)
    VSOM_CUDA(ctx, cudaMalloc(&flags, 2048 * kCand));
    VSOM_CUDA(ctx, cudaMalloc(&out, sizeof(long long)));
    VSOM_CUDA(ctx, cudaMalloc(&smids, 2 * sizeof(int)));
    VSOM_CUDA(ctx, cudaMemsetAsync(flags, 0, 2048 * kCand, ctx->stream));
    const int iters = 96;
    u64 base = 0;
    bool ok = true;
    int sm0 = -1;
    auto pingpong = [&](int blk, int peer, float &cycles, int &peerSm) -> int {
        u64 *f1 = flags + static_cast<size_t>(blk) * 256, *f2 = f1 + 16;
        int a = 0, it = iters;
        VSOM_CUDA(ctx, cudaMemsetAsync(out, 0, sizeof(long long), ctx->stream));
        void *args[] = {&f1, &f2, &a, &peer, &it, &base, &out, &smids};
        VSOM_CUDA(ctx, cudaLaunchCooperativeKernel(reinterpret_cast<void *>(die_pingpong_kernel), dim3(n), dim3(32), args, 0, ctx->stream));
        long long cyc = 0;
        int ids[2] = {0, 0};
        VSOM_CUDA(ctx, cudaMemcpyAsync(&cyc, out, sizeof(cyc), cudaMemcpyDeviceToHost, ctx->stream));
        VSOM_CUDA(ctx, cudaMemcpyAsync(ids, smids, sizeof(ids), cudaMemcpyDeviceToHost, ctx->stream));
        VSOM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        base += iters + 8;
        if (cyc <= 0 || ids[1] < 0 || ids[1] > 255 || (sm0 >= 0 && ids[0] != sm0))
            ok = false; // timed out, or CTA 0 moved between launches
        sm0 = ids[0];
        cycles = static_cast<float>(cyc) / iters;
        peerSm = ids[1];
        return VSOM_OK;
    };
    // the flag block must be homed on CTA 0's own die, or the two modes of the scan below are hard to tell apart (a far
    // home adds its latency to every pair): take the candidate with the shortest round trip to the neighbouring CTA
    int flagBlk = 0;
    float bestRt = 0.f;
    for (int k = 0; k < kCand && ok; ++k)
    {
        float c = 0.f;
        int psm = 0;
        int rc = pingpong(k, 1, c, psm);
        if (rc)
            return rc;
        if (k == 0 || c < bestRt)
        {
            bestRt = c;
            flagBlk = k;
        }
    }
    std::vector<float> rt;
    std::vector<int> sm;
    for (int peer = 1; peer < n && ok; ++peer)
    {
        float c = 0.f;
        int psm = 0;
        int rc = pingpong(flagBlk, peer, c, psm);
        if (rc)
            return rc;
        rt.push_back(c);
        sm.push_back(psm);
    }
    cudaFree(flags);
    cudaFree(out);
    cudaFree(smids);
    float thr = 0.f;
    const bool bimodal = ok && split_bimodal(rt, thr);
    if (!bimodal)
    {
        std::vector<float> srt = rt;
        std::sort(srt.begin(), srt.end());
        fprintf(stderr, "[vsom] SM die calibration: ok=%d bimodal=%d thr=%.0f n=%zu min=%.0f q1=%.0f median=%.0f q3=%.0f max=%.0f\n", ok ? 1 : 0, bimodal ? 1 : 0, thr,
                srt.size(), srt.empty() ? 0.f : srt.front(), srt.empty() ? 0.f : srt[srt.size() / 4], srt.empty() ? 0.f : srt[srt.size() / 2],
                srt.empty() ? 0.f : srt[3 * srt.size() / 4], srt.empty() ? 0.f : srt.back());
    }
    if (!bimodal)
        return VSOM_OK; // leave the map invalid: rows are then taken in pool order (still correct, only slower)
    dm.dieOfSm[sm0 & 255] = 0;
    dm.count[0] = 1;
    for (size_t i = 0; i < rt.size(); ++i)
    {
        const int d = rt[i] > thr ? 1 : 0;
        dm.dieOfSm[sm[i] & 255] = d;
        dm.count[d] += 1;
    }
    dm.valid = true;
    return VSOM_OK;
}

// row pool of the context + the home die of each of its 2 KB blocks -> rowBlocks[die][slot][buffer]
static int build_row_pool(vsom_ctx *ctx)
{
    if (ctx->rowPool)
        return VSOM_OK;
    int rc = calibrate_die_map(ctx);
    if (rc)
        return rc;
    const DieMap &dm = g_dieMap[ctx->device & 63];
    VSOM_CUDA(ctx, cudaMalloc(&ctx->rowPool, static_cast<size_t>(kFPoolBlocks) * 2048));
    VSOM_CUDA(ctx, cudaMalloc(&ctx->rowMeta, sizeof(int) * (256 + 2 * 2 * kFMaxCtas + kFMaxCtas) + sizeof(unsigned) * 4));
    std::vector<int> home(kFPoolBlocks, -1);
    bool haveHomes = false;
    if (dm.valid)
    {
        // pairs of die-0 SMs, by SM id
        std::vector<int> pairOf(256, -1), roleOf(256, 0), die0;
        for (int s = 0; s < 256; ++s)
            if (dm.dieOfSm[s] == 0)
                die0.push_back(s);
        // dieOfSm defaults to 0 for ids that were never seen; keep only SM ids below the SM count
        die0.erase(std::remove_if(die0.begin(), die0.end(), [&](int s) { return s >= ctx->numSMs; }), die0.end());
        const int nPairs = static_cast<int>(die0.size()) / 2;
        for (int i = 0; i < nPairs; ++i)
        {
            pairOf[die0[2 * i]] = i;
            roleOf[die0[2 * i]] = 0;
            pairOf[die0[2 * i + 1]] = i;
            roleOf[die0[2 * i + 1]] = 1;
        }
        if (nPairs >= 4)
        {
            int *tab = nullptr;
            float *rtDev = nullptr;
            VSOM_CUDA(ctx, cudaMalloc(&tab, sizeof(int) * 512));
            VSOM_CUDA(ctx, cudaMalloc(&rtDev, sizeof(float) * kFPoolBlocks));
            VSOM_CUDA(ctx, cudaMemcpyAsync(tab, pairOf.data(), sizeof(int) * 256, cudaMemcpyHostToDevice, ctx->stream));
            VSOM_CUDA(ctx, cudaMemcpyAsync(tab + 256, roleOf.data(), sizeof(int) * 256, cudaMemcpyHostToDevice, ctx->stream));
            VSOM_CUDA(ctx, cudaMemsetAsync(rtDev, 0, sizeof(float) * kFPoolBlocks, ctx->stream));
            VSOM_CUDA(ctx, cudaMemsetAsync(ctx->rowPool, 0, static_cast<size_t>(kFPoolBlocks) * 2048, ctx->stream));
            u64 *pool = ctx->rowPool;
            int nb = kFPoolBlocks, np = nPairs, iters = 48;
            const int *pairDev = tab, *roleDev = tab + 256;
            void *args[] = {&pool, &nb, &pairDev, &roleDev, &np, &iters, &rtDev};
            VSOM_CUDA(ctx, cudaLaunchCooperativeKernel(reinterpret_cast<void *>(die_classify_blocks_kernel), dim3(ctx->numSMs), dim3(32), args, 0, ctx->stream));
            std::vector<float> rt(kFPoolBlocks);
            VSOM_CUDA(ctx, cudaMemcpyAsync(rt.data(), rtDev, sizeof(float) * kFPoolBlocks, cudaMemcpyDeviceToHost, ctx->stream));
            VSOM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            cudaFree(tab);
            cudaFree(rtDev);
            float thr = 0.f;
            bool complete = true;
            for (float v : rt)
                complete = complete && v > 0.f;
            const bool bimodal = complete && split_bimodal(rt, thr);
            if (!bimodal)
            {
                std::vector<float> srt = rt;
                std::sort(srt.begin(), srt.end());
                size_t near = 0;
                for (float x : srt)
                    near += (x > thr - 0.15f * (srt[3 * srt.size() / 4] - srt[srt.size() / 4]) && x < thr + 0.15f * (srt[3 * srt.size() / 4] - srt[srt.size() / 4])) ? 1 : 0;
                fprintf(stderr, "[vsom] block die calibration: pairs=%d complete=%d bimodal=%d thr=%.0f min=%.0f q1=%.0f median=%.0f q3=%.0f max=%.0f near=%zu\n", nPairs,
                        complete ? 1 : 0, bimodal ? 1 : 0, thr, srt.front(), srt[srt.size() / 4], srt[srt.size() / 2], srt[3 * srt.size() / 4], srt.back(), near);
            }
            if (bimodal)
            {
                for (int k = 0; k < kFPoolBlocks; ++k)
                    home[k] = rt[k] > thr ? 1 : 0; // measured by die-0 pairs: fast = homed on die 0
                haveHomes = true;
            }
        }
    }
    // rowBlocks[(die * kFMaxCtas + slot) * 2 + buffer] = block index; every (die, slot, buffer) gets its own block
    std::vector<int> rowBlocks(2 * 2 * kFMaxCtas, 0), dieOfSm(256, 0);
    std::vector<int> byDie[2];
    for (int k = 0; k < kFPoolBlocks; ++k)
        byDie[haveHomes ? home[k] : (k & 1)].push_back(k);
    ctx->dieAware = haveHomes ? 1 : 0;
    if (haveHomes)
        for (int s = 0; s < 256; ++s)
            dieOfSm[s] = dm.dieOfSm[s];
    bool enough = byDie[0].size() >= 2 * 100 && byDie[1].size() >= 2 * 100; // a die has at most ~80 SMs
    if (!enough)
    {
        ctx->dieAware = 0;
        byDie[0].clear();
        byDie[1].clear();
        for (int k = 0; k < kFPoolBlocks; ++k)
            byDie[k & 1].push_back(k);
        std::fill(dieOfSm.begin(), dieOfSm.end(), 0);
    }
    for (int d = 0; d < 2; ++d)
        for (int slot = 0; slot < kFMaxCtas; ++slot)
            for (int buf = 0; buf < 2; ++buf)
            {
                const size_t i = static_cast<size_t>(slot) * 2 + buf;
                // past the die's own blocks (more CTAs on one die than any B200 has SMs there) borrow from the other list
                const std::vector<int> &own = byDie[d], &other = byDie[1 - d];
                rowBlocks[(d * kFMaxCtas + slot) * 2 + buf] = i < own.size() ? own[i] : other[other.size() - 1 - (i - own.size())];
            }
    int *meta = ctx->rowMeta;
    VSOM_CUDA(ctx, cudaMemcpyAsync(meta, dieOfSm.data(), sizeof(int) * 256, cudaMemcpyHostToDevice, ctx->stream));
    VSOM_CUDA(ctx, cudaMemcpyAsync(meta + 256, rowBlocks.data(), sizeof(int) * rowBlocks.size(), cudaMemcpyHostToDevice, ctx->stream));
    VSOM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return VSOM_OK;
}

// K1F's plan, left unset where K1F cannot run the context (launch_online_step states the rule)
void configure_online_step_fast(vsom_ctx *ctx)
{
    const char *env = getenv("VSOM_ONLINE_KERNEL"); // "generic": every chunk on K1 (A/B measurements)
    if ((env && std::string(env) == "generic") || ctx->order == VSOM_ORDER_LANES || ctx->world > 1 || ctx->W > 4096 || ctx->H > 4096)
        return;
    if (ctx->transform == VSOM_CLR && ((ctx->Din + 3) & ~3) + 4 > 65535)
        return; // pair tables are 16-bit
    int G = ctx->localN < ctx->numSMs ? ctx->localN : ctx->numSMs;
    if (G > kFMaxCtas)
        G = kFMaxCtas;
    const int stride = fast_stride(ctx);
    const size_t bytes = fast_smem(ctx, G, stride);
    if (bytes + kFStaticSmem > static_cast<size_t>(ctx->smemOptin))
        return;
    const int Lmax = (ctx->localN + G - 1) / G;
    if (Lmax > kFThreads)
        return; // one scan lane per owned node
    StepPlan pl;
    const int ipw = fast_ipw(ctx, G);
    for (int prof = 0; prof < 2; ++prof)
    {
        FastKernel k = pick_fast(ctx->transform, ipw, prof != 0);
        if (cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, ctx->smemOptin - static_cast<int>(kFStaticSmem)) != cudaSuccess)
        {
            cudaGetLastError();
            return;
        }
        int perSm = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSm, k, kFThreads, bytes) != cudaSuccess || perSm < 1)
        {
            cudaGetLastError();
            return;
        }
        pl.kernel[prof] = k;
    }
    pl.grid = G;
    pl.threads = kFThreads;
    pl.smem = bytes;
    pl.smemCap = static_cast<size_t>(ctx->smemOptin) - kFStaticSmem;
    pl.resident = 1;
    pl.smStride = stride;
    // Eigen order: eight lanes per node cut the chain from Dr to Dr / 8 dependent adds; worth it when the rows are long or when
    // all the CTA's nodes still fit one warp (no extra CTA-level reduction).
    pl.lanesPerNode = ctx->order == VSOM_ORDER_EIGEN_SSE && Lmax * 8 <= kFThreads && (Lmax * 8 <= 32 || ctx->Dr >= 256) ? 8 : 1;
    // slots: chain, CTA min, exchange, coefficients, barrier, update (+ the next sample's squared residuals), barrier.  No
    // wait-for-sample phase; the other four phases of the profile are sums of these.
    pl.profStride = 8;
    const unsigned char fold[5] = {0, 0x03, 0x04, 0x18, 0x60};
    std::copy(fold, fold + 5, pl.profFold);
    ctx->k1f = pl;
}

// [start,end) of the update window per BMU column and row: the f64 expressions of src/Som.cpp:899-903
static int build_window_table(vsom_ctx *ctx, double sigma)
{
    if (ctx->winTab && ctx->winSigma == sigma)
        return VSOM_OK;
    if (!ctx->winTab)
        VSOM_CUDA(ctx, cudaMalloc(&ctx->winTab, sizeof(unsigned) * (static_cast<size_t>(ctx->W) + ctx->H)));
    std::vector<unsigned> h(static_cast<size_t>(ctx->W) + ctx->H);
    const double dW = static_cast<double>(ctx->W), dH = static_cast<double>(ctx->H);
    for (int i = 0; i < ctx->W + ctx->H; ++i)
    {
        const bool isX = i < ctx->W;
        const double c = static_cast<double>(isX ? i : i - ctx->W), lim = isX ? dW : dH;
        const double lo = c - 2.5 * sigma, hi = c + 2.5 * sigma;
        const size_t start = static_cast<size_t>(lo > 0. ? lo : 0.);
        const size_t end = static_cast<size_t>(hi < lim ? hi : lim);
        h[i] = static_cast<unsigned>(start > 0xffff ? 0xffff : start) | (static_cast<unsigned>(end) << 16);
    }
    VSOM_CUDA(ctx, cudaMemcpyAsync(ctx->winTab, h.data(), sizeof(unsigned) * h.size(), cudaMemcpyHostToDevice, ctx->stream));
    ctx->winSigma = sigma;
    return VSOM_OK;
}

// K1F's per-chunk state: the local walk's tagged distances, the exchange rows (the first chunk measures the L2 dies) and the
// update window table
int prepare_online_step_fast(vsom_ctx *ctx, StepParams &p, double sigma)
{
    if (p.localSearch)
    {
        const size_t bytes = sizeof(u64) * 2 * kWalkReplicas * static_cast<size_t>(ctx->N);
        if (!ctx->distTag)
            VSOM_CUDA(ctx, cudaMalloc(&ctx->distTag, bytes));
        VSOM_CUDA(ctx, cudaMemsetAsync(ctx->distTag, 0xff, bytes, ctx->stream)); // no word carries a tag of this launch yet
    }
    p.distTag = ctx->distTag;
    int rc = build_row_pool(ctx);
    if (rc)
        return rc;
    rc = build_window_table(ctx, sigma);
    if (rc)
        return rc;
    VSOM_CUDA(ctx, cudaMemsetAsync(ctx->rowPool, 0xff, static_cast<size_t>(kFPoolBlocks) * 2048, ctx->stream));
    unsigned *ctr = reinterpret_cast<unsigned *>(ctx->rowMeta + 256 + 2 * 2 * kFMaxCtas + kFMaxCtas);
    VSOM_CUDA(ctx, cudaMemsetAsync(ctr, 0, sizeof(unsigned) * 4, ctx->stream));
    p.winTab = ctx->winTab;
    p.dieOfSm = ctx->rowMeta;
    p.rowBlocks = ctx->rowMeta + 256;
    p.rowOf = ctx->rowMeta + 256 + 2 * 2 * kFMaxCtas;
    p.rowCtr = ctr;
    p.rowPool = ctx->rowPool;
    return VSOM_OK;
}

} // namespace vsom
