// score_tc.cu — K2: batch BMU search as a dense contraction on the 5th-generation tensor cores, + exact rescore.
//
// Replaces the same row loops as score_exact.cu (Som::evaluate src/Som.cpp:503-520, findBmu :291-309,
// findRestrictedBmu :313-332 over a loaded DataSet) when the batch is large:
//     d(r,p) = |x_r|^2 - 2 x_r . m_p + |m_p|^2            (Standard / Median Comparer, src/Transformation.cpp:7-8)
// The cross term X[R x K] . M^T[K x N] runs as tcgen05.mma (fp16 operands, fp32 accumulators in TMEM), operands
// staged by TMA (128-byte swizzle).  The tensor cores only SELECT candidates; the exact pass re-evaluates them in
// the reference's own f32 arithmetic and order (bit-identical distances) and applies findBmu's lowest-index rule.
//
// Operands are IEEE half (fp16, u = 2^-11), not bf16: same tensor-core rate, 8x tighter products — on a TRAINED map the
// neighbours of the BMU differ from it by less than a bf16 product's error, and the candidate lists would hold the whole
// neighbourhood.  fp16's narrow range is handled by power-of-two scales (exact): one per ROW of the data, s_r, putting the
// row's largest |x_k| in [2^9, 2^10), and one for the map, s_m, likewise (values far below the largest one may become fp16
// subnormals: their absolute error 2^-25 is part of the bound below).
//
// The node constant rides in the contraction: the map operand holds -2 s_m m_p followed by three columns with a hi / mid / lo
// fp16 split of s_m c_p / tau (c_p = |m_p|^2, tau a power of two that keeps the pieces inside fp16), the row operand s_r x
// followed by three columns s_r tau, so the f32 accumulator IS the scaled approximate score
//     a'_p = S_r (c_p - 2 x^ . m^_p),  S_r = s_r s_m,
// and the epilogue only takes minima (K = D + 3, rounded up to 16 per MMA).  Everything per row (best, threshold, margins)
// lives in that row's scaled units; powers of two commute with every comparison.
//
// Candidate rule (margin list + certificate).  |a'_p + S_r |x|^2 - S_r d_p| <= E', with
//     E' = 2 (2u + u^2) |s_r x| max_p |s_m m_p|  +  2^-25 sqrt(D) (2 max|s_m m_p| + |s_r x|)  +  slack
// (rounding of both operands + Cauchy-Schwarz; the subnormal term; a relative slack for every f32 effect: tensor-core
// accumulation, the norms, the reference's own f32 chain).  While streaming over the node tiles each row keeps its running
// best score and appends every node with a'_p < best + Delta' to a small per-row list (tc_margins: Delta' = 1.25 E' + slack).
// Delta' alone proves nothing; the proof is the CERTIFICATE checked after the exact rescore: every node NOT in the list had
// a'_q >= best_final + Delta', hence S_r times its reference distance is >= best_final + S_r |x|^2 + Delta' - E'.  If that
// bound is strictly above S_r times the best EXACT distance among the listed nodes, no unlisted node can be the BMU or tie
// with it, and the row is done; otherwise the row is re-scored by the exact full scan.  So the result never depends on a
// statistical recall argument: Delta' only trades list length against the share of rows that need the full scan.  Up to
// 48 survivors per row go to the exact rescore (which also re-checks min_hits eligibility, so nothing depends on the large
// constant given to excluded nodes); rows with more (or whose list overflowed) take the exact full scan as well.
// What the certificate covers: nodes with finite approximate scores.  A NaN score drops out of the epilogue's minima and is
// never listed, which is right for every node but node 0: findBmu seeds with node 0, so a NaN distance there wins every
// row (src/Som.cpp:293).  When node 0 has a NaN component (TcScale::nanNode0, set by map_stats_kernel) no row is certified
// and the probes hand the call to the exact scan.  Rows with a NaN or infinite element, and rows whose best listed distance
// overflows to inf, fail the certificate on their own (NaN / inf bound); an infinite map component collapses s_m so that
// every node sits inside every margin.  All of these end in the exact scan.
//
// Kernel structure (one CTA per SM, persistent; 384 threads; by default two CTAs — the SMs of a TPC — form a cluster and
// work as ONE tcgen05 cta_group::2 unit on 256 rows, see score_tc_kernel):
//   warp 0   TMA producer : A tile (128 rows x K; resident for the row tile when K <= 320, else its k-blocks ride in the
//                           ring) + B tiles (this CTA's half of 256 nodes x 64) through an mbarrier ring (6 / 5 stages)
//   warp 1   MMA issuer   : the whole warp walks the loop, one elected lane (elect.sync) issues tcgen05.mma kind::f16
//                           (M = 128 per CTA, N = 256, K = 16) into one of two 256-column TMEM accumulators;
//                           tcgen05.commit frees the smem stage / publishes the accumulator (multicast to both CTAs)
//   warp 2   TMEM allocator (512 columns)
//   warps 4-11 epilogue   : two threads per row (TMEM lane), 128 columns each; tcgen05.ld 32 columns at a time (next
//                           chunk in flight); per chunk a tree of FMNMX3 (the accumulators ARE the scores), one vote, and
//                           only for flagged groups of four columns the predicated appends to the thread's list
// Two precision tiers (one fp16 per operand element / hi-lo pairs, three products) — see tc_score_tiers.
// Measured (round 2, 128x128x256, ncu): pipeline without epilogue 93 % / 97 % tensor-pipe active (tier 1 / 2); an epilogue that only
// reads the accumulators (tcgen05.ld, no scoring) 92 % / 97 %; the real one 72 % / 95 %.  So the TMEM reads fit under the K = 272
// contraction of a tile; what costs tier 1 its last 20 % is the latency chain of the scoring code (min tree -> vote -> branch) with two
// epilogue warps per scheduler, and the per-tile handshake of 16 warps in two CTAs.  Tier 2 runs into the chip's power limit
// (SM clock 1.35-1.5 GHz at > 90 % activity).
// Limits: Standard / Median transformation (not CLR), Dm <= 2048; other shapes use K3.
#include "common.cuh"

#include <cuda.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>

namespace vsom
{

constexpr int TC_BM = 128, TC_BN = 256, TC_BK = 64, TC_STAGES = 3, TC_TOPK = 48, TC_THREADS = 384;
constexpr int TC_MAXSTAGES = 6; // ring stages at most (CTA pairs hold half B tiles: twice the stages in the same space)
constexpr int TC_LIST = 24;    // per-thread candidate list (shared memory); a full list sends the row to the exact scan
constexpr int TC_LIST_HI = 16; // lists are compacted against the current threshold when one passes this length
constexpr unsigned TC_OVERFLOW = 255;
constexpr int TC_MAXK = 256;   // longest model vector; the operands carry 3 more columns for the node constant (below)
constexpr int TC_MAXKB = (TC_MAXK + 16 + TC_BK - 1) / TC_BK; // k-blocks of the extended operands at most (5)
constexpr float TC_BIG = 1.0e38f; // node constant of nodes that must never be selected (padding, below min_hits)
constexpr int TC_A_BYTES = TC_BM * TC_BK * 2;  // 16 KB per k-block
constexpr int TC_B_BYTES = TC_BN * TC_BK * 2;  // 32 KB per stage

// ------------------------------------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ unsigned smem_u32(const void *p) { return static_cast<unsigned>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(void *bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(void *bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(void *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(void *bar, unsigned parity)
{
    unsigned ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok)
                 : "r"(smem_u32(bar)), "r"(parity)
                 : "memory");
    return ok != 0;
}
// bounded wait: a pipeline bug must end the kernel (error flag), not hang the GPU
__device__ __forceinline__ bool mbar_wait(void *bar, unsigned parity, int *err)
{
    unsigned long long t0 = 0;
#pragma unroll 1
    for (unsigned spin = 1;; ++spin)
    {
        if (mbar_try_wait(bar, parity))
            return true;
        if ((spin & 1023u) == 0)
        {
            unsigned long long t;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            if (t0 == 0)
                t0 = t;
            else if (t - t0 > 4000000000ull) // 4 s: no legitimate wait of this pipeline lasts longer than a tile
                break;
        }
    }
    *err = 2;
    return false;
}
// In a CTA pair the shared::cluster address of the SAME offset in the even (leader) CTA: clear the peer bit (cute's Sm100MmaPeerBitMask)
constexpr unsigned TC_LEADER_MASK = 0xFEFFFFFFu;
// PAIR: the load lands in this CTA's shared memory, its bytes complete on the LEADER CTA's barrier
template <bool PAIR>
__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *map, void *bar, int c0, int c1)
{
    if (PAIR)
        asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(dst)),
                     "l"(map), "r"(smem_u32(bar) & TC_LEADER_MASK), "r"(c0), "r"(c1)
                     : "memory");
    else
        asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(dst)),
                     "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
                     : "memory");
}
// PAIR: the arrival is delivered to the barrier at this offset in BOTH CTAs
template <bool PAIR>
__device__ __forceinline__ void umma_commit(void *bar)
{
    if (PAIR)
        asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)), "h"(static_cast<unsigned short>(3))
                     : "memory");
    else
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
template <bool PAIR>
__device__ __forceinline__ void mbar_arrive_leader(void *bar)
{
    if (PAIR)
        asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & TC_LEADER_MASK) : "memory"); // no .release.cluster: that is a MEMBAR.GPU per tile; the TMEM reads are ordered by tcgen05.fence::before_thread_sync
    else
        asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// one lane of a converged warp (elect.sync): the compiler knows the guarded code runs in exactly one thread
__device__ __forceinline__ bool elect_one()
{
    unsigned pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void cluster_sync()
{
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld32(unsigned addr, unsigned (&v)[32])
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, "
                 "%20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]),
                   "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]),
                   "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]),
                   "=r"(v[31])
                 : "r"(addr)
                 : "memory");
}
__device__ __forceinline__ void sts64(unsigned addr, unsigned lo, unsigned hi)
{
    asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(addr), "r"(lo), "r"(hi) : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// shared-memory matrix descriptor, K-major, 128-byte swizzle (cute::UMMA::SmemDescriptor bit layout):
// start address >> 4 in [0,14), LBO (ignored for swizzled K-major, set 1) in [16,30), SBO = 1024 B (8 rows x 128 B)
// in [32,46), version 1 in [46,48), layout SWIZZLE_128B = 2 in [61,64)
__device__ __forceinline__ u64 umma_desc_sw128(unsigned smemAddr)
{
    return static_cast<u64>((smemAddr & 0x3ffff) >> 4) | (1ull << 16) | (static_cast<u64>(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
// instruction descriptor (cute::UMMA::InstrDescriptor): c=f32 (1<<4), a=b=f16 (format 0 at bits 7 and 10; bf16 would be 1), both K-major, N>>3 at 17, M>>4 at 24
__host__ __device__ constexpr unsigned tc_idesc(int m) { return (1u << 4) | (static_cast<unsigned>(TC_BN >> 3) << 17) | (static_cast<unsigned>(m >> 4) << 24); }
constexpr unsigned kIdesc = tc_idesc(TC_BM), kIdescPair = tc_idesc(2 * TC_BM);
// PAIR: one instruction for both CTAs (M = 256: rows 0..127 from the leader's A tile into its TMEM, 128..255 the peer's);
// each CTA's shared memory supplies its 128 of the 256 B rows; the descriptors address the same offsets in both
template <bool PAIR>
__device__ __forceinline__ void umma_f16(unsigned tmemC, u64 descA, u64 descB, unsigned accumulate)
{
    if (PAIR)
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmemC), "l"(descA),
                     "l"(descB), "r"(kIdescPair), "r"(accumulate)
                     : "memory");
    else
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmemC), "l"(descA),
                     "l"(descB), "r"(kIdesc), "r"(accumulate)
                     : "memory");
}

// scales of one scoring call, computed on the device (tc_scale_kernel)
struct TcScale
{
    float sm;       // power of two: map values are multiplied by it
    float tau;      // power of two: the node-constant columns hold s_m c_p / tau, the rows' tail columns s_r tau
    float mm;       // max_p |s_m m_p|^2
    float maxAbs;   // max |m_pk| (bits, via atomicMax) — input of the scale
    float maxNorm2; // max_p |m_p|^2                   — input of the scale
    int split;      // 1: operands are hi / lo pairs of halves (three products per element), 0: one half each
    int nanNode0;   // node 0 has a NaN component: no row can be certified (see "Candidate rule")
};

// Error bound E' and list margin Delta' of one row in its scaled units (see "Candidate rule" above).
// xn = |s_r x|^2, mm = max_p |s_m m_p|^2, ratio = s_m / s_r (so that S_r |x|^2 = xn ratio and S_r max|m|^2 = mm / ratio).
// split: the precise tier — X = xh + xl + ex, M = mh + ml + em with |ex_k| <= u^2 |X_k| + 2^-25, the contraction computes
// xh.mh + xl.mh + xh.ml, so X.M - (...) = xl.ml + ex.M + (X - ex).em  <=  3 u^2 (1 + ...) |X||M| + 2^-25 sqrt(D) (|M| + |X|).
// slack: f32 accumulation of K products inside the tensor core (assumed no better than truncation, 2^-23 each), the
// reference's own f32 chain and the f32 norms (D 2^-24 each).
__device__ __forceinline__ void tc_margins(float xn, float mm, float ratio, int Kpad, int D, int split, float &E, float &delta)
{
    const float slack = static_cast<float>(Kpad + D + 64) * 1.1920928955078125e-7f * (xn * ratio + mm / ratio); // (K + D + 64) 2^-23 S (|x|^2 + max|m|^2)
    const float sx = sqrtf(xn), smx = sqrtf(mm);
    // one half each: 2 (2u + u^2) = 2^-9 (1 + 2^-12) < 0.00196; hi / lo pairs: 6 u^2 (1 + ...) < 1.45e-6; 2^-25 (1 + u) < 2.99e-8
    E = (split ? 1.45e-6f : 0.00196f) * sx * smx + 2.99e-8f * sqrtf(static_cast<float>(D)) * (2.0f * smx + sx) + slack;
    delta = 1.25f * E + 0.25f * slack;
}

struct TcShared
{
    // offsets inside the dynamic shared buffer (1024-byte aligned base)
    static constexpr int A_OFF = 0;                                   // up to 5 k-blocks x 16 KB
    static constexpr int B_OFF = A_OFF + TC_MAXKB * TC_A_BYTES;        // 3 stages x 32 KB
    static constexpr int BAR_OFF = B_OFF + TC_STAGES * TC_B_BYTES;     // mbarriers
    static constexpr int LIST_OFF = BAR_OFF + 256;                     // TC_LIST x 256 x {score, node}: per-thread candidate lists
    static constexpr int MERGE_OFF = LIST_OFF + TC_LIST * 256 * 8;     // 256 floats + 256 ints: merge of the two half rows
    static constexpr int TOTAL = MERGE_OFF + 256 * 8;
};

// PAIR = true: two CTAs of a cluster (the two SMs of a TPC) work as one tcgen05 cta_group::2 unit on 256 rows.  Each CTA
// holds its own 128 rows of A and HALF of the B tile (128 of the 256 nodes); one MMA (M = 256) issued by the even CTA reads
// both halves, so every B byte crosses L2 -> SMEM once per 256 rows instead of once per 128, and each SM's shared memory
// serves 8 KB per K = 16 step instead of 12 KB.  Barrier protocol (same offsets in both CTAs):
//   bFull / aFull : the LEADER's; its producer expects both CTAs' bytes, the peer's TMA completes on it (cta_group::2 load)
//   bEmpty / aEmpty / tFull : each CTA's own, signalled by the leader's tcgen05.commit multicast to both
//   tEmpty : the leader's; one arrival per epilogue warp of BOTH CTAs (the peer's arrive through shared::cluster)
//
// TOP = 2 (vsom_find_bmu2): the list must hold the runner-up too, so each thread keeps an upper bound `second` of the
// second-smallest score it has seen and lists every node below second + Delta'.  Per chunk:
//     second = min(second, max(best, chunk min), second-smallest of the eight group minima m4[])
// (each term bounds the second-smallest of the scores seen so far; the group minima are eight different columns), so the
// threshold still only falls.  The half-row merge combines the two (best, second) pairs the same way, and bestOut receives the
// final threshold base: every unlisted node had a' >= that base + Delta' (see rescore_kernel's certificate).
template <bool PAIR, int TOP>
__global__ void __launch_bounds__(TC_THREADS, 1)
score_tc_kernel(const __grid_constant__ CUtensorMap mapX, const __grid_constant__ CUtensorMap mapM, int kSteps, int rowsTotal,
                int numRowTiles, int numNodeTiles, int kBlocks, int kCols, int stagger, int D, const float *__restrict__ xnorm2, const float *__restrict__ xratio, const TcScale *__restrict__ scale,
                unsigned *__restrict__ candOut,
                unsigned *__restrict__ countOut, float *__restrict__ bestOut, int *err)
{
    // 128-byte-swizzled TMA / UMMA tiles need a 1024-byte aligned base; declaring the alignment (instead of rounding
    // a pointer up by hand) also lets the compiler keep every derived pointer in the shared address space (LDS/STS)
    extern __shared__ __align__(1024) unsigned char smem[];
    constexpr int BST = PAIR ? TC_B_BYTES / 2 : TC_B_BYTES;       // B bytes of one stage in THIS CTA's shared memory
    constexpr int NCTA = PAIR ? 2 : 1;
    unsigned char *sA = smem + TcShared::A_OFF;
    unsigned char *sB = smem + TcShared::B_OFF;
    u64 *bars = reinterpret_cast<u64 *>(smem + TcShared::BAR_OFF);
    u64 *bFull = bars, *bEmpty = bars + TC_MAXSTAGES, *aFull = bars + 2 * TC_MAXSTAGES, *aEmpty = aFull + 1, *tFull = aEmpty + 1, *tEmpty = tFull + 2;
    unsigned *tmemBaseSlot = reinterpret_cast<unsigned *>(tEmpty + 2);
    uint2 *lists = reinterpret_cast<uint2 *>(smem + TcShared::LIST_OFF);
    float *sBest = reinterpret_cast<float *>(smem + TcShared::MERGE_OFF);
    int *sCnt = reinterpret_cast<int *>(sBest + 256);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool streamed = kBlocks > TC_MAXKB; // the row tile's K does not fit the resident A area: A k-blocks ride in the stage ring
    const int stageBytes = streamed ? TC_A_BYTES + BST : BST;
    // stages of the ring: whatever fits the operand area (resident: the 96 KB behind A; streamed: A and B areas together)
    const unsigned numStages = streamed ? static_cast<unsigned>((TcShared::BAR_OFF) / (TC_A_BYTES + BST) < TC_MAXSTAGES ? (TcShared::BAR_OFF) / (TC_A_BYTES + BST) : TC_MAXSTAGES)
                                        : static_cast<unsigned>(TC_STAGES * TC_B_BYTES / BST);
    unsigned char *ring = streamed ? smem : sB;
    unsigned crank = 0;
    if (PAIR)
        asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(crank));
    const bool leader = crank == 0;
    // work units: PAIR -> 256 rows (row tiles 2u and 2u + 1, one per CTA; an odd last one is a tile of zero rows)
    const int unitIdx = PAIR ? blockIdx.x >> 1 : blockIdx.x, unitStride = PAIR ? gridDim.x >> 1 : gridDim.x;
    const int numUnits = PAIR ? (numRowTiles + 1) >> 1 : numRowTiles;
    // units walk the node tiles from different starting points so that at any moment they pull DIFFERENT B tiles out
    // of L2 (all starting at tile 0 makes 148 SMs ask the same lines at once)
    const int ntStart = (stagger & 1) ? static_cast<int>((static_cast<unsigned>(unitIdx) * 7u) % static_cast<unsigned>(numNodeTiles)) : 0;

    if (warp == 1 && lane == 0)
    {
        for (int s = 0; s < TC_MAXSTAGES; ++s)
        {
            mbar_init(&bFull[s], 1);
            mbar_init(&bEmpty[s], 1);
        }
        mbar_init(aFull, 1);
        mbar_init(aEmpty, 1);
        for (int a = 0; a < 2; ++a)
        {
            mbar_init(&tFull[a], 1);
            mbar_init(&tEmpty[a], 8 * NCTA); // one arrival per epilogue warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (PAIR)
        cluster_sync(); // the peer's barriers exist before anything of ours can reach them; both CTAs are resident for the paired allocation
    if (warp == 2)
    {
        if (PAIR)
        {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmemBaseSlot)), "r"(512) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        }
        else
        {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmemBaseSlot)), "r"(512) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const unsigned tmemBase = *tmemBaseSlot;

    if (warp == 0)
    {
        // ===================================================== TMA producer (both CTAs of a pair: own A rows, own half of B)
        // The WHOLE warp walks the loop (waits included) and one elected lane issues: with a divergent `if (lane == 0)` around
        // the loop every TMA / MMA instruction (uniform datapath) is wrapped in an ELECT / R2UR.BROADCAST retry loop and the
        // per-k-block issue path grows to ~150 dependent instructions — as long as the 4 MMAs it feeds (ncu, round 2).
        {
            unsigned stage = 0, phase = 0, aPhase = 0;
            bool ok = true;
            for (int u = unitIdx; u < numUnits && ok; u += unitStride)
            {
                const int rt = PAIR ? 2 * u + static_cast<int>(crank) : u;
                if (!streamed)
                {
                    ok = mbar_wait(aEmpty, aPhase ^ 1, err); // previous row tile's MMAs are done with A
                    aPhase ^= 1;
                    if (elect_one())
                    {
                        if (leader)
                            mbar_expect_tx(aFull, static_cast<unsigned>(kBlocks) * TC_A_BYTES * NCTA);
                        for (int kb = 0; kb < kBlocks; ++kb)
                            tma_load_2d<PAIR>(sA + kb * TC_A_BYTES, &mapX, aFull, kb * TC_BK, rt * TC_BM);
                    }
                    __syncwarp();
                }
                for (int i = 0; i < numNodeTiles && ok; ++i)
                {
                    int nt = i + ntStart;
                    nt -= nt >= numNodeTiles ? numNodeTiles : 0;
                    const int node0 = nt * TC_BN + static_cast<int>(crank) * (TC_BN / 2); // PAIR: this CTA's half of the node tile (box of 128 rows)
                    for (int kb = 0; kb < kBlocks && ok; ++kb)
                    {
                        ok = mbar_wait(&bEmpty[stage], phase ^ 1, err);
                        unsigned char *st = ring + stage * stageBytes;
                        if (elect_one())
                        {
                            if (leader)
                                mbar_expect_tx(&bFull[stage], static_cast<unsigned>(stageBytes) * NCTA);
                            if (streamed)
                            {
                                // long rows: the A k-block travels with the B k-block (re-read from L2 for every node tile)
                                tma_load_2d<PAIR>(st, &mapX, &bFull[stage], kb * TC_BK, rt * TC_BM);
                                st += TC_A_BYTES;
                            }
                            tma_load_2d<PAIR>(st, &mapM, &bFull[stage], kb * TC_BK, node0);
                        }
                        __syncwarp();
                        if (++stage == numStages)
                        {
                            stage = 0;
                            phase ^= 1;
                        }
                    }
                }
            }
        }
    }
    else if (warp == 1)
    {
        // ===================================================== MMA issuer (whole warp walks, one elected lane issues; PAIR: leader CTA only)
        if (leader)
        {
            unsigned stage = 0, phase = 0, aPhase = 0, acc = 0, accPhase = 0;
            bool ok = true;
            const unsigned ringAddr = smem_u32(ring), sAAddr = smem_u32(sA);
            for (int u = unitIdx; u < numUnits && ok; u += unitStride)
            {
                if (!streamed)
                {
                    ok = mbar_wait(aFull, aPhase, err);
                    aPhase ^= 1;
                }
                for (int nt = 0; nt < numNodeTiles && ok; ++nt)
                {
                    ok = mbar_wait(&tEmpty[acc], accPhase ^ 1, err); // epilogue drained this accumulator
                    const unsigned tmemC = tmemBase + acc * TC_BN;
                    for (int kb = 0; kb < kBlocks && ok; ++kb)
                    {
                        ok = mbar_wait(&bFull[stage], phase, err);
                        tc_fence_after();
                        const unsigned stAddr = ringAddr + stage * static_cast<unsigned>(stageBytes);
                        const unsigned aAddr = streamed ? stAddr : sAAddr + static_cast<unsigned>(kb) * TC_A_BYTES;
                        const unsigned bAddr = streamed ? stAddr + TC_A_BYTES : stAddr;
                        const int steps = min(TC_BK / 16, kSteps - kb * (TC_BK / 16)); // the last k-block may be partly used
                        if (elect_one())
                        {
                            // +32 bytes per K=16 step inside the 128-byte swizzle row: +2 in the descriptor's address field
                            const u64 da = umma_desc_sw128(aAddr), db = umma_desc_sw128(bAddr);
#pragma unroll
                            for (int k = 0; k < TC_BK / 16; ++k)
                                if (k < steps)
                                    umma_f16<PAIR>(tmemC, da + 2u * k, db + 2u * k, (kb | k) != 0 ? 1u : 0u);
                            umma_commit<PAIR>(&bEmpty[stage]); // frees the stage (in both CTAs) when the MMAs above have read it
                            if (kb == kBlocks - 1)
                                umma_commit<PAIR>(&tFull[acc]); // accumulator complete
                        }
                        __syncwarp();
                        if (++stage == numStages)
                        {
                            stage = 0;
                            phase ^= 1;
                        }
                    }
                    if (++acc == 2)
                    {
                        acc = 0;
                        accPhase ^= 1;
                    }
                }
                if (!streamed)
                {
                    if (elect_one())
                        umma_commit<PAIR>(aEmpty); // all MMAs of this row tile are done reading A
                    __syncwarp();
                }
            }
        }
    }
    else if (warp >= 4)
    {
        // ===================================================== epilogue: 8 warps, two threads per row of the tile
        // Warps 4-7 score columns 0..127 of every accumulator, warps 8-11 columns 128..255 (warp w may only touch the
        // TMEM lane quarter w % 4, so both halves cover all 128 rows).  Two resident warps per scheduler hide each
        // other's LDS / ALU latencies; each thread keeps its own running best and its own short list, merged per row
        // at the end of the row tile.
        const int q = warp & 3;            // TMEM lane quarter this warp may access
        const int half = (warp - 4) >> 2;  // 0: columns 0..127, 1: columns 128..255
        const int rowInTile = q * 32 + lane;
        const int et = threadIdx.x - 128;  // 0..255 ; partner thread of the same row: et ^ 128
        uint2 *mine = lists + et;          // entry e of this thread at mine[e * 256]
        const unsigned mineAddr = smem_u32(mine);
        const unsigned mineEnd = mineAddr + TC_LIST * 2048u;
        unsigned acc = 0, accPhase = 0;
        bool ok = true;
        const float mm = scale->mm;
        const float inf = __int_as_float(0x7f800000);

        // drop list entries that are no longer below the (tightened) threshold; warp-uniform control flow
        auto compact = [&](int &cnt, float thr) {
            const int maxc = __reduce_max_sync(0xffffffffu, cnt);
            int k = 0;
#pragma unroll 1
            for (int e = 0; e < maxc; ++e)
                if (e < cnt)
                {
                    const uint2 v = mine[e * 256];
                    if (__uint_as_float(v.x) < thr)
                    {
                        mine[k * 256] = v;
                        ++k;
                    }
                }
            cnt = k;
        };

        for (int u = unitIdx; u < numUnits && ok; u += unitStride)
        {
            const int rt = PAIR ? 2 * u + static_cast<int>(crank) : u;
            const long long row = static_cast<long long>(rt) * TC_BM + rowInTile;
            const float xn = row < rowsTotal ? xnorm2[row] : 0.0f, ratio = row < rowsTotal ? xratio[row] : 1.0f;
            float E, delta;
            tc_margins(xn, mm, ratio, kCols, D, scale->split, E, delta);
            float best = inf, thr = inf, thrC = inf; // thrC: threshold at this list's last compaction
            float second = inf;                      // TOP = 2: upper bound of the second-smallest score so far
            int cnt = 0;
            bool ovf = false;
            unsigned wp = mineAddr; // shared address of the next free entry of this thread's list (2048 bytes apart)
            for (int i = 0; i < numNodeTiles && ok; ++i)
            {
                int nt = i + ntStart; // ntStart < numNodeTiles: one conditional subtraction instead of a division per tile
                nt -= nt >= numNodeTiles ? numNodeTiles : 0;
                ok = mbar_wait(&tFull[acc], accPhase, err);
                tc_fence_after();
                const unsigned taddr = tmemBase + (static_cast<unsigned>(q * 32) << 16) + acc * TC_BN + half * (TC_BN / 2);
                unsigned v[2][32];
                bool released = false;
                if (stagger & 4) // bit 2 of the debug word: read the accumulator, do nothing with it (TMEM-read-only timing)
                {
                    // bit 3: two loads in flight per warp (is the read rate bound by the port or by the requests in flight?)
#pragma unroll 1
                    for (int c = 0; c < TC_BN / 64; c += 2)
                    {
                        tmem_ld32(taddr + c * 32, v[0]);
                        if (!(stagger & 8))
                            tmem_wait_ld();
                        tmem_ld32(taddr + (c + 1) * 32, v[1]);
                        tmem_wait_ld();
                        unsigned x = 0;
#pragma unroll
                        for (int j = 0; j < 32; ++j)
                            x |= v[0][j] | v[1][j];
                        if (x == 0x7fc00123u) // keeps the loads alive; never true for sums of finite products
                            ovf = true;
                    }
                }
                else if ((stagger & 2) == 0) // bit 1 of the debug word: skip the column work (pipeline-only timing)
                {
                    // one 32-column chunk of this thread's row.  Kept as ONE copy of the code per TMEM buffer (the loop below is
                    // not unrolled further): fully unrolled, the epilogue was 48 KB of SASS and its warps spent 40 % of their
                    // time waiting for instructions (ncu: stall_no_inst, profiles/r02_k2_ncu_details.txt)
                    auto chunk = [&](unsigned(&w)[32], int c) {
                        const unsigned nodeBase = static_cast<unsigned>(nt * TC_BN + half * (TC_BN / 2) + c * 32);
                        // The accumulators ARE the scores.  Group minima (of four columns) and the chunk minimum first: a tree of
                        // independent min instructions (FMNMX3 where it fits), nothing else on the common path.
                        float m4[8];
#pragma unroll
                        for (int j4 = 0; j4 < 8; ++j4)
                            m4[j4] = fminf(fminf(__uint_as_float(w[j4 * 4 + 0]), __uint_as_float(w[j4 * 4 + 1])),
                                           fminf(__uint_as_float(w[j4 * 4 + 2]), __uint_as_float(w[j4 * 4 + 3])));
                        const float cm = fminf(fminf(fminf(m4[0], m4[1]), fminf(m4[2], m4[3])), fminf(fminf(m4[4], m4[5]), fminf(m4[6], m4[7])));
                        const float thrOld = thr; // valid, possibly stale: whatever must be appended lies below it
                        // the chunk's own minimum tightens the threshold BEFORE anything is appended
                        if (TOP == 2)
                        {
                            // second-smallest of the group minima: (min, second) of pairs, merged twice
                            float lo[4], hi[4];
#pragma unroll
                            for (int j = 0; j < 4; ++j)
                            {
                                lo[j] = fminf(m4[2 * j], m4[2 * j + 1]);
                                hi[j] = fmaxf(m4[2 * j], m4[2 * j + 1]);
                            }
#pragma unroll
                            for (int w2 = 2; w2; w2 >>= 1)
#pragma unroll
                                for (int j = 0; j < w2; ++j)
                                {
                                    hi[j] = fminf(fmaxf(lo[j], lo[j + w2]), fminf(hi[j], hi[j + w2]));
                                    lo[j] = fminf(lo[j], lo[j + w2]);
                                }
                            second = fminf(second, fminf(fmaxf(best, cm), hi[0]));
                            best = fminf(best, cm);
                            thr = second + delta;
                        }
                        else
                        {
                            best = fminf(best, cm);
                            thr = best + delta;
                        }
                        if (!__any_sync(0xffffffffu, cm < thrOld))
                            return; // no lane of the warp has a candidate in this chunk (the common case once the rows have settled)
                        // Lists only grow here, so this is where a long one is compacted — and only when the threshold has tightened
                        // since its last compaction: otherwise nothing would go, and rows with many genuine near-candidates would pay
                        // the loop at every chunk.  (The check used to sit at the top of every chunk: a second vote on the common path.)
                        cnt = static_cast<int>((wp - mineAddr) >> 11);
                        if (__any_sync(0xffffffffu, cnt > TC_LIST_HI && thr < thrC))
                        {
                            compact(cnt, thr);
                            thrC = thr;
                            wp = mineAddr + (static_cast<unsigned>(cnt) << 11);
                        }
                        unsigned gm = 0; // groups of four columns in which this row may have something to append
#pragma unroll
                        for (int j4 = 0; j4 < 8; ++j4)
                            gm |= (m4[j4] < thrOld) ? (1u << j4) : 0u;
                        // one REDUX tells the whole warp which groups need the (predicated) appends; the branches below are on a
                        // warp-uniform value.  (Re-reading the flagged groups from TMEM in a short loop makes the code 4x smaller and measured the same on a
                        // random map, 5 % slower on a candidate-rich one: its tcgen05.wait::ld also waits for the prefetched next chunk.)
                        const unsigned any = __reduce_or_sync(0xffffffffu, gm);
#pragma unroll
                        for (int j4 = 0; j4 < 8; ++j4)
                            if (any & (1u << j4))
                            {
#pragma unroll
                                for (int k = 0; k < 4; ++k)
                                    if (__uint_as_float(w[j4 * 4 + k]) < thr)
                                    {
                                        if (wp < mineEnd)
                                        {
                                            sts64(wp, w[j4 * 4 + k], nodeBase + j4 * 4 + k);
                                            wp += 2048;
                                        }
                                        else
                                            ovf = true; // list full: this row takes the exact scan
                                    }
                            }
                    };
                    tmem_ld32(taddr, v[0]);
#pragma unroll 1
                    for (int cp = 0; cp < TC_BN / 128; ++cp)
                    {
                        tmem_wait_ld();
                        tmem_ld32(taddr + (2 * cp + 1) * 32, v[1]);
                        chunk(v[0], 2 * cp);
                        tmem_wait_ld();
                        if (2 * cp + 2 < TC_BN / 64)
                            tmem_ld32(taddr + (2 * cp + 2) * 32, v[0]);
                        else
                        {
                            // the tile's last chunk is in registers: the accumulator goes back to the MMA warp BEFORE that chunk is
                            // scored (the slowest of the 16 epilogue warps of a pair gates the next tile but one)
                            tc_fence_before();
                            __syncwarp();
                            if (lane == 0)
                                mbar_arrive_leader<PAIR>(&tEmpty[acc]);
                            released = true;
                        }
                        chunk(v[1], 2 * cp + 1);
                    }
                }
                if (!released)
                {
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0)
                        mbar_arrive_leader<PAIR>(&tEmpty[acc]);
                }
                if (++acc == 2)
                {
                    acc = 0;
                    accPhase ^= 1;
                }
            }
            // merge the two halves of the row: common best -> final threshold -> filter both lists -> candidates
            cnt = static_cast<int>((wp - mineAddr) >> 11);
            sBest[et] = best;
            if (TOP == 2)
                reinterpret_cast<float *>(sCnt)[et] = second; // sCnt is free until the counts below
            asm volatile("bar.sync 1, 256;" ::: "memory");
            float bestF, thrF;
            if (TOP == 2)
            {
                // the pair's threshold base: an upper bound of the row's second-smallest score, below both halves' thresholds
                const float bo = sBest[et ^ 128], so = reinterpret_cast<const float *>(sCnt)[et ^ 128];
                bestF = fminf(fmaxf(best, bo), fminf(second, so));
                thrF = bestF + delta;
                asm volatile("bar.sync 1, 256;" ::: "memory"); // both halves have read sCnt's floats
            }
            else
            {
                bestF = fminf(best, sBest[et ^ 128]);
                thrF = bestF + delta;
            }
            compact(cnt, thrF);
            sCnt[et] = ovf ? 1000 : cnt;
            asm volatile("bar.sync 1, 256;" ::: "memory");
            const int other = sCnt[et ^ 128], total = sCnt[et] + other;
            if (row < rowsTotal)
            {
                const bool bad = total > TC_TOPK || total == 0;
                if (!bad)
                {
                    const int off = half ? other : 0;
                    for (int e = 0; e < cnt; ++e)
                        candOut[row * TC_TOPK + off + e] = mine[e * 256].y;
                }
                if (half == 0)
                {
                    countOut[row] = bad ? TC_OVERFLOW : static_cast<unsigned>(total);
                    bestOut[row] = bestF; // the certificate's lower bound starts from the best APPROXIMATE score (TOP = 2: the threshold base)
                }
            }
            asm volatile("bar.sync 1, 256;" ::: "memory"); // sBest / sCnt are reused by the next row tile
        }
    }

    tc_fence_before();
    if (PAIR)
        cluster_sync(); // neither CTA leaves (or frees TMEM) while the other may still signal its barriers
    else
        __syncthreads();
    if (warp == 2)
    {
        if (PAIR)
            asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmemBase), "r"(512) : "memory");
        else
            asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmemBase), "r"(512) : "memory");
    }
}

// ------------------------------------------------------------------------------------------------ operand preparation

// power of two 2^(target - e) for v = f 2^e, f in [0.5, 1): v times it lies in [2^(target-1), 2^target); 1 for 0 / NaN / inf
__device__ __forceinline__ float pow2_scale(float v, int target, int lo, int hi)
{
    if (!(v > 0.0f) || v > 3.0e38f)
        return 1.0f;
    int e;
    frexpf(v, &e);
    int k = target - e;
    k = k < lo ? lo : (k > hi ? hi : k);
    return ldexpf(1.0f, k);
}

// map statistics: |m_p|^2 per node (f32, any order: margins only), max |m_pk| and max |m_p|^2 (atomic max on the bits of
// non-negative floats).  One warp per node.
__global__ void map_stats_kernel(const float *__restrict__ mean, int N, int D, int rowStride, float *__restrict__ norm2, TcScale *__restrict__ scale)
{
    const int p = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (p >= N)
        return;
    float s = 0.0f, mx = 0.0f;
    for (int k = lane; k < D; k += 32)
    {
        const float v = mean[static_cast<size_t>(p) * rowStride + k];
        s += v * v;
        mx = fmaxf(mx, fabsf(v)); // NaN is ignored here; a NaN node gets the large constant below
    }
    for (int o = 16; o; o >>= 1)
    {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    if (lane == 0)
    {
        norm2[p] = s;
        if (p == 0 && s != s)
            scale->nanNode0 = 1;
        atomicMax(reinterpret_cast<int *>(&scale->maxAbs), __float_as_int(fminf(mx, 3.0e38f)));
        if (s == s)
            atomicMax(reinterpret_cast<int *>(&scale->maxNorm2), __float_as_int(fminf(s, 3.0e38f)));
    }
}

__global__ void tc_scale_kernel(TcScale *scale, int split)
{
    scale->split = split;
    const float sm = pow2_scale(scale->maxAbs, 10, -100, 100); // max |s_m m| in [2^9, 2^10)
    const float cmax = sm * scale->maxNorm2;                    // largest s_m c_p
    scale->sm = sm;
    scale->tau = 1.0f / pow2_scale(cmax, 13, -120, 120);        // s_m c_p / tau in [2^12, 2^13) for the largest node constant
    scale->mm = sm * sm * scale->maxNorm2;
}

// map rows -> fp16 operand rows of Kpad columns: -2 s_m m_p, then the hi / mid / lo split of s_m c_p / tau in columns
// D .. D+2, zeros behind.  c_p = |m_p|^2 for nodes that may win; padding rows and nodes below min_hits get a constant above
// every real one (node 0 always competes: it seeds findRestrictedBmu regardless of its hit count, src/Som.cpp:316-322).
__global__ void map_operand_kernel(const float *__restrict__ mean, const float *__restrict__ norm2, const u64 *__restrict__ hits, u64 minHits, int N, int Npad, int D,
                                   int rowStride, const TcScale *__restrict__ scale, __half *__restrict__ Mb, int Kpad)
{
    const int p = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (p >= Npad)
        return;
    const float sm = scale->sm, tau = scale->tau;
    const int split = scale->split, cbase = split ? 3 * D : D;
    __half *row = Mb + static_cast<size_t>(p) * Kpad;
    for (int k = lane; k < Kpad; k += 32)
        if (k >= cbase + 3 || (k < cbase && p >= N)) // padding columns, and the data columns of padding rows
            row[k] = __float2half_rn(0.0f);
    if (p < N)
        for (int k = lane; k < D; k += 32)
        {
            const float v = -2.0f * sm * mean[static_cast<size_t>(p) * rowStride + k];
            const __half h = __float2half_rn(v);
            row[k] = h;
            if (split) // columns [0, D) and [D, 2D) meet the rows' hi and lo halves, [2D, 3D) carries the map's lo half
            {
                row[D + k] = h;
                row[2 * D + k] = __float2half_rn(v - __half2float(h));
            }
        }
    if (lane == 0)
    {
        float c = 60000.0f; // pieces of real nodes stay below 2^13
        if (p < N && restricted_eligible(p, hits, minHits) && norm2[p] == norm2[p])
            c = fminf(sm * norm2[p] / tau, 60000.0f);
        const __half hi = __float2half_rn(c);
        const float r1 = c - __half2float(hi);
        const __half mid = __float2half_rn(r1);
        row[cbase] = hi;
        row[cbase + 1] = mid;
        row[cbase + 2] = __float2half_rn(r1 - __half2float(mid));
    }
}

// data rows -> fp16 operand rows: s_r x (s_r = the row's own power-of-two scale), then s_r tau in the three columns D .. D+2,
// zeros behind; per row |s_r x|^2 and the ratio s_m / s_r (margins and certificate).  One warp per row.
__global__ void row_operand_kernel(const float *__restrict__ src, long long rows, int D, const TcScale *__restrict__ scale, __half *__restrict__ dst, int Kpad,
                                   float *__restrict__ norm2, float *__restrict__ ratio)
{
    const long long row = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows)
        return;
    const float *x = src + row * D;
    float mx = 0.0f;
    for (int k = lane; k < D; k += 32)
        mx = fmaxf(mx, fabsf(x[k]));
    for (int o = 16; o; o >>= 1)
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    const float tau = scale->tau;
    int te;
    frexpf(tau, &te); // tau = 2^(te - 1); the tail s_r tau must stay inside [2^-14, 2^15]
    const float sr = pow2_scale(mx, 10, -14 - (te - 1), 15 - (te - 1));
    float s = 0.0f;
    const int split = scale->split, cbase = split ? 3 * D : D;
    __half *out = dst + row * Kpad;
    for (int k = lane; k < Kpad; k += 32)
        if (k >= cbase)
            out[k] = __float2half_rn(k < cbase + 3 ? sr * tau : 0.0f);
    for (int k = lane; k < D; k += 32)
    {
        const float v = sr * x[k]; // a NaN / inf element poisons the row's scores: it takes the exact scan
        const __half h = __float2half_rn(v);
        out[k] = h;
        if (split) // hi | lo | hi against the map's hi | hi | lo
        {
            out[D + k] = __float2half_rn(v - __half2float(h));
            out[2 * D + k] = h;
        }
        s += v * v;
    }
    for (int o = 16; o; o >>= 1)
        s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0)
    {
        norm2[row] = s;
        ratio[row] = scale->sm / sr;
    }
}

// ------------------------------------------------------------------------------------------------ exact rescore + certificate

// Re-evaluation of the candidates with the reference's sequential f32 chain.  Rows keep 1-3 candidates on average, so a
// thread per (row, slot) would leave nine lanes in ten idle: a CTA takes 128 rows, compacts their (row, candidate) items into
// a list (block scan of the counts) and its 256 threads walk the list, all lanes busy; the per-row winner is an atomic min of
// the (distance, node) key in shared memory — lowest index on ties, like the reference.  Then the certificate (see the
// head of this file): the row is final only if no unlisted node can reach the winner's exact distance.  Rows that fail it,
// rows whose list overflowed and rows whose winner is NaN go to the fallback list (exact full scan).
// TOP = 2: the two smallest keys of the row (two shared-memory atomic mins per candidate, key_top2_atomic), and the certificate
// must clear the RUNNER-UP's exact distance: bestA then holds the kernel's final threshold base, every unlisted node q had
// a'_q >= bestA + Delta', so S_r d_q >= bestA + S_r |x|^2 + 0.25 E' > S_r d2 >= S_r d1 — no unlisted node can be either of the
// two or tie with them.  A row without two listed eligible nodes, or with a NaN among its two, takes the exact scan.
constexpr int RS_ROWS = 128;
constexpr int RS_THREADS = 256;
template <int TOP>
__global__ void __launch_bounds__(RS_THREADS) rescore_kernel(const float *__restrict__ x, long long rows, int D, const float *__restrict__ mean, int rowStride,
                                                             const unsigned *__restrict__ cand, const unsigned *__restrict__ count, const float *__restrict__ bestA,
                                                             const float *__restrict__ xnorm2, const float *__restrict__ xratio, const TcScale *__restrict__ scale,
                                                             int Kpad, int order, int N, const u64 *__restrict__ hits, u64 minHits, unsigned *__restrict__ outBmu,
                                                             float *__restrict__ outDist, unsigned *__restrict__ fallbackRows, unsigned *__restrict__ fallbackCount,
                                                             unsigned long long *__restrict__ stats, unsigned *__restrict__ outBmu2, float *__restrict__ outDist2)
{
    __shared__ unsigned sOff[RS_ROWS + 1];
    __shared__ unsigned sWarpTot[RS_ROWS / 32];
    __shared__ u64 sKey[RS_ROWS];
    __shared__ u64 sKey2[TOP == 2 ? 2 * RS_ROWS : 1]; // TOP = 2: (best, second) of row r at 2 r
    __shared__ unsigned short sItem[RS_ROWS * TC_TOPK];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long row0 = static_cast<long long>(blockIdx.x) * RS_ROWS;
    unsigned cnt = 0, c = 0;
    if (tid < RS_ROWS)
    {
        const long long row = row0 + tid;
        cnt = row < rows ? count[row] : 0u;
        c = cnt == TC_OVERFLOW ? 0u : cnt;
        sKey[tid] = ~0ull;
        if (TOP == 2)
            sKey2[2 * tid] = sKey2[2 * tid + 1] = ~0ull;
        unsigned inc = c; // inclusive scan inside the warp
#pragma unroll
        for (int o = 1; o < 32; o <<= 1)
        {
            const unsigned v = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o)
                inc += v;
        }
        if (lane == 31)
            sWarpTot[warp] = inc;
        sOff[tid] = inc - c; // exclusive, warp-local for now
    }
    __syncthreads();
    if (tid < RS_ROWS)
    {
        unsigned base = 0;
        for (int w = 0; w < warp; ++w)
            base += sWarpTot[w];
        const unsigned off = sOff[tid] + base;
        for (unsigned j = 0; j < c; ++j)
            sItem[off + j] = static_cast<unsigned short>((tid << 6) | j);
        if (tid == RS_ROWS - 1)
            sOff[RS_ROWS] = off + c;
    }
    __syncthreads();
    const unsigned total = sOff[RS_ROWS];
    for (unsigned i = tid; i < total; i += RS_THREADS)
    {
        const unsigned it = sItem[i];
        const int r = static_cast<int>(it >> 6), j = static_cast<int>(it & 63u);
        const long long row = row0 + r;
        const unsigned node = cand[row * TC_TOPK + j];
        // eligibility is re-checked here: padding nodes and nodes below min_hits may be listed when their large constant does
        // not dominate (rows much larger than the map); they must not win
        if (node >= static_cast<unsigned>(N) || !restricted_eligible(node, hits, minHits))
            continue;
        const float s = dist_rows_f32(mean + static_cast<size_t>(node) * rowStride, x + row * D, D, order);
        if (TOP == 2)
            key_top2_atomic(&sKey2[2 * r], score_key(s, node), ~0ull);
        else
            atomicMin(&sKey[r], score_key(s, node));
    }
    __syncthreads();
    if (tid < RS_ROWS && row0 + tid < rows)
    {
        const long long row = row0 + tid;
        const u64 key = TOP == 2 ? sKey2[2 * tid] : sKey[tid];
        const u64 key2 = TOP == 2 ? sKey2[2 * tid + 1] : 0ull; // TOP = 2: the runner-up, whose distance the bound must clear
        const u64 keyC = TOP == 2 ? key2 : key;
        const bool nan = (key & 1ull) != 0 || (TOP == 2 && (key2 & 1ull) != 0) || scale->nanNode0;
        bool certified = false;
        if (cnt != TC_OVERFLOW && !nan && keyC != ~0ull)
        {
            // unlisted nodes, in the row's scaled units (S_r = s_r s_m = s_m^2 / ratio): S_r d_q >= best approximate score +
            // S_r |x|^2 + Delta' - E' = ... + 0.25 E' + slack (tc_margins)
            const float xn = xnorm2[row], ratio = xratio[row], sm = scale->sm;
            float E, delta;
            tc_margins(xn, scale->mm, ratio, Kpad, D, scale->split, E, delta);
            const float lower = __fadd_rn(__fadd_rn(bestA[row], __fmul_rn(xn, ratio)), __fmul_rn(0.25f, E));
            const float sd = __fmul_rn(__fdiv_rn(__fmul_rn(sm, sm), ratio), __uint_as_float(static_cast<unsigned>(keyC >> 32))); // S_r d*: a power of two times d*
            certified = lower > sd;
        }
        if (!certified)
        {
            fallbackRows[atomicAdd(fallbackCount, 1u)] = static_cast<unsigned>(row);
            // diagnostics: why (1: list overflow / empty, 2: NaN or nothing eligible, 3: the certificate's bound did not clear d*)
            atomicAdd(stats + (cnt == TC_OVERFLOW ? 1 : (nan || keyC == ~0ull ? 2 : 3)), 1ull);
        }
        else
            store_row_outputs<TOP>(outBmu, outDist, outBmu2, outDist2, static_cast<u64>(row), key, key2);
    }
}

__global__ void add_count_kernel(const unsigned *count, unsigned long long *total) { *total += *count; }

// ------------------------------------------------------------------------------------------------ host side

EncodeTiledFn tensor_map_encoder()
{
    static EncodeTiledFn fn = nullptr;
    if (!fn)
    {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

static int make_map(vsom_ctx *ctx, CUtensorMap *map, void *base, unsigned long long rows, int Kpad, int boxRows)
{
    EncodeTiledFn enc = tensor_map_encoder();
    if (!enc)
        return set_error(ctx, VSOM_ERR_CUDA, "score_tc: cuTensorMapEncodeTiled entry point not available");
    const cuuint64_t dims[2] = {static_cast<cuuint64_t>(Kpad), static_cast<cuuint64_t>(rows)};
    const cuuint64_t strides[1] = {static_cast<cuuint64_t>(Kpad) * 2};
    const cuuint32_t box[2] = {static_cast<cuuint32_t>(TC_BK), static_cast<cuuint32_t>(boxRows)};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
        return set_error(ctx, VSOM_ERR_CUDA, "score_tc: cuTensorMapEncodeTiled failed (" + std::to_string(static_cast<int>(r)) + ")");
    return VSOM_OK;
}

// One batched scoring call: tc_begin (map side, once) -> tc_enqueue per slab of rows (no host synchronisation) -> tc_finish.
// stage slots used: 6 = fp16 map operand + statistics, 7 = fp16 rows of the current slab, 8 = per-row scratch (two sets).
struct TcCall
{
    int D = 0, N = 0, Kpad = 0, kBlocks = 0, kSteps = 0, Npad = 0, nodeTiles = 0, split = 0;
    int top = 1; // 2: best and second-best node of every row (vsom_find_bmu2)
    bool pair = true;
    uint64_t minHits = 0;
    size_t slabRows = 0, setBytes = 0, slab = 0;
    __half *Xb = nullptr;
    TcScale *scale = nullptr;
    unsigned long long *totalDev = nullptr;
    CUtensorMap mapM;
    ScanMap map; // the nodes the rows are scored against
};

static int tc_begin(vsom_ctx *ctx, TcCall &c, const ScanMap &map, size_t maxSlabRows, uint64_t minHits, int split, int top)
{
    const int D = map.Dr, N = map.N;
    c.map = map;
    c.top = top;
    c.D = D;
    c.N = N;
    c.split = split;
    c.kSteps = ((split ? 3 * D : D) + 3 + 15) / 16; // K = 16 per MMA: the model vector (three segments in the precise tier) + the three node-constant columns
    c.Kpad = c.kSteps * 16; // columns of the operand rows; the last 64-wide TMA box may reach past them: zero fill, no memory traffic
    c.kBlocks = (c.Kpad + TC_BK - 1) / TC_BK;
    c.Npad = (N + TC_BN - 1) / TC_BN * TC_BN;
    c.nodeTiles = c.Npad / TC_BN;
    c.minHits = minHits;

    // ---- map side: statistics -> scales -> fp16 operand with the node constants folded in
    const size_t mbBytes = sizeof(__half) * static_cast<size_t>(c.Npad) * c.Kpad;
    int rc = stage_reserve(ctx, 6, mbBytes + sizeof(float) * (static_cast<size_t>(c.Npad) + 64));
    if (rc)
        return rc;
    __half *Mb = static_cast<__half *>(ctx->stage[6]);
    float *mnorm = reinterpret_cast<float *>(static_cast<unsigned char *>(ctx->stage[6]) + mbBytes);
    c.scale = reinterpret_cast<TcScale *>(mnorm + c.Npad);
    VSOM_CUDA(ctx, cudaMemsetAsync(c.scale, 0, sizeof(TcScale), ctx->stream));
    map_stats_kernel<<<(N + 7) / 8, 256, 0, ctx->stream>>>(map.mean, N, D, map.rowStride, mnorm, c.scale);
    tc_scale_kernel<<<1, 1, 0, ctx->stream>>>(c.scale, split);
    map_operand_kernel<<<(c.Npad + 7) / 8, 256, 0, ctx->stream>>>(map.mean, mnorm, map.hits, minHits, N, c.Npad, D, map.rowStride, c.scale, Mb, c.Kpad);
    ctx->launches += 3;
    // function attributes are per device: set them for every context (not once per process), and ask once whether the device can
    // co-schedule a cluster of two of these CTAs (it cannot on a partition without whole TPCs; then the single-CTA kernel runs)
    if (!ctx->tcAttrSet)
    {
        VSOM_CUDA(ctx, cudaFuncSetAttribute(score_tc_kernel<false, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcShared::TOTAL));
        VSOM_CUDA(ctx, cudaFuncSetAttribute(score_tc_kernel<true, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcShared::TOTAL));
        VSOM_CUDA(ctx, cudaFuncSetAttribute(score_tc_kernel<false, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcShared::TOTAL));
        VSOM_CUDA(ctx, cudaFuncSetAttribute(score_tc_kernel<true, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcShared::TOTAL));
        cudaLaunchConfig_t q = {};
        cudaLaunchAttribute qa[1];
        q.gridDim = dim3(2);
        q.blockDim = dim3(TC_THREADS);
        q.dynamicSmemBytes = TcShared::TOTAL;
        qa[0].id = cudaLaunchAttributeClusterDimension;
        qa[0].val.clusterDim.x = 2;
        qa[0].val.clusterDim.y = 1;
        qa[0].val.clusterDim.z = 1;
        q.attrs = qa;
        q.numAttrs = 1;
        int clusters = 0;
        const cudaError_t qe = cudaOccupancyMaxActiveClusters(&clusters, score_tc_kernel<true, 1>, &q); // the TOP = 2 kernel has the same launch shape
        if (qe != cudaSuccess)
            cudaGetLastError(); // not an error of the scoring call
        ctx->tcPairOk = qe == cudaSuccess && clusters >= 1 ? 1 : 0;
        ctx->tcAttrSet = 1;
    }
    // CTA pairs (tcgen05 cta_group::2, the default): each CTA of a pair loads half of a node tile (box of 128 nodes)
    const char *pairEnv = getenv("VSOM_TC_PAIR"); // read per call: the tests run both variants in one process
    c.pair = (pairEnv ? atoi(pairEnv) != 0 : true) && ctx->numSMs >= 2 && ctx->tcPairOk;
    ctx->lastScorePair = c.pair ? 1 : 0;
    rc = make_map(ctx, &c.mapM, Mb, static_cast<unsigned long long>(c.Npad), c.Kpad, c.pair ? TC_BN / 2 : TC_BN);
    if (rc)
        return rc;
    // ---- rows go through in slabs (the fp16 staging buffer: 2.7 GB at K = 256 + 3 for 4M rows).  Two streams: the context's
    // stream converts a slab and runs the tensor-core search; an auxiliary stream re-scores the slab's candidates (and scans
    // the few rows the certificate rejected) while the next slab is already being searched.  Candidate scratch is
    // double-buffered by slab parity; nothing returns to the host in between.
    c.slabRows = maxSlabRows;
    rc = stage_reserve(ctx, 7, sizeof(__half) * c.slabRows * c.Kpad);
    if (rc)
        return rc;
    // per-row scratch: candidates, their count, |s_r x|^2, s_m / s_r, best approximate score, fallback list; per set: fallback count
    const size_t perRow = sizeof(unsigned) * TC_TOPK + sizeof(unsigned) + 3 * sizeof(float) + sizeof(unsigned) + sizeof(u64) * top; // + key(s) of the exact scan's node splits
    c.setBytes = (perRow * c.slabRows + 512 + 255) & ~static_cast<size_t>(255);
    rc = stage_reserve(ctx, 8, 2 * c.setBytes + 256);
    if (rc)
        return rc;
    if (!ctx->auxStream)
    {
        VSOM_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->auxStream, cudaStreamNonBlocking));
        VSOM_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->copyStream, cudaStreamNonBlocking));
        for (int i = 0; i < 2; ++i)
        {
            VSOM_CUDA(ctx, cudaEventCreateWithFlags(&ctx->evScore[i], cudaEventDisableTiming));
            VSOM_CUDA(ctx, cudaEventCreateWithFlags(&ctx->evDone[i], cudaEventDisableTiming));
        }
        for (int i = 0; i < 3; ++i)
        {
            VSOM_CUDA(ctx, cudaEventCreateWithFlags(&ctx->evCopied[i], cudaEventDisableTiming));
            VSOM_CUDA(ctx, cudaEventCreateWithFlags(&ctx->evSlabDone[i], cudaEventDisableTiming));
        }
    }
    c.Xb = static_cast<__half *>(ctx->stage[7]);
    c.totalDev = reinterpret_cast<unsigned long long *>(static_cast<unsigned char *>(ctx->stage[8]) + 2 * c.setBytes);
    VSOM_CUDA(ctx, cudaMemsetAsync(c.totalDev, 0, 4 * sizeof(unsigned long long), ctx->stream));
    VSOM_CUDA(ctx, cudaMemsetAsync(ctx->errFlag, 0, sizeof(int), ctx->stream));
    c.slab = 0;
    return VSOM_OK;
}

// Host rows: the results of a slab are final in `dev` (device staging).  Behind them on `stream`: the similarity pass, then the
// copies to the caller's buffers in `host`.  The predicted columns (host.q) are filled into host.meanDev / sigmaDev and copied out on
// `outStream` behind the slab's BMUs: on the pipelined path a stream of their own, so that copying out 8q bytes per row overlaps the
// next slab's re-scoring and the H2D copies instead of queuing in front of them.
static int slab_to_host(vsom_ctx *ctx, const float *xs, size_t rows, const ScoreOut &dev, const ScoreOut &host, cudaStream_t stream, cudaStream_t outStream)
{
    if (host.k != 0.0f)
    {
        const int rc = launch_similarity_rowmax(ctx, xs, rows, dev.bmu, host.k, host.rowMaxDev, stream);
        if (rc)
            return rc;
        VSOM_CUDA(ctx, cudaMemcpyAsync(host.rowMax, host.rowMaxDev, sizeof(float) * rows, cudaMemcpyDeviceToHost, stream));
    }
    if (host.q && (host.mean || host.sigma))
    {
        if (outStream != stream)
        {
            VSOM_CUDA(ctx, cudaEventRecord(ctx->evOut, stream));
            VSOM_CUDA(ctx, cudaStreamWaitEvent(outStream, ctx->evOut, 0));
        }
        const int rc = launch_predict_fill(ctx, dev.bmu, rows, host, true, outStream);
        if (rc)
            return rc;
        const size_t bytes = sizeof(float) * rows * static_cast<size_t>(host.q);
        if (host.mean)
            VSOM_CUDA(ctx, cudaMemcpyAsync(host.mean, host.meanDev, bytes, cudaMemcpyDeviceToHost, outStream));
        if (host.sigma)
            VSOM_CUDA(ctx, cudaMemcpyAsync(host.sigma, host.sigmaDev, bytes, cudaMemcpyDeviceToHost, outStream));
    }
    if (host.bmu)
        VSOM_CUDA(ctx, cudaMemcpyAsync(host.bmu, dev.bmu, sizeof(unsigned) * rows, cudaMemcpyDeviceToHost, stream));
    if (host.dist)
        VSOM_CUDA(ctx, cudaMemcpyAsync(host.dist, dev.dist, sizeof(float) * rows, cudaMemcpyDeviceToHost, stream));
    if (host.bmu2)
        VSOM_CUDA(ctx, cudaMemcpyAsync(host.bmu2, dev.bmu2, sizeof(unsigned) * rows, cudaMemcpyDeviceToHost, stream));
    if (host.dist2)
        VSOM_CUDA(ctx, cudaMemcpyAsync(host.dist2, dev.dist2, sizeof(float) * rows, cudaMemcpyDeviceToHost, stream));
    return VSOM_OK;
}

// One slab: xs = rows x D f32 in device memory (must stay valid until the slab's evDone event).  Results go to `dev` (device
// memory, top = c.top) and, for host rows, from there to `host` on the re-scoring stream.
static int tc_enqueue(vsom_ctx *ctx, TcCall &c, const float *xs, size_t rows, const ScoreOut &dev, const ScoreOut *host)
{
    const int par = static_cast<int>(c.slab & 1);
    unsigned char *set = static_cast<unsigned char *>(ctx->stage[8]) + par * c.setBytes;
    unsigned *cand = reinterpret_cast<unsigned *>(set);
    unsigned *candCount = cand + c.slabRows * TC_TOPK;
    float *xnorm = reinterpret_cast<float *>(candCount + c.slabRows);
    float *xratio = xnorm + c.slabRows;
    float *bestA = xratio + c.slabRows;
    unsigned *fbRows = reinterpret_cast<unsigned *>(bestA + c.slabRows);
    u64 *fbKeys = reinterpret_cast<u64 *>(set + ((reinterpret_cast<unsigned char *>(fbRows + c.slabRows) - set + 7) & ~static_cast<size_t>(7)));
    unsigned *fbCount = reinterpret_cast<unsigned *>(fbKeys + c.slabRows * c.top);
    const int order = ctx->order == VSOM_ORDER_EIGEN_SSE ? VSOM_ORDER_EIGEN_SSE : VSOM_ORDER_REFERENCE;

    if (c.slab >= 2)
        VSOM_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->evDone[par], 0)); // slab - 2 is done with this scratch set
    row_operand_kernel<<<static_cast<unsigned>((rows + 7) / 8), 256, 0, ctx->stream>>>(xs, static_cast<long long>(rows), c.D, c.scale, c.Xb, c.Kpad, xnorm, xratio);
    CUtensorMap mapX;
    int rc = make_map(ctx, &mapX, c.Xb, rows, c.Kpad, TC_BM);
    if (rc)
        return rc;
    const int rowTiles = static_cast<int>((rows + TC_BM - 1) / TC_BM);
    VSOM_CUDA(ctx, cudaMemsetAsync(fbCount, 0, sizeof(unsigned), ctx->stream));
    {
        cudaLaunchConfig_t cfg = {};
        cudaLaunchAttribute attr[1];
        cfg.blockDim = dim3(TC_THREADS);
        cfg.dynamicSmemBytes = TcShared::TOTAL;
        cfg.stream = ctx->stream;
        if (c.pair)
        {
            // one cluster of two CTAs (the two SMs of a TPC) per 256 rows
            const int units = (rowTiles + 1) / 2;
            cfg.gridDim = dim3(static_cast<unsigned>(2 * std::min(units, ctx->numSMs / 2)));
            attr[0].id = cudaLaunchAttributeClusterDimension;
            attr[0].val.clusterDim.x = 2;
            attr[0].val.clusterDim.y = 1;
            attr[0].val.clusterDim.z = 1;
            cfg.attrs = attr;
            cfg.numAttrs = 1;
        }
        else
            cfg.gridDim = dim3(static_cast<unsigned>(std::min(rowTiles, ctx->numSMs)));
        const int rowsI = static_cast<int>(rows);
        const float *xn = xnorm, *xr = xratio;
        const TcScale *sc = c.scale;
        // the kernel's debug word is 1: staggered node-tile starts, none of the timing-only variants
        auto kern = c.top == 2 ? (c.pair ? score_tc_kernel<true, 2> : score_tc_kernel<false, 2>) : (c.pair ? score_tc_kernel<true, 1> : score_tc_kernel<false, 1>);
        VSOM_CUDA(ctx, cudaLaunchKernelEx(&cfg, kern, mapX, c.mapM, c.kSteps, rowsI, rowTiles, c.nodeTiles, c.kBlocks, c.Kpad, 1, c.D, xn, xr, sc, cand, candCount, bestA,
                                          ctx->errFlag));
    }
    cudaStream_t rs = ctx->auxStream;
    VSOM_CUDA(ctx, cudaEventRecord(ctx->evScore[par], ctx->stream));
    VSOM_CUDA(ctx, cudaStreamWaitEvent(rs, ctx->evScore[par], 0));
    (c.top == 2 ? rescore_kernel<2> : rescore_kernel<1>)<<<static_cast<unsigned>((rows + RS_ROWS - 1) / RS_ROWS), RS_THREADS, 0, rs>>>(
        xs, static_cast<long long>(rows), c.D, c.map.mean, c.map.rowStride, cand, candCount, bestA, xnorm, xratio, c.scale, c.Kpad, order, c.N, c.map.hits, c.minHits, dev.bmu,
        dev.dist, fbRows, fbCount, c.totalDev, dev.bmu2, dev.dist2);
    // rows the certificate rejected: exact scan (K3 tiles over the row list; the count stays on the device)
    add_count_kernel<<<1, 1, 0, rs>>>(fbCount, c.totalDev);
    rc = launch_find_bmu_list(ctx, xs, rows, fbRows, fbCount, c.minHits, dev, rs, fbKeys, c.map);
    if (rc)
        return rc;
    if (host)
    {
        rc = slab_to_host(ctx, xs, rows, dev, *host, rs, ctx->outStream);
        if (rc)
            return rc;
    }
    VSOM_CUDA(ctx, cudaEventRecord(ctx->evDone[par], rs));
    ctx->launches += 4;
    VSOM_CUDA(ctx, cudaGetLastError());
    ++c.slab;
    return VSOM_OK;
}

// fallbackRows: rows of this run that took the exact scan
static int tc_finish(vsom_ctx *ctx, TcCall &c, unsigned long long &fallbackRows)
{
    // the context's stream owns the results again
    for (int i = 0; i < 2 && static_cast<size_t>(i) < c.slab; ++i)
        VSOM_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->evDone[i], 0));
    unsigned long long st[4] = {0, 0, 0, 0};
    int flag = 0;
    VSOM_CUDA(ctx, cudaMemcpyAsync(st, c.totalDev, sizeof(st), cudaMemcpyDeviceToHost, ctx->stream));
    VSOM_CUDA(ctx, cudaMemcpyAsync(&flag, ctx->errFlag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    VSOM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (flag)
        return set_error(ctx, VSOM_ERR_TIMEOUT, "score_tc: pipeline barrier timed out (kernel bug)");
    VSOM_CUDA(ctx, cudaGetLastError());
    fallbackRows = st[0];
    for (int i = 0; i < 3; ++i)
        ctx->tcStats[i] += st[i + 1];
    return VSOM_OK;
}

// Which tier scores this call.  Tier 1 (one half per operand) costs 2 N D tensor flops per row; on a trained map the BMU's
// neighbours differ from it by less than its product error and most rows would end in the exact scan, so tier 2 (hi / lo
// pairs, 6 N D flops, ~2^-20 relative error) takes over when a probe of the first rows sends more than 4 % of them there
// (tier 1 at f fallback costs ~ t1 + f t_exact per row, tier 2 ~ 3 t1: break-even near 4 %).  VSOM_TC_TIER=1|2 forces one.
static const size_t kTcProbeRows = 8192;
static const double kTcTierSwitch = 0.04;
static const double kTcExactSwitch = 0.25; // tier-2 probe fallback above this: the tensor cores select nothing useful, the rest is scanned exactly (tier "3")

// rows per slab such that the fp16 operand staging of a slab stays below 2.5 GiB
static size_t tc_slab_cap(const ScanMap &map, int split)
{
    const size_t kext = static_cast<size_t>(split ? 3 * map.Dr : map.Dr) + 3, kpad = (kext + 15) / 16 * 16;
    return std::max<size_t>(TC_BM, ((size_t{5} << 29) / (kpad * 2)) & ~static_cast<size_t>(TC_BM - 1));
}

// The tier policy of both forms.  run(r0, rows, tier, fb) scores rows [r0, r0 + rows) through tier 1 or 2 and sets fb to the
// number of them that took the exact scan.  On return `tier` is the tier chosen, `done` rows have been scored (all n, unless
// the tier-2 probe chose tier 3: then rows [done, n) are left to the exact scan) and `fallback` of them took the exact scan.
template <class Run>
static int tc_score_tiers(size_t n, const Run &run, int &tier, size_t &done, unsigned long long &fallback)
{
    const char *e = getenv("VSOM_TC_TIER");
    const int forced = e ? atoi(e) : 0;
    tier = forced;
    unsigned long long fb = 0;
    done = 0;
    fallback = 0;
    if (tier != 1 && tier != 2)
    {
        // probe: the first rows through tier 1 (their results stand), then decide
        done = std::min(n, kTcProbeRows);
        const int rc = run(0, done, 1, fb);
        if (rc)
            return rc;
        fallback += fb;
        tier = static_cast<double>(fb) > kTcTierSwitch * static_cast<double>(done) ? 2 : 1;
    }
    if (tier == 2 && !forced && n - done > kTcProbeRows)
    {
        // second probe: the next rows through tier 2 (their results stand).  Data whose norms dwarf the map's (or a map whose nodes
        // nearly coincide) leaves more candidates than the lists hold even at 2^-20: the remainder goes straight to the exact scan
        const int rc = run(done, kTcProbeRows, 2, fb);
        if (rc)
            return rc;
        fallback += fb;
        done += kTcProbeRows;
        if (static_cast<double>(fb) > kTcExactSwitch * static_cast<double>(kTcProbeRows))
            tier = 3;
    }
    if (done < n && tier != 3)
    {
        const int rc = run(done, n - done, tier, fb);
        if (rc)
            return rc;
        fallback += fb;
        done = n;
    }
    return VSOM_OK;
}

// rows [0, n) of xDev through one tier; slabs of the given size
static int tc_run_device(vsom_ctx *ctx, const ScanMap &map, const float *xDev, size_t n, uint64_t minHits, int split, size_t slabRows, const ScoreOut &out,
                         unsigned long long &fallbackRows)
{
    slabRows = std::min(n, std::min(slabRows, tc_slab_cap(map, split)));
    TcCall c;
    int rc = tc_begin(ctx, c, map, slabRows, minHits, split, out.top);
    if (rc)
        return rc;
    for (size_t r0 = 0; r0 < n; r0 += slabRows)
    {
        rc = tc_enqueue(ctx, c, xDev + r0 * c.D, std::min(slabRows, n - r0), out.at(r0), nullptr);
        if (rc)
            return rc;
    }
    return tc_finish(ctx, c, fallbackRows);
}

// Rows in HOST memory (the call Som::evaluate / measureSimilarity / mapDataSet make), rows [0, n) through one tier: the chunk
// crosses PCIe in slabs on a copy stream into one of three staging buffers while the previous slabs are searched and re-scored,
// and each slab's results return to the host behind its re-scoring.  With pinned host memory the three engines (H2D, SMs, D2H)
// overlap fully; the call is then bound by the slower of PCIe (4 D bytes per row) and the kernel.  stage slots: 0 = three row
// slabs, 1 / 2 = BMU / distance of the whole run, 4 = runner-ups and their distances (top = 2), 11 = the three slabs gathered to the
// map's columns (map.cols: the copies carry srcDin floats per row, the search reads D), 12 = three slabs of predicted columns (out.q).
// The predictions of slab s go out on ctx->outStream; the fill of slab s + 3 reuses slab s's staging behind its copies there.
static int tc_run_host(vsom_ctx *ctx, const ScanMap &map, const float *xHost, size_t n, uint64_t minHits, int split, size_t slabRows, const ScoreOut &out,
                       unsigned long long &fallbackRows)
{
    slabRows = std::min(n, std::min(slabRows, tc_slab_cap(map, split)));
    const size_t D = static_cast<size_t>(map.Din), xD = map.cols ? static_cast<size_t>(map.srcDin) : D;
    // THREE staging buffers: the copy of slab s + 1 must not wait for the re-scoring (and the exact scan of the rejected rows) of
    // slab s - 1, which with two buffers sat on the critical path (measured: 14.6 ms per 512 K-row slab instead of 11.5)
    int rc = stage_reserve(ctx, 0, sizeof(float) * 3 * slabRows * xD);
    if (rc)
        return rc;
    float *cbuf[3] = {};
    if (map.cols)
    {
        rc = stage_reserve(ctx, 11, sizeof(float) * 3 * slabRows * D);
        if (rc)
            return rc;
        for (int i = 0; i < 3; ++i)
            cbuf[i] = static_cast<float *>(ctx->stage[11]) + static_cast<size_t>(i) * slabRows * D;
    }
    rc = stage_reserve(ctx, 1, sizeof(unsigned) * n);
    if (rc)
        return rc;
    rc = stage_reserve(ctx, 2, sizeof(float) * n);
    if (rc)
        return rc;
    float *xbuf[3];
    for (int i = 0; i < 3; ++i)
        xbuf[i] = static_cast<float *>(ctx->stage[0]) + static_cast<size_t>(i) * slabRows * xD;
    ScoreOut dev;
    dev.bmu = static_cast<unsigned *>(ctx->stage[1]);
    dev.dist = static_cast<float *>(ctx->stage[2]);
    dev.top = out.top;
    if (out.top == 2)
    {
        rc = stage_reserve(ctx, 4, (sizeof(unsigned) + sizeof(float)) * n);
        if (rc)
            return rc;
        dev.bmu2 = static_cast<unsigned *>(ctx->stage[4]);
        dev.dist2 = reinterpret_cast<float *>(dev.bmu2 + n);
    }
    const bool predict = out.q && (out.mean || out.sigma);
    const size_t slabVals = slabRows * static_cast<size_t>(out.q);
    if (predict)
    {
        rc = stage_reserve(ctx, 12, sizeof(float) * 2 * 3 * slabVals);
        if (rc)
            return rc;
        if (!ctx->outStream)
        {
            VSOM_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->outStream, cudaStreamNonBlocking));
            VSOM_CUDA(ctx, cudaEventCreateWithFlags(&ctx->evOut, cudaEventDisableTiming));
        }
    }
    TcCall c;
    rc = tc_begin(ctx, c, map, slabRows, minHits, split, out.top);
    if (rc)
        return rc;
    // the staging buffers may still be in use by earlier work of the context's stream
    VSOM_CUDA(ctx, cudaEventRecord(ctx->evCopied[0], ctx->stream));
    VSOM_CUDA(ctx, cudaStreamWaitEvent(ctx->copyStream, ctx->evCopied[0], 0));
    auto copy_in = [&](size_t slab) -> int {
        const size_t r0 = slab * slabRows, rows = std::min(slabRows, n - r0);
        const int b = static_cast<int>(slab % 3);
        if (slab >= 3)
            VSOM_CUDA(ctx, cudaStreamWaitEvent(ctx->copyStream, ctx->evSlabDone[b], 0)); // slab - 3 (same buffer) is fully re-scored
        VSOM_CUDA(ctx, cudaMemcpyAsync(xbuf[b], xHost + r0 * xD, sizeof(float) * rows * xD, cudaMemcpyHostToDevice, ctx->copyStream));
        VSOM_CUDA(ctx, cudaEventRecord(ctx->evCopied[b], ctx->copyStream));
        return VSOM_OK;
    };
    const size_t slabs = (n + slabRows - 1) / slabRows;
    rc = copy_in(0);
    if (rc)
        return rc;
    size_t issued = 1;
    for (size_t sl = 0; sl < slabs; ++sl)
    {
        const size_t r0 = sl * slabRows, rows = std::min(slabRows, n - r0);
        const int b = static_cast<int>(sl % 3);
        VSOM_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->evCopied[b], 0));
        const float *xs = xbuf[b];
        if (map.cols)
        {
            // cbuf[b] is free: slab sl - 3 was re-scored before the copy of this slab began (evSlabDone -> evCopied)
            rc = launch_gather_columns(ctx, xbuf[b], rows, xD, map.cols, static_cast<int>(D), static_cast<int>(D), cbuf[b], ctx->stream);
            if (rc)
                return rc;
            xs = cbuf[b];
        }
        ScoreOut host = out.at(r0);
        if (predict)
        {
            host.meanDev = static_cast<float *>(ctx->stage[12]) + 2 * static_cast<size_t>(b) * slabVals;
            host.sigmaDev = host.meanDev + slabVals;
        }
        rc = tc_enqueue(ctx, c, xs, rows, dev.at(r0), &host);
        if (rc)
            return rc;
        VSOM_CUDA(ctx, cudaEventRecord(ctx->evSlabDone[b], ctx->auxStream)); // behind the slab's re-scoring and result copies
        // up to two copies ahead, enqueued AFTER the search of slab sl: a pageable source blocks the host here, not the device
        while (issued < std::min(slabs, sl + 3))
        {
            rc = copy_in(issued++);
            if (rc)
                return rc;
        }
    }
    if (predict)
    {
        // the context's stream owns the predictions again once they have been copied out
        VSOM_CUDA(ctx, cudaEventRecord(ctx->evOut, ctx->outStream));
        VSOM_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->evOut, 0));
    }
    return tc_finish(ctx, c, fallbackRows);
}

// The exact scan of rows in HOST memory, in slabs (VSOM_EXACT_HOST_SLAB_LOG2, default 2^20 rows): staging stays bounded and each
// slab's results return before the next slab is copied in.  stage slots as tc_run_host, sized by the slab (one buffer each).
static int score_exact_host(vsom_ctx *ctx, const ScanMap &map, const float *xHost, size_t n, uint64_t minHits, const ScoreOut &out)
{
    const char *slabEnv = getenv("VSOM_EXACT_HOST_SLAB_LOG2");
    const size_t slab = std::min(n, static_cast<size_t>(1) << (slabEnv ? atoi(slabEnv) : 20));
    const size_t D = static_cast<size_t>(map.Din), xD = map.cols ? static_cast<size_t>(map.srcDin) : D;
    int rc = stage_reserve(ctx, 0, sizeof(float) * slab * xD);
    if (rc)
        return rc;
    float *cDev = nullptr;
    if (map.cols)
    {
        rc = stage_reserve(ctx, 11, sizeof(float) * slab * D);
        if (rc)
            return rc;
        cDev = static_cast<float *>(ctx->stage[11]);
    }
    rc = stage_reserve(ctx, 1, sizeof(unsigned) * slab);
    if (rc)
        return rc;
    rc = stage_reserve(ctx, 2, sizeof(float) * slab);
    if (rc)
        return rc;
    float *xDev = static_cast<float *>(ctx->stage[0]);
    float *predDev = nullptr;
    if (out.q && (out.mean || out.sigma))
    {
        rc = stage_reserve(ctx, 12, sizeof(float) * 2 * slab * out.q);
        if (rc)
            return rc;
        predDev = static_cast<float *>(ctx->stage[12]);
    }
    ScoreOut dev;
    dev.bmu = static_cast<unsigned *>(ctx->stage[1]);
    dev.dist = static_cast<float *>(ctx->stage[2]);
    dev.top = out.top;
    if (out.top == 2)
    {
        rc = stage_reserve(ctx, 4, (sizeof(unsigned) + sizeof(float)) * slab);
        if (rc)
            return rc;
        dev.bmu2 = static_cast<unsigned *>(ctx->stage[4]);
        dev.dist2 = reinterpret_cast<float *>(dev.bmu2 + slab);
    }
    for (size_t r0 = 0; r0 < n; r0 += slab)
    {
        const size_t rows = std::min(slab, n - r0);
        VSOM_CUDA(ctx, cudaMemcpyAsync(xDev, xHost + r0 * xD, sizeof(float) * rows * xD, cudaMemcpyHostToDevice, ctx->stream));
        const float *xs = xDev;
        if (map.cols)
        {
            rc = launch_gather_columns(ctx, xDev, rows, xD, map.cols, static_cast<int>(D), static_cast<int>(D), cDev, ctx->stream);
            if (rc)
                return rc;
            xs = cDev;
        }
        rc = launch_find_bmu_list(ctx, xs, rows, nullptr, nullptr, minHits, dev, ctx->stream, nullptr, map);
        if (rc)
            return rc;
        ScoreOut host = out.at(r0);
        if (predDev)
        {
            host.meanDev = predDev;
            host.sigmaDev = predDev + slab * out.q;
        }
        rc = slab_to_host(ctx, xs, rows, dev, host, ctx->stream, ctx->stream);
        if (rc)
            return rc;
        VSOM_CUDA(ctx, cudaStreamSynchronize(ctx->stream)); // the staging buffers are reused by the next slab
    }
    return VSOM_OK;
}

// Batches of at least kTcMinRows rows on a shape K2 covers take the tensor-core candidate search + exact rescore (same results,
// bit for bit); everything else the exact scan.  K2 covers the Standard / Median Comparer (the contraction form of |m - x|^2) up to
// 2048 model columns; rows longer than TC_MAXK stream their A k-blocks.
static const size_t kTcMinRows = 1024;

int score_rows(vsom_ctx *ctx, const float *x, bool hostRows, size_t n, uint64_t minHits, bool allowTc, const ScoreOut &out, uint64_t *fallbackRows,
               const ScanMap &map)
{
    // floats between the caller's rows
    const size_t xD = static_cast<size_t>(hostRows && map.cols ? map.srcDin : map.Din);
    if (fallbackRows)
        *fallbackRows = 0;
    if (hostRows && n == 0)
        return VSOM_OK; // nothing ran: vsom_debug_last_score_tc keeps reporting the previous call
    int tier = 0;
    size_t done = 0;
    unsigned long long fallback = 0;
    if (allowTc && map.transform != VSOM_CLR && map.Dr <= 2048 && n >= kTcMinRows)
    {
        // test knobs; smaller device slabs measured slower (per-slab ramp and tail of the persistent kernel)
        const char *slabEnv = getenv(hostRows ? "VSOM_TC_HOST_SLAB_LOG2" : "VSOM_TC_SLAB_LOG2");
        const size_t slab1 = static_cast<size_t>(1) << (slabEnv ? atoi(slabEnv) : hostRows ? 19 : 22);
        const size_t slab2 = hostRows ? slab1 : std::min<size_t>(slab1, static_cast<size_t>(1) << 20);
        const int rc = tc_score_tiers(
            n,
            [&](size_t r0, size_t rows, int t, unsigned long long &fb) {
                const int split = t == 2 ? 1 : 0;
                const size_t slab = t == 2 ? slab2 : slab1;
                return hostRows ? tc_run_host(ctx, map, x + r0 * xD, rows, minHits, split, slab, out.at(r0), fb)
                                : tc_run_device(ctx, map, x + r0 * xD, rows, minHits, split, slab, out.at(r0), fb);
            },
            tier, done, fallback);
        if (rc)
            return rc;
    }
    ctx->lastScoreTier = tier;
    if (done < n) // every row, or the rows the probes sent to the exact scan (tier 3)
    {
        const float *xr = x + done * xD;
        const int rc = hostRows ? score_exact_host(ctx, map, xr, n - done, minHits, out.at(done))
                                : launch_find_bmu_list(ctx, xr, n - done, nullptr, nullptr, minHits, out.at(done), ctx->stream, nullptr, map);
        if (rc)
            return rc;
        fallback += n - done;
    }
    if (!hostRows && out.q && (out.mean || out.sigma))
    {
        // device rows: the predicted columns behind the final BMUs, which the context's stream owns again (tc_finish joined the
        // re-scoring stream)
        const int rc = launch_predict_fill(ctx, out.bmu, n, out, false, ctx->stream);
        if (rc)
            return rc;
    }
    if (fallbackRows)
        *fallbackRows = fallback;
    return VSOM_OK;
}

} // namespace vsom
