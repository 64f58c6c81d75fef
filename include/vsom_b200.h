/* vsom_b200.h — C-ABI of libvsom_b200.so, the B200 (sm_100a) implementation of the VSOM training and
 * scoring hot path.
 *
 * The reference (PereUbu7/Variational-Self-Organizing-Maps) has no FFI layer: its boundary is the C++
 * class surface in include/SOM.hpp.  The host classes shipped in this repository's include/SOM.hpp keep
 * that surface and forward the hot methods to the entry points below; each entry point names the
 * reference method it replaces (file:line relative to the reference tree).  Only plain pointers and
 * sizes cross this boundary — no Eigen, no torch, no C++ types.
 *
 * Conventions
 *   - every function returns 0 (VSOM_OK) or a negative vsom_status; vsom_last_error() gives the text.
 *     Nothing throws, nothing calls exit().  There is NO CPU fallback: without a usable CUDA device
 *     vsom_create() fails with VSOM_ERR_NO_DEVICE.
 *   - one context is driven by one host thread at a time.
 *   - "host" entry points take pageable or pinned host pointers, copy in/out on the context's stream and
 *     are complete on return.  "_device" entry points take device pointers, only enqueue work on the
 *     context's stream (vsom_stream) and return immediately; call vsom_synchronize() before reading.
 *   - planes are row-major: node p = y*W + x (src/Som.cpp:119,191,895), N = W*H rows of Dm floats, where
 *     Dm = vsom_model_length(d_in, transform) (Transformation::Length, src/Transformation.cpp:31-35,162-165).
 */
#ifndef VSOM_B200_H
#define VSOM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define VSOM_API __attribute__((visibility("default")))
#else
#define VSOM_API
#endif

typedef struct vsom_ctx vsom_ctx;

typedef enum vsom_status
{
    VSOM_OK = 0,
    VSOM_ERR_INVALID = -1,     /* bad argument */
    VSOM_ERR_CUDA = -2,        /* CUDA runtime error (text in vsom_last_error) */
    VSOM_ERR_UNSUPPORTED = -3, /* a regime this build does not run on the device (never silently on the CPU) */
    VSOM_ERR_TIMEOUT = -4,     /* a persistent kernel gave up waiting for a peer CTA / rank */
    VSOM_ERR_NO_DEVICE = -5
} vsom_status;

/* The three shipped Transformation factories (src/Transformation.cpp:3-39, :41-77, :79-167). */
typedef enum vsom_transform_kind
{
    VSOM_STANDARD = 0, /* Comparer m-v, Stepper v-m */
    VSOM_MEDIAN = 1,   /* Comparer m-v, Stepper sign(v-m) */
    VSOM_CLR = 2       /* combinatorial linear regression over the J(J-1)/2 pairs i<j */
} vsom_transform_kind;

/* Som::WeigthDecayFunction (include/SOM.hpp:70-75).  BatchMap is not an online mode. */
typedef enum vsom_decay_kind
{
    VSOM_EXPONENTIAL = 0,
    VSOM_INVERSE_PROPORTIONAL = 1
} vsom_decay_kind;

/* Order in which the squared residuals of one distance are summed (f32).
 *   REFERENCE: k = 0,1,2,... sequentially — the order of `comparer.dot(comparer)` (src/Som.cpp:140) as the
 *              reference compiles in this repository's oracle.  Distances, BMUs and the whole training
 *              trajectory are then bit-identical to the reference.
 *   LANES:     32 interleaved partial sums (k mod 32) each sequential, combined by a fixed xor-butterfly
 *              (16,8,4,2,1).  Deterministic; BMUs can differ from the reference only at near-ties (relative
 *              distance gap below 2*Dm*2^-24, see DESIGN.md).  It runs on the generic online-step kernel; since
 *              K1F (online_step_fast.cu) the REFERENCE order is the faster of the two for maps that fit on chip.
 *              Only the online step sums in the lanes order: every other path of such a context (scoring, all_dists,
 *              soft assignment, U-matrix, the batch-map trainer) sums in the REFERENCE order and returns its bits.
 *   EIGEN_SSE: the order `dot()` / `squaredNorm()` have when the reference is built against real Eigen (3.3 / 3.4) with
 *              its release flags (-msse2, README.md:64-69, build/Makefile:18): Eigen's vectorised redux over Packet4f —
 *              two 4-wide accumulators over strides of 8 elements (eight interleaved sequential chains), res0 + res1,
 *              one more packet when 4..7 elements remain, the horizontal sum (p0 + p2) + (p1 + p3), then the scalar tail.
 *              Bit-identical to the reference compiled with -DVSOM_COMPAT_EIGEN_SSE_REDUX (oracle/Makefile), which makes
 *              the stand-in Eigen header reduce in that published order.  Applies to every distance on the path
 *              (training, scoring, evaluate, batch-map MSE) and to euclidianWeightedDistRaw's dot (U-matrix). */
typedef enum vsom_reduction_order
{
    VSOM_ORDER_REFERENCE = 0,
    VSOM_ORDER_LANES = 1,
    VSOM_ORDER_EIGEN_SSE = 2
} vsom_reduction_order;

/* -------------------------------------------------------------------------------- context / state */

/* Som::Som(width, height, depth, transformation) + Som::Construct (include/SOM.hpp:83-87, src/Som.cpp:11-48):
 * all planes zero.  `device` is a CUDA ordinal. */
VSOM_API int vsom_create(vsom_ctx **out, int device, int width, int height, int d_in, int transform, int order);
VSOM_API void vsom_destroy(vsom_ctx *ctx);
/* Node-sharded training of a large map across the GPUs of one NVLink box (BASELINE config 5).  Grid rows are dealt to the
 * ranks round-robin in blocks of a few rows (vsom_shard_rows; block b of 4 rows -> rank b % world), so that every update
 * window — and the U-matrix — spreads over all GPUs.  Every rank calls vsom_train_chunk[_device] with the SAME samples;
 * inside the persistent kernel each GPU scans its rows, CTA 0 pushes the GPU-local (distance, node) key into every rank's
 * memory over NVLink (peer-mapped pointers, system-scope stores) and every CTA takes the min of the `world` keys — one
 * 8-byte exchange per sample, no host round trip, no NCCL call on the data path.
 * Setup, one process per GPU: each rank exports two handles — its exchange slots (vsom_peer_export) and its mean plane
 * (vsom_peer_export_planes, read by the neighbours for the U-matrix halo); the caller all-gathers them (e.g.
 * torch.distributed) and imports them (vsom_peer_import, vsom_peer_import_planes) before the first chunk.  Several ranks
 * inside ONE process (a thread per GPU) attach each other directly with vsom_peer_attach.
 * upload / download / vsom_update_umatrix take FULL-map arrays and touch only the rank's own grid rows.
 * vsom_update_umatrix on a sharded context is a collective in the caller's hands: every rank's training stream must be
 * idle before any rank calls it (the kernel reads one border row of means per neighbouring block straight out of the owners'
 * planes over NVLink peer memory — no staging copy),
 * and no rank may train again before every rank has returned.  Scoring and index entry points need an unsharded context;
 * the findLocalBmu regime (sigma <= 1) is not available on sharded contexts. */
VSOM_API int vsom_create_sharded(vsom_ctx **out, int device, int width, int height, int d_in, int transform, int order, int rank, int world);
VSOM_API int vsom_peer_export(vsom_ctx *ctx, unsigned char handle[64]);
VSOM_API int vsom_peer_import(vsom_ctx *ctx, int rank, const unsigned char handle[64]);
VSOM_API int vsom_peer_export_planes(vsom_ctx *ctx, unsigned char handle[64]);
VSOM_API int vsom_peer_import_planes(vsom_ctx *ctx, int rank, const unsigned char handle[64]);
VSOM_API int vsom_peer_attach(vsom_ctx *ctx, int rank, vsom_ctx *peer);
/* Layout of this rank's share: rows per block, number of local rows, and (global_rows, may be NULL, local_rows entries)
 * the grid row of every local row in local order.  Unsharded: one block of all `height` rows. */
VSOM_API int vsom_shard_rows(const vsom_ctx *ctx, int *block_rows, int *local_rows, int *global_rows);
/* Text of the last error on ctx (or of the last failed vsom_create when ctx is NULL). */
VSOM_API const char *vsom_last_error(const vsom_ctx *ctx);
/* Transformation::Length (src/Transformation.cpp:31-35, :69-73, :162-165). */
VSOM_API int vsom_model_length(int d_in, int transform);
VSOM_API int vsom_depth(const vsom_ctx *ctx);      /* Som::getDepth  (src/Som.cpp:184-187) */
VSOM_API int vsom_node_count(const vsom_ctx *ctx); /* width*height */
/* cudaStream_t of the context, as void*: callers timing with CUDA events record on this stream. */
VSOM_API void *vsom_stream(const vsom_ctx *ctx);
VSOM_API int vsom_synchronize(vsom_ctx *ctx);
/* Number of kernels this library has launched on ctx since creation (bench.py's gpu_launches). */
VSOM_API uint64_t vsom_launch_count(const vsom_ctx *ctx);
/* 1 when the online step keeps the three planes resident in shared memory for this map, else 0. */
VSOM_API int vsom_planes_resident(const vsom_ctx *ctx);

/* Diagnostics of the online step (K1): when enabled, thread 0 of every CTA accumulates clock64() deltas of the
 * five phases of each sample (wait-for-sample, scan + CTA min, grid-wide min-loc exchange, broadcast barrier,
 * window update); vsom_debug_phase_cycles returns their mean over CTAs in cycles per sample for the last chunk. */
VSOM_API int vsom_debug_profile(vsom_ctx *ctx, int enable);
/* Which kernel the last vsom_train_chunk[_device] call ran: 1 = K1F (online_step_fast.cu), 0 = the generic online-step
 * kernel.  K1F runs chunks of fewer than 2^32 - 1 samples on one GPU in the reference and Eigen orders, for every
 * transformation and both sigma regimes, when the map fits on chip (grid sides <= 4096, at most 512 nodes per CTA, planes
 * in shared memory).  The environment variable VSOM_ONLINE_KERNEL=generic, read by vsom_create, keeps a context on the
 * generic kernel (A/B measurements). */
VSOM_API int vsom_debug_last_train_fast(const vsom_ctx *ctx);
VSOM_API int vsom_debug_phase_cycles(vsom_ctx *ctx, double out[5]);
/* The unfolded slots of the last launch.  K1F: chain, CTA min, exchange, coefficients, barrier, update, barrier, 0;
 * generic kernel: the five phases above, then zeros. */
VSOM_API int vsom_debug_phase_cycles_raw(vsom_ctx *ctx, double out[8]);
/* 1 when K1F's exchange rows were placed by L2 die (the SM -> die and block -> die maps were measured and are clean). */
VSOM_API int vsom_debug_die_aware(const vsom_ctx *ctx);

/* Measured on-chip bandwidth of this device (not a product path; bench.py's roofline denominators for maps that stay on
 * chip): out[0] = aggregate shared-memory read bandwidth (GB/s, conflict-free LDS.128 on every SM), out[1] = the same per SM,
 * out[2] = L2 read bandwidth (GB/s, every SM reading one L2-resident buffer with L2-only 128-bit loads), out[3] = size of
 * that buffer in MiB. */
VSOM_API int vsom_debug_measure_peaks(vsom_ctx *ctx, double out[4]);

/* Replace / read the model state: Som::map, SMap, sigmaMap, weightMap, bmuHits (include/SOM.hpp:56-61).
 * Any pointer may be NULL (skipped).  Initial planes come from the host (Som::randomInitialize,
 * src/Som.cpp:977-997, runs on the host so that glibc's rand() sequence is the reference's). */
VSOM_API int vsom_upload_state(vsom_ctx *ctx, const float *mean, const float *S, const float *sigma, const float *weight, const uint64_t *hits);
VSOM_API int vsom_download_state(vsom_ctx *ctx, float *mean, float *S, float *sigma, float *weight, uint64_t *hits);

/* Linear initialisation (not in the reference; SOM_PAK lininit / SOM Toolbox som_lininit): the map's mean plane spans the
 * plane of the data's two leading principal components.  Standard and Median contexts (D = d_in = Dm).
 *   1. mu = (1/n) sum_r x_r and C = (1/(n-1)) sum_r (x_r - mu)(x_r - mu)^T, both in f64.
 *   2. lambda_1 >= lambda_2: the two largest eigenvalues of C, each clamped at 0; v_1, v_2 orthonormal eigenvectors for them, each
 *      signed so that its component of largest magnitude is positive (the lowest index among equal magnitudes).  D = 1: v_1 = [1],
 *      lambda_2 = 0, v_2 = 0.
 *   3. The first axis runs along the longer side of the grid: with W >= H, x goes with (lambda_1, v_1) and y with (lambda_2, v_2);
 *      otherwise the two are swapped.  Grid coordinate c_L(i) = (2i - (L-1)) / (L-1) for L >= 2, c_1(0) = 0.
 *   4. m[y*W + x][k] = f32( (mu_k + (c_W(x) * s_x) * v_x[k]) + (c_H(y) * s_y) * v_y[k] ), s = sqrt(lambda), evaluated in f64 with
 *      round-to-nearest in exactly that order and rounded to f32 once (so the plane can be recomputed bit for bit from the call's own
 *      out_mean, out_lambda and out_axes).
 *   5. S, sigma, weight and hits are set to 0 (the state Som::randomInitialize leaves).
 * The bits depend only on the rows: not on the device, the summation order, Standard vs Median, or node sharding.  On node-sharded
 * contexts every rank calls with the same rows and writes only its own grid rows (no communication).
 * Method: one f64 pass over the rows shifted by the first row (host rows stream in slabs of VSOM_LINEAR_INIT_SLAB_ROWS rows), then
 * subspace iteration on min(D, 8) vectors until |C v_i - lambda_i v_i| <= 1e-11 lambda_1 for i = 1, 2, or 300 iterations.  When the
 * cap ends it (lambda_1, lambda_2, lambda_3 nearly equal: the data does not determine the axes) the call still succeeds with the Ritz
 * pairs it has.
 * x: n x d_in host rows (pageable or pinned).  out_mean[D], out_lambda[2], out_axes[2*D] (axis 1, then axis 2); each may be NULL.
 * Errors: n < 2 or a non-finite element -> VSOM_ERR_INVALID; a CLR context -> VSOM_ERR_UNSUPPORTED (its model vector holds regression
 * coefficients, not a point in data space).  A refused call leaves the state unchanged. */
#define VSOM_LINEAR_INIT_SLAB_ROWS 16384
VSOM_API int vsom_linear_init(vsom_ctx *ctx, const float *x, size_t n, double *out_mean, double *out_lambda, double *out_axes);
/* Host wall time of the three phases of the last vsom_linear_init on ctx (ms): out[0] co-moment pass (including the copies of the
 * rows), out[1] eigen step, out[2] fill; out[3] subspace iterations. */
VSOM_API int vsom_debug_linear_init_phases(const vsom_ctx *ctx, double out[4]);

/* Clustering of the map's nodes (not in the reference; SOM Toolbox som_kmeans / kmeans_clusters after Vesanto & Alhoniemi (2000),
 * somoclu's Somoclu.cluster): k-means++ seeding, then Lloyd iterations, over the N rows of the mean plane (Dm floats each; on a CLR
 * context the regression coefficients, so the call clusters the regression models).  Read-only: the planes, hits and U-matrix are
 * unchanged afterwards.  Weights: w_p = 1 under VSOM_CLUSTER_UNIFORM, (double)hits[p] under VSOM_CLUSTER_HITS.
 *   Distance: d(p, c) = sum_k (m_p[k] - c[k])^2 in f32 in the context's summation order (a LANES context sums in the REFERENCE
 *     order, as every path but the online step does), c = the f32 rounding (RN) of the f64 centroid: the bits vsom_find_bmu_exact
 *     returns for the row m_p on a Standard context of k nodes whose mean plane holds those f32 centroids.
 *   Seeding: splitmix64 with state = seed (state += 0x9E3779B97F4A7C15; z = state; z = (z ^ z>>30) * 0xBF58476D1CE4E5B9;
 *     z = (z ^ z>>27) * 0x94D049BB133111EB; draw z ^ z>>31).  Pick j = 0 .. k-1 takes one draw, u_j = (draw >> 11) * 2^-53.  Pick
 *     weights: q_p = w_p for pick 0, q_p = w_p * D_p (f64) after, D_p = (double) min over the earlier centroids i of d(p, c_i).
 *     T_b = sequential f64 sum of q over nodes [VSOM_CLUSTER_BLOCK b, VSOM_CLUSTER_BLOCK (b + 1)) in node order; total = sequential
 *     sum of the T_b; target = u_j * total.  The block: the first b whose running sum over blocks (running + T_b) exceeds the target,
 *     else the last block with T_b > 0.  The node: inside it, from the sum of the earlier blocks, add q_p in node order and take the
 *     first p whose sum exceeds the target, else the last p with q_p > 0.  Centroid j = that row, exact in f64.  A total of 0 (fewer
 *     than k distinct nodes carry weight; under HITS a map that has seen no data) or one that is not finite -> VSOM_ERR_INVALID.
 *   Lloyd, i = 1 .. max_iter: (1) label(p) = the j with the smallest (d(p, c_j), j).  (2) Stop when i > 1 and no label changed
 *     (converged = 1), else when i = max_iter (converged = 0).  (3) Update: c_j[k] = (sum of w_p * (double)m_p[k]) / W_j,
 *     W_j = sum of w_p, over the members in ascending node order, in consecutive groups of VSOM_CLUSTER_BLOCK members, each group
 *     summed sequentially from 0 and the group sums added sequentially from 0; one f64 division.  A cluster with W_j = 0 keeps its
 *     centroid.  Stopping before the update keeps the outputs consistent: the labels are the assignment to the returned centroids.
 *   Outputs (each may be NULL): out_label[N], out_centroids[k * Dm] (f64), out_weight[k] = W_j of the final labels, out_inertia =
 *     sum_p w_p * (double)d(p, c_label(p)) in the seeding's block order, out_iterations = the number of assignments, out_converged.
 * Errors (no output written, no state changed): k < 1, k > N, max_iter < 1, an unknown weighting or a NaN / infinite element of the
 * mean plane -> VSOM_ERR_INVALID; a node-sharded context -> VSOM_ERR_UNSUPPORTED.
 * Device work: the seeding streams the plane once per pick with the block sums and the pick on the device; the assignment is the exact
 * scan (K3) with the centroids as its map; the update groups the members with the index build (K5). */
#define VSOM_CLUSTER_BLOCK 1024
typedef enum vsom_cluster_weighting
{
    VSOM_CLUSTER_UNIFORM = 0,
    VSOM_CLUSTER_HITS = 1
} vsom_cluster_weighting;
VSOM_API int vsom_cluster_nodes(vsom_ctx *ctx, int k, uint64_t seed, int weighting, int max_iter, int32_t *out_label, double *out_centroids, double *out_weight,
                                double *out_inertia, int *out_iterations, int *out_converged);
/* Device time (CUDA events on the context's stream, ms) of the phases of the last successful vsom_cluster_nodes on ctx: out[0] the
 * seeding (the plane check included), out[1] all assignments, out[2] all updates, out[3] the outputs (the weights of the final
 * labels and the inertia); out[4] the number of assignments (updates: one fewer). */
VSOM_API int vsom_debug_cluster_phases(const vsom_ctx *ctx, double out[5]);

/* One node's rows: Som::getNeuron / Som::getSigmaNeuron (src/Som.cpp:194-212).  Either output may be NULL. */
VSOM_API int vsom_get_node(vsom_ctx *ctx, size_t node, float *mean, float *sigma);

/* -------------------------------------------------------------------------------- online training */

/* n consecutive Som::trainSingle + Som::addBmu calls at fixed (eta, sigma): the inner loop of
 * Som::trainBasicSom (src/Som.cpp:1161-1171; trainSingle :885-947, findBmu :291-309,
 * euclidianWeightedDist :124-141, calculateNeighbourhoodWeight :949-975, addBmu :1189-1192), in row order.
 *   x          n x d_in, row-major
 *   last_bmu   in/out per row like DataSet::getLastBMU(j) (src/DataSet.cpp:60-69); may be NULL (= zeros).
 *              Read only when sigma <= 1 (findLocalBmu regime, src/Som.cpp:335-454); always written.
 *   out_bmu    linear BMU index per row; out_dist = (float)dist(bmu) on the updated map (:946);
 *   out_resid2 = residual.squaredNorm() (the term of src/Som.cpp:1167).  Each may be NULL. */
VSOM_API int vsom_train_chunk(vsom_ctx *ctx, const float *x, size_t n, double eta, double sigma, int decay, uint64_t *last_bmu,
                     uint32_t *out_bmu, float *out_dist, float *out_resid2);
/* Same with x / outputs in device memory; enqueue only.  With sigma <= 1 every row's local walk starts at node 0, which is
 * what DataSet gives the reference too (lastBMU is zeroed at every chunk load, src/DataSet.cpp:136-137). */
VSOM_API int vsom_train_chunk_device(vsom_ctx *ctx, const float *x_dev, size_t n, double eta, double sigma, int decay,
                            uint32_t *out_bmu_dev, float *out_dist_dev);

/* One chunk-epoch of the batch-map trainer: Som::trainBatchSomEpoch (src/Som.cpp:756-879).  Phase A finds every row's BMU
 * (is_first != 0: global search; else the local walk from last_bmu[row]), counts the hits and returns the mean squared
 * residual in *out_mse; phase B replaces every neuron by the incrementally weighted mean of all rows of the chunk (and its
 * sigma and weight).  last_bmu is in/out per row; x is n x d_in row-major on the host.
 * Limits: Standard / Median need Dm <= 5888; CLR needs P = d_in (d_in - 1) / 2 <= 2944 (d_in <= 77); rows of up to 6400
 * values fit phase B's shared-memory row buffers.  A call past a limit returns VSOM_ERR_UNSUPPORTED and changes nothing: not
 * the map, its hit counts or last_bmu.  Afterwards vsom_debug_last_score_tc reports phase A's search: K2's tier when a first
 * epoch ran the tensor-core search (>= 1024 rows on a shape K2 covers), 0 for the exact scan and for the local walks. */
VSOM_API int vsom_batch_epoch(vsom_ctx *ctx, const float *x, size_t n, double sigma, int is_first, uint64_t *last_bmu, float *out_mse);

/* -------------------------------------------------------------------------------- scoring */

/* Per row: Som::findBmu (min_hits == 0, src/Som.cpp:291-309) or Som::findRestrictedBmu (src/Som.cpp:313-332),
 * and out_dist = (float)euclidianWeightedDist(bmu, row) (src/Som.cpp:124-141).  Outputs may be NULL.
 * This is the call behind Som::evaluate (:490-523), Som::measureSimilarity (:631-714) and Som::mapDataSet.
 * Dispatch: batches of >= 1024 rows on shapes K2 covers (Standard / Median, Dm <= 2048) run the tensor-core candidate
 * search (tcgen05 + TMA, fp16 operands with exact power-of-two scaling; one value per element, or hi / lo pairs when a probe
 * of the first rows shows the map needs the precision) + exact f32 rescore of the <= 48 listed candidates per row + a
 * certificate that no unlisted node can win; rows that fail it are re-scored by the exact scan.  Everything else runs the
 * exact scan.
 * Results are bit-identical either way.  The host-pointer form streams the rows through three staging buffers (H2D of the
 * next slab overlaps the search of the current one; pinned host memory gives full overlap). */
VSOM_API int vsom_find_bmu(vsom_ctx *ctx, const float *x, size_t n, uint64_t min_hits, uint32_t *out_bmu, float *out_dist);
VSOM_API int vsom_find_bmu_device(vsom_ctx *ctx, const float *x_dev, size_t n, uint64_t min_hits, uint32_t *out_bmu_dev, float *out_dist_dev);
/* Same contract, always the exact scan (K3) — what the tests compare the dispatching calls with. */
VSOM_API int vsom_find_bmu_exact(vsom_ctx *ctx, const float *x, size_t n, uint64_t min_hits, uint32_t *out_bmu, float *out_dist);
VSOM_API int vsom_find_bmu_exact_device(vsom_ctx *ctx, const float *x_dev, size_t n, uint64_t min_hits, uint32_t *out_bmu_dev, float *out_dist_dev);
/* Prediction of unobserved columns (not in the reference; SOM Toolbox som_fillnans, kohonen predict(whatmap=)).
 * match[Dm]: 1 = the column is observed and is matched, 0 = the column is predicted; any other value -> VSOM_ERR_INVALID.
 * S = the matched columns in ascending order (|S| >= 1), Q = the predicted ones in ascending order (q = Dm - |S| >= 0).
 * Per row r of x (n x d_in, full width; the columns in Q are never read and may hold anything, NaN included):
 *   out_bmu[r], out_dist[r]: exactly what vsom_find_bmu_exact returns, with the same min_hits, on a Standard context of the
 *     same grid and summation order whose mean plane is the columns S of this map, for the row x[r][S].  That is
 *     d_S(p) = sum over j of (m_p[S_j] - x_r[S_j])^2 in f32 in the context's order over the compacted sequence (a LANES
 *     context sums in the REFERENCE order, as every path but the online step does).  It inherits findRestrictedBmu's
 *     eligibility (hits >= min_hits, node 0 always) and the NaN-at-node-0 rule.
 *   out_mean[r*q + j] = mean[out_bmu[r]][Q_j], out_sigma[r*q + j] = sigma[out_bmu[r]][Q_j] (copies of the plane's f32 bits).
 * Every output may be NULL.  |S| = Dm gives vsom_find_bmu's bits.  Read-only: planes, hits and U-matrix are unchanged.
 * Errors (nothing written): match NULL, no matched column, a value other than 0 / 1 -> VSOM_ERR_INVALID; a CLR context
 * (its model vector holds regression coefficients, not data columns) or a node-sharded one -> VSOM_ERR_UNSUPPORTED.
 * Dispatch as vsom_find_bmu, over the compacted operands: >= 1024 rows with |S| <= 2048 run K2 (tiers, probes, exact
 * rescore, certificate, exact scan of the rows it leaves); everything else runs K3.  vsom_debug_last_score_tc / _pair /
 * _tc_stats report these calls like vsom_find_bmu's.  The host form copies full-width rows in vsom_find_bmu's slabs and
 * gathers the columns S on the device; the predictions return per slab through 2 q floats per row of device staging for three
 * slabs (one slab on the exact scan), on a stream of their own.  The device form gathers all n rows once (n x |S| floats of
 * staging).  Staging is grow-only: it is kept until the context is destroyed. */
VSOM_API int vsom_predict_columns(vsom_ctx *ctx, const float *x, size_t n, const uint8_t *match, uint64_t min_hits,
                                  uint32_t *out_bmu, float *out_dist, float *out_mean, float *out_sigma);
VSOM_API int vsom_predict_columns_device(vsom_ctx *ctx, const float *x_dev, size_t n, const uint8_t *match /* host */, uint64_t min_hits,
                                         uint32_t *out_bmu_dev, float *out_dist_dev, float *out_mean_dev, float *out_sigma_dev);
/* vsom_find_bmu[_device] that also reports how many rows took the exact full scan (fallback_rows, may be NULL; = n when
 * the whole batch ran on the exact scan). */
VSOM_API int vsom_find_bmu_batch(vsom_ctx *ctx, const float *x, size_t n, uint64_t min_hits, uint32_t *out_bmu, float *out_dist, uint64_t *fallback_rows);
VSOM_API int vsom_find_bmu_batch_device(vsom_ctx *ctx, const float *x_dev, size_t n, uint64_t min_hits, uint32_t *out_bmu_dev, float *out_dist_dev,
                                        uint64_t *fallback_rows);
/* Best AND second-best matching node of every row — what the topographic error needs.  out_bmu / out_dist are exactly what
 * vsom_find_bmu returns for the same rows and min_hits (the NaN-at-node-0 rule included).  out_bmu2 / out_dist2: the eligible
 * node (hits >= min_hits, or node 0) other than out_bmu with the smallest (distance, index) key — a smaller distance wins,
 * equal distances go to the lower index, a NaN distance ranks after every number (lower index first among NaNs).  A row
 * without such a node (one node, or one eligible node) gets out_bmu2 = 0xFFFFFFFF and a NaN out_dist2.  Every output may be
 * NULL; fallback_rows (may be NULL) as in vsom_find_bmu_batch.
 * Topographic error of n rows: the share of rows whose out_bmu and out_bmu2 are not 8-neighbours on the rectangular,
 * non-wrapping grid (max(|dx|, |dy|) == 1, diagonals included: the U-matrix's neighbourhood); rows without a runner-up are
 * not errors.  Som::topographicError (include/SOM.hpp) computes it from these outputs.
 * Dispatch and tiers as vsom_find_bmu: >= 1024 rows on a shape K2 covers run the tensor-core search in its top-2 mode (the list
 * threshold follows an upper bound of the second-smallest approximate score, and the certificate must clear the runner-up's
 * exact distance), everything else the exact scan.  vsom_debug_last_score_tc / _pair / _tc_stats report these calls like
 * vsom_find_bmu's.  Node-sharded contexts return VSOM_ERR_UNSUPPORTED. */
VSOM_API int vsom_find_bmu2(vsom_ctx *ctx, const float *x, size_t n, uint64_t min_hits, uint32_t *out_bmu, float *out_dist, uint32_t *out_bmu2,
                            float *out_dist2, uint64_t *fallback_rows);
VSOM_API int vsom_find_bmu2_device(vsom_ctx *ctx, const float *x_dev, size_t n, uint64_t min_hits, uint32_t *out_bmu_dev, float *out_dist_dev,
                                   uint32_t *out_bmu2_dev, float *out_dist2_dev, uint64_t *fallback_rows);
/* Same contract, always the exact scan (K3) — what the tests compare the dispatching calls with. */
VSOM_API int vsom_find_bmu2_exact(vsom_ctx *ctx, const float *x, size_t n, uint64_t min_hits, uint32_t *out_bmu, float *out_dist, uint32_t *out_bmu2,
                                  float *out_dist2);
/* 0 when the last scoring call on ctx ran the exact scan, else the precision tier of its tensor-core search: 1 = one fp16
 * value per operand element, 2 = hi / lo pairs (three products per element; chosen when a probe of the first rows shows that
 * tier 1 cannot separate the BMU from its neighbours on this map), 3 = both probes (8192 rows each, whose results stand)
 * left more than a quarter of their rows uncertified and the remainder went to the exact scan. */
VSOM_API int vsom_debug_last_score_tc(const vsom_ctx *ctx);
/* 1 when that search ran as CTA pairs (tcgen05 cta_group::2, the default wherever the device can co-schedule clusters of two),
 * 0 for the single-CTA kernel (VSOM_TC_PAIR=0, or a device partition without whole TPCs). */
VSOM_API int vsom_debug_last_score_pair(const vsom_ctx *ctx);
/* Why rows of the tensor-core path went to the exact scan, counted since vsom_create: out[0] candidate list overflowed (more
 * than 48 nodes inside the margin), out[1] NaN distance / no eligible candidate, out[2] the certificate could not exclude an
 * unlisted node. */
VSOM_API int vsom_debug_tc_stats(const vsom_ctx *ctx, uint64_t out[3]);

/* Som::evaluate for all-continuous columns (src/Som.cpp:490-523): f64 running mean of the BMU distance in row
 * order.  (With binary columns the reference adds a cross-entropy term; that is host work on top of the
 * BMU indices this call family returns.) */
VSOM_API int vsom_evaluate(vsom_ctx *ctx, const float *x, size_t n, double *mean_error);
/* The per-row pass of Som::measureSimilarity (src/Som.cpp:631-714) for n host rows in ONE trip over PCIe: every row's restricted
 * BMU (as vsom_find_bmu, out_bmu may be NULL) and out_row_max[i] = max over the columns of ((x - m_bmu) / sM) / number_of_sigmas
 * with the reference's capped sigma sM (:648) and its three f32 operations; NaN deltas never win (the reference compares with
 * `>`), -inf when a row has none.  The reference's running maximum over all rows and columns is, after its first update, the
 * running maximum of these values in row order, which is how Som::measureSimilarity (host/Som.cpp) finds the row it judges.
 * Needs a Standard / Median context (model vector as long as the rows). */
VSOM_API int vsom_measure_similarity(vsom_ctx *ctx, const float *x, size_t n, uint64_t min_hits, int number_of_sigmas, uint32_t *out_bmu, float *out_row_max);
/* Distance of one row to every node: N x euclidianWeightedDist (src/Som.cpp:124-141), as the double it returns. */
VSOM_API int vsom_all_dists(vsom_ctx *ctx, const float *v, double *out);

/* Soft assignment of a batch of rows: Som::findRestrictedBmd (src/Som.cpp:457-487) per row — out_prob[r*N + i] =
 * exp(-d_i^2 / 2) / C for nodes with hits >= min_hits (d_i = the already squared distance, as the reference has it), 0 for
 * the others; C sums the terms in node order.  What Som::variationalAutoEncoder / autoEncoder (:525-623) sample from
 * (the sampling itself stays on the host: std::discrete_distribution over these probabilities).  Distances are the
 * reference's bits; exp() is the device's f64 exp, so probabilities agree with the reference to a few ulp (1e-14 relative). */
VSOM_API int vsom_soft_assign(vsom_ctx *ctx, const float *x, size_t n, uint64_t min_hits, double *out_prob);

/* -------------------------------------------------------------------------------- U-matrix / index */

/* Som::updateUMatrix + Som::getUMatrix (src/Som.cpp:999-1111, :159-162; euclidianWeightedDistRaw :143-157).
 * out: N doubles, may be NULL (the matrix is kept on the device either way).  Needs width, height >= 2.
 * Node-sharded contexts compute their own grid rows (halo rows come from the neighbouring ranks, see vsom_create_sharded). */
VSOM_API int vsom_update_umatrix(vsom_ctx *ctx, double *out);
/* "SomIndex build": histogram of BMU ids (what Som::addBmu accumulates, src/Som.cpp:1189-1192) and the rows
 * grouped by BMU in ascending row order (the per-neuron row set of src/Som.cpp:845-868).
 * counts[N], offsets[N+1], row_ids[n]; each may be NULL. */
VSOM_API int vsom_build_index(vsom_ctx *ctx, const uint32_t *bmu, size_t n, uint64_t *counts, uint64_t *offsets, uint32_t *row_ids);
/* Same on device arrays (enqueue only; an out-of-range BMU id raises the context's error flag, reported by the host form). */
VSOM_API int vsom_build_index_device(vsom_ctx *ctx, const uint32_t *bmu_dev, size_t n, uint64_t *counts_dev, uint64_t *offsets_dev, uint32_t *row_ids_dev);

#ifdef __cplusplus
}
#endif
#endif /* VSOM_B200_H */
