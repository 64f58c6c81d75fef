// capi.cu — the extern "C" surface of libvsom_b200.so (include/vsom_b200.h): context, state transfer and the
// host-buffer entry points that stage data through the context's stream around the kernel launchers.
#include "common.cuh"

#include <cstdlib>

#include <algorithm>
#include <cstdio>
#include <cstring>

namespace vsom
{

static std::string g_createError;

int set_error(vsom_ctx *ctx, int code, const std::string &msg)
{
    if (ctx)
        ctx->err = msg;
    else
        g_createError = msg;
    return code;
}

int cuda_fail(vsom_ctx *ctx, cudaError_t e, const char *what, const char *file, int line)
{
    char buf[512];
    std::snprintf(buf, sizeof(buf), "%s failed: %s (%s:%d)", what, cudaGetErrorString(e), file, line);
    return set_error(ctx, VSOM_ERR_CUDA, buf);
}

int stage_reserve(vsom_ctx *ctx, int slot, size_t bytes)
{
    if (bytes <= ctx->stageCap[slot])
        return VSOM_OK;
    if (ctx->stage[slot])
    {
        VSOM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        VSOM_CUDA(ctx, cudaFree(ctx->stage[slot]));
        ctx->stage[slot] = nullptr;
        ctx->stageCap[slot] = 0;
    }
    const size_t cap = bytes + bytes / 4 + 256;
    VSOM_CUDA(ctx, cudaMalloc(&ctx->stage[slot], cap));
    ctx->stageCap[slot] = cap;
    return VSOM_OK;
}

static int check_error_flag(vsom_ctx *ctx, const char *what)
{
    int flag = 0;
    VSOM_CUDA(ctx, cudaMemcpyAsync(&flag, ctx->errFlag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    VSOM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (flag)
    {
        ctx->poisoned = true; // only the online step raises the flag through this path (vsom_build_index re-maps it and clears this)
        return set_error(ctx, VSOM_ERR_TIMEOUT, std::string(what) + ": device reported an error flag");
    }
    return VSOM_OK;
}

} // namespace vsom

using namespace vsom;

extern "C"
{

int vsom_model_length(int d_in, int transform) { return transform == VSOM_CLR ? d_in * (d_in - 1) : d_in; }

static int create_impl(vsom_ctx **out, int device, int width, int height, int d_in, int transform, int order, int rank, int world)
{
    if (!out)
        return set_error(nullptr, VSOM_ERR_INVALID, "vsom_create: out is NULL");
    *out = nullptr;
    if (width < 1 || height < 1 || d_in < 1 || transform < VSOM_STANDARD || transform > VSOM_CLR || order < VSOM_ORDER_REFERENCE ||
        order > VSOM_ORDER_EIGEN_SSE || (transform == VSOM_CLR && d_in < 2))
        return set_error(nullptr, VSOM_ERR_INVALID, "vsom_create: bad width/height/d_in/transform/order");
    if (static_cast<long long>(width) * height >= (1ll << 24))
        return set_error(nullptr, VSOM_ERR_INVALID, "vsom_create: at most 2^24 - 1 nodes");
    if (transform == VSOM_CLR && d_in > 65535)
        return set_error(nullptr, VSOM_ERR_INVALID, "vsom_create: CLR pair tables are 16-bit");
    if (world < 1 || world > 8 || rank < 0 || rank >= world || world > height)
        return set_error(nullptr, VSOM_ERR_INVALID, "vsom_create_sharded: need 1 <= world <= 8, 0 <= rank < world, world <= height");
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count < 1 || device < 0 || device >= count)
    {
        char buf[256];
        std::snprintf(buf, sizeof(buf), "vsom_create: no usable CUDA device %d (%s; %d visible). This library has no CPU path.", device,
                      e == cudaSuccess ? "ok" : cudaGetErrorString(e), count);
        return set_error(nullptr, VSOM_ERR_NO_DEVICE, buf);
    }
    vsom_ctx *ctx = new vsom_ctx();
    ctx->device = device;
    ctx->W = width;
    ctx->H = height;
    ctx->N = width * height;
    ctx->Din = d_in;
    ctx->transform = transform;
    ctx->order = order;
    ctx->Dm = vsom_model_length(d_in, transform);
    ctx->P = transform == VSOM_CLR ? ctx->Dm / 2 : 0;
    ctx->Dr = transform == VSOM_CLR ? ctx->P : ctx->Dm;
    ctx->rowStride = (ctx->Dm + 3) & ~3;
    ctx->rank = rank;
    ctx->world = world;
    {
        // Node sharding: grid rows are dealt to the ranks round-robin in blocks of shardBlock rows (block b -> rank b % world).
        // Contiguous bands (SURVEY.md §8e's first proposal) put a whole update window (80 x 80 nodes at sigma = 16 on a
        // 512 x 512 map) on one or two GPUs; small blocks spread it over all of them, at the price of more U-matrix halo rows.
        int block = world == 1 ? height : 4;
        if (world > 1 && block * world > height)
            block = height / world; // every rank holds at least one row (world <= height was checked above)
        ctx->shardBlock = block;
        for (int y = 0; y < height; ++y)
            if ((y / block) % world == rank)
                ctx->localRowY.push_back(y);
        ctx->localRows = static_cast<int>(ctx->localRowY.size());
        ctx->node0 = 0;
        ctx->localN = ctx->localRows * width;
    }

    auto fail = [&](int rc) {
        g_createError = ctx->err;
        vsom_destroy(ctx);
        return rc;
    };
#define CREATE_CUDA(call)                                                                  \
    do                                                                                     \
    {                                                                                      \
        cudaError_t _e = (call);                                                           \
        if (_e != cudaSuccess)                                                             \
            return fail(cuda_fail(ctx, _e, #call, __FILE__, __LINE__));                    \
    } while (0)

    CREATE_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    CREATE_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
    {
        ctx->err = "vsom_create: this library is built for sm_100a (B200) only; device is sm_" + std::to_string(prop.major) + std::to_string(prop.minor);
        return fail(VSOM_ERR_NO_DEVICE);
    }
    ctx->numSMs = prop.multiProcessorCount;
    {
        // diagnostics / A-B measurements: VSOM_ONLINE_KERNEL=generic keeps every online step on the generic kernel
        const char *e = getenv("VSOM_ONLINE_KERNEL");
        ctx->fastDisabled = (e && std::string(e) == "generic") ? 1 : 0;
    }
    ctx->smemOptin = static_cast<int>(prop.sharedMemPerBlockOptin);
    CREATE_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    const size_t plane = sizeof(float) * static_cast<size_t>(ctx->localN) * ctx->rowStride;
    // the mean plane carries a tail of zero rows: the streamed scan's TMA descriptor (online_step.cu) addresses rows as
    // (owner CTA, owned-row index) and its last index may reach up to one grid of rows past the map
    const size_t meanTail = sizeof(float) * 160 * static_cast<size_t>(ctx->rowStride);
    CREATE_CUDA(cudaMalloc(&ctx->mean, plane + meanTail));
    CREATE_CUDA(cudaMemsetAsync(reinterpret_cast<char *>(ctx->mean) + plane, 0, meanTail, ctx->stream));
    CREATE_CUDA(cudaMalloc(&ctx->S, plane));
    CREATE_CUDA(cudaMalloc(&ctx->sigma, plane));
    CREATE_CUDA(cudaMalloc(&ctx->weight, sizeof(float) * ctx->localN));
    CREATE_CUDA(cudaMalloc(&ctx->hits, sizeof(u64) * ctx->localN));
    CREATE_CUDA(cudaMalloc(&ctx->rankSlots, sizeof(u64) * 2 * 8));
    CREATE_CUDA(cudaMemsetAsync(ctx->rankSlots, 0xff, sizeof(u64) * 2 * 8, ctx->stream));
    ctx->peerSlots[rank] = ctx->rankSlots;
    ctx->peerMean[rank] = ctx->mean;
    CREATE_CUDA(cudaMalloc(&ctx->umatrix, sizeof(double) * ctx->N));
    CREATE_CUDA(cudaMalloc(&ctx->slots, sizeof(u64) * 2 * static_cast<size_t>(ctx->numSMs) * ((ctx->numSMs + 15) & ~15)));
    CREATE_CUDA(cudaMalloc(&ctx->errFlag, sizeof(int)));
    CREATE_CUDA(cudaMemsetAsync(ctx->mean, 0, plane, ctx->stream));
    CREATE_CUDA(cudaMemsetAsync(ctx->S, 0, plane, ctx->stream));
    CREATE_CUDA(cudaMemsetAsync(ctx->sigma, 0, plane, ctx->stream));
    CREATE_CUDA(cudaMemsetAsync(ctx->weight, 0, sizeof(float) * ctx->localN, ctx->stream));
    CREATE_CUDA(cudaMemsetAsync(ctx->hits, 0, sizeof(u64) * ctx->localN, ctx->stream));
    CREATE_CUDA(cudaMemsetAsync(ctx->umatrix, 0, sizeof(double) * ctx->N, ctx->stream));
    CREATE_CUDA(cudaMemsetAsync(ctx->errFlag, 0, sizeof(int), ctx->stream));
    if (transform == VSOM_CLR)
    {
        // pairs (i<j) in row-major upper-triangle order: x'_q = v_i, y'_q = v_j (src/Transformation.cpp:94-101)
        std::vector<unsigned short> pi(ctx->P), pj(ctx->P);
        int q = 0;
        for (int i = 0; i < d_in; ++i)
            for (int j = i + 1; j < d_in; ++j)
            {
                pi[q] = static_cast<unsigned short>(i);
                pj[q] = static_cast<unsigned short>(j);
                ++q;
            }
        CREATE_CUDA(cudaMalloc(&ctx->pairI, sizeof(unsigned short) * ctx->P));
        CREATE_CUDA(cudaMalloc(&ctx->pairJ, sizeof(unsigned short) * ctx->P));
        CREATE_CUDA(cudaMemcpy(ctx->pairI, pi.data(), sizeof(unsigned short) * ctx->P, cudaMemcpyHostToDevice));
        CREATE_CUDA(cudaMemcpy(ctx->pairJ, pj.data(), sizeof(unsigned short) * ctx->P, cudaMemcpyHostToDevice));
    }
    int rc = configure_online_step(ctx);
    if (rc)
        return fail(rc);
    CREATE_CUDA(cudaStreamSynchronize(ctx->stream));
#undef CREATE_CUDA
    *out = ctx;
    return VSOM_OK;
}

int vsom_create(vsom_ctx **out, int device, int width, int height, int d_in, int transform, int order)
{
    return create_impl(out, device, width, height, d_in, transform, order, 0, 1);
}

int vsom_create_sharded(vsom_ctx **out, int device, int width, int height, int d_in, int transform, int order, int rank, int world)
{
    return create_impl(out, device, width, height, d_in, transform, order, rank, world);
}

int vsom_peer_export(vsom_ctx *ctx, unsigned char handle[64])
{
    if (!ctx || !handle)
        return VSOM_ERR_INVALID;
    VSOM_CUDA(ctx, cudaSetDevice(ctx->device));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    cudaIpcMemHandle_t h;
    VSOM_CUDA(ctx, cudaIpcGetMemHandle(&h, ctx->rankSlots));
    std::memcpy(handle, &h, 64);
    return VSOM_OK;
}

int vsom_peer_import(vsom_ctx *ctx, int rank, const unsigned char handle[64])
{
    if (!ctx || !handle || rank < 0 || rank >= ctx->world)
        return ctx ? set_error(ctx, VSOM_ERR_INVALID, "vsom_peer_import: bad rank") : VSOM_ERR_INVALID;
    if (rank == ctx->rank)
        return VSOM_OK;
    VSOM_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, 64);
    void *ptr = nullptr;
    VSOM_CUDA(ctx, cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
    ctx->peerSlots[rank] = static_cast<u64 *>(ptr);
    ctx->peerOpened[rank] = true;
    return VSOM_OK;
}

int vsom_peer_export_planes(vsom_ctx *ctx, unsigned char handle[64])
{
    if (!ctx || !handle)
        return VSOM_ERR_INVALID;
    VSOM_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    VSOM_CUDA(ctx, cudaIpcGetMemHandle(&h, ctx->mean));
    std::memcpy(handle, &h, 64);
    return VSOM_OK;
}

int vsom_peer_import_planes(vsom_ctx *ctx, int rank, const unsigned char handle[64])
{
    if (!ctx || !handle || rank < 0 || rank >= ctx->world)
        return ctx ? set_error(ctx, VSOM_ERR_INVALID, "vsom_peer_import_planes: bad rank") : VSOM_ERR_INVALID;
    if (rank == ctx->rank)
        return VSOM_OK;
    VSOM_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, 64);
    void *ptr = nullptr;
    VSOM_CUDA(ctx, cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
    ctx->peerMean[rank] = static_cast<float *>(ptr);
    ctx->peerMeanOpened[rank] = true;
    return VSOM_OK;
}

int vsom_peer_attach(vsom_ctx *ctx, int rank, vsom_ctx *peer)
{
    if (!ctx || !peer || rank < 0 || rank >= ctx->world || peer->rank != rank || peer->world != ctx->world || peer->W != ctx->W || peer->H != ctx->H ||
        peer->Dm != ctx->Dm)
        return ctx ? set_error(ctx, VSOM_ERR_INVALID, "vsom_peer_attach: peer is not rank `rank` of the same sharded map") : VSOM_ERR_INVALID;
    if (rank == ctx->rank)
        return VSOM_OK;
    VSOM_CUDA(ctx, cudaSetDevice(ctx->device));
    if (peer->device != ctx->device)
    {
        int can = 0;
        VSOM_CUDA(ctx, cudaDeviceCanAccessPeer(&can, ctx->device, peer->device));
        if (!can)
            return set_error(ctx, VSOM_ERR_UNSUPPORTED, "vsom_peer_attach: no peer access between the two devices");
        const cudaError_t e = cudaDeviceEnablePeerAccess(peer->device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
            return cuda_fail(ctx, e, "cudaDeviceEnablePeerAccess", __FILE__, __LINE__);
        cudaGetLastError();
    }
    ctx->peerSlots[rank] = peer->rankSlots;
    ctx->peerMean[rank] = peer->mean;
    return VSOM_OK;
}

int vsom_shard_rows(const vsom_ctx *ctx, int *block_rows, int *local_rows, int *global_rows)
{
    if (!ctx)
        return VSOM_ERR_INVALID;
    if (block_rows)
        *block_rows = ctx->shardBlock;
    if (local_rows)
        *local_rows = ctx->localRows;
    if (global_rows)
        for (int i = 0; i < ctx->localRows; ++i)
            global_rows[i] = ctx->localRowY[i];
    return VSOM_OK;
}

void vsom_destroy(vsom_ctx *ctx)
{
    if (!ctx)
        return;
    cudaSetDevice(ctx->device);
    if (ctx->stream)
        cudaStreamSynchronize(ctx->stream);
    cudaFree(ctx->mean);
    cudaFree(ctx->S);
    cudaFree(ctx->sigma);
    cudaFree(ctx->weight);
    cudaFree(ctx->hits);
    cudaFree(ctx->umatrix);
    cudaFree(ctx->pairI);
    cudaFree(ctx->pairJ);
    cudaFree(ctx->slots);
    for (int r = 0; r < 8; ++r)
    {
        if (ctx->peerOpened[r])
            cudaIpcCloseMemHandle(ctx->peerSlots[r]);
        if (ctx->peerMeanOpened[r])
            cudaIpcCloseMemHandle(ctx->peerMean[r]);
    }
    cudaFree(ctx->rankSlots);
    cudaFree(ctx->errFlag);
    cudaFree(ctx->lut);
    cudaFree(ctx->distBuf);
    cudaFree(ctx->winTab);
    cudaFree(ctx->distTag);
    cudaFree(ctx->scanMapDev);
    cudaFree(ctx->rowPool);
    cudaFree(ctx->rowMeta);
    cudaFree(ctx->profDev);
    cudaFree(ctx->umTab);
    for (void *p : ctx->stage)
        cudaFree(p);
    if (ctx->auxStream)
    {
        cudaStreamSynchronize(ctx->auxStream);
        cudaStreamDestroy(ctx->auxStream);
        if (ctx->copyStream)
        {
            cudaStreamSynchronize(ctx->copyStream);
            cudaStreamDestroy(ctx->copyStream);
        }
        for (int i = 0; i < 2; ++i)
        {
            cudaEventDestroy(ctx->evScore[i]);
            cudaEventDestroy(ctx->evDone[i]);
        }
        for (int i = 0; i < 3; ++i)
        {
            cudaEventDestroy(ctx->evCopied[i]);
            cudaEventDestroy(ctx->evSlabDone[i]);
        }
    }
    if (ctx->stream)
        cudaStreamDestroy(ctx->stream);
    delete ctx;
}

const char *vsom_last_error(const vsom_ctx *ctx) { return ctx ? ctx->err.c_str() : g_createError.c_str(); }
int vsom_depth(const vsom_ctx *ctx) { return ctx ? ctx->Dm : 0; }
int vsom_node_count(const vsom_ctx *ctx) { return ctx ? ctx->N : 0; }
void *vsom_stream(const vsom_ctx *ctx) { return ctx ? static_cast<void *>(ctx->stream) : nullptr; }
uint64_t vsom_launch_count(const vsom_ctx *ctx) { return ctx ? ctx->launches : 0; }
int vsom_planes_resident(const vsom_ctx *ctx) { return ctx ? ctx->residentTrain : 0; }

int vsom_debug_last_train_fast(const vsom_ctx *ctx) { return ctx ? ctx->lastTrainFast : 0; }

int vsom_debug_profile(vsom_ctx *ctx, int enable)
{
    if (!ctx)
        return VSOM_ERR_INVALID;
    VSOM_CUDA(ctx, cudaSetDevice(ctx->device));
    VSOM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (enable && !ctx->profDev)
    {
        VSOM_CUDA(ctx, cudaMalloc(&ctx->profDev, sizeof(long long) * 8 * ctx->numSMs));
        VSOM_CUDA(ctx, cudaMemset(ctx->profDev, 0, sizeof(long long) * 8 * ctx->numSMs));
    }
    else if (!enable && ctx->profDev)
    {
        VSOM_CUDA(ctx, cudaFree(ctx->profDev));
        ctx->profDev = nullptr;
    }
    return VSOM_OK;
}

// raw per-phase cycle sums of the last online-step launch, averaged over CTAs, per sample: the generic kernel fills
// 5 slots (stride 5), K1F 7 (stride 8)
static int read_phase_cycles(vsom_ctx *ctx, double raw[8])
{
    if (!ctx->profDev || !ctx->profSamples || !ctx->gridTrain)
        return set_error(ctx, VSOM_ERR_INVALID, "vsom_debug_phase_cycles: profiling not enabled or no chunk trained yet");
    VSOM_CUDA(ctx, cudaSetDevice(ctx->device));
    const int stride = ctx->lastTrainFast ? 8 : 5, grid = ctx->lastTrainFast ? ctx->fastGrid : ctx->gridTrain;
    std::vector<long long> h(static_cast<size_t>(stride) * grid);
    VSOM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    VSOM_CUDA(ctx, cudaMemcpy(h.data(), ctx->profDev, sizeof(long long) * h.size(), cudaMemcpyDeviceToHost));
    for (int i = 0; i < 8; ++i)
    {
        double s = 0;
        for (int b = 0; i < stride && b < grid; ++b)
            s += static_cast<double>(h[static_cast<size_t>(b) * stride + i]);
        raw[i] = s / grid / static_cast<double>(ctx->profSamples);
    }
    return VSOM_OK;
}

int vsom_debug_phase_cycles(vsom_ctx *ctx, double out[5])
{
    if (!ctx || !out)
        return VSOM_ERR_INVALID;
    double raw[8];
    int rc = read_phase_cycles(ctx, raw);
    if (rc)
        return rc;
    if (ctx->lastTrainFast)
    {
        // K1F has no wait-for-sample phase; fold its seven slots into the five documented ones
        out[0] = 0.0;
        out[1] = raw[0] + raw[1]; // FADD chain + CTA min
        out[2] = raw[2];          // grid-wide exchange
        out[3] = raw[3] + raw[4]; // coefficients + barrier
        out[4] = raw[5] + raw[6]; // update (+ next sample's squared residuals) + barrier
    }
    else
        for (int i = 0; i < 5; ++i)
            out[i] = raw[i];
    return VSOM_OK;
}

int vsom_debug_phase_cycles_raw(vsom_ctx *ctx, double out[8])
{
    if (!ctx || !out)
        return VSOM_ERR_INVALID;
    return read_phase_cycles(ctx, out);
}

int vsom_debug_die_aware(const vsom_ctx *ctx) { return ctx ? ctx->dieAware : 0; }

int vsom_synchronize(vsom_ctx *ctx)
{
    if (!ctx)
        return VSOM_ERR_INVALID;
    VSOM_CUDA(ctx, cudaSetDevice(ctx->device));
    VSOM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->trainEnqueued) // a chunk enqueued by vsom_train_chunk_device may have aborted: report it here
    {
        ctx->trainEnqueued = false;
        return check_error_flag(ctx, "vsom_synchronize (after vsom_train_chunk_device)");
    }
    return VSOM_OK;
}

// Planes cross the boundary as FULL-map arrays; a node-sharded context touches only its own blocks of grid rows.
// `toDevice`: host -> device, else device -> host.
static int copy_state(vsom_ctx *ctx, bool toDevice, float *mean, float *S, float *sigma, float *weight, uint64_t *hits)
{
    VSOM_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t w = sizeof(float) * ctx->Dm, pitch = sizeof(float) * ctx->rowStride;
    const cudaMemcpyKind kind = toDevice ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost;
    for (int lr = 0; lr < ctx->localRows;)
    {
        int rows = 1; // run of local rows that are also consecutive grid rows (one block; the whole map when unsharded)
        while (lr + rows < ctx->localRows && ctx->localRowY[lr + rows] == ctx->localRowY[lr] + rows)
            ++rows;
        const size_t nodes = static_cast<size_t>(rows) * ctx->W, lnode = static_cast<size_t>(lr) * ctx->W, gnode = static_cast<size_t>(ctx->localRowY[lr]) * ctx->W;
        float *planesHost[3] = {mean, S, sigma}, *planesDev[3] = {ctx->mean, ctx->S, ctx->sigma};
        for (int k = 0; k < 3; ++k)
            if (planesHost[k])
            {
                float *h = planesHost[k] + gnode * ctx->Dm, *d = planesDev[k] + lnode * ctx->rowStride;
                if (toDevice)
                    VSOM_CUDA(ctx, cudaMemcpy2DAsync(d, pitch, h, w, w, nodes, kind, ctx->stream));
                else
                    VSOM_CUDA(ctx, cudaMemcpy2DAsync(h, w, d, pitch, w, nodes, kind, ctx->stream));
            }
        if (weight)
            VSOM_CUDA(ctx, cudaMemcpyAsync(toDevice ? ctx->weight + lnode : weight + gnode, toDevice ? weight + gnode : ctx->weight + lnode, sizeof(float) * nodes, kind, ctx->stream));
        if (hits)
            VSOM_CUDA(ctx, cudaMemcpyAsync(toDevice ? static_cast<void *>(ctx->hits + lnode) : static_cast<void *>(hits + gnode),
                                           toDevice ? static_cast<const void *>(hits + gnode) : static_cast<const void *>(ctx->hits + lnode), sizeof(u64) * nodes, kind, ctx->stream));
        lr += rows;
    }
    VSOM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return VSOM_OK;
}

int vsom_upload_state(vsom_ctx *ctx, const float *mean, const float *S, const float *sigma, const float *weight, const uint64_t *hits)
{
    if (!ctx)
        return VSOM_ERR_INVALID;
    return copy_state(ctx, true, const_cast<float *>(mean), const_cast<float *>(S), const_cast<float *>(sigma), const_cast<float *>(weight), const_cast<uint64_t *>(hits));
}

int vsom_download_state(vsom_ctx *ctx, float *mean, float *S, float *sigma, float *weight, uint64_t *hits)
{
    if (!ctx)
        return VSOM_ERR_INVALID;
    return copy_state(ctx, false, mean, S, sigma, weight, hits);
}

int vsom_get_node(vsom_ctx *ctx, size_t node, float *mean, float *sigma)
{
    if (ctx && ctx->world > 1)
        return set_error(ctx, VSOM_ERR_UNSUPPORTED, "this entry point needs an unsharded context (scoring, U-matrix and index run on replicated maps)");
    if (!ctx || node >= static_cast<size_t>(ctx->N))
        return ctx ? set_error(ctx, VSOM_ERR_INVALID, "vsom_get_node: node out of range") : VSOM_ERR_INVALID;
    VSOM_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t off = node * ctx->rowStride;
    if (mean)
        VSOM_CUDA(ctx, cudaMemcpyAsync(mean, ctx->mean + off, sizeof(float) * ctx->Dm, cudaMemcpyDeviceToHost, ctx->stream));
    if (sigma)
        VSOM_CUDA(ctx, cudaMemcpyAsync(sigma, ctx->sigma + off, sizeof(float) * ctx->Dm, cudaMemcpyDeviceToHost, ctx->stream));
    VSOM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return VSOM_OK;
}

int vsom_train_chunk_device(vsom_ctx *ctx, const float *x_dev, size_t n, double eta, double sigma, int decay, uint32_t *out_bmu_dev,
                            float *out_dist_dev)
{
    if (!ctx || (!x_dev && n))
        return ctx ? set_error(ctx, VSOM_ERR_INVALID, "vsom_train_chunk_device: x is NULL") : VSOM_ERR_INVALID;
    VSOM_CUDA(ctx, cudaSetDevice(ctx->device));
    ctx->trainEnqueued = true;
    return launch_online_step(ctx, x_dev, n, eta, sigma, decay, out_bmu_dev, out_dist_dev);
}

int vsom_train_chunk(vsom_ctx *ctx, const float *x, size_t n, double eta, double sigma, int decay, uint64_t *last_bmu, uint32_t *out_bmu,
                     float *out_dist, float *out_resid2)
{
    if (!ctx || (!x && n))
        return ctx ? set_error(ctx, VSOM_ERR_INVALID, "vsom_train_chunk: x is NULL") : VSOM_ERR_INVALID;
    if (n == 0)
        return VSOM_OK;
    VSOM_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc = stage_reserve(ctx, 0, sizeof(float) * n * ctx->Din);
    if (rc)
        return rc;
    rc = stage_reserve(ctx, 1, sizeof(unsigned) * n);
    if (rc)
        return rc;
    rc = stage_reserve(ctx, 2, sizeof(float) * n);
    if (rc)
        return rc;
    float *xDev = static_cast<float *>(ctx->stage[0]);
    unsigned *bmuDev = static_cast<unsigned *>(ctx->stage[1]);
    float *distDev = static_cast<float *>(ctx->stage[2]);
    VSOM_CUDA(ctx, cudaMemcpyAsync(xDev, x, sizeof(float) * n * ctx->Din, cudaMemcpyHostToDevice, ctx->stream));
    if (ctx->world > 1) // only the rank that owns a sample's BMU reports its distance; the others keep NaN
        VSOM_CUDA(ctx, cudaMemsetAsync(distDev, 0xff, sizeof(float) * n, ctx->stream));
    const u64 *lastDev = nullptr;
    if (!(sigma > 1.0) && last_bmu) // findLocalBmu starts its walk at the row's lastBMU (src/Som.cpp:891)
    {
        rc = stage_reserve(ctx, 3, sizeof(u64) * n);
        if (rc)
            return rc;
        for (size_t r = 0; r < n; ++r)
            if (last_bmu[r] >= static_cast<uint64_t>(ctx->N))
                return set_error(ctx, VSOM_ERR_INVALID, "vsom_train_chunk: last_bmu out of range");
        VSOM_CUDA(ctx, cudaMemcpyAsync(ctx->stage[3], last_bmu, sizeof(u64) * n, cudaMemcpyHostToDevice, ctx->stream));
        lastDev = static_cast<const u64 *>(ctx->stage[3]);
    }
    rc = launch_online_step(ctx, xDev, n, eta, sigma, decay, bmuDev, distDev, lastDev);
    if (rc)
        return rc;
    std::vector<unsigned> tmp;
    unsigned *bmuHost = out_bmu;
    if (!bmuHost && last_bmu)
    {
        tmp.resize(n);
        bmuHost = tmp.data();
    }
    if (bmuHost)
        VSOM_CUDA(ctx, cudaMemcpyAsync(bmuHost, bmuDev, sizeof(unsigned) * n, cudaMemcpyDeviceToHost, ctx->stream));
    if (out_dist)
        VSOM_CUDA(ctx, cudaMemcpyAsync(out_dist, distDev, sizeof(float) * n, cudaMemcpyDeviceToHost, ctx->stream));
    // residual.squaredNorm() (src/Som.cpp:1167) and distanceError (:946) are the same f32 sum of the same residual
    if (out_resid2)
        VSOM_CUDA(ctx, cudaMemcpyAsync(out_resid2, distDev, sizeof(float) * n, cudaMemcpyDeviceToHost, ctx->stream));
    rc = check_error_flag(ctx, "vsom_train_chunk");
    if (rc)
        return rc;
    if (last_bmu)
        for (size_t r = 0; r < n; ++r)
            last_bmu[r] = bmuHost[r]; // src/Som.cpp:895
    return VSOM_OK;
}

int vsom_batch_epoch(vsom_ctx *ctx, const float *x, size_t n, double sigma, int is_first, uint64_t *last_bmu, float *out_mse)
{
    if (!ctx || (!x && n) || (!last_bmu && n))
        return ctx ? set_error(ctx, VSOM_ERR_INVALID, "vsom_batch_epoch: NULL argument") : VSOM_ERR_INVALID;
    if (out_mse)
        *out_mse = 0.0f;
    if (n == 0)
        return VSOM_OK;
    VSOM_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc = stage_reserve(ctx, 0, sizeof(float) * n * ctx->Din);
    if (rc)
        return rc;
    rc = stage_reserve(ctx, 1, sizeof(unsigned) * n);
    if (rc)
        return rc;
    rc = stage_reserve(ctx, 2, sizeof(float) * n);
    if (rc)
        return rc;
    rc = stage_reserve(ctx, 3, sizeof(u64) * n);
    if (rc)
        return rc;
    float *xDev = static_cast<float *>(ctx->stage[0]);
    unsigned *bmuDev = static_cast<unsigned *>(ctx->stage[1]);
    float *distDev = static_cast<float *>(ctx->stage[2]);
    u64 *lastDev = static_cast<u64 *>(ctx->stage[3]);
    for (size_t r = 0; r < n; ++r)
        if (last_bmu[r] >= static_cast<uint64_t>(ctx->N))
            return set_error(ctx, VSOM_ERR_INVALID, "vsom_batch_epoch: last_bmu out of range");
    VSOM_CUDA(ctx, cudaMemcpyAsync(xDev, x, sizeof(float) * n * ctx->Din, cudaMemcpyHostToDevice, ctx->stream));
    VSOM_CUDA(ctx, cudaMemcpyAsync(lastDev, last_bmu, sizeof(u64) * n, cudaMemcpyHostToDevice, ctx->stream));
    rc = launch_batch_epoch(ctx, xDev, n, sigma, is_first, lastDev, bmuDev, distDev);
    if (rc)
        return rc;
    std::vector<unsigned> bmu(n);
    std::vector<float> dist(n);
    VSOM_CUDA(ctx, cudaMemcpyAsync(bmu.data(), bmuDev, sizeof(unsigned) * n, cudaMemcpyDeviceToHost, ctx->stream));
    VSOM_CUDA(ctx, cudaMemcpyAsync(dist.data(), distDev, sizeof(float) * n, cudaMemcpyDeviceToHost, ctx->stream));
    VSOM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    float mse = 0.0f;
    for (size_t r = 0; r < n; ++r)
    {
        last_bmu[r] = bmu[r];                       // :777 / :800
        mse = mse + dist[r] / static_cast<float>(n); // :781 / :804, f32, row order
    }
    if (out_mse)
        *out_mse = mse;
    return VSOM_OK;
}

// Batches of at least kTcMinRows rows on a shape K2 covers take the tensor-core candidate search + exact rescore (same
// results, bit for bit); everything else the exact scan.
static const size_t kTcMinRows = 1024;
static const char *kUnshardedOnly = "this entry point needs an unsharded context (scoring and index run on replicated maps)";

static int find_bmu_device_impl(vsom_ctx *ctx, const float *x_dev, size_t n, uint64_t min_hits, uint32_t *out_bmu_dev, float *out_dist_dev, bool allowTc,
                                uint64_t *fallback_rows, const char *who)
{
    if (ctx && ctx->world > 1)
        return set_error(ctx, VSOM_ERR_UNSUPPORTED, kUnshardedOnly);
    if (!ctx || (!x_dev && n))
        return ctx ? set_error(ctx, VSOM_ERR_INVALID, std::string(who) + ": x is NULL") : VSOM_ERR_INVALID;
    VSOM_CUDA(ctx, cudaSetDevice(ctx->device));
    if (fallback_rows)
        *fallback_rows = 0;
    if (!allowTc || !score_tc_supported(ctx) || n < kTcMinRows)
    {
        if (fallback_rows)
            *fallback_rows = n;
        ctx->lastScoreTc = 0;
        return launch_find_bmu(ctx, x_dev, n, min_hits, out_bmu_dev, out_dist_dev);
    }
    unsigned long long fb = 0;
    ctx->lastScoreTc = 1;
    const int rc = launch_find_bmu_tc(ctx, x_dev, n, min_hits, out_bmu_dev, out_dist_dev, &fb);
    if (fallback_rows)
        *fallback_rows = fb;
    return rc;
}

static int find_bmu_host_impl(vsom_ctx *ctx, const float *x, size_t n, uint64_t min_hits, uint32_t *out_bmu, float *out_dist, bool allowTc, uint64_t *fallback_rows,
                              const char *who)
{
    if (ctx && ctx->world > 1)
        return set_error(ctx, VSOM_ERR_UNSUPPORTED, kUnshardedOnly);
    if (!ctx || (!x && n))
        return ctx ? set_error(ctx, VSOM_ERR_INVALID, std::string(who) + ": x is NULL") : VSOM_ERR_INVALID;
    if (fallback_rows)
        *fallback_rows = 0;
    if (n == 0)
        return VSOM_OK;
    VSOM_CUDA(ctx, cudaSetDevice(ctx->device));
    if (allowTc && score_tc_supported(ctx) && n >= kTcMinRows)
    {
        // pipelined: H2D of slab i + 1, search + re-scoring of slab i and D2H of slab i - 1 overlap (score_tc.cu)
        unsigned long long fb = 0;
        size_t done = 0;
        ctx->lastScoreTc = 1;
        const int rc = launch_find_bmu_tc_host(ctx, x, n, min_hits, out_bmu, out_dist, &fb, &done);
        if (rc)
            return rc;
        if (done < n) // the probes found the map / data unsuited to the candidate search: the rest takes the exact path below
        {
            uint64_t rest = 0;
            const int rc2 = find_bmu_host_impl(ctx, x + done * ctx->Din, n - done, min_hits, out_bmu ? out_bmu + done : nullptr, out_dist ? out_dist + done : nullptr, false,
                                               &rest, who);
            ctx->lastScoreTc = 1;
            fb += rest;
            if (rc2)
                return rc2;
        }
        if (fallback_rows)
            *fallback_rows = fb;
        return VSOM_OK;
    }
    // exact scan from host rows, in slabs (a call can be the remainder of a very large batch that the probes took off the
    // tensor-core path): staging stays bounded, results return per slab
    const char *slabEnv = getenv("VSOM_EXACT_HOST_SLAB_LOG2"); // test knob
    const size_t slab = std::min(n, static_cast<size_t>(1) << (slabEnv ? atoi(slabEnv) : 20));
    int rc = stage_reserve(ctx, 0, sizeof(float) * slab * ctx->Din);
    if (rc)
        return rc;
    rc = stage_reserve(ctx, 1, sizeof(unsigned) * slab);
    if (rc)
        return rc;
    rc = stage_reserve(ctx, 2, sizeof(float) * slab);
    if (rc)
        return rc;
    float *xDev = static_cast<float *>(ctx->stage[0]);
    unsigned *bmuDev = static_cast<unsigned *>(ctx->stage[1]);
    float *distDev = static_cast<float *>(ctx->stage[2]);
    if (fallback_rows)
        *fallback_rows = n;
    ctx->lastScoreTc = 0;
    for (size_t r0 = 0; r0 < n; r0 += slab)
    {
        const size_t rows = std::min(slab, n - r0);
        VSOM_CUDA(ctx, cudaMemcpyAsync(xDev, x + r0 * ctx->Din, sizeof(float) * rows * ctx->Din, cudaMemcpyHostToDevice, ctx->stream));
        rc = launch_find_bmu(ctx, xDev, rows, min_hits, bmuDev, distDev);
        if (rc)
            return rc;
        rc = similarity_hook(ctx, xDev, rows, bmuDev, 0, ctx->stream); // armed by vsom_measure_similarity only
        if (rc)
            return rc;
        ctx->simRowBase += rows;
        if (out_bmu)
            VSOM_CUDA(ctx, cudaMemcpyAsync(out_bmu + r0, bmuDev, sizeof(unsigned) * rows, cudaMemcpyDeviceToHost, ctx->stream));
        if (out_dist)
            VSOM_CUDA(ctx, cudaMemcpyAsync(out_dist + r0, distDev, sizeof(float) * rows, cudaMemcpyDeviceToHost, ctx->stream));
        VSOM_CUDA(ctx, cudaStreamSynchronize(ctx->stream)); // the staging buffers are reused by the next slab
    }
    return VSOM_OK;
}

int vsom_find_bmu_device(vsom_ctx *ctx, const float *x_dev, size_t n, uint64_t min_hits, uint32_t *out_bmu_dev, float *out_dist_dev)
{
    return find_bmu_device_impl(ctx, x_dev, n, min_hits, out_bmu_dev, out_dist_dev, true, nullptr, "vsom_find_bmu_device");
}

int vsom_find_bmu(vsom_ctx *ctx, const float *x, size_t n, uint64_t min_hits, uint32_t *out_bmu, float *out_dist)
{
    return find_bmu_host_impl(ctx, x, n, min_hits, out_bmu, out_dist, true, nullptr, "vsom_find_bmu");
}

int vsom_find_bmu_exact_device(vsom_ctx *ctx, const float *x_dev, size_t n, uint64_t min_hits, uint32_t *out_bmu_dev, float *out_dist_dev)
{
    return find_bmu_device_impl(ctx, x_dev, n, min_hits, out_bmu_dev, out_dist_dev, false, nullptr, "vsom_find_bmu_exact_device");
}

int vsom_find_bmu_exact(vsom_ctx *ctx, const float *x, size_t n, uint64_t min_hits, uint32_t *out_bmu, float *out_dist)
{
    return find_bmu_host_impl(ctx, x, n, min_hits, out_bmu, out_dist, false, nullptr, "vsom_find_bmu_exact");
}

int vsom_find_bmu_batch_device(vsom_ctx *ctx, const float *x_dev, size_t n, uint64_t min_hits, uint32_t *out_bmu_dev, float *out_dist_dev,
                               uint64_t *fallback_rows)
{
    return find_bmu_device_impl(ctx, x_dev, n, min_hits, out_bmu_dev, out_dist_dev, true, fallback_rows, "vsom_find_bmu_batch_device");
}

int vsom_find_bmu_batch(vsom_ctx *ctx, const float *x, size_t n, uint64_t min_hits, uint32_t *out_bmu, float *out_dist, uint64_t *fallback_rows)
{
    return find_bmu_host_impl(ctx, x, n, min_hits, out_bmu, out_dist, true, fallback_rows, "vsom_find_bmu_batch");
}

int vsom_debug_tc_stats(const vsom_ctx *ctx, uint64_t out[3])
{
    if (!ctx || !out)
        return VSOM_ERR_INVALID;
    for (int i = 0; i < 3; ++i)
        out[i] = ctx->tcStats[i];
    return VSOM_OK;
}

int vsom_debug_last_score_tc(const vsom_ctx *ctx) { return ctx ? (ctx->lastScoreTc ? ctx->lastScoreTier : 0) : 0; }
int vsom_debug_last_score_pair(const vsom_ctx *ctx) { return ctx ? (ctx->lastScoreTc ? ctx->lastScorePair : 0) : 0; }

int vsom_evaluate(vsom_ctx *ctx, const float *x, size_t n, double *mean_error)
{
    if (!ctx || !mean_error)
        return ctx ? set_error(ctx, VSOM_ERR_INVALID, "vsom_evaluate: mean_error is NULL") : VSOM_ERR_INVALID;
    std::vector<float> dist(n);
    int rc = vsom_find_bmu(ctx, x, n, 0, nullptr, dist.data());
    if (rc)
        return rc;
    // src/Som.cpp:519 — Finch's incremental mean in double, in row order; with all-continuous columns the
    // binary cross-entropy vector is multiplied by zeros, so its norm contributes sqrt(0) = 0.
    double error = 0;
    for (size_t i = 0; i < n; ++i)
        error += 1. / (static_cast<double>(i) + 1.0) * (static_cast<double>(dist[i]) + 0.0 - error);
    *mean_error = error;
    return VSOM_OK;
}

int vsom_measure_similarity(vsom_ctx *ctx, const float *x, size_t n, uint64_t min_hits, int number_of_sigmas, uint32_t *out_bmu, float *out_row_max)
{
    if (!ctx || (!x && n) || (!out_row_max && n))
        return ctx ? set_error(ctx, VSOM_ERR_INVALID, "vsom_measure_similarity: NULL argument") : VSOM_ERR_INVALID;
    if (ctx->world > 1)
        return set_error(ctx, VSOM_ERR_UNSUPPORTED, kUnshardedOnly);
    if (ctx->Dm != ctx->Din)
        return set_error(ctx, VSOM_ERR_UNSUPPORTED, "vsom_measure_similarity: the model vector must have the rows' length (Standard / Median transformation)");
    if (number_of_sigmas == 0)
        return set_error(ctx, VSOM_ERR_INVALID, "vsom_measure_similarity: number_of_sigmas is 0");
    if (n == 0)
        return VSOM_OK;
    VSOM_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc = stage_reserve(ctx, 9, sizeof(float) * n);
    if (rc)
        return rc;
    ctx->simK = static_cast<float>(number_of_sigmas);
    ctx->simHost = out_row_max;
    ctx->simRowBase = 0;
    rc = find_bmu_host_impl(ctx, x, n, min_hits, out_bmu, nullptr, true, nullptr, "vsom_measure_similarity");
    ctx->simK = 0.0f;
    ctx->simHost = nullptr;
    if (rc)
        return rc;
    // the tensor-core path's result copies run on its re-scoring stream; tc_finish joined it to the context's stream
    VSOM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return VSOM_OK;
}

int vsom_all_dists(vsom_ctx *ctx, const float *v, double *out)
{
    if (ctx && ctx->world > 1)
        return set_error(ctx, VSOM_ERR_UNSUPPORTED, "this entry point needs an unsharded context (scoring, U-matrix and index run on replicated maps)");
    if (!ctx || !v || !out)
        return ctx ? set_error(ctx, VSOM_ERR_INVALID, "vsom_all_dists: NULL argument") : VSOM_ERR_INVALID;
    VSOM_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc = stage_reserve(ctx, 0, sizeof(float) * ctx->Din);
    if (rc)
        return rc;
    rc = stage_reserve(ctx, 5, sizeof(double) * ctx->N);
    if (rc)
        return rc;
    VSOM_CUDA(ctx, cudaMemcpyAsync(ctx->stage[0], v, sizeof(float) * ctx->Din, cudaMemcpyHostToDevice, ctx->stream));
    rc = launch_all_dists(ctx, static_cast<float *>(ctx->stage[0]), static_cast<double *>(ctx->stage[5]));
    if (rc)
        return rc;
    VSOM_CUDA(ctx, cudaMemcpyAsync(out, ctx->stage[5], sizeof(double) * ctx->N, cudaMemcpyDeviceToHost, ctx->stream));
    VSOM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return VSOM_OK;
}

int vsom_soft_assign(vsom_ctx *ctx, const float *x, size_t n, uint64_t min_hits, double *out_prob)
{
    if (ctx && ctx->world > 1)
        return set_error(ctx, VSOM_ERR_UNSUPPORTED, kUnshardedOnly);
    if (!ctx || (!x && n) || (!out_prob && n))
        return ctx ? set_error(ctx, VSOM_ERR_INVALID, "vsom_soft_assign: NULL argument") : VSOM_ERR_INVALID;
    if (n == 0)
        return VSOM_OK;
    VSOM_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t N = ctx->N, batch = std::max<size_t>(1, std::min<size_t>(n, (size_t{256} << 20) / (sizeof(double) * N))); // <= 256 MiB of probabilities at a time
    int rc = stage_reserve(ctx, 0, sizeof(float) * batch * ctx->Din);
    if (rc)
        return rc;
    rc = stage_reserve(ctx, 5, sizeof(double) * (batch * N + batch));
    if (rc)
        return rc;
    float *xDev = static_cast<float *>(ctx->stage[0]);
    double *probDev = static_cast<double *>(ctx->stage[5]), *sumsDev = probDev + batch * N;
    for (size_t r0 = 0; r0 < n; r0 += batch)
    {
        const size_t rows = std::min(batch, n - r0);
        VSOM_CUDA(ctx, cudaMemcpyAsync(xDev, x + r0 * ctx->Din, sizeof(float) * rows * ctx->Din, cudaMemcpyHostToDevice, ctx->stream));
        rc = launch_soft_assign(ctx, xDev, rows, min_hits, probDev, sumsDev);
        if (rc)
            return rc;
        VSOM_CUDA(ctx, cudaMemcpyAsync(out_prob + r0 * N, probDev, sizeof(double) * rows * N, cudaMemcpyDeviceToHost, ctx->stream));
        VSOM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return VSOM_OK;
}

// per-grid-row pointer tables of K4 (umatrix.cu): [H] mean rows, [H] sigma rows, then the tiles to compute.  A
// node-sharded context reads its neighbours' border rows straight out of the owners' planes (peer-mapped pointers).
static int umatrix_tables(vsom_ctx *ctx)
{
    if (ctx->umTab)
        return VSOM_OK;
    const int H = ctx->H;
    const size_t rowFloats = static_cast<size_t>(ctx->W) * ctx->rowStride;
    std::vector<const float *> rows(2 * static_cast<size_t>(H), nullptr);
    for (int lr = 0; lr < ctx->localRows; ++lr)
    {
        const int y = ctx->localRowY[lr];
        rows[y] = ctx->mean + lr * rowFloats;
        rows[H + y] = ctx->sigma + lr * rowFloats;
    }
    // Halo rows (grid rows of other ranks that border this rank's rows) are not copied: their table entries point INTO the
    // owner's mean plane (peer-mapped over NVLink), and the kernels' cp.async copies read them from there while they
    // compute — one border row of means per neighbouring block (sigma is the centre's own, SURVEY.md §8e).
    for (int lr = 0; lr < ctx->localRows; ++lr)
        for (int dy = -1; dy <= 1; dy += 2)
        {
            const int y = ctx->localRowY[lr] + dy;
            if (y < 0 || y >= H || rows[y])
                continue;
            const int owner = (y / ctx->shardBlock) % ctx->world, ly = shard_local_row(y, ctx->shardBlock, owner, ctx->world);
            if (!ctx->peerMean[owner])
                return set_error(ctx, VSOM_ERR_INVALID, "vsom_update_umatrix: sharded context without vsom_peer_import_planes / vsom_peer_attach for every rank");
            rows[y] = ctx->peerMean[owner] + ly * rowFloats;
        }
    // tiles of the tiled kernel: runs of at most umatrix_tile_rows() consecutive grid rows this context owns
    std::vector<int2> tiles;
    for (int lr = 0; lr < ctx->localRows;)
    {
        int rows_ = 1;
        while (rows_ < umatrix_tile_rows() && lr + rows_ < ctx->localRows && ctx->localRowY[lr + rows_] == ctx->localRowY[lr] + rows_)
            ++rows_;
        tiles.push_back(make_int2(ctx->localRowY[lr], rows_));
        lr += rows_;
    }
    const size_t ptrBytes = sizeof(float *) * rows.size();
    VSOM_CUDA(ctx, cudaMalloc(&ctx->umTab, ptrBytes + sizeof(int2) * tiles.size()));
    VSOM_CUDA(ctx, cudaMemcpy(ctx->umTab, rows.data(), ptrBytes, cudaMemcpyHostToDevice));
    VSOM_CUDA(ctx, cudaMemcpy(static_cast<unsigned char *>(ctx->umTab) + ptrBytes, tiles.data(), sizeof(int2) * tiles.size(), cudaMemcpyHostToDevice));
    ctx->umTiles = static_cast<int>(tiles.size());
    return VSOM_OK;
}

int vsom_update_umatrix(vsom_ctx *ctx, double *out)
{
    if (!ctx)
        return VSOM_ERR_INVALID;
    VSOM_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc = umatrix_tables(ctx);
    if (rc)
        return rc;
    const float *const *meanRows = static_cast<const float *const *>(ctx->umTab);
    rc = launch_umatrix_tiles(ctx, meanRows, meanRows + ctx->H, reinterpret_cast<const int2 *>(meanRows + 2 * ctx->H), ctx->umTiles);
    if (rc)
        return rc;
    if (out) // full-map array; a sharded context fills in its own grid rows only
        for (int lr = 0; lr < ctx->localRows;)
        {
            int rows = 1;
            while (lr + rows < ctx->localRows && ctx->localRowY[lr + rows] == ctx->localRowY[lr] + rows)
                ++rows;
            const size_t g = static_cast<size_t>(ctx->localRowY[lr]) * ctx->W;
            VSOM_CUDA(ctx, cudaMemcpyAsync(out + g, ctx->umatrix + g, sizeof(double) * rows * ctx->W, cudaMemcpyDeviceToHost, ctx->stream));
            lr += rows;
        }
    VSOM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return VSOM_OK;
}

int vsom_build_index_device(vsom_ctx *ctx, const uint32_t *bmu_dev, size_t n, uint64_t *counts_dev, uint64_t *offsets_dev, uint32_t *row_ids_dev)
{
    if (ctx && ctx->world > 1)
        return set_error(ctx, VSOM_ERR_UNSUPPORTED, kUnshardedOnly);
    if (!ctx || (!bmu_dev && n) || !counts_dev || !offsets_dev)
        return ctx ? set_error(ctx, VSOM_ERR_INVALID, "vsom_build_index_device: NULL argument") : VSOM_ERR_INVALID;
    VSOM_CUDA(ctx, cudaSetDevice(ctx->device));
    return launch_build_index(ctx, bmu_dev, n, reinterpret_cast<u64 *>(counts_dev), reinterpret_cast<u64 *>(offsets_dev), row_ids_dev);
}

int vsom_build_index(vsom_ctx *ctx, const uint32_t *bmu, size_t n, uint64_t *counts, uint64_t *offsets, uint32_t *row_ids)
{
    if (ctx && ctx->world > 1)
        return set_error(ctx, VSOM_ERR_UNSUPPORTED, "this entry point needs an unsharded context (scoring, U-matrix and index run on replicated maps)");
    if (!ctx || (!bmu && n))
        return ctx ? set_error(ctx, VSOM_ERR_INVALID, "vsom_build_index: bmu is NULL") : VSOM_ERR_INVALID;
    VSOM_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t N = ctx->N;
    int rc = stage_reserve(ctx, 1, sizeof(unsigned) * (n ? n : 1));
    if (rc)
        return rc;
    rc = stage_reserve(ctx, 2, sizeof(unsigned) * (n ? n : 1));
    if (rc)
        return rc;
    rc = stage_reserve(ctx, 5, sizeof(u64) * (2 * N + 1));
    if (rc)
        return rc;
    unsigned *bmuDev = static_cast<unsigned *>(ctx->stage[1]);
    unsigned *rowDev = static_cast<unsigned *>(ctx->stage[2]);
    u64 *countsDev = static_cast<u64 *>(ctx->stage[5]);
    u64 *offsetsDev = countsDev + N;
    if (n)
        VSOM_CUDA(ctx, cudaMemcpyAsync(bmuDev, bmu, sizeof(unsigned) * n, cudaMemcpyHostToDevice, ctx->stream));
    rc = launch_build_index(ctx, bmuDev, n, countsDev, offsetsDev, row_ids ? rowDev : nullptr);
    if (rc)
        return rc;
    if (counts)
        VSOM_CUDA(ctx, cudaMemcpyAsync(counts, countsDev, sizeof(u64) * N, cudaMemcpyDeviceToHost, ctx->stream));
    if (offsets)
        VSOM_CUDA(ctx, cudaMemcpyAsync(offsets, offsetsDev, sizeof(u64) * (N + 1), cudaMemcpyDeviceToHost, ctx->stream));
    if (row_ids && n)
        VSOM_CUDA(ctx, cudaMemcpyAsync(row_ids, rowDev, sizeof(unsigned) * n, cudaMemcpyDeviceToHost, ctx->stream));
    rc = check_error_flag(ctx, "vsom_build_index");
    if (rc)
    {
        ctx->poisoned = false;
        return set_error(ctx, VSOM_ERR_INVALID, "vsom_build_index: a BMU id is >= width*height");
    }
    return VSOM_OK;
}

} // extern "C"
