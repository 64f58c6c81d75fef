// Som.cpp — host side of class Som: the reference's public surface (include/SOM.hpp of the reference,
// implementation in its src/Som.cpp) on top of the C-ABI of libvsom_b200.so.  Epoch schedules, the DataSet
// chunk protocol, metrics and the mutex / atomic contract stay on the host exactly where the reference has
// them (src/Som.cpp:1113-1187); everything per-sample or per-node runs in the CUDA kernels.
#include "SOM.hpp"

#include "vsom_b200.h"

#include <algorithm>
#include <cassert>
#include <cmath>
#include <cstdlib>
#include <cctype>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <ctime>
#include <fstream>
#include <iostream>
#include <random>
#include <stdexcept>

struct Som::Device
{
    vsom_ctx *ctx{nullptr};
    ~Device()
    {
        if (ctx)
            vsom_destroy(ctx);
    }
};

namespace
{
[[noreturn]] void fail(vsom_ctx *ctx, const char *what)
{
    throw std::runtime_error(std::string(what) + ": " + vsom_last_error(ctx));
}
[[noreturn]] void offPath(const char *what)
{
    throw std::logic_error(std::string(what) + " is not on the B200 hot path of this build (see DESIGN.md, out of scope)");
}
std::vector<float> flatten(const std::vector<Eigen::VectorXf> &rows, size_t depth)
{
    std::vector<float> out(rows.size() * depth);
    for (size_t p = 0; p < rows.size(); ++p)
        std::memcpy(out.data() + p * depth, rows[p].data(), depth * sizeof(float));
    return out;
}
void unflatten(const std::vector<float> &flat, std::vector<Eigen::VectorXf> &rows, size_t depth)
{
    for (size_t p = 0; p < rows.size(); ++p)
        std::memcpy(rows[p].data(), flat.data() + p * depth, depth * sizeof(float));
}
// the order dot() has in the Eigen this translation unit sees (see the note at the top of SOM.hpp)
int defaultReductionOrder()
{
    if (const char *e = std::getenv("VSOM_REDUCTION_ORDER"))
    {
        const std::string v(e);
        if (v == "eigen_sse")
            return VSOM_ORDER_EIGEN_SSE;
        if (v == "lanes")
            return VSOM_ORDER_LANES;
        if (v == "reference" || v == "sequential")
            return VSOM_ORDER_REFERENCE;
    }
#if !defined(VSOM_COMPAT_EIGEN_DENSE) || defined(VSOM_COMPAT_EIGEN_SSE_REDUX)
    return VSOM_ORDER_EIGEN_SSE;
#else
    return VSOM_ORDER_REFERENCE;
#endif
}
// f32 sum of squares in a given order, for the few reductions that stay on the host (binary cross-entropy term of evaluate)
float orderedSquaredNorm(const std::vector<float> &t, int order)
{
    const size_t n = t.size();
    if (order != VSOM_ORDER_EIGEN_SSE || n < 4)
    {
        float s = 0.0f;
        for (float v : t)
            s = s + v * v;
        return s;
    }
    const size_t a2 = n / 8 * 8, a = n / 4 * 4;
    float p0[4], p1[4];
    for (size_t j = 0; j < 4; ++j)
        p0[j] = t[j] * t[j];
    if (a > 4)
    {
        for (size_t j = 0; j < 4; ++j)
            p1[j] = t[4 + j] * t[4 + j];
        for (size_t i = 8; i < a2; i += 8)
            for (size_t j = 0; j < 4; ++j)
            {
                p0[j] = p0[j] + t[i + j] * t[i + j];
                p1[j] = p1[j] + t[i + 4 + j] * t[i + 4 + j];
            }
        for (size_t j = 0; j < 4; ++j)
            p0[j] = p0[j] + p1[j];
        if (a > a2)
            for (size_t j = 0; j < 4; ++j)
                p0[j] = p0[j] + t[a2 + j] * t[a2 + j];
    }
    float s = (p0[0] + p0[2]) + (p0[1] + p0[3]);
    for (size_t i = a; i < n; ++i)
        s = s + t[i] * t[i];
    return s;
}
} // namespace

// ------------------------------------------------------------------------------------------------ construction

void Som::Construct(size_t inWidth, size_t inHeight, size_t inDepth, std::vector<std::string> names)
{
    width = inWidth;
    height = inHeight;
    depth = inDepth;
    const size_t nodes = width * height;
    map.assign(nodes, Eigen::VectorXf::Zero(static_cast<Eigen::Index>(depth)));
    sigmaMap = map;
    SMap = map;
    weightMap = Eigen::VectorXf::Zero(static_cast<Eigen::Index>(nodes));
    bmuHits.assign(nodes, 0u);
    uMatrix.assign(nodes, 0.0);
    transform.names = names;
    _isTraining = false;
    hostIsStale = false;
    deviceIsStale = true;
}

// Som(const char*) of the reference (src/Som.cpp:51-83): size from the file, zero planes, then load().
Som::Som(const char *filename) : transform{}
{
    const Eigen::VectorXf shape = getSizeFromFile(filename);
    Construct(width, height, static_cast<size_t>(shape.size()), std::vector<std::string>{});
    load(filename);
}

Som::Som(const Som &som)
    : transform{som.transform}, metrics{}, _isTraining{}, height{som.height}, width{som.width}, depth{som.depth}, metricsMutex{}
{
    som.pull();
    map = som.map;
    sigmaMap = som.sigmaMap;
    SMap = som.SMap;
    weightMap = som.weightMap;
    bmuHits = som.bmuHits;
    uMatrix = som.uMatrix;
    reductionOrder = som.reductionOrder;
    _isTraining.store(som._isTraining.load());
    hostIsStale = false;
    deviceIsStale = true; // the copy gets its own context on first use
}

Som &Som::operator=(const Som &other)
{
    if (this == &other)
        return *this;
    other.pull();
    transform = other.transform;
    map = other.map;
    sigmaMap = other.sigmaMap;
    SMap = other.SMap;
    weightMap = other.weightMap;
    bmuHits = other.bmuHits;
    uMatrix = other.uMatrix;
    height = other.height;
    width = other.width;
    depth = other.depth;
    reductionOrder = other.reductionOrder;
    _isTraining.store(other._isTraining.load());
    device.reset();
    hostIsStale = false;
    deviceIsStale = true;
    return *this;
}

Som::~Som() = default;

size_t Som::inputLength() const
{
    if (transform.deviceKind() != Transformation::DeviceKind::LinearRegression)
        return depth;
    // depth = J (J - 1)  (Transformation::Length of CLR, reference src/Transformation.cpp:162-165)
    size_t j = static_cast<size_t>((1.0 + std::sqrt(1.0 + 4.0 * static_cast<double>(depth))) / 2.0 + 0.5);
    while (j * (j - 1) > depth)
        --j;
    while (j * (j - 1) < depth)
        ++j;
    if (j * (j - 1) != depth)
        throw std::invalid_argument("Som: depth is not J*(J-1) for a linear-regression transformation");
    return j;
}

vsom_ctx *Som::context() const
{
    if (!device)
        device = std::make_shared<Device>();
    if (!device->ctx)
    {
        const auto kind = transform.deviceKind();
        if (kind == Transformation::DeviceKind::Custom)
            throw std::runtime_error("Som: this Transformation is not one of the shipped factories (Standard, StandardMedianEstimator, "
                                     "CombinatorialLinearRegression); std::function strategies cannot run on the device and there is no CPU fallback");
        const int rc = vsom_create(&device->ctx, 0, static_cast<int>(width), static_cast<int>(height), static_cast<int>(inputLength()),
                                   static_cast<int>(kind), getReductionOrder());
        if (rc != VSOM_OK)
            throw std::runtime_error(std::string("Som: vsom_create failed: ") + vsom_last_error(nullptr));
        deviceIsStale = true;
    }
    if (deviceIsStale)
    {
        const auto m = flatten(map, depth), s = flatten(SMap, depth), g = flatten(sigmaMap, depth);
        std::vector<uint64_t> hits(bmuHits.begin(), bmuHits.end());
        if (vsom_upload_state(device->ctx, m.data(), s.data(), g.data(), weightMap.data(), hits.data()) != VSOM_OK)
            fail(device->ctx, "Som: upload");
        deviceIsStale = false;
        hostIsStale = false;
    }
    return device->ctx;
}

void Som::pull() const
{
    if (!hostIsStale || !device || !device->ctx)
        return;
    const size_t nodes = width * height;
    std::vector<float> m(nodes * depth), s(nodes * depth), g(nodes * depth);
    std::vector<uint64_t> hits(nodes);
    if (vsom_download_state(device->ctx, m.data(), s.data(), g.data(), weightMap.data(), hits.data()) != VSOM_OK)
        fail(device->ctx, "Som: download");
    unflatten(m, map, depth);
    unflatten(s, SMap, depth);
    unflatten(g, sigmaMap, depth);
    for (size_t p = 0; p < nodes; ++p)
        bmuHits[p] = static_cast<size_t>(hits[p]);
    hostIsStale = false;
}

int Som::getReductionOrder() const { return reductionOrder >= 0 ? reductionOrder : defaultReductionOrder(); }

void Som::setReductionOrder(int order)
{
    if (order < VSOM_ORDER_REFERENCE || order > VSOM_ORDER_EIGEN_SSE)
        throw std::invalid_argument("Som::setReductionOrder: 0 (sequential), 1 (lanes) or 2 (Eigen SSE2)");
    if (order == getReductionOrder() && reductionOrder >= 0)
        return;
    pull();
    device.reset();
    deviceIsStale = true;
    reductionOrder = order;
}

void Som::setFastReductionOrder(bool lanes) { setReductionOrder(lanes ? VSOM_ORDER_LANES : VSOM_ORDER_REFERENCE); }

// Som::randomInitialize of the reference (src/Som.cpp:977-997): host-side, glibc rand() in node-major order,
// so that the initial planes are the reference's for the same seed.
void Som::randomInitialize(int seed, float sigma)
{
    std::srand(static_cast<unsigned>(seed));
    metrics = Metrics{depth};
    const int span = static_cast<int>(2000 * sigma);
    for (size_t p = 0; p < width * height; ++p)
    {
        for (Eigen::Index k = 0; k < map[p].size(); ++k)
        {
            map[p](k) = (static_cast<float>(std::rand() % span) - (1000.f * sigma)) / 1000.f;
            sigmaMap[p](k) = 0.0f;
            SMap[p](k) = 0.0f;
        }
        weightMap[static_cast<Eigen::Index>(p)] = 0.0f;
        bmuHits[p] = 0u;
        uMatrix[p] = 0.0;
    }
    hostIsStale = false;
    deviceIsStale = true;
}

// Linear initialisation (an addition, not in the reference): vsom_linear_init on the loaded chunk writes the device planes; the
// host mirror is refreshed from them on demand.
void Som::linearInitialize(const DataSet &dataset)
{
    if (dataset.vectorLength() != inputLength())
        throw std::invalid_argument("Som::linearInitialize: the rows' length differs from the map's input length");
    vsom_ctx *ctx = context();
    if (vsom_linear_init(ctx, dataset.contiguousRows(), dataset.size(), nullptr, nullptr, nullptr) != VSOM_OK)
        fail(ctx, "Som::linearInitialize");
    metrics = Metrics{depth};
    std::fill(uMatrix.begin(), uMatrix.end(), 0.0);
    hostIsStale = true;
}

// Clustering of the nodes (an addition, not in the reference): vsom_cluster_nodes over the device planes, which it leaves unchanged.
double Som::clusterNodes(size_t k, std::vector<int> &labels, std::vector<Eigen::VectorXd> &centroids, uint64_t seed, bool weightByHits, int maxIterations) const
{
    const size_t nodes = width * height;
    if (k < 1 || k > nodes)
        throw std::invalid_argument("Som::clusterNodes: k must lie in 1 .. width*height");
    vsom_ctx *ctx = context();
    std::vector<int32_t> lab(nodes);
    std::vector<double> cent(k * depth);
    double inertia = 0.0;
    if (vsom_cluster_nodes(ctx, static_cast<int>(k), seed, weightByHits ? VSOM_CLUSTER_HITS : VSOM_CLUSTER_UNIFORM, maxIterations, lab.data(), cent.data(), nullptr,
                           &inertia, nullptr, nullptr) != VSOM_OK)
        fail(ctx, "Som::clusterNodes");
    labels.assign(lab.begin(), lab.end());
    centroids.assign(k, Eigen::VectorXd(static_cast<Eigen::Index>(depth)));
    for (size_t j = 0; j < k; ++j)
        std::memcpy(centroids[j].data(), cent.data() + j * depth, depth * sizeof(double));
    return inertia;
}

// ------------------------------------------------------------------------------------------------ training

void Som::train(DataSet &data, size_t numberOfEpochs, double eta0, double etaDecay, double sigma0, double sigmaDecay,
                WeigthDecayFunction weightDecayFunction, bool updateUMatrixAfterEpoch)
{
    // same contract as the reference (src/Som.cpp:1113-1132): exceptions end the run with a message on
    // std::cerr and the flag is cleared either way, so a polling thread never hangs on isTraining()
    _isTraining = true;
    try
    {
        if (weightDecayFunction == WeigthDecayFunction::BatchMap)
            trainBatchSom(data, numberOfEpochs, sigma0, sigmaDecay, updateUMatrixAfterEpoch);
        else
            trainBasicSom(data, numberOfEpochs, eta0, etaDecay, sigma0, sigmaDecay, weightDecayFunction, updateUMatrixAfterEpoch);
    }
    catch (const std::exception &e)
    {
        std::cerr << e.what() << '\n';
    }
    _isTraining = false;
}

void Som::trainBasicSom(DataSet &data, size_t numberOfEpochs, double eta0, double etaDecay, double sigma0, double sigmaDecay,
                        WeigthDecayFunction weightDecayFunction, bool updateUMatrixAfterEpoch)
{
    if (weightDecayFunction == WeigthDecayFunction::BatchMap)
        offPath("trainBasicSom(BatchMap)");
    vsom_ctx *ctx = context();
    metrics = Metrics(numberOfEpochs);
    const int decay = weightDecayFunction == WeigthDecayFunction::Exponential ? VSOM_EXPONENTIAL : VSOM_INVERSE_PROPORTIONAL;
    std::vector<float> resid2;
    std::vector<uint64_t> last;
    for (size_t epoch = 0; epoch < numberOfEpochs; ++epoch)
    {
        // schedules of src/Som.cpp:1145-1149 (sigma is clamped UP to 1)
        const double eta = eta0 * std::exp(-etaDecay * static_cast<double>(epoch));
        double sigma = sigma0 * std::exp(-sigmaDecay * static_cast<double>(epoch));
        if (sigma < 1.0)
            sigma = 1.0;
        float meanSquareError{0.0};
        size_t chunks{0};
        while (!data.hasReadWholeDataStream())
        {
            data.loadNextDataFromStream();
            const size_t rows = data.size();
            resid2.resize(rows);
            auto &lastColumn = data.lastBmuColumn();
            last.assign(lastColumn.begin(), lastColumn.end());
            // one persistent kernel runs the whole chunk: trainSingle + addBmu for every row, in row order
            if (vsom_train_chunk(ctx, data.contiguousRows(), rows, eta, sigma, decay, last.data(), nullptr, nullptr, resid2.data()) != VSOM_OK)
                fail(ctx, "Som::trainBasicSom");
            hostIsStale = true;
            for (size_t j = 0; j < rows; ++j)
            {
                lastColumn[j] = static_cast<size_t>(last[j]);
                meanSquareError += resid2[j] / static_cast<float>(rows); // src/Som.cpp:1167, f32, row order
            }
            ++chunks;
        }
        meanSquareError /= static_cast<float>(chunks);
        {
            const std::lock_guard<std::mutex> lock(metricsMutex);
            metrics.MeanSquaredError[epoch] = meanSquareError;
        }
        data.resetStreamLoadPosition();
        if (updateUMatrixAfterEpoch)
            updateUMatrix(data.getWeights());
    }
}

// Batch-map trainer (reference src/Som.cpp:716-754): sigma schedule without clamp — the run RETURNS at the first epoch
// whose sigma drops below 1 — one trainBatchSomEpoch per loaded chunk, MSE averaged over the chunks of the epoch.
void Som::trainBatchSom(DataSet &data, size_t numberOfEpochs, double sigma0, double sigmaDecay, bool updateUMatrixAfterEpoch)
{
    metrics = Metrics(numberOfEpochs);
    for (size_t epoch = 0; epoch < numberOfEpochs; ++epoch)
    {
        const double sigma = sigma0 * std::exp(-sigmaDecay * static_cast<double>(epoch));
        if (sigma < 1.0)
            return;
        float meanSquareError{0.0f};
        size_t chunks{0};
        while (!data.hasReadWholeDataStream())
        {
            data.loadNextDataFromStream();
            meanSquareError += trainBatchSomEpoch(data, sigma, epoch == 0);
            ++chunks;
        }
        meanSquareError /= static_cast<float>(chunks);
        {
            const std::lock_guard<std::mutex> lock(metricsMutex);
            metrics.MeanSquaredError[epoch] = meanSquareError;
        }
        data.resetStreamLoadPosition();
        if (updateUMatrixAfterEpoch)
            updateUMatrix(data.getWeights());
    }
}

// One chunk-epoch on the device (K6, csrc/batch_map.cu): BMU per row, hits, squared residuals, then every neuron's
// incrementally weighted mean / variance over the chunk's rows (reference src/Som.cpp:756-879).
float Som::trainBatchSomEpoch(DataSet &data, double currentSigma, bool isFirst)
{
    vsom_ctx *ctx = context();
    auto &lastColumn = data.lastBmuColumn();
    std::vector<uint64_t> last(lastColumn.begin(), lastColumn.end());
    float mse = 0.0f;
    if (vsom_batch_epoch(ctx, data.contiguousRows(), data.size(), currentSigma, isFirst ? 1 : 0, last.data(), &mse) != VSOM_OK)
        fail(ctx, "Som::trainBatchSomEpoch");
    hostIsStale = true;
    for (size_t j = 0; j < last.size(); ++j)
        lastColumn[j] = static_cast<size_t>(last[j]);
    return mse;
}

Som::TrainingReturnValue Som::trainSingle(const Eigen::VectorXf &v, const Eigen::VectorXf &valid, const Eigen::VectorXf &weights, const double eta,
                                          const double sigma, size_t &lastBMU, const WeigthDecayFunction weightDecayFunction)
{
    if (weightDecayFunction == WeigthDecayFunction::BatchMap)
        offPath("trainSingle(BatchMap)");
    vsom_ctx *ctx = context();
    uint64_t last = lastBMU;
    uint32_t bmu = 0;
    float dist = 0;
    const int decay = weightDecayFunction == WeigthDecayFunction::Exponential ? VSOM_EXPONENTIAL : VSOM_INVERSE_PROPORTIONAL;
    // NB: unlike trainBasicSom this does NOT count the hit: the reference's caller does that with addBmu()
    if (vsom_train_chunk(ctx, v.data(), 1, eta, sigma, decay, &last, &bmu, &dist, nullptr) != VSOM_OK)
        fail(ctx, "Som::trainSingle");
    hostIsStale = true;
    lastBMU = static_cast<size_t>(last);
    Eigen::VectorXf neuron(static_cast<Eigen::Index>(depth)), spread(static_cast<Eigen::Index>(depth));
    if (vsom_get_node(ctx, bmu, neuron.data(), spread.data()) != VSOM_OK)
        fail(ctx, "Som::trainSingle");
    // the kernel's chunk entry point already did addBmu for its row; undo it so that trainSingle + addBmu
    // by the caller counts once, like in the reference (src/Som.cpp:1163-1165)
    pull();
    bmuHits[bmu] -= 1;
    deviceIsStale = true;
    Eigen::VectorXf mask = (valid.array() * weights.array()).matrix();
    return TrainingReturnValue{SomIndex(bmu % width, bmu / width), transform.Comparer(v, neuron, spread, mask), dist};
}

void Som::addBmu(SomIndex position)
{
    pull();
    bmuHits[getIndex(position)] += 1;
    deviceIsStale = true;
}

// ------------------------------------------------------------------------------------------------ scoring

void Som::mapDataSet(const DataSet &dataset, std::vector<size_t> &bmuOut, std::vector<float> &distOut, size_t minBmuHits) const
{
    vsom_ctx *ctx = context();
    const size_t rows = dataset.size();
    std::vector<uint32_t> bmu(rows);
    distOut.resize(rows);
    if (vsom_find_bmu(ctx, dataset.contiguousRows(), rows, minBmuHits, bmu.data(), distOut.data()) != VSOM_OK)
        fail(ctx, "Som::mapDataSet");
    bmuOut.assign(bmu.begin(), bmu.end());
}

// Prediction from a column subset (an addition, not in the reference): vsom_predict_columns over the loaded chunk.
void Som::predictColumns(const DataSet &dataset, const std::vector<bool> &matchColumns, std::vector<size_t> &bmuOut, std::vector<float> &distOut,
                         std::vector<float> &meanOut, std::vector<float> &sigmaOut, size_t minBmuHits) const
{
    if (transform.deviceKind() == Transformation::DeviceKind::LinearRegression)
        throw std::invalid_argument("Som::predictColumns: a CLR map's model vector holds regression coefficients, not data columns");
    if (matchColumns.size() != depth)
        throw std::invalid_argument("Som::predictColumns: the mask's length differs from getDepth()");
    std::vector<uint8_t> match(depth);
    size_t matched = 0;
    for (size_t j = 0; j < depth; ++j)
        matched += match[j] = matchColumns[j] ? 1 : 0;
    if (matched == 0)
        throw std::invalid_argument("Som::predictColumns: the mask has no matched column");
    vsom_ctx *ctx = context();
    const size_t rows = dataset.size(), q = depth - matched;
    std::vector<uint32_t> bmu(rows);
    distOut.resize(rows);
    meanOut.resize(rows * q);
    sigmaOut.resize(rows * q);
    if (vsom_predict_columns(ctx, dataset.contiguousRows(), rows, match.data(), minBmuHits, bmu.data(), distOut.data(), meanOut.data(), sigmaOut.data()) != VSOM_OK)
        fail(ctx, "Som::predictColumns");
    bmuOut.assign(bmu.begin(), bmu.end());
}

void Som::mapDataSetTopTwo(const DataSet &dataset, std::vector<size_t> &bmuOut, std::vector<float> &distOut, std::vector<size_t> &bmu2Out,
                           std::vector<float> &dist2Out, size_t minBmuHits) const
{
    vsom_ctx *ctx = context();
    const size_t rows = dataset.size();
    std::vector<uint32_t> bmu(rows), bmu2(rows);
    distOut.resize(rows);
    dist2Out.resize(rows);
    if (vsom_find_bmu2(ctx, dataset.contiguousRows(), rows, minBmuHits, bmu.data(), distOut.data(), bmu2.data(), dist2Out.data(), nullptr) != VSOM_OK)
        fail(ctx, "Som::mapDataSetTopTwo");
    bmuOut.assign(bmu.begin(), bmu.end());
    bmu2Out.resize(rows);
    for (size_t i = 0; i < rows; ++i)
        bmu2Out[i] = bmu2[i] == 0xFFFFFFFFu ? SIZE_MAX : static_cast<size_t>(bmu2[i]);
}

double Som::topographicError(const DataSet &dataset) const
{
    std::vector<size_t> bmu, bmu2;
    std::vector<float> dist, dist2;
    mapDataSetTopTwo(dataset, bmu, dist, bmu2, dist2, 0);
    if (bmu.empty())
        return 0.0;
    size_t errors = 0;
    for (size_t i = 0; i < bmu.size(); ++i)
    {
        if (bmu2[i] == SIZE_MAX)
            continue;
        const long long dx = static_cast<long long>(bmu[i] % width) - static_cast<long long>(bmu2[i] % width);
        const long long dy = static_cast<long long>(bmu[i] / width) - static_cast<long long>(bmu2[i] / width);
        if (std::max(std::llabs(dx), std::llabs(dy)) != 1)
            ++errors;
    }
    return static_cast<double>(errors) / static_cast<double>(bmu.size());
}

void Som::buildIndex(const std::vector<size_t> &bmu, std::vector<size_t> &counts, std::vector<size_t> &offsets, std::vector<unsigned> &rowIds) const
{
    vsom_ctx *ctx = context();
    std::vector<uint32_t> b(bmu.begin(), bmu.end());
    std::vector<uint64_t> c(width * height), o(width * height + 1);
    rowIds.resize(bmu.size());
    if (vsom_build_index(ctx, b.data(), b.size(), c.data(), o.data(), rowIds.data()) != VSOM_OK)
        fail(ctx, "Som::buildIndex");
    counts.assign(c.begin(), c.end());
    offsets.assign(o.begin(), o.end());
}

SomIndex Som::findBmu(const Eigen::VectorXf &v) const
{
    const Eigen::VectorXf ones = Eigen::VectorXf::Ones(v.size());
    return findBmu(v, ones, ones);
}

SomIndex Som::findBmu(const Eigen::VectorXf &v, const Eigen::VectorXf &, const Eigen::VectorXf &) const
{
    // validity and weights are built and then ignored by every shipped Comparer (SURVEY.md §0.3)
    vsom_ctx *ctx = context();
    uint32_t bmu = 0;
    if (vsom_find_bmu(ctx, v.data(), 1, 0, &bmu, nullptr) != VSOM_OK)
        fail(ctx, "Som::findBmu");
    return SomIndex(bmu % width, bmu / width);
}

SomIndex Som::findRestrictedBmu(const Eigen::VectorXf &v, const Eigen::VectorXf &, const size_t minBmuHits, const Eigen::VectorXf &) const
{
    vsom_ctx *ctx = context();
    uint32_t bmu = 0;
    if (vsom_find_bmu(ctx, v.data(), 1, minBmuHits, &bmu, nullptr) != VSOM_OK)
        fail(ctx, "Som::findRestrictedBmu");
    return SomIndex(bmu % width, bmu / width);
}

// findLocalBmu (reference src/Som.cpp:335-454): the greedy walk itself is a handful of comparisons; the
// distances it compares come from the device (one pass over all nodes), so they are the device's bits.
SomIndex Som::findLocalBmu(const Eigen::VectorXf &v, const Eigen::VectorXf &, const size_t &lastBMUref, const Eigen::VectorXf &) const
{
    vsom_ctx *ctx = context();
    std::vector<double> dist(width * height);
    if (vsom_all_dists(ctx, v.data(), dist.data()) != VSOM_OK)
        fail(ctx, "Som::findLocalBmu");
    const size_t W = width, H = height, M1 = static_cast<size_t>(-1);
    // size_t arithmetic on purpose: "-1" is 2^64-1, so min(x + off, W-1) wraps the left/up neighbour of
    // column/row 0 to the last column/row (SURVEY.md App. B.3)
    auto clampX = [&](size_t x) { return std::max<size_t>(std::min<size_t>(x, W - 1), 0); };
    auto clampY = [&](size_t y) { return std::max<size_t>(std::min<size_t>(y, H - 1), 0); };
    const size_t offX[8] = {M1, 0, 1, 1, 1, 0, M1, M1}, offY[8] = {1, 1, 1, 0, M1, M1, M1, 0};
    size_t from = lastBMUref, best = from, probe = from;
    double bestDist = dist[from];
    auto consider = [&](size_t cx, size_t cy) {
        const size_t at = cy * W + cx;
        if (dist[at] < bestDist)
        {
            bestDist = dist[at];
            best = at;
        }
    };
    for (;;)
    {
        const size_t px = probe % W, py = probe / W, fx = from % W, fy = from / W;
        if (probe == from)
        {
            for (int k = 0; k < 8; ++k)
                consider(clampX(px + offX[k]), clampY(py + offY[k]));
            if (best == from)
                break;
            probe = best;
        }
        else
        {
            if (px - fx) // continue in the X direction: three cells one step further
                for (int k = -1; k < 2; ++k)
                    consider(clampX(px + px - fx), clampY(py + static_cast<size_t>(static_cast<long long>(k))));
            // the reference's Y-direction continuation starts its column loop at size_t(-1) and therefore never
            // runs (src/Som.cpp:411-426); nothing to do here
            if (best == probe)
                break;
            from = probe;
            probe = best;
        }
    }
    return SomIndex(best % W, best / W);
}

std::vector<double> Som::findRestrictedBmd(const Eigen::VectorXf &v, const Eigen::VectorXf &, size_t minBmuHits, const Eigen::VectorXf &) const
{
    vsom_ctx *ctx = context();
    std::vector<double> out(width * height);
    if (vsom_all_dists(ctx, v.data(), out.data()) != VSOM_OK)
        fail(ctx, "Som::findRestrictedBmd");
    pull();
    // reference src/Som.cpp:457-487: exp(-d*d/2) of the (already squared) distance, normalised by the sum
    double total = 0;
    for (size_t p = 0; p < out.size(); ++p)
    {
        out[p] = bmuHits[p] >= minBmuHits ? std::exp(-out[p] * out[p] / 2) : 0.0;
        total += out[p];
    }
    for (double &d : out)
        d /= total;
    return out;
}

double Som::euclidianWeightedDist(const SomIndex &pos, const Eigen::VectorXf &v, const Eigen::VectorXf &valid, const Eigen::VectorXf &weights) const
{
    const size_t at = getIndex(pos);
    return euclidianWeightedDist(at, v, valid, weights);
}

double Som::euclidianWeightedDist(const size_t &pos, const Eigen::VectorXf &v, const Eigen::VectorXf &, const Eigen::VectorXf &) const
{
    vsom_ctx *ctx = context();
    std::vector<double> dist(width * height);
    if (vsom_all_dists(ctx, v.data(), dist.data()) != VSOM_OK)
        fail(ctx, "Som::euclidianWeightedDist");
    return dist[pos];
}

// reference src/Som.cpp:143-157 — only updateUMatrix uses it there; single calls are evaluated on the mirror
double Som::euclidianWeightedDistRaw(const size_t &pos, const Eigen::VectorXf &v, const Eigen::VectorXf &valid, const Eigen::VectorXf &weights) const
{
    pull();
    float sum = 0.0f;
    for (Eigen::Index k = 0; k < map[pos].size(); ++k)
    {
        const float s = sigmaMap[pos][k] < 0.00001f ? 0.00001f : sigmaMap[pos][k];
        const float d = map[pos][k] - v[k];
        const float a = d / s;
        const float b = (d * (valid[k] * weights[k])) / s;
        sum = sum + a * b;
    }
    return static_cast<double>(sum);
}

double Som::evaluate(const DataSet &dataset) const
{
    vsom_ctx *ctx = context();
    const Eigen::ArrayXi binary = dataset.getBinary();
    bool anyBinary = false;
    for (Eigen::Index k = 0; k < binary.size(); ++k)
        anyBinary = anyBinary || binary[k] != 0;
    const size_t rows = dataset.size();
    if (!anyBinary)
    {
        double error = 0;
        if (vsom_evaluate(ctx, dataset.contiguousRows(), rows, &error) != VSOM_OK)
            fail(ctx, "Som::evaluate");
        return error;
    }
    // binary columns: BMUs and distances from the device, the cross-entropy term of src/Som.cpp:509-519 here
    // (the reference reads an uninitialised `ones` array at :495; the evident intent, 1.0, is used)
    std::vector<uint32_t> bmu(rows);
    std::vector<float> dist(rows);
    if (vsom_find_bmu(ctx, dataset.contiguousRows(), rows, 0, bmu.data(), dist.data()) != VSOM_OK)
        fail(ctx, "Som::evaluate");
    pull();
    double error = 0;
    for (size_t i = 0; i < rows; ++i)
    {
        const Eigen::VectorXf x = dataset.getData(i);
        const Eigen::VectorXi ok = dataset.getValidity(i);
        const Eigen::ArrayXi cont = dataset.getContinuous();
        std::vector<float> ce(static_cast<size_t>(x.size()));
        for (Eigen::Index k = 0; k < x.size(); ++k)
        {
            const float m = map[bmu[i]][k];
            float e = std::log(m) * x[k] + std::log(1.0f - m) * (1.0f - x[k]);
            if (std::isnan(e) || std::isinf(e))
                e = -99999;
            ce[static_cast<size_t>(k)] = e * static_cast<float>(binary[k]) * static_cast<float>(ok[k] * cont[k]);
        }
        const float ce2 = orderedSquaredNorm(ce, getReductionOrder()); // binaryError.dot(binaryError), src/Som.cpp:519
        error += 1. / (static_cast<double>(i) + 1.0) * (static_cast<double>(dist[i]) + std::sqrt(ce2) - error);
    }
    return error;
}

// reference src/Som.cpp:631-714 with its quirks (reversed sigma clamp :658, signed delta against a stored
// |delta| :686-688, re-visit of the arg-max row :643-647); the per-row BMU search is one device pass.
int Som::measureSimilarity(const DataSet *dataset, int numberOfSigmas, size_t minBmuHits) const
{
    vsom_ctx *ctx = context();
    const size_t rows = dataset->size();
    if (rows == 0)
        return 1;
    const size_t D = dataset->vectorLength();
    // One pass over PCIe: per row the restricted BMU and the row's largest delta (device, the reference's f32 operations); the
    // O(rows x columns) loop of the reference (:640-706) would otherwise keep one host core busy ~50x longer than the BMU search.
    // CLR maps (model vector longer than the rows) and numberOfSigmas == 0 (division by zero: every delta is +-inf / NaN) keep the
    // reference's loop on the host.
    const bool onDevice = vsom_depth(ctx) == static_cast<int>(D) && numberOfSigmas != 0;
    std::vector<uint32_t> bmu(rows);
    std::vector<float> rowMax;
    if (onDevice)
    {
        rowMax.resize(rows);
        if (vsom_measure_similarity(ctx, dataset->contiguousRows(), rows, minBmuHits, numberOfSigmas, bmu.data(), rowMax.data()) != VSOM_OK)
            fail(ctx, "Som::measureSimilarity");
    }
    else if (vsom_find_bmu(ctx, dataset->contiguousRows(), rows, minBmuHits, bmu.data(), nullptr) != VSOM_OK)
        fail(ctx, "Som::measureSimilarity");
    pull();
    const float k = static_cast<float>(numberOfSigmas);
    float largest = -99999999.f;
    size_t largestRow = 0;
    int success = 1;
    auto visit = [&](size_t i, bool judge) {
        const float *v = dataset->contiguousRows() + i * D;
        const Eigen::VectorXf &m = map[bmu[i]], &sg = sigmaMap[bmu[i]];
        const Eigen::VectorXi ok = dataset->getValidity(i);
        for (size_t d = 0; d < D; ++d)
        {
            const float sM = sg[d] > 0.00001f ? 0.00001f : sg[d];
            const float delta = ((v[d] - m[d]) / sM) / k;
            if (delta > largest)
            {
                largest = static_cast<float>(std::fabs(static_cast<double>(delta)));
                largestRow = i;
            }
            // only columns that are present in the row are judged (src/Som.cpp:697-703)
            if (judge && ok[static_cast<Eigen::Index>(d)] && (v[d] < m[d] - sM * k || v[d] > m[d] + sM * k))
                success = 0;
        }
    };
    size_t i = 0;
    // The reference's running maximum starts at -99999999 and stores |delta| on its FIRST update (which may be a negative delta);
    // until then the rows are replayed element by element.  From then on the value is >= 0, an update needs delta > value >= 0 and
    // stores delta itself, so a row can only raise it to its own largest delta: the device's per-row maxima carry the scan.
    for (; i < rows && (!onDevice || largest < 0.0f); ++i)
        visit(i, false);
    for (; i < rows; ++i)
        if (rowMax[i] > largest)
        {
            largest = rowMax[i];
            largestRow = i;
        }
    visit(largestRow, true);
    return success;
}

// reference src/Som.cpp:525-566.  Every row's distribution is computed and sampled there, but only the LAST row's sample
// is returned and the generator is freshly seeded from std::random_device on every call, so the earlier rows have no
// observable effect: the device computes the last row's soft assignment (vsom_soft_assign) and one sample is drawn on
// the host exactly like the reference draws it (std::mt19937 + std::discrete_distribution).
size_t Som::variationalAutoEncoder(const DataSet *dataset, size_t minBmuHits) const
{
    const size_t rows = dataset->size();
    if (rows == 0)
        return 0;
    vsom_ctx *ctx = context();
    std::vector<double> probability(width * height);
    const float *lastRow = dataset->contiguousRows() + (rows - 1) * dataset->vectorLength();
    if (vsom_soft_assign(ctx, lastRow, 1, minBmuHits, probability.data()) != VSOM_OK)
        fail(ctx, "Som::variationalAutoEncoder");
    std::random_device rd;
    std::mt19937 gen(rd());
    std::discrete_distribution<size_t> d(probability.begin(), probability.end());
    return d(gen);
}

// reference src/Som.cpp:568-623: per row, a model vector drawn from the (last row's, see above) soft assignment, then per
// column the record value and a logistic approximation of a normal sample around that neuron, printed to std::cout.
int Som::autoEncoder(const DataSet *dataset, size_t minBmuHits) const
{
    const size_t rows = dataset->size();
    if (rows == 0)
        return 1;
    vsom_ctx *ctx = context();
    std::vector<double> probability(width * height);
    const float *lastRow = dataset->contiguousRows() + (rows - 1) * dataset->vectorLength();
    if (vsom_soft_assign(ctx, lastRow, 1, minBmuHits, probability.data()) != VSOM_OK)
        fail(ctx, "Som::autoEncoder");
    pull();
    std::srand(static_cast<unsigned>(std::time(nullptr) + std::clock()));
    std::random_device rd;
    std::mt19937 gen(rd());
    std::discrete_distribution<size_t> draw(probability.begin(), probability.end());
    for (size_t i = 0; i < rows; ++i)
    {
        const Eigen::VectorXf v = dataset->getData(i);
        const size_t node = draw(gen);
        for (Eigen::Index n = 0; n < v.size(); ++n)
        {
            std::cout << v(n) << "\n";
            const double L = static_cast<double>(std::rand() % 1000) / 1000;
            const double N = std::log(L / (1 - L)) / 1.6 * sigmaMap[node][n] + map[node][n];
            std::cout << dataset->getName(static_cast<size_t>(n)) << "\t" << N << "\t"
                      << "\n";
        }
        std::cout << "\n";
    }
    return 1;
}

// ------------------------------------------------------------------------------------------------ U-matrix

void Som::updateUMatrix(const Eigen::VectorXf &)
{
    // the argument is ignored by the reference too (it overwrites it with ones, src/Som.cpp:1002-1003)
    vsom_ctx *ctx = context();
    if (vsom_update_umatrix(ctx, uMatrix.data()) != VSOM_OK)
        fail(ctx, "Som::updateUMatrix");
}

UMatrix Som::getUMatrix() const noexcept { return UMatrix{uMatrix, width, height}; }

// ------------------------------------------------------------------------------------------------ accessors

Eigen::VectorXf Som::getWeigthMap() const noexcept
{
    pull();
    return weightMap;
}
std::vector<size_t> Som::getBmuHits() const noexcept
{
    pull();
    return bmuHits;
}
size_t Som::getHeight() const noexcept { return height; }
size_t Som::getWidth() const noexcept { return width; }
size_t Som::getDepth() const noexcept { return depth; }
size_t Som::getIndex(SomIndex index) const noexcept { return index.getY() * width + index.getX(); }
Eigen::VectorXf Som::getNeuron(SomIndex index) const noexcept { return getNeuron(getIndex(index)); }
Eigen::VectorXf Som::getNeuron(size_t index) const noexcept
{
    pull();
    return map[index];
}
Eigen::VectorXf Som::getSigmaNeuron(SomIndex index) const noexcept { return getSigmaNeuron(getIndex(index)); }
Eigen::VectorXf Som::getSigmaNeuron(size_t index) const noexcept
{
    pull();
    return sigmaMap[index];
}
std::vector<std::string> Som::getNeuronStrings(SomIndex index) const noexcept { return transform.Displayer(getNeuron(index)); }
std::vector<std::string> Som::getSigmaNeuronStrings(SomIndex index) const noexcept { return transform.Displayer(getSigmaNeuron(index)); }

namespace
{
template <typename Pick> float extreme(const std::vector<Eigen::VectorXf> &plane, size_t feature, Pick better)
{
    assert(feature < static_cast<size_t>(plane.at(0).size()));
    float best = plane[0][static_cast<Eigen::Index>(feature)];
    for (const auto &row : plane)
        if (better(row[static_cast<Eigen::Index>(feature)], best))
            best = row[static_cast<Eigen::Index>(feature)];
    return best;
}
} // namespace

float Som::getMaxValueOfFeature(size_t f) const
{
    pull();
    return extreme(map, f, [](float a, float b) { return a > b; });
}
float Som::getMinValueOfFeature(size_t f) const
{
    pull();
    return extreme(map, f, [](float a, float b) { return a < b; });
}
float Som::getMaxSigmaOfFeature(size_t f) const
{
    pull();
    return extreme(sigmaMap, f, [](float a, float b) { return a > b; });
}
float Som::getMinSigmaOfFeature(size_t f) const
{
    pull();
    return extreme(sigmaMap, f, [](float a, float b) { return a < b; });
}

Som::Metrics Som::getMetrics() const noexcept { return metrics; }
bool Som::isTraining() const noexcept { return _isTraining; }
bool Som::isCompatibleWithData(DataSet &data) const noexcept { return transform.Length(data.vectorLength()) == depth; }

void Som::display() const
{
    pull();
    for (size_t p = 0; p < map.size(); ++p)
        std::cout << "node " << p << ": " << map[p].transpose() << "\n";
}
void Som::displayUMatrix() const
{
    for (size_t y = 0; y < height; ++y)
    {
        for (size_t x = 0; x < width; ++x)
            std::cout << uMatrix[y * width + x] << (x + 1 < width ? " " : "");
        std::cout << "\n";
    }
}

// ------------------------------------------------------------------------------------------------ persistence
// Octave-text checkpoint of the reference (src/Som.cpp:1209-1294 save, :1296-1341 getSizeFromFile, :1343-1598 load).
// Layout: sections "som" and "sigmaSom" (ndims 3: width height depth; one " %f" per line, node index fastest, then
// dimension), then "weightMap", "bmuHits", "U" as `width` text rows of `height` tab-separated values taken from the
// linear arrays in order (a plain reshape: "# rows" carries the WIDTH and "# columns" the HEIGHT).  SMap is not
// persisted, %f keeps six decimals, and the reader only accepts value lines whose first significant character is a
// digit (or '-' in the 3-D sections) — all as in the reference; the state is pulled from the device before writing
// and pushed again after reading.
void Som::save(const char *filename) const
{
    pull();
    FILE *fp = std::fopen(filename, "w");
    if (!fp)
    {
        std::cout << "Could not open file " << filename << " for writing. Quitting...\n";
        std::exit(EXIT_FAILURE);
    }
    const unsigned long W = width, H = height, D = depth;
    std::fprintf(fp, "# This file is generated by Som.exe\n# It contains all data needed to evaluate a sample according to the SOM trained by Som.exe\n");
    auto cube = [&](const char *name, const std::vector<Eigen::VectorXf> &plane) {
        std::fprintf(fp, "# name: %s\n# type: matrix\n# ndims: 3\n %lu %lu %lu\n", name, W, H, D);
        for (unsigned long k = 0; k < D; ++k)
            for (unsigned long p = 0; p < W * H; ++p)
                std::fprintf(fp, " %f\n", plane[p](static_cast<Eigen::Index>(k)));
    };
    auto sheetHeader = [&](const char *name) { std::fprintf(fp, "\n\n# name: %s\n# type: matrix\n# rows: %lu\n# columns: %lu\n", name, W, H); };
    cube("som", map);
    std::fprintf(fp, "\n\n");
    cube("sigmaSom", sigmaMap);
    sheetHeader("weightMap");
    for (unsigned long r = 0; r < W; ++r)
    {
        for (unsigned long c = 0; c < H; ++c)
            std::fprintf(fp, "%f\t", weightMap[static_cast<Eigen::Index>(r * H + c)]);
        std::fprintf(fp, "\n");
    }
    sheetHeader("bmuHits");
    for (unsigned long r = 0; r < W; ++r)
    {
        for (unsigned long c = 0; c < H; ++c)
            std::fprintf(fp, "%lu\t", static_cast<unsigned long>(bmuHits[r * H + c]));
        std::fprintf(fp, "\n");
    }
    sheetHeader("U");
    for (unsigned long r = 0; r < W; ++r)
    {
        for (unsigned long c = 0; c < H; ++c)
            std::fprintf(fp, "%f\t", uMatrix[r * H + c]);
        std::fprintf(fp, "\n");
    }
    std::fclose(fp);
}

Eigen::VectorXf Som::getSizeFromFile(const char *filename)
{
    std::ifstream file(filename);
    if (!file.is_open())
    {
        std::cout << "Could not open file " << filename << " for reading. Quitting...\n";
        std::exit(EXIT_FAILURE);
    }
    Eigen::VectorXf shape(1);
    std::string line;
    while (std::getline(file, line))
    {
        if (line.compare(0, 9, "# ndims: ") == 0)
        {
            std::getline(file, line); // " W H D": the vector length is the last number
            shape.resize(static_cast<Eigen::Index>(std::stoul(line.substr(line.find_last_of(" ") + 1))));
        }
        else if (line.compare(0, 8, "# rows: ") == 0)
            height = std::stoul(line.substr(8)); // sic: swapped here, swapped back by load() (reference :1327-1336)
        else if (line.compare(0, 11, "# columns: ") == 0)
            width = std::stoul(line.substr(11));
    }
    return shape;
}

void Som::load(const char *filename)
{
    std::ifstream file(filename);
    if (!file.is_open() || !file.good())
    {
        std::cout << "Could not open file " << filename << " for reading. Quitting...\n";
        std::exit(EXIT_FAILURE);
    }
    pull();
    enum Section { None, Mean, Sigma, Weight, Hits, U } section = None;
    auto at = [](const std::string &s, size_t i) { return i < s.size() ? s[i] : '\0'; };
    auto digit = [](char c) { return std::isdigit(static_cast<unsigned char>(c)) != 0; };
    unsigned k = 0, node = 0; // 3-D sections: node index runs fastest, then the dimension
    std::string line;
    // text rows of a 2-D sheet: `width` lines of `height` numbers each, starting at the current line
    auto sheet = [&](auto store) {
        for (unsigned r = 0; r < width; ++r)
        {
            char *cursor = const_cast<char *>(line.c_str());
            for (unsigned c = 0; c < height; ++c)
                store(r * height + c, cursor);
            std::getline(file, line);
        }
    };
    while (!file.eof())
    {
        std::getline(file, line);
        if (at(line, 0) == '#')
        {
            if (line.compare(0, 8, "# name: ") == 0)
            {
                const std::string name = line.substr(8, 20);
                if (name == "som")
                    section = Mean;
                else if (name == "sigmaSom")
                    section = Sigma;
                else if (name == "weightMap")
                    section = Weight;
                else if (name == "bmuHits")
                    section = Hits;
                else if (name == "U")
                    section = U;
                else
                {
                    std::cout << "No name for vector in SOM file!\n";
                    std::exit(EXIT_FAILURE);
                }
            }
            else if (line.compare(0, 8, "# type: ") == 0)
            {
                if (line.compare(8, 20, "matrix") != 0)
                {
                    std::cout << "Incorrect type in SOM file!\n";
                    std::exit(EXIT_FAILURE);
                }
            }
            else if (line.compare(0, 9, "# ndims: ") == 0)
                std::getline(file, line); // the shape line was consumed by getSizeFromFile
            else if (line.compare(0, 8, "# rows: ") == 0)
                width = std::stoul(line.substr(8));
            else if (line.compare(0, 11, "# columns: ") == 0)
                height = std::stoul(line.substr(11));
            continue;
        }
        if ((section == Mean || section == Sigma) && (digit(at(line, 1)) || at(line, 1) == '-'))
        {
            auto &plane = section == Mean ? map : sigmaMap;
            plane[node](static_cast<Eigen::Index>(k)) = static_cast<float>(std::stod(line));
            if (++node >= height * width)
            {
                node = 0;
                if (++k >= static_cast<unsigned>(plane[0].size()))
                {
                    k = 0;
                    section = None;
                }
            }
        }
        else if (section == Weight && digit(at(line, 0)))
            sheet([&](unsigned i, char *&cur) { weightMap(static_cast<Eigen::Index>(i)) = static_cast<float>(std::strtod(cur, &cur)); });
        else if (section == Hits && digit(at(line, 0)))
            sheet([&](unsigned i, char *&cur) { bmuHits[i] = std::strtoul(cur, &cur, 10); });
        else if (section == U && digit(at(line, 0)))
            sheet([&](unsigned i, char *&cur) { uMatrix[i] = std::strtod(cur, &cur); });
    }
    device.reset(); // the file may carry another shape: the next device call builds a fresh context from the mirror
    hostIsStale = false;
    deviceIsStale = true;
}

// reference src/Som.cpp:949-975, same division order; host libm exp() like the kernel's table builder
double Som::calculateNeighbourhoodWeight(const size_t &currentX, const size_t &currentY, const size_t &bmuX, const size_t &bmuY,
                                         const double &currentSigma)
{
    if (currentSigma > 1.0)
    {
        const double dx = static_cast<double>(currentX) - static_cast<double>(bmuX), dy = static_cast<double>(currentY) - static_cast<double>(bmuY);
        return std::exp(-(dx * dx / 2.0 / currentSigma / currentSigma + dy * dy / 2.0 / currentSigma / currentSigma));
    }
    return (currentX == bmuX && currentY == bmuY) ? 1.0 : 0.0;
}
