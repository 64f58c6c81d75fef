// SOM.hpp — class Som with the public surface of the reference (include/SOM.hpp:39-189), re-implemented for
// B200: the model state lives on the GPU behind the C-ABI of vsom_b200.h and the hot methods
//   train / trainBasicSom / trainSingle              -> vsom_train_chunk   (K1F / K1, persistent online-step kernels)
//   train(BatchMap) / trainBatchSom[Epoch]           -> vsom_batch_epoch   (K6)
//   evaluate / measureSimilarity / mapDataSet         -> vsom_find_bmu / vsom_evaluate: batches of >= 1024 rows run the
//                                                        tensor-core candidate search + exact rescore (K2), smaller ones
//                                                        the exact scan (K3); same bits either way
//   mapDataSetTopTwo / topographicError (additions)   -> vsom_find_bmu2 (K2 / K3 in their top-2 mode)
//   linearInitialize (addition)                       -> vsom_linear_init (co-moment pass + subspace iteration, lininit.cu)
//   clusterNodes (addition)                           -> vsom_cluster_nodes (k-means++ seeding + Lloyd over the mean plane, cluster.cu)
//   predictColumns (addition)                         -> vsom_predict_columns (K2 / K3 over the matched columns, predict.cu)
//   findBmu / findRestrictedBmu (one row)             -> vsom_find_bmu      (K3)
//   euclidianWeightedDist / findLocalBmu / findRestrictedBmd -> vsom_all_dists
//   variationalAutoEncoder / autoEncoder              -> vsom_soft_assign + host sampling
//   updateUMatrix / getUMatrix                        -> vsom_update_umatrix (K4)
// forward to it.  Getters read a host mirror that is refreshed from the device on demand.  There is no CPU
// implementation of the hot path behind this class: if the CUDA library cannot run, the methods throw.
//
// save / load / getSizeFromFile / Som(const char*) keep the reference's Octave-text checkpoint format byte for byte
// (host code over the mirror).
//
// Summation order of dot() / squaredNorm() (the one order-dependent operation of the path): by default the order of the
// Eigen this library is compiled against — real Eigen: its SSE2 packet redux (VSOM_ORDER_EIGEN_SSE); the stand-in header
// of include/compat: sequential, or the packet order with -DVSOM_COMPAT_EIGEN_SSE_REDUX.  The environment variable
// VSOM_REDUCTION_ORDER=reference|eigen_sse|lanes, or setReductionOrder(), overrides it.
#pragma once

#include "DataSet.hpp"
#include "SomIndex.hpp"
#include "Transformation.hpp"
#include "UMatrix.hpp"

#include <atomic>
#include <memory>
#include <mutex>
#include <vector>

#include "Eigen/Dense"

#define SIGMA_SWITCH_TO_LOCAL 1

struct vsom_ctx;

class Som
{
  protected:
    struct TrainingReturnValue
    {
        SomIndex bmu;
        Eigen::VectorXf residual;
        float distanceError;
    };
    struct Metrics
    {
        std::vector<float> MeanSquaredError;
        std::vector<float> DistanceError;
        Metrics() : MeanSquaredError{}, DistanceError{} {}
        Metrics(size_t size) : MeanSquaredError(size), DistanceError(size) {}
    };
    Transformation transform;
    // host mirror of the device planes (refreshed lazily; see pull())
    mutable std::vector<Eigen::VectorXf> map;
    mutable std::vector<Eigen::VectorXf> sigmaMap;
    mutable std::vector<Eigen::VectorXf> SMap;
    Metrics metrics;
    mutable Eigen::VectorXf weightMap;
    mutable std::vector<size_t> bmuHits;
    mutable std::vector<double> uMatrix;
    std::atomic<bool> _isTraining;
    size_t height, width, depth;

    void Construct(size_t inWidth, size_t inHeight, size_t inDepth, std::vector<std::string> names);

    // ---- device side
    struct Device; // owns the vsom_ctx
    mutable std::shared_ptr<Device> device;
    mutable bool hostIsStale{false};   // the device holds newer planes than the mirror
    mutable bool deviceIsStale{true};  // the mirror holds planes the device has not seen
    mutable int reductionOrder{-1};    // vsom_reduction_order; -1: the build's default (see the note at the top)
    vsom_ctx *context() const;         // creates the context on first use, pushes the mirror if needed
    void pull() const;                 // refresh the mirror from the device
    size_t inputLength() const;        // sample length the model vector was built for

  public:
    enum class WeigthDecayFunction
    {
        Exponential,
        InverseProportional,
        BatchMap
    };
    std::mutex metricsMutex;

    Som(size_t width, size_t height, DataSet dataset, Transformation transformation = Transformation{}) : transform{transformation}
    {
        Construct(width, height, dataset.vectorLength(), dataset.getNames());
    }
    Som(size_t width, size_t height, size_t depth, Transformation transformation = Transformation{}) : transform{transformation}
    {
        Construct(width, height, depth, std::vector<std::string>{});
    }
    Som(const char *filename);
    Som(const Som &som);
    Som &operator=(const Som &other);
    ~Som();

    void train(DataSet &data, size_t numberOfEpochs, double eta0, double etaDecay, double sigma0, double sigmaDecay,
               WeigthDecayFunction weightDecayFunction, bool updateUMatrixAfterEpoch = false);
    void trainBasicSom(DataSet &data, size_t numberOfEpochs, double eta0, double etaDecay, double sigma0, double sigmaDecay,
                       WeigthDecayFunction weightDecayFunction, bool updateUMatrixAfterEpoch = false);
    void trainBatchSom(DataSet &data, size_t numberOfEpochs, double sigma0, double sigmaDecay, bool updateUMatrixAfterEpoch = false);
    float trainBatchSomEpoch(DataSet &data, double currentSigma, bool isFirst);
    double evaluate(const DataSet &dataset) const;
    TrainingReturnValue trainSingle(const Eigen::VectorXf &v, const Eigen::VectorXf &valid, const Eigen::VectorXf &weights, const double eta,
                                    const double sigma, size_t &lastBMU, const WeigthDecayFunction weightDecayFunction);
    int measureSimilarity(const DataSet *dataset, int numberOfSigmas, size_t minBmuHits) const;
    int autoEncoder(const DataSet *dataset, size_t minBmuHits) const;
    size_t variationalAutoEncoder(const DataSet *dataset, size_t minBmuHits) const;
    SomIndex findBmu(const Eigen::VectorXf &v) const;
    SomIndex findBmu(const Eigen::VectorXf &v, const Eigen::VectorXf &valid, const Eigen::VectorXf &weights) const;
    SomIndex findLocalBmu(const Eigen::VectorXf &v, const Eigen::VectorXf &valid, const size_t &lastBMUref, const Eigen::VectorXf &weights) const;
    SomIndex findRestrictedBmu(const Eigen::VectorXf &v, const Eigen::VectorXf &valid, const size_t minBmuHits, const Eigen::VectorXf &weights) const;
    std::vector<double> findRestrictedBmd(const Eigen::VectorXf &v, const Eigen::VectorXf &valid, size_t minBmuHits, const Eigen::VectorXf &weights) const;
    double euclidianWeightedDist(const SomIndex &pos, const Eigen::VectorXf &v, const Eigen::VectorXf &valid, const Eigen::VectorXf &weights) const;
    double euclidianWeightedDist(const size_t &pos, const Eigen::VectorXf &v, const Eigen::VectorXf &valid, const Eigen::VectorXf &weights) const;
    double euclidianWeightedDistRaw(const size_t &pos, const Eigen::VectorXf &v, const Eigen::VectorXf &valid, const Eigen::VectorXf &weights) const;
    void display() const;
    void displayUMatrix() const;
    UMatrix getUMatrix() const noexcept;
    Eigen::VectorXf getWeigthMap() const noexcept;
    std::vector<size_t> getBmuHits() const noexcept;
    size_t getHeight() const noexcept;
    size_t getWidth() const noexcept;
    size_t getDepth() const noexcept;
    size_t getIndex(SomIndex index) const noexcept;
    Eigen::VectorXf getNeuron(SomIndex index) const noexcept;
    Eigen::VectorXf getNeuron(size_t index) const noexcept;
    Eigen::VectorXf getSigmaNeuron(SomIndex index) const noexcept;
    Eigen::VectorXf getSigmaNeuron(size_t index) const noexcept;
    std::vector<std::string> getNeuronStrings(SomIndex index) const noexcept;
    std::vector<std::string> getSigmaNeuronStrings(SomIndex index) const noexcept;
    float getMaxValueOfFeature(size_t modelVectorIndex) const;
    float getMinValueOfFeature(size_t modelVectorIndex) const;
    float getMaxSigmaOfFeature(size_t modelVectorIndex) const;
    float getMinSigmaOfFeature(size_t modelVectorIndex) const;
    Metrics getMetrics() const noexcept;
    bool isTraining() const noexcept;
    bool isCompatibleWithData(DataSet &data) const noexcept;
    void randomInitialize(int seed, float sigma);
    void addBmu(SomIndex position);
    void updateUMatrix(const Eigen::VectorXf &weights);
    void save(const char *filename) const;
    void load(const char *filename);
    Eigen::VectorXf getSizeFromFile(const char *filename);

    double static calculateNeighbourhoodWeight(const size_t &currentX, const size_t &currentY, const size_t &bmuX, const size_t &bmuY,
                                               const double &currentSigma);

    // ---- additions of this implementation (not in the reference)
    // Batch scoring of the loaded chunk in one device pass: BMU index and distance per row.
    void mapDataSet(const DataSet &dataset, std::vector<size_t> &bmuOut, std::vector<float> &distOut, size_t minBmuHits = 0) const;
    // The same pass with every row's second-best node as well (vsom_find_bmu2): bmuOut / distOut as mapDataSet, bmu2Out / dist2Out the
    // runner-up among the eligible nodes (smallest (distance, index) key, NaN distances last); SIZE_MAX and NaN for rows without one.
    void mapDataSetTopTwo(const DataSet &dataset, std::vector<size_t> &bmuOut, std::vector<float> &distOut, std::vector<size_t> &bmu2Out,
                          std::vector<float> &dist2Out, size_t minBmuHits = 0) const;
    // Topographic error of the loaded chunk (min_hits 0): the share of rows whose best and second-best nodes are not 8-neighbours
    // on the grid (max(|dx|, |dy|) == 1, no wrap-around); rows without a runner-up (a 1 x 1 map) are not errors.  0 for an empty chunk.
    double topographicError(const DataSet &dataset) const;
    // Linear initialisation of the map from the loaded chunk (vsom_linear_init): the mean plane spans the plane of the rows' two
    // principal components, the first axis along the longer side of the grid; S, sigma, weight, hits and the U-matrix are zeroed and
    // the metrics reset, as randomInitialize does.  Standard / Median maps only (a CLR map throws), at least two finite rows.
    void linearInitialize(const DataSet &dataset);
    // k-means over the map's nodes (vsom_cluster_nodes): k-means++ seeding from `seed`, then at most maxIterations Lloyd iterations over
    // the mean plane, each node weighted by 1 or (weightByHits) by its hit count.  labels[N] gets every node's cluster, centroids the k
    // centroids (Dm values each, f64); returns the inertia (the weighted sum of the nodes' f32 distances to their centroids).  Throws
    // on a refused call (k outside 1..N, a non-finite plane, fewer than k distinct nodes carrying weight).  Reads the map only.
    double clusterNodes(size_t k, std::vector<int> &labels, std::vector<Eigen::VectorXd> &centroids, uint64_t seed = 0, bool weightByHits = false,
                        int maxIterations = 300) const;
    // Prediction of unobserved columns for the loaded chunk (vsom_predict_columns): each row's BMU over the columns whose matchColumns
    // entry is true (bmuOut / distOut, as mapDataSet on a map of those columns only), and that node's mean and sigma at the other
    // columns, q = getDepth() - (matched columns) values per row in ascending column order (meanOut / sigmaOut, n * q).  The rows'
    // unmatched columns are never read.  Throws on a CLR map, on a mask whose length is not getDepth() and on a mask with no matched
    // column.  Reads the map only.
    void predictColumns(const DataSet &dataset, const std::vector<bool> &matchColumns, std::vector<size_t> &bmuOut, std::vector<float> &distOut,
                        std::vector<float> &meanOut, std::vector<float> &sigmaOut, size_t minBmuHits = 0) const;
    // Rows grouped by BMU: counts[N], offsets[N+1], rowIds[n] (the "SomIndex build").
    void buildIndex(const std::vector<size_t> &bmu, std::vector<size_t> &counts, std::vector<size_t> &offsets, std::vector<unsigned> &rowIds) const;
    // Summation order of the distances (vsom_reduction_order of vsom_b200.h): 0 sequential, 1 lanes (online step only, near-tie
    // rule), 2 Eigen's SSE2 packet order.  Re-creates the device context on the next call.
    void setReductionOrder(int order);
    int getReductionOrder() const;
    void setFastReductionOrder(bool lanes); // kept from round 1: lanes ? order 1 : order 0
};
