// lininit_driver.cpp — drives Som::linearInitialize (include/SOM.hpp) on a MemoryDataLoader, then one epoch of Som::train from the
// initialised map.  tests/test_gpu_linear_init.py writes the case and compares the output with the binding's linear_init followed
// by the oracle's training.
//
// usage: lininit_driver <case.bin> <out.bin>
// case.bin: int32 W, H, Din, transform, n, chunk ; float64 eta0, etaDecay, sigma0, sigmaDecay ; float32 x[n*Din]
//           (sequential summation order, Exponential decay)
// out.bin:  int32 status (0: initialised; 1: linearInitialize threw — nothing follows) ; then, after the initialisation,
//           float32 mean[N*Dm] ; float32 sigma[N*Dm] ; float32 weight[N] ; uint64 hits[N] ; float64 umatrix[N] ; uint64 metrics length ;
//           and after the epoch: float32 mse[1] ; float32 mean[N*Dm] ; float32 sigma[N*Dm] ; float32 weight[N] ; uint64 hits[N]
#include "DataSet.hpp"
#include "MemoryDataLoader.hpp"
#include "SOM.hpp"
#include "Transformation.hpp"

#include <cstdint>
#include <cstdio>
#include <exception>
#include <vector>

namespace
{
template <typename T> void put(FILE *f, const T *p, size_t n) { std::fwrite(p, sizeof(T), n, f); }

void putState(FILE *f, const Som &som)
{
    const size_t N = som.getWidth() * som.getHeight();
    for (size_t p = 0; p < N; ++p)
    {
        const Eigen::VectorXf m = som.getNeuron(p);
        put(f, m.data(), static_cast<size_t>(m.size()));
    }
    for (size_t p = 0; p < N; ++p)
    {
        const Eigen::VectorXf s = som.getSigmaNeuron(p);
        put(f, s.data(), static_cast<size_t>(s.size()));
    }
    const Eigen::VectorXf wm = som.getWeigthMap();
    put(f, wm.data(), static_cast<size_t>(wm.size()));
    for (size_t v : som.getBmuHits())
    {
        const uint64_t u = v;
        put(f, &u, 1);
    }
}
} // namespace

int main(int argc, char **argv)
{
    if (argc != 3)
        return 2;
    FILE *in = std::fopen(argv[1], "rb");
    if (!in)
        return 3;
    int32_t h[6];
    double sched[4];
    if (std::fread(h, sizeof(int32_t), 6, in) != 6 || std::fread(sched, sizeof(double), 4, in) != 4)
        return 4;
    const size_t W = static_cast<size_t>(h[0]), H = static_cast<size_t>(h[1]), Din = static_cast<size_t>(h[2]), n = static_cast<size_t>(h[4]),
                 chunk = static_cast<size_t>(h[5]);
    const int transform = h[3];
    std::vector<float> x(n * Din);
    if (std::fread(x.data(), sizeof(float), x.size(), in) != x.size())
        return 5;
    std::fclose(in);

    std::vector<std::string> names;
    Transformation t = transform == 1 ? Transformation::StandardMedianEstimator(names)
                       : transform == 2 ? Transformation::CombinatorialLinearRegression(names)
                                        : Transformation::Standard(names);
    Som som(W, H, t.Length(Din), t);
    som.setReductionOrder(0);
    MemoryDataLoader initLoader(x.data(), n, Din);
    DataSet initRows(initLoader);
    initRows.loadNextDataFromStream();

    FILE *out = std::fopen(argv[2], "wb");
    if (!out)
        return 6;
    int32_t status = 0;
    try
    {
        som.linearInitialize(initRows);
    }
    catch (const std::exception &)
    {
        status = 1;
    }
    put(out, &status, 1);
    if (status)
    {
        std::fclose(out);
        return 0;
    }
    putState(out, som);
    const UMatrix um = som.getUMatrix();
    put(out, um.getData().data(), um.getData().size());
    const uint64_t metricsLength = som.getMetrics().MeanSquaredError.size();
    put(out, &metricsLength, 1);

    MemoryDataLoader trainLoader(x.data(), n, Din, chunk);
    DataSet trainRows(trainLoader);
    som.train(trainRows, 1, sched[0], sched[1], sched[2], sched[3], Som::WeigthDecayFunction::Exponential, false);
    const auto metrics = som.getMetrics();
    put(out, metrics.MeanSquaredError.data(), metrics.MeanSquaredError.size());
    putState(out, som);
    std::fclose(out);
    return 0;
}
