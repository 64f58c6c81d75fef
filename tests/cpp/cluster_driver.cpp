// cluster_driver.cpp — trains a small map through Som (include/SOM.hpp) on a MemoryDataLoader, then calls Som::clusterNodes.
// tests/test_gpu_cluster.py uploads the trained state into a binding context, calls cluster_nodes there and compares.
//
// usage: cluster_driver <case.bin> <state.bin>
// case.bin:  int32 W, H, Din, transform, order, n, chunk, k, weightByHits, maxIterations ; uint64 seed ;
//            float64 eta0, etaDecay, sigma0, sigmaDecay ; float32 x[n*Din]   (one online epoch, Exponential decay)
// state.bin: float32 mean[N*Dm] ; float32 sigma[N*Dm] ; float32 weight[N] ; uint64 hits[N] of the trained map
// stdout:    "inertia <%a>", "labels <N ints>", then k lines "centroid <j> <Dm values %a>"
#include "DataSet.hpp"
#include "MemoryDataLoader.hpp"
#include "SOM.hpp"
#include "Transformation.hpp"

#include <cstdint>
#include <cstdio>
#include <vector>

int main(int argc, char **argv)
{
    if (argc != 3)
        return 2;
    FILE *in = std::fopen(argv[1], "rb");
    if (!in)
        return 3;
    int32_t h[10];
    uint64_t seed = 0;
    double sched[4];
    if (std::fread(h, sizeof(int32_t), 10, in) != 10 || std::fread(&seed, sizeof(seed), 1, in) != 1 || std::fread(sched, sizeof(double), 4, in) != 4)
        return 4;
    const size_t W = static_cast<size_t>(h[0]), H = static_cast<size_t>(h[1]), Din = static_cast<size_t>(h[2]), n = static_cast<size_t>(h[5]),
                 chunk = static_cast<size_t>(h[6]), k = static_cast<size_t>(h[7]);
    const int transform = h[3], order = h[4], byHits = h[8], maxIterations = h[9];
    std::vector<float> x(n * Din);
    if (std::fread(x.data(), sizeof(float), x.size(), in) != x.size())
        return 5;
    std::fclose(in);

    std::vector<std::string> names;
    Transformation t = transform == 1 ? Transformation::StandardMedianEstimator(names)
                       : transform == 2 ? Transformation::CombinatorialLinearRegression(names)
                                        : Transformation::Standard(names);
    Som som(W, H, t.Length(Din), t);
    som.setReductionOrder(order);
    som.randomInitialize(7, 1.0f);
    MemoryDataLoader loader(x.data(), n, Din, chunk);
    DataSet rows(loader);
    som.train(rows, 1, sched[0], sched[1], sched[2], sched[3], Som::WeigthDecayFunction::Exponential, false);

    std::vector<int> labels;
    std::vector<Eigen::VectorXd> centroids;
    const double inertia = som.clusterNodes(k, labels, centroids, seed, byHits != 0, maxIterations);

    const size_t N = W * H, Dm = som.getDepth();
    FILE *out = std::fopen(argv[2], "wb");
    if (!out)
        return 6;
    for (int plane = 0; plane < 2; ++plane)
        for (size_t p = 0; p < N; ++p)
        {
            const Eigen::VectorXf v = plane == 0 ? som.getNeuron(p) : som.getSigmaNeuron(p);
            std::fwrite(v.data(), sizeof(float), Dm, out);
        }
    const Eigen::VectorXf wm = som.getWeigthMap();
    std::fwrite(wm.data(), sizeof(float), N, out);
    for (size_t v : som.getBmuHits())
    {
        const uint64_t u = v;
        std::fwrite(&u, sizeof(u), 1, out);
    }
    std::fclose(out);

    std::printf("inertia %a\nlabels", inertia);
    for (int l : labels)
        std::printf(" %d", l);
    std::printf("\n");
    for (size_t j = 0; j < k; ++j)
    {
        std::printf("centroid %zu", j);
        for (Eigen::Index c = 0; c < centroids[j].size(); ++c)
            std::printf(" %a", centroids[j](c));
        std::printf("\n");
    }
    return 0;
}
