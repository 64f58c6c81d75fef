// predict_driver.cpp — trains a small map through Som (include/SOM.hpp) on a MemoryDataLoader, then calls Som::predictColumns on the
// same rows.  tests/test_gpu_predict_columns.py uploads the trained state into a binding context, calls predict_columns there and
// compares.
//
// usage: predict_driver <case.bin> <state.bin> <out.bin>
// case.bin:  int32 W, H, Din, transform, order, n, chunk, minHits ; float64 eta0, etaDecay, sigma0, sigmaDecay ;
//            uint8 match[Dm] ; float32 x[n*Din]   (one online epoch, Exponential decay)
// state.bin: float32 mean[N*Dm] ; float32 sigma[N*Dm] ; float32 weight[N] ; uint64 hits[N] of the trained map
// out.bin:   uint64 bmu[n] ; float32 dist[n] ; float32 mean[n*q] ; float32 sigma[n*q]
// exit code 0; 7 when predictColumns threw (the message goes to stderr)
#include "DataSet.hpp"
#include "MemoryDataLoader.hpp"
#include "SOM.hpp"
#include "Transformation.hpp"

#include <cstdint>
#include <cstdio>
#include <exception>
#include <vector>

int main(int argc, char **argv)
{
    if (argc != 4)
        return 2;
    FILE *in = std::fopen(argv[1], "rb");
    if (!in)
        return 3;
    int32_t h[8];
    double sched[4];
    if (std::fread(h, sizeof(int32_t), 8, in) != 8 || std::fread(sched, sizeof(double), 4, in) != 4)
        return 4;
    const size_t W = static_cast<size_t>(h[0]), H = static_cast<size_t>(h[1]), Din = static_cast<size_t>(h[2]), n = static_cast<size_t>(h[5]),
                 chunk = static_cast<size_t>(h[6]), minHits = static_cast<size_t>(h[7]);
    const int transform = h[3], order = h[4];
    std::vector<std::string> names;
    Transformation t = transform == 1 ? Transformation::StandardMedianEstimator(names)
                       : transform == 2 ? Transformation::CombinatorialLinearRegression(names)
                                        : Transformation::Standard(names);
    const size_t Dm = t.Length(Din);
    std::vector<uint8_t> m(Dm);
    std::vector<float> x(n * Din);
    if (std::fread(m.data(), 1, Dm, in) != Dm || std::fread(x.data(), sizeof(float), x.size(), in) != x.size())
        return 5;
    std::fclose(in);

    Som som(W, H, Dm, t);
    som.setReductionOrder(order);
    som.randomInitialize(7, 1.0f);
    {
        MemoryDataLoader loader(x.data(), n, Din, chunk);
        DataSet rows(loader);
        som.train(rows, 1, sched[0], sched[1], sched[2], sched[3], Som::WeigthDecayFunction::Exponential, false);
    }

    MemoryDataLoader loader(x.data(), n, Din, n);
    DataSet rows(loader);
    rows.loadNextDataFromStream();
    std::vector<bool> match(m.begin(), m.end());
    std::vector<size_t> bmu;
    std::vector<float> dist, mean, sigma;
    try
    {
        som.predictColumns(rows, match, bmu, dist, mean, sigma, minHits);
    }
    catch (const std::exception &e)
    {
        std::fprintf(stderr, "%s\n", e.what());
        return 7;
    }

    const size_t N = W * H;
    FILE *st = std::fopen(argv[2], "wb");
    if (!st)
        return 6;
    for (int plane = 0; plane < 2; ++plane)
        for (size_t p = 0; p < N; ++p)
        {
            const Eigen::VectorXf v = plane == 0 ? som.getNeuron(p) : som.getSigmaNeuron(p);
            std::fwrite(v.data(), sizeof(float), Dm, st);
        }
    const Eigen::VectorXf wm = som.getWeigthMap();
    std::fwrite(wm.data(), sizeof(float), N, st);
    for (size_t v : som.getBmuHits())
    {
        const uint64_t u = v;
        std::fwrite(&u, sizeof(u), 1, st);
    }
    std::fclose(st);

    FILE *out = std::fopen(argv[3], "wb");
    if (!out)
        return 6;
    for (size_t b : bmu)
    {
        const uint64_t u = b;
        std::fwrite(&u, sizeof(u), 1, out);
    }
    std::fwrite(dist.data(), sizeof(float), dist.size(), out);
    std::fwrite(mean.data(), sizeof(float), mean.size(), out);
    std::fwrite(sigma.data(), sizeof(float), sigma.size(), out);
    std::fclose(out);
    return 0;
}
