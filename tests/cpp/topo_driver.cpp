// topo_driver.cpp — drives Som::mapDataSetTopTwo and Som::topographicError (include/SOM.hpp) on a given map and rows.
// tests/test_gpu_top2.py writes the case and checks the output against the topographic error it computes from the oracle's
// distances.
//
// usage: topo_driver <case.bin> <out.bin>
// case.bin: int32 W, H, D, n ; float32 mean[W*H*D] ; float32 x[n*D]   (Standard transformation, sequential summation order)
// out.bin:  float64 topographicError ; uint64 bmu[n] ; float32 dist[n] ; uint64 bmu2[n] ; float32 dist2[n]
#include "DataSet.hpp"
#include "IDataLoader.hpp"
#include "SOM.hpp"
#include "Transformation.hpp"

#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

namespace
{
// the whole row array as one chunk
class RowsLoader : public IDataLoader
{
  public:
    RowsLoader(const float *x, size_t n, size_t depth) : _x{x}, _n{n}, _depth{depth}, _w(depth, 1.0f), _bin(depth, 0), _cont(depth, 1), _names(depth, "c") {}
    size_t load() override
    {
        data.clear();
        for (size_t r = 0; r < _n; ++r)
        {
            RowData row{Eigen::VectorXf(_depth), std::vector<int>(_depth, 1)};
            std::memcpy(row.values.data(), _x + r * _depth, _depth * sizeof(float));
            data.push_back(row);
        }
        return data.size();
    }
    std::vector<RowData> getPreview(size_t) override { return {}; }
    bool open(const char *) override { return true; }
    std::vector<std::string> findAllColumns() override { return _names; }
    void setColumnSpec(const std::vector<ColumnSpec>) noexcept override {}
    const std::vector<ColumnSpec> getColumnSpec() noexcept override { return {}; }
    float getWeight(size_t i) override { return _w[i]; }
    const std::vector<float> getWeights() const noexcept override { return _w; }
    const std::vector<int> &getBinary() const noexcept override { return _bin; }
    const std::vector<int> &getContinuous() const noexcept override { return _cont; }
    std::string getName(size_t i) const noexcept override { return _names[i]; }
    const std::vector<std::string> getNames() const noexcept override { return _names; }
    size_t getDepth() const noexcept override { return _depth; }
    bool isAtStartOfDataStream() const noexcept override { return true; }

  private:
    const float *_x;
    size_t _n, _depth;
    std::vector<float> _w;
    std::vector<int> _bin, _cont;
    std::vector<std::string> _names;
};

// a Som whose model vectors are set directly (the mirror is pushed to the device on the next call)
struct MapSom : Som
{
    MapSom(size_t w, size_t h, size_t d) : Som(w, h, d) {}
    void setMap(const float *mean)
    {
        for (size_t p = 0; p < map.size(); ++p)
            std::memcpy(map[p].data(), mean + p * depth, depth * sizeof(float));
        deviceIsStale = true;
    }
};

template <typename T> void put(FILE *f, const T *p, size_t n) { std::fwrite(p, sizeof(T), n, f); }
} // namespace

int main(int argc, char **argv)
{
    if (argc != 3)
        return 2;
    FILE *in = std::fopen(argv[1], "rb");
    if (!in)
        return 3;
    int32_t h[4];
    if (std::fread(h, sizeof(int32_t), 4, in) != 4)
        return 4;
    const size_t W = static_cast<size_t>(h[0]), H = static_cast<size_t>(h[1]), D = static_cast<size_t>(h[2]), n = static_cast<size_t>(h[3]);
    std::vector<float> mean(W * H * D), x(n * D);
    if (std::fread(mean.data(), sizeof(float), mean.size(), in) != mean.size() || std::fread(x.data(), sizeof(float), x.size(), in) != x.size())
        return 5;
    std::fclose(in);

    MapSom som(W, H, D);
    som.setReductionOrder(0);
    som.setMap(mean.data());
    RowsLoader loader(x.data(), n, D);
    DataSet ds(loader);
    ds.loadNextDataFromStream();

    const double te = som.topographicError(ds);
    std::vector<size_t> bmu, bmu2;
    std::vector<float> dist, dist2;
    som.mapDataSetTopTwo(ds, bmu, dist, bmu2, dist2);
    std::vector<uint64_t> b(bmu.begin(), bmu.end()), b2(bmu2.begin(), bmu2.end());

    FILE *out = std::fopen(argv[2], "wb");
    if (!out)
        return 6;
    put(out, &te, 1);
    put(out, b.data(), n);
    put(out, dist.data(), n);
    put(out, b2.data(), n);
    put(out, dist2.data(), n);
    std::fclose(out);
    return 0;
}
