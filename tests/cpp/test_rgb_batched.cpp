// C++ host-mirror self-test of batched colour segmentation: pcc::findPointNeighboursBatched and pcc::RegionGrowingRGBBatched
// (include/pcc/grid_search.hpp) against per-cluster pcc::findPointNeighbours and pcc::RegionGrowingRGB, and pcc::RegionGrowingRGB on a
// cluster under 100 points against pcc_region_growing_rgb called on its stride-100 table.  Prints PASS and returns 0 when every check holds.
#include <cmath>
#include <cstdio>
#include <cstring>
#include <random>
#include <vector>

#include "../../include/pcc/grid_search.hpp"

using Pt = pcc::PointXYZRGB;
using Cloud = pcc::PointCloud<Pt>;
static int failures = 0;
#define CHECK(c, ...) do { if (!(c)) { ++failures; std::printf("FAIL %s:%d ", __FILE__, __LINE__); std::printf(__VA_ARGS__); std::printf("\n"); } } while (0)

// n points uniform in a side x side square around (x0, y0); `stripes` vertical colour stripes (distinct base colours, +-1 jitter)
static std::shared_ptr<Cloud> patch(int n, float side, float x0, float y0, int stripes, unsigned seed) {
    static const int base[4][3] = {{200, 60, 60}, {60, 60, 200}, {60, 200, 60}, {200, 200, 60}};
    std::mt19937 rng(seed);
    std::uniform_real_distribution<float> u(0.f, 1.f);
    std::uniform_int_distribution<int> jit(-1, 1);
    auto cloud = std::make_shared<Cloud>();
    for (int i = 0; i < n; ++i) {
        Pt p;
        const float fx = u(rng), fy = u(rng);
        p.x = x0 + side * (fx - 0.5f); p.y = y0 + side * (fy - 0.5f); p.z = 0.5f + 0.05f * std::sin(7.f * p.x);
        const int s = std::min((int)(fx * stripes), stripes - 1);
        p.r = (std::uint8_t)(base[s][0] + jit(rng)); p.g = (std::uint8_t)(base[s][1] + jit(rng)); p.b = (std::uint8_t)(base[s][2] + jit(rng)); p.a = 255;
        cloud->push_back(p);
    }
    return cloud;
}

static std::vector<pcc::PointIndices> per_cluster(const std::shared_ptr<const Cloud> &cloud, int min_size) {
    pcc::RegionGrowingRGB<Pt> rg;
    rg.setInputCloud(cloud);
    rg.setDistanceThreshold(10); rg.setPointColorThreshold(6); rg.setRegionColorThreshold(5); rg.setMinClusterSize(min_size);
    std::vector<pcc::PointIndices> out;
    rg.extract(out);
    return out;
}

int main() {
    std::vector<std::shared_ptr<const Cloud> > clusters;
    clusters.push_back(patch(800, 0.4f, 0.f, 0.f, 3, 1));
    clusters.push_back(std::make_shared<Cloud>());                                  // empty
    clusters.push_back(patch(60, 0.1f, 0.1f, 0.f, 2, 2));                           // 60 points, two colours (under the table's 100 columns)
    clusters.push_back(patch(500, 0.3f, 0.05f, 0.02f, 2, 3));                       // overlaps the first cluster in space
    clusters.push_back(patch(300, 0.3f, 40.f, 5.f, 4, 4));                          // far away
    const std::shared_ptr<const Cloud> &small = clusters[2];

    // findPointNeighboursBatched == findPointNeighbours per cluster, bit for bit
    for (int k : {16, 100}) {
        std::vector<std::vector<int> > nb; std::vector<std::vector<float> > nd;
        const std::vector<int> keff = pcc::findPointNeighboursBatched<Pt>(clusters, k, nb, nd);
        CHECK(keff.size() == clusters.size(), "k_eff size %zu", keff.size());
        for (size_t c = 0; c < clusters.size(); ++c) {
            const int n = (int)clusters[c]->points.size();
            CHECK(keff[c] == std::min(k, n), "k=%d cluster %zu: k_eff %d", k, c, keff[c]);
            if (n == 0) { CHECK(nb[c].empty(), "empty cluster has rows"); continue; }
            auto tree = std::make_shared<pcc::search::GridSearch<Pt> >();
            tree->setKHint(k); tree->setInputCloud(clusters[c]);
            std::vector<int> ni; std::vector<float> di;
            pcc::findPointNeighbours(*tree, k, ni, di);
            CHECK(ni == nb[c] && di.size() == nd[c].size() && std::memcmp(di.data(), nd[c].data(), di.size() * 4) == 0, "k=%d cluster %zu: tables differ", k, c);
        }
    }

    // RegionGrowingRGB on the 60-point cluster == pcc_region_growing_rgb over the stride-100 table findPointNeighbours fills
    {
        pcc::search::GridSearch<Pt> tree;
        tree.setKHint(100); tree.setInputCloud(small);
        std::vector<int> ni; std::vector<float> di;
        pcc::findPointNeighbours(tree, 100, ni, di);
        const int n = (int)small->points.size();
        std::vector<int32_t> lab((size_t)n);
        int64_t nc = 0;
        const uint32_t *rgba = reinterpret_cast<const uint32_t *>(reinterpret_cast<const char *>(small->points.data()) + 16);
        pcc::check(pcc_region_growing_rgb(ni.data(), di.data(), n, 100, rgba, (int)sizeof(Pt), 10.f, 6.f, 5.f, 30, 10, std::numeric_limits<int>::max(), lab.data(), &nc));
        const std::vector<pcc::PointIndices> got = per_cluster(small, 10);
        std::vector<int32_t> from_class((size_t)n, -1);
        for (size_t j = 0; j < got.size(); ++j)
            for (int i : got[j].indices) from_class[(size_t)i] = (int32_t)j;
        CHECK(nc == 2 && got.size() == 2, "60-point cluster: %lld colour clusters from the table, %zu from RegionGrowingRGB", (long long)nc, got.size());
        for (int i = 0; i < n; ++i)
            CHECK(from_class[(size_t)i] == lab[(size_t)i], "60-point cluster: point %d in cluster %d, the table says %d", i, from_class[(size_t)i], lab[(size_t)i]);
    }

    // RegionGrowingRGBBatched == RegionGrowingRGB per cluster
    for (int min_size : {10, 200}) {
        pcc::RegionGrowingRGBBatched<Pt> rb;
        rb.setInputClouds(clusters);
        rb.setDistanceThreshold(10); rb.setPointColorThreshold(6); rb.setRegionColorThreshold(5); rb.setMinClusterSize(min_size);
        std::vector<std::vector<pcc::PointIndices> > out;
        rb.extract(out);
        CHECK(out.size() == clusters.size(), "%zu results", out.size());
        size_t split = 0;
        for (size_t c = 0; c < clusters.size() && c < out.size(); ++c) {
            const std::vector<pcc::PointIndices> want = clusters[c]->points.empty() ? std::vector<pcc::PointIndices>() : per_cluster(clusters[c], min_size);
            bool same = want.size() == out[c].size();
            for (size_t j = 0; same && j < want.size(); ++j) same = want[j].indices == out[c][j].indices;
            CHECK(same, "min %d cluster %zu: %zu colour clusters batched, %zu alone", min_size, c, out[c].size(), want.size());
            split += out[c].size() >= 2;
        }
        CHECK(split >= 2, "min %d: only %zu clusters split by colour", min_size, split);
    }

    if (failures) { std::printf("%d failures\n", failures); return 1; }
    std::printf("PASS\n");
    return 0;
}
