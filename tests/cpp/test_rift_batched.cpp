// C++ host-mirror self-test of batched processRIFT: pcc::processRIFTBatched (include/pcc/grid_search.hpp) against the per-cluster
// chain pcc::NormalEstimation (radius) -> drop NaN normals -> pcc::IntensityGradientEstimation -> pcc::RIFTEstimation -> drop the
// rows with a non-finite bin.  Prints PASS and returns 0 when every check holds.
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

// n points uniform in a side x side square around (x0, y0), on a gentle bump, random colours
static std::shared_ptr<Cloud> patch(int n, float side, float x0, float y0, unsigned seed) {
    std::mt19937 rng(seed);
    std::uniform_real_distribution<float> u(-0.5f * side, 0.5f * side);
    std::uniform_int_distribution<int> col(0, 255);
    auto cloud = std::make_shared<Cloud>();
    for (int i = 0; i < n; ++i) {
        Pt p;
        p.x = x0 + u(rng); p.y = y0 + u(rng); p.z = 0.5f + 0.2f * (p.x - x0) * (p.x - x0) + 0.1f * std::sin(20.f * p.y);
        p.r = (std::uint8_t)col(rng); p.g = (std::uint8_t)col(rng); p.b = (std::uint8_t)col(rng); p.a = 255;
        cloud->push_back(p);
    }
    return cloud;
}

// processRIFT on one cluster through the single-cluster classes
static void per_cluster(const std::shared_ptr<const Cloud> &cloud, int nd, int ng, std::vector<pcc::Histogram32> &desc, std::vector<int> &kept) {
    desc.clear(); kept.clear();
    if (cloud->points.empty()) return;
    pcc::NormalEstimation<Pt> ne;
    ne.setInputCloud(cloud); ne.setRadiusSearch(0.03);
    std::vector<pcc::Normal> normals;
    ne.compute(normals);
    auto filtered = std::make_shared<Cloud>();
    std::vector<pcc::Normal> nrm1;
    std::vector<float> inten;
    std::vector<int> keep1;
    for (size_t i = 0; i < normals.size(); ++i) {
        const pcc::Normal &m = normals[i];
        if (!std::isfinite(m.normal_x) || !std::isfinite(m.normal_y) || !std::isfinite(m.normal_z)) continue;
        const Pt &p = cloud->points[i];
        filtered->push_back(p); nrm1.push_back(m); inten.push_back(pcc::rgbToIntensity(p.r, p.g, p.b)); keep1.push_back((int)i);
    }
    if (filtered->points.empty()) return;
    auto tree = std::make_shared<pcc::search::GridSearch<Pt> >();
    pcc::IntensityGradientEstimation<Pt> ge;
    ge.setSearchMethod(tree); ge.setInputCloud(filtered); ge.setInputNormals(&nrm1); ge.setInputIntensities(&inten); ge.setRadiusSearch(0.03);
    std::vector<pcc::IntensityGradient> grad;
    ge.compute(grad);
    pcc::RIFTEstimation<Pt> re;
    re.setSearchMethod(tree); re.setInputCloud(filtered); re.setInputGradient(&grad); re.setRadiusSearch(0.05);
    re.setNrDistanceBins(nd); re.setNrGradientBins(ng);
    std::vector<pcc::Histogram32> h;
    re.compute(h);
    for (size_t i = 0; i < h.size(); ++i) {
        bool ok = true;
        for (int k = 0; k < nd * ng; ++k) ok = ok && std::isfinite(h[i].histogram[k]);
        if (ok) { desc.push_back(h[i]); kept.push_back(keep1[i]); }
    }
}

int main() {
    // two clusters that overlap in space, a sparse one (drops at both stages), a 2-point cluster and an empty cluster
    std::vector<std::shared_ptr<const Cloud> > clusters = {patch(700, 0.12f, 0.f, 0.f, 5), patch(500, 0.10f, 0.03f, 0.01f, 6),
                                                           patch(200, 0.40f, 0.f, 0.f, 7), patch(2, 0.01f, 0.3f, 0.3f, 8), std::make_shared<Cloud>()};
    size_t total = 0;
    int dropped = 0;
    for (int shape = 0; shape < 2; ++shape) {
        const int nd = shape ? 3 : 4, ng = shape ? 7 : 8;
        std::vector<std::vector<pcc::Histogram32> > desc;
        std::vector<std::vector<int> > kept;
        pcc::processRIFTBatched<Pt>(clusters, desc, kept, 0.03, 0.03, 0.05, nd, ng);
        CHECK(desc.size() == clusters.size() && kept.size() == clusters.size(), "%zu descriptor lists for %zu clusters", desc.size(), clusters.size());
        for (size_t c = 0; c < clusters.size() && c < desc.size(); ++c) {
            std::vector<pcc::Histogram32> want;
            std::vector<int> want_rows;
            per_cluster(clusters[c], nd, ng, want, want_rows);
            CHECK(desc[c].size() == want.size() && kept[c] == want_rows, "%dx%d cluster %zu: %zu descriptors, alone %zu", nd, ng, c, desc[c].size(), want.size());
            for (size_t i = 0; i < want.size() && i < desc[c].size(); ++i)
                CHECK(std::memcmp(&desc[c][i], &want[i], sizeof(pcc::Histogram32)) == 0, "%dx%d cluster %zu descriptor %zu differs", nd, ng, c, i);
            if (shape == 0) { total += want.size(); dropped += (int)(clusters[c]->points.size() - want.size()); }
        }
        CHECK(desc.size() == 5 && desc[4].empty() && desc[0].size() > 600, "cluster sizes");
    }
    CHECK(dropped > 0, "no row dropped");
    bool threw = false;
    try { std::vector<std::vector<pcc::Histogram32> > d; std::vector<std::vector<int> > k; pcc::processRIFTBatched<Pt>(clusters, d, k, 0.03, 0.03, 0.05, 4, 9); }
    catch (const pcc::Error &) { threw = true; }
    CHECK(threw, "4 x 9 bins accepted");
    std::printf("%zu clusters: %zu descriptors (%d rows dropped), identical to the per-cluster chain\n", clusters.size(), total, dropped);
    if (failures) { std::printf("%d failures\n", failures); return 1; }
    std::printf("PASS\n");
    return 0;
}
