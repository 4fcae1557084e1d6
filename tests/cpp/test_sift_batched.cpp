// C++ host-mirror self-test of batched SIFT keypoint detection: pcc::SIFTKeypointBatched (include/pcc/grid_search.hpp) against
// pcc::SIFTKeypoint::compute and pcc_first_within on each cluster alone.  Prints PASS and returns 0 when every check holds.
#include <cmath>
#include <cstdio>
#include <cstring>
#include <random>
#include <vector>

#include "../../include/pcc/grid_search.hpp"

using Pt = pcc::PointXYZRGB;
static int failures = 0;
#define CHECK(c, ...) do { if (!(c)) { ++failures; std::printf("FAIL %s:%d ", __FILE__, __LINE__); std::printf(__VA_ARGS__); std::printf("\n"); } } while (0)

// a jittered 4 mm grid of a x b points on z = z0 with a bright Gaussian blob of sigma 0.02 at (cx, cy)
static std::shared_ptr<pcc::PointCloud<Pt> > blob_patch(int a_n, int b_n, float z0, double cx, double cy, unsigned seed) {
    std::mt19937 rng(seed);
    std::uniform_real_distribution<float> j(-0.0004f, 0.0004f);
    auto cloud = std::make_shared<pcc::PointCloud<Pt> >();
    for (int a = 0; a < a_n; ++a)
        for (int b = 0; b < b_n; ++b) {
            Pt p;
            p.x = 0.004f * a + j(rng); p.y = 0.004f * b + j(rng); p.z = z0;
            const double d = std::hypot(p.x - cx, p.y - cy);
            const std::uint8_t c = (std::uint8_t)std::lround(std::fmin(255.0, 128 + 100 * std::exp(-d * d / (2 * 0.02 * 0.02))));
            p.r = p.g = p.b = c; p.a = 255;
            cloud->push_back(p);
        }
    return cloud;
}

static bool same(const pcc::PointWithScale &a, const pcc::PointWithScale &b) { return std::memcmp(&a, &b, sizeof(a)) == 0; }

int main() {
    // two patches that overlap in space, a 12-point cluster (no octave) and an empty cluster
    std::vector<std::shared_ptr<const pcc::PointCloud<Pt> > > clouds = {blob_patch(60, 60, 0.5f, 0.12, 0.12, 5), blob_patch(40, 70, 0.5f, 0.08, 0.14, 6),
                                                                     blob_patch(3, 4, 0.2f, 0.0, 0.0, 7), std::make_shared<pcc::PointCloud<Pt> >()};
    pcc::SIFTKeypointBatched<Pt> batched;
    batched.setInputClouds(clouds);
    batched.setScales(0.005f, 5, 5);
    batched.setMinimumContrast(0.001f);
    std::vector<std::vector<pcc::PointWithScale> > kp;
    std::vector<std::vector<int> > snap;
    batched.compute(kp, &snap, 0.05);
    CHECK(kp.size() == clouds.size() && snap.size() == clouds.size(), "%zu keypoint lists for %zu clusters", kp.size(), clouds.size());
    size_t total = 0;
    for (size_t c = 0; c < clouds.size() && c < kp.size(); ++c) {
        std::vector<pcc::PointWithScale> want;
        if (!clouds[c]->points.empty()) {
            pcc::SIFTKeypoint<Pt> single;
            single.setInputCloud(clouds[c]);
            single.compute(want);
        }
        CHECK(kp[c].size() == want.size(), "cluster %zu: %zu keypoints, alone %zu", c, kp[c].size(), want.size());
        for (size_t i = 0; i < want.size() && i < kp[c].size(); ++i) CHECK(same(kp[c][i], want[i]), "cluster %zu keypoint %zu differs", c, i);
        total += want.size();
        if (want.empty()) { CHECK(snap[c].empty(), "cluster %zu: snaps without keypoints", c); continue; }
        pcc_index *ix = nullptr;
        pcc::check(pcc_create(0, &ix));
        std::vector<int32_t> first(want.size());
        pcc::check(pcc_build(ix, clouds[c]->points.data(), (int64_t)clouds[c]->points.size(), (int)sizeof(Pt), nullptr, 0, 0.05f, 0, PCC_HOST, nullptr));
        pcc::check(pcc_first_within(ix, want.data(), (int64_t)want.size(), (int)sizeof(pcc::PointWithScale), 0.05, first.data(), PCC_HOST, nullptr));
        pcc_destroy(ix);
        CHECK(snap[c].size() == want.size(), "cluster %zu: %zu snaps", c, snap[c].size());
        for (size_t i = 0; i < first.size() && i < snap[c].size(); ++i) CHECK(snap[c][i] == first[i], "cluster %zu snap %zu: %d, alone %d", c, i, snap[c][i], first[i]);
    }
    CHECK(total > 0 && kp.size() == 4 && kp[2].empty() && kp[3].empty(), "%zu keypoints in all", total);
    bool threw = false;
    try { pcc::SIFTKeypointBatched<Pt> b2; b2.setInputClouds(clouds); b2.setScales(0.005f, 5, 14); std::vector<std::vector<pcc::PointWithScale> > k2; b2.compute(k2); }
    catch (const pcc::Error &) { threw = true; }
    CHECK(threw, "14 scales per octave accepted");
    std::printf("%zu clusters: %zu keypoints, identical to the per-cluster calls\n", clouds.size(), total);
    if (failures) { std::printf("%d failures\n", failures); return 1; }
    std::printf("PASS\n");
    return 0;
}
