// C++ host-mirror self-test of SIFT keypoint detection: pcc::SIFTKeypoint (include/pcc/grid_search.hpp) through the C ABI, on
// known answers.  Prints PASS and returns 0 when every check holds.
#include <cmath>
#include <cstdio>
#include <random>
#include <vector>

#include "../../include/pcc/grid_search.hpp"

using Pt = pcc::PointXYZRGB;
static int failures = 0;
#define CHECK(c, ...) do { if (!(c)) { ++failures; std::printf("FAIL %s:%d ", __FILE__, __LINE__); std::printf(__VA_ARGS__); std::printf("\n"); } } while (0)

// a jittered 4 mm grid on z = 0.5 carrying a bright (+100) and a dark (-100) grey Gaussian blob of sigma 0.02
static std::shared_ptr<pcc::PointCloud<Pt> > blob_plane(bool constant) {
    std::mt19937 rng(5);
    std::uniform_real_distribution<float> j(-0.0004f, 0.0004f);
    auto cloud = std::make_shared<pcc::PointCloud<Pt> >();
    const double sb = 0.02;
    for (int a = 0; a < 100; ++a)
        for (int b = 0; b < 100; ++b) {
            Pt p;
            p.x = 0.004f * a + j(rng); p.y = 0.004f * b + j(rng); p.z = 0.5f;
            const double d1 = std::hypot(p.x - 0.12, p.y - 0.2), d2 = std::hypot(p.x - 0.28, p.y - 0.2);
            const double v = 128 + 100 * std::exp(-d1 * d1 / (2 * sb * sb)) - 100 * std::exp(-d2 * d2 / (2 * sb * sb));
            const std::uint8_t c = constant ? 1 : (std::uint8_t)std::lround(std::fmin(255.0, std::fmax(0.0, v)));
            p.r = p.g = p.b = c; p.a = 255;
            cloud->push_back(p);
        }
    return cloud;
}

int main() {
    {   // constant value 1.0: every response is exactly 1, the DoG is 0 and nothing is a keypoint
        pcc::SIFTKeypoint<Pt> sift;
        sift.setInputCloud(blob_plane(true));
        std::vector<pcc::PointWithScale> kp;
        sift.compute(kp);
        CHECK(kp.empty(), "constant cloud gave %zu keypoints", kp.size());
    }
    auto cloud = blob_plane(false);
    pcc::SIFTKeypoint<Pt> sift;
    auto tree = std::make_shared<pcc::search::GridSearch<Pt> >();
    sift.setSearchMethod(tree);
    sift.setScales(0.005f, 5, 5);
    sift.setMinimumContrast(0.001f);
    sift.setInputCloud(cloud);
    std::vector<pcc::PointWithScale> kp;
    sift.compute(kp);
    CHECK(!kp.empty(), "no keypoints on the blob plane");
    // every scale is an entry of an octave table (columns 1 .. nr_scales_per_octave), and each blob has a keypoint near its centre
    // at the blob's sigma (octave base 0.02, column 1)
    int near_bright = 0, near_dark = 0;
    for (const auto &k : kp) {
        bool in_table = false;
        for (float base = 0.005f; base < 0.1f; base *= 2)
            for (int i = 1; i <= 5; ++i) in_table |= k.scale == base * powf(2.0f, (1.0f * (float)i - 1.0f) / 5.0f);
        CHECK(in_table, "scale %g is not a table entry", k.scale);
        if (k.scale == 0.02f && std::hypot(k.x - 0.12, k.y - 0.2) < 0.02) ++near_bright;
        if (k.scale == 0.02f && std::hypot(k.x - 0.28, k.y - 0.2) < 0.02) ++near_dark;
    }
    CHECK(near_bright > 0 && near_dark > 0, "blob centres: %d bright, %d dark keypoints at scale 0.02", near_bright, near_dark);
    // cap convention: the full count always, at most cap rows written, the same leading rows
    {
        pcc_index *ws = nullptr;
        pcc::check(pcc_create(0, &ws));
        std::vector<pcc::PointWithScale> few(3);
        int64_t found = -1;
        pcc::check(pcc_sift_keypoints(ws, cloud->points.data(), (int64_t)cloud->points.size(), (int)sizeof(Pt), 16, 0.005f, 5, 5, 0.001f,
                                      reinterpret_cast<float *>(few.data()), 3, &found, PCC_HOST, nullptr));
        pcc_destroy(ws);
        CHECK(found == (int64_t)kp.size(), "capped call counted %lld, full call %zu", (long long)found, kp.size());
        for (int i = 0; i < 3 && i < (int)kp.size(); ++i)
            CHECK(few[i].x == kp[i].x && few[i].y == kp[i].y && few[i].z == kp[i].z && few[i].scale == kp[i].scale, "capped row %d differs", i);
    }
    bool threw = false;
    try { pcc::SIFTKeypoint<Pt> s2; s2.setInputCloud(cloud); s2.setScales(0.005f, 5, 14); std::vector<pcc::PointWithScale> k2; s2.compute(k2); }
    catch (const pcc::Error &) { threw = true; }
    CHECK(threw, "14 scales per octave accepted");
    std::printf("blob plane: %zu keypoints, %d at the bright centre, %d at the dark centre\n", kp.size(), near_bright, near_dark);
    if (failures) { std::printf("%d failures\n", failures); return 1; }
    std::printf("PASS\n");
    return 0;
}
