// C++ host-mirror self-test of the descriptor stage: pcc::IntensityGradientEstimation and pcc::RIFTEstimation (include/pcc/grid_search.hpp)
// through the C ABI, checked against an in-test brute force.  Prints PASS and returns 0 when every check holds.
#include <cmath>
#include <cstdio>
#include <random>
#include <vector>

#include "../../include/pcc/grid_search.hpp"

using Pt = pcc::PointXYZ;
static int failures = 0;
#define CHECK(c, ...) do { if (!(c)) { ++failures; std::printf("FAIL %s:%d ", __FILE__, __LINE__); std::printf(__VA_ARGS__); std::printf("\n"); } } while (0)

static float d2f(const Pt &a, const Pt &b) { const float dx = a.x - b.x, dy = a.y - b.y, dz = a.z - b.z; return (dx * dx + dy * dy) + dz * dz; }

int main() {
    std::mt19937 rng(7);
    std::uniform_real_distribution<float> u(0.f, 0.3f);
    auto cloud = std::make_shared<pcc::PointCloud<Pt> >();
    const int n = 3000;
    for (int i = 0; i < n; ++i) cloud->push_back(Pt(u(rng), u(rng), 0.5f));          // an exactly planar patch on z = 0.5
    // linear intensity over the plane, built from colours like the reference's XYZRGB -> XYZI step
    const double ax = 200.0, ay = -120.0;
    std::vector<float> inten(n);
    for (int i = 0; i < n; ++i) {
        const double v = 100.0 + ax * cloud->points[i].x + ay * cloud->points[i].y;
        const std::uint8_t r = (std::uint8_t)std::lround(std::fmin(255.0, std::fmax(0.0, v)));
        inten[i] = v - r + pcc::rgbToIntensity(r, r, r);           // grey: 0.299 r + 0.587 r + 0.114 r == r up to rounding
    }
    CHECK(std::fabs(pcc::rgbToIntensity(255, 255, 255) - 255.f) < 1e-4f, "rgbToIntensity(255,255,255)");
    CHECK(pcc::rgbToIntensity(1, 0, 0) == 0.299f && pcc::rgbToIntensity(0, 1, 0) == 0.587f && pcc::rgbToIntensity(0, 0, 1) == 0.114f, "rgbToIntensity weights");

    auto tree = std::make_shared<pcc::search::GridSearch<Pt> >();
    pcc::NormalEstimation<Pt> ne;
    ne.setSearchMethod(tree); ne.setInputCloud(cloud); ne.setRadiusSearch(0.03);
    std::vector<pcc::Normal> normals;
    ne.compute(normals);

    pcc::IntensityGradientEstimation<Pt> ge;
    ge.setSearchMethod(tree); ge.setInputCloud(cloud); ge.setInputNormals(&normals); ge.setInputIntensities(&inten); ge.setRadiusSearch(0.03);
    std::vector<pcc::IntensityGradient> grad;
    ge.compute(grad);
    CHECK(grad.size() == (size_t)n, "gradient size");
    const float r2g = (float)(0.03 * 0.03);
    int nan_rows = 0, checked = 0;
    for (int i = 0; i < n; ++i) {
        int cnt = 0;
        for (int j = 0; j < n; ++j) cnt += d2f(cloud->points[i], cloud->points[j]) < r2g;
        const bool isnan_row = std::isnan(grad[i].gradient_x);
        CHECK(isnan_row == (cnt < 3), "row %d: %d neighbours, gradient %g", i, cnt, grad[i].gradient_x);
        nan_rows += isnan_row;
        if (!isnan_row && cnt >= 20) {       // linear intensity on a plane: the in-plane gradient is (ax, ay), the normal component 0
            ++checked;
            CHECK(std::fabs(grad[i].gradient_x - ax) < 2e-3 * ax && std::fabs(grad[i].gradient_y - ay) < 2e-3 * std::fabs(ay) && std::fabs(grad[i].gradient_z) < 1e-3,
                  "row %d gradient (%g, %g, %g)", i, grad[i].gradient_x, grad[i].gradient_y, grad[i].gradient_z);
        }
    }
    CHECK(checked > n / 2, "only %d rows checked", checked);

    // RIFT over the gradients above, against computeRIFT restated here in double precision on brute-force neighbours
    for (int shape = 0; shape < 2; ++shape) {
        const int nd = shape ? 2 : 4, ng = shape ? 5 : 8;
        pcc::RIFTEstimation<Pt> re;
        auto tree2 = std::make_shared<pcc::search::GridSearch<Pt> >();
        re.setSearchMethod(tree2); re.setInputCloud(cloud); re.setInputGradient(&grad); re.setRadiusSearch(0.05);
        re.setNrDistanceBins(nd); re.setNrGradientBins(ng);
        std::vector<pcc::Histogram32> h;
        re.compute(h);
        CHECK(h.size() == (size_t)n, "rift size");
        const float r2 = (float)(0.05 * 0.05);
        double worst = 0;
        for (int i = 0; i < n; i += 7) {
            std::vector<double> ref((size_t)nd * ng, 0.0);
            const Pt &p0 = cloud->points[i];
            bool poisoned = false;
            for (int j = 0; j < n; ++j) {
                const float dd = d2f(p0, cloud->points[j]);
                if (!(dd < r2)) continue;
                const double gx = grad[j].gradient_x, gy = grad[j].gradient_y, gz = grad[j].gradient_z;
                if (std::isnan(gx)) { poisoned = true; continue; }
                const double m = std::sqrt(gx * gx + gy * gy + gz * gz);
                double vx = cloud->points[j].x - p0.x, vy = cloud->points[j].y - p0.y, vz = cloud->points[j].z - p0.z;
                const double l = std::sqrt(vx * vx + vy * vy + vz * vz);
                if (l > 0) { vx /= l; vy /= l; vz /= l; }
                double ang = std::acos((gx * vx + gy * vy + gz * vz) / m);
                if (!std::isfinite(ang)) ang = 0;
                const double d = nd * std::sqrt((double)dd) / (0.05 + 1.1920929e-7), g = ng * ang / (M_PI + 1.1920929e-7);
                for (int gi = (int)std::ceil(g - 1); gi <= (int)std::floor(g + 1); ++gi)
                    for (int di = std::max((int)std::ceil(d - 1), 0); di <= std::min((int)std::floor(d + 1), nd - 1); ++di)
                        ref[(size_t)(((gi + ng) % ng) * nd + di)] += (1 - std::fabs(d - di)) * (1 - std::fabs(g - gi)) * m;
            }
            if (poisoned) continue;
            double z = 0; for (double v : ref) z += v * v;
            z = std::sqrt(z);
            for (int k = 0; k < 32; ++k) {
                const double want = k < nd * ng ? (z > 0 ? ref[(size_t)k] / z : 0.0) : 0.0;
                worst = std::fmax(worst, std::fabs(h[i].histogram[k] - want));
            }
        }
        CHECK(worst < 1e-4, "RIFT %dx%d: max |gpu - brute force| = %g", nd, ng, worst);
        std::printf("RIFT %dx%d vs brute force: max bin error %.3g\n", nd, ng, worst);
    }
    bool threw = false;
    try { pcc::RIFTEstimation<Pt> re; re.setInputCloud(cloud); re.setInputGradient(&grad); re.setNrDistanceBins(4); re.setNrGradientBins(9); std::vector<pcc::Histogram32> h; re.compute(h); }
    catch (const pcc::Error &) { threw = true; }
    CHECK(threw, "4 x 9 bins accepted");
    std::printf("gradient rows: %d, NaN (< 3 neighbours): %d, checked against the plane's gradient: %d\n", n, nan_rows, checked);
    if (failures) { std::printf("%d failures\n", failures); return 1; }
    std::printf("PASS\n");
    return 0;
}
