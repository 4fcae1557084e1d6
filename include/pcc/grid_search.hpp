// pcc/grid_search.hpp -- C++ host mirror of the reference's search plug-in, header-only over the C ABI (pcc/search.h).
//
// pcc::search::GridSearch<PointT> keeps pcl::search::Search<PointT>'s interface method for method (PCL 1.7
// pcl/search/search.h [upstream]; reference call sites src/segmentation.cpp:120-122,129,169-171,182,232-237,262 and
// src/comparator.cpp:456-462,495-497,632-634,768-770): setInputCloud / nearestKSearch / radiusSearch with the
// point, (cloud, index), (index) and batched overloads, same return values (number of neighbours, 0 = none), same
// output-resizing convention, k clamped to the indexed point count.  Every overload is ONE batched GPU call;
// single-point overloads are a batch of one.  When PCL headers are on the include path the class derives from
// pcl::search::Search<PointT>, so `consumer.setSearchMethod(tree)` accepts it unchanged (INTEGRATION.md).
//
// The drivers below the class restate the per-point loops of the reference's consumers as single fused calls:
//   pcc::NormalEstimation            <- pcl::NormalEstimation            (src/segmentation.cpp:236-240, src/comparator.cpp:628-635)
//   pcc::StatisticalOutlierRemoval   <- pcl::StatisticalOutlierRemoval   (src/comparator.cpp:1523-1527,1537-1541)
//   pcc::EuclideanClusterExtraction  <- pcl::EuclideanClusterExtraction  (src/segmentation.cpp:125-131)
//   pcc::IterativeClosestPoint       <- pcl::IterativeClosestPoint       (src/comparator.cpp:1089-1110)
//   pcc::findPointNeighbours         <- RegionGrowing(RGB)::findPointNeighbours (src/segmentation.cpp:271,190)
//   pcc::VoxelGrid                   <- pcl::VoxelGrid                   (src/segmentation.cpp:69-74,223-228)
//   pcc::RegionGrowing               <- pcl::RegionGrowing               (src/segmentation.cpp:249-271)
//   pcc::IntensityGradientEstimation <- pcl::IntensityGradientEstimation (src/comparator.cpp:649-656)
//   pcc::RIFTEstimation              <- pcl::RIFTEstimation              (src/comparator.cpp:659-673)
//   pcc::processRIFTBatched          <- processRIFT on every cluster     (src/comparator.cpp:590-684, 1224-1366)
//   pcc::findPointNeighboursBatched, pcc::RegionGrowingRGBBatched
//                                    <- color_growing_segmentation on every cluster (src/segmentation.cpp:161-216, src/comparator.cpp:1457-1460)
// There is no CPU fallback: a failing CUDA call throws pcc::Error.
#ifndef PCC_GRID_SEARCH_HPP_
#define PCC_GRID_SEARCH_HPP_

#include <algorithm>
#include <cmath>
#include <cstddef>
#include <cstdint>
#include <limits>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "search.h"

#if defined(__has_include)
#if __has_include(<pcl/search/search.h>) && !defined(PCC_NO_PCL)
#include <pcl/point_cloud.h>
#include <pcl/search/search.h>
#define PCC_HAVE_PCL 1
#endif
#endif

namespace pcc {

struct Error : std::runtime_error {
    explicit Error(const std::string &what) : std::runtime_error(what) {}
};
inline void check(int rc) {
    if (rc != PCC_OK) throw Error(std::string("libpcc_search: ") + pcc_last_error());
}

#ifndef PCC_HAVE_PCL
// Minimal stand-ins with PCL's memory layout (xyz in the first 12 bytes of a 16-byte-aligned struct) so the class below
// compiles and is testable without PCL.  With PCL present the real pcl:: types are used instead.
struct alignas(16) PointXYZ { float x, y, z, _pad; PointXYZ() : x(0), y(0), z(0), _pad(1.f) {} PointXYZ(float a, float b, float c) : x(a), y(b), z(c), _pad(1.f) {} };
struct alignas(16) PointXYZRGB { float x, y, z, _pad; union { struct { std::uint8_t b, g, r, a; }; float rgb; }; float _pad2[3]; PointXYZRGB() : x(0), y(0), z(0), _pad(1.f), rgb(0) { _pad2[0] = _pad2[1] = _pad2[2] = 0; } };
struct alignas(16) Normal { float normal_x, normal_y, normal_z, _pad; float curvature; float _pad2[3]; };
template <typename PointT>
struct PointCloud {
    typedef std::shared_ptr<PointCloud<PointT> > Ptr;
    typedef std::shared_ptr<const PointCloud<PointT> > ConstPtr;
    std::vector<PointT> points;
    std::uint32_t width = 0, height = 1;
    bool is_dense = true;
    std::size_t size() const { return points.size(); }
    const PointT &operator[](std::size_t i) const { return points[i]; }
    PointT &operator[](std::size_t i) { return points[i]; }
    void push_back(const PointT &p) { points.push_back(p); width = (std::uint32_t)points.size(); }
};
struct PointIndices { std::vector<int> indices; };
#define PCC_CLOUD_T ::pcc::PointCloud
#define PCC_SHARED std::shared_ptr
#else
using Normal = ::pcl::Normal;
using PointIndices = ::pcl::PointIndices;
#define PCC_CLOUD_T ::pcl::PointCloud
#define PCC_SHARED boost::shared_ptr
#endif

namespace search {

template <typename PointT>
class GridSearch
#ifdef PCC_HAVE_PCL
    : public ::pcl::search::Search<PointT>
#endif
{
  public:
    typedef PCC_CLOUD_T<PointT> PointCloud;
    typedef PCC_SHARED<PointCloud> PointCloudPtr;
    typedef PCC_SHARED<const PointCloud> PointCloudConstPtr;
    typedef PCC_SHARED<std::vector<int> > IndicesPtr;
    typedef PCC_SHARED<const std::vector<int> > IndicesConstPtr;
    typedef PCC_SHARED<GridSearch<PointT> > Ptr;
    typedef PCC_SHARED<const GridSearch<PointT> > ConstPtr;

    // pcl::search::KdTree(bool sorted = true)
    explicit GridSearch(bool sorted = true, int device = 0)
#ifdef PCC_HAVE_PCL
        : ::pcl::search::Search<PointT>("pcc::search::GridSearch", sorted)
#endif
    {
        name_ = "pcc::search::GridSearch";
        sorted_ = sorted;
        check(pcc_create(device, &idx_));
    }
    virtual ~GridSearch() { pcc_destroy(idx_); }
    GridSearch(const GridSearch &) = delete;
    GridSearch &operator=(const GridSearch &) = delete;

    virtual const std::string &getName() const { return name_; }
    virtual void setSortedResults(bool sorted) { sorted_ = sorted; }
    virtual bool getSortedResults() { return sorted_; }
    // grid tuning hints (optional): expected k of the coming kNN calls, or a fixed cell edge for radius-only work
    void setKHint(int k) { k_hint_ = k; }
    void setCellHint(float cell) { cell_hint_ = cell; }

    virtual void setInputCloud(const PointCloudConstPtr &cloud, const IndicesConstPtr &indices = IndicesConstPtr()) {
        input_ = cloud;
        indices_ = indices;
        const bool use_idx = indices_ && !indices_->empty();
        check(pcc_build(idx_, cloud->points.data(), (int64_t)cloud->points.size(), (int)sizeof(PointT), use_idx ? indices_->data() : nullptr,
                        use_idx ? (int64_t)indices_->size() : 0, cell_hint_, k_hint_, PCC_HOST, nullptr));
    }
    virtual PointCloudConstPtr getInputCloud() const { return input_; }
    virtual IndicesConstPtr getIndices() const { return indices_; }
    pcc_index *handle() const { return idx_; }

    // ---- nearestKSearch --------------------------------------------------------------------------------------
    virtual int nearestKSearch(const PointT &point, int k, std::vector<int> &k_indices, std::vector<float> &k_sqr_distances) const {
        int keff = 0;
        k_indices.assign((size_t)k, -1);
        k_sqr_distances.assign((size_t)k, std::numeric_limits<float>::infinity());
        if (k <= 0) return 0;
        check(pcc_knn(idx_, &point, 1, (int)sizeof(PointT), k, k_indices.data(), k_sqr_distances.data(), &keff, PCC_HOST, nullptr));
        if (k_indices[0] < 0) keff = 0;      // non-finite query
        k_indices.resize((size_t)keff);
        k_sqr_distances.resize((size_t)keff);
        return keff;
    }
    virtual int nearestKSearch(const PointCloud &cloud, int index, int k, std::vector<int> &k_indices, std::vector<float> &k_sqr_distances) const {
        return nearestKSearch(cloud.points[(size_t)index], k, k_indices, k_sqr_distances);
    }
    virtual int nearestKSearch(int index, int k, std::vector<int> &k_indices, std::vector<float> &k_sqr_distances) const {
        const bool use_idx = indices_ && !indices_->empty();
        return nearestKSearch(input_->points[(size_t)(use_idx ? (*indices_)[(size_t)index] : index)], k, k_indices, k_sqr_distances);
    }
    // batched overload: empty `indices` means every point of `cloud`
    virtual void nearestKSearch(const PointCloud &cloud, const std::vector<int> &indices, int k, std::vector<std::vector<int> > &k_indices,
                                std::vector<std::vector<float> > &k_sqr_distances) const {
        std::vector<PointT> gathered;
        const PointT *q = cloud.points.data();
        size_t nq = cloud.points.size();
        if (!indices.empty()) {
            gathered.reserve(indices.size());
            for (int i : indices) gathered.push_back(cloud.points[(size_t)i]);
            q = gathered.data(); nq = gathered.size();
        }
        std::vector<int> flat_i(nq * (size_t)k);
        std::vector<float> flat_d(nq * (size_t)k);
        int keff = 0;
        if (nq) check(pcc_knn(idx_, q, (int64_t)nq, (int)sizeof(PointT), k, flat_i.data(), flat_d.data(), &keff, PCC_HOST, nullptr));
        k_indices.resize(nq); k_sqr_distances.resize(nq);
        for (size_t r = 0; r < nq; ++r) {
            const int n = flat_i[r * k] < 0 ? 0 : keff;
            k_indices[r].assign(flat_i.begin() + r * k, flat_i.begin() + r * k + n);
            k_sqr_distances[r].assign(flat_d.begin() + r * k, flat_d.begin() + r * k + n);
        }
    }
    // flat variant for consumers that want the dense N x k table (RegionGrowing::findPointNeighbours); q == nullptr = the input cloud
    int nearestKSearchTable(const PointT *q, size_t nq, int k, std::vector<int> &flat_indices, std::vector<float> &flat_sqr_distances) const {
        const size_t rows = q ? nq : input_->points.size();
        flat_indices.resize(rows * (size_t)k); flat_sqr_distances.resize(rows * (size_t)k);
        int keff = 0;
        if (rows) check(pcc_knn(idx_, q, (int64_t)nq, (int)sizeof(PointT), k, flat_indices.data(), flat_sqr_distances.data(), &keff, PCC_HOST, nullptr));
        return keff;
    }

    // ---- radiusSearch ------------------------------------------------------------------------------------------
    virtual int radiusSearch(const PointT &point, double radius, std::vector<int> &k_indices, std::vector<float> &k_sqr_distances, unsigned int max_nn = 0) const {
        std::vector<int64_t> off(2, 0);
        csr(&point, 1, radius, max_nn, off, k_indices, k_sqr_distances);
        return (int)k_indices.size();
    }
    virtual int radiusSearch(const PointCloud &cloud, int index, double radius, std::vector<int> &k_indices, std::vector<float> &k_sqr_distances, unsigned int max_nn = 0) const {
        return radiusSearch(cloud.points[(size_t)index], radius, k_indices, k_sqr_distances, max_nn);
    }
    virtual int radiusSearch(int index, double radius, std::vector<int> &k_indices, std::vector<float> &k_sqr_distances, unsigned int max_nn = 0) const {
        const bool use_idx = indices_ && !indices_->empty();
        return radiusSearch(input_->points[(size_t)(use_idx ? (*indices_)[(size_t)index] : index)], radius, k_indices, k_sqr_distances, max_nn);
    }
    virtual void radiusSearch(const PointCloud &cloud, const std::vector<int> &indices, double radius, std::vector<std::vector<int> > &k_indices,
                              std::vector<std::vector<float> > &k_sqr_distances, unsigned int max_nn = 0) const {
        std::vector<PointT> gathered;
        const PointT *q = cloud.points.data();
        size_t nq = cloud.points.size();
        if (!indices.empty()) {
            gathered.reserve(indices.size());
            for (int i : indices) gathered.push_back(cloud.points[(size_t)i]);
            q = gathered.data(); nq = gathered.size();
        }
        std::vector<int64_t> off;
        std::vector<int> fi;
        std::vector<float> fd;
        csr(q, nq, radius, max_nn, off, fi, fd);
        k_indices.resize(nq); k_sqr_distances.resize(nq);
        for (size_t r = 0; r < nq; ++r) {
            k_indices[r].assign(fi.begin() + off[r], fi.begin() + off[r + 1]);
            k_sqr_distances[r].assign(fd.begin() + off[r], fd.begin() + off[r + 1]);
        }
    }
    // CSR variant (offsets[nq+1]); q == nullptr = the input cloud
    void csr(const PointT *q, size_t nq, double radius, unsigned max_nn, std::vector<int64_t> &offsets, std::vector<int> &indices, std::vector<float> &sqr_distances) const {
        const size_t rows = q ? nq : input_->points.size();
        offsets.assign(rows + 1, 0);
        int64_t total = 0;
        check(pcc_radius_count(idx_, q, (int64_t)nq, (int)sizeof(PointT), radius, max_nn, offsets.data(), &total, PCC_HOST, nullptr));
        indices.resize((size_t)total); sqr_distances.resize((size_t)total);
        if (total) check(pcc_radius_fill(idx_, q, (int64_t)nq, (int)sizeof(PointT), radius, max_nn, sorted_ ? 1 : 0, offsets.data(), indices.data(), sqr_distances.data(), PCC_HOST, nullptr));
    }

  protected:
    pcc_index *idx_ = nullptr;
    PointCloudConstPtr input_;
    IndicesConstPtr indices_;
    std::string name_;
    bool sorted_ = true;
    int k_hint_ = 0;
    float cell_hint_ = 0.f;
};

}  // namespace search

// ---- consumers: the reference's per-point loops as single fused calls ---------------------------------------------

// pcl::NormalEstimation::compute with setKSearch(k) or setRadiusSearch(r) over the tree's input cloud.
// out[i] = (normal_x, normal_y, normal_z, curvature); NaN when a point has < 3 neighbours.
template <typename PointT>
class NormalEstimation {
  public:
    void setSearchMethod(const typename search::GridSearch<PointT>::Ptr &tree) { tree_ = tree; }
    void setInputCloud(const typename search::GridSearch<PointT>::PointCloudConstPtr &cloud) { input_ = cloud; }
    void setKSearch(int k) { k_ = k; }
    void setRadiusSearch(double r) { radius_ = r; }
    void setViewPoint(float x, float y, float z) { vp_[0] = x; vp_[1] = y; vp_[2] = z; }
    void compute(std::vector<Normal> &out) {
        if (!tree_) tree_.reset(new search::GridSearch<PointT>());
        if (k_ > 0) tree_->setKHint(k_); else tree_->setCellHint((float)radius_);
        if (tree_->getInputCloud() != input_) tree_->setInputCloud(input_);
        const size_t n = input_->points.size();
        std::vector<float> flat(n * 4);
        if (n) {
            if (k_ > 0) check(pcc_normals_knn(tree_->handle(), nullptr, 0, (int)sizeof(PointT), k_, vp_, flat.data(), PCC_HOST, nullptr));
            else check(pcc_normals_radius(tree_->handle(), nullptr, 0, (int)sizeof(PointT), radius_, vp_, flat.data(), PCC_HOST, nullptr));
        }
        out.resize(n);
        for (size_t i = 0; i < n; ++i) { out[i].normal_x = flat[4 * i]; out[i].normal_y = flat[4 * i + 1]; out[i].normal_z = flat[4 * i + 2]; out[i].curvature = flat[4 * i + 3]; }
    }
  private:
    typename search::GridSearch<PointT>::Ptr tree_;
    typename search::GridSearch<PointT>::PointCloudConstPtr input_;
    int k_ = 0; double radius_ = 0; float vp_[3] = {0, 0, 0};
};

// pcl::StatisticalOutlierRemoval::applyFilterIndices: indices kept (distance <= mean + mul * stddev).
template <typename PointT>
class StatisticalOutlierRemoval {
  public:
    void setInputCloud(const typename search::GridSearch<PointT>::PointCloudConstPtr &cloud) { input_ = cloud; }
    void setMeanK(int k) { mean_k_ = k; }
    void setStddevMulThresh(double m) { mul_ = m; }
    void filter(std::vector<int> &kept_indices) {
        search::GridSearch<PointT> tree(false);
        tree.setKHint(mean_k_ + 1);
        tree.setInputCloud(input_);
        const size_t n = input_->points.size();
        std::vector<float> dist(n);
        std::vector<std::uint8_t> keep(n);
        int64_t kept = 0;
        if (n) {
            check(pcc_knn_mean_dist(tree.handle(), nullptr, 0, (int)sizeof(PointT), mean_k_, dist.data(), PCC_HOST, nullptr));
            check(pcc_sor_threshold(tree.handle(), dist.data(), (int64_t)n, pcc_size(tree.handle()), mul_, stats_, keep.data(), &kept, PCC_HOST, nullptr));
        }
        kept_indices.clear();
        kept_indices.reserve((size_t)kept);
        for (size_t i = 0; i < n; ++i) if (keep[i]) kept_indices.push_back((int)i);
    }
    double mean() const { return stats_[0]; }
    double stddev() const { return stats_[1]; }
    double threshold() const { return stats_[2]; }
  private:
    typename search::GridSearch<PointT>::PointCloudConstPtr input_;
    int mean_k_ = 1; double mul_ = 0; double stats_[3] = {0, 0, 0};
};

// pcl::EuclideanClusterExtraction::extract: clusters by size descending, indices ascending inside a cluster.
template <typename PointT>
class EuclideanClusterExtraction {
  public:
    void setClusterTolerance(double t) { tol_ = t; }
    void setMinClusterSize(int n) { min_ = n; }
    void setMaxClusterSize(int n) { max_ = n; }
    void setSearchMethod(const typename search::GridSearch<PointT>::Ptr &tree) { tree_ = tree; }
    void setInputCloud(const typename search::GridSearch<PointT>::PointCloudConstPtr &cloud) { input_ = cloud; }
    void extract(std::vector<PointIndices> &clusters) {
        if (!tree_) tree_.reset(new search::GridSearch<PointT>());
        tree_->setCellHint((float)tol_);
        if (tree_->getInputCloud() != input_) tree_->setInputCloud(input_);
        const size_t n = input_->points.size();
        std::vector<int32_t> labels(n ? n : 1);
        std::vector<int64_t> sizes(n / (size_t)(min_ > 0 ? min_ : 1) + 1);
        int64_t nc = 0;
        check(pcc_euclidean_labels(tree_->handle(), tol_, min_, max_, labels.data(), &nc, sizes.data(), (int64_t)sizes.size(), PCC_HOST, nullptr));
        clusters.assign((size_t)nc, PointIndices());
        for (int64_t c = 0; c < nc; ++c) clusters[(size_t)c].indices.reserve((size_t)sizes[(size_t)c]);
        for (size_t i = 0; i < n; ++i) if (labels[i] >= 0) clusters[(size_t)labels[i]].indices.push_back((int)i);
    }
  private:
    typename search::GridSearch<PointT>::Ptr tree_;
    typename search::GridSearch<PointT>::PointCloudConstPtr input_;
    double tol_ = 0; int min_ = 1; int max_ = std::numeric_limits<int>::max();
};

// pcl::IterativeClosestPoint as the reference uses it: setMaximumIterations, align, hasConverged, getFitnessScore.
template <typename PointT>
class IterativeClosestPoint {
  public:
    void setMaximumIterations(int n) { max_iter_ = n; }
    void setInputSource(const typename search::GridSearch<PointT>::PointCloudConstPtr &c) { source_ = c; }
    void setInputTarget(const typename search::GridSearch<PointT>::PointCloudConstPtr &c) { target_ = c; }
    void align() {
        search::GridSearch<PointT> tree;
        tree.setKHint(32);     // coarse cells: the first iterations search from far away (measured 2.4x faster than k_hint = 1 on the 10 M pair)
        tree.setInputCloud(target_);
        check(pcc_icp_align(tree.handle(), source_->points.data(), (int64_t)source_->points.size(), (int)sizeof(PointT), max_iter_, T_, &converged_, &fitness_, &iterations_, PCC_HOST, nullptr));
    }
    bool hasConverged() const { return converged_ != 0; }
    double getFitnessScore() const { return fitness_; }
    const float *getFinalTransformation() const { return T_; }   // row-major 4x4
    int iterations() const { return iterations_; }
  private:
    typename search::GridSearch<PointT>::PointCloudConstPtr source_, target_;
    int max_iter_ = 10, converged_ = 0, iterations_ = 0; double fitness_ = 0; float T_[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
};

// pcl::VoxelGrid<PointT>: setLeafSize + filter (src/segmentation.cpp:69-74, 223-228).  One centroid per occupied voxel, ordered
// by voxel index; for colour points pass the byte offset of the packed rgb word (16 for pcl::PointXYZRGB), else -1.
template <typename PointT>
class VoxelGrid {
  public:
    explicit VoxelGrid(int rgb_offset_bytes = -1, int device = 0) : rgb_off_(rgb_offset_bytes) { check(pcc_create(device, &ws_)); }
    ~VoxelGrid() { pcc_destroy(ws_); }
    VoxelGrid(const VoxelGrid &) = delete;
    VoxelGrid &operator=(const VoxelGrid &) = delete;
    void setInputCloud(const typename search::GridSearch<PointT>::PointCloudConstPtr &cloud) { input_ = cloud; }
    void setLeafSize(float lx, float ly, float lz) { leaf_[0] = lx; leaf_[1] = ly; leaf_[2] = lz; }
    void setMinimumPointsNumberPerVoxel(int n) { min_points_ = n; }
    void filter(typename search::GridSearch<PointT>::PointCloud &output) {
        const size_t n = input_->points.size();
        std::vector<PointT> out(n);
        int64_t n_out = 0;
        if (n) check(pcc_voxel_grid(ws_, input_->points.data(), (int64_t)n, (int)sizeof(PointT), rgb_off_, leaf_, min_points_, out.data(), &n_out, PCC_HOST, nullptr));
        out.resize((size_t)n_out);
        output.points.swap(out);
        output.width = (std::uint32_t)output.points.size(); output.height = 1; output.is_dense = true;
    }
  private:
    pcc_index *ws_ = nullptr;
    typename search::GridSearch<PointT>::PointCloudConstPtr input_;
    float leaf_[3] = {0.01f, 0.01f, 0.01f};
    int rgb_off_ = -1, min_points_ = 0;
};

// RegionGrowing(RGB)::findPointNeighbours: the dense N x k neighbour (and distance) table the sequential grow phase consumes.
template <typename PointT>
inline int findPointNeighbours(search::GridSearch<PointT> &tree, int k, std::vector<int> &neighbours, std::vector<float> &sqr_distances) {
    return tree.nearestKSearchTable(nullptr, 0, k, neighbours, sqr_distances);
}

// pcl::RegionGrowing<PointT, Normal>::extract: the N x k table comes from one batched GPU query, the order-dependent grow
// phase runs on the host over it (pcc_region_growing).  Clusters come out in creation order, members ascending, as PCL's
// assembleRegions leaves them.
template <typename PointT>
class RegionGrowing {
  public:
    void setSearchMethod(const typename search::GridSearch<PointT>::Ptr &tree) { tree_ = tree; }
    void setInputCloud(const typename search::GridSearch<PointT>::PointCloudConstPtr &cloud) { input_ = cloud; }
    void setInputNormals(const std::vector<Normal> *normals) { normals_ = normals; }
    void setNumberOfNeighbours(unsigned int k) { k_ = (int)k; }
    void setMinClusterSize(int n) { min_size_ = n; }
    void setMaxClusterSize(int n) { max_size_ = n; }
    void setSmoothnessThreshold(float theta) { theta_ = theta; }
    void setCurvatureThreshold(float c) { curvature_ = c; }
    void extract(std::vector<PointIndices> &clusters) {
        clusters.clear();
        if (!input_ || !normals_ || normals_->size() != input_->points.size()) throw Error("RegionGrowing: cloud and normals must be set and of equal size");
        const size_t n = input_->points.size();
        if (n == 0) return;
        if (!tree_) tree_.reset(new search::GridSearch<PointT>());
        tree_->setKHint(k_);
        if (tree_->getInputCloud() != input_) tree_->setInputCloud(input_);
        std::vector<int> nbrs; std::vector<float> d2;
        findPointNeighbours(*tree_, k_, nbrs, d2);
        std::vector<float> flat(n * 4);
        for (size_t i = 0; i < n; ++i) { const Normal &m = (*normals_)[i]; flat[4 * i] = m.normal_x; flat[4 * i + 1] = m.normal_y; flat[4 * i + 2] = m.normal_z; flat[4 * i + 3] = m.curvature; }
        labels_.assign(n, -1);
        int64_t nc = 0;
        check(pcc_region_growing(nbrs.data(), (int64_t)n, k_, flat.data(), theta_, curvature_, min_size_, max_size_, labels_.data(), &nc));
        clusters.resize((size_t)nc);
        for (size_t i = 0; i < n; ++i) if (labels_[i] >= 0) clusters[(size_t)labels_[i]].indices.push_back((int)i);
    }
    const std::vector<int32_t> &labels() const { return labels_; }
  private:
    typename search::GridSearch<PointT>::Ptr tree_;
    typename search::GridSearch<PointT>::PointCloudConstPtr input_;
    const std::vector<Normal> *normals_ = nullptr;
    std::vector<int32_t> labels_;
    int k_ = 30; int64_t min_size_ = 1, max_size_ = std::numeric_limits<int>::max();
    float theta_ = 30.0f / 180.0f * 3.14159265358979f, curvature_ = 0.05f;
};

// pcl::RegionGrowingRGB<PointT>::extract as color_growing_segmentation uses it (src/segmentation.cpp:179-190: distance 10, point colour 6,
// region colour 5, min cluster 200; neither the search k nor the neighbour number is set, so the table has PCL's 100 columns and the
// grow phase walks the first 30).  The N x 100 table + squared distances come from one batched GPU query; grow / merge / fold of small
// regions run on the host over it (pcc_region_growing_rgb).  PointT must carry PCL's packed colour word at `rgba_offset` bytes
// (16 for pcl::PointXYZRGB and for the stand-in above).
template <typename PointT>
class RegionGrowingRGB {
  public:
    explicit RegionGrowingRGB(int rgba_offset = 16) : rgba_off_(rgba_offset) {}
    void setSearchMethod(const typename search::GridSearch<PointT>::Ptr &tree) { tree_ = tree; }
    void setInputCloud(const typename search::GridSearch<PointT>::PointCloudConstPtr &cloud) { input_ = cloud; }
    void setDistanceThreshold(float d) { distance_ = d; }
    void setPointColorThreshold(float t) { point_color_ = t; }
    void setRegionColorThreshold(float t) { region_color_ = t; }
    void setNumberOfRegionNeighbours(unsigned int k) { table_k_ = (int)k; }       // RegionGrowingRGB::region_neighbour_number_ (the table's width)
    void setNumberOfNeighbours(unsigned int k) { grow_k_ = (int)k; }              // RegionGrowing::neighbour_number_ (what growRegion walks)
    void setMinClusterSize(int n) { min_size_ = n; }
    void setMaxClusterSize(int n) { max_size_ = n; }
    void extract(std::vector<PointIndices> &clusters) {
        clusters.clear();
        if (!input_) throw Error("RegionGrowingRGB: no input cloud");
        const size_t n = input_->points.size();
        if (n == 0) return;
        if (!tree_) tree_.reset(new search::GridSearch<PointT>());
        tree_->setKHint(table_k_);
        if (tree_->getInputCloud() != input_) tree_->setInputCloud(input_);
        std::vector<int> nbrs; std::vector<float> d2;
        findPointNeighbours(*tree_, table_k_, nbrs, d2);          // rows of stride table_k_; a cluster under table_k_ points ends its rows with -1
        labels_.assign(n, -1);
        int64_t nc = 0;
        const uint32_t *rgba = reinterpret_cast<const uint32_t *>(reinterpret_cast<const char *>(input_->points.data()) + rgba_off_);
        check(pcc_region_growing_rgb(nbrs.data(), d2.data(), (int64_t)n, table_k_, rgba, (int)sizeof(PointT), distance_, point_color_, region_color_,
                                     std::min(grow_k_, table_k_), min_size_, max_size_, labels_.data(), &nc));
        clusters.resize((size_t)nc);
        for (size_t i = 0; i < n; ++i) if (labels_[i] >= 0) clusters[(size_t)labels_[i]].indices.push_back((int)i);
    }
    const std::vector<int32_t> &labels() const { return labels_; }
  private:
    typename search::GridSearch<PointT>::Ptr tree_;
    typename search::GridSearch<PointT>::PointCloudConstPtr input_;
    std::vector<int32_t> labels_;
    int rgba_off_, table_k_ = 100, grow_k_ = 30;
    int64_t min_size_ = 1, max_size_ = std::numeric_limits<int>::max();
    float distance_ = 10.f, point_color_ = 1225.f, region_color_ = 10.f;          // PCL 1.7 constructor defaults
};

// findPointNeighbours of every cluster in one call (pcc_knn_batched): neighbours[c] / sqr_distances[c] get exactly the table
// findPointNeighbours fills for cluster c alone (stride k, cluster-local indices, -1 / +inf past the cluster's k_eff); returns k_eff per
// cluster.  Clusters are copied into one concatenated cloud for the call.
template <typename PointT>
inline std::vector<int> findPointNeighboursBatched(const std::vector<typename search::GridSearch<PointT>::PointCloudConstPtr> &clusters, int k,
                                                   std::vector<std::vector<int> > &neighbours, std::vector<std::vector<float> > &sqr_distances, int device = 0) {
    std::vector<PointT> all;
    std::vector<int64_t> off(1, 0);
    for (const auto &c : clusters) {
        if (!c) throw Error("findPointNeighboursBatched: null input cloud");
        all.insert(all.end(), c->points.begin(), c->points.end());
        off.push_back((int64_t)all.size());
    }
    const int64_t n_clouds = (int64_t)clusters.size(), n = (int64_t)all.size();
    std::vector<int> fi((size_t)n * (size_t)std::max(k, 0)), keff((size_t)n_clouds + 1);
    std::vector<float> fd(fi.size());
    pcc_index *ws = nullptr;
    check(pcc_create(device, &ws));
    const int rc = pcc_knn_batched(ws, all.data(), n, (int)sizeof(PointT), off.data(), n_clouds, k, fi.data(), fd.data(), keff.data(), PCC_HOST, nullptr);
    pcc_destroy(ws);
    check(rc);
    neighbours.assign((size_t)n_clouds, std::vector<int>());
    sqr_distances.assign((size_t)n_clouds, std::vector<float>());
    for (int64_t c = 0; c < n_clouds; ++c) {
        neighbours[c].assign(fi.begin() + off[c] * k, fi.begin() + off[c + 1] * k);
        sqr_distances[c].assign(fd.begin() + off[c] * k, fd.begin() + off[c + 1] * k);
    }
    keff.resize((size_t)n_clouds);
    return keff;
}

// RegionGrowingRGB over every cluster of a cloud in one call (pcc_region_growing_rgb_batched), as computeSimilarity runs
// color_growing_segmentation on both clouds of every matched pair (src/comparator.cpp:1457-1460): extract fills clusters[c] with exactly what
// RegionGrowingRGB::extract returns on cluster c alone, members as cluster-local rows.  One GPU pass builds every cluster's table; the grow /
// merge runs on the host, one cluster after another.  The reference segments only clouds of more than 10 points
// (src/segmentation.cpp:167): that test stays with the caller.  Setters and defaults are RegionGrowingRGB's.
template <typename PointT>
class RegionGrowingRGBBatched {
  public:
    explicit RegionGrowingRGBBatched(int rgba_offset = 16, int device = 0) : rgba_off_(rgba_offset) { check(pcc_create(device, &ws_)); }
    ~RegionGrowingRGBBatched() { pcc_destroy(ws_); }
    RegionGrowingRGBBatched(const RegionGrowingRGBBatched &) = delete;
    RegionGrowingRGBBatched &operator=(const RegionGrowingRGBBatched &) = delete;
    void setInputClouds(const std::vector<typename search::GridSearch<PointT>::PointCloudConstPtr> &clouds) { inputs_ = clouds; }
    void setDistanceThreshold(float d) { distance_ = d; }
    void setPointColorThreshold(float t) { point_color_ = t; }
    void setRegionColorThreshold(float t) { region_color_ = t; }
    void setNumberOfRegionNeighbours(unsigned int k) { table_k_ = (int)k; }
    void setNumberOfNeighbours(unsigned int k) { grow_k_ = (int)k; }
    void setMinClusterSize(int n) { min_size_ = n; }
    void setMaxClusterSize(int n) { max_size_ = n; }
    void extract(std::vector<std::vector<PointIndices> > &clusters) {
        std::vector<PointT> all;
        std::vector<int64_t> off(1, 0);
        for (const auto &c : inputs_) {
            if (!c) throw Error("RegionGrowingRGBBatched: null input cloud");
            all.insert(all.end(), c->points.begin(), c->points.end());
            off.push_back((int64_t)all.size());
        }
        const int64_t n_clouds = (int64_t)inputs_.size();
        std::vector<int32_t> labels(all.size());
        std::vector<int64_t> nc((size_t)n_clouds + 1);
        check(pcc_region_growing_rgb_batched(ws_, all.data(), (int64_t)all.size(), (int)sizeof(PointT), rgba_off_, off.data(), n_clouds, table_k_, distance_,
                                             point_color_, region_color_, std::min(grow_k_, table_k_), min_size_, max_size_, labels.data(), nc.data(),
                                             PCC_HOST, nullptr));
        clusters.assign((size_t)n_clouds, std::vector<PointIndices>());
        for (int64_t c = 0; c < n_clouds; ++c) {
            clusters[c].resize((size_t)nc[c]);
            for (int64_t i = off[c]; i < off[c + 1]; ++i) if (labels[i] >= 0) clusters[c][(size_t)labels[i]].indices.push_back((int)(i - off[c]));
        }
    }
  private:
    pcc_index *ws_ = nullptr;
    std::vector<typename search::GridSearch<PointT>::PointCloudConstPtr> inputs_;
    int rgba_off_, table_k_ = 100, grow_k_ = 30;
    int64_t min_size_ = 1, max_size_ = std::numeric_limits<int>::max();
    float distance_ = 10.f, point_color_ = 1225.f, region_color_ = 10.f;          // PCL 1.7 constructor defaults
};

// PCL 1.7 PointXYZRGBtoXYZI (src/comparator.cpp:597): 0.299f r + 0.587f g + 0.114f b, left to right in fp32.
inline float rgbToIntensity(std::uint8_t r, std::uint8_t g, std::uint8_t b) {
    volatile float t = 0.299f * (float)r;          // volatile: no contraction into an FMA whatever the caller's flags
    t = t + 0.587f * (float)g;
    return t + 0.114f * (float)b;
}

struct IntensityGradient { float gradient_x, gradient_y, gradient_z, _pad; };
struct Histogram32 { float histogram[32]; };

// pcl::IntensityGradientEstimation<PointT, Normal, IntensityGradient>::compute with setRadiusSearch(r) over the tree's input
// cloud (the reference's surface): one fused GPU call (pcc_intensity_gradient).  Intensities are one float per input point
// (rgbToIntensity for colour clouds); normals as pcc::NormalEstimation fills them.  NaN gradients with < 3 neighbours.
template <typename PointT>
class IntensityGradientEstimation {
  public:
    void setSearchMethod(const typename search::GridSearch<PointT>::Ptr &tree) { tree_ = tree; }
    void setInputCloud(const typename search::GridSearch<PointT>::PointCloudConstPtr &cloud) { input_ = cloud; }
    void setInputNormals(const std::vector<Normal> *normals) { normals_ = normals; }
    void setInputIntensities(const std::vector<float> *intensity) { intensity_ = intensity; }
    void setRadiusSearch(double r) { radius_ = r; }
    void compute(std::vector<IntensityGradient> &out) {
        if (!input_ || !normals_ || !intensity_ || normals_->size() != input_->points.size() || intensity_->size() != input_->points.size())
            throw Error("IntensityGradientEstimation: cloud, normals and intensities must be set and of equal size");
        if (!tree_) tree_.reset(new search::GridSearch<PointT>());
        tree_->setCellHint((float)radius_);
        if (tree_->getInputCloud() != input_) tree_->setInputCloud(input_);
        const size_t n = input_->points.size();
        std::vector<float> nrm(n * 4), flat(n * 4);
        for (size_t i = 0; i < n; ++i) { const Normal &m = (*normals_)[i]; nrm[4 * i] = m.normal_x; nrm[4 * i + 1] = m.normal_y; nrm[4 * i + 2] = m.normal_z; nrm[4 * i + 3] = m.curvature; }
        if (n) check(pcc_intensity_gradient(tree_->handle(), nullptr, 0, (int)sizeof(PointT), radius_, intensity_->data(), nrm.data(), flat.data(), PCC_HOST, nullptr));
        out.resize(n);
        for (size_t i = 0; i < n; ++i) { out[i].gradient_x = flat[4 * i]; out[i].gradient_y = flat[4 * i + 1]; out[i].gradient_z = flat[4 * i + 2]; out[i]._pad = 0.f; }
    }
  private:
    typename search::GridSearch<PointT>::Ptr tree_;
    typename search::GridSearch<PointT>::PointCloudConstPtr input_;
    const std::vector<Normal> *normals_ = nullptr;
    const std::vector<float> *intensity_ = nullptr;
    double radius_ = 0;
};

// pcl::RIFTEstimation<PointT, IntensityGradient, Histogram<32>>::compute over the tree's input cloud (pcc_rift).  Bins beyond
// nd * ng stay 0; a point without neighbours gets a NaN histogram.  Order: histogram[g * nd + d], as PCL copies it out.
template <typename PointT>
class RIFTEstimation {
  public:
    void setSearchMethod(const typename search::GridSearch<PointT>::Ptr &tree) { tree_ = tree; }
    void setInputCloud(const typename search::GridSearch<PointT>::PointCloudConstPtr &cloud) { input_ = cloud; }
    void setInputGradient(const std::vector<IntensityGradient> *gradient) { gradient_ = gradient; }
    void setRadiusSearch(double r) { radius_ = r; }
    void setNrDistanceBins(int n) { nd_ = n; }
    void setNrGradientBins(int n) { ng_ = n; }
    void compute(std::vector<Histogram32> &out) {
        if (!input_ || !gradient_ || gradient_->size() != input_->points.size())
            throw Error("RIFTEstimation: the gradient cloud must be set and of the input cloud's size");
        if (nd_ * ng_ > 32) throw Error("RIFTEstimation: nr_distance_bins * nr_gradient_bins must be <= 32 (Histogram<32>)");
        if (!tree_) tree_.reset(new search::GridSearch<PointT>());
        tree_->setCellHint((float)radius_);
        if (tree_->getInputCloud() != input_) tree_->setInputCloud(input_);
        const size_t n = input_->points.size();
        const int nb = nd_ * ng_;
        std::vector<float> flat(n * (size_t)nb);
        if (n) check(pcc_rift(tree_->handle(), nullptr, 0, (int)sizeof(PointT), radius_, reinterpret_cast<const float *>(gradient_->data()), nd_, ng_, flat.data(), PCC_HOST, nullptr));
        out.assign(n, Histogram32());
        for (size_t i = 0; i < n; ++i) for (int k = 0; k < 32; ++k) out[i].histogram[k] = k < nb ? flat[i * nb + k] : 0.f;
    }
  private:
    typename search::GridSearch<PointT>::Ptr tree_;
    typename search::GridSearch<PointT>::PointCloudConstPtr input_;
    const std::vector<IntensityGradient> *gradient_ = nullptr;
    double radius_ = 0;
    int nd_ = 4, ng_ = 8;
};

// pcl::PointWithScale: a SIFT keypoint (x, y, z of the octave point and the scale it was detected at)
struct PointWithScale { float x, y, z, scale; };

// pcl::SIFTKeypoint<PointT, PointWithScale>::compute as processSift configures it (src/comparator.cpp:449-465): one call
// (pcc_sift_keypoints) runs the whole octave loop on the GPU.  The class owns its workspace index, as VoxelGrid does; after compute
// it indexes the last octave's grid.  setSearchMethod is accepted for PCL's call pattern and not used: PCL 1.7 re-points the tree at
// every octave's grid itself.  PointT needs PCL's packed `rgb` member.  Defaults are the reference's parameters.
template <typename PointT>
class SIFTKeypoint {
  public:
    explicit SIFTKeypoint(int device = 0) { check(pcc_create(device, &ws_)); }
    ~SIFTKeypoint() { pcc_destroy(ws_); }
    SIFTKeypoint(const SIFTKeypoint &) = delete;
    SIFTKeypoint &operator=(const SIFTKeypoint &) = delete;
    void setInputCloud(const typename search::GridSearch<PointT>::PointCloudConstPtr &cloud) { input_ = cloud; }
    void setSearchMethod(const typename search::GridSearch<PointT>::Ptr &) {}
    void setScales(float min_scale, int nr_octaves, int nr_scales_per_octave) { min_scale_ = min_scale; nr_octaves_ = nr_octaves; nr_scales_per_octave_ = nr_scales_per_octave; }
    void setMinimumContrast(float min_contrast) { min_contrast_ = min_contrast; }
    void compute(std::vector<PointWithScale> &out) {
        if (!input_) throw Error("SIFTKeypoint: no input cloud");
        const int64_t n = (int64_t)input_->points.size();
        int64_t cap = std::max<int64_t>(n, 1), found = 0;
        for (;;) {                                   // the keypoint count is known after the call: retry once with room for all
            out.resize((size_t)cap);
            check(pcc_sift_keypoints(ws_, input_->points.data(), n, (int)sizeof(PointT), (int)offsetof(PointT, rgb), min_scale_, nr_octaves_,
                                     nr_scales_per_octave_, min_contrast_, reinterpret_cast<float *>(out.data()), cap, &found, PCC_HOST, nullptr));
            if (found <= cap) break;
            cap = found;
        }
        out.resize((size_t)found);
    }
  private:
    pcc_index *ws_ = nullptr;
    typename search::GridSearch<PointT>::PointCloudConstPtr input_;
    float min_scale_ = 0.005f, min_contrast_ = 0.001f;
    int nr_octaves_ = 5, nr_scales_per_octave_ = 5;
};

// SIFTKeypoint over every cluster of a cloud in one call (pcc_sift_keypoints_batched), as processRIFTwithSIFT runs it per cluster
// (src/comparator.cpp:1228, 1264): compute fills out[c] with exactly what SIFTKeypoint::compute returns on cluster c alone, and, when
// `snap` is given, (*snap)[c] with the cluster-local row of the first point of cluster c within snap_threshold of each keypoint
// (-1 if none; src/comparator.cpp:696-713).  Clusters are copied into one concatenated cloud for the call.
template <typename PointT>
class SIFTKeypointBatched {
  public:
    explicit SIFTKeypointBatched(int device = 0) { check(pcc_create(device, &ws_)); }
    ~SIFTKeypointBatched() { pcc_destroy(ws_); }
    SIFTKeypointBatched(const SIFTKeypointBatched &) = delete;
    SIFTKeypointBatched &operator=(const SIFTKeypointBatched &) = delete;
    void setInputClouds(const std::vector<typename search::GridSearch<PointT>::PointCloudConstPtr> &clouds) { inputs_ = clouds; }
    void setScales(float min_scale, int nr_octaves, int nr_scales_per_octave) { min_scale_ = min_scale; nr_octaves_ = nr_octaves; nr_scales_per_octave_ = nr_scales_per_octave; }
    void setMinimumContrast(float min_contrast) { min_contrast_ = min_contrast; }
    void compute(std::vector<std::vector<PointWithScale> > &out, std::vector<std::vector<int> > *snap = nullptr, double snap_threshold = 0.05) {
        std::vector<PointT> all;
        std::vector<int64_t> off(1, 0);
        for (const auto &c : inputs_) {
            if (!c) throw Error("SIFTKeypointBatched: null input cloud");
            all.insert(all.end(), c->points.begin(), c->points.end());
            off.push_back((int64_t)all.size());
        }
        const int64_t n_clouds = (int64_t)inputs_.size();
        std::vector<int64_t> kp_off(off.size());
        std::vector<PointWithScale> kp;
        std::vector<int32_t> sn;
        int64_t cap = std::max<int64_t>((int64_t)all.size(), 1);
        for (;;) {                                   // the keypoint count is known after the call: retry once with room for all
            kp.resize((size_t)cap);
            if (snap) sn.resize((size_t)cap);
            check(pcc_sift_keypoints_batched(ws_, all.data(), (int64_t)all.size(), (int)sizeof(PointT), (int)offsetof(PointT, rgb), off.data(), n_clouds,
                                             min_scale_, nr_octaves_, nr_scales_per_octave_, min_contrast_, snap_threshold,
                                             reinterpret_cast<float *>(kp.data()), snap ? sn.data() : nullptr, cap, kp_off.data(), PCC_HOST, nullptr));
            if (kp_off.back() <= cap) break;
            cap = kp_off.back();
        }
        out.assign((size_t)n_clouds, std::vector<PointWithScale>());
        if (snap) snap->assign((size_t)n_clouds, std::vector<int>());
        for (int64_t c = 0; c < n_clouds; ++c) {
            out[c].assign(kp.begin() + kp_off[c], kp.begin() + kp_off[c + 1]);
            if (snap) (*snap)[c].assign(sn.begin() + kp_off[c], sn.begin() + kp_off[c + 1]);
        }
    }
  private:
    pcc_index *ws_ = nullptr;
    std::vector<typename search::GridSearch<PointT>::PointCloudConstPtr> inputs_;
    float min_scale_ = 0.005f, min_contrast_ = 0.001f;
    int nr_octaves_ = 5, nr_scales_per_octave_ = 5;
};

// processRIFT (src/comparator.cpp:590-684) on every cluster in one call (pcc_rift_batched), as computeSimilarity runs it per cluster:
// descriptors[c] and kept_rows[c] are exactly what cluster c alone gets from NormalEstimation(radius) -> drop the NaN normals ->
// IntensityGradientEstimation -> RIFTEstimation -> drop the rows with a non-finite bin.  kept_rows[c] are rows of cluster c; bins beyond
// nd * ng stay 0.  Intensity is rgbToIntensity of each point's colour, so PointT needs PCL's r, g, b members.  Clusters are copied into
// one concatenated cloud for the call.
template <typename PointT>
inline void processRIFTBatched(const std::vector<typename search::GridSearch<PointT>::PointCloudConstPtr> &clusters,
                               std::vector<std::vector<Histogram32> > &descriptors, std::vector<std::vector<int> > &kept_rows, double normal_radius = 0.03,
                               double gradient_radius = 0.03, double rift_radius = 0.05, int nr_distance_bins = 4, int nr_gradient_bins = 8, int device = 0) {
    std::vector<PointT> all;
    std::vector<float> inten;
    std::vector<int64_t> off(1, 0);
    for (const auto &c : clusters) {
        if (!c) throw Error("processRIFTBatched: null input cloud");
        for (const PointT &p : c->points) { all.push_back(p); inten.push_back(rgbToIntensity(p.r, p.g, p.b)); }
        off.push_back((int64_t)all.size());
    }
    const int64_t n_clouds = (int64_t)clusters.size(), n = (int64_t)all.size();
    const int nb = nr_distance_bins * nr_gradient_bins;
    std::vector<int64_t> desc_off(off.size());
    std::vector<float> flat((size_t)std::max<int64_t>(n, 1) * (size_t)std::max(nb, 1));
    std::vector<int32_t> rows((size_t)std::max<int64_t>(n, 1));
    pcc_index *ws = nullptr;
    check(pcc_create(device, &ws));
    // at most one descriptor per point: a cap of n always holds the result
    const int rc = pcc_rift_batched(ws, all.data(), n, (int)sizeof(PointT), inten.data(), off.data(), n_clouds, normal_radius, gradient_radius, rift_radius,
                                    nr_distance_bins, nr_gradient_bins, flat.data(), rows.data(), n, desc_off.data(), PCC_HOST, nullptr);
    pcc_destroy(ws);
    check(rc);
    descriptors.assign((size_t)n_clouds, std::vector<Histogram32>());
    kept_rows.assign((size_t)n_clouds, std::vector<int>());
    for (int64_t c = 0; c < n_clouds; ++c) {
        for (int64_t i = desc_off[c]; i < desc_off[c + 1]; ++i) {
            Histogram32 h;
            for (int k = 0; k < 32; ++k) h.histogram[k] = k < nb ? flat[(size_t)i * nb + k] : 0.f;
            descriptors[c].push_back(h);
            kept_rows[c].push_back(rows[(size_t)i]);
        }
    }
}

// matchRIFTFeaturesKnn (src/comparator.cpp:560-588): KdTreeFLANN<Histogram<32>> over descriptors1, nearestKSearch(k = 1) for every
// descriptor of descriptors2, kept when the squared distance is < 0.05.  The returned vector starts with one 0, as the reference's
// `std::vector<int> correspondence(1)` does (its callers use size()).  HistT is any POD whose first floats are the histogram
// (pcl::Histogram<32>: 32 floats).  match_dims = 3 reproduces the reference binary, where PCL 1.7's DefaultPointRepresentation
// clamps the unregistered Histogram<32> to its first three floats; match_dims = 32 matches on the whole histogram (INTEGRATION.md).
template <typename HistT>
inline std::vector<int> matchRIFTFeaturesKnn(const std::vector<HistT> &descriptors1, const std::vector<HistT> &descriptors2, int match_dims = 3,
                                             float threshold = 0.05f, int device = 0) {
    static_assert(sizeof(HistT) % sizeof(float) == 0, "descriptor rows must be whole floats");
    std::vector<int> correspondence(1);
    if (descriptors1.empty() || descriptors2.empty()) return correspondence;
    pcc_index *ws = nullptr;
    check(pcc_create(device, &ws));
    std::vector<int32_t> idx(descriptors2.size()); std::vector<float> d2(descriptors2.size());
    const int rc = pcc_descriptor_nn(ws, reinterpret_cast<const float *>(descriptors1.data()), (int64_t)descriptors1.size(),
                                     reinterpret_cast<const float *>(descriptors2.data()), (int64_t)descriptors2.size(), match_dims,
                                     (int)(sizeof(HistT) / sizeof(float)), idx.data(), d2.data(), PCC_HOST, nullptr);
    pcc_destroy(ws);
    check(rc);
    for (size_t i = 0; i < idx.size(); ++i) if (idx[i] >= 0 && d2[i] < threshold) correspondence.push_back(idx[i]);
    return correspondence;
}

}  // namespace pcc
#endif  // PCC_GRID_SEARCH_HPP_
