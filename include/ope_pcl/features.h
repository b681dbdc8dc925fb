// ope_pcl/features.h — pcl::NormalEstimation and pcl::FPFHEstimation with the call surface the reference uses:
//   NormalEstimation<PointT, PointOutT>  setSearchMethod, setKSearch or setRadiusSearch, setInputCloud, compute
//                                        (D&L/src/poseestimator.cpp:151-156; BM/src/regmeshpcd.cpp:74-90). As in PCL's
//                                        Feature::initCompute, exactly one of k and the radius must be set: k > 0 runs
//                                        ope_normals_knn, a radius > 0 runs ope_normals_radius, both or neither print PCL's
//                                        error and compute nothing.
//   FPFHEstimation<PointT, Normal, FPFHSignature33>  setInputCloud, setRadiusSearch, setInputNormals, compute
//                                        (D&L/src/poseestimator.cpp:121-125)
// compute() uploads the cloud, runs the device kernels (ope_normals_knn / ope_normals_radius / ope_fpfh) and writes the caller's output
// cloud; nothing is computed on the host.
#pragma once
#include "filters.h"

namespace OPE_PCL_NAMESPACE {

template <typename PointInT, typename PointOutT>
class Feature : public PCLBase<PointInT> {
 public:
  typedef typename search::KdTree<PointInT>::Ptr KdTreePtr;
  void setSearchMethod(const KdTreePtr& tree) { tree_ = tree; }
  KdTreePtr getSearchMethod() const { return tree_; }
  void setKSearch(int k) { k_ = k; }
  int getKSearch() const { return k_; }
  void setRadiusSearch(double r) { search_radius_ = r; }
  double getRadiusSearch() const { return search_radius_; }

 protected:
  KdTreePtr tree_;
  int k_ = 0;
  double search_radius_ = 0.0;
};

// ---- pcl::NormalEstimation ----------------------------------------------------------------------------------------------
template <typename PointInT, typename PointOutT>
class NormalEstimation : public Feature<PointInT, PointOutT> {
 public:
  using PCLBase<PointInT>::input_;
  using Feature<PointInT, PointOutT>::k_;
  using Feature<PointInT, PointOutT>::search_radius_;
  void setViewPoint(float vpx, float vpy, float vpz) { vp_[0] = vpx; vp_[1] = vpy; vp_[2] = vpz; use_sensor_origin_ = false; }
  // writes normal_x/y/z and curvature of every output point; other fields of PointOutT are left alone (SURVEY A.4)
  void compute(PointCloud<PointOutT>& output) {
    if (!input_) { detail::pcl_error("pcl::NormalEstimation::compute", "No input dataset given!"); output.clear(); return; }
    const size_t n = input_->points.size();
    output.points.resize(n);
    output.width = input_->width ? input_->width : (std::uint32_t)n;
    output.height = input_->height ? input_->height : 1;
    output.is_dense = true;
    if (n == 0) return;
    if (search_radius_ != 0.0 && k_ != 0) {
      char msg[160];
      std::snprintf(msg, sizeof(msg), "Both radius (%f) and K (%d) defined! Set one of them to zero first and then re-run compute ().",
                    search_radius_, k_);
      detail::pcl_error("pcl::NormalEstimation::compute", msg);
      return;
    }
    if (!(search_radius_ > 0) && k_ <= 0) {
      detail::pcl_error("pcl::NormalEstimation::compute", "Neither radius nor K defined! Set one of them to a positive number first and then re-run compute ().");
      return;
    }
    ope_ctx* ctx = detail::context();
    detail::DeviceCloud dc;
    if (!ctx || !detail::upload(*input_, dc, "pcl::NormalEstimation::compute")) return;
    float vp[3] = {vp_[0], vp_[1], vp_[2]};
    if (use_sensor_origin_) { vp[0] = input_->sensor_origin_[0]; vp[1] = input_->sensor_origin_[1]; vp[2] = input_->sensor_origin_[2]; }
    std::vector<float> out4(4 * n);
    const int rc = k_ > 0 ? ope_normals_knn(ctx, dc.get(), k_, vp, out4.data())
                          : ope_normals_radius(ctx, dc.get(), (float)search_radius_, vp, out4.data());
    if (!detail::check(rc, "pcl::NormalEstimation::compute")) return;
    for (size_t i = 0; i < n; ++i) {
      PointOutT& o = output.points[i];
      o.normal_x = out4[4 * i]; o.normal_y = out4[4 * i + 1]; o.normal_z = out4[4 * i + 2]; o.curvature = out4[4 * i + 3];
      if (!std::isfinite(o.normal_x)) output.is_dense = false;
    }
  }

 private:
  float vp_[3] = {0, 0, 0};
  bool use_sensor_origin_ = true;
};

// ---- pcl::FPFHEstimation ------------------------------------------------------------------------------------------------
template <typename PointInT, typename PointNT, typename PointOutT = FPFHSignature33>
class FPFHEstimation : public Feature<PointInT, PointOutT> {
 public:
  using PCLBase<PointInT>::input_;
  using Feature<PointInT, PointOutT>::search_radius_;
  typedef typename PointCloud<PointNT>::ConstPtr PointCloudNConstPtr;
  void setInputNormals(const PointCloudNConstPtr& normals) { normals_ = normals; }
  void compute(PointCloud<PointOutT>& output) {
    if (!input_) { detail::pcl_error("pcl::FPFHEstimation::compute", "No input dataset given!"); output.clear(); return; }
    if (!normals_) { detail::pcl_error("pcl::FPFHEstimation::compute", "No input dataset containing normals was given!"); output.clear(); return; }
    const size_t n = input_->points.size();
    output.points.resize(n);
    output.width = (std::uint32_t)n; output.height = 1; output.is_dense = true;
    if (n == 0) return;
    if (!(search_radius_ > 0)) { detail::pcl_error("pcl::FPFHEstimation::compute", "only setRadiusSearch(r) is supported (D&L/src/poseestimator.cpp:122)"); return; }
    ope_ctx* ctx = detail::context();
    detail::DeviceCloud dc;
    if (!ctx || !detail::upload_with_normals(*input_, *normals_, dc, "pcl::FPFHEstimation::compute")) { output.clear(); return; }
    static_assert(sizeof(PointOutT) == 33 * sizeof(float), "FPFHSignature33");
    if (!detail::check(ope_fpfh(ctx, dc.get(), (float)search_radius_, reinterpret_cast<float*>(output.points.data()), nullptr),
                       "pcl::FPFHEstimation::compute")) return;
    for (size_t i = 0; i < n && output.is_dense; ++i)
      if (!std::isfinite(output.points[i].histogram[0])) output.is_dense = false;
  }

 private:
  PointCloudNConstPtr normals_;
};

}  // namespace OPE_PCL_NAMESPACE
