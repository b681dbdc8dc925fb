// ope_pcl/registration.h — the PCL-style Registration API of the reference, backed by libope_cuda.so.
//
//   pcl::Registration<Src, Tgt, Scalar>            VP/registration_mod.h:68-610, VP/impl/registration_mod.hpp:57-219
//   pcl::IterativeClosestPoint / ...WithNormals    VP/icp_mod.h:92-379, VP/impl/icp_mod.hpp:118-318
//   pcl::SampleConsensusInitialAlignment           [UPSTREAM ia_ransac.h]; call site D&L/src/poseestimator.cpp:50-65
//   pcl::registration::CorrespondenceEstimation / CorrespondenceEstimationNormalShooting
//                                                   VP/correspondence_estimation_mod.h, VP/impl/..normal_shooting_weighted.hpp:104-145
//   pcl::registration::CorrespondenceRejectorSurfaceNormal / SelfOccludedNormal
//                                                   VP/correspondence_rejection_mod.h:368-391, VP/impl/..self_occluded_normal.cpp:43-64
//   pcl::registration::TransformationEstimationSVD / PointToPlane / PointToPlaneLLS
//                                                   call sites D&L/src/poseestimator.cpp:298-306,341,435; BM/src/regmeshpcd.cpp:162,193
//
// Same setters, same defaults, same error behaviour (PCL_ERROR-style line on stderr, no exception, transforms left at
// identity); the bodies marshal the configuration into ope_icp_params / ope_sacia_params and call ope_icp_align /
// ope_sacia_align / ope_fitness. Clouds are uploaded once per setInputSource/setInputTarget and stay on the device; the
// target's spatial index is rebuilt when the target changes (target_cloud_updated_, VP/impl/registration_mod.hpp:57-67,80-84).
#pragma once
#include <cfloat>
#include <string>

#include "features.h"

namespace OPE_PCL_NAMESPACE {
namespace registration {

// ---- correspondence estimation ------------------------------------------------------------------------------------------
template <typename PointSource, typename PointTarget, typename Scalar = float>
class CorrespondenceEstimationBase {
 public:
  typedef std::shared_ptr<CorrespondenceEstimationBase<PointSource, PointTarget, Scalar>> Ptr;
  typedef typename PointCloud<PointSource>::ConstPtr PointCloudSourceConstPtr;
  typedef typename PointCloud<PointTarget>::ConstPtr PointCloudTargetConstPtr;
  virtual ~CorrespondenceEstimationBase() {}
  void setInputSource(const PointCloudSourceConstPtr& cloud) { input_ = cloud; src_dirty_ = true; }
  void setInputCloud(const PointCloudSourceConstPtr& cloud) { setInputSource(cloud); }  // deprecated PCL spelling
  void setInputTarget(const PointCloudTargetConstPtr& cloud) { target_ = cloud; tgt_dirty_ = true; }
  PointCloudSourceConstPtr getInputSource() const { return input_; }
  PointCloudTargetConstPtr getInputTarget() const { return target_; }
  // which estimator the ICP loop should run on the device (OPE_EST_*) and its k
  virtual int opeEstimator() const = 0;
  virtual int opeKSearch() const { return 1; }

  // one estimation pass on the clouds as given (D&L/src/poseestimator.cpp:247)
  virtual void determineCorrespondences(Correspondences& correspondences, double max_distance = std::numeric_limits<double>::max()) {
    correspondences.clear();
    if (!input_ || !target_ || target_->points.empty()) { detail::pcl_error("pcl::registration::CorrespondenceEstimation::compute", "No input target dataset was given!"); return; }
    ope_ctx* ctx = detail::context();
    if (!ctx || !sync()) return;
    ope_icp_params prm;
    ope_icp_params_default(&prm);
    prm.estimator = opeEstimator();
    prm.k_search = opeKSearch();
    prm.max_correspondence_distance = max_distance;
    std::vector<ope_correspondence> out(input_->points.size() + 1);
    size_t n = 0;
    if (!detail::check(ope_correspondences(ctx, dsrc_.get(), dtgt_.get(), &prm, out.data(), &n), "determineCorrespondences")) return;
    correspondences.resize(n);
    for (size_t i = 0; i < n; ++i) correspondences[i] = Correspondence(out[i].index_query, out[i].index_match, out[i].distance);
  }

 protected:
  virtual bool sync() {
    if (src_dirty_) { if (!detail::upload(*input_, dsrc_, "CorrespondenceEstimation::setInputSource")) return false; src_dirty_ = false; }
    if (tgt_dirty_) { if (!detail::upload(*target_, dtgt_, "CorrespondenceEstimation::setInputTarget")) return false; tgt_dirty_ = false; }
    return true;
  }
  PointCloudSourceConstPtr input_;
  PointCloudTargetConstPtr target_;
  detail::DeviceCloud dsrc_, dtgt_;
  bool src_dirty_ = true, tgt_dirty_ = true;
};

template <typename PointSource, typename PointTarget, typename Scalar = float>
class CorrespondenceEstimation : public CorrespondenceEstimationBase<PointSource, PointTarget, Scalar> {
 public:
  typedef std::shared_ptr<CorrespondenceEstimation<PointSource, PointTarget, Scalar>> Ptr;
  int opeEstimator() const override { return OPE_EST_NEAREST; }
};

template <typename PointSource, typename PointTarget, typename NormalT, typename Scalar = float>
class CorrespondenceEstimationNormalShooting : public CorrespondenceEstimationBase<PointSource, PointTarget, Scalar> {
  typedef CorrespondenceEstimationBase<PointSource, PointTarget, Scalar> Base;

 public:
  typedef std::shared_ptr<CorrespondenceEstimationNormalShooting<PointSource, PointTarget, NormalT, Scalar>> Ptr;
  typedef typename PointCloud<NormalT>::ConstPtr NormalsConstPtr;
  void setSourceNormals(const NormalsConstPtr& normals) { source_normals_ = normals; this->src_dirty_ = true; }
  NormalsConstPtr getSourceNormals() const { return source_normals_; }
  void setKSearch(unsigned int k) { k_ = k; }
  unsigned int getKSearch() const { return k_; }
  int opeEstimator() const override { return OPE_EST_NORMAL_SHOOTING; }
  int opeKSearch() const override { return (int)k_; }

 protected:
  bool sync() override {
    if (this->src_dirty_) {
      if (!source_normals_) { detail::pcl_error("pcl::registration::CorrespondenceEstimationNormalShooting::initCompute", "Datasets containing normals for source have not been given!"); return false; }
      if (!detail::upload_with_normals(*this->input_, *source_normals_, this->dsrc_, "CorrespondenceEstimationNormalShooting")) return false;
      this->src_dirty_ = false;
    }
    return Base::sync();
  }
  NormalsConstPtr source_normals_;
  unsigned int k_ = 10;  // [UPSTREAM] default
};

// ---- correspondence rejection --------------------------------------------------------------------------------------------
class CorrespondenceRejector {
 public:
  typedef std::shared_ptr<CorrespondenceRejector> Ptr;
  virtual ~CorrespondenceRejector() {}
  virtual int opeKind() const = 0;        // OPE_REJ_*
  virtual double opeThreshold() const = 0;
  virtual const std::string& getClassName() const { return name_; }

 protected:
  std::string name_ = "CorrespondenceRejector";
};

// keep iff n_src . n_tgt > threshold (VP/correspondence_rejection_mod.h:368-376). The standalone pass
// (getRemainingCorrespondences, D&L/src/poseestimator.cpp:264-273) scores on the host exactly like DataContainer does:
// a double-precision dot product of the float normals.
class CorrespondenceRejectorSurfaceNormal : public CorrespondenceRejector {
 public:
  typedef std::shared_ptr<CorrespondenceRejectorSurfaceNormal> Ptr;
  CorrespondenceRejectorSurfaceNormal() { name_ = "CorrespondenceRejectorSurfaceNormal"; }
  template <typename PointT, typename NormalT> void initializeDataContainer() {}
  template <typename PointT> void setInputSource(const typename PointCloud<PointT>::ConstPtr&) {}
  template <typename PointT> void setInputCloud(const typename PointCloud<PointT>::ConstPtr&) {}
  template <typename PointT> void setInputTarget(const typename PointCloud<PointT>::ConstPtr&) {}
  template <typename PointT, typename NormalT> void setInputNormals(const typename PointCloud<NormalT>::ConstPtr& n) { copy_normals(*n, src_n_); }
  template <typename PointT, typename NormalT> void setTargetNormals(const typename PointCloud<NormalT>::ConstPtr& n) { copy_normals(*n, tgt_n_); }
  void setThreshold(double threshold) { threshold_ = threshold; }
  double getThreshold() const { return threshold_; }
  void getRemainingCorrespondences(const Correspondences& in, Correspondences& out) {
    out.clear();
    for (const Correspondence& c : in) {
      if (c.index_query < 0 || (size_t)c.index_query * 3 + 2 >= src_n_.size() || c.index_match < 0 || (size_t)c.index_match * 3 + 2 >= tgt_n_.size()) continue;
      const float* a = &src_n_[3 * (size_t)c.index_query];
      const float* b = &tgt_n_[3 * (size_t)c.index_match];
      const double score = (double)((a[0] * b[0]) + (a[1] * b[1]) + (a[2] * b[2]));
      if (score > threshold_) out.push_back(c);
    }
  }
  int opeKind() const override { return OPE_REJ_SURFACE_NORMAL; }
  double opeThreshold() const override { return threshold_; }

 private:
  template <typename NormalT> static void copy_normals(const PointCloud<NormalT>& c, std::vector<float>& v) {
    v.resize(3 * c.points.size());
    for (size_t i = 0; i < c.points.size(); ++i) { v[3 * i] = c.points[i].normal_x; v[3 * i + 1] = c.points[i].normal_y; v[3 * i + 2] = c.points[i].normal_z; }
  }
  double threshold_ = 1.0;  // [UPSTREAM] default
  std::vector<float> src_n_, tgt_n_;
};

// keep iff n_src . (-p_src / |p_src|) > threshold (VP/correspondence_rejection_mod.h:382-391)
class CorrespondenceRejectorSelfOccludedNormal : public CorrespondenceRejector {
 public:
  typedef std::shared_ptr<CorrespondenceRejectorSelfOccludedNormal> Ptr;
  CorrespondenceRejectorSelfOccludedNormal() { name_ = "CorrespondenceRejectorSelfOccludedNormal"; }
  void setThreshold(double threshold) { threshold_ = threshold; }
  double getThreshold() const { return threshold_; }
  int opeKind() const override { return OPE_REJ_SELF_OCCLUDED_NORMAL; }
  double opeThreshold() const override { return threshold_; }

 private:
  double threshold_ = 1.0;
};

// ---- transformation estimation ---------------------------------------------------------------------------------------------
template <typename PointSource, typename PointTarget, typename Scalar = float>
class TransformationEstimation {
 public:
  typedef std::shared_ptr<TransformationEstimation<PointSource, PointTarget, Scalar>> Ptr;
  typedef Eigen::Matrix4f Matrix4;
  virtual ~TransformationEstimation() {}
  virtual int opeKind() const = 0;  // OPE_TE_*, or a negative value for estimators the device loop does not implement
};

template <typename PointSource, typename PointTarget, typename Scalar = float>
class TransformationEstimationSVD : public TransformationEstimation<PointSource, PointTarget, Scalar> {
 public:
  typedef std::shared_ptr<TransformationEstimationSVD<PointSource, PointTarget, Scalar>> Ptr;
  typedef Eigen::Matrix4f Matrix4;
  int opeKind() const override { return OPE_TE_SVD; }
  // identity correspondences over the whole clouds (D&L/src/poseestimator.cpp:429-435)
  void estimateRigidTransformation(const PointCloud<PointSource>& src, const PointCloud<PointTarget>& tgt, Matrix4& T) const {
    T.setIdentity();
    if (src.points.size() != tgt.points.size()) { detail::pcl_error("pcl::TransformationEstimationSVD::estimateRigidTransformation", "Number or points in source differs than target!"); return; }
    run(src, tgt, nullptr, nullptr, src.points.size(), T);
  }
  void estimateRigidTransformation(const PointCloud<PointSource>& src, const PointCloud<PointTarget>& tgt,
                                   const Correspondences& corr, Matrix4& T) const {
    T.setIdentity();
    std::vector<int32_t> is(corr.size()), it(corr.size());
    for (size_t i = 0; i < corr.size(); ++i) { is[i] = corr[i].index_query; it[i] = corr[i].index_match; }
    run(src, tgt, is.data(), it.data(), corr.size(), T);
  }

 private:
  static void run(const PointCloud<PointSource>& src, const PointCloud<PointTarget>& tgt, const int32_t* is, const int32_t* it, size_t n,
                  Matrix4& T) {
    ope_ctx* ctx = detail::context();
    detail::DeviceCloud a, b;
    if (!ctx || n == 0 || !detail::upload(src, a, "TransformationEstimationSVD") || !detail::upload(tgt, b, "TransformationEstimationSVD")) return;
    float M[16];
    if (detail::check(ope_umeyama(ctx, a.get(), b.get(), is, it, n, M), "pcl::TransformationEstimationSVD::estimateRigidTransformation"))
      T = detail::from_c(M);
  }
};
// shared front end of TransformationEstimationPointToPlaneLLS / TransformationEstimationPointToPlane
template <typename PointSource, typename PointTarget, typename Scalar, int Kind>
class TransformationEstimationPointToPlaneBase : public TransformationEstimation<PointSource, PointTarget, Scalar> {
 public:
  typedef Eigen::Matrix4f Matrix4;
  int opeKind() const override { return Kind; }
  void estimateRigidTransformation(const PointCloud<PointSource>& src, const PointCloud<PointTarget>& tgt, Matrix4& T) const {
    T.setIdentity();
    if (src.points.size() != tgt.points.size()) { detail::pcl_error(name(), "Number or points in source differs than target!"); return; }
    run(src, tgt, nullptr, nullptr, src.points.size(), T);
  }
  void estimateRigidTransformation(const PointCloud<PointSource>& src, const PointCloud<PointTarget>& tgt,
                                   const Correspondences& corr, Matrix4& T) const {
    T.setIdentity();
    std::vector<int32_t> is(corr.size()), it(corr.size());
    for (size_t i = 0; i < corr.size(); ++i) { is[i] = corr[i].index_query; it[i] = corr[i].index_match; }
    run(src, tgt, is.data(), it.data(), corr.size(), T);
  }

 private:
  // the target point type carries the normals (PointXYZRGBNormal / PointNormal), as PCL requires of these estimators;
  // detail::upload() takes normal_x.. along when PointT has them
  static void run(const PointCloud<PointSource>& src, const PointCloud<PointTarget>& tgt, const int32_t* is, const int32_t* it, size_t n,
                  Matrix4& T) {
    ope_ctx* ctx = detail::context();
    detail::DeviceCloud a, b;
    if (!ctx || n == 0 || !detail::upload(src, a, name()) || !detail::upload(tgt, b, name())) return;
    float M[16];
    if (detail::check(ope_point_to_plane(ctx, a.get(), b.get(), is, it, n, Kind, M, nullptr), name())) T = detail::from_c(M);
  }
  static const char* name() {
    return Kind == OPE_TE_POINT_TO_PLANE_LLS ? "pcl::registration::TransformationEstimationPointToPlaneLLS::estimateRigidTransformation"
                                             : "pcl::registration::TransformationEstimationLM::estimateRigidTransformation";
  }
};
// 6x6 linear least squares, the default of IterativeClosestPointWithNormals (VP/icp_mod.h:352-357)
template <typename PointSource, typename PointTarget, typename Scalar = float>
class TransformationEstimationPointToPlaneLLS
    : public TransformationEstimationPointToPlaneBase<PointSource, PointTarget, Scalar, OPE_TE_POINT_TO_PLANE_LLS> {
 public:
  typedef std::shared_ptr<TransformationEstimationPointToPlaneLLS<PointSource, PointTarget, Scalar>> Ptr;
};
// Levenberg-Marquardt over the 6-parameter rigid warp, what BuildModel plugs in (BM/src/regmeshpcd.cpp:162,193)
template <typename PointSource, typename PointTarget, typename Scalar = float>
class TransformationEstimationPointToPlane
    : public TransformationEstimationPointToPlaneBase<PointSource, PointTarget, Scalar, OPE_TE_POINT_TO_PLANE> {
 public:
  typedef std::shared_ptr<TransformationEstimationPointToPlane<PointSource, PointTarget, Scalar>> Ptr;
};

// DefaultConvergenceCriteria::ConvergenceState (VP/default_convergence_criteria_mod.h:73-81)
template <typename Scalar = float>
struct DefaultConvergenceCriteria {
  enum ConvergenceState {
    CONVERGENCE_CRITERIA_NOT_CONVERGED = OPE_CONV_NOT_CONVERGED,
    CONVERGENCE_CRITERIA_ITERATIONS = OPE_CONV_ITERATIONS,
    CONVERGENCE_CRITERIA_TRANSFORM = OPE_CONV_TRANSFORM,
    CONVERGENCE_CRITERIA_ABS_MSE = OPE_CONV_ABS_MSE,
    CONVERGENCE_CRITERIA_REL_MSE = OPE_CONV_REL_MSE,
    CONVERGENCE_CRITERIA_NO_CORRESPONDENCES = OPE_CONV_NO_CORRESPONDENCES
  };
};

}  // namespace registration

// ---- pcl::Registration ------------------------------------------------------------------------------------------------------
template <typename PointSource, typename PointTarget, typename Scalar = float>
class Registration {
 public:
  typedef Eigen::Matrix4f Matrix4;
  typedef PointCloud<PointSource> PointCloudSource;
  typedef typename PointCloudSource::Ptr PointCloudSourcePtr;
  typedef typename PointCloudSource::ConstPtr PointCloudSourceConstPtr;
  typedef PointCloud<PointTarget> PointCloudTarget;
  typedef typename PointCloudTarget::ConstPtr PointCloudTargetConstPtr;
  typedef typename search::KdTree<PointTarget>::Ptr KdTreePtr;
  typedef typename search::KdTree<PointSource>::Ptr KdTreeReciprocalPtr;
  typedef typename registration::TransformationEstimation<PointSource, PointTarget, Scalar>::Ptr TransformationEstimationPtr;
  typedef typename registration::CorrespondenceEstimationBase<PointSource, PointTarget, Scalar>::Ptr CorrespondenceEstimationPtr;
  typedef registration::CorrespondenceRejector::Ptr CorrespondenceRejectorPtr;

  // defaults: VP/registration_mod.h:102-130
  Registration()
      : final_transformation_(Matrix4::Identity()), transformation_(Matrix4::Identity()), previous_transformation_(Matrix4::Identity()) {}
  virtual ~Registration() {}

  void setTransformationEstimation(const TransformationEstimationPtr& te) { transformation_estimation_ = te; }
  void setCorrespondenceEstimation(const CorrespondenceEstimationPtr& ce) { correspondence_estimation_ = ce; }
  virtual void setInputSource(const PointCloudSourceConstPtr& cloud) {
    if (!cloud || cloud->points.empty()) { detail::pcl_error(reg_name_.c_str(), "setInputSource: Invalid or empty point cloud dataset given!"); return; }
    input_ = cloud; source_cloud_updated_ = true;
  }
  void setInputCloud(const PointCloudSourceConstPtr& cloud) { setInputSource(cloud); }  // PCL 1.7 deprecated spelling
  PointCloudSourceConstPtr const getInputSource() { return input_; }
  virtual void setInputTarget(const PointCloudTargetConstPtr& cloud) {
    if (!cloud || cloud->points.empty()) { detail::pcl_error(reg_name_.c_str(), "setInputTarget: Invalid or empty point cloud dataset given!"); return; }
    target_ = cloud; target_cloud_updated_ = true;
  }
  PointCloudTargetConstPtr const getInputTarget() { return target_; }
  // the index lives on the device with the target cloud; the tree object is accepted and kept for API compatibility
  void setSearchMethodTarget(const KdTreePtr& tree, bool force_no_recompute = false) { tree_ = tree; force_no_recompute_ = force_no_recompute; }
  KdTreePtr getSearchMethodTarget() const { return tree_; }
  void setSearchMethodSource(const KdTreeReciprocalPtr& tree, bool force_no_recompute = false) { tree_reciprocal_ = tree; (void)force_no_recompute; }
  KdTreeReciprocalPtr getSearchMethodSource() const { return tree_reciprocal_; }
  Matrix4 getFinalTransformation() { return final_transformation_; }
  Matrix4 getLastIncrementalTransformation() { return transformation_; }
  void setMaximumIterations(int nr_iterations) { max_iterations_ = nr_iterations; }
  int getMaximumIterations() { return max_iterations_; }
  void setRANSACIterations(int ransac_iterations) { ransac_iterations_ = ransac_iterations; }
  double getRANSACIterations() { return ransac_iterations_; }
  void setRANSACOutlierRejectionThreshold(double inlier_threshold) { inlier_threshold_ = inlier_threshold; }
  double getRANSACOutlierRejectionThreshold() { return inlier_threshold_; }
  void setMaxCorrespondenceDistance(double distance_threshold) { corr_dist_threshold_ = distance_threshold; }
  double getMaxCorrespondenceDistance() { return corr_dist_threshold_; }
  void setTransformationEpsilon(double epsilon) { transformation_epsilon_ = epsilon; }
  double getTransformationEpsilon() { return transformation_epsilon_; }
  void setEuclideanFitnessEpsilon(double epsilon) { euclidean_fitness_epsilon_ = epsilon; }
  double getEuclideanFitnessEpsilon() { return euclidean_fitness_epsilon_; }
  void addCorrespondenceRejector(const CorrespondenceRejectorPtr& rejector) { correspondence_rejectors_.push_back(rejector); }
  std::vector<CorrespondenceRejectorPtr> getCorrespondenceRejectors() { return correspondence_rejectors_; }
  bool removeCorrespondenceRejector(unsigned int i) {
    if (i >= correspondence_rejectors_.size()) return false;
    correspondence_rejectors_.erase(correspondence_rejectors_.begin() + i);
    return true;
  }
  void clearCorrespondenceRejectors() { correspondence_rejectors_.clear(); }
  bool hasConverged() { return converged_; }
  const std::string& getClassName() const { return reg_name_; }

  // mean squared nearest-neighbour distance of the transformed source (VP/impl/registration_mod.hpp:131-165)
  double getFitnessScore(double max_range = std::numeric_limits<double>::max()) {
    ope_ctx* ctx = detail::context();
    if (!ctx || !input_ || !target_ || !sync_clouds()) return std::numeric_limits<double>::max();
    float T[16];
    detail::to_c(final_transformation_, T);
    double out = std::numeric_limits<double>::max();
    detail::check(ope_fitness(ctx, dsrc_.get(), dtgt_.get(), T, max_range, &out), "pcl::Registration::getFitnessScore");
    return out;
  }

  void align(PointCloudSource& output) { align(output, Matrix4::Identity()); }
  // VP/impl/registration_mod.hpp:176-219
  void align(PointCloudSource& output, const Matrix4& guess) {
    if (!initCompute()) return;
    // resize / copy the output from the input (:182-201)
    output.points = input_->points;
    output.width = (std::uint32_t)input_->points.size(); output.height = 1; output.is_dense = input_->is_dense;
    output.sensor_origin_ = input_->sensor_origin_;
    converged_ = false;
    final_transformation_ = transformation_ = previous_transformation_ = Matrix4::Identity();
    computeTransformation(output, guess);
  }

 protected:
  virtual void computeTransformation(PointCloudSource& output, const Matrix4& guess) = 0;

  // Registration::initCompute, VP/impl/registration_mod.hpp:70-98
  bool initCompute() {
    if (!target_) { detail::pcl_error((reg_name_ + "::compute").c_str(), "No input target dataset was given!"); return false; }
    if (!input_) { detail::pcl_error((reg_name_ + "::compute").c_str(), "No input source dataset was given!"); return false; }
    return detail::context() != nullptr && sync_clouds();
  }
  // PCL re-reads *input_ / *target_ on every align(): a cloud modified in place since the last upload (the reference does
  // `*p_sourceCloud = *alignedCloud` and aligns again) is detected by its fingerprint and uploaded again; a changed target also
  // drops its search index, like target_cloud_updated_ does to the kd-tree (VP/impl/registration_mod.hpp:80-84)
  bool sync_clouds() {
    const detail::CloudFingerprint fs = detail::fingerprint(*input_), ft = detail::fingerprint(*target_);
    if (source_cloud_updated_ || fs != src_print_) {
      if (!detail::upload(*input_, dsrc_, reg_name_.c_str())) return false;
      source_cloud_updated_ = false; src_print_ = fs;
    }
    if (target_cloud_updated_ || ft != tgt_print_) {
      if (!detail::upload(*target_, dtgt_, reg_name_.c_str())) return false;
      target_cloud_updated_ = false; tgt_print_ = ft;
    }
    return true;
  }
  detail::CloudFingerprint src_print_, tgt_print_;
  // download a device cloud (`output`, same size and order as input_) into the caller's point structs
  void fetch_output(ope_cloud* aligned, PointCloudSource& output) {
    ope_ctx* ctx = detail::context();
    const size_t n = output.points.size();
    if (!ctx || !aligned || n != ope_cloud_size(aligned)) return;
    std::vector<float> xyz(3 * n), nrm;
    const bool with_n = detail::has_normal<PointSource>::value && ope_cloud_has_normals(aligned);
    if (with_n) nrm.resize(4 * n);
    if (!detail::check(ope_cloud_download(ctx, aligned, xyz.data(), with_n ? nrm.data() : nullptr), "align: download")) return;
    for (size_t i = 0; i < n; ++i) {
      output.points[i].x = xyz[3 * i]; output.points[i].y = xyz[3 * i + 1]; output.points[i].z = xyz[3 * i + 2];
      if (with_n) set_normal(output.points[i], &nrm[4 * i], detail::has_normal<PointSource>());
    }
  }
  template <typename P> static void set_normal(P& p, const float* v, std::true_type) { p.normal_x = v[0]; p.normal_y = v[1]; p.normal_z = v[2]; }
  template <typename P> static void set_normal(P&, const float*, std::false_type) {}

  std::string reg_name_ = "Registration";
  KdTreePtr tree_;
  KdTreeReciprocalPtr tree_reciprocal_;
  bool force_no_recompute_ = false;
  int nr_iterations_ = 0;
  int max_iterations_ = 10;
  int ransac_iterations_ = 0;
  PointCloudSourceConstPtr input_;
  PointCloudTargetConstPtr target_;
  Matrix4 final_transformation_, transformation_, previous_transformation_;
  double transformation_epsilon_ = 0.0;
  double euclidean_fitness_epsilon_ = -std::numeric_limits<double>::max();
  double corr_dist_threshold_ = std::sqrt(std::numeric_limits<double>::max());
  double inlier_threshold_ = 0.05;
  bool converged_ = false;
  int min_number_correspondences_ = 3;
  CorrespondenceEstimationPtr correspondence_estimation_;
  TransformationEstimationPtr transformation_estimation_;
  std::vector<CorrespondenceRejectorPtr> correspondence_rejectors_;
  bool target_cloud_updated_ = true, source_cloud_updated_ = true;
  detail::DeviceCloud dsrc_, dtgt_;
};

// ---- pcl::IterativeClosestPoint ---------------------------------------------------------------------------------------------
template <typename PointSource, typename PointTarget, typename Scalar = float>
class IterativeClosestPoint : public Registration<PointSource, PointTarget, Scalar> {
  typedef Registration<PointSource, PointTarget, Scalar> Base;

 public:
  typedef typename Base::Matrix4 Matrix4;
  typedef typename Base::PointCloudSource PointCloudSource;
  typedef std::shared_ptr<IterativeClosestPoint<PointSource, PointTarget, Scalar>> Ptr;
  IterativeClosestPoint() {
    this->reg_name_ = "IterativeClosestPoint";
    // ctor defaults of VP/icp_mod.h:136-152: SVD, nearest-neighbour estimation, no reciprocal correspondences
    this->transformation_estimation_.reset(new registration::TransformationEstimationSVD<PointSource, PointTarget, Scalar>());
    this->correspondence_estimation_.reset(new registration::CorrespondenceEstimation<PointSource, PointTarget, Scalar>());
  }
  void setUseReciprocalCorrespondences(bool use) { use_reciprocal_correspondence_ = use; }
  bool getUseReciprocalCorrespondences() const { return use_reciprocal_correspondence_; }
  // the vendored class's fixed correspondences, VP/icp_mod.h:267-281: the caller keeps ownership; align() rewrites the distances
  // when the nearest-neighbour estimator puts the pairs in front (see ope_icp_align_fixed)
  void setFixedCorrespondences(Correspondences* correspondences) { corres_fixed_ = correspondences; }
  Correspondences& getFixedCorrespondences() { return *corres_fixed_; }
  void clearCorrespondences() { if (corres_fixed_) corres_fixed_->clear(); }
  // additions of the vendored class: VP/icp_mod.h:249-260
  double getAlignStrength() {
    const double total = (double)((this->input_ ? this->input_->points.size() : 0) + (this->target_ ? this->target_->points.size() : 0));
    return total > 0 ? (double)last_.n_correspondences / total : 0.0;
  }
  // DefaultConvergenceCriteria::getConvergenceState of the last align()
  int getConvergenceState() const { return last_.state; }
  int getNumberOfIterations() const { return last_.iterations; }
  // which vendored loop to reproduce (SURVEY 3.2): OPE_ICP_VARIANT_MOD (PCL x.7.2 branch, default) or OPE_ICP_VARIANT_MODCORR
  void setLoopVariant(int variant) { variant_ = variant; }

 protected:
  virtual bool withNormals() const { return false; }
  // VP/impl/icp_mod.hpp:118-272, run as one persistent kernel (DESIGN.md section 4)
  void computeTransformation(PointCloudSource& output, const Matrix4& guess) override {
    ope_ctx* ctx = detail::context();
    ope_icp_params prm;
    ope_icp_params_default(&prm);
    prm.max_iterations = this->max_iterations_;
    prm.transformation_epsilon = this->transformation_epsilon_;
    prm.euclidean_fitness_epsilon = this->euclidean_fitness_epsilon_;
    prm.max_correspondence_distance = this->corr_dist_threshold_;
    prm.min_number_correspondences = this->min_number_correspondences_;
    prm.use_reciprocal = use_reciprocal_correspondence_ ? 1 : 0;
    prm.estimator = this->correspondence_estimation_ ? this->correspondence_estimation_->opeEstimator() : OPE_EST_NEAREST;
    prm.k_search = this->correspondence_estimation_ ? this->correspondence_estimation_->opeKSearch() : 1;
    prm.variant = variant_;
    prm.with_normals = withNormals() ? 1 : 0;
    if (this->correspondence_rejectors_.size() > OPE_MAX_REJECTORS) { detail::pcl_error(this->reg_name_.c_str(), "too many correspondence rejectors"); return; }
    prm.n_rejectors = (int)this->correspondence_rejectors_.size();
    for (int r = 0; r < prm.n_rejectors; ++r) {
      prm.rejector_kind[r] = this->correspondence_rejectors_[r]->opeKind();
      prm.rejector_threshold[r] = this->correspondence_rejectors_[r]->opeThreshold();
    }
    const int te = this->transformation_estimation_ ? this->transformation_estimation_->opeKind() : OPE_TE_SVD;
    if (te < 0) {
      detail::pcl_error(this->reg_name_.c_str(), "this TransformationEstimation is not implemented on the device");
      return;
    }
    prm.transformation = te;
    float G[16];
    detail::to_c(guess, G);
    ope_cloud* aligned = nullptr;
    std::memset(&last_, 0, sizeof(last_));
    static_assert(sizeof(Correspondence) == sizeof(ope_correspondence), "pcl::Correspondence layout");
    const size_t n_fixed = corres_fixed_ ? corres_fixed_->size() : 0;
    const int rc = ope_icp_align_fixed(ctx, this->dsrc_.get(), this->dtgt_.get(), &prm, G,
                                       n_fixed ? reinterpret_cast<ope_correspondence*>(corres_fixed_->data()) : nullptr, n_fixed, &last_,
                                       nullptr, &aligned);
    if (!detail::check(rc, (this->reg_name_ + "::computeTransformation").c_str())) return;
    this->final_transformation_ = detail::from_c(last_.T);
    this->converged_ = last_.converged != 0;
    this->nr_iterations_ = last_.iterations;
    this->fetch_output(aligned, output);
    if (aligned) ope_cloud_free(ctx, aligned);
  }
  bool use_reciprocal_correspondence_ = false;
  Correspondences* corres_fixed_ = nullptr;
  int variant_ = OPE_ICP_VARIANT_MOD;
  ope_reg_result last_{};
};

// VP/icp_mod.h:340-379: default estimator point-to-plane LLS, transformCloud rotates the normals too
template <typename PointSource, typename PointTarget, typename Scalar = float>
class IterativeClosestPointWithNormals : public IterativeClosestPoint<PointSource, PointTarget, Scalar> {
 public:
  typedef std::shared_ptr<IterativeClosestPointWithNormals<PointSource, PointTarget, Scalar>> Ptr;
  IterativeClosestPointWithNormals() {
    this->reg_name_ = "IterativeClosestPointWithNormals";
    this->transformation_estimation_.reset(new registration::TransformationEstimationPointToPlaneLLS<PointSource, PointTarget, Scalar>());
  }

 protected:
  bool withNormals() const override { return true; }
};

// ---- pcl::SampleConsensusInitialAlignment [UPSTREAM ia_ransac.h] ------------------------------------------------------------
template <typename PointSource, typename PointTarget, typename FeatureT>
class SampleConsensusInitialAlignment : public Registration<PointSource, PointTarget> {
  typedef Registration<PointSource, PointTarget> Base;

 public:
  typedef typename Base::Matrix4 Matrix4;
  typedef typename Base::PointCloudSource PointCloudSource;
  typedef typename PointCloud<FeatureT>::ConstPtr FeatureCloudConstPtr;
  SampleConsensusInitialAlignment() { this->reg_name_ = "SampleConsensusInitialAlignment"; this->max_iterations_ = 1000; }
  void setSourceFeatures(const FeatureCloudConstPtr& features) { input_features_ = features; }
  FeatureCloudConstPtr const getSourceFeatures() { return input_features_; }
  void setTargetFeatures(const FeatureCloudConstPtr& features) { target_features_ = features; }
  FeatureCloudConstPtr const getTargetFeatures() { return target_features_; }
  void setMinSampleDistance(float d) { min_sample_distance_ = d; }
  float getMinSampleDistance() { return min_sample_distance_; }
  void setNumberOfSamples(int n) { nr_samples_ = n; }
  int getNumberOfSamples() { return nr_samples_; }
  void setCorrespondenceRandomness(int k) { k_correspondences_ = k; }
  int getCorrespondenceRandomness() { return k_correspondences_; }
  // replay a pre-drawn libc rand() decision table instead of drawing from rand() (parity tests, sharded pools)
  void setDecisionTable(const ope_rng_table* table) { table_ = table; }
  double getLowestError() const { return last_.best_error; }
  int getBestIteration() const { return last_.best_iteration; }

 protected:
  void computeTransformation(PointCloudSource& output, const Matrix4& guess) override {
    (void)guess;  // [UPSTREAM]: the guess is ignored by SAC-IA
    const char* where = "pcl::SampleConsensusInitialAlignment::computeTransformation";
    if (!input_features_) { detail::pcl_error(where, "No source features were given! Call setSourceFeatures before aligning."); return; }
    if (!target_features_) { detail::pcl_error(where, "No target features were given! Call setTargetFeatures before aligning."); return; }
    if (this->input_->size() != input_features_->size()) { detail::pcl_error(where, "The source points and source feature points need to be in a one-to-one relationship!"); return; }
    if (this->target_->size() != target_features_->size()) { detail::pcl_error(where, "The target points and target feature points need to be in a one-to-one relationship!"); return; }
    static_assert(sizeof(FeatureT) == 33 * sizeof(float), "the device path takes FPFHSignature33 features");
    ope_ctx* ctx = detail::context();
    ope_sacia_params prm;
    ope_sacia_params_default(&prm);
    prm.max_iterations = this->max_iterations_;
    prm.nr_samples = nr_samples_;
    prm.k_correspondences = k_correspondences_;
    prm.min_sample_distance = min_sample_distance_;
    prm.max_correspondence_distance = this->corr_dist_threshold_;
    std::memset(&last_, 0, sizeof(last_));
    const int rc = ope_sacia_align(ctx, this->dsrc_.get(), reinterpret_cast<const float*>(input_features_->points.data()), this->dtgt_.get(),
                                   reinterpret_cast<const float*>(target_features_->points.data()), &prm, table_, &last_, nullptr);
    if (!detail::check(rc, where)) return;
    this->final_transformation_ = detail::from_c(last_.T);
    this->converged_ = last_.converged != 0;
    if (!table_) min_sample_distance_ = (float)last_.last_mse;   // selectSamples halves the MEMBER; it stays halved across align()s
    // transformPointCloud(*input_, output, final_transformation_)
    transformPointCloud(*this->input_, output, this->final_transformation_);
  }
  FeatureCloudConstPtr input_features_, target_features_;
  int nr_samples_ = 3;
  float min_sample_distance_ = 0.0f;
  int k_correspondences_ = 10;
  const ope_rng_table* table_ = nullptr;
  ope_reg_result last_{};
};

}  // namespace OPE_PCL_NAMESPACE
