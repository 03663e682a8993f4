// KeypointLearning.h -- pcl::keypoints::KeypointLearningDetector over the C ABI of include/kpl.h.
//
// Same class name, template parameters, constructor defaults and method names as the reference's
// include/KeypointLearning.h:55-206 (+ the pcl::Keypoint members its driver calls: setRadiusSearch,
// compute, getKeypointsIndices), so src/main_test_detector.cpp:123-187 compiles against this header
// unchanged apart from the include lines.  Every call forwards to libkpl_b200.so; nothing is computed
// on the host.  Error behaviour follows the reference: loadForest -> false, initCompute failure ->
// message on stderr and an empty output cloud (impl/KeypointLearning.hpp:119-123,149-153,165-174).
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <memory>
#include <string>
#include <vector>
#include "kpl.h"
#include "pcl_shim.h"

namespace pcl {
namespace keypoints {

template <typename PointInT, typename PointOutT, typename NormalT = pcl::Normal>
class KeypointLearningDetector {
public:
    typedef std::shared_ptr<KeypointLearningDetector<PointInT, PointOutT, NormalT>> Ptr;
    typedef std::shared_ptr<const KeypointLearningDetector<PointInT, PointOutT, NormalT>> ConstPtr;
    typedef pcl::PointCloud<PointInT> PointCloudIn;
    typedef pcl::PointCloud<PointOutT> PointCloudOut;
    typedef typename PointCloudIn::ConstPtr PointCloudInConstPtr;
    typedef pcl::PointCloud<NormalT> PointCloudN;
    typedef typename PointCloudN::Ptr PointCloudNPtr;
    typedef typename PointCloudN::ConstPtr PointCloudNConstPtr;

    // include/KeypointLearning.h:81-90
    KeypointLearningDetector(double prediction_th = 0.5f, bool non_maxima = true, bool non_maxima_draws_remove = true,
                             double non_max_radius = 0.0f, int n_annulus = 5, int n_bins = 10, int device = 0)
        : name_("Keypoint_Learnining_Detector"), keypoints_indices_(new pcl::PointIndices)
    {
        kpl_params_default(&p_);
        p_.threshold = prediction_th;
        p_.non_maxima = non_maxima;
        p_.draws_remove = non_maxima_draws_remove;
        p_.radius_nms = (float)non_max_radius;
        p_.n_annulus = n_annulus;
        p_.n_bins = n_bins;
        p_.radius_features = 0.f;            // pcl::Keypoint::search_radius_ starts at 0: setRadiusSearch is mandatory
        create_rc_ = kpl_create(device, &ctx_);
        if (create_rc_ != KPL_OK) std::fprintf(stderr, "[pcl::%s] no usable sm_100 device (kpl_create -> %d); there is no CPU path\n", name_.c_str(), create_rc_);
    }
    virtual ~KeypointLearningDetector() { kpl_destroy(ctx_); }
    KeypointLearningDetector(const KeypointLearningDetector&) = delete;
    KeypointLearningDetector& operator=(const KeypointLearningDetector&) = delete;

    // impl/KeypointLearning.hpp:49-57
    virtual void setInputCloud(const PointCloudInConstPtr& cloud)
    {
        if (normals_ && input_ && cloud != input_) normals_.reset();
        input_ = cloud;
    }
    virtual void setNormals(const PointCloudNConstPtr& normals) { normals_ = normals; }
    virtual void setNonMaxima(bool v) { p_.non_maxima = v; }
    virtual void setNonMaximaDrawsRemove(bool v) { p_.draws_remove = v; }
    virtual void setNonMaximaDrawsThreshold(float v) { p_.draws_threshold = v; }
    virtual void setPredictionThreshold(double th) { p_.threshold = th; }
    virtual void setNonMaxRadius(double r) { p_.radius_nms = (float)r; }
    virtual void setNAnnulus(int n) { p_.n_annulus = n; }
    virtual void setNBins(int n) { p_.n_bins = n; }
    // ---- inherited from pcl::Keypoint in the reference (include/KeypointLearning.h:55-56)
    void setRadiusSearch(double r) { p_.radius_features = (float)r; }
    // pcl::Keypoint::initCompute refuses a radius AND a k; a k alone would make computePointFeatures divide by a zero
    // support (hpp:345 passes search_radius_): both cases fail in initCompute() below, as they do upstream
    void setKSearch(int k) { k_ = k; }
    // Neighbour searches of this build always run on the uniform grid inside libkpl_b200 with the radiusSearch
    // semantics of the kd-tree the reference installs (hpp:116-124): any search object is accepted and has no effect.
    void setSearchMethod(const typename pcl::search::KdTree<PointInT>::Ptr&) {}
    // The reference indexes normals_, response and the kd-tree with ONE index space (hpp:203-253,334-342), which only
    // holds when the search surface is the input cloud: another surface is refused in initCompute().
    void setSearchSurface(const PointCloudInConstPtr& cloud) { surface_ = cloud; }
    // ---- B200 build only
    void setCellsPerRadius(int cpr) { p_.cells_per_radius = cpr; }
    void setReportFragile(bool on) { p_.report_fragile = on; }                 // kpl_stats.n_fragile_points
    void setEigen32Normalize(bool on) { p_.eigen32_normalize = on; }           // row.normalize() as Eigen 3.2.x (x * 1/norm)
    const kpl_params& params() const { return p_; }

    // impl/KeypointLearning.hpp:159-176
    virtual bool loadForest(const std::string& path)
    {
        if (!ctx_) return false;
        if (kpl_load_forest(ctx_, path.c_str()) != KPL_OK) {
            std::fprintf(stderr, "[pcl::%s::loadForest] impossible to load random forest with path %s (%s)\n", name_.c_str(), path.c_str(), kpl_last_error(ctx_));
            return false;
        }
        int32_t ntrees = 0;
        kpl_forest_info(ctx_, &ntrees, nullptr, nullptr, nullptr);
        return ntrees != 0;
    }
    // B200 build only: appends a forest to the set computeForests() scores (loadForest's forest is forest 0 and drops the others)
    bool addForest(const std::string& path)
    {
        if (!ctx_) return false;
        if (kpl_add_forest(ctx_, path.c_str(), nullptr) != KPL_OK) {
            std::fprintf(stderr, "[pcl::%s::addForest] impossible to load random forest with path %s (%s)\n", name_.c_str(), path.c_str(), kpl_last_error(ctx_));
            return false;
        }
        return true;
    }

    // pcl::Keypoint::compute -> initCompute / detectKeypoints (impl/KeypointLearning.hpp:116-156,179-263)
    void compute(PointCloudOut& output)
    {
        output.points.clear(); output.width = output.height = 0;
        keypoints_indices_.reset(new pcl::PointIndices);
        if (!initCompute()) return;
        const int64_t n = (int64_t)input_->size();
        // result buffers are written by the library: sized, not cleared (clearing 10 M-point buffers costs milliseconds)
        if (response_.size() != (size_t)n) response_.resize((size_t)n);
        std::unique_ptr<int32_t[]> idx(new int32_t[(size_t)std::max<int64_t>(n, 1)]);
        int64_t nkp = 0;
        std::unique_ptr<float[]> xyzi(new float[(size_t)std::max<int64_t>(n, 1) * 4]);   // keypoint cloud, gathered on the device
        std::vector<int32_t> finite;
        std::vector<float> sc;
        bool compacted = false;
        int rc = detectFinite([&](const PointInT* pts, const float* nrm, int64_t m) {
            float* scores = response_.data();
            if (compacted) { sc.resize((size_t)std::max<int64_t>(m, 1)); scores = sc.data(); }
            return kpl_detect_xyzi(ctx_, reinterpret_cast<const float*>(pts), (int32_t)sizeof(PointInT), nrm, (int32_t)sizeof(NormalT), nullptr, m,
                                   scores, idx.get(), xyzi.get(), &nkp);
        }, finite, compacted);
        if (rc == KPL_OK && compacted) {
            response_.assign((size_t)n, std::nanf(""));
            for (size_t k = 0; k < finite.size(); ++k) response_[(size_t)finite[k]] = sc[k];
            for (int64_t k = 0; k < nkp; ++k) idx[(size_t)k] = finite[(size_t)idx[(size_t)k]];
        }
        if (rc != KPL_OK) {
            std::fprintf(stderr, "[pcl::%s::compute] %s\n", name_.c_str(), kpl_last_error(ctx_));
            return;
        }
        output.points.reserve((size_t)nkp);
        for (int64_t k = 0; k < nkp; ++k) {                                       // hpp:246-253
            PointOutT o;
            o.x = xyzi[(size_t)k * 4]; o.y = xyzi[(size_t)k * 4 + 1]; o.z = xyzi[(size_t)k * 4 + 2];
            o.intensity = xyzi[(size_t)k * 4 + 3];
            output.points.push_back(o);
            keypoints_indices_->indices.push_back(idx[(size_t)k]);
        }
        output.height = 1;
        output.width = (uint32_t)output.points.size();
        output.is_dense = p_.non_maxima ? true : input_->is_dense;               // hpp:192-193,258-260
    }
    pcl::PointIndicesConstPtr getKeypointsIndices() const { return keypoints_indices_; }

    // B200 build only: every forest of the set (loadForest + addForest) over the input cloud from one feature pass
    // (kpl_detect_forests).  outputs[k] is what compute() returns with only forest k loaded, at threshold (*thresholds)[k]
    // (default: the prediction threshold); (*indices)[k], when asked for, its keypoint indices.  Non-dense clouds and the
    // initCompute checks are handled as in compute().  The detector's response and keypoint indices are left as they are.
    bool computeForests(std::vector<PointCloudOut>& outputs, std::vector<pcl::PointIndices>* indices = nullptr,
                        const std::vector<double>* thresholds = nullptr)
    {
        outputs.clear();
        if (indices) indices->clear();
        if (!initCompute()) return false;
        int32_t K = 0;
        kpl_forest_count(ctx_, &K);
        if (thresholds && thresholds->size() != (size_t)K) {
            std::fprintf(stderr, "[pcl::%s::computeForests] %zu thresholds for %d forests\n", name_.c_str(), thresholds->size(), K);
            return false;
        }
        std::vector<float> scores;
        std::vector<int32_t> idx, finite;
        std::vector<int64_t> off((size_t)K + 1);
        bool compacted = false;
        int rc = detectFinite([&](const PointInT* pts, const float* nrm, int64_t m) {
            scores.resize((size_t)K * (size_t)std::max<int64_t>(m, 1));
            idx.resize((size_t)K * (size_t)std::max<int64_t>(m, 1));
            return kpl_detect_forests(ctx_, reinterpret_cast<const float*>(pts), (int32_t)sizeof(PointInT), nrm, (int32_t)sizeof(NormalT), m,
                                      thresholds ? thresholds->data() : nullptr, scores.data(), idx.data(), off.data());
        }, finite, compacted);
        if (rc != KPL_OK) {
            std::fprintf(stderr, "[pcl::%s::compute] %s\n", name_.c_str(), kpl_last_error(ctx_));
            return false;
        }
        const size_t m = compacted ? finite.size() : input_->size();
        outputs.assign((size_t)K, PointCloudOut());
        if (indices) indices->assign((size_t)K, pcl::PointIndices());
        for (size_t k = 0; k < (size_t)K; ++k) {
            PointCloudOut& out = outputs[k];
            out.points.reserve((size_t)(off[k + 1] - off[k]));
            for (int64_t j = off[k]; j < off[k + 1]; ++j) {                     // hpp:246-253
                const int32_t local = idx[(size_t)j];
                const int32_t i = compacted ? finite[(size_t)local] : local;
                const PointInT& p = input_->points[(size_t)i];
                PointOutT o;
                o.x = p.x; o.y = p.y; o.z = p.z;
                o.intensity = scores[k * m + (size_t)local];
                out.points.push_back(o);
                if (indices) (*indices)[k].indices.push_back(i);
            }
            out.height = 1;
            out.width = (uint32_t)out.points.size();
            out.is_dense = p_.non_maxima ? true : input_->is_dense;             // hpp:192-193,258-260
        }
        return true;
    }
    const std::vector<float>& getResponse() const { return response_; }          // the `response` cloud's intensities (hpp:181-187)

    // impl/KeypointLearning.hpp:299-318 (cv::Mat -> KplFeatureMatrix)
    KplFeatureMatrix computePointsForTrainingFeatures(pcl::PointIndicesConstPtr indices)
    {
        KplFeatureMatrix m;
        if (!indices || !initCompute()) return m;
        const int F = p_.n_annulus * p_.n_bins;
        m.data.assign(indices->indices.size() * (size_t)F, 0.f);
        const float* nrm = normals_ ? reinterpret_cast<const float*>(normals_->points.data()) : nullptr;
        int rc = kpl_features(ctx_, reinterpret_cast<const float*>(input_->points.data()), (int32_t)sizeof(PointInT), nrm, (int32_t)sizeof(NormalT),
                              (int64_t)input_->size(), indices->indices.data(), (int64_t)indices->indices.size(), m.data.data());
        if (rc != KPL_OK) {
            std::fprintf(stderr, "[pcl::%s::computePointsForTrainingFeatures] %s\n", name_.c_str(), kpl_last_error(ctx_));
            m.data.clear();
            return m;
        }
        m.rows = (int)indices->indices.size(); m.cols = F;
        return m;
    }

    // A stream of organized frames of one width x height (a depth camera) in one pass (kpl_detect_batch_organized): for
    // every frame what compute() returns for it alone with no normals set -- integral-image normals (hpp:138-145) flipped
    // towards the frame's sensor_origin_, the detection over its finite points.  outputs[f] is frame f's keypoint cloud
    // (x, y, z, intensity = response); (*indices)[f], when asked for, its keypoint indices.  The input cloud, normals,
    // response and keypoint indices of the detector are left as they are.
    bool computeOrganizedBatch(const std::vector<PointCloudInConstPtr>& frames, std::vector<PointCloudOut>& outputs,
                               std::vector<pcl::PointIndices>* indices = nullptr)
    {
        return detectOrganizedFrames(frames, 1, outputs, indices, [&](const float* pts, const float* vps, int32_t W, int32_t H, int32_t F,
                                                                      float* scores, int32_t* idx, int64_t* off) {
            return kpl_detect_batch_organized(ctx_, pts, (int32_t)sizeof(PointInT), nullptr, 0, W, H, F, 5.0f, vps, scores, idx, off);
        });
    }

    // B200 build only: computeOrganizedBatch for every forest of the set (loadForest + addForest) from one feature pass
    // (kpl_detect_batch_organized_forests).  outputs[k][f] is what computeOrganizedBatch returns for frame f with only forest
    // k loaded, at threshold (*thresholds)[k] (default: the prediction threshold); (*indices)[k][f], when asked for, its
    // keypoint indices.  A thresholds vector that does not hold one value per forest is refused.
    bool computeOrganizedBatchForests(const std::vector<PointCloudInConstPtr>& frames, std::vector<std::vector<PointCloudOut>>& outputs,
                                      std::vector<std::vector<pcl::PointIndices>>* indices = nullptr,
                                      const std::vector<double>* thresholds = nullptr)
    {
        outputs.clear();
        if (indices) indices->clear();
        int32_t K = 0;
        if (ctx_) kpl_forest_count(ctx_, &K);
        if (thresholds && thresholds->size() != (size_t)K) {
            std::fprintf(stderr, "[pcl::%s::computeOrganizedBatchForests] %zu thresholds for %d forests\n", name_.c_str(), thresholds->size(), K);
            return false;
        }
        std::vector<PointCloudOut> flat;
        std::vector<pcl::PointIndices> flat_idx;
        const bool ok = detectOrganizedFrames(frames, std::max(K, 1), flat, indices ? &flat_idx : nullptr,
                                              [&](const float* pts, const float* vps, int32_t W, int32_t H, int32_t F, float* scores, int32_t* idx,
                                                  int64_t* off) {
            return kpl_detect_batch_organized_forests(ctx_, pts, (int32_t)sizeof(PointInT), nullptr, 0, W, H, F, 5.0f, vps,
                                                      thresholds ? thresholds->data() : nullptr, scores, idx, off);
        });
        if (!ok) return false;
        const size_t F = frames.size();
        for (size_t k = 0; k < (size_t)K; ++k) {
            outputs.emplace_back(flat.begin() + k * F, flat.begin() + (k + 1) * F);
            if (indices) indices->emplace_back(flat_idx.begin() + k * F, flat_idx.begin() + (k + 1) * F);
        }
        return true;
    }

    kpl_ctx* context() { return ctx_; }

protected:
    // The frame checks and packing of computeOrganizedBatch(Forests): detect(points, viewpoints, W, H, F, scores, indices,
    // offsets) runs K forests over the packed frames; outputs[k * F + f] (and (*indices)[k * F + f]) receive forest k's
    // keypoints of frame f.
    template <typename Detect>
    bool detectOrganizedFrames(const std::vector<PointCloudInConstPtr>& frames, int K, std::vector<PointCloudOut>& outputs,
                               std::vector<pcl::PointIndices>* indices, Detect detect)
    {
        outputs.assign((size_t)K * frames.size(), PointCloudOut());
        if (indices) indices->assign((size_t)K * frames.size(), pcl::PointIndices());
        if (!ctx_ || frames.empty() || !frames[0]) {
            std::fprintf(stderr, "[pcl::%s::initCompute] init failed!\n", name_.c_str());
            return false;
        }
        const uint32_t W = frames[0]->width, H = frames[0]->height;
        for (const PointCloudInConstPtr& f : frames)
            if (!f || !f->isOrganized() || f->width != W || f->height != H || f->size() != (size_t)W * H) {
                std::fprintf(stderr, "[pcl::%s::initCompute] the frames of a batch must be organized clouds of one width x height\n", name_.c_str());
                return false;
            }
        if (!checkSearch()) return false;
        const size_t n = (size_t)W * H, F = frames.size();
        std::vector<PointInT> pts(n * F);
        std::vector<float> vps(3 * F), scores((size_t)K * n * F);
        for (size_t f = 0; f < F; ++f) {
            std::copy(frames[f]->points.begin(), frames[f]->points.end(), pts.begin() + f * n);
            for (int a = 0; a < 3; ++a) vps[3 * f + a] = frames[f]->sensor_origin_[a];
        }
        std::vector<int32_t> idx((size_t)K * n * F);
        std::vector<int64_t> off((size_t)K * F + 1);
        if (kpl_set_params(ctx_, &p_) != KPL_OK ||
            detect(reinterpret_cast<const float*>(pts.data()), vps.data(), (int32_t)W, (int32_t)H, (int32_t)F, scores.data(), idx.data(),
                   off.data()) != KPL_OK) {
            std::fprintf(stderr, "[pcl::%s::compute] %s\n", name_.c_str(), kpl_last_error(ctx_));
            return false;
        }
        for (size_t r = 0; r < (size_t)K * F; ++r) {
            const size_t f = r % F;
            PointCloudOut& out = outputs[r];
            for (int64_t k = off[r]; k < off[r + 1]; ++k) {                      // hpp:246-253
                const int32_t i = idx[(size_t)k];
                const PointInT& p = frames[f]->points[(size_t)i];
                PointOutT o;
                o.x = p.x; o.y = p.y; o.z = p.z;
                o.intensity = scores[r * n + (size_t)i];
                out.points.push_back(o);
                if (indices) (*indices)[r].indices.push_back(i);
            }
            out.height = 1;
            out.width = (uint32_t)out.points.size();
            out.is_dense = p_.non_maxima ? true : frames[f]->is_dense;             // hpp:192-193,258-260
        }
        return true;
    }

    // detect(points, normals or nullptr, count) on the input cloud.  Non-dense clouds (Kinect / organized PCDs carry NaN
    // points; found by the device's bounding-box pass, KPL_E_NONFINITE): the reference's kd-tree ignores them and runForest
    // skips them (hpp:277), so detect runs again on the compacted finite points, whose input indices `finite` then lists
    // and `compacted` is set.  The caller maps the results back: a skipped point has a NaN response and is never a keypoint.
    template <typename Detect>
    int detectFinite(Detect detect, std::vector<int32_t>& finite, bool& compacted)
    {
        finite.clear();
        compacted = false;
        const int64_t n = (int64_t)input_->size();
        int rc = detect(input_->points.data(), normals_ ? reinterpret_cast<const float*>(normals_->points.data()) : nullptr, n);
        if (rc != KPL_E_NONFINITE) return rc;
        for (int64_t i = 0; i < n; ++i)
            if (pcl::isFinite(input_->points[(size_t)i])) finite.push_back((int32_t)i);
        const int64_t m = (int64_t)finite.size();
        std::vector<PointInT> pts((size_t)m);
        std::vector<NormalT> nrs(normals_ ? (size_t)m : 0);
        for (int64_t k = 0; k < m; ++k) {
            pts[(size_t)k] = input_->points[(size_t)finite[(size_t)k]];
            if (normals_) nrs[(size_t)k] = normals_->points[(size_t)finite[(size_t)k]];
        }
        compacted = true;
        return detect(pts.data(), normals_ ? reinterpret_cast<const float*>(nrs.data()) : nullptr, m);
    }

    // pcl::Keypoint::initCompute's search checks
    bool checkSearch() const
    {
        if (p_.radius_features > 0.f && k_ != 0) {   // pcl::Keypoint::initCompute
            std::fprintf(stderr, "[pcl::%s::initCompute] Both radius (%f) and K (%d) defined! Set one of them to zero first and then re-run compute ().\n",
                         name_.c_str(), p_.radius_features, k_);
            return false;
        }
        if (!(p_.radius_features > 0.f)) {
            if (k_ != 0)
                std::fprintf(stderr, "[pcl::%s::initCompute] a k search gives computePointFeatures a zero support (hpp:345): set a radius with setRadiusSearch\n", name_.c_str());
            else
                std::fprintf(stderr, "[pcl::%s::initCompute] Neither radius nor K defined! Set one of them to zero first and then re-run compute ().\n", name_.c_str());
            return false;
        }
        return true;
    }

    bool initCompute()
    {
        if (!ctx_ || !input_) {
            std::fprintf(stderr, "[pcl::%s::initCompute] init failed!\n", name_.c_str());
            return false;
        }
        if (surface_ && surface_ != input_) {
            std::fprintf(stderr, "[pcl::%s::initCompute] a search surface other than the input cloud is not supported: normals, response and "
                                 "neighbour indices share one index space (hpp:203-253,334-342)\n", name_.c_str());
            return false;
        }
        if (!checkSearch()) return false;
        if (normals_ && normals_->size() != input_->size()) {
            std::fprintf(stderr, "[pcl::%s::initCompute] normals given, but the number of normals does not match the number of input points!\n", name_.c_str());
            return false;
        }
        kpl_params q = p_;
        if (!normals_) {
            // hpp:125-148: unorganized -> NormalEstimation.setRadiusSearch(search_radius_); organized -> integral images (unsupported)
            std::printf("Computing normals for KPL\n");
            if (input_->isOrganized()) {
                // hpp:138-145: IntegralImageNormalEstimation, SIMPLE_3D_GRADIENT, setNormalSmoothingSize(5.0); like the
                // reference the result becomes this->normals_ and stays for later calls on the same cloud
                q.viewpoint[0] = input_->sensor_origin_[0]; q.viewpoint[1] = input_->sensor_origin_[1]; q.viewpoint[2] = input_->sensor_origin_[2];
                const size_t n = input_->size();
                std::vector<float> buf(n * 4);
                if (kpl_set_params(ctx_, &q) != KPL_OK ||
                    kpl_normals_organized(ctx_, reinterpret_cast<const float*>(input_->points.data()), (int32_t)sizeof(PointInT), (int32_t)input_->width,
                                          (int32_t)input_->height, 5.0f, buf.data()) != KPL_OK) {
                    std::fprintf(stderr, "[pcl::%s::initCompute] %s\n", name_.c_str(), kpl_last_error(ctx_));
                    return false;
                }
                PointCloudNPtr normals(new PointCloudN());
                normals->points.resize(n);
                for (size_t i = 0; i < n; ++i) {
                    NormalT& o = normals->points[i];
                    o.normal_x = buf[4 * i]; o.normal_y = buf[4 * i + 1]; o.normal_z = buf[4 * i + 2]; o.curvature = buf[4 * i + 3];
                }
                normals->width = input_->width; normals->height = input_->height; normals->is_dense = false;
                normals_ = normals;
                return true;
            }
            q.normals_mode = KPL_NORMALS_RADIUS;
            q.viewpoint[0] = input_->sensor_origin_[0]; q.viewpoint[1] = input_->sensor_origin_[1]; q.viewpoint[2] = input_->sensor_origin_[2];
        }
        if (kpl_set_params(ctx_, &q) != KPL_OK) {
            std::fprintf(stderr, "[pcl::%s::initCompute] %s\n", name_.c_str(), kpl_last_error(ctx_));
            return false;
        }
        return true;
    }

    std::string name_;
    kpl_ctx* ctx_ = nullptr;
    int create_rc_ = KPL_OK;
    kpl_params p_;
    int k_ = 0;
    PointCloudInConstPtr input_, surface_;
    PointCloudNConstPtr normals_;
    pcl::PointIndicesPtr keypoints_indices_;
    std::vector<float> response_;
};

}  // namespace keypoints
}  // namespace pcl
