// KeypointLearningSharded.h -- the detector of KeypointLearning.h over SEVERAL GPUs of one node: the multi-GPU form of
// the reference driver's `detector->compute(*keypoint)` (src/main_test_detector.cpp:123-187).  The cloud is cut into
// x slabs (kpl_slab_plan_make), one host thread per GPU drives one rank of the kpl_shard_* entry points of
// include/kpl.h (NCCL halo + score exchange inside libkpl_b200.so), and the result is the keypoint cloud the
// single-GPU detector returns, bit for bit.  Without setNormals(), normals are estimated on the devices (k-NN, the
// TestDetector setting :162-169, viewpoint = sensor origin), each slab for its halo as well; with setNormals() the
// caller's normals are partitioned like the points and travel with the halo strips (kpl_shard_set_slab_normals).
//
// Same setter names as the single-GPU class; every setter is forwarded to all ranks.
#pragma once
#include <cmath>
#include <cstdio>
#include <memory>
#include <string>
#include <thread>
#include <vector>
#include "KeypointLearning.h"

namespace pcl {
namespace keypoints {

template <typename PointInT, typename PointOutT>
class ShardedKeypointLearningDetector {
public:
    typedef KeypointLearningDetector<PointInT, PointOutT> Single;
    typedef typename Single::PointCloudInConstPtr PointCloudInConstPtr;
    typedef typename Single::PointCloudNConstPtr PointCloudNConstPtr;
    typedef pcl::Normal NormalT;                              // Single's (the default NormalT of KeypointLearningDetector)
    typedef pcl::PointCloud<PointOutT> PointCloudOut;

    // More ranks than devices (e.g. a test on one GPU): the ranks share the devices round-robin and form an in-process
    // group (NCCL refuses two ranks on one device).
    explicit ShardedKeypointLearningDetector(int gpus) : gpus_(gpus)
    {
        const int devices = std::max(kpl_device_count(), 1);
        share_devices_ = gpus > devices;
        for (int g = 0; g < gpus; ++g) ranks_.emplace_back(new Single(0.5f, true, true, 0.0f, 5, 10, g % devices));
    }
    int gpus() const { return gpus_; }
    // as KeypointLearningDetector (impl/KeypointLearning.hpp:49-57): another cloud drops the normals
    void setInputCloud(const PointCloudInConstPtr& cloud)
    {
        if (normals_ && input_ && cloud != input_) normals_.reset();
        input_ = cloud;
    }
    void setNormals(const PointCloudNConstPtr& normals) { normals_ = normals; }
    void setNonMaxima(bool v) { for (auto& r : ranks_) r->setNonMaxima(v); }
    void setNonMaximaDrawsRemove(bool v) { for (auto& r : ranks_) r->setNonMaximaDrawsRemove(v); }
    void setNonMaximaDrawsThreshold(float v) { for (auto& r : ranks_) r->setNonMaximaDrawsThreshold(v); }
    void setPredictionThreshold(double th) { for (auto& r : ranks_) r->setPredictionThreshold(th); }
    void setNonMaxRadius(double v) { for (auto& r : ranks_) r->setNonMaxRadius(v); }
    void setNAnnulus(int n) { for (auto& r : ranks_) r->setNAnnulus(n); }
    void setNBins(int n) { for (auto& r : ranks_) r->setNBins(n); }
    void setRadiusSearch(double v) { for (auto& r : ranks_) r->setRadiusSearch(v); }
    // the normal estimation TestDetector runs before the detector (ne.setKSearch(10), --flipNormals)
    void setNormalEstimation(int k, bool flip) { k_normals_ = k; flip_ = flip; }
    void setNormalSupportCells(int c) { support_ = c; }
    bool loadForest(const std::string& path)
    {
        bool ok = true;
        for (auto& r : ranks_) ok = r->loadForest(path) && ok;
        return ok;
    }
    // B200 build only: appends a forest to the set computeForests() scores, on every rank (loadForest's is forest 0)
    bool addForest(const std::string& path)
    {
        bool ok = true;
        for (auto& r : ranks_) ok = r->addForest(path) && ok;
        return ok;
    }
    pcl::PointIndicesConstPtr getKeypointsIndices() const { return keypoints_indices_; }
    const std::vector<float>& getResponse() const { return response_; }
    const kpl_slab_plan& plan() const { return plan_; }
    const std::vector<kpl_shard_info>& info() const { return info_; }
    Single& rank(int r) { return *ranks_[(size_t)r]; }

    // Returns false (output empty, message on stderr) on failure, like initCompute -> false upstream.
    bool compute(PointCloudOut& output)
    {
        output.points.clear(); output.width = output.height = 0;
        keypoints_indices_.reset(new pcl::PointIndices);
        std::vector<int32_t> kp;
        std::vector<int64_t> off;
        if (!detect("compute", false, nullptr, response_, kp, off)) return false;
        emit(output, kp.data() + off[0], kp.data() + off[1], response_.data(), &keypoints_indices_->indices);
        return true;
    }

    // B200 build only: every forest of the set (loadForest + addForest) over the input cloud from one feature pass per rank
    // (kpl_shard_detect_forests).  outputs[k] is what compute() returns with only forest k loaded, at threshold
    // (*thresholds)[k] (default: the prediction threshold); (*indices)[k], when asked for, its keypoint indices -- as
    // KeypointLearningDetector::computeForests.  The detector's response and keypoint indices are left as they are.
    bool computeForests(std::vector<PointCloudOut>& outputs, std::vector<pcl::PointIndices>* indices = nullptr,
                        const std::vector<double>* thresholds = nullptr)
    {
        outputs.clear();
        if (indices) indices->clear();
        int32_t K = 0;
        if (ranks_[0]->context()) kpl_forest_count(ranks_[0]->context(), &K);
        if (thresholds && thresholds->size() != (size_t)K) {
            std::fprintf(stderr, "[ShardedKeypointLearningDetector::computeForests] %zu thresholds for %d forests\n", thresholds->size(), K);
            return false;
        }
        std::vector<float> scores;
        std::vector<int32_t> kp;
        std::vector<int64_t> off;
        if (!detect("computeForests", true, thresholds, scores, kp, off)) return false;
        const size_t n = input_->size();
        outputs.assign(off.size() - 1, PointCloudOut());
        if (indices) indices->assign(off.size() - 1, pcl::PointIndices());
        for (size_t k = 0; k + 1 < off.size(); ++k)
            emit(outputs[k], kp.data() + off[k], kp.data() + off[k + 1], scores.data() + k * n, indices ? &(*indices)[k].indices : nullptr);
        return true;
    }

private:
    // the keypoint cloud of [kp, kp_end): positions and the responses of `response` (hpp:246-253)
    void emit(PointCloudOut& output, const int32_t* kp, const int32_t* kp_end, const float* response, std::vector<int>* idx) const
    {
        output.points.clear();
        output.points.reserve((size_t)(kp_end - kp));
        for (; kp != kp_end; ++kp) {
            const PointInT& in = input_->points[(size_t)*kp];
            PointOutT o;
            o.x = in.x; o.y = in.y; o.z = in.z;
            o.intensity = response[(size_t)*kp];
            output.points.push_back(o);
            if (idx) idx->push_back(*kp);
        }
        output.height = 1;
        output.width = (uint32_t)output.points.size();
        output.is_dense = true;
    }

    // The checks of compute(), then one detection through the re-plan loop: forest 0, or every forest of the set
    // (forests).  scores: K x n responses in input order; forest k's keypoints are kp[off[k] .. off[k + 1]).
    bool detect(const char* who, bool forests, const std::vector<double>* thresholds, std::vector<float>& scores, std::vector<int32_t>& kp,
                std::vector<int64_t>& off)
    {
        if (!input_ || input_->empty()) { std::fprintf(stderr, "[ShardedKeypointLearningDetector::%s] no input cloud\n", who); return false; }
        const int64_t n = (int64_t)input_->size();
        if (normals_ && (int64_t)normals_->size() != n) {       // pcl::KeypointLearningDetector::initCompute (hpp:149-153)
            std::fprintf(stderr, "[ShardedKeypointLearningDetector::%s] normals given, but the number of normals does not match the number of input points!\n", who);
            return false;
        }
        const float* xyz = reinterpret_cast<const float*>(input_->points.data());
        std::vector<kpl_params> P((size_t)gpus_);
        for (int g = 0; g < gpus_; ++g) {
            kpl_params q = ranks_[(size_t)g]->params();
            q.normals_mode = KPL_NORMALS_KNN; q.k_normals = k_normals_; q.flip_normals = flip_;
            for (int a = 0; a < 3; ++a) q.viewpoint[a] = input_->sensor_origin_[a];
            if (!ranks_[(size_t)g]->context() || kpl_set_params(ranks_[(size_t)g]->context(), &q) != KPL_OK) {
                std::fprintf(stderr, "[ShardedKeypointLearningDetector::%s] rank %d: %s\n", who, g,
                             ranks_[(size_t)g]->context() ? kpl_last_error(ranks_[(size_t)g]->context()) : "no usable sm_100 device");
                return false;
            }
            P[(size_t)g] = q;
        }
        int32_t K = 1;
        if (forests) kpl_forest_count(ranks_[0]->context(), &K);
        scores.assign((size_t)std::max(K, 1) * (size_t)n, std::nanf(""));
        kp.resize((size_t)std::max(K, 1) * (size_t)n);
        off.assign((size_t)K + 1, 0);
        // a k-NN normal that matters may be clipped by a slab face (KPL_E_HALO, reported by every rank): widen the support
        // (1 after 0).  Given normals need no k-NN support: one plan with support 0, which cannot fail that way.
        for (int support = normals_ ? 0 : support_; ; support = std::max(support * 2, 1)) {
            int rc = kpl_slab_plan_make(xyz, (int32_t)sizeof(PointInT), n, &P[0], gpus_, support, &plan_);
            if (rc != KPL_OK) {
                std::fprintf(stderr, "[ShardedKeypointLearningDetector::%s] the cloud cannot be cut into %d slabs with a halo of %d + %d cell columns "
                                     "(kpl_slab_plan_make -> %d): use fewer GPUs\n", who, gpus_, plan_.reach_feat, support, rc);
                return false;
            }
            rc = run(xyz, n, forests, K, thresholds ? thresholds->data() : nullptr, scores.data(), kp.data(), off.data());
            if (rc == KPL_OK) return true;
            if (rc != KPL_E_HALO || normals_ || support > 64) {
                std::fprintf(stderr, "[ShardedKeypointLearningDetector::%s] %s\n", who, error_.c_str());
                return false;
            }
        }
    }

    // one detection with the current plan: one host thread per rank (ncclCommInitRank blocks until all ranks joined).
    // K score slices: kpl_shard_detect_forests (forests) or kpl_shard_detect (K = 1).
    int run(const float* xyz, int64_t n, bool forests, int K, const double* thresholds, float* scores_out, int32_t* kp_out, int64_t* off_out)
    {
        unsigned char id[128];
        const bool nccl = !share_devices_ && kpl_nccl_unique_id(id) == KPL_OK;   // no NCCL on this host: ranks of an in-process group instead
        std::vector<kpl_shard*> shards((size_t)gpus_, nullptr);
        std::vector<int> rcs((size_t)gpus_, KPL_OK);
        std::vector<std::string> errs((size_t)gpus_);
        std::vector<std::vector<int32_t>> gidx((size_t)gpus_);
        std::vector<std::vector<float>> scores((size_t)gpus_);
        std::vector<int64_t> nk((size_t)gpus_, 0);
        const int64_t cap = (int64_t)std::max(K, 1) * n;
        info_.assign((size_t)gpus_, kpl_shard_info());
        auto setup = [&](int g) {
            kpl_ctx* ctx = ranks_[(size_t)g]->context();
            auto& rc = rcs[(size_t)g];
            gidx[(size_t)g].resize((size_t)n);
            int64_t m = 0;
            rc = kpl_slab_partition(&plan_, xyz, (int32_t)sizeof(PointInT), n, g, gidx[(size_t)g].data(), &m);
            if (rc) { errs[(size_t)g] = "kpl_slab_partition failed"; return; }
            gidx[(size_t)g].resize((size_t)m);
            std::vector<PointInT> own((size_t)m);
            std::vector<NormalT> own_n(normals_ ? (size_t)m : 0);
            for (int64_t k = 0; k < m; ++k) {
                own[(size_t)k] = input_->points[(size_t)gidx[(size_t)g][(size_t)k]];
                if (normals_) own_n[(size_t)k] = normals_->points[(size_t)gidx[(size_t)g][(size_t)k]];
            }
            scores[(size_t)g].assign((size_t)std::max(K, 1) * (size_t)m, 0.f);
            rc = kpl_shard_create(ctx, &plan_, g, nccl ? id : nullptr, &shards[(size_t)g]);
            const float* p = reinterpret_cast<const float*>(own.data());
            if (!rc && normals_)
                rc = kpl_shard_set_slab_normals(shards[(size_t)g], p, (int32_t)sizeof(PointInT), reinterpret_cast<const float*>(own_n.data()),
                                                (int32_t)sizeof(NormalT), gidx[(size_t)g].data(), m);
            else if (!rc)
                rc = kpl_shard_set_slab(shards[(size_t)g], p, (int32_t)sizeof(PointInT), gidx[(size_t)g].data(), m);
            if (rc) errs[(size_t)g] = kpl_last_error(ctx);
        };
        auto detect = [&](int g) {
            if (rcs[(size_t)g]) return;
            int32_t* kp = g == 0 ? kp_out : nullptr;
            rcs[(size_t)g] = forests ? kpl_shard_detect_forests(shards[(size_t)g], thresholds, scores[(size_t)g].data(), kp, cap, g == 0 ? off_out : nullptr, &nk[(size_t)g])
                                     : kpl_shard_detect(shards[(size_t)g], scores[(size_t)g].data(), kp, cap, &nk[(size_t)g]);
            if (rcs[(size_t)g]) errs[(size_t)g] = kpl_last_error(ranks_[(size_t)g]->context());
            else kpl_shard_get_info(shards[(size_t)g], &info_[(size_t)g]);
        };
        auto all = [&](auto&& fn) {
            std::vector<std::thread> th;
            for (int g = 0; g < gpus_; ++g) th.emplace_back(fn, g);
            for (auto& t : th) t.join();
        };
        int rc = KPL_OK;
        all(setup);
        bool ready = true;
        for (int g = 0; g < gpus_; ++g) ready = ready && rcs[(size_t)g] == KPL_OK;
        if (ready) {
            if (nccl) all(detect);
            else {
                std::vector<float*> sp((size_t)gpus_);
                for (int g = 0; g < gpus_; ++g) sp[(size_t)g] = scores[(size_t)g].data();
                rcs[0] = forests ? kpl_shard_detect_forests_group(shards.data(), gpus_, thresholds, sp.data(), kp_out, cap, off_out, &nk[0])
                                 : kpl_shard_detect_group(shards.data(), gpus_, sp.data(), kp_out, cap, &nk[0]);
                if (rcs[0]) errs[0] = kpl_last_error(ranks_[0]->context());
                else for (int g = 0; g < gpus_; ++g) kpl_shard_get_info(shards[(size_t)g], &info_[(size_t)g]);
            }
        }
        for (int g = 0; g < gpus_; ++g)
            if (rcs[(size_t)g] && !rc) { rc = rcs[(size_t)g]; error_ = "rank " + std::to_string(g) + ": " + errs[(size_t)g]; }
        for (int g = 0; g < gpus_; ++g) kpl_shard_destroy(shards[(size_t)g]);
        if (rc) return rc;
        for (int g = 0; g < gpus_; ++g) {
            const size_t m = gidx[(size_t)g].size();
            for (int k = 0; k < K; ++k)
                for (size_t j = 0; j < m; ++j) scores_out[(size_t)k * (size_t)n + (size_t)gidx[(size_t)g][j]] = scores[(size_t)g][(size_t)k * m + j];
        }
        if (!forests) { off_out[0] = 0; off_out[1] = nk[0]; }
        return KPL_OK;
    }

    int gpus_;
    int k_normals_ = 10, support_ = 1;
    bool flip_ = false, share_devices_ = false;
    std::vector<std::unique_ptr<Single>> ranks_;
    PointCloudInConstPtr input_;
    PointCloudNConstPtr normals_;
    pcl::PointIndicesPtr keypoints_indices_{new pcl::PointIndices};
    std::vector<float> response_;
    kpl_slab_plan plan_;
    std::vector<kpl_shard_info> info_;
    std::string error_;
};

}  // namespace keypoints
}  // namespace pcl
