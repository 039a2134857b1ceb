// stereo/multiviewstereo.hpp — MultiViewStereo with the reference's public interface
// (stereo/multiviewstereo.hpp:44-63) on top of the B200 C ABI (include/sr_b200.h).
//
// initialize() loads the default image of every view from the image set, scales it, and turns a
// PNG alpha channel into the mask (alpha != 255 -> BLACK), as multiviewstereo.cpp:193-247 does.
// runTask() is the reference's task (:325-475) with every per-pixel stage on the GPU:
//   neighbour selection (:335-360)        sr_select_neighbours
//   computeInitialEstimate (:524-662)     sr_run_view, MultiViewStereo selection over depth labels
//   crossCheck (:666-729)                 sr_cross_check
//   colourisation (:257-278, :381-395)    sr_get_depth_image
//   point cloud (:291-315, :740-750)      sr_get_points (with setKeepPointCloud(true))
// No CPU fallback: a missing CUDA device makes run() throw from sr_ctx_create.
#ifndef SR_STEREO_MULTIVIEWSTEREO_HPP
#define SR_STEREO_MULTIVIEWSTEREO_HPP
#include <fstream>

#include "gui/task.hpp"
#include "project/camera.hpp"
#include "project/imageset.hpp"
#include "project/project.hpp"
#include "project/projectimage.hpp"
#include "stereo/sr_session.hpp"
#include "util/ray.hpp"
#include "util/vectorimage.hpp"

typedef std::pair<Ray3d::Point, RGBA> PLYPoint;

//! Output a set of points to an ASCII PLY file (multiviewstereo.cpp:291-315)
inline void outputPLYFile(const std::string &path, const std::vector<PLYPoint> &points) {
    std::ofstream out(path.c_str());
    out << "ply\nformat ascii 1.0\nelement vertex " << points.size()
        << "\nproperty float x\nproperty float y\nproperty float z\n"
        << "property uchar diffuse_red\nproperty uchar diffuse_green\nproperty uchar diffuse_blue\nend_header\n";
    for (const PLYPoint &pp : points)
        out << pp.first[0] << ' ' << pp.first[1] << ' ' << pp.first[2] << ' ' << (int)pp.second.r << ' '
            << (int)pp.second.g << ' ' << (int)pp.second.b << '\n';
}

class MultiViewStereo : public Task {
public:
    MultiViewStereo() : minDepth(10), maxDepth(100), numDepthLevels(100), crossCheckThreshold(1), imageScale(1) {
        sr_params_default(&params_, 1);
    }

    void initialize(ProjectPtr project, ImageSetPtr imageSet, const std::vector<CameraPtr> &views, double minDepth,
                    double maxDepth, int numDepthLevels, double crossCheckThreshold, double imageScale = 1.0) {
        this->project = project;
        imageSet_ = imageSet;
        this->minDepth = minDepth;
        this->maxDepth = maxDepth;
        this->numDepthLevels = numDepthLevels;
        this->crossCheckThreshold = crossCheckThreshold;
        this->imageScale = imageScale;
        this->views.clear();
        peakPairs_.clear();
        keptCloud_.clear();
        cloudKept_ = false;
        inMemory_ = false;
        images.clear();
        masks.clear();
        results.clear();
        computedDepths.clear();
        depthIndices.clear();
        for (const CameraPtr &view : views) {
            if (!view || !imageSet) continue;
            ProjectImagePtr pi = imageSet->defaultImageForCamera(view);
            if (!pi) continue;
            QImage base(pi->file());
            if (base.isNull()) continue;  // QFileInfo(file).exists() in the reference (:218)
            addView(view, base);
        }
        neighbours.assign(this->views.size(), std::vector<size_t>());
    }

    //! Extension: the same as initialize() with images handed over in memory (no files, no project).
    void initializeFromImages(const std::vector<CameraPtr> &views, const std::vector<QImage> &baseImages, double minDepth,
                              double maxDepth, int numDepthLevels, double crossCheckThreshold, double imageScale = 1.0) {
        initialize(ProjectPtr(), ImageSetPtr(), std::vector<CameraPtr>(), minDepth, maxDepth, numDepthLevels,
                   crossCheckThreshold, imageScale);
        for (size_t i = 0; i < views.size() && i < baseImages.size(); ++i)
            if (views[i] && !baseImages[i].isNull()) addView(views[i], baseImages[i]);
        neighbours.assign(this->views.size(), std::vector<size_t>());
        inMemory_ = true;
    }

    // Task implementation
    std::string title() const { return "Multi-view Stereo"; }
    int numSteps() const { return 2 * (int)views.size(); }

    //! The depth map of `view` (gray: black = close, white = far or unknown); null image if unknown view.
    QImage depthMap(CameraPtr view) const {
        for (size_t i = 0; i < views.size(); ++i)
            if (views[i] == view) return VectorImage::toQImage(results[i], false);
        return QImage();
    }
    ImageSetPtr imageSet() const { return imageSet_; }

    // ---- extensions ------------------------------------------------------------------------
    sr_params &params() { return params_; }
    void setDevice(int device) { device_ = device; }
    //! true (default): search along the rasterised epipolar curve, depth from the rays' closest approach —
    //! the reference's live formulation (multiviewstereo.cpp:574-602), so a caller switched over unchanged
    //! gets the reference's depth maps; false: the depth-label cost volume + WTA of the same rule
    //! (SURVEY §8a S4 applied to S2: the reference's compiled-out branch, about twice as fast here).
    //! NOTE imageScale != 1: addView() rescales with this repository's QImage stand-in (bilinear), not Qt's
    //! scaledToWidth (multiviewstereo.cpp:221) — the scaled pixels, and with them the depth maps, can differ
    //! from the reference's in the last gray levels.  Pass pre-scaled images to stay bit-comparable.
    void setCurveMode(bool on) { curveMode_ = on; }
    //! true: also keep, per pixel, the K = 9 largest (ncc, depth) candidates of the search — the
    //! reference's CostFunction::peakPairs (multiviewstereo.cpp:479-482,589-602), the input of its
    //! MRF stage; read with peakPairs() after run().  Works in label and in curve mode.
    void setKeepPeaks(bool on) { params_.keep_cost_volume = on ? (params_.keep_cost_volume | 2) : (params_.keep_cost_volume & ~2); }
    //! [h][w][9][2] (ncc, depth), ascending, padded with (0, -1); the last pair is the pixel's result
    //! before the cross-check.  Empty unless setKeepPeaks(true).
    const std::vector<double> &peakPairs(size_t viewIndex) const { return peakPairs_[viewIndex]; }
    //! true: runTask() also computes every view's coloured point cloud on the GPU (sr_get_points) after the
    //! cross-check, and pointCloud() returns it.  Off by default: the cloud costs a kernel, ~60 MB of copies
    //! per 1080p view and the PLYPoint vector on every run.
    void setKeepPointCloud(bool on) { keepPointCloud_ = on; }
    size_t numViews() const { return views.size(); }
    const std::vector<double> &depths(size_t viewIndex) const { return computedDepths[viewIndex]; }
    const std::vector<int32_t> &indices(size_t viewIndex) const { return depthIndices[viewIndex]; }
    const std::vector<std::vector<size_t> > &selectedNeighbours() const { return neighbours; }
    //! Depth maps as a coloured point cloud (what the GUI's PLY export consumes), views in order, pixels
    //! row-major.  The cloud the last run kept (setKeepPointCloud(true)), else unprojected here on the host.
    std::vector<PLYPoint> pointCloud() const {
        if (cloudKept_) return keptCloud_;
        std::vector<PLYPoint> pts;
        for (size_t v = 0; v < views.size(); ++v) {
            const int w = images[v].width(), h = images[v].height();
            const Eigen::Vector3d n = views[v]->principleRay().direction();
            for (int y = 0; y < h; ++y)
                for (int x = 0; x < w; ++x) {
                    const double d = computedDepths[v][(size_t)y * w + x];
                    if (!std::isfinite(d) || d + 1e-5 < minDepth) continue;
                    Ray3d::Point p;
                    const Ray3d ray = views[v]->unproject((x + 0.5) / imageScale, (y + 0.5) / imageScale);
                    if (intersect(ray, Plane3d(n, views[v]->C() + n * d), p)) pts.push_back(PLYPoint(p, images[v].pixel(x, y)));
                }
        }
        return pts;
    }

protected:
    void runTask() {
        keptCloud_.clear();
        cloudKept_ = false;
        if ((!inMemory_ && (!project || !imageSet_)) || views.empty()) return;  // multiviewstereo.cpp:326-327
        const int V = (int)views.size();
        const int w = images[0].width(), h = images[0].height();
        for (const VectorImage &im : images)
            if (im.width() != w || im.height() != h) throw std::runtime_error("MultiViewStereo: the B200 path needs equally sized views");
        sr_host::Session s(device_);
        std::vector<sr_camera> cams(V);
        std::vector<std::vector<uint8_t> > rgba(V), msk(V);
        std::vector<const uint8_t *> ip(V), mp(V);
        for (int v = 0; v < V; ++v) {
            cams[v] = views[v]->toPod();
            rgba[v] = images[v].toRGBA8();
            msk[v] = masks[v].toMask8();
            ip[v] = rgba[v].data();
            mp[v] = msk[v].data();
        }
        s.check(sr_set_views(s.get(), V, cams.data(), ip.data(), mp.data(), w, h), "sr_set_views");
        params_.min_depth = minDepth;
        params_.max_depth = maxDepth;
        params_.num_levels = numDepthLevels;
        params_.image_scale = imageScale;
        s.check(sr_set_params(s.get(), &params_), "sr_set_params");

        const int maxN = 3;  // NUM_NEIGHBOURING_VIEWS, multiviewstereo.cpp:96
        std::vector<int32_t> nb((size_t)V * maxN), cnt(V);
        s.check(sr_select_neighbours(s.get(), maxN, nb.data(), cnt.data()), "sr_select_neighbours");
        for (int v = 0; v < V; ++v) neighbours[v].assign(nb.begin() + (size_t)v * maxN, nb.begin() + (size_t)v * maxN + cnt[v]);

        int step = 0;
        for (int v = 0; v < V; ++v) {
            progressUpdate(step++);
            if (isCancelled()) { sr_request_cancel(s.get()); return; }
            stageUpdate("Computing cost volume for camera " + views[v]->name());
            if (cnt[v] > 0) {
                if (curveMode_) s.check(sr_run_view_curve(s.get(), v, &nb[(size_t)v * maxN], cnt[v]), "sr_run_view_curve");
                else s.check(sr_run_view(s.get(), v, &nb[(size_t)v * maxN], cnt[v]), "sr_run_view");
                if (params_.keep_cost_volume & 2) {  // the library keeps the lists of the last view only
                    peakPairs_[v].resize((size_t)w * h * 18);
                    s.check(sr_get_peaks(s.get(), v, peakPairs_[v].data()), "sr_get_peaks");
                }
            } else {
                // no neighbour was selected: the reference's loops find no candidate, which leaves -1 on the
                // in-mask pixels and +INF on the others (multiviewstereo.cpp:559-565,604)
                std::vector<double> fill((size_t)w * h);
                for (int y = 0; y < h; ++y)
                    for (int x = 0; x < w; ++x)
                        fill[(size_t)y * w + x] = (masks[v].pixel(x, y) == WHITE) ? -1.0 : std::numeric_limits<double>::infinity();
                s.check(sr_set_depth(s.get(), v, fill.data()), "sr_set_depth");
            }
        }
        stageUpdate("Constructing depth maps");
        fetch(s, w, h);
        coverage_before_ = coverage();
        stageUpdate("Cross-checking");
        for (int v = 0; v < V; ++v) progressUpdate(step++);
        if (isCancelled()) return;
        s.check(sr_cross_check(s.get(), 0, crossCheckThreshold), "sr_cross_check");
        stageUpdate("Constructing depth maps");
        fetch(s, w, h);
        coverage_after_ = coverage();
        if (keepPointCloud_) keepPointCloud(s);
    }

public:
    //! Fraction of in-mask pixels with a finite depth, per view, before / after the cross-check
    //! (what the reference prints with qDebug, multiviewstereo.cpp:419-420,472-473).
    const std::vector<double> &coverageBeforeCrossCheck() const { return coverage_before_; }
    const std::vector<double> &coverageAfterCrossCheck() const { return coverage_after_; }

private:
    void addView(const CameraPtr &view, const QImage &base) {
        QImage image = base.scaledToWidth((int)(base.width() * imageScale));
        images.push_back(VectorImage::fromQImage(image));
        masks.push_back(VectorImage(image.width(), image.height(), WHITE));
        if (base.hasAlphaChannel()) {  // anything not fully opaque is ignored (:225-237)
            for (int y = 0; y < image.height(); ++y)
                for (int x = 0; x < image.width(); ++x)
                    if (image.pixel(x, y)[3] != 255) masks.back().setPixel(x, y, BLACK);
        }
        results.push_back(VectorImage(image.width(), image.height()));
        computedDepths.push_back(std::vector<double>((size_t)image.width() * image.height(), std::numeric_limits<double>::quiet_NaN()));
        depthIndices.push_back(std::vector<int32_t>((size_t)image.width() * image.height(), -1));
        peakPairs_.push_back(std::vector<double>());
        views.push_back(view);
    }

    void fetch(sr_host::Session &s, int w, int h) {
        std::vector<uint8_t> img((size_t)w * h * 4);
        for (size_t v = 0; v < views.size(); ++v) {
            s.check(sr_get_depth(s.get(), (int)v, computedDepths[v].data()), "sr_get_depth");
            s.check(sr_get_depth_index(s.get(), (int)v, depthIndices[v].data()), "sr_get_depth_index");
            s.check(sr_get_depth_image(s.get(), (int)v, 1, img.data()), "sr_get_depth_image");
            results[v] = VectorImage::fromQImage(QImage(img.data(), w, h, false));
        }
    }

    void keepPointCloud(sr_host::Session &s) {
        std::vector<double> xyz;
        std::vector<uint8_t> rgb;
        for (size_t v = 0; v < views.size(); ++v) {
            int64_t n = 0;
            s.check(sr_get_points(s.get(), (int)v, 0, nullptr, nullptr, nullptr, &n), "sr_get_points");
            if (n == 0) continue;
            xyz.resize((size_t)n * 3);
            rgb.resize((size_t)n * 3);
            s.check(sr_get_points(s.get(), (int)v, n, xyz.data(), rgb.data(), nullptr, &n), "sr_get_points");
            keptCloud_.reserve(keptCloud_.size() + (size_t)n);
            for (size_t i = 0; i < (size_t)n; ++i)
                keptCloud_.push_back(PLYPoint(Ray3d::Point(xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2]),
                                              RGBA(rgb[3 * i], rgb[3 * i + 1], rgb[3 * i + 2])));
        }
        cloudKept_ = true;
    }

    std::vector<double> coverage() const {
        std::vector<double> out;
        for (size_t v = 0; v < views.size(); ++v) {
            size_t total = 0, have = 0;
            const int w = images[v].width(), h = images[v].height();
            for (int y = 0; y < h; ++y)
                for (int x = 0; x < w; ++x)
                    if (masks[v].pixel(x, y) == WHITE) {
                        ++total;
                        if (std::isfinite(computedDepths[v][(size_t)y * w + x])) ++have;
                    }
            out.push_back(total ? (double)have / total : 0.0);
        }
        return out;
    }

    ProjectPtr project;
    ImageSetPtr imageSet_;
    std::vector<CameraPtr> views;
    std::vector<std::vector<size_t> > neighbours;
    std::vector<VectorImage> images, masks, results;
    std::vector<std::vector<double> > computedDepths;
    std::vector<std::vector<int32_t> > depthIndices;
    std::vector<std::vector<double> > peakPairs_;
    std::vector<double> coverage_before_, coverage_after_;
    std::vector<PLYPoint> keptCloud_;
    bool keepPointCloud_ = false;
    bool cloudKept_ = false;  // keptCloud_ belongs to the last run
    double minDepth, maxDepth;
    int numDepthLevels;
    double crossCheckThreshold;
    double imageScale;
    sr_params params_;
    int device_ = 0;
    bool inMemory_ = false;
    bool curveMode_ = true;   // the reference's live formulation; setCurveMode(false) = depth-label cost volume
};
#endif
