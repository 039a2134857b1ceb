// point_cloud_test — MultiViewStereo::pointCloud() with the cloud kept on the GPU (setKeepPointCloud(true),
// sr_get_points) against the host loop of the same class (the flag off), on the same in-memory views.
// Used by tests/test_gpu_point_cloud.py, and by tools/point_cloud_timing.py for the host loop's time.
//
//   point_cloud_test <scene.bin> <outdir|-> <minDepth> <maxDepth> <levels> <crossCheck> <curve 0|1>
//
// scene.bin: int32 V, w, h; V sr_camera PODs; V images of h*w RGBA8 (alpha != 255: masked).
// Prints one line "points kept=<n> host=<n> same_rgb=<0|1> max_rel=<e> host_ms=<ms>"; max_rel is the largest
// |kept - host| / max(1, |host|) over all coordinates (inf when the counts differ).  With an outdir, also
// writes kept_xyz.bin, kept_rgb.bin, host_xyz.bin, host_rgb.bin (float64 [n][3], uint8 [n][3]).
#include <chrono>
#include <cmath>
#include <cstdio>
#include <fstream>
#include <limits>

#include "stereo/multiviewstereo.hpp"

static void dump_cloud(const std::string &prefix, const std::vector<PLYPoint> &pts) {
    std::vector<double> xyz;
    std::vector<uint8_t> rgb;
    for (const PLYPoint &p : pts) {
        for (int k = 0; k < 3; ++k) xyz.push_back(p.first[k]);
        rgb.push_back((uint8_t)p.second.r);
        rgb.push_back((uint8_t)p.second.g);
        rgb.push_back((uint8_t)p.second.b);
    }
    std::ofstream(prefix + "_xyz.bin", std::ios::binary).write(reinterpret_cast<const char *>(xyz.data()), (std::streamsize)(xyz.size() * 8));
    std::ofstream(prefix + "_rgb.bin", std::ios::binary).write(reinterpret_cast<const char *>(rgb.data()), (std::streamsize)rgb.size());
}

int main(int argc, char **argv) {
    if (argc != 8) {
        std::fprintf(stderr, "usage: %s scene.bin outdir|- minDepth maxDepth levels crossCheck curve\n", argv[0]);
        return 2;
    }
    try {
        std::ifstream f(argv[1], std::ios::binary);
        int32_t hdr[3] = {0, 0, 0};
        f.read(reinterpret_cast<char *>(hdr), sizeof(hdr));
        const int V = hdr[0], w = hdr[1], h = hdr[2];
        std::vector<sr_camera> pods(V);
        f.read(reinterpret_cast<char *>(pods.data()), (std::streamsize)(sizeof(sr_camera) * V));
        std::vector<CameraPtr> views;
        std::vector<QImage> images;
        std::vector<uint8_t> rgba((size_t)w * h * 4);
        for (int v = 0; v < V; ++v) {
            const sr_camera &c = pods[v];
            Eigen::Matrix3d K, R;
            for (int i = 0; i < 3; ++i)
                for (int j = 0; j < 3; ++j) {
                    K(i, j) = c.K[3 * i + j];
                    R(i, j) = c.R[3 * i + j];
                }
            CameraPtr cam(new Camera("cam" + std::to_string(v), "view " + std::to_string(v)));
            cam->set(K, R, Eigen::Vector3d(c.t[0], c.t[1], c.t[2]));
            cam->setLensDistortion(LensDistortions{{c.dist[0], c.dist[1], c.dist[2], c.dist[3], c.dist[4]}});
            cam->setRefractiveIndex(c.n);
            cam->setPlane(Plane3d(Eigen::Vector3d(c.plane_n[0], c.plane_n[1], c.plane_n[2]), c.plane_d));
            views.push_back(cam);
            f.read(reinterpret_cast<char *>(rgba.data()), (std::streamsize)rgba.size());
            images.push_back(QImage(rgba.data(), w, h, true));
        }
        if (!f) throw std::runtime_error("short scene file");

        MultiViewStereo mvs;
        mvs.initializeFromImages(views, images, std::atof(argv[3]), std::atof(argv[4]), std::atoi(argv[5]), std::atof(argv[6]));
        mvs.setCurveMode(std::atoi(argv[7]) != 0);
        mvs.setKeepPointCloud(true);
        mvs.run();
        const std::vector<PLYPoint> kept = mvs.pointCloud();
        mvs.setKeepPointCloud(false);
        mvs.run();
        const auto t0 = std::chrono::steady_clock::now();
        const std::vector<PLYPoint> host = mvs.pointCloud();
        const double host_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();

        bool same_rgb = kept.size() == host.size();
        double max_rel = kept.size() == host.size() ? 0.0 : std::numeric_limits<double>::infinity();
        for (size_t i = 0; i < kept.size() && i < host.size(); ++i) {
            for (int k = 0; k < 3; ++k) {
                const double a = kept[i].first[k], b = host[i].first[k];
                const double rel = std::fabs(a - b) / std::max(1.0, std::fabs(b));
                max_rel = (rel > max_rel || !(rel == rel)) ? rel : max_rel;
            }
            same_rgb = same_rgb && kept[i].second.r == host[i].second.r && kept[i].second.g == host[i].second.g &&
                       kept[i].second.b == host[i].second.b;
        }
        if (std::string(argv[2]) != "-") {
            dump_cloud(std::string(argv[2]) + "/kept", kept);
            dump_cloud(std::string(argv[2]) + "/host", host);
        }
        std::printf("points kept=%zu host=%zu same_rgb=%d max_rel=%.3e host_ms=%.1f\n", kept.size(), host.size(), (int)same_rgb,
                    max_rel, host_ms);
    } catch (const std::exception &e) {
        std::fprintf(stderr, "point_cloud_test: %s\n", e.what());
        return 1;
    }
    return 0;
}
