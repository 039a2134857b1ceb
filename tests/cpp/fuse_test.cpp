// fuse_test — MultiViewStereo with setFusePointCloud(true, k) for k = 1 and 2, and with the flag off, on the same
// in-memory views.  Used by tests/test_gpu_fuse.py, which compares the fused clouds with Context.fuse_points on
// the dumped depth maps.
//
//   fuse_test <scene.bin> <outdir> <minDepth> <maxDepth> <levels> <crossCheck> <curve 0|1>
//
// scene.bin: int32 V, w, h; V sr_camera PODs; V images of h*w RGBA8 (alpha != 255: masked).
// Writes depth_off.bin, depth_1.bin, depth_2.bin (float64 [V][h][w]), off_xyz.bin / off_rgb.bin (pointCloud()
// with the flag off) and fused<k>_xyz.bin / fused<k>_rgb.bin (float64 [n][3], uint8 [n][3]).  Prints one line
// "fuse off_fused=<n> off_points=<n> fused1=<n> fused2=<n>".
#include <cstdio>
#include <fstream>

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

static void dump_depths(const std::string &path, const MultiViewStereo &mvs) {
    std::ofstream out(path, std::ios::binary);
    for (size_t v = 0; v < mvs.numViews(); ++v)
        out.write(reinterpret_cast<const char *>(mvs.depths(v).data()), (std::streamsize)(mvs.depths(v).size() * 8));
}

int main(int argc, char **argv) {
    if (argc != 8) {
        std::fprintf(stderr, "usage: %s scene.bin outdir minDepth maxDepth levels crossCheck curve\n", argv[0]);
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

        const std::string out = argv[2];
        MultiViewStereo mvs;
        mvs.initializeFromImages(views, images, std::atof(argv[3]), std::atof(argv[4]), std::atoi(argv[5]), std::atof(argv[6]));
        mvs.setCurveMode(std::atoi(argv[7]) != 0);
        mvs.run();
        dump_depths(out + "/depth_off.bin", mvs);
        const std::vector<PLYPoint> off = mvs.pointCloud();
        dump_cloud(out + "/off", off);
        const size_t off_fused = mvs.fusedPointCloud().size();
        size_t fused[3] = {0, 0, 0};
        for (int k = 1; k <= 2; ++k) {
            mvs.setFusePointCloud(true, k);
            mvs.run();
            dump_depths(out + "/depth_" + std::to_string(k) + ".bin", mvs);
            dump_cloud(out + "/fused" + std::to_string(k), mvs.fusedPointCloud());
            fused[k] = mvs.fusedPointCloud().size();
        }
        std::printf("fuse off_fused=%zu off_points=%zu fused1=%zu fused2=%zu\n", off_fused, off.size(), fused[1], fused[2]);
    } catch (const std::exception &e) {
        std::fprintf(stderr, "fuse_test: %s\n", e.what());
        return 1;
    }
    return 0;
}
