// mrf_class_test — MultiViewStereo with setMrf(true) (sr_mrf_select after each view's search, before the
// cross-check) or without it, on in-memory views; writes every view's final depth map and index map.
// Used by tests/test_gpu_mrf.py, which compares them with the C-ABI sequence run -> sr_mrf_select -> cross-check.
//
//   mrf_class_test <scene.bin> <outdir> <minDepth> <maxDepth> <levels> <crossCheck> <curve 0|1> <mrf 0|1>
//
// scene.bin: int32 V, w, h; V sr_camera PODs; V images of h*w RGBA8 (alpha != 255: masked).
// Writes <outdir>/depth.bin (float64 [V][h][w]) and <outdir>/index.bin (int32 [V][h][w]); prints
// "mrf views=<V> w=<w> h=<h>".
#include <cstdio>
#include <fstream>

#include "stereo/multiviewstereo.hpp"

int main(int argc, char **argv) {
    if (argc != 9) {
        std::fprintf(stderr, "usage: %s scene.bin outdir minDepth maxDepth levels crossCheck curve mrf\n", argv[0]);
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
        mvs.setMrf(std::atoi(argv[8]) != 0);
        mvs.run();
        std::ofstream d(std::string(argv[2]) + "/depth.bin", std::ios::binary), i(std::string(argv[2]) + "/index.bin", std::ios::binary);
        for (int v = 0; v < V; ++v) {
            d.write(reinterpret_cast<const char *>(mvs.depths(v).data()), (std::streamsize)(mvs.depths(v).size() * 8));
            i.write(reinterpret_cast<const char *>(mvs.indices(v).data()), (std::streamsize)(mvs.indices(v).size() * 4));
        }
        std::printf("mrf views=%d w=%d h=%d\n", V, w, h);
    } catch (const std::exception &e) {
        std::fprintf(stderr, "mrf_class_test: %s\n", e.what());
        return 1;
    }
    return 0;
}
