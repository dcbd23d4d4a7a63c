// The shim's camera constructor frame(camera_image, cols, rows, channels) against its gray constructor: a keyframe and frames built
// from BGR camera images (gray, undistortion and resize on the GPU) track to the same poses as the same sequence built from the
// level-0 images the CPU oracle computes from those camera images.
// Input blob (written by tests/test_host_shim_ingest.py): int32 w, h, W, H, n; f32 fx fy cx cy; f64 K[9], dist[5], alpha; u8 keyframe
// camera image (W x H x 3); 4 depth levels; 4 variance levels; n camera images; u8 keyframe gray (w x h); n gray images.
// Prints "img <0|1>" per frame (level-0 image equal to the oracle's) and one "pose <pass> <i> ..." line per track.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "DepthPropagation.h"
#include "ExternVariable.h"
#include "Frame.h"
#include "ImageFunc.h"

static void rd(FILE* f, void* p, size_t n) { if (fread(p, 1, n, f) != n) { fprintf(stderr, "short read\n"); exit(2); } }

int main(int argc, char** argv) {
    if (argc < 2) { fprintf(stderr, "usage: test_shim_ingest blob\n"); return 2; }
    FILE* f = fopen(argv[1], "rb");
    if (!f) return 2;
    int w, h, W, H, n; float k[4]; double K[9], dist[5], alpha;
    rd(f, &w, 4); rd(f, &h, 4); rd(f, &W, 4); rd(f, &H, 4); rd(f, &n, 4); rd(f, k, 16);
    rd(f, K, sizeof(K)); rd(f, dist, sizeof(dist)); rd(f, &alpha, 8);
    std::vector<unsigned char> kf_cam((size_t)W * H * 3), kf_gray((size_t)w * h);
    rd(f, kf_cam.data(), kf_cam.size());
    std::vector<std::vector<float> > depth(4), var(4);
    for (int l = 0; l < 4; ++l) { depth[l].resize((size_t)(w >> l) * (h >> l)); rd(f, depth[l].data(), depth[l].size() * 4); }
    for (int l = 0; l < 4; ++l) { var[l].resize((size_t)(w >> l) * (h >> l)); rd(f, var[l].data(), var[l].size() * 4); }
    std::vector<std::vector<unsigned char> > cams(n, std::vector<unsigned char>((size_t)W * H * 3)), grays(n, std::vector<unsigned char>((size_t)w * h));
    for (auto& c : cams) rd(f, c.data(), c.size());
    rd(f, kf_gray.data(), kf_gray.size());
    for (auto& g : grays) rd(f, g.data(), g.size());
    fclose(f);
    try {
        util::configure(w, h, k[0], k[1], k[2], k[3]);
        util::configure_camera(W, H, 3, K, dist, true, (float)W / w, alpha);
        printf("size %d %d\n", util::ORIG_COLS, util::ORIG_ROWS);
        for (int pass = 0; pass < 2; ++pass) {                      // 0: camera constructor, 1: gray constructor
            frame* kf = pass == 0 ? new frame(kf_cam.data(), W, H, 3) : new frame(kf_gray.data(), w, h);
            if (pass == 0) printf("img %d\n", std::memcmp(kf->image.ptr<unsigned char>(0), kf_gray.data(), kf_gray.size()) == 0 ? 1 : 0);
            depthMap dm;
            dm.keyFrame = kf;
            for (int l = 0; l < 4; ++l) {
                std::memcpy(kf->depth_pyramid[l].ptr<float>(0), depth[l].data(), depth[l].size() * 4);
                std::memcpy(dm.depthvararrptr[l], var[l].data(), var[l].size() * 4);
            }
            dm.markDepthUpdated();
            frame* prev = kf;
            std::vector<frame*> frames;
            for (int i = 0; i < n; ++i) {
                frame* cur = pass == 0 ? new frame(cams[i].data(), W, H, 3) : new frame(grays[i].data(), w, h);
                if (pass == 0) printf("img %d\n", std::memcmp(cur->image.ptr<unsigned char>(0), grays[i].data(), grays[i].size()) == 0 ? 1 : 0);
                frames.push_back(cur);
                float init[6] = {0, 0, 0, 0, 0, 0};
                std::vector<float> p = GetImagePoseEstimate(kf, cur, i + 2, &dm, prev, init);
                printf("pose %d %d %.9g %.9g %.9g %.9g %.9g %.9g\n", pass, i, p[0], p[1], p[2], p[3], p[4], p[5]);
                prev = cur;
            }
            for (frame* c : frames) delete c;
            delete kf;
        }
        ellc_host::shutdown();
    } catch (const std::exception& e) {
        fprintf(stderr, "error: %s\n", e.what());
        return 1;
    }
    return 0;
}
