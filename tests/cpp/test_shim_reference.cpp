// The C++ host shim with util::GPU_ARITHMETIC = ELLC_ARITH_REFERENCE: one GetImagePoseEstimate of a frame on a keyframe at the
// origin with the t-1 frame at the origin, as the reference's own driver ran it for tests/golden/reference_track_480x270.npz.
// Input blob (written by tests/test_host_shim_reference.py): int32 w, h, n_frames (= 1); f32 fx fy cx cy; u8 keyframe image;
// 4 depth levels; 4 variance levels; one u8 frame image.  Prints the returned pose, poseWrtOrigin and poseWrtWorld.
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "../../include/ellc_gn.h"
#include "DepthPropagation.h"
#include "ExternVariable.h"
#include "Frame.h"
#include "ImageFunc.h"

static void rd(FILE* f, void* p, size_t n) { if (fread(p, 1, n, f) != n) { fprintf(stderr, "short read\n"); exit(2); } }

int main(int argc, char** argv) {
    if (argc < 2) return 2;
    FILE* f = fopen(argv[1], "rb");
    if (!f) return 2;
    int w, h, n; float k[4];
    rd(f, &w, 4); rd(f, &h, 4); rd(f, &n, 4); rd(f, k, 16);
    util::configure(w, h, k[0], k[1], k[2], k[3]);
    util::GPU_ARITHMETIC = ELLC_ARITH_REFERENCE;
    std::vector<unsigned char> img((size_t)w * h);
    rd(f, img.data(), img.size());
    try {
        frame kf(img.data(), w, h);
        depthMap dm;
        dm.keyFrame = &kf;
        for (int l = 0; l < 4; ++l) rd(f, kf.depth_pyramid[l].ptr<float>(0), (size_t)(w >> l) * (h >> l) * 4);
        for (int l = 0; l < 4; ++l) rd(f, dm.depthvararrptr[l], (size_t)(w >> l) * (h >> l) * 4);
        dm.markDepthUpdated();
        rd(f, img.data(), img.size());
        frame cur(img.data(), w, h);
        float init[6] = {0, 0, 0, 0, 0, 0};
        std::vector<float> p = GetImagePoseEstimate(&kf, &cur, 2, &dm, &kf, init);
        printf("pose %.9g %.9g %.9g %.9g %.9g %.9g\n", p[0], p[1], p[2], p[3], p[4], p[5]);
        printf("origin %.9g %.9g %.9g %.9g %.9g %.9g\n", cur.poseWrtOrigin[0], cur.poseWrtOrigin[1], cur.poseWrtOrigin[2],
               cur.poseWrtOrigin[3], cur.poseWrtOrigin[4], cur.poseWrtOrigin[5]);
        printf("world %.9g %.9g %.9g %.9g %.9g %.9g\n", cur.poseWrtWorld[0], cur.poseWrtWorld[1], cur.poseWrtWorld[2],
               cur.poseWrtWorld[3], cur.poseWrtWorld[4], cur.poseWrtWorld[5]);
    } catch (const std::exception& e) {
        fprintf(stderr, "%s\n", e.what());
        return 1;
    }
    ellc_host::shutdown();
    fclose(f);
    return 0;
}
