// The video flow of one Detector per stream segment: detect(img, thresh, use_mean) and then tracking(result, story)
// for every frame in order (yolo_v2_class.cpp:173-304).  tests/test_track_gpu.py compares the tracked streams entries
// with its lines.
//
//   detector_track <cfg> <weights> <thresh> <nms> <story> <frames.u8> <spec.txt> <gpu_id>
// spec.txt, one line each: "new" (a fresh Detector for the frames below) or "frame <byte offset> <w> <h> <use_mean>"
// (uint8 interleaved RGB in frames.u8, converted as load_image does: (float)byte / 255.).
#include <cstdio>
#include <cstdlib>
#include <memory>
#include <string>
#include <vector>

#include "yolo_v2_class.hpp"

static void dump(int k, const std::vector<bbox_t> &v)
{
    printf("track %d %zu", k, v.size());
    for (const bbox_t &b : v) printf(" %u %u %u %u %.9g %u %u", b.x, b.y, b.w, b.h, b.prob, b.obj_id, b.track_id);
    printf("\n");
}

int main(int argc, char **argv)
{
    if (argc < 9) {
        fprintf(stderr, "usage: detector_track cfg weights thresh nms story frames.u8 spec.txt gpu_id\n");
        return 1;
    }
    const float thresh = (float)atof(argv[3]), nms = (float)atof(argv[4]);
    const int story = atoi(argv[5]), gpu = atoi(argv[8]);
    FILE *f = fopen(argv[6], "rb");
    if (!f) return 2;
    fseek(f, 0, SEEK_END);
    std::vector<unsigned char> bytes((size_t)ftell(f));
    fseek(f, 0, SEEK_SET);
    if (fread(bytes.data(), 1, bytes.size(), f) != bytes.size()) return 2;
    fclose(f);
    FILE *spec = fopen(argv[7], "r");
    if (!spec) return 3;
    std::unique_ptr<Detector> det;
    char word[16];
    int k = 0;
    while (fscanf(spec, "%15s", word) == 1) {
        if (std::string(word) == "new") {
            det.reset();
            det.reset(new Detector(argv[1], argv[2], gpu));
            det->nms = nms;
            continue;
        }
        long long off = 0;
        int w = 0, h = 0, use_mean = 0;
        if (fscanf(spec, "%lld %d %d %d", &off, &w, &h, &use_mean) != 4 || !det) return 4;
        std::vector<float> planar((size_t)3 * w * h);
        for (int c = 0; c < 3; ++c)
            for (int y = 0; y < h; ++y)
                for (int x = 0; x < w; ++x)
                    planar[((size_t)c * h + y) * w + x] = (float)bytes[off + ((size_t)y * w + x) * 3 + c] / 255.;
        image_t im;
        im.w = w;
        im.h = h;
        im.c = 3;
        im.data = planar.data();
        dump(k++, det->tracking(det->detect(im, thresh, use_mean != 0), story));
    }
    fclose(spec);
    return 0;
}
