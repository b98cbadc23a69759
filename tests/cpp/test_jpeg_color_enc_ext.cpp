// test_jpeg_color_enc_ext.cpp -- jpegEncodeColor and degradeJPEGColor of include/filter_ext.h called through cv::Mat
// (oracle/refshim's stand-in here).  Reads a rows x cols x 3 BGR file and, for every sampling, writes the stream to
// <in>.<sampling>.jpg and the round trip to <in>.<sampling>.bgr, printing the round trip's byte count; the comparison
// with cv2 is done by tests/test_cpp_jpeg_color_enc_ext.py.  A CV_8UC1 source must be refused.
//   test_jpeg_color_enc_ext <in.bgr> <rows> <cols> <quality>
#include "filter.h"
#include "filter_ext.h"
#include <cstdio>
#include <cstdlib>
#include <string>

static bool write_file(const std::string& path, const void* p, size_t n) {
    FILE* o = fopen(path.c_str(), "wb");
    return o && fwrite(p, 1, n, o) == n && fclose(o) == 0;
}

int main(int argc, char** argv) {
    if (argc != 5) { fprintf(stderr, "usage: %s in.bgr rows cols quality\n", argv[0]); return 2; }
    const int rows = atoi(argv[2]), cols = atoi(argv[3]), quality = atoi(argv[4]);
    Mat src(rows, cols, CV_8UC3);
    FILE* f = fopen(argv[1], "rb");
    if (!f || fread(src.data, 1, (size_t)rows * cols * 3, f) != (size_t)rows * cols * 3) { fprintf(stderr, "cannot read %s\n", argv[1]); return 2; }
    fclose(f);
    const struct { const char* name; int sampling; } samplings[] = {{"444", DMC_JPEG_SAMPLING_444}, {"422", DMC_JPEG_SAMPLING_422}, {"420", DMC_JPEG_SAMPLING_420},
                                                                    {"440", DMC_JPEG_SAMPLING_440}, {"411", DMC_JPEG_SAMPLING_411}};
    for (const auto& s : samplings) {
        vector<uchar> buf;
        jpegEncodeColor(src, buf, quality, s.sampling);
        Mat dec;
        const int bytes = degradeJPEGColor(src, dec, quality, s.sampling);
        if (dec.type() != CV_8UC3 || dec.rows != rows || dec.cols != cols) { printf("FAIL %s: bad round-trip image\n", s.name); return 1; }
        const std::string base = std::string(argv[1]) + "." + s.name;
        if (!write_file(base + ".jpg", buf.data(), buf.size()) || !write_file(base + ".bgr", dec.data, (size_t)rows * cols * 3)) return 2;
        printf("sampling %s %zu %d\n", s.name, buf.size(), bytes);
    }
    vector<uchar> def;
    jpegEncodeColor(src, def, quality);
    if (!write_file(std::string(argv[1]) + ".default.jpg", def.data(), def.size())) return 2;
    try {
        Mat gray(rows, cols, CV_8UC1);
        vector<uchar> buf;
        jpegEncodeColor(gray, buf, quality);
        printf("FAIL: CV_8UC1 accepted\n");
        return 1;
    } catch (const cv::Exception& e) {
        printf("refused gray: %s\n", e.what());
    }
    printf("ALL OK\n");
    return 0;
}
