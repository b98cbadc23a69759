// test_rd_sweep_ext.cpp -- jpegRateDistortionGray of include/filter_ext.h called through cv::Mat (oracle/refshim's stand-in
// here).  Reads a raw rows x cols 8-bit image and prints one line per (mode, quality); tests/test_cpp_rd_sweep_ext.py
// compares them with cv2 and the port.
//   test_rd_sweep_ext <in.raw> <rows> <cols> <quality>...
#include "filter.h"
#include "filter_ext.h"
#include <cstdio>
#include <cstdlib>
#include <vector>

int main(int argc, char** argv) {
    if (argc < 5) { fprintf(stderr, "usage: %s in.raw rows cols quality...\n", argv[0]); return 2; }
    const int rows = atoi(argv[2]), cols = atoi(argv[3]);
    Mat img(rows, cols, CV_8U);
    FILE* f = fopen(argv[1], "rb");
    if (!f || fread(img.data, 1, (size_t)rows * cols, f) != (size_t)rows * cols) { fprintf(stderr, "cannot read %s\n", argv[1]); return 2; }
    fclose(f);
    vector<int> qualities;
    for (int i = 4; i < argc; i++) qualities.push_back(atoi(argv[i]));
    for (int optimize = 0; optimize < 2; optimize++) {
        vector<int> bytes; vector<double> pc, pf;
        jpegRateDistortionGray(img, qualities, bytes, pc, pf, 2, 1, 3, 5, 10, optimize != 0);
        if (bytes.size() != qualities.size() || pc.size() != qualities.size() || pf.size() != qualities.size()) return 3;
        for (size_t k = 0; k < qualities.size(); k++) printf("rd %d %d %d %.17g %.17g\n", optimize, qualities[k], bytes[k], pc[k], pf[k]);
    }
    printf("ALL OK\n");
    return 0;
}
