// test_brf_rd_sweep_ext.cpp -- the BRF overloads of jpegRateDistortionGray and jpegViewRateDistortionGray of include/filter_ext.h,
// called through cv::Mat (oracle/refshim's stand-in here).  Reads a raw rows x cols 8-bit disparity and a raw rows x cols x 3
// texture, runs both sweeps with the chain and BRF 13x13 (1, 1, 1) and prints one line per (mode, quality) and per (mode,
// quality, camera); tests/test_cpp_brf_rd_sweep_ext.py compares them with jpegRateDistortion / jpegViewRateDistortion.
//   test_brf_rd_sweep_ext <disp.raw> <texture.raw> <rows> <cols> <f> <tx> <quality>...
#include "filter.h"
#include "filter_ext.h"
#include <cstdio>
#include <cstdlib>
#include <vector>

static bool read_raw(const char* path, void* dst, size_t bytes) {
    FILE* f = fopen(path, "rb");
    const bool ok = f && fread(dst, 1, bytes, f) == bytes;
    if (f) fclose(f);
    return ok;
}

int main(int argc, char** argv) {
    if (argc < 8) { fprintf(stderr, "usage: %s disp.raw texture.raw rows cols f tx quality...\n", argv[0]); return 2; }
    const int rows = atoi(argv[3]), cols = atoi(argv[4]);
    const double f = atof(argv[5]), tx = atof(argv[6]);
    Mat disp(rows, cols, CV_8U), tex(rows, cols, CV_8UC3);
    if (!read_raw(argv[1], disp.data, (size_t)rows * cols) || !read_raw(argv[2], tex.data, (size_t)rows * cols * 3)) { fprintf(stderr, "cannot read the inputs\n"); return 2; }
    vector<int> qualities;
    for (int i = 7; i < argc; i++) qualities.push_back(atoi(argv[i]));
    Mat K = Mat::zeros(3, 3, CV_64F);
    K.at<double>(0, 0) = f; K.at<double>(1, 1) = f; K.at<double>(0, 2) = (cols - 1) * 0.5; K.at<double>(1, 2) = (rows - 1) * 0.5; K.at<double>(2, 2) = 1.0;
    vector<Mat> R, t;
    for (int v = 0; v < 2; v++) {
        Mat r = Mat::zeros(3, 3, CV_64F), tt = Mat::zeros(3, 1, CV_64F);
        for (int i = 0; i < 3; i++) r.at<double>(i, i) = 1.0;
        tt.at<double>(0, 0) = v ? -tx : tx;
        R.push_back(r); t.push_back(tt);
    }
    for (int optimize = 0; optimize < 2; optimize++) {
        vector<int> bytes; vector<double> pc, pf, pb;
        jpegRateDistortionGray(disp, qualities, bytes, pc, pf, 2, 1, 3, 5, 10, Size(13, 13), 1.f, 1.f, 1.f, pb, optimize != 0);
        if (bytes.size() != qualities.size() || pb.size() != qualities.size()) return 3;
        for (size_t k = 0; k < qualities.size(); k++) printf("gray %d %d %d %.17g %.17g %.17g\n", optimize, qualities[k], bytes[k], pc[k], pf[k], pb[k]);
        vector<vector<double> > vc, vf, vb;
        jpegViewRateDistortionGray(disp, tex, qualities, 75.0, 575.0, 2.6, 1, 0, 1, 3, 65.f, f, R, t, K, true, bytes, vc, vf, Size(13, 13), 1.f, 1.f, 1.f, vb, optimize != 0);
        if (bytes.size() != qualities.size() || vb.size() != qualities.size()) return 3;
        for (size_t k = 0; k < qualities.size(); k++)
            for (size_t v = 0; v < R.size(); v++) printf("view %d %d %d %d %.17g %.17g %.17g\n", optimize, qualities[k], (int)v, bytes[k], vc[k][v], vf[k][v], vb[k][v]);
    }
    printf("ALL OK\n");
    return 0;
}
