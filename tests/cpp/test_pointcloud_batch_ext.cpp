// test_pointcloud_batch_ext.cpp -- prepareDisparityBatch and renderViewBatch of include/filter_ext.h called through cv::Mat
// (oracle/refshim's stand-in here).  Reads n raw rows x cols 16-bit depth frames and n raw rows x cols x 3 textures,
// prepares the disparity (both pass counts), converts it to depth (disp8U2depth32F) and renders two cameras (R = I,
// t = (+-tx, 0, 0), K of pointcloudTest); writes the disparities and the views as raw files next to the inputs.
// tests/test_cpp_pointcloud_batch_ext.py compares them with prepareDisparityBatch and renderViewBatch.
//   test_pointcloud_batch_ext <depth16.raw> <texture.raw> <n> <rows> <cols> <f> <tx> <outdir>
#include "filter.h"
#include "filter_ext.h"
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

static bool read_raw(const char* path, std::vector<unsigned char>& dst) {
    FILE* f = fopen(path, "rb");
    const bool ok = f && fread(dst.data(), 1, dst.size(), f) == dst.size();
    if (f) fclose(f);
    return ok;
}

static bool write_raw(const std::string& path, const Mat& m) {
    FILE* f = fopen(path.c_str(), "ab");
    const size_t bytes = (size_t)m.rows * m.cols * m.elemSize();
    const bool ok = f && fwrite(m.data, 1, bytes, f) == bytes;
    if (f) fclose(f);
    return ok;
}

int main(int argc, char** argv) {
    if (argc != 9) { fprintf(stderr, "usage: %s depth16.raw texture.raw n rows cols f tx outdir\n", argv[0]); return 2; }
    const int n = atoi(argv[3]), rows = atoi(argv[4]), cols = atoi(argv[5]);
    const double f = atof(argv[6]), tx = atof(argv[7]);
    const std::string out = argv[8];
    const size_t px = (size_t)rows * cols;
    std::vector<unsigned char> d16(2 * px * n), tex(3 * px * n);
    if (!read_raw(argv[1], d16) || !read_raw(argv[2], tex)) { fprintf(stderr, "cannot read the inputs\n"); return 2; }
    vector<Mat> depth16(n), texture(n);
    for (int i = 0; i < n; i++) {
        depth16[i].create(rows, cols, CV_16UC1); memcpy(depth16[i].data, &d16[2 * px * i], 2 * px);
        texture[i].create(rows, cols, CV_8UC3); memcpy(texture[i].data, &tex[3 * px * i], 3 * px);
    }
    Mat K = Mat::zeros(3, 3, CV_64F);
    K.at<double>(0, 0) = f; K.at<double>(1, 1) = f; K.at<double>(0, 2) = (cols - 1) * 0.5; K.at<double>(1, 2) = (rows - 1) * 0.5; K.at<double>(2, 2) = 1.0;
    vector<Mat> R, t;
    for (int v = 0; v < 2; v++) {
        Mat r = Mat::zeros(3, 3, CV_64F), tt = Mat::zeros(3, 1, CV_64F);
        for (int i = 0; i < 3; i++) r.at<double>(i, i) = 1.0;
        tt.at<double>(0, 0) = v ? -tx : tx;
        R.push_back(r); t.push_back(tt);
    }
    for (int passes = 1; passes <= 2; passes++) {
        vector<Mat> disp;
        prepareDisparityBatch(depth16, disp, 75.f * 575.f, 2.6f, 0.f, passes);
        if ((int)disp.size() != n) return 3;
        const std::string dp = out + "/disp" + std::to_string(passes) + ".raw";
        for (int i = 0; i < n; i++) if (disp[i].type() != CV_8UC1 || !write_raw(dp, disp[i])) return 4;
        if (passes == 1) continue;
        vector<Mat> depth(n);
        for (int i = 0; i < n; i++) { depth[i] = Mat::zeros(rows, cols, CV_32F); disp8U2depth32F(disp[i], depth[i], 75.f * 575.f, 2.6f, 0.f); }
        vector<vector<Mat> > views;
        renderViewBatch(depth, texture, f, R, t, K, true, views);
        if (views.size() != 2) return 5;
        for (int v = 0; v < 2; v++)
            for (int i = 0; i < n; i++) if (views[v][i].type() != CV_8UC3 || !write_raw(out + "/views.raw", views[v][i])) return 6;
    }
    printf("ALL OK\n");
    return 0;
}
