// test_jpeg_ext_opt.cpp -- the optimised-table mode of the JPEG extensions of include/filter_ext.h (jpegEncodeGray and
// degradeJPEGGray with optimize = true) called through cv::Mat (oracle/refshim's stand-in here).  Reads a raw rows x cols
// 8-bit image, writes what the calls produce; the comparison with cv2 is done by tests/test_cpp_jpeg_ext_opt.py.
//   test_jpeg_ext_opt <in.raw> <rows> <cols> <quality> <out_dir>
#include "filter.h"
#include "filter_ext.h"
#include <cstdio>
#include <string>
#include <vector>

static bool write_file(const std::string& path, const void* p, size_t n) {
    FILE* f = fopen(path.c_str(), "wb");
    if (!f) return false;
    const bool ok = fwrite(p, 1, n, f) == n;
    return fclose(f) == 0 && ok;
}

int main(int argc, char** argv) {
    if (argc != 6) { fprintf(stderr, "usage: %s in.raw rows cols quality out_dir\n", argv[0]); return 2; }
    const int rows = atoi(argv[2]), cols = atoi(argv[3]), q = atoi(argv[4]);
    const std::string out = argv[5];
    Mat img(rows, cols, CV_8U);
    FILE* f = fopen(argv[1], "rb");
    if (!f || fread(img.data, 1, (size_t)rows * cols, f) != (size_t)rows * cols) { fprintf(stderr, "cannot read %s\n", argv[1]); return 2; }
    fclose(f);

    vector<uchar> buf, std_buf;
    jpegEncodeGray(img, buf, q, true);
    jpegEncodeGray(img, std_buf, q);                  // the default stays the standard tables
    Mat dec;
    const int n = degradeJPEGGray(img, dec, q, true);
    if (!write_file(out + "/stream.jpg", buf.data(), buf.size()) || !write_file(out + "/standard.jpg", std_buf.data(), std_buf.size()) ||
        !write_file(out + "/degraded.raw", dec.data, (size_t)rows * cols)) return 2;
    printf("bytes %zu %d\n", buf.size(), n);

    // a region of interest (row step larger than the row) and an in-place call
    if (rows > 2 && cols > 2) {
        Mat roi = img(Rect(1, 1, cols - 2, rows - 2));
        vector<uchar> rbuf;
        jpegEncodeGray(roi, rbuf, q, true);
        Mat inplace = roi.clone();
        const int rn = degradeJPEGGray(inplace, inplace, q, true);
        if (!write_file(out + "/roi.jpg", rbuf.data(), rbuf.size()) || !write_file(out + "/roi_degraded.raw", inplace.data, (size_t)(rows - 2) * (cols - 2))) return 2;
        printf("roi %zu %d\n", rbuf.size(), rn);
    }
    printf("ALL OK\n");
    return 0;
}
