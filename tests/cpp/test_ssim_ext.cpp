// test_ssim_ext.cpp -- structuralSimilarity of include/filter_ext.h, called through cv::Mat (oracle/refshim's stand-in here).
// Reads two raw rows x cols x 3 images a and b and prints one line per case: the SSIM of the CV_8UC3 pair, of their first
// channels as CV_8UC1 (whole, and a region of interest with a row step wider than its rows), and of a with itself;
// tests/test_cpp_ssim_ext.py compares them with frameSSIM.  A pair of mismatched types must be refused.
//   test_ssim_ext <a.raw> <b.raw> <rows> <cols>
#include "filter.h"
#include "filter_ext.h"
#include <cstdio>
#include <cstdlib>

static bool read_raw(const char* path, void* dst, size_t bytes) {
    FILE* f = fopen(path, "rb");
    const bool ok = f && fread(dst, 1, bytes, f) == bytes;
    if (f) fclose(f);
    return ok;
}

int main(int argc, char** argv) {
    if (argc != 5) { fprintf(stderr, "usage: %s a.raw b.raw rows cols\n", argv[0]); return 2; }
    const int rows = atoi(argv[3]), cols = atoi(argv[4]);
    Mat a(rows, cols, CV_8UC3), b(rows, cols, CV_8UC3);
    if (!read_raw(argv[1], a.data, (size_t)rows * cols * 3) || !read_raw(argv[2], b.data, (size_t)rows * cols * 3)) { fprintf(stderr, "cannot read the inputs\n"); return 2; }
    Mat ga(rows, cols, CV_8UC1), gb(rows, cols, CV_8UC1);
    for (int y = 0; y < rows; y++)
        for (int x = 0; x < cols; x++) { ga.ptr(y)[x] = a.ptr(y)[3 * x]; gb.ptr(y)[x] = b.ptr(y)[3 * x]; }
    printf("c3 %.17g\n", structuralSimilarity(a, b));
    printf("c1 %.17g\n", structuralSimilarity(ga, gb));
    const Rect roi(3, 2, cols - 7, rows - 5);
    printf("roi %.17g\n", structuralSimilarity(ga(roi), gb(roi)));
    printf("self %.17g\n", structuralSimilarity(a, a));
    bool refused = false;
    try { structuralSimilarity(a, gb); } catch (const cv::Exception&) { refused = true; }
    if (!refused) { fprintf(stderr, "a type mismatch was not refused\n"); return 3; }
    printf("ALL OK\n");
    return 0;
}
