// test_jpeg_color_ext.cpp -- jpegDecodeColor of include/filter_ext.h called through cv::Mat (oracle/refshim's stand-in
// here).  Decodes each stream file to <stream>.bgr (rows x cols x 3 bytes); the comparison with cv2.imdecode is done by
// tests/test_cpp_jpeg_color_ext.py.  A stream that is refused prints "refused <file>: <reason>".
//   test_jpeg_color_ext <a.jpg> [<b.jpg> ...]
#include "filter.h"
#include "filter_ext.h"
#include <cstdio>
#include <string>
#include <vector>

int main(int argc, char** argv) {
    if (argc < 2) { fprintf(stderr, "usage: %s a.jpg [b.jpg ...]\n", argv[0]); return 2; }
    for (int a = 1; a < argc; a++) {
        FILE* f = fopen(argv[a], "rb");
        if (!f) { fprintf(stderr, "cannot read %s\n", argv[a]); return 2; }
        vector<uchar> buf;
        uchar tmp[65536]; size_t n;
        while ((n = fread(tmp, 1, sizeof tmp, f)) > 0) buf.insert(buf.end(), tmp, tmp + n);
        fclose(f);
        Mat dst;
        try {
            jpegDecodeColor(buf, dst);
        } catch (const cv::Exception& e) {
            printf("refused %s: %s\n", argv[a], e.what());
            continue;
        }
        if (dst.type() != CV_8UC3) { printf("FAIL %s: not CV_8UC3\n", argv[a]); return 1; }
        const std::string out = std::string(argv[a]) + ".bgr";
        FILE* o = fopen(out.c_str(), "wb");
        const size_t bytes = (size_t)dst.rows * dst.cols * 3;
        if (!o || fwrite(dst.data, 1, bytes, o) != bytes || fclose(o) != 0) return 2;
        printf("decoded %s %d %d\n", argv[a], dst.rows, dst.cols);
    }
    printf("ALL OK\n");
    return 0;
}
