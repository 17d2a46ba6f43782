// fic_cli -- headless stand-in for the reference's GUI action openDecodedImage
// (RLEAppController.java:172-188): encode an image to a .run stream, decode a stream.
//   fic_cli encode in.pgm|in.ppm out.run [blockgroesse] [widthKernel]   (binary P5 / P6)
//   fic_cli decode in.run out.pgm|out.ppm
//   fic_cli roundtrip in.pgm|in.ppm [blockgroesse] [widthKernel]        (prints "MSE <avgError>" like the GUI label)
//   fic_cli qtroundtrip in.pgm b_max b_min widthKernel max_mse            (quadtree extension, grey: stream size, bits
//                                                                          per pixel, iterations, avgError, PSNR)
//   fic_cli qtroundtrip_rgb in.ppm b_max b_min widthKernel max_mse        (the same, RGB: PSNR over the 3*W*H samples)
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <sstream>

#include "fractal_compression.hpp"

using namespace bvk_ss19;

static RasterImage read_pnm(const char *path)
{
    std::ifstream f(path, std::ios::binary);
    if (!f) throw std::runtime_error(std::string("cannot open ") + path);
    std::string magic;
    int w, h, maxv;
    f >> magic >> w >> h >> maxv;
    f.get();
    if ((magic != "P5" && magic != "P6") || maxv != 255) throw std::runtime_error("need binary P5/P6 with maxval 255");
    RasterImage img(w, h);
    std::vector<unsigned char> buf((size_t)w * h * (magic == "P6" ? 3 : 1));
    f.read((char *)buf.data(), (std::streamsize)buf.size());
    for (size_t i = 0; i < (size_t)w * h; i++) {
        unsigned r, g, b;
        if (magic == "P6") { r = buf[3 * i]; g = buf[3 * i + 1]; b = buf[3 * i + 2]; }
        else r = g = b = buf[i];
        img.argb[i] = (int32_t)(0xff000000u | (r << 16) | (g << 8) | b);
    }
    return img;
}

static void write_pnm(const char *path, const RasterImage &img)
{
    bool grey = FractalCompression::isGreyScale(img);
    std::ofstream f(path, std::ios::binary);
    f << (grey ? "P5" : "P6") << "\n" << img.width << " " << img.height << "\n255\n";
    for (int32_t p : img.argb) {
        unsigned char rgb[3] = {(unsigned char)((p >> 16) & 0xff), (unsigned char)((p >> 8) & 0xff), (unsigned char)(p & 0xff)};
        f.write((const char *)rgb, grey ? 1 : 3);
    }
}

// Quadtree round trip on the GPU: grey (the red channel, fic_encode_quadtree) or RGB (three planes,
// fic_encode_quadtree_rgb).  Prints the stream size, bits per pixel, iterations, avgError and the PSNR over every sample.
static int qt_roundtrip(const RasterImage &img, bool rgb, int b_max, int b_min, int wk, double max_mse)
{
    const int W = img.width, H = img.height, C = rgb ? 3 : 1;
    const size_t plane_px = (size_t)W * H;
    std::vector<uint8_t> planes(C * plane_px), out(C * plane_px);
    for (int c = 0; c < C; c++)  // R, G, B planes; grey: the red channel
        for (size_t i = 0; i < plane_px; i++) planes[c * plane_px + i] = (uint8_t)((img.argb[i] >> (16 - 8 * c)) & 0xff);
    std::vector<uint8_t> stream((rgb ? fic_quadtree_rgb_stream_bound : fic_quadtree_stream_bound)(W, H, b_max, b_min) + 1);
    fic_handle *h = nullptr;
    size_t n = 0;
    float avg = 0;
    int iters = 0;
    int rc = fic_create(0, &h);
    if (!rc) rc = (rgb ? fic_encode_quadtree_rgb : fic_encode_quadtree)(h, planes.data(), W, H, b_max, b_min, wk, max_mse, stream.data(), stream.size(), &n);
    if (!rc) rc = (rgb ? fic_decode_quadtree_rgb : fic_decode_quadtree)(h, stream.data(), n, 50, out.data(), &avg, &iters);
    if (rc) {
        fprintf(stderr, "fic_cli: error %d: %s\n", rc, fic_last_error(h));
        fic_destroy(h);
        return 1;
    }
    fic_destroy(h);
    double se = 0;
    for (size_t i = 0; i < planes.size(); i++) se += ((double)planes[i] - out[i]) * ((double)planes[i] - out[i]);
    const double mse = se / (double)planes.size();
    printf("bytes %zu bpp %.4f iterations %d MSE %.9g PSNR %.3f dB\n", n, 8.0 * n / plane_px, iters, avg,
           mse > 0 ? 10.0 * std::log10(255.0 * 255.0 / mse) : INFINITY);
    return 0;
}

int main(int argc, char **argv)
{
    // a trailing "iso" selects the isometry extension for encode / roundtrip
    if (argc > 2 && !strcmp(argv[argc - 1], "iso")) {
        FractalCompression::isometries = true;
        argc--;
    }
    try {
        if (argc >= 4 && !strcmp(argv[1], "encode")) {
            if (argc > 4) FractalCompression::blockgroesse = atoi(argv[4]);
            if (argc > 5) FractalCompression::widthKernel = atoi(argv[5]);
            std::ofstream out(argv[3], std::ios::binary);
            FractalCompression::encode(read_pnm(argv[2]), out);
            return 0;
        }
        if (argc >= 4 && !strcmp(argv[1], "decode")) {
            std::ifstream in(argv[2], std::ios::binary);
            write_pnm(argv[3], FractalCompression::decode(in));
            printf("MSE %.9g (%d iterations)\n", FractalCompression::getAvgError(), FractalCompression::lastIterations);
            return 0;
        }
        if (argc >= 3 && !strcmp(argv[1], "roundtrip")) {
            if (argc > 3) FractalCompression::blockgroesse = atoi(argv[3]);
            if (argc > 4) FractalCompression::widthKernel = atoi(argv[4]);
            std::stringstream ss(std::ios::in | std::ios::out | std::ios::binary);
            FractalCompression::encode(read_pnm(argv[2]), ss);
            ss.seekg(0);
            FractalCompression::decode(ss);
            printf("MSE %.9g (%d iterations)\n", FractalCompression::getAvgError(), FractalCompression::lastIterations);
            return 0;
        }
        if (argc >= 7 && (!strcmp(argv[1], "qtroundtrip") || !strcmp(argv[1], "qtroundtrip_rgb")))
            return qt_roundtrip(read_pnm(argv[2]), !strcmp(argv[1], "qtroundtrip_rgb"), atoi(argv[3]), atoi(argv[4]),
                                atoi(argv[5]), atof(argv[6]));
        fprintf(stderr, "usage: fic_cli encode in.pnm out.run [B] [wk] [iso] | decode in.run out.pnm | roundtrip in.pnm [B] [wk] [iso]"
                        " | qtroundtrip in.pgm b_max b_min wk max_mse | qtroundtrip_rgb in.ppm b_max b_min wk max_mse\n");
        return 2;
    } catch (const std::exception &e) {
        fprintf(stderr, "fic_cli: %s\n", e.what());
        return 1;
    }
}
