#pragma once
#include <cstdint>
#include <string>
#include <vector>
namespace moxh {
void accumToRgb8(const float* accum, uint32_t W, uint32_t H, float nAccum, uint8_t* out);
// The same with a sample count per pixel (W*H, row 0 = bottom, as the accumulator); a count of 0 gives black.
void accumToRgb8Counts(const float* accum, uint32_t W, uint32_t H, const uint32_t* counts, uint8_t* out);
bool writeImage(const std::string& path, const uint8_t* rgb, uint32_t W, uint32_t H, std::string& err);
// Decode an image file (PNG 8-bit non-interlaced, binary PPM/PGM, PFM) into RGBA float texels with
// row 0 = BOTTOM of the picture and alpha = 1, which is how the reference fills its texture buffers
// from a QImage (MinimalOptiX.cpp:459-470).
bool readImageRgba(const std::string& path, int& w, int& h, std::vector<float>& texels, std::string& err);
bool writeAccum(const std::string& path, const float* accum, uint32_t W, uint32_t H, uint64_t launches, std::string& err);
bool readAccum(const std::string& path, float* accum, uint32_t W, uint32_t H, uint64_t* launches, std::string& err);
}
