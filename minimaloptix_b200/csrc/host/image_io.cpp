// image_io.cpp — display conversion and file output of the accumulation buffer
// (reference: MinimalOptiX::updateContent / saveCurrentFrame, MinimalOptiX.cpp:43-84; Qt's
// QImage/QColor replaced by a dependency-free PNG/PPM writer).
#include "image_io.h"
#include "jpeg_decode.h"

#include <algorithm>
#include <cctype>
#include <cmath>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

namespace moxh {

// QColor::setRedF stores round(v * 65535) as 16 bit; QImage RGB888 keeps the high byte.
static inline uint8_t quantise(float v) {
  v = fmaxf(0.f, fminf(v, 1.f));
  return (uint8_t)(((uint32_t)floorf(v * 65535.0f + 0.5f)) >> 8);
}

void accumToRgb8(const float* accum, uint32_t W, uint32_t H, float nAccum, uint8_t* out) {
  for (uint32_t i = 0; i < H; ++i)
    for (uint32_t j = 0; j < W; ++j) {
      const float* src = accum + 3 * ((size_t)i * W + j);
      uint8_t* dst = out + 3 * ((size_t)(H - 1 - i) * W + j);  // accumulator row 0 is the image bottom
      dst[0] = quantise(src[0] / nAccum);
      dst[1] = quantise(src[1] / nAccum);
      dst[2] = quantise(src[2] / nAccum);
    }
}

void accumToRgb8Counts(const float* accum, uint32_t W, uint32_t H, const uint32_t* counts, uint8_t* out) {
  for (uint32_t i = 0; i < H; ++i)
    for (uint32_t j = 0; j < W; ++j) {
      const size_t p = (size_t)i * W + j;
      const float* src = accum + 3 * p;
      uint8_t* dst = out + 3 * ((size_t)(H - 1 - i) * W + j);
      if (!counts[p]) { dst[0] = dst[1] = dst[2] = 0; continue; }   // a pixel nobody rendered
      const float n = (float)counts[p];
      dst[0] = quantise(src[0] / n);
      dst[1] = quantise(src[1] / n);
      dst[2] = quantise(src[2] / n);
    }
}

namespace {
uint32_t crcTable[256];
bool crcInit = false;
uint32_t crc32(uint32_t crc, const uint8_t* p, size_t n) {
  if (!crcInit) {
    for (uint32_t i = 0; i < 256; ++i) {
      uint32_t c = i;
      for (int k = 0; k < 8; ++k) c = c & 1 ? 0xEDB88320u ^ (c >> 1) : c >> 1;
      crcTable[i] = c;
    }
    crcInit = true;
  }
  crc = ~crc;
  for (size_t i = 0; i < n; ++i) crc = crcTable[(crc ^ p[i]) & 0xFF] ^ (crc >> 8);
  return ~crc;
}
void put32(std::vector<uint8_t>& v, uint32_t x) { v.push_back(x >> 24); v.push_back(x >> 16); v.push_back(x >> 8); v.push_back(x); }
void chunk(FILE* f, const char* type, const std::vector<uint8_t>& data) {
  std::vector<uint8_t> buf;
  put32(buf, (uint32_t)data.size());
  fwrite(buf.data(), 1, 4, f);
  std::vector<uint8_t> body(type, type + 4);
  body.insert(body.end(), data.begin(), data.end());
  fwrite(body.data(), 1, body.size(), f);
  buf.clear();
  put32(buf, crc32(0, body.data(), body.size()));
  fwrite(buf.data(), 1, 4, f);
}
}  // namespace

bool writeImage(const std::string& path, const uint8_t* rgb, uint32_t W, uint32_t H, std::string& err) {
  FILE* f = fopen(path.c_str(), "wb");
  if (!f) { err = "cannot open " + path; return false; }
  bool ppm = path.size() > 4 && path.substr(path.size() - 4) == ".ppm";
  if (ppm) {
    fprintf(f, "P6\n%u %u\n255\n", W, H);
    fwrite(rgb, 1, (size_t)W * H * 3, f);
    fclose(f);
    return true;
  }
  static const uint8_t sig[8] = {0x89, 'P', 'N', 'G', '\r', '\n', 0x1a, '\n'};
  fwrite(sig, 1, 8, f);
  std::vector<uint8_t> ihdr;
  put32(ihdr, W); put32(ihdr, H);
  ihdr.push_back(8); ihdr.push_back(2); ihdr.push_back(0); ihdr.push_back(0); ihdr.push_back(0);
  chunk(f, "IHDR", ihdr);
  // zlib stream of stored (uncompressed) deflate blocks over the filtered scanlines.
  std::vector<uint8_t> raw;
  raw.reserve((size_t)H * (3 * W + 1));
  for (uint32_t y = 0; y < H; ++y) { raw.push_back(0); raw.insert(raw.end(), rgb + (size_t)y * W * 3, rgb + (size_t)(y + 1) * W * 3); }
  std::vector<uint8_t> z;
  z.push_back(0x78); z.push_back(0x01);
  size_t pos = 0;
  uint32_t a = 1, b = 0;
  while (pos < raw.size() || raw.empty()) {
    size_t n = std::min<size_t>(65535, raw.size() - pos);
    bool last = pos + n >= raw.size();
    z.push_back(last ? 1 : 0);
    z.push_back(n & 0xFF); z.push_back(n >> 8); z.push_back(~n & 0xFF); z.push_back((~n >> 8) & 0xFF);
    z.insert(z.end(), raw.begin() + pos, raw.begin() + pos + n);
    for (size_t i = pos; i < pos + n; ++i) { a = (a + raw[i]) % 65521; b = (b + a) % 65521; }
    pos += n;
    if (last) break;
  }
  put32(z, (b << 16) | a);
  chunk(f, "IDAT", z);
  chunk(f, "IEND", {});
  fclose(f);
  return true;
}

// ------------------------------------------------------------------ image decoding (textures)
namespace {

// RFC 1951 inflate: stored, fixed and dynamic Huffman blocks.
struct Inflater {
  const uint8_t* in; size_t n, pos = 0; uint32_t bitBuf = 0; int bitCnt = 0;
  std::vector<uint8_t>& out;
  bool ok = true;
  Inflater(const uint8_t* p, size_t len, std::vector<uint8_t>& o) : in(p), n(len), out(o) {}
  uint32_t bits(int need) {
    while (bitCnt < need) {
      if (pos >= n) { ok = false; return 0; }
      bitBuf |= (uint32_t)in[pos++] << bitCnt;
      bitCnt += 8;
    }
    uint32_t v = bitBuf & ((need == 32) ? 0xffffffffu : ((1u << need) - 1u));
    bitBuf >>= need; bitCnt -= need;
    return v;
  }
  struct Huff { uint16_t count[16]; uint16_t symbol[288]; };
  static void build(Huff& h, const uint8_t* len, int nsym) {
    memset(h.count, 0, sizeof h.count);
    for (int i = 0; i < nsym; ++i) h.count[len[i]]++;
    h.count[0] = 0;
    uint16_t offs[16]; offs[1] = 0;
    for (int i = 1; i < 15; ++i) offs[i + 1] = offs[i] + h.count[i];
    for (int i = 0; i < nsym; ++i) if (len[i]) h.symbol[offs[len[i]]++] = (uint16_t)i;
  }
  int decode(const Huff& h) {
    int code = 0, first = 0, index = 0;
    for (int len = 1; len <= 15; ++len) {
      code |= (int)bits(1);
      if (!ok) return -1;
      int count = h.count[len];
      if (code - count < first) return h.symbol[index + (code - first)];
      index += count; first += count; first <<= 1; code <<= 1;
    }
    ok = false;
    return -1;
  }
  bool codes(const Huff& lit, const Huff& dist) {
    static const uint16_t lbase[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
    static const uint16_t lext[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
    static const uint16_t dbase[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
    static const uint16_t dext[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
    for (;;) {
      int sym = decode(lit);
      if (!ok) return false;
      if (sym < 256) out.push_back((uint8_t)sym);
      else if (sym == 256) return true;
      else {
        sym -= 257;
        if (sym >= 29) return false;
        int len = lbase[sym] + (int)bits(lext[sym]);
        int ds = decode(dist);
        if (!ok || ds < 0 || ds >= 30) return false;
        size_t d = dbase[ds] + bits(dext[ds]);
        if (!ok || d > out.size()) return false;
        size_t from = out.size() - d;
        for (int k = 0; k < len; ++k) out.push_back(out[from + k]);
      }
    }
  }
  bool run() {
    for (;;) {
      uint32_t last = bits(1), type = bits(2);
      if (!ok) return false;
      if (type == 0) {
        bitBuf = 0; bitCnt = 0;
        if (pos + 4 > n) return false;
        uint32_t len = in[pos] | (in[pos + 1] << 8);
        pos += 4;
        if (pos + len > n) return false;
        out.insert(out.end(), in + pos, in + pos + len);
        pos += len;
      } else if (type == 1) {
        uint8_t l[288];
        for (int i = 0; i < 144; ++i) l[i] = 8;
        for (int i = 144; i < 256; ++i) l[i] = 9;
        for (int i = 256; i < 280; ++i) l[i] = 7;
        for (int i = 280; i < 288; ++i) l[i] = 8;
        Huff lit, dist;
        build(lit, l, 288);
        uint8_t dl[30];
        for (int i = 0; i < 30; ++i) dl[i] = 5;
        build(dist, dl, 30);
        if (!codes(lit, dist)) return false;
      } else if (type == 2) {
        int nlen = (int)bits(5) + 257, ndist = (int)bits(5) + 1, ncode = (int)bits(4) + 4;
        if (!ok || nlen > 286 || ndist > 30) return false;
        static const uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
        uint8_t lengths[320];
        memset(lengths, 0, sizeof lengths);
        for (int i = 0; i < ncode; ++i) lengths[order[i]] = (uint8_t)bits(3);
        Huff lencode;
        build(lencode, lengths, 19);
        uint8_t ll[320];
        memset(ll, 0, sizeof ll);
        int idx = 0;
        while (idx < nlen + ndist) {
          int sym = decode(lencode);
          if (!ok) return false;
          if (sym < 16) ll[idx++] = (uint8_t)sym;
          else {
            int rep, val = 0;
            if (sym == 16) { if (idx == 0) return false; val = ll[idx - 1]; rep = 3 + (int)bits(2); }
            else if (sym == 17) rep = 3 + (int)bits(3);
            else rep = 11 + (int)bits(7);
            if (idx + rep > nlen + ndist) return false;
            while (rep--) ll[idx++] = (uint8_t)val;
          }
        }
        Huff lit, dist;
        build(lit, ll, nlen);
        build(dist, ll + nlen, ndist);
        if (!codes(lit, dist)) return false;
      } else {
        return false;
      }
      if (last) return ok;
    }
  }
};

bool readWhole(const std::string& path, std::vector<uint8_t>& data) {
  FILE* f = fopen(path.c_str(), "rb");
  if (!f) return false;
  uint8_t buf[1 << 16];
  size_t n;
  while ((n = fread(buf, 1, sizeof buf, f)) > 0) data.insert(data.end(), buf, buf + n);
  fclose(f);
  return true;
}

inline uint32_t be32(const uint8_t* p) { return ((uint32_t)p[0] << 24) | (p[1] << 16) | (p[2] << 8) | p[3]; }

// rows top-down, `ch` channels of 8 bit -> RGBA float, flipped so row 0 is the bottom
void toTexels(const std::vector<uint8_t>& px, int w, int h, int ch, const uint8_t* palette, std::vector<float>& texels) {
  texels.resize((size_t)w * h * 4);
  for (int y = 0; y < h; ++y)
    for (int x = 0; x < w; ++x) {
      const uint8_t* s = &px[((size_t)y * w + x) * ch];
      float r, g, b;
      if (palette) { const uint8_t* q = palette + 3 * s[0]; r = q[0]; g = q[1]; b = q[2]; }
      else if (ch <= 2) { r = g = b = s[0]; }
      else { r = s[0]; g = s[1]; b = s[2]; }
      float* d = &texels[((size_t)(h - 1 - y) * w + x) * 4];
      d[0] = r / 255.0f; d[1] = g / 255.0f; d[2] = b / 255.0f; d[3] = 1.f;  // QColor::redF() == value / 255
    }
}

// PNG as QImage (libpng) presents it to the reference's texel loop (MinimalOptiX.cpp:445-479): grey / RGB /
// palette with or without alpha at 1, 2, 4, 8 or 16 bits, Adam7 interlacing; 16-bit samples keep their
// high byte, low-depth grey is scaled to 0..255, alpha is ignored (the loop reads red/green/blue only).
bool readPng(const std::vector<uint8_t>& f, int& w, int& h, std::vector<float>& texels, std::string& err) {
  size_t pos = 8;
  int depth = 0, ctype = 0, interlace = 0;
  std::vector<uint8_t> idat, palette;
  while (pos + 12 <= f.size()) {
    uint32_t len = be32(&f[pos]);
    const uint8_t* type = &f[pos + 4];
    if (pos + 12 + (size_t)len > f.size()) break;
    const uint8_t* body = &f[pos + 8];
    if (!memcmp(type, "IHDR", 4) && len >= 13) { w = (int)be32(body); h = (int)be32(body + 4); depth = body[8]; ctype = body[9]; interlace = body[12]; }
    else if (!memcmp(type, "PLTE", 4)) palette.assign(body, body + len);
    else if (!memcmp(type, "IDAT", 4)) idat.insert(idat.end(), body, body + len);
    else if (!memcmp(type, "IEND", 4)) break;
    pos += 12 + len;
  }
  const int ch = ctype == 0 ? 1 : ctype == 2 ? 3 : ctype == 3 ? 1 : ctype == 4 ? 2 : ctype == 6 ? 4 : 0;
  const bool depthOk = ctype == 0 ? (depth == 1 || depth == 2 || depth == 4 || depth == 8 || depth == 16)
                     : ctype == 3 ? (depth == 1 || depth == 2 || depth == 4 || depth == 8) : (depth == 8 || depth == 16);
  if (w <= 0 || h <= 0 || (int64_t)w * h > ((int64_t)1 << 28) || !ch || !depthOk || interlace > 1) { err = "unsupported PNG header"; return false; }
  if (ctype == 3) palette.resize(3 * 256, 0);
  if (idat.size() < 6) { err = "corrupt PNG data"; return false; }
  std::vector<uint8_t> raw;
  Inflater inf(idat.data() + 2, idat.size() - 2, raw);  // skip the zlib header; the Adler-32 trailer is ignored
  const bool inflated = inf.run();
  const int bpp = depth * ch;                    // bits per pixel
  const size_t fu = (size_t)std::max(1, bpp / 8);  // filter unit in bytes
  std::vector<uint8_t> px((size_t)w * h * 3);
  std::vector<uint8_t> prev, cur;
  size_t rp = 0;
  // Adam7: pass p covers pixels (x0 + i*dx, y0 + j*dy); a non-interlaced image is one pass with unit steps
  static const int X0[7] = {0, 4, 0, 2, 0, 1, 0}, Y0[7] = {0, 0, 4, 0, 2, 0, 1}, DX[7] = {8, 8, 4, 4, 2, 2, 1}, DY[7] = {8, 8, 8, 4, 4, 2, 2};
  const int npass = interlace ? 7 : 1;
  for (int p = 0; p < npass; ++p) {
    const int x0 = interlace ? X0[p] : 0, y0 = interlace ? Y0[p] : 0, dx = interlace ? DX[p] : 1, dy = interlace ? DY[p] : 1;
    const int pw = (w - x0 + dx - 1) / dx, ph = (h - y0 + dy - 1) / dy;
    if (pw <= 0 || ph <= 0) continue;
    const size_t stride = ((size_t)pw * bpp + 7) / 8;
    prev.assign(stride, 0);
    cur.resize(stride);
    for (int j = 0; j < ph; ++j) {
      if (rp + 1 + stride > raw.size()) { err = inflated ? "truncated PNG data" : "corrupt PNG data"; return false; }
      const int ft = raw[rp];
      const uint8_t* src = &raw[rp + 1];
      rp += 1 + stride;
      for (size_t i = 0; i < stride; ++i) {
        const int a = i >= fu ? cur[i - fu] : 0, b = prev[i], c = i >= fu ? prev[i - fu] : 0;
        int v = src[i];
        switch (ft) {
          case 1: v += a; break;
          case 2: v += b; break;
          case 3: v += (a + b) >> 1; break;
          case 4: { int q = a + b - c, pa = abs(q - a), pb = abs(q - b), pc = abs(q - c); v += (pa <= pb && pa <= pc) ? a : (pb <= pc ? b : c); break; }
          default: break;
        }
        cur[i] = (uint8_t)v;
      }
      const int y = y0 + j * dy;
      for (int i = 0; i < pw; ++i) {
        uint8_t s[4] = {0, 0, 0, 0};
        if (depth == 8) for (int k = 0; k < ch; ++k) s[k] = cur[(size_t)i * ch + k];
        else if (depth == 16) for (int k = 0; k < ch; ++k) s[k] = cur[((size_t)i * ch + k) * 2];
        else {
          const int bit = i * depth, v = (cur[bit >> 3] >> (8 - depth - (bit & 7))) & ((1 << depth) - 1);
          s[0] = ctype == 3 ? (uint8_t)v : (uint8_t)(v * 255 / ((1 << depth) - 1));
        }
        uint8_t* d = &px[((size_t)y * w + x0 + i * dx) * 3];
        if (ctype == 3) { const uint8_t* q = &palette[3 * s[0]]; d[0] = q[0]; d[1] = q[1]; d[2] = q[2]; }
        else if (ch <= 2) d[0] = d[1] = d[2] = s[0];
        else { d[0] = s[0]; d[1] = s[1]; d[2] = s[2]; }
      }
      prev.swap(cur);
    }
  }
  toTexels(px, w, h, 3, nullptr, texels);
  return true;
}

}  // namespace

bool readImageRgba(const std::string& path, int& w, int& h, std::vector<float>& texels, std::string& err) {
  std::vector<uint8_t> f;
  if (!readWhole(path, f)) { err = "cannot open " + path; return false; }
  static const uint8_t sig[8] = {0x89, 'P', 'N', 'G', '\r', '\n', 0x1a, '\n'};
  if (f.size() > 8 && !memcmp(f.data(), sig, 8)) return readPng(f, w, h, texels, err);
  if (f.size() > 3 && f[0] == 0xff && f[1] == 0xd8) {
    std::vector<uint8_t> px;
    if (!decodeJpeg(f.data(), f.size(), w, h, px, err)) { err += ": " + path; return false; }
    toTexels(px, w, h, 3, nullptr, texels);
    return true;
  }
  if (f.size() > 2 && f[0] == 'P' && (f[1] == '6' || f[1] == '5' || f[1] == 'F' || f[1] == 'f')) {
    // netpbm header: magic, width, height, maxval (or scale for PFM), one whitespace, data
    // The header is text of unknown length inside a binary buffer: parse a NUL-terminated copy
    // of its first bytes so strtod can never run past the end of a truncated file.
    const std::string head((const char*)f.data(), std::min<size_t>(f.size(), 512));
    size_t pos = 2;
    double vals[3];
    for (int k = 0; k < 3; ++k) {
      while (pos < head.size() && (isspace((unsigned char)head[pos]) || head[pos] == '#')) { if (head[pos] == '#') while (pos < head.size() && head[pos] != '\n') ++pos; else ++pos; }
      if (pos >= head.size()) { err = "truncated netpbm header"; return false; }
      char* end = nullptr;
      vals[k] = strtod(head.c_str() + pos, &end);
      if (end == head.c_str() + pos) { err = "bad netpbm header"; return false; }
      pos = (size_t)(end - head.c_str());
    }
    if (pos >= f.size()) { err = "truncated netpbm header"; return false; }
    ++pos;
    w = (int)vals[0]; h = (int)vals[1];
    if (w <= 0 || h <= 0) { err = "bad netpbm header"; return false; }
    if (f[1] == '6' || f[1] == '5') {
      int ch = f[1] == '6' ? 3 : 1;
      if (vals[2] != 255 || pos + (size_t)w * h * ch > f.size()) { err = "unsupported netpbm file"; return false; }
      std::vector<uint8_t> px(f.begin() + pos, f.begin() + pos + (size_t)w * h * ch);
      toTexels(px, w, h, ch, nullptr, texels);
      return true;
    }
    int ch = f[1] == 'F' ? 3 : 1;  // PFM: rows bottom-up already, little-endian when scale < 0
    if (vals[2] >= 0 || pos + (size_t)w * h * ch * 4 > f.size()) { err = "unsupported PFM (need little-endian)"; return false; }
    texels.resize((size_t)w * h * 4);
    const uint8_t* src = &f[pos];   // not 4-byte aligned in general: the header has any length
    auto at = [&](size_t k) { float v; memcpy(&v, src + 4 * k, 4); return v; };
    for (size_t i = 0; i < (size_t)w * h; ++i) {
      float r = at(i * ch), g = ch == 3 ? at(i * ch + 1) : r, b = ch == 3 ? at(i * ch + 2) : r;
      texels[4 * i] = r; texels[4 * i + 1] = g; texels[4 * i + 2] = b; texels[4 * i + 3] = 1.f;
    }
    return true;
  }
  err = "unknown image format: " + path;
  return false;
}

bool writeAccum(const std::string& path, const float* accum, uint32_t W, uint32_t H, uint64_t launches, std::string& err) {
  FILE* f = fopen(path.c_str(), "wb");
  if (!f) { err = "cannot open " + path; return false; }
  fwrite("MOXA", 1, 4, f);
  fwrite(&W, 4, 1, f); fwrite(&H, 4, 1, f); fwrite(&launches, 8, 1, f);
  fwrite(accum, sizeof(float), (size_t)W * H * 3, f);
  fclose(f);
  return true;
}

bool readAccum(const std::string& path, float* accum, uint32_t W, uint32_t H, uint64_t* launches, std::string& err) {
  FILE* f = fopen(path.c_str(), "rb");
  if (!f) { err = "cannot open " + path; return false; }
  char magic[4]; uint32_t w = 0, h = 0; uint64_t n = 0;
  bool ok = fread(magic, 1, 4, f) == 4 && memcmp(magic, "MOXA", 4) == 0 && fread(&w, 4, 1, f) == 1 && fread(&h, 4, 1, f) == 1 &&
            fread(&n, 8, 1, f) == 1 && w == W && h == H && fread(accum, sizeof(float), (size_t)W * H * 3, f) == (size_t)W * H * 3;
  fclose(f);
  if (!ok) { err = "bad accumulator file " + path; return false; }
  if (launches) *launches = n;
  return true;
}

}  // namespace moxh
