// md2_png_host.cpp - a serial host restatement of md2_png.cu's passes over md2_png.h for one image: every bit position
// through the block finder, every candidate's count decode, the walk from bit 0 (decoding a block itself where no
// candidate is), every walked candidate's write with markers, marker resolution, the Adler-32 check and the row
// filters.  tests/test_png_decode.py compiles it with g++.
#include <stdlib.h>
#include <string.h>
#include <vector>
#include "md2_png.h"

namespace {
struct Cand {
  uint32_t pos;
  Md2PngEnd e;
  long long g;
};
}  // namespace

// `use_finder` = 0 skips the finder, so the walk decodes every block itself.  Returns the status word; *n_cands and
// *n_walked (when given) get the candidates found and the ones the walk took.
extern "C" int decode_host(const unsigned char* data, const md2_png_job* j, unsigned char* frame, int use_finder,
                           int* n_cands, int* n_walked) {
  const long long limit = (long long)j->height * (3LL * j->width + 1), rowb = 3LL * j->width + 1;
  Md2PngBits bits;
  md2_png_bits_init(bits, data + j->stream_offset, (uint32_t)j->stream_bytes);
  std::vector<Cand> cands;
  uint8_t cl_lut[128];
  Md2PngHuff* h = new Md2PngHuff;
  for (uint32_t b = 0; use_finder && b < (uint32_t)j->stream_bytes; ++b) {
    for (int k = 0; k < 8; ++k) {                     // the window test of md2_png_find, one position at a time
      const uint32_t pos = b * 8u + (uint32_t)k;
      md2_png_seek(bits, pos);
      const uint64_t v = bits.buf;
      const uint32_t type = (uint32_t)(v >> 1) & 3u;
      bool cand = false;
      if (type == 2) {
        cand = ((v >> 3) & 31u) <= 29u && ((v >> 8) & 31u) <= 29u && md2_png_header_plausible(bits, pos, cl_lut);
      } else if (type == 0) {
        const uint32_t at = b + (k <= 5 ? 1 : 2);
        const uint32_t len = md2_png_byte(bits, at) | md2_png_byte(bits, at + 1) << 8;
        const uint32_t nlen = md2_png_byte(bits, at + 2) | md2_png_byte(bits, at + 3) << 8;
        cand = len == (nlen ^ 0xFFFFu);
      }
      if (cand) cands.push_back({pos, {0u, 0, 0u, 0, 0}, -1});
    }
  }
  for (Cand& c : cands) c.e = md2_png_block<false>(bits, *h, c.pos, 0, limit, nullptr);
  std::vector<uint32_t> out32((size_t)limit);
  unsigned st = 0;
  long long g = 0;
  uint32_t pos = 0;
  int check = 0, walked = 0;
  uint32_t trailer = 0;
  for (;;) {                                           // md2_png_chain
    Cand* c = nullptr;
    for (Cand& x : cands)
      if (x.pos == pos) c = &x;
    Md2PngEnd e;
    if (c) {
      c->g = g;
      e = c->e;
      ++walked;
    } else {
      e = md2_png_block<true>(bits, *h, pos, g, limit, out32.data());
      st |= md2_png_block_status(e, g, limit);
    }
    const long long at = g + e.out;
    const bool last = e.flags || e.stop || e.final || at > limit;
    if (e.final && !e.flags && !e.stop && at <= limit) {
      const uint32_t tb = (e.end + 7u) >> 3;
      if ((long long)tb + 4 > j->stream_bytes) {
        if (at < limit) st |= MD2_PNG_EXHAUSTED;
      } else {
        check = at < limit && (at == 0 || at % rowb) ? 2 : 1;
        trailer = md2_png_byte(bits, tb) << 24 | md2_png_byte(bits, tb + 1) << 16 | md2_png_byte(bits, tb + 2) << 8 |
                  md2_png_byte(bits, tb + 3);
      }
    }
    g = at;
    pos = e.end;
    if (last) break;
  }
  const long long produced = g < limit ? g : limit;
  for (const Cand& c : cands) {                        // md2_png_write
    if (c.g < 0) continue;
    const Md2PngEnd e = md2_png_block<true>(bits, *h, c.pos, c.g, limit, out32.data());
    st |= md2_png_block_status(e, c.g, limit);
    if (e.flags)
      for (long long q = c.g + e.out; q < c.g + c.e.out && q < limit; ++q) out32[q] = 0;
  }
  std::vector<unsigned char> raw((size_t)limit);
  unsigned long long s1 = 0, sq = 0;
  for (long long q = 0; q < limit; ++q) {              // md2_png_resolve
    uint32_t v = 0;
    if (q < produced) {
      v = out32[q];
      long long cur = q;
      while (v >= 256u) {
        const long long src = (long long)(v - 256u);
        if (src >= cur) { v = 0; break; }
        cur = src;
        v = out32[src];
      }
    }
    raw[q] = (unsigned char)v;
    s1 = (s1 + v) % MD2_PNG_ADLER_MOD;
    sq = (sq + (unsigned long long)q * v) % MD2_PNG_ADLER_MOD;
  }
  if (check) {
    const unsigned long long M = MD2_PNG_ADLER_MOD, n = (unsigned long long)produced % M;
    const unsigned a = (unsigned)((1 + s1) % M), b = (unsigned)((n + n * s1 % M + M - sq) % M);
    if ((b << 16 | a) != trailer)
      st |= MD2_PNG_CHECKSUM;
    else if (check == 2)
      st |= MD2_PNG_EXHAUSTED;
  }
  for (int y = 0; y < j->height; ++y) {                // md2_png_unfilter, a tile at a time as the wavefront does
    int f = raw[y * rowb];
    if (f > 4) { st |= MD2_PNG_BAD_FILTER; f = 0; }
    unsigned char left[3] = {0, 0, 0}, upleft[3] = {0, 0, 0};
    for (int x0 = 0; x0 < j->width; x0 += 16)
      md2_png_unfilter_span(f, &raw[y * rowb + 1], y ? frame + (long long)(y - 1) * 3 * j->width : nullptr,
                            frame + (long long)y * 3 * j->width, x0, x0 + 16 < j->width ? x0 + 16 : j->width, left,
                            upleft);
  }
  delete h;
  if (n_cands) *n_cands = (int)cands.size();
  if (n_walked) *n_walked = walked;
  return (int)st;
}

#ifdef MD2_PNG_HOST_MAIN
// md2_png_host <packed buffer file> <use finder>: decodes the one image whose md2_png_job is at offset 0 of the
// buffer and prints its status word (the AddressSanitizer build checks every access on corrupt streams).
#include <stdio.h>
int main(int argc, char** argv) {
  if (argc != 3) return 2;
  FILE* f = fopen(argv[1], "rb");
  if (!f) return 2;
  fseek(f, 0, SEEK_END);
  const long n = ftell(f);
  fseek(f, 0, SEEK_SET);
  unsigned char* buf = (unsigned char*)malloc(n);
  if (fread(buf, 1, n, f) != (size_t)n) return 2;
  fclose(f);
  md2_png_job j;
  memcpy(&j, buf, sizeof(j));
  unsigned char* out = (unsigned char*)malloc((size_t)j.height * j.width * 3);
  const int st = decode_host(buf, &j, out, atoi(argv[2]), nullptr, nullptr);
  printf("%d\n", st);
  free(out);
  free(buf);
  return 0;
}
#endif
