// md2_jpeg_host.cpp - a serial host restatement of md2_jpeg.cu's four passes over md2_jpeg.h, the chunk size a
// parameter: every chunk re-decodes from its predecessor's previous exit, all at once, until no exit changes (the
// self-synchronising search), then writes its blocks, then the IDCT and the colour pass.  tests/test_jpeg_decode.py
// compiles it with g++.
#include <stdlib.h>
#include <string.h>
#include <vector>
#include "md2_jpeg.h"

extern "C" int decode_host(const unsigned char* data, const md2_jpeg_job* j, int chunk_bytes, unsigned char* out,
                           short* coefs_out, int* rounds_out) {
  const int mx = (j->width + 8 * j->h_samp - 1) / (8 * j->h_samp), my = (j->height + 8 * j->v_samp - 1) / (8 * j->v_samp);
  const int luma = j->h_samp * j->v_samp, bpm = luma + 2, mcus = mx * my;
  const long long nblk = (long long)mcus * bpm;
  const md2_jpeg_tables* tab = (const md2_jpeg_tables*)(data + j->tables_offset);
  const md2_jpeg_segment* segs = (const md2_jpeg_segment*)(data + j->segments_offset);
  Md2JpegImage im;
  im.tab = tab;
  im.luma_blocks = luma;
  im.tables = 0;
  for (int c = 0; c < 3; ++c) im.tables |= (unsigned)(j->dc_table[c] & 1) << c | (unsigned)(j->ac_table[c] & 1) << (3 + c);
  std::vector<short> coefs(nblk * 64, 0);
  unsigned flags = 0;
  const int per = j->restart_interval > 0 ? j->restart_interval : mcus;
  int rounds = 0;
  for (int s = 0; s < j->n_segments; ++s) {
    Md2JpegBits b;
    b.d = data + j->entropy_offset + (long long)segs[s].chunk * MD2_JPEG_CHUNK_BYTES;
    b.n = (unsigned)segs[s].bytes;
    b.bp = 0; b.nb = 0; b.buf = 0;
    const unsigned seg_bits = b.n * 8u;
    const int nch = seg_bits ? (int)((seg_bits + chunk_bytes * 8 - 1) / (chunk_bytes * 8)) : 1;
    std::vector<Md2JpegState> entry(nch), ex(nch);
    std::vector<int> cnt(nch);
    std::vector<Md2JpegDc> dc(nch);
    auto end_of = [&](int c) { unsigned e = (unsigned)(c + 1) * chunk_bytes * 8; return e < seg_bits ? e : seg_bits; };
    auto run = [&](int c) {
      cnt[c] = 0; dc[c] = {0, 0, 0};
      ex[c] = md2_jpeg_run_chunk(b, im, entry[c], end_of(c), &cnt[c], &dc[c], nullptr, 0, 0, seg_bits, nullptr);
    };
    for (int c = 0; c < nch; ++c) { entry[c] = {c ? (unsigned)c * chunk_bytes * 8 : 0u, 0, 0}; run(c); }
    for (;;) {                            // every chunk from its predecessor's previous exit, all at once
      std::vector<Md2JpegState> prev = ex;
      bool changed = false;
      for (int c = 1; c < nch; ++c) {
        const Md2JpegState in = prev[c - 1];
        if (in.pos != entry[c].pos || in.blk != entry[c].blk || in.z != entry[c].z) { entry[c] = in; run(c); changed = true; }
      }
      ++rounds;
      if (!changed) break;
    }
    const int first_mcu = s * per, n_mcu = per < mcus - first_mcu ? per : mcus - first_mcu;
    int before = 0;
    Md2JpegDc run_dc = {0, 0, 0};
    for (int c = 0; c < nch; ++c) {
      Md2JpegDc d = run_dc;
      int n = 0;
      md2_jpeg_run_chunk(b, im, entry[c], end_of(c), &n, &d, coefs.data(), (long long)first_mcu * bpm + before,
                         n_mcu * bpm - before, seg_bits, &flags);
      before += cnt[c];
      run_dc.y += dc[c].y; run_dc.cb += dc[c].cb; run_dc.cr += dc[c].cr;
    }
  }
  const int lw = mx * 8 * j->h_samp, lh = my * 8 * j->v_samp, cw8 = mx * 8, ch8 = my * 8;
  std::vector<unsigned char> planes((size_t)nblk * 64);
  for (long long g = 0; g < nblk; ++g) {
    const int mcu = (int)(g / bpm), k = (int)(g % bpm), mr = mcu / mx, mc = mcu % mx;
    int comp, stride, by, bx;
    unsigned char* base = planes.data();
    if (k < luma) { comp = 0; stride = lw; by = mr * j->v_samp + k / j->h_samp; bx = mc * j->h_samp + k % j->h_samp; }
    else { comp = k - luma + 1; base += (size_t)lw * lh + (size_t)(comp - 1) * cw8 * ch8; stride = cw8; by = mr; bx = mc; }
    md2_jpeg_idct_islow(&coefs[g * 64], tab->quant[j->quant_table[comp]], base + (size_t)by * 8 * stride + bx * 8, stride);
  }
  const unsigned char* Y = planes.data();
  const unsigned char* Cb = Y + (size_t)lw * lh;
  const unsigned char* Cr = Cb + (size_t)cw8 * ch8;
  const int ch = md2_jpeg_comp_size(j->height, 1, j->v_samp), cw = md2_jpeg_comp_size(j->width, 1, j->h_samp);
  for (int y = 0; y < j->height; ++y)
    for (int x = 0; x < j->width; ++x)
      md2_jpeg_ycc_rgb(Y[(size_t)y * lw + x], md2_jpeg_chroma(Cb, cw8, ch, cw, j->h_samp, j->v_samp, y, x),
                       md2_jpeg_chroma(Cr, cw8, ch, cw, j->h_samp, j->v_samp, y, x), out + ((size_t)y * j->width + x) * 3);
  if (coefs_out) memcpy(coefs_out, coefs.data(), coefs.size() * 2);
  if (rounds_out) *rounds_out = rounds;
  return (int)flags;
}

#ifdef MD2_JPEG_HOST_MAIN
// md2_jpeg_host <packed buffer file> <chunk bytes>: decodes the one image whose md2_jpeg_job is at offset 0 of the
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
  md2_jpeg_job j;
  memcpy(&j, buf, sizeof(j));
  unsigned char* out = (unsigned char*)malloc((size_t)j.height * j.width * 3);
  const int st = decode_host(buf, &j, atoi(argv[2]), out, nullptr, nullptr);
  printf("%d\n", st);
  free(out);
  free(buf);
  return 0;
}
#endif
