// md2_jpeg.h - the per-symbol, per-block and per-pixel arithmetic of md2_jpeg_decode, shared by the CUDA kernels and a
// g++ build (tests/test_jpeg_decode.py compiles it on the host and holds it to oracle/jpeg_decode.py and Pillow).
//
// Everything here is libjpeg-turbo's integer arithmetic for baseline streams, as Pillow runs it:
//   jdhuff.c     - the lookahead / maxcode Huffman decode, HUFF_EXTEND, the fake zero symbol after 17 bits of a bad
//                  code, and zero bits past the end of a segment (fill_bit_buffer at a marker);
//   jidctint.c   - jpeg_idct_islow with the range_limit[x & RANGE_MASK] table of prepare_range_limit_table;
//   jdsample.c   - h2v1 / h2v2 fancy up-sampling (edge samples repeated, as its SIMD form does; jdmainct.c's context
//                  rows repeat the first and last real row), plain replication for components <= 2 samples wide;
//   jdcolor.c    - ycc_rgb_convert's tables.
//
// Entropy decoding is split into chunks of a segment (a restart interval).  md2_jpeg_run_chunk decodes from an entry
// state (bit position, block of the MCU, zig-zag index) to the first symbol that starts at or after the chunk's end and
// returns that exit state; in count mode it also sums the DC differences and the blocks whose DC symbol lies in the
// chunk, in write mode it writes those blocks' coefficients.  A chunk whose entry is its predecessor's exit decodes
// exactly what the serial decoder decodes there, which is what the self-synchronising search in md2_jpeg.cu finds.
#ifndef MD2_JPEG_H_
#define MD2_JPEG_H_

#include <stdint.h>

#include "../../include/md2_loss.h"

#ifdef __CUDACC__
#define MD2_JHD __host__ __device__ __forceinline__
#else
#define MD2_JHD inline
#endif

// jpeg_natural_order with jdhuff.c's 16 extra entries: a corrupt run past 63 writes coefficient 63
#define MD2_JPEG_NATURAL_ORDER                                                                                         \
  {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13,        \
   6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31,        \
   39, 46, 53, 60, 61, 54, 47, 55, 62, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63}
#ifdef __CUDACC__
__constant__ unsigned char md2_jpeg_natural_dev[80] = MD2_JPEG_NATURAL_ORDER;
#endif
static const unsigned char md2_jpeg_natural_host[80] = MD2_JPEG_NATURAL_ORDER;

MD2_JHD int md2_jpeg_natural(int k) {
#ifdef __CUDA_ARCH__
  return md2_jpeg_natural_dev[k];
#else
  return md2_jpeg_natural_host[k];
#endif
}

// ------------------------------------------------------------------ bit reader
// Bits of one segment, MSB first; bytes at or past `n` read as zeros.  buf holds nb valid bits, left-aligned.
struct Md2JpegBits {
  const unsigned char* d;
  unsigned n;
  unsigned bp;
  int nb;
  unsigned long long buf;
};

MD2_JHD void md2_jpeg_fill(Md2JpegBits& b) {
  while (b.nb <= 56) {
    const unsigned long long v = b.bp < b.n ? b.d[b.bp] : 0u;
    b.buf |= v << (56 - b.nb);
    ++b.bp;
    b.nb += 8;
  }
}

MD2_JHD void md2_jpeg_seek(Md2JpegBits& b, unsigned pos) {
  b.bp = pos >> 3;
  b.nb = 0;
  b.buf = 0;
  md2_jpeg_fill(b);
  b.buf <<= (pos & 7);
  b.nb -= (int)(pos & 7);
}

MD2_JHD unsigned md2_jpeg_pos(const Md2JpegBits& b) { return b.bp * 8u - (unsigned)b.nb; }

// n <= 16 bits; the caller has filled the buffer (nb >= 33 holds a code of up to 17 bits and then 16 more bits)
MD2_JHD unsigned md2_jpeg_get(Md2JpegBits& b, int n) {
  if (n == 0) return 0;
  const unsigned v = (unsigned)(b.buf >> (64 - n));
  b.buf <<= n;
  b.nb -= n;
  return v;
}

// HUFF_DECODE / jpeg_huff_decode.  *bad is set for a code no table holds (17 bits consumed, symbol 0).
MD2_JHD int md2_jpeg_huff_decode(Md2JpegBits& b, const md2_jpeg_huff& t, bool* bad) {
  md2_jpeg_fill(b);
  const unsigned look = t.look[(unsigned)(b.buf >> 56)];
  const int l8 = (int)(look >> 8);
  if (l8 != 0) {
    const int l = l8 > 8 ? 8 : l8;
    b.buf <<= l;
    b.nb -= l;
    return (int)(look & 0xFFu);
  }
  for (int l = 9; l <= 16; ++l) {
    const int code = (int)(b.buf >> (64 - l));
    if (code <= t.maxcode[l]) {
      b.buf <<= l;
      b.nb -= l;
      return t.huffval[(code + t.valoffset[l]) & 0xFF];
    }
  }
  b.buf <<= 17;
  b.nb -= 17;
  *bad = true;
  return 0;
}

MD2_JHD int md2_jpeg_extend(unsigned x, int s) {  // HUFF_EXTEND
  return s == 0 ? 0 : ((int)x < (1 << (s - 1)) ? (int)x + (int)(~0u << s) + 1 : (int)x);
}

// ------------------------------------------------------------------ chunk decode
struct Md2JpegState {
  unsigned pos;   // bit position in the segment
  int blk;        // block of the MCU the next symbol belongs to
  int z;          // zig-zag index it decodes: 0 the DC, 1..63 an AC
};

struct Md2JpegImage {   // what the chunk decode needs of an image
  const md2_jpeg_tables* tab;
  int luma_blocks;      // h_samp * v_samp
  unsigned tables;      // bit c: the DC table of component c, bit 3 + c: its AC table
};

struct Md2JpegDc {      // per-component DC sums (kept in registers: no indexed arrays)
  int y, cb, cr;
};

MD2_JHD int md2_jpeg_dc_add(Md2JpegDc& s, int c, int d) {   // last_dc_val += d, wrapping as int does
  const unsigned u = (unsigned)d;
  if (c == 0) return s.y = (int)((unsigned)s.y + u);
  if (c == 1) return s.cb = (int)((unsigned)s.cb + u);
  return s.cr = (int)((unsigned)s.cr + u);
}

MD2_JHD int md2_jpeg_comp(const Md2JpegImage& im, int blk) {
  return blk < im.luma_blocks ? 0 : blk - im.luma_blocks + 1;
}

// Decodes one symbol at state s (DC or AC per s.z), advancing s.  Returns the DC difference for a DC symbol (z was 0)
// and writes the AC coefficient (natural order) into blkout when it is non-null.
MD2_JHD int md2_jpeg_step(Md2JpegBits& b, const Md2JpegImage& im, Md2JpegState& s, short* blkout, unsigned* flags) {
  const int c = md2_jpeg_comp(im, s.blk);
  bool bad = false;
  int dc = 0;
  if (s.z == 0) {
    const int t = md2_jpeg_huff_decode(b, im.tab->dc[(im.tables >> c) & 1u], &bad) & 15;
    dc = md2_jpeg_extend(md2_jpeg_get(b, t), t);
    s.z = 1;
  } else {
    const int sym = md2_jpeg_huff_decode(b, im.tab->ac[(im.tables >> (3 + c)) & 1u], &bad);
    const int r = sym >> 4, sz = sym & 15;
    if (sz) {
      s.z += r;
      if (s.z > 63) *flags |= MD2_JPEG_BAD_INDEX;
      const int v = md2_jpeg_extend(md2_jpeg_get(b, sz), sz);
      if (blkout) blkout[md2_jpeg_natural(s.z)] = (short)v;
      s.z += 1;
    } else if (r == 15) {
      s.z += 16;
    } else {
      s.z = 64;
    }
  }
  if (bad) *flags |= MD2_JPEG_BAD_CODE;
  md2_jpeg_fill(b);
  return dc;
}

MD2_JHD void md2_jpeg_end_block(Md2JpegState& s, int blocks_per_mcu) {
  if (s.z >= 64) {
    s.z = 0;
    s.blk = s.blk + 1 == blocks_per_mcu ? 0 : s.blk + 1;
  }
}

// Count mode (coefs == null): from `s` decode every symbol starting before bit `end`; returns the exit state, and adds
// to *n_blocks and dc_sum[c] the blocks whose DC symbol lies in the chunk and their DC differences.
// Write mode: the same walk, but the rest of a block begun before the chunk is skipped and every block whose DC lies in
// the chunk is decoded to its end and written, DC value = dc_run[c] after adding its difference (int wraps as
// last_dc_val does; the int16 store is (JCOEF)), as block first_block + i of `coefs` (natural order, 64 shorts), for
// i < max_blocks only; the segment's last chunk (end == seg_bits) flags MD2_JPEG_EXHAUSTED when the segment's
// blocks run out first.
MD2_JHD Md2JpegState md2_jpeg_run_chunk(Md2JpegBits& b, const Md2JpegImage& im, Md2JpegState s, unsigned end,
                                        int* n_blocks, Md2JpegDc* dc_sum, short* coefs, long long first_block,
                                        int max_blocks, unsigned seg_bits, unsigned* flags) {
  const int bpm = im.luma_blocks + 2;
  md2_jpeg_seek(b, s.pos);
  if (!coefs) {
    unsigned dummy = 0;
    while (md2_jpeg_pos(b) < end) {
      if (s.z == 0) ++*n_blocks;
      const int c = md2_jpeg_comp(im, s.blk);
      const int d = md2_jpeg_step(b, im, s, nullptr, &dummy);
      if (s.z == 1) md2_jpeg_dc_add(*dc_sum, c, d);
      md2_jpeg_end_block(s, bpm);
    }
    s.pos = md2_jpeg_pos(b);
    return s;
  }
  // one step call site: the tail of a block its predecessor writes is skipped (blk == null), then blocks are written
  short* blk = nullptr;
  int i = 0;
  for (;;) {
    if (s.z == 0) {
      if (md2_jpeg_pos(b) >= end || i >= max_blocks) break;
      blk = coefs + (first_block + i) * 64;
      for (int k = 0; k < 16; ++k) reinterpret_cast<unsigned long long*>(blk)[k] = 0ull;
    } else if (!blk && md2_jpeg_pos(b) >= end) {
      break;
    }
    const int c = md2_jpeg_comp(im, s.blk);
    const unsigned keep = *flags;
    const int d = md2_jpeg_step(b, im, s, blk, flags);
    if (!blk) {
      *flags = keep;                                   // the predecessor reports that block
      md2_jpeg_end_block(s, bpm);
      continue;
    }
    if (s.z == 1) blk[0] = (short)md2_jpeg_dc_add(*dc_sum, c, d);
    if (s.z >= 64) {
      if (md2_jpeg_pos(b) > seg_bits) *flags |= MD2_JPEG_EXHAUSTED;
      ++i;
    }
    md2_jpeg_end_block(s, bpm);
  }
  if (end == seg_bits && i < max_blocks) *flags |= MD2_JPEG_EXHAUSTED;   // the segment's last chunk: MCUs missing
  *n_blocks = i;
  s.pos = md2_jpeg_pos(b);
  return s;
}

// ------------------------------------------------------------------ IDCT
MD2_JHD int md2_jpeg_range_limit(int x) {   // idct_table[x & RANGE_MASK] (prepare_range_limit_table, 8-bit samples)
  x &= 1023;
  return x < 128 ? x + 128 : (x < 512 ? 255 : (x < 896 ? 0 : x - 896));
}

#define MD2_JPEG_IDCT_1D(c0, c1, c2, c3, c4, c5, c6, c7, o0, o1, o2, o3, o4, o5, o6, o7, SH)                            \
  do {                                                                                                                 \
    const int z1_ = ((c2) + (c6)) * 4433;                                                                              \
    const int t2_ = z1_ + (c6) * -15137, t3_ = z1_ + (c2) * 6270;                                                      \
    const int t0_ = ((c0) + (c4)) * 8192, t1_ = ((c0) - (c4)) * 8192;                                                  \
    const int t10 = t0_ + t3_, t13 = t0_ - t3_, t11 = t1_ + t2_, t12 = t1_ - t2_;                                      \
    int a0 = (c7), a1 = (c5), a2 = (c3), a3 = (c1);                                                                    \
    int y1 = a0 + a3, y2 = a1 + a2, y3 = a0 + a2, y4 = a1 + a3;                                                        \
    const int y5 = (y3 + y4) * 9633;                                                                                   \
    a0 *= 2446; a1 *= 16819; a2 *= 25172; a3 *= 12299;                                                                 \
    y1 *= -7373; y2 *= -20995; y3 *= -16069; y4 *= -3196;                                                              \
    y3 += y5; y4 += y5;                                                                                                \
    a0 += y1 + y3; a1 += y2 + y4; a2 += y2 + y3; a3 += y1 + y4;                                                        \
    const int r_ = 1 << ((SH) - 1);                                                                                    \
    o0 = (t10 + a3 + r_) >> (SH); o7 = (t10 - a3 + r_) >> (SH);                                                        \
    o1 = (t11 + a2 + r_) >> (SH); o6 = (t11 - a2 + r_) >> (SH);                                                        \
    o2 = (t12 + a1 + r_) >> (SH); o5 = (t12 - a1 + r_) >> (SH);                                                        \
    o3 = (t13 + a0 + r_) >> (SH); o4 = (t13 - a0 + r_) >> (SH);                                                        \
  } while (0)

// jpeg_idct_islow of one natural-order block with its natural-order quant table into 8 rows of `out` (row stride
// `stride`).  The all-zero-AC shortcuts of jidctint.c give the values the full formulas give, so they are not taken.
MD2_JHD void md2_jpeg_idct_islow(const short* coef, const unsigned short* q, unsigned char* out, int stride) {
  int ws[64];
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    int v[8];
#pragma unroll
    for (int r = 0; r < 8; ++r) v[r] = (int)coef[r * 8 + c] * (int)(short)q[r * 8 + c];   // ISLOW_MULT_TYPE
    MD2_JPEG_IDCT_1D(v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7], ws[c], ws[8 + c], ws[16 + c], ws[24 + c],
                     ws[32 + c], ws[40 + c], ws[48 + c], ws[56 + c], 13 - 2);
  }
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    const int* w = ws + r * 8;
    int o[8];
    MD2_JPEG_IDCT_1D(w[0], w[1], w[2], w[3], w[4], w[5], w[6], w[7], o[0], o[1], o[2], o[3], o[4], o[5], o[6], o[7],
                     13 + 2 + 3);
#pragma unroll
    for (int k = 0; k < 8; ++k) out[r * stride + k] = (unsigned char)md2_jpeg_range_limit(o[k]);
  }
}

// ------------------------------------------------------------------ up-sampling and colour
MD2_JHD int md2_jpeg_clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// The up-sampled chroma sample at output (y, x) of a (ch, cw) component plane (row stride `stride`) for luma
// sampling (hs, vs): 1x1 the sample itself, else h2v1 / h2v2 fancy up-sampling, or replication when cw <= 2.
MD2_JHD int md2_jpeg_chroma(const unsigned char* p, int stride, int ch, int cw, int hs, int vs, int y, int x) {
  if (hs == 1) return p[(long long)y * stride + x];
  const int j = x >> 1;
  const int i = vs == 2 ? y >> 1 : y;
  if (cw <= 2) return p[(long long)i * stride + j];
  const int jn = md2_jpeg_clampi((x & 1) ? j + 1 : j - 1, 0, cw - 1);
  const unsigned char* row = p + (long long)i * stride;
  if (vs == 1) {
    const int a = 3 * row[j];
    return (x & 1) ? (a + row[jn] + 2) >> 2 : (a + row[jn] + 1) >> 2;
  }
  const int in = md2_jpeg_clampi((y & 1) ? i + 1 : i - 1, 0, ch - 1);
  const unsigned char* other = p + (long long)in * stride;
  const int cs = 3 * row[j] + other[j];
  const int cn = 3 * row[jn] + other[jn];
  return (x & 1) ? (3 * cs + cn + 7) >> 4 : (3 * cs + cn + 8) >> 4;
}

// ycc_rgb_convert (build_ycc_rgb_table: FIX(1.40200) = 91881, FIX(1.77200) = 116130, FIX(0.71414) = 46802,
// FIX(0.34414) = 22554, SCALEBITS 16) with the sample range limit
MD2_JHD void md2_jpeg_ycc_rgb(int y, int cb, int cr, unsigned char* rgb) {
  const int xb = cb - 128, xr = cr - 128;
  const int r = y + ((91881 * xr + 32768) >> 16);
  const int g = y + ((-22554 * xb + 32768 + -46802 * xr) >> 16);
  const int b = y + ((116130 * xb + 32768) >> 16);
  rgb[0] = (unsigned char)md2_jpeg_clampi(r, 0, 255);
  rgb[1] = (unsigned char)md2_jpeg_clampi(g, 0, 255);
  rgb[2] = (unsigned char)md2_jpeg_clampi(b, 0, 255);
}

// jdiv_round_up(image size * sampling, max sampling)
MD2_JHD int md2_jpeg_comp_size(int n, int samp, int max_samp) { return (n * samp + max_samp - 1) / max_samp; }

#endif  // MD2_JPEG_H_
