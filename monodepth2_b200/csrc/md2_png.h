// md2_png.h - the per-bit, per-symbol, per-block and per-row arithmetic of md2_png_decode, shared by the CUDA kernels
// and a g++ build (tests/test_png_decode.py compiles it on the host and holds it to oracle/png_decode.py and Pillow).
//
// Inflate follows zlib's inflate.c / inftrees.c, as Pillow's ZipDecode runs it:
//   - a code-length code must be complete; a literal/length or distance code must not be over-subscribed and may be
//     incomplete only when its longest code is one bit; a distance code may be empty; symbol 256 must have a code;
//   - HLIT > 29, HDIST > 29, BTYPE 3, a repeat with nothing before it or past the last length, a stored block whose
//     NLEN is not ~LEN, literal/length 286-287 and distance 30-31 (fixed code) are errors;
//   - a distance longer than the output so far is an error.
// Pillow asks zlib for exactly height * (3 * width + 1) bytes.  zlib stops at the first symbol that would write past
// them, so whatever follows that symbol is never looked at: more data, a bad code, a missing final block, a wrong
// Adler-32.  Symbols that write nothing (an end-of-block code, the next block's header) are still decoded, so an
// error there counts when the output is exactly complete, and after the final block the Adler-32 trailer is checked
// when its four bytes are there.  A final block that ends early is zlib's stream end: Pillow checks the Adler-32 over
// the shorter data and keeps the image, the missing rows zero, when that data is a positive whole number of rows.
// Any other early end (mid-row, no row at all, no trailer, no final block) is the "truncated" error.
//
// md2_png_block decodes one block from a bit position into a uint32 output where a byte that copies from before the
// block's first byte is a marker (256 + its source position), which md2_png.cu resolves once every block is written.
#ifndef MD2_PNG_H_
#define MD2_PNG_H_

#include <stdint.h>

#include "../../include/md2_loss.h"

#ifdef __CUDACC__
#define MD2_PHD __host__ __device__ __forceinline__
#else
#define MD2_PHD inline
#endif

#define MD2_PNG_CL_ORDER {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15}
#ifdef __CUDACC__
__constant__ unsigned char md2_png_cl_order_dev[19] = MD2_PNG_CL_ORDER;
#endif
static const unsigned char md2_png_cl_order_host[19] = MD2_PNG_CL_ORDER;

MD2_PHD int md2_png_cl_order(int i) {
#ifdef __CUDA_ARCH__
  return md2_png_cl_order_dev[i];
#else
  return md2_png_cl_order_host[i];
#endif
}

// ------------------------------------------------------------------ bit reader
// Bits of one stream, LSB first; bytes at or past the stream's end read as zeros.  The stream starts 4-byte aligned
// and its last word lies inside the caller's buffer (md2_png_decode checks both); bytes of that word past the end are
// masked off.
struct Md2PngBits {
  const uint32_t* w;
  uint32_t nw;          // words holding the stream's bytes
  uint32_t last_mask;   // valid bits of word nw - 1
  uint32_t len_bits;    // 8 * stream bytes
  uint32_t next;        // next word to load
  int cnt;              // valid bits in buf
  uint64_t buf;
};

MD2_PHD void md2_png_bits_init(Md2PngBits& b, const unsigned char* d, uint32_t n) {
  b.w = reinterpret_cast<const uint32_t*>(d);
  b.nw = (n + 3) >> 2;
  b.last_mask = (n & 3) ? (1u << (8 * (n & 3))) - 1u : 0xFFFFFFFFu;
  b.len_bits = n * 8u;
  b.next = 0;
  b.cnt = 0;
  b.buf = 0;
}

MD2_PHD uint32_t md2_png_word(const Md2PngBits& b, uint32_t k) {
  if (k >= b.nw) return 0u;
  const uint32_t v = b.w[k];
  return k + 1 == b.nw ? v & b.last_mask : v;
}

MD2_PHD unsigned md2_png_byte(const Md2PngBits& b, uint32_t k) { return (md2_png_word(b, k >> 2) >> (8 * (k & 3))) & 0xFFu; }

MD2_PHD void md2_png_refill(Md2PngBits& b) {          // leaves at least 33 bits
  if (b.cnt <= 32) {
    b.buf |= (uint64_t)md2_png_word(b, b.next) << b.cnt;
    ++b.next;
    b.cnt += 32;
  }
}

MD2_PHD void md2_png_seek(Md2PngBits& b, uint32_t pos) {
  b.next = pos >> 5;
  b.buf = md2_png_word(b, b.next) >> (pos & 31);
  b.cnt = 32 - (int)(pos & 31);
  ++b.next;
  md2_png_refill(b);
}

MD2_PHD uint32_t md2_png_pos(const Md2PngBits& b) { return b.next * 32u - (uint32_t)b.cnt; }

MD2_PHD uint32_t md2_png_get(Md2PngBits& b, int n) {  // n <= 32, cnt >= n
  const uint32_t v = (uint32_t)(b.buf & ((1ull << n) - 1ull));
  b.buf >>= n;
  b.cnt -= n;
  return v;
}

// ------------------------------------------------------------------ Huffman codes
// A canonical code: a lookup table of 2^lutbits entries (length << 9 | symbol for codes of at most lutbits bits, 0
// for the rest), the count of codes per length and the symbols in code order for the longer ones.
struct Md2PngHuff {
  uint16_t lut[512];          // literal/length, 9 bits
  uint16_t dlut[256];         // distance, 8 bits (the code-length code while the header is read, 7 bits)
  uint16_t lcount[16], dcount[16];
  uint16_t lsym[288];
  uint16_t dsym[32];
  uint16_t offs[16];
  uint8_t lens[340];          // the code lengths of both codes, then (from 320) the code-length code's
};

MD2_PHD uint32_t md2_png_reverse(uint32_t code, int len) {
  uint32_t r = 0;
  for (int i = 0; i < len; ++i) r |= ((code >> i) & 1u) << (len - 1 - i);
  return r;
}

// inflate_table's rules: returns false for an over-subscribed code, for an incomplete one when `complete_only` or its
// longest code has more than one bit, and for an empty one unless `empty_ok`.
MD2_PHD bool md2_png_build(const uint8_t* lens, int n, uint16_t* count, uint16_t* sym, uint16_t* offs, uint16_t* lut,
                           int lutbits, bool complete_only, bool empty_ok) {
  for (int l = 0; l < 16; ++l) count[l] = 0;
  for (int s = 0; s < n; ++s) ++count[lens[s]];
  int max = 0;
  for (int l = 1; l < 16; ++l)
    if (count[l]) max = l;
  if (max == 0) {
    if (!empty_ok) return false;
  } else {
    int left = 1;
    for (int l = 1; l < 16; ++l) {
      left = (left << 1) - count[l];
      if (left < 0) return false;
    }
    if (left > 0 && (complete_only || max != 1)) return false;
  }
  offs[1] = 0;
  for (int l = 1; l < 15; ++l) offs[l + 1] = offs[l] + count[l];
  for (int s = 0; s < n; ++s)
    if (lens[s]) sym[offs[lens[s]]++] = (uint16_t)s;
  const int size = 1 << lutbits;
  for (int i = 0; i < size; ++i) lut[i] = 0;
  uint32_t code = 0;
  int k = 0;
  for (int l = 1; l <= lutbits; ++l) {
    for (int c = 0; c < count[l]; ++c, ++k, ++code) {
      const uint16_t e = (uint16_t)(l << 9 | sym[k]);
      for (uint32_t i = md2_png_reverse(code, l); i < (uint32_t)size; i += 1u << l) lut[i] = e;
    }
    code <<= 1;
  }
  return true;
}

// One symbol (the caller has refilled: at least 15 bits), -1 for a code the table does not hold.
MD2_PHD int md2_png_decode_sym(Md2PngBits& b, const uint16_t* lut, int lutbits, const uint16_t* count,
                               const uint16_t* sym) {
  const uint32_t e = lut[b.buf & ((1u << lutbits) - 1u)];
  if (e) {
    b.buf >>= (e >> 9);
    b.cnt -= (int)(e >> 9);
    return (int)(e & 511u);
  }
  uint64_t v = b.buf;
  int code = 0, first = 0, index = 0;
  for (int l = 1; l < 16; ++l) {
    code |= (int)(v & 1u);
    v >>= 1;
    const int c = count[l];
    if (code - first < c) {
      b.buf >>= l;
      b.cnt -= l;
      return sym[index + code - first];
    }
    index += c;
    first = (first + c) << 1;
    code <<= 1;
  }
  return -1;
}

MD2_PHD void md2_png_fixed(Md2PngHuff& h) {
  for (int s = 0; s < 288; ++s) h.lens[s] = s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8;
  md2_png_build(h.lens, 288, h.lcount, h.lsym, h.offs, h.lut, 9, true, false);
  for (int s = 0; s < 32; ++s) h.lens[s] = 5;
  md2_png_build(h.lens, 32, h.dcount, h.dsym, h.offs, h.dlut, 8, true, false);
}

// A dynamic block's header, from after BTYPE: builds both codes in h.  Returns 0 or MD2_PNG_BAD_CODE /
// MD2_PNG_EXHAUSTED.
MD2_PHD unsigned md2_png_dynamic(Md2PngBits& b, Md2PngHuff& h) {
  md2_png_refill(b);
  const int nlen = (int)md2_png_get(b, 5) + 257, ndist = (int)md2_png_get(b, 5) + 1, ncl = (int)md2_png_get(b, 4) + 4;
  if (nlen > 286 || ndist > 30) return MD2_PNG_BAD_CODE;
  uint8_t* cl = h.lens + 320;
  for (int i = 0; i < 19; ++i) cl[i] = 0;
  for (int i = 0; i < ncl; ++i) {
    md2_png_refill(b);
    cl[md2_png_cl_order(i)] = (uint8_t)md2_png_get(b, 3);
  }
  if (md2_png_pos(b) > b.len_bits) return MD2_PNG_EXHAUSTED;
  if (!md2_png_build(cl, 19, h.dcount, h.dsym, h.offs, h.dlut, 7, true, false)) return MD2_PNG_BAD_CODE;
  const int total = nlen + ndist;
  int i = 0;
  while (i < total) {
    md2_png_refill(b);
    const int s = md2_png_decode_sym(b, h.dlut, 7, h.dcount, h.dsym);
    if (s < 0) return MD2_PNG_BAD_CODE;
    int v = 0, rep = 1;
    if (s < 16) {
      v = s;
    } else if (s == 16) {
      if (i == 0) return MD2_PNG_BAD_CODE;
      v = h.lens[i - 1];
      rep = 3 + (int)md2_png_get(b, 2);
    } else if (s == 17) {
      rep = 3 + (int)md2_png_get(b, 3);
    } else {
      rep = 11 + (int)md2_png_get(b, 7);
    }
    if (md2_png_pos(b) > b.len_bits) return MD2_PNG_EXHAUSTED;
    if (i + rep > total) return MD2_PNG_BAD_CODE;
    for (int k = 0; k < rep; ++k) h.lens[i++] = (uint8_t)v;
  }
  if (h.lens[256] == 0) return MD2_PNG_BAD_CODE;
  if (!md2_png_build(h.lens, nlen, h.lcount, h.lsym, h.offs, h.lut, 9, false, false)) return MD2_PNG_BAD_CODE;
  if (!md2_png_build(h.lens + nlen, ndist, h.dcount, h.dsym, h.offs, h.dlut, 8, false, true)) return MD2_PNG_BAD_CODE;
  return 0u;
}

// Would md2_png_dynamic accept a dynamic header at bit `pos` (BFINAL, BTYPE = 2, HLIT and HDIST in range already
// seen)?  Exactly its rules, without building the codes: a 128-entry table of the code-length code in `cl_lut` and the
// Kraft sums of the two codes.  The block finder runs this at every bit position that gets this far.
MD2_PHD bool md2_png_header_plausible(Md2PngBits& b, uint32_t pos, uint8_t* cl_lut) {
  md2_png_seek(b, pos + 3);
  const int nlen = (int)md2_png_get(b, 5) + 257, ndist = (int)md2_png_get(b, 5) + 1, ncl = (int)md2_png_get(b, 4) + 4;
  uint64_t cl = 0;                                       // 3 bits per symbol
  int kraft = 0;
  for (int i = 0; i < ncl; ++i) {
    md2_png_refill(b);
    const uint32_t l = md2_png_get(b, 3);
    cl |= (uint64_t)l << (3 * md2_png_cl_order(i));
    if (l) kraft += 128 >> l;
  }
  if (kraft != 128 || md2_png_pos(b) > b.len_bits) return false;
  for (int i = 0; i < 128; ++i) cl_lut[i] = 0;
  uint32_t code = 0;
  for (int l = 1; l <= 7; ++l) {
    for (int s = 0; s < 19; ++s) {
      if ((int)((cl >> (3 * s)) & 7u) != l) continue;
      for (uint32_t i = md2_png_reverse(code, l); i < 128u; i += 1u << l) cl_lut[i] = (uint8_t)(l << 5 | s);
      ++code;
    }
    code <<= 1;
  }
  const int total = nlen + ndist;
  int lk = 0, dk = 0, lmax = 0, dmax = 0, prev = 0, i = 0;
  bool eob = false;
  while (i < total) {
    md2_png_refill(b);
    const uint32_t e = cl_lut[b.buf & 127u];
    b.buf >>= (e >> 5);
    b.cnt -= (int)(e >> 5);
    const int s = (int)(e & 31u);
    int v = 0, rep = 1;
    if (s < 16) {
      v = s;
    } else if (s == 16) {
      if (i == 0) return false;
      v = prev;
      rep = 3 + (int)md2_png_get(b, 2);
    } else if (s == 17) {
      rep = 3 + (int)md2_png_get(b, 3);
    } else {
      rep = 11 + (int)md2_png_get(b, 7);
    }
    if (i + rep > total || md2_png_pos(b) > b.len_bits) return false;
    if (v) {
      const int nl = i < nlen ? (i + rep < nlen ? rep : nlen - i) : 0;
      lk += nl << (15 - v);
      dk += (rep - nl) << (15 - v);
      if (nl && v > lmax) lmax = v;
      if (rep > nl && v > dmax) dmax = v;
      if (i <= 256 && 256 < i + rep) eob = true;
      if (lk > 32768 || dk > 32768) return false;
    }
    prev = v;
    i += rep;
  }
  return eob && (lk == 32768 || lmax == 1) && (dk == 32768 || dmax <= 1);
}

// ------------------------------------------------------------------ one block
struct Md2PngEnd {
  uint32_t end;         // bit position after the block (valid when flags == 0 and !stop)
  int out;              // bytes the block produced
  unsigned flags;       // MD2_PNG_BAD_CODE / DISTANCE / EXHAUSTED where decoding stopped on an error
  int final;            // BFINAL
  int stop;             // a symbol would have written at or past `limit`: zlib stops there
};

// Decodes the block at bit `pos` whose first byte is byte g of the inflated data.  With kWrite, bytes g.. go to
// out[g..] up to `limit` (a byte copied from before g is stored as 256 + its source position), and a distance past
// the data's start is an error; without, nothing is written and g should be 0.
template <bool kWrite>
MD2_PHD Md2PngEnd md2_png_block(Md2PngBits& b, Md2PngHuff& h, uint32_t pos, long long g, long long limit,
                                uint32_t* out) {
  Md2PngEnd r = {0u, 0, 0u, 0, 0};
  md2_png_seek(b, pos);
  r.final = (int)md2_png_get(b, 1);
  const uint32_t type = md2_png_get(b, 2);
  if (md2_png_pos(b) > b.len_bits) {
    r.flags = MD2_PNG_EXHAUSTED;
    return r;
  }
  long long o = 0;
  if (type == 0) {                                       // stored
    const uint32_t p = (md2_png_pos(b) + 7u) & ~7u;
    const uint32_t at = p >> 3;
    if (p + 32u > b.len_bits) {
      r.flags = MD2_PNG_EXHAUSTED;
      return r;
    }
    const uint32_t len = md2_png_byte(b, at) | md2_png_byte(b, at + 1) << 8;
    const uint32_t nlen = md2_png_byte(b, at + 2) | md2_png_byte(b, at + 3) << 8;
    if (len != (nlen ^ 0xFFFFu)) {
      r.flags = MD2_PNG_BAD_CODE;
      return r;
    }
    const uint32_t first = at + 4u, n_bytes = b.len_bits >> 3;
    for (uint32_t k = 0; k < len; ++k, ++o) {
      if (first + k >= n_bytes) {
        r.flags = MD2_PNG_EXHAUSTED;
        r.out = (int)o;
        return r;
      }
      if (g + o >= limit) {
        r.stop = 1;
        r.out = (int)o;
        return r;
      }
      if (kWrite) out[g + o] = md2_png_byte(b, first + k);
    }
    r.out = (int)o;
    r.end = (first + len) * 8u;
    return r;
  }
  if (type == 3) {
    r.flags = MD2_PNG_BAD_CODE;
    return r;
  }
  if (type == 1) {
    md2_png_fixed(h);
  } else {
    r.flags = md2_png_dynamic(b, h);
    if (r.flags) return r;
  }
  for (;;) {
    md2_png_refill(b);
    const int s = md2_png_decode_sym(b, h.lut, 9, h.lcount, h.lsym);
    if (md2_png_pos(b) > b.len_bits) {
      r.flags = MD2_PNG_EXHAUSTED;
      break;
    }
    if (s < 0 || s > 285) {
      r.flags = MD2_PNG_BAD_CODE;
      break;
    }
    if (s < 256) {
      if (g + o >= limit) {
        r.stop = 1;
        break;
      }
      if (kWrite) out[g + o] = (uint32_t)s;
      ++o;
      continue;
    }
    if (s == 256) {
      r.end = md2_png_pos(b);
      break;
    }
    int len;
    const int li = s - 257;
    if (li < 8) {
      len = li + 3;
    } else if (li == 28) {
      len = 258;
    } else {
      const int e = (li - 4) >> 2;
      len = ((((li - 8) & 3) + 4) << e) + 3 + (int)md2_png_get(b, e);
    }
    md2_png_refill(b);
    const int d = md2_png_decode_sym(b, h.dlut, 8, h.dcount, h.dsym);
    if (d < 0 || d > 29) {
      r.flags = md2_png_pos(b) > b.len_bits ? MD2_PNG_EXHAUSTED : MD2_PNG_BAD_CODE;
      break;
    }
    int dist;
    if (d < 4) {
      dist = d + 1;
    } else {
      const int e = (d >> 1) - 1;
      dist = ((2 + (d & 1)) << e) + 1 + (int)md2_png_get(b, e);
    }
    if (md2_png_pos(b) > b.len_bits) {
      r.flags = MD2_PNG_EXHAUSTED;
      break;
    }
    if (kWrite && dist > g + o) {
      r.flags = MD2_PNG_DISTANCE;
      break;
    }
    if (g + o >= limit) {
      r.stop = 1;
      break;
    }
    for (int k = 0; k < len; ++k) {
      const long long q = g + o + k;
      if (q >= limit) break;
      if (kWrite) {
        const long long src = q - dist;
        out[q] = src >= g ? out[src] : 256u + (uint32_t)src;
      }
    }
    o += len;
  }
  r.out = (int)o;
  return r;
}

// The status bits of a block decoded at byte g: an error counts when zlib would have reached it, that is before the
// output was complete, or exactly at its end for anything but running out of data.
MD2_PHD unsigned md2_png_block_status(const Md2PngEnd& e, long long g, long long limit) {
  const long long at = g + e.out;
  if (at > limit) return 0u;
  return at == limit ? e.flags & ~MD2_PNG_EXHAUSTED : e.flags;
}

// ------------------------------------------------------------------ Adler-32 and the row filters
#define MD2_PNG_ADLER_MOD 65521u

// Pixels [x0, x1) of row y (bpp 3): filtered bytes `raw` (after the filter byte), the unfiltered row above `prior`
// (null for row 0), writes the unfiltered bytes to `cur`.  left / upleft carry the pixel before x0 of this row and
// the row above (zeros at x0 = 0).
MD2_PHD void md2_png_unfilter_span(int f, const unsigned char* __restrict__ raw, const unsigned char* __restrict__ prior,
                                   unsigned char* __restrict__ cur, int x0, int x1, unsigned char left[3],
                                   unsigned char upleft[3]) {
#pragma unroll 4
  for (int x = x0; x < x1; ++x) {
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const int i = 3 * x + c;
      const int a = left[c], bb = prior ? prior[i] : 0, cc = upleft[c];
      int v = raw[i];
      if (f == 1) {
        v += a;
      } else if (f == 2) {
        v += bb;
      } else if (f == 3) {
        v += (a + bb) >> 1;
      } else if (f == 4) {
        const int p = a + bb - cc;
        const int pa = p > a ? p - a : a - p, pb = p > bb ? p - bb : bb - p, pc = p > cc ? p - cc : cc - p;
        v += (pa <= pb && pa <= pc) ? a : (pb <= pc ? bb : cc);
      }
      cur[i] = (unsigned char)v;
      left[c] = (unsigned char)v;
      upleft[c] = (unsigned char)bb;
    }
  }
}

#endif  // MD2_PNG_H_
