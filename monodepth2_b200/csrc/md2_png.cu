// md2_png.cu - PNG decoding on the GPU, byte for byte what Pillow gives (md2_png.h).
//
// A deflate stream is one serial dependency: where a block starts is known only once the block before it is decoded.
// One call decodes every image of a batch in six launches after a memset:
//   md2_png_find    - every bit position of every stream is tested as a block header: a dynamic header that zlib
//                     would accept (md2_png_header_plausible: ranges, a complete code-length code, code lengths that
//                     form valid codes with an end-of-block code), or a stored header whose LEN / NLEN agree.  Most
//                     positions fail within a few operations; the rest become candidates.
//   md2_png_count   - every candidate decodes its block to the end-of-block code (md2_png_block without writing):
//                     end position, output length, final flag, or where it failed.
//   md2_png_chain   - one CTA per image walks from bit 0 through the blocks, taking each block's end from its
//                     candidate record.  A block that starts where no candidate is (a fixed-Huffman block, or any
//                     header the finder passed over) is decoded here, serially, into its place.  The candidates on the
//                     walk get their output offsets; the rest were false positives and are ignored.
//   md2_png_write   - every candidate on the walk decodes again into its place.  A byte copied from before the block's
//                     first byte is stored as a marker (256 + its source position): that byte is not written yet.
//   md2_png_resolve - every marker follows its source (a source is always earlier, so the chain ends) to a byte; the
//                     Adler-32 sums of the inflated data as a parallel reduction.
//   md2_png_unfilter - one CTA per image undoes the row filters as a wavefront (row y runs 16 pixels behind row y - 1)
//                     straight into the HWC frame, and checks the Adler-32 trailer.
// Correctness never rests on speculation: a candidate's record is a function of its bit position alone, the chain
// follows only positions that the true decode reaches, and a position without a record is decoded where it is.  It may
// be slow, never wrong.  Grids and scratch depend only on the image count and the capacity (stream bytes, inflated
// bytes), so one CUDA graph serves every batch within it.  Malformed data only sets status bits: every read is bounded
// by its stream (zeros past the end), every write by the image's inflated size or its frame, and every loop by the
// stream's bits or the marker chain's strictly decreasing positions.  The kernels check every image against the
// buffers and the capacity again (job_fits), so a replayed graph fed a batch over its capacity skips that image and
// flags it instead of writing past the scratch.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/md2_loss.h"
#include "md2_png.h"

namespace {

constexpr int kFindThreads = 256;       // one stream byte (eight bit positions) per thread
constexpr int kDecThreads = 16;         // md2_png_count / md2_png_write: one candidate per thread, its codes in shared
constexpr int kDecCtas = 148 * 5;
constexpr int kChainThreads = 128;
constexpr int kResolveThreads = 256;
constexpr int kResolveCtas = 32;        // per image
constexpr int kUnfilterThreads = 512;   // rows per wavefront band
constexpr int kTile = 16;               // pixels a row advances per wavefront step

struct ImageState {
  unsigned long long s1, sq;            // Adler-32: sum of bytes, sum of position * byte (mod 65521 per CTA)
  long long produced;                   // inflated bytes the walk placed (at most the image's)
  int check;                            // 1: check the trailer over `produced` bytes; 2: and if it matches, the data
                                        // still ended before a whole row (Pillow's "truncated")
  unsigned trailer;
};
static_assert(sizeof(ImageState) == 32, "32 bytes per image");

struct Cand {
  uint32_t pos;
  int img;
  uint32_t end;
  int out;
  unsigned flags;
  int final_stop;                       // final | stop << 1
  long long g;                          // output offset on the walk, -1 off it
};
static_assert(sizeof(Cand) == 32, "32 bytes per candidate");

inline size_t align256(size_t n) { return (n + 255) / 256 * 256; }

struct Layout {
  size_t states, counter, cands, out32, raw8, total;
  long long cap;
};
inline Layout layout(int n_images, long long max_stream, long long max_raw) {
  Layout L;
  L.cap = max_stream / 32 + 256LL * n_images;
  L.states = 0;
  L.counter = align256(sizeof(ImageState) * (size_t)n_images);
  L.cands = L.counter + 256;
  L.out32 = L.cands + align256(sizeof(Cand) * (size_t)L.cap);
  L.raw8 = L.out32 + align256((size_t)max_raw * 4);
  L.total = L.raw8 + align256((size_t)max_raw);
  return L;
}

__device__ __forceinline__ long long raw_bytes(const md2_png_job& j) { return (long long)j.height * (3LL * j.width + 1); }

// The image lies inside the buffers and the capacity the call was sized for.  md2_png_decode checks this on the host;
// a replayed CUDA graph skips that check, so every kernel checks it again and skips the image (md2_png_chain flags it).
__device__ __forceinline__ bool job_fits(const md2_png_job& j, size_t data_bytes, size_t frames_bytes,
                                         long long max_stream, long long max_raw) {
  if (j.height < 1 || j.width < 1 || j.height > MD2_PNG_MAX_SIDE || j.width > MD2_PNG_MAX_SIDE || j.stream_bytes < 0 ||
      j.stream_bytes > (1 << 28) || j.stream_offset < 0 || (j.stream_offset & 3) || j.out_offset < 0 ||
      j.stream_index < 0 || j.raw_offset < 0)
    return false;
  return j.stream_index + j.stream_bytes <= max_stream && j.raw_offset + raw_bytes(j) <= max_raw &&
         (unsigned long long)(j.stream_offset + ((long long)j.stream_bytes + 3) / 4 * 4) <= data_bytes &&
         (unsigned long long)(j.out_offset + 3LL * j.height * j.width) <= frames_bytes;
}

__device__ __forceinline__ void bits_of(const unsigned char* data, const md2_png_job& j, Md2PngBits& b) {
  md2_png_bits_init(b, data + j.stream_offset, (uint32_t)j.stream_bytes);
}

__device__ __forceinline__ int image_of_byte(long long t, const md2_png_job* __restrict__ jobs, int n_images) {
  int lo = 0, hi = n_images - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (jobs[mid].stream_index <= t) lo = mid; else hi = mid - 1;
  }
  return lo;
}

__device__ __forceinline__ void add_candidate(Cand* cands, unsigned* counter, long long cap, uint32_t pos, int img) {
  const unsigned i = atomicAdd(counter, 1u);
  if (i < cap) {                         // past the capacity the walk decodes the block itself
    Cand c;
    c.pos = pos;
    c.img = img;
    c.end = 0;
    c.out = 0;
    c.flags = 0;
    c.final_stop = 0;
    c.g = -1;
    cands[i] = c;
  }
}

__global__ void __launch_bounds__(kFindThreads) md2_png_find(const unsigned char* __restrict__ data,
                                                             const md2_png_job* __restrict__ jobs, int n_images,
                                                             long long max_stream, Cand* cands, unsigned* counter,
                                                             long long cap, size_t data_bytes, size_t frames_bytes,
                                                             long long max_raw) {
  __shared__ uint8_t cl_lut[kFindThreads][128];
  const long long t = (long long)blockIdx.x * kFindThreads + threadIdx.x;
  if (t >= max_stream) return;
  const int img = image_of_byte(t, jobs, n_images);
  const md2_png_job& j = jobs[img];
  const long long local = t - j.stream_index;
  if (local < 0 || local >= j.stream_bytes || !job_fits(j, data_bytes, frames_bytes, max_stream, max_raw)) return;
  const uint32_t b = (uint32_t)local;
  Md2PngBits bits;
  bits_of(data, j, bits);
  const uint64_t lo = md2_png_word(bits, b >> 2) | (uint64_t)md2_png_word(bits, (b >> 2) + 1) << 32;
  const uint64_t hi = md2_png_word(bits, (b >> 2) + 2);
  const int sh = 8 * (b & 3);
  const uint64_t win = sh ? (lo >> sh) | (hi << (64 - sh)) : lo;      // the stream's bits from byte b on
  for (int k = 0; k < 8; ++k) {
    const uint64_t v = win >> k;
    const uint32_t type = (uint32_t)(v >> 1) & 3u;
    const uint32_t pos = b * 8u + (uint32_t)k;
    if (type == 2) {
      if (((v >> 3) & 31u) <= 29u && ((v >> 8) & 31u) <= 29u &&
          md2_png_header_plausible(bits, pos, cl_lut[threadIdx.x]))
        add_candidate(cands, counter, cap, pos, img);
    } else if (type == 0) {
      const int at = k <= 5 ? 8 : 16;                                  // LEN / NLEN at the next byte boundary
      const uint32_t len = (uint32_t)(win >> at) & 0xFFFFu, nlen = (uint32_t)(win >> (at + 16)) & 0xFFFFu;
      if (len == (nlen ^ 0xFFFFu)) add_candidate(cands, counter, cap, pos, img);
    }
  }
}

__global__ void __launch_bounds__(kDecThreads) md2_png_count(const unsigned char* __restrict__ data,
                                                             const md2_png_job* __restrict__ jobs, Cand* cands,
                                                             const unsigned* __restrict__ counter, long long cap) {
  __shared__ Md2PngHuff h[kDecThreads];
  const long long n = min((long long)*counter, cap);
  for (long long c = (long long)blockIdx.x * kDecThreads + threadIdx.x; c < n; c += (long long)gridDim.x * kDecThreads) {
    Cand k = cands[c];
    const md2_png_job& j = jobs[k.img];
    Md2PngBits bits;
    bits_of(data, j, bits);
    const Md2PngEnd e = md2_png_block<false>(bits, h[threadIdx.x], k.pos, 0, raw_bytes(j), nullptr);
    cands[c].end = e.end;
    cands[c].out = e.out;
    cands[c].flags = e.flags;
    cands[c].final_stop = e.final | e.stop << 1;
  }
}

__global__ void __launch_bounds__(kChainThreads) md2_png_chain(const unsigned char* __restrict__ data,
                                                               const md2_png_job* __restrict__ jobs, Cand* cands,
                                                               const unsigned* __restrict__ counter, long long cap,
                                                               uint32_t* out32, ImageState* states, unsigned* status,
                                                               size_t data_bytes, size_t frames_bytes,
                                                               long long max_stream, long long max_raw) {
  __shared__ Md2PngHuff h;
  __shared__ int found, done;
  __shared__ uint32_t pos;
  const int img = blockIdx.x;
  const md2_png_job& j = jobs[img];
  if (!job_fits(j, data_bytes, frames_bytes, max_stream, max_raw)) {
    if (threadIdx.x == 0) atomicOr(status + img, MD2_PNG_CAPACITY);
    return;
  }
  const long long limit = raw_bytes(j);
  const long long rowb = 3LL * j.width + 1;
  uint32_t* out = out32 + j.raw_offset;
  const long long n = min((long long)*counter, cap);
  long long g = 0;                                         // thread 0's
  unsigned st = 0;
  if (threadIdx.x == 0) pos = 0;
  for (;;) {
    if (threadIdx.x == 0) found = -1;
    __syncthreads();
    const uint32_t p = pos;
    for (long long c = threadIdx.x; c < n; c += kChainThreads)
      if (cands[c].pos == p && cands[c].img == img) found = (int)c;  // positions are unique per image
    __syncthreads();
    if (threadIdx.x == 0) {
      Md2PngEnd e;
      if (found >= 0) {
        Cand& k = cands[found];
        k.g = g;
        e.end = k.end;
        e.out = k.out;
        e.flags = k.flags;
        e.final = k.final_stop & 1;
        e.stop = k.final_stop >> 1;
      } else {
        Md2PngBits bits;
        bits_of(data, j, bits);
        e = md2_png_block<true>(bits, h, p, g, limit, out);
        st |= md2_png_block_status(e, g, limit);
      }
      const long long at = g + e.out;
      int last = e.flags || e.stop || e.final || at > limit;
      if (e.final && !e.flags && !e.stop && at <= limit) {
        // The trailer, big-endian, after the final block.  A stream that ends early with its trailer is zlib's
        // Z_STREAM_END: Pillow checks the Adler-32 over what came, keeps it when it is a positive whole number of
        // rows (the rest stays zero) and is "truncated" otherwise.  Without the trailer only a complete image stands.
        const uint32_t tb = (e.end + 7u) >> 3;
        if ((long long)tb + 4 <= j.stream_bytes) {
          Md2PngBits bits;
          bits_of(data, j, bits);
          states[img].check = at < limit && (at == 0 || at % rowb) ? 2 : 1;
          states[img].trailer = md2_png_byte(bits, tb) << 24 | md2_png_byte(bits, tb + 1) << 16 |
                                md2_png_byte(bits, tb + 2) << 8 | md2_png_byte(bits, tb + 3);
        } else if (at < limit) {
          st |= MD2_PNG_EXHAUSTED;
        }
      }
      g = at;
      pos = e.end;
      done = last;
    }
    __syncthreads();
    if (done) break;
  }
  if (threadIdx.x == 0) {
    states[img].produced = g < limit ? g : limit;
    if (st) atomicOr(status + img, st);
  }
}

__global__ void __launch_bounds__(kDecThreads) md2_png_write(const unsigned char* __restrict__ data,
                                                             const md2_png_job* __restrict__ jobs,
                                                             const Cand* __restrict__ cands,
                                                             const unsigned* __restrict__ counter, long long cap,
                                                             uint32_t* out32, unsigned* status) {
  __shared__ Md2PngHuff h[kDecThreads];
  const long long n = min((long long)*counter, cap);
  for (long long c = (long long)blockIdx.x * kDecThreads + threadIdx.x; c < n; c += (long long)gridDim.x * kDecThreads) {
    const Cand k = cands[c];
    if (k.g < 0) continue;
    const md2_png_job& j = jobs[k.img];
    const long long limit = raw_bytes(j);
    uint32_t* out = out32 + j.raw_offset;
    Md2PngBits bits;
    bits_of(data, j, bits);
    const Md2PngEnd e = md2_png_block<true>(bits, h[threadIdx.x], k.pos, k.g, limit, out);
    const unsigned st = md2_png_block_status(e, k.g, limit);
    if (st) atomicOr(status + k.img, st);
    if (e.flags)                                         // a distance error the count pass could not see: the walk
      for (long long q = k.g + e.out; q < k.g + k.out && q < limit; ++q) out[q] = 0;   // placed more bytes here
  }
}

__global__ void __launch_bounds__(kResolveThreads) md2_png_resolve(const md2_png_job* __restrict__ jobs,
                                                                   const uint32_t* __restrict__ out32,
                                                                   unsigned char* raw8, ImageState* states,
                                                                   size_t data_bytes, size_t frames_bytes,
                                                                   long long max_stream, long long max_raw) {
  const int img = blockIdx.y;
  const md2_png_job& j = jobs[img];
  if (!job_fits(j, data_bytes, frames_bytes, max_stream, max_raw)) return;
  const long long limit = raw_bytes(j);
  const long long produced = states[img].produced;
  const uint32_t* in = out32 + j.raw_offset;
  unsigned char* r8 = raw8 + j.raw_offset;
  unsigned long long s1 = 0, sq = 0;
  for (long long q = (long long)blockIdx.x * kResolveThreads + threadIdx.x; q < limit;
       q += (long long)gridDim.x * kResolveThreads) {
    uint32_t v = 0;
    if (q < produced) {
      v = in[q];
      long long cur = q;
      while (v >= 256u) {                                 // sources strictly decrease
        const long long src = (long long)(v - 256u);
        if (src >= cur) {
          v = 0;
          break;
        }
        cur = src;
        v = in[src];
      }
    }
    r8[q] = (unsigned char)v;
    s1 += v;
    sq += (unsigned long long)q * v;
  }
  s1 %= MD2_PNG_ADLER_MOD;
  sq %= MD2_PNG_ADLER_MOD;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s1 += __shfl_down_sync(0xFFFFFFFFu, s1, o);
    sq += __shfl_down_sync(0xFFFFFFFFu, sq, o);
  }
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(&states[img].s1, s1);
    atomicAdd(&states[img].sq, sq);
  }
}

__global__ void __launch_bounds__(kUnfilterThreads) md2_png_unfilter(const md2_png_job* __restrict__ jobs,
                                                                     const unsigned char* __restrict__ raw8,
                                                                     const ImageState* __restrict__ states,
                                                                     unsigned char* frames, unsigned* status,
                                                                     size_t data_bytes, size_t frames_bytes,
                                                                     long long max_stream, long long max_raw) {
  const int img = blockIdx.x;
  const md2_png_job& j = jobs[img];
  if (!job_fits(j, data_bytes, frames_bytes, max_stream, max_raw)) return;
  const int H = j.height, W = j.width;
  const long long rowb = 3LL * W + 1;
  const unsigned char* r8 = raw8 + j.raw_offset;
  unsigned char* out = frames + j.out_offset;
  if (threadIdx.x == 0 && states[img].check) {
    const unsigned long long M = MD2_PNG_ADLER_MOD, n = (unsigned long long)states[img].produced % M;
    const unsigned long long s1 = states[img].s1 % M, sq = states[img].sq % M;
    const unsigned a = (unsigned)((1 + s1) % M);
    const unsigned b = (unsigned)((n + n * s1 % M + M - sq) % M);   // sum over bytes of (n - i) * byte, plus n
    if ((b << 16 | a) != states[img].trailer)
      atomicOr(status + img, MD2_PNG_CHECKSUM);
    else if (states[img].check == 2)
      atomicOr(status + img, MD2_PNG_EXHAUSTED);
  }
  const int tiles = (W + kTile - 1) / kTile;
  for (int band = 0; band < H; band += kUnfilterThreads) {
    const int y = band + threadIdx.x;
    const bool active = y < H;
    int f = 0;
    if (active) {
      f = r8[y * rowb];
      if (f > 4) {
        atomicOr(status + img, MD2_PNG_BAD_FILTER);
        f = 0;
      }
    }
    unsigned char left[3] = {0, 0, 0}, upleft[3] = {0, 0, 0};
    const int rows = min(kUnfilterThreads, H - band);
    for (int s = 0; s < rows + tiles - 1; ++s) {
      const int k = s - (int)threadIdx.x;
      if (active && k >= 0 && k < tiles)
        md2_png_unfilter_span(f, r8 + y * rowb + 1, y ? out + (long long)(y - 1) * 3 * W : nullptr,
                         out + (long long)y * 3 * W, k * kTile, min(W, (k + 1) * kTile), left, upleft);
      __syncthreads();
    }
  }
}

}  // namespace

extern "C" {

int md2_png_decode_scratch_bytes(int n_images, long long max_stream_bytes, long long max_raw_bytes, size_t* bytes) {
  if (!bytes || n_images < 1 || max_stream_bytes < 1 || max_raw_bytes < 1) return MD2_ERR_INVALID_ARGUMENT;
  if (n_images > 65535 || max_stream_bytes > (1LL << 31) || max_raw_bytes > (1LL << 36)) return MD2_ERR_UNSUPPORTED;
  *bytes = layout(n_images, max_stream_bytes, max_raw_bytes).total;
  return MD2_OK;
}

int md2_png_decode(const unsigned char* data, size_t data_bytes, const md2_png_job* jobs, const md2_png_job* jobs_dev,
                   int n_images, unsigned char* frames, size_t frames_bytes, unsigned int* status,
                   long long max_stream_bytes, long long max_raw_bytes, void* scratch, size_t scratch_bytes,
                   void* stream) {
  if (!data || !jobs || !jobs_dev || !frames || !status || n_images < 1 || max_stream_bytes < 1 || max_raw_bytes < 1)
    return MD2_ERR_INVALID_ARGUMENT;
  if (n_images > 65535 || max_stream_bytes > (1LL << 31) || max_raw_bytes > (1LL << 36)) return MD2_ERR_UNSUPPORTED;
  long long streams = 0, raws = 0;
  for (int i = 0; i < n_images; ++i) {
    const md2_png_job& j = jobs[i];
    if (j.height < 1 || j.width < 1 || j.height > MD2_PNG_MAX_SIDE || j.width > MD2_PNG_MAX_SIDE ||
        j.stream_bytes < 0 || j.stream_bytes > (1 << 28))
      return MD2_ERR_INVALID_ARGUMENT;
    if (j.stream_index != streams || j.raw_offset != raws) return MD2_ERR_INVALID_ARGUMENT;   // running sums
    streams += j.stream_bytes;
    raws += (long long)j.height * (3LL * j.width + 1);
    auto inside = [&](long long off, long long n, long long align, size_t total) {
      return off >= 0 && off % align == 0 && (unsigned long long)off <= total && (unsigned long long)n <= total - off;
    };
    if (!inside(j.stream_offset, ((long long)j.stream_bytes + 3) / 4 * 4, 4, data_bytes) ||
        !inside(j.out_offset, 3LL * j.height * j.width, 1, frames_bytes))
      return MD2_ERR_INVALID_ARGUMENT;
  }
  if (streams > max_stream_bytes || raws > max_raw_bytes) return MD2_ERR_UNSUPPORTED;   // over the stated capacity
  const Layout L = layout(n_images, max_stream_bytes, max_raw_bytes);
  if (!scratch || scratch_bytes < L.total) return MD2_ERR_WORKSPACE_TOO_SMALL;
  cudaStream_t s = (cudaStream_t)stream;
  unsigned char* base = (unsigned char*)scratch;
  ImageState* states = (ImageState*)(base + L.states);
  unsigned* counter = (unsigned*)(base + L.counter);
  Cand* cands = (Cand*)(base + L.cands);
  uint32_t* out32 = (uint32_t*)(base + L.out32);
  unsigned char* raw8 = base + L.raw8;
  if (cudaMemsetAsync(base, 0, L.cands, s) != cudaSuccess) return MD2_ERR_CUDA;
  if (cudaMemsetAsync(status, 0, sizeof(unsigned) * n_images, s) != cudaSuccess) return MD2_ERR_CUDA;
  md2_png_find<<<(unsigned)((max_stream_bytes + kFindThreads - 1) / kFindThreads), kFindThreads, 0, s>>>(
      data, jobs_dev, n_images, max_stream_bytes, cands, counter, L.cap, data_bytes, frames_bytes, max_raw_bytes);
  md2_png_count<<<kDecCtas, kDecThreads, 0, s>>>(data, jobs_dev, cands, counter, L.cap);
  md2_png_chain<<<n_images, kChainThreads, 0, s>>>(data, jobs_dev, cands, counter, L.cap, out32, states, status,
                                                    data_bytes, frames_bytes, max_stream_bytes, max_raw_bytes);
  md2_png_write<<<kDecCtas, kDecThreads, 0, s>>>(data, jobs_dev, cands, counter, L.cap, out32, status);
  md2_png_resolve<<<dim3(kResolveCtas, n_images), kResolveThreads, 0, s>>>(jobs_dev, out32, raw8, states, data_bytes,
                                                                            frames_bytes, max_stream_bytes,
                                                                            max_raw_bytes);
  md2_png_unfilter<<<n_images, kUnfilterThreads, 0, s>>>(jobs_dev, raw8, states, frames, status, data_bytes,
                                                         frames_bytes, max_stream_bytes, max_raw_bytes);
  return cudaGetLastError() == cudaSuccess ? MD2_OK : MD2_ERR_CUDA;
}

}  // extern "C"
