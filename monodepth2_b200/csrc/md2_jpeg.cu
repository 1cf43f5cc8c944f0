// md2_jpeg.cu - baseline JPEG decoding on the GPU, byte for byte what Pillow's libjpeg-turbo gives (md2_jpeg.h).
//
// One call decodes every image of a batch in four launches after a memset:
//   md2_jpeg_sync    - self-synchronising parallel Huffman decoding (Weissenberger & Schmidt, ICPP 2018).  Every
//                      segment (an image, or one restart interval) is cut into MD2_JPEG_CHUNK_BYTES chunks, one thread
//                      each.  A thread decodes its chunk from a guessed entry state (the chunk's first bit, block 0 of
//                      the MCU, a DC symbol) to its exit state; then, in shared memory, every chunk re-decodes from
//                      its predecessor's exit until no exit changes.  A decode from a wrong guess usually falls into
//                      step with the true symbol boundaries within a few symbols, so few rounds are needed, but the
//                      loop ends only when every entry is its predecessor's exit, so the result is exact however slowly
//                      the chunks resynchronise.  Across CTAs an ordered look-back chain carries the exit state: a CTA
//                      takes a ticket with atomicAdd (tickets, not blockIdx, number the chunks, so a CTA only ever waits
//                      on one that started before it), waits for its predecessor's published exit when its first chunk
//                      continues a segment, re-runs the loop from it, and publishes its own.  Each CTA also decodes
//                      the last kOverlap chunks of its predecessor's range: by the end of them its guess has almost
//                      always fallen into step with the true decode, so the published exit rarely changes anything
//                      and the chain costs a flag hand-off per CTA instead of a serial re-decode.  A segmented scan then
//                      gives every chunk the index of its first block in the segment and the per-component sums of
//                      the DC differences before it.
//   md2_jpeg_huffman - every chunk decodes again from its exact entry and writes its blocks' int16 coefficients
//                      (natural order), DC differences already summed into DC values (the segmented DC scan).
//   md2_jpeg_idct    - one thread per block: dequantisation and jpeg_idct_islow into the padded component planes.
//   md2_jpeg_color   - fancy up-sampling and ycc_rgb_convert into (height, width, 3) uint8 at each image's offset.
// Grids and scratch depend only on the image count and the capacity (chunks, blocks), so one CUDA graph serves every
// batch within it.  Malformed data only sets status bits: every read is bounded by its segment (zeros past the end),
// every write by the image's blocks, and every loop by the chunk's bits.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/md2_loss.h"
#include "md2_jpeg.h"

namespace {

constexpr int kChunkBits = MD2_JPEG_CHUNK_BYTES * 8;
constexpr int kSyncThreads = 256;       // threads per CTA of md2_jpeg_sync / md2_jpeg_huffman (one chunk each)
constexpr int kOverlap = 32;            // md2_jpeg_sync: chunks a CTA also decodes from its predecessor's range
constexpr int kOwned = kSyncThreads - kOverlap;
constexpr int kIdctThreads = 128;
constexpr int kColorThreads = 256;
constexpr int kColorCtas = 96;          // per image

struct ChunkRec {           // a chunk's exact entry, its first block in the segment and the DC sums before it
  unsigned pos;
  int blk_z;                // blk << 8 | z
  int blocks;
  int dc[3];
  int pad[2];
};
static_assert(sizeof(ChunkRec) == 32, "32 bytes per chunk");

struct Publish {            // a CTA's exit: its last chunk's exit state and the segment's sums through it
  int flag;
  unsigned pos;
  int blk_z;
  int blocks;
  int dc[3];
  int pad;
};
static_assert(sizeof(Publish) == 32, "32 bytes per CTA");

inline size_t align256(size_t n) { return (n + 255) / 256 * 256; }

struct Layout {
  size_t pub, recs, coefs, planes, total;
};
inline Layout layout(long long max_chunks, long long max_blocks) {
  Layout L;
  const long long ctas = (max_chunks + kOwned - 1) / kOwned;
  L.pub = 0;                                                   // the ticket counter, then one Publish per CTA
  L.recs = align256(sizeof(Publish) * (size_t)(ctas + 1));
  L.coefs = L.recs + align256(sizeof(ChunkRec) * (size_t)max_chunks);
  L.planes = L.coefs + align256((size_t)max_blocks * 128);
  L.total = L.planes + align256((size_t)max_blocks * 64);
  return L;
}

__device__ __forceinline__ int mcus_x(const md2_jpeg_job& j) { return (j.width + 8 * j.h_samp - 1) / (8 * j.h_samp); }
__device__ __forceinline__ int mcus_y(const md2_jpeg_job& j) { return (j.height + 8 * j.v_samp - 1) / (8 * j.v_samp); }

struct Where {
  int img, seg;
  bool first;               // the segment's first chunk
  unsigned cb, ce, seg_bits;
  int seg_blocks;           // blocks of the segment
  long long seg_block0;     // first block of the segment in the coefficient buffer
};

// The image and segment of global chunk c; false for a chunk past the last image's or inside no segment (the latter
// flags the image when `status` is given).
__device__ __forceinline__ bool locate(long long c, const unsigned char* __restrict__ data, const md2_jpeg_job* __restrict__ jobs,
                       int n_images, unsigned* status, Where* w) {
  int lo = 0, hi = n_images - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (jobs[mid].chunk_offset <= c) lo = mid; else hi = mid - 1;
  }
  const md2_jpeg_job& j = jobs[lo];
  const long long local = c - j.chunk_offset;
  if (local < 0 || local >= j.n_chunks) return false;
  const md2_jpeg_segment* segs = reinterpret_cast<const md2_jpeg_segment*>(data + j.segments_offset);
  int a = 0, b = j.n_segments - 1;
  while (a < b) {
    const int mid = (a + b + 1) >> 1;
    if (segs[mid].chunk <= local) a = mid; else b = mid - 1;
  }
  const md2_jpeg_segment s = segs[a];
  const long long nch = s.bytes > 0 ? (s.bytes + MD2_JPEG_CHUNK_BYTES - 1) / MD2_JPEG_CHUNK_BYTES : 1;
  if (s.chunk < 0 || s.bytes < 0 || s.chunk + nch > j.n_chunks || local < s.chunk || local >= s.chunk + nch) {
    if (status) atomicOr(status + lo, MD2_JPEG_BAD_SEGMENT);
    return false;
  }
  const int mcus = mcus_x(j) * mcus_y(j);
  const int per = j.restart_interval > 0 ? j.restart_interval : mcus;
  const int first_mcu = a * per;
  const int n_mcu = min(per, mcus - first_mcu);
  const int bpm = j.h_samp * j.v_samp + 2;
  w->img = lo;
  w->seg = a;
  w->first = local == s.chunk;
  w->seg_bits = (unsigned)s.bytes * 8u;
  w->cb = (unsigned)(local - s.chunk) * kChunkBits;
  w->ce = min(w->cb + kChunkBits, w->seg_bits);
  w->seg_blocks = n_mcu > 0 ? n_mcu * bpm : 0;
  w->seg_block0 = j.block_offset + (long long)first_mcu * bpm;
  return true;
}

__device__ __forceinline__ Md2JpegImage image_of(const unsigned char* data, const md2_jpeg_job& j) {
  Md2JpegImage im;
  im.tab = reinterpret_cast<const md2_jpeg_tables*>(data + j.tables_offset);
  im.luma_blocks = j.h_samp * j.v_samp;
  im.tables = 0;
#pragma unroll
  for (int c = 0; c < 3; ++c) im.tables |= (unsigned)(j.dc_table[c] & 1) << c | (unsigned)(j.ac_table[c] & 1) << (3 + c);
  return im;
}

__device__ __forceinline__ Md2JpegBits bits_of(const unsigned char* data, const md2_jpeg_job& j, int seg) {
  const md2_jpeg_segment s = reinterpret_cast<const md2_jpeg_segment*>(data + j.segments_offset)[seg];
  Md2JpegBits b;
  b.d = data + j.entropy_offset + (long long)s.chunk * MD2_JPEG_CHUNK_BYTES;
  b.n = (unsigned)s.bytes;
  b.bp = 0;
  b.nb = 0;
  b.buf = 0;
  return b;
}

struct SyncShared {
  unsigned pos[kSyncThreads];
  int blk_z[kSyncThreads];
  int cnt[kSyncThreads];
  int dc[3][kSyncThreads];
  int head[kSyncThreads];
  unsigned ticket;
  int waited;
  Publish prev;
};

__global__ void __launch_bounds__(kSyncThreads) md2_jpeg_sync(const unsigned char* __restrict__ data,
                                                               const md2_jpeg_job* __restrict__ jobs, int n_images,
                                                               long long max_chunks, Publish* pub, ChunkRec* recs,
                                                               unsigned* status) {
  __shared__ SyncShared sh;
  const int tid = threadIdx.x;
  if (tid == 0) sh.ticket = atomicAdd(reinterpret_cast<unsigned*>(pub), 1u);
  __syncthreads();
  const unsigned t = sh.ticket;
  Publish* mine_pub = pub + 1 + t;
  const long long c = (long long)t * kOwned - kOverlap + tid;   // threads < kOverlap: the predecessor's last chunks
  const bool owned = tid >= kOverlap;
  Where w;
  const bool located = c >= 0 && c < max_chunks && locate(c, data, jobs, n_images, owned ? status : nullptr, &w);
  Md2JpegImage im;
  Md2JpegBits bits;
  Md2JpegState entry = {0u, 0, 0};
  int cnt = 0;
  Md2JpegDc dc = {0, 0, 0};
  if (located) {
    const md2_jpeg_job& j = jobs[w.img];
    im = image_of(data, j);
    bits = bits_of(data, j, w.seg);
    if (!w.first) entry.pos = w.cb;                            // the guess: a DC symbol of block 0 at the chunk start
  }
  Md2JpegState in = entry;
  bool follows = located && !w.first && tid > 0;
  auto check = [&]() {                                         // does the predecessor's exit differ from my entry?
    in = entry;
    if (!follows) return false;
    in.pos = sh.pos[tid - 1];
    in.blk = sh.blk_z[tid - 1] >> 8;
    in.z = sh.blk_z[tid - 1] & 0xFF;
    return in.pos != entry.pos || in.blk != entry.blk || in.z != entry.z;
  };
  if (!located) {
    sh.pos[tid] = 0xFFFFFFFFu;
    sh.blk_z[tid] = 0;
  }
  bool need = located;                                         // the first pass decodes from the guess
  bool waits = false;
  // Phase 0 settles the CTA on its own; phase 1 is the look-back.  The first owned chunk continues a segment begun in
  // the previous CTA: the overlap chunks decoded the end of that CTA's range from a guess and have almost always
  // fallen into step with the true decode, so the published exit usually equals the overlap's and nothing is decoded
  // again.  Either way the owned chunks are settled once more from the published exit, which is exact.
  for (int phase = 0; phase < 2; ++phase) {
    if (phase == 1) {
      waits = located && tid == kOverlap && !w.first;
      if (tid == kOverlap) sh.waited = waits;
      if (waits) {
        const volatile Publish* p = pub + t;                   // pub + 1 + (t - 1)
        while (p->flag == 0) __nanosleep(64);
        __threadfence();
        sh.prev.pos = p->pos;
        sh.prev.blk_z = p->blk_z;
        sh.prev.blocks = p->blocks;
        for (int k = 0; k < 3; ++k) sh.prev.dc[k] = p->dc[k];
      }
      __syncthreads();
      if (tid == kOverlap - 1 && sh.waited) {                  // the overlap's last exit becomes the published one
        sh.pos[tid] = sh.prev.pos;
        sh.blk_z[tid] = sh.prev.blk_z;
      }
      follows = follows && owned;
      __syncthreads();
      need = check();
      __syncthreads();
    }
    for (;;) {                                                 // until every entry is its predecessor's exit
      if (need) {
        entry = in;
        cnt = 0;
        dc = {0, 0, 0};
        const Md2JpegState e = md2_jpeg_run_chunk(bits, im, entry, w.ce, &cnt, &dc, nullptr, 0, 0, w.seg_bits, nullptr);
        sh.pos[tid] = e.pos;
        sh.blk_z[tid] = e.blk << 8 | e.z;
      }
      if (!__syncthreads_or(need)) break;
      need = check();
      __syncthreads();
    }
  }
  // segmented inclusive scan of the block counts and DC sums; the predecessor's sums enter at chunk 0
  int v[4] = {cnt, dc.y, dc.cb, dc.cr};
  if (waits) {
    v[0] += sh.prev.blocks;
    for (int k = 0; k < 3; ++k) v[1 + k] = (int)((unsigned)v[1 + k] + (unsigned)sh.prev.dc[k]);
  }
  int head = !located || w.first || tid <= kOverlap;
  if (!owned) v[0] = v[1] = v[2] = v[3] = 0;
  __syncthreads();
  for (int d = 1; d < kSyncThreads; d <<= 1) {
    sh.cnt[tid] = v[0];
    sh.dc[0][tid] = v[1];
    sh.dc[1][tid] = v[2];
    sh.dc[2][tid] = v[3];
    sh.head[tid] = head;
    __syncthreads();
    if (!head && tid >= d) {
      v[0] += sh.cnt[tid - d];
      for (int k = 0; k < 3; ++k) v[1 + k] = (int)((unsigned)v[1 + k] + (unsigned)sh.dc[k][tid - d]);
      head = sh.head[tid - d];
    }
    __syncthreads();
  }
  if (located && owned) {
    ChunkRec r;
    r.pos = entry.pos;
    r.blk_z = entry.blk << 8 | entry.z;
    r.blocks = v[0] - cnt;
    r.dc[0] = (int)((unsigned)v[1] - (unsigned)dc.y);
    r.dc[1] = (int)((unsigned)v[2] - (unsigned)dc.cb);
    r.dc[2] = (int)((unsigned)v[3] - (unsigned)dc.cr);
    r.pad[0] = r.pad[1] = 0;
    recs[c] = r;
  }
  if (tid == kSyncThreads - 1) {
    mine_pub->pos = sh.pos[tid];
    mine_pub->blk_z = sh.blk_z[tid];
    mine_pub->blocks = v[0];
    for (int k = 0; k < 3; ++k) mine_pub->dc[k] = v[1 + k];
    __threadfence();
    atomicExch(&mine_pub->flag, 1);
  }
}

__global__ void __launch_bounds__(kSyncThreads) md2_jpeg_huffman(const unsigned char* __restrict__ data,
                                                                  const md2_jpeg_job* __restrict__ jobs, int n_images,
                                                                  long long max_chunks, const ChunkRec* __restrict__ recs,
                                                                  short* coefs, unsigned* status) {
  const long long c = (long long)blockIdx.x * kSyncThreads + threadIdx.x;
  Where w;
  if (c >= max_chunks || !locate(c, data, jobs, n_images, status, &w)) return;
  const md2_jpeg_job& j = jobs[w.img];
  const Md2JpegImage im = image_of(data, j);
  Md2JpegBits bits = bits_of(data, j, w.seg);
  const ChunkRec r = recs[c];
  const Md2JpegState entry = {r.pos, r.blk_z >> 8, r.blk_z & 0xFF};
  Md2JpegDc dc = {r.dc[0], r.dc[1], r.dc[2]};
  int n = 0;
  unsigned flags = 0;
  md2_jpeg_run_chunk(bits, im, entry, w.ce, &n, &dc, coefs, w.seg_block0 + r.blocks, w.seg_blocks - r.blocks,
                     w.seg_bits, &flags);
  if (flags) atomicOr(status + w.img, flags);
}

__device__ __forceinline__ int image_of_block(long long g, const md2_jpeg_job* __restrict__ jobs, int n_images) {
  int lo = 0, hi = n_images - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (jobs[mid].block_offset <= g) lo = mid; else hi = mid - 1;
  }
  return lo;
}

__global__ void __launch_bounds__(kIdctThreads) md2_jpeg_idct(const unsigned char* __restrict__ data,
                                                               const md2_jpeg_job* __restrict__ jobs, int n_images,
                                                               long long max_blocks, const short* __restrict__ coefs,
                                                               unsigned char* planes) {
  const long long g = (long long)blockIdx.x * kIdctThreads + threadIdx.x;
  if (g >= max_blocks) return;
  const int i = image_of_block(g, jobs, n_images);
  const md2_jpeg_job& j = jobs[i];
  const int mx = mcus_x(j), my = mcus_y(j);
  const int luma = j.h_samp * j.v_samp, bpm = luma + 2;
  const long long local = g - j.block_offset;
  if (local < 0 || local >= (long long)mx * my * bpm) return;
  const int mcu = (int)(local / bpm), k = (int)(local % bpm);
  const int mr = mcu / mx, mc = mcu % mx;
  unsigned char* base = planes + j.block_offset * 64;
  const int lw = mx * 8 * j.h_samp, lh = my * 8 * j.v_samp, cw = mx * 8, ch = my * 8;
  int comp, stride, by, bx;
  if (k < luma) {
    comp = 0;
    stride = lw;
    by = mr * j.v_samp + k / j.h_samp;
    bx = mc * j.h_samp + k % j.h_samp;
  } else {
    comp = k - luma + 1;
    base += (long long)lw * lh + (long long)(comp - 1) * cw * ch;
    stride = cw;
    by = mr;
    bx = mc;
  }
  const md2_jpeg_tables* tab = reinterpret_cast<const md2_jpeg_tables*>(data + j.tables_offset);
  short blk[64];
  const int4* src = reinterpret_cast<const int4*>(coefs + g * 64);
#pragma unroll
  for (int q = 0; q < 8; ++q) reinterpret_cast<int4*>(blk)[q] = src[q];
  md2_jpeg_idct_islow(blk, tab->quant[j.quant_table[comp]], base + (long long)by * 8 * stride + bx * 8, stride);
}

__global__ void __launch_bounds__(kColorThreads) md2_jpeg_color(const md2_jpeg_job* __restrict__ jobs,
                                                                 const unsigned char* __restrict__ planes,
                                                                 unsigned char* frames) {
  const md2_jpeg_job& j = jobs[blockIdx.y];
  const int H = j.height, W = j.width, hs = j.h_samp, vs = j.v_samp;
  const int mx = mcus_x(j), my = mcus_y(j);
  const int lw = mx * 8 * hs, lh = my * 8 * vs, cws = mx * 8, chs = my * 8;
  const unsigned char* Y = planes + j.block_offset * 64;
  const unsigned char* Cb = Y + (long long)lw * lh;
  const unsigned char* Cr = Cb + (long long)cws * chs;
  const int ch = md2_jpeg_comp_size(H, 1, vs), cw = md2_jpeg_comp_size(W, 1, hs);
  unsigned char* out = frames + j.out_offset;
  const long long n = (long long)H * W;
  for (long long p = (long long)blockIdx.x * kColorThreads + threadIdx.x; p < n;
       p += (long long)gridDim.x * kColorThreads) {
    const int y = (int)(p / W), x = (int)(p % W);
    unsigned char rgb[3];
    md2_jpeg_ycc_rgb(Y[(long long)y * lw + x], md2_jpeg_chroma(Cb, cws, ch, cw, hs, vs, y, x),
                     md2_jpeg_chroma(Cr, cws, ch, cw, hs, vs, y, x), rgb);
    out[p * 3] = rgb[0];
    out[p * 3 + 1] = rgb[1];
    out[p * 3 + 2] = rgb[2];
  }
}

inline long long host_mcus(const md2_jpeg_job& j) {
  return (long long)((j.width + 8 * j.h_samp - 1) / (8 * j.h_samp)) * ((j.height + 8 * j.v_samp - 1) / (8 * j.v_samp));
}

}  // namespace

extern "C" {

int md2_jpeg_decode_scratch_bytes(int n_images, long long max_chunks, long long max_blocks, size_t* bytes) {
  if (!bytes || n_images < 1 || max_chunks < 1 || max_blocks < 1) return MD2_ERR_INVALID_ARGUMENT;
  if (max_chunks > (1LL << 31) - kSyncThreads || max_blocks > (1LL << 40)) return MD2_ERR_UNSUPPORTED;
  *bytes = layout(max_chunks, max_blocks).total;
  return MD2_OK;
}

int md2_jpeg_decode(const unsigned char* data, size_t data_bytes, const md2_jpeg_job* jobs, const md2_jpeg_job* jobs_dev,
                    int n_images, unsigned char* frames, size_t frames_bytes, unsigned int* status,
                    long long max_chunks, long long max_blocks, void* scratch, size_t scratch_bytes, void* stream) {
  if (!data || !jobs || !jobs_dev || !frames || !status || n_images < 1 || max_chunks < 1 || max_blocks < 1)
    return MD2_ERR_INVALID_ARGUMENT;
  if (n_images > 65535 || max_chunks > (1LL << 31) - kSyncThreads || max_blocks > (1LL << 40))
    return MD2_ERR_UNSUPPORTED;
  long long chunks = 0, blocks = 0;
  for (int i = 0; i < n_images; ++i) {
    const md2_jpeg_job& j = jobs[i];
    const bool samp = (j.h_samp == 1 && j.v_samp == 1) || (j.h_samp == 2 && j.v_samp == 1) ||
                      (j.h_samp == 2 && j.v_samp == 2);
    if (!samp) return MD2_ERR_UNSUPPORTED;
    if (j.height < 1 || j.width < 1 || j.height > 65535 || j.width > 65535 || j.restart_interval < 0)
      return MD2_ERR_INVALID_ARGUMENT;
    for (int c = 0; c < 3; ++c)
      if (j.dc_table[c] < 0 || j.dc_table[c] > 1 || j.ac_table[c] < 0 || j.ac_table[c] > 1 || j.quant_table[c] < 0 ||
          j.quant_table[c] > 3)
        return MD2_ERR_INVALID_ARGUMENT;
    const long long mcus = host_mcus(j);
    const long long segs = j.restart_interval > 0 ? (mcus + j.restart_interval - 1) / j.restart_interval : 1;
    if (j.n_segments != segs || j.n_chunks < j.n_segments) return MD2_ERR_INVALID_ARGUMENT;
    if (j.chunk_offset != chunks || j.block_offset != blocks) return MD2_ERR_INVALID_ARGUMENT;   // running sums
    chunks += j.n_chunks;
    blocks += mcus * (j.h_samp * j.v_samp + 2);
    auto inside = [&](long long off, long long n, long long align, size_t total) {
      return off >= 0 && off % align == 0 && (unsigned long long)off <= total && (unsigned long long)n <= total - off;
    };
    if (!inside(j.entropy_offset, (long long)j.n_chunks * MD2_JPEG_CHUNK_BYTES, 1, data_bytes) ||
        !inside(j.segments_offset, (long long)j.n_segments * (long long)sizeof(md2_jpeg_segment), 8, data_bytes) ||
        !inside(j.tables_offset, (long long)sizeof(md2_jpeg_tables), 8, data_bytes) ||
        !inside(j.out_offset, 3LL * j.height * j.width, 1, frames_bytes))
      return MD2_ERR_INVALID_ARGUMENT;
  }
  if (chunks > max_chunks || blocks > max_blocks) return MD2_ERR_UNSUPPORTED;        // over the stated capacity
  const Layout L = layout(max_chunks, max_blocks);
  if (!scratch || scratch_bytes < L.total) return MD2_ERR_WORKSPACE_TOO_SMALL;
  cudaStream_t s = (cudaStream_t)stream;
  unsigned char* base = (unsigned char*)scratch;
  Publish* pub = (Publish*)(base + L.pub);
  ChunkRec* recs = (ChunkRec*)(base + L.recs);
  short* coefs = (short*)(base + L.coefs);
  unsigned char* planes = base + L.planes;
  const long long sync_ctas = (max_chunks + kOwned - 1) / kOwned;
  const long long ctas = (max_chunks + kSyncThreads - 1) / kSyncThreads;
  if (cudaMemsetAsync(base, 0, L.recs, s) != cudaSuccess) return MD2_ERR_CUDA;
  if (cudaMemsetAsync(status, 0, sizeof(unsigned) * n_images, s) != cudaSuccess) return MD2_ERR_CUDA;
  md2_jpeg_sync<<<(unsigned)sync_ctas, kSyncThreads, 0, s>>>(data, jobs_dev, n_images, max_chunks, pub, recs, status);
  md2_jpeg_huffman<<<(unsigned)ctas, kSyncThreads, 0, s>>>(data, jobs_dev, n_images, max_chunks, recs, coefs, status);
  md2_jpeg_idct<<<(unsigned)((max_blocks + kIdctThreads - 1) / kIdctThreads), kIdctThreads, 0, s>>>(
      data, jobs_dev, n_images, max_blocks, coefs, planes);
  md2_jpeg_color<<<dim3(kColorCtas, n_images), kColorThreads, 0, s>>>(jobs_dev, planes, frames);
  return cudaGetLastError() == cudaSuccess ? MD2_OK : MD2_ERR_CUDA;
}

}  // extern "C"
