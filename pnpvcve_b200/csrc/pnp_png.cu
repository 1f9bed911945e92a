// PNG encoder on the device: F uint8 (3,H,W) frames -> F complete 8-bit RGB PNG files (pnp_png_* in
// include/pnp_vcve.h).  Replaces the host's mmcv.imwrite(tensor2img(frame)) of the reference's test loop.
//
// A frame's filtered scanlines are cut into SEGMENTS of whole rows (about kSegTarget bytes, the row count depends on W
// only).  png_segment_kernel encodes one segment per CTA, independently of every other one:
//   filter   : per row the PNG filter with the smallest sum of |signed byte| (libpng's heuristic); the filters read the
//              raw previous row from the frame, also across a segment edge
//   LZ77     : each thread parses its own slice of the segment greedily; a match is the longest of a fixed set of
//              candidate distances (the previous pixels, the row above and its neighbours), stays inside the segment,
//              is at most 32 KB back and ends at the end of the slice
//   encode   : one fixed-Huffman block (bit offsets of the slices by a block scan, shared-memory atomics), or one stored
//              block when that is not larger; a non-final segment ends with a sync flush (empty stored block), so the
//              segments concatenate into one deflate stream, and the last one carries BFINAL
//   checksums: Adler-32 sums of the filtered bytes and the CRC-32 of the coded bytes (per-thread pieces combined in GF(2))
// png_assemble_kernel then writes each segment as one IDAT chunk behind the signature and IHDR, adds the zlib header and
// the Adler-32 trailer, finishes the chunk CRCs and appends IEND.  A file depends on its pixels and (H, W) only.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/pnp_vcve.h"

namespace {

constexpr int kThreads = 256;
constexpr int kSegTarget = 32768;   // filtered bytes per segment: 2-3 CTAs of ~70 KB shared memory per SM at 720p
constexpr int kMaxW = 21844;        // 3 W + 1 <= 65533: every segment fits one stored block (LEN <= 65535)
constexpr int kMaxDist = 32768;
constexpr uint32_t kAdlerMod = 65521;

struct Geo {
  int L;          // bytes per filtered scanline: filter byte + 3 W
  int rows;       // scanlines per segment (the last segment may hold fewer)
  int nseg;
  int smax;       // filtered bytes of the largest segment
  int64_t cap;    // workspace bytes per segment: stored form, rounded up to 16
};

__host__ __device__ inline Geo geometry(int H, int W) {
  Geo g;
  g.L = 3 * W + 1;
  g.rows = kSegTarget / g.L > 0 ? kSegTarget / g.L : 1;
  if (g.rows > H) g.rows = H;
  g.nseg = (H + g.rows - 1) / g.rows;
  g.smax = g.rows * g.L;
  g.cap = ((int64_t)g.smax + 5 + 15) & ~(int64_t)15;
  return g;
}

// signature + IHDR chunk + one IDAT chunk (12 bytes of framing + stored block) per segment + zlib header and trailer
// + IEND
__host__ __device__ inline int64_t frame_bound(int H, int W) {
  const Geo g = geometry(H, W);
  return 8 + 25 + 2 + 4 + 12 + (int64_t)H * g.L + 17LL * g.nseg;
}

struct SegMeta {
  uint32_t len;   // coded bytes of the segment
  uint32_t crc;   // CRC-32 of the coded bytes
  uint32_t s1;    // sum of the filtered bytes mod 65521
  uint32_t s2;    // sum of (n - i) * byte_i mod 65521 (n filtered bytes)
};

// ------------------------------------------------------------------ CRC-32 (reflected 0xEDB88320) in GF(2)
// a * b mod P, reflected bit order (x^0 is bit 31); a != 0
__device__ inline uint32_t multmodp(uint32_t a, uint32_t b) {
  uint32_t m = 1u << 31, p = 0;
  for (;;) {
    if (a & m) {
      p ^= b;
      if ((a & (m - 1)) == 0) break;
    }
    m >>= 1;
    b = (b & 1) ? (b >> 1) ^ 0xEDB88320u : b >> 1;
  }
  return p;
}

// x^(8 n) mod P
__device__ inline uint32_t x8n(uint32_t n) {
  uint32_t p = 1u << 31, sq = 1u << 23;
  while (n) {
    if (n & 1) p = multmodp(sq, p);
    n >>= 1;
    if (n) sq = multmodp(sq, sq);
  }
  return p;
}

// CRC-32 of A || B from crc(A), crc(B) and the length of B
__device__ inline uint32_t crc_combine(uint32_t ca, uint32_t cb, uint32_t len_b) {
  return len_b ? multmodp(x8n(len_b), ca) ^ cb : ca;
}

// continues a (finished) CRC-32 over n more bytes, bit by bit (headers and trailers only)
__device__ inline uint32_t crc_bytes(uint32_t crc, const uint8_t* p, int n) {
  crc = ~crc;
  for (int i = 0; i < n; ++i) {
    crc ^= p[i];
    for (int k = 0; k < 8; ++k) crc = (crc & 1) ? (crc >> 1) ^ 0xEDB88320u : crc >> 1;
  }
  return ~crc;
}

__device__ inline void put_be32(uint8_t* p, uint32_t v) {
  p[0] = (uint8_t)(v >> 24);
  p[1] = (uint8_t)(v >> 16);
  p[2] = (uint8_t)(v >> 8);
  p[3] = (uint8_t)v;
}

// ------------------------------------------------------------------ fixed-Huffman symbols (RFC 1951 3.2.5 / 3.2.6)
struct Code {
  uint32_t bits;  // in stream order (Huffman codes already bit-reversed)
  int n;
};

__device__ inline uint32_t rev(uint32_t code, int n) { return __brev(code) >> (32 - n); }

__device__ inline Code literal_code(int v) {
  return v < 144 ? Code{rev(0x30 + v, 8), 8} : Code{rev(0x190 + v - 144, 9), 9};
}

// length 3..258 -> length code + extra bits, one field of at most 8 + 5 bits
__device__ inline Code length_code(int len) {
  int sym, ne = 0, ev = 0;
  if (len == 258) {
    sym = 285;
  } else {
    const int l = len - 3;
    if (l < 8) {
      sym = 257 + l;
    } else {
      const int e = 31 - __clz(l);
      sym = 257 + 4 * (e - 1) + ((l >> (e - 2)) & 3);
      ne = e - 2;
      ev = l & ((1 << ne) - 1);
    }
  }
  Code c = sym < 280 ? Code{rev(sym - 256, 7), 7} : Code{rev(0xC0 + sym - 280, 8), 8};
  c.bits |= (uint32_t)ev << c.n;
  c.n += ne;
  return c;
}

// distance 1..32768 -> 5-bit code + extra bits (at most 18 bits)
__device__ inline Code dist_code(int d) {
  int code, ne = 0, ev = 0;
  if (d <= 4) {
    code = d - 1;
  } else {
    const int e = 31 - __clz(d - 1);
    code = 2 * e + (((d - 1) >> (e - 1)) & 1);
    ne = e - 1;
    ev = (d - 1) & ((1 << ne) - 1);
  }
  return Code{rev(code, 5) | ((uint32_t)ev << 5), 5 + ne};
}

__device__ inline int match_len(const uint8_t* buf, int p, int d, int maxlen) {
  int n = 0;
  while (n < maxlen && buf[p + n] == buf[p + n - d]) ++n;
  return n;
}

// LSB-first bit writer into a zeroed shared-memory word buffer that neighbouring threads share at their edges
struct BitWriter {
  uint32_t* words;
  int64_t pos;      // next word
  uint64_t acc;
  int nacc;
  __device__ BitWriter(uint32_t* w, int64_t bit) : words(w), pos(bit >> 5), acc(0), nacc((int)(bit & 31)) {}
  __device__ inline void put(uint32_t bits, int n) {
    acc |= (uint64_t)bits << nacc;
    nacc += n;
    if (nacc >= 32) {
      atomicOr(&words[pos++], (uint32_t)acc);
      acc >>= 32;
      nacc -= 32;
    }
  }
  __device__ inline void flush() {
    if (nacc > 0) atomicOr(&words[pos], (uint32_t)acc);
  }
};

// Greedy LZ77 parse of buf[b0, b1) with matches from the candidate distances; EMIT = false counts the coded bits.
template <bool EMIT>
__device__ uint32_t parse(const uint8_t* buf, int b0, int b1, int L, BitWriter* bw) {
  const int cand[8] = {1, 3, 6, 2, L, L - 3, L + 3, 2 * L};
  uint32_t bits = 0;
  int p = b0;
  while (p < b1) {
    const int maxlen = min(258, b1 - p);
    int best = 0, bd = 0;
    if (maxlen >= 3) {
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int d = cand[k];
        if (d < 1 || d > p || d > kMaxDist) continue;
        const int n = match_len(buf, p, d, maxlen);
        if (n > best) {
          best = n;
          bd = d;
          if (best == maxlen) break;
        }
      }
    }
    if (best >= 3) {
      const Code lc = length_code(best), dc = dist_code(bd);
      bits += lc.n + dc.n;
      if (EMIT) {
        bw->put(lc.bits, lc.n);
        bw->put(dc.bits, dc.n);
      }
      p += best;
    } else {
      const Code c = literal_code(buf[p]);
      bits += c.n;
      if (EMIT) bw->put(c.bits, c.n);
      ++p;
    }
  }
  return bits;
}

// exclusive block scan of one value per thread; returns the total in *total
__device__ uint32_t block_scan(uint32_t v, uint32_t* scratch, uint32_t* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) scratch[warp] = x;
  __syncthreads();
  uint32_t before = 0, sum = 0;
  for (int w = 0; w < kThreads / 32; ++w) {
    if (w < warp) before += scratch[w];
    sum += scratch[w];
  }
  *total = sum;
  __syncthreads();
  return before + x - v;
}

__device__ inline uint32_t sabs(int v) { return v < 128 ? v : 256 - v; }

__device__ inline int paeth(int a, int b, int c) {
  const int p = a + b - c, pa = abs(p - a), pb = abs(p - b), pc = abs(p - c);
  return (pa <= pb && pa <= pc) ? a : (pb <= pc ? b : c);
}

// grid (nseg, F), kThreads threads; dynamic shared memory: filtered bytes | coded words | scratch
__global__ void __launch_bounds__(kThreads) png_segment_kernel(const uint8_t* __restrict__ frames, int64_t sf, int64_t sc,
                                                               int64_t sy, int H, int W, uint8_t* __restrict__ ws) {
  extern __shared__ __align__(16) uint8_t smem[];
  const Geo g = geometry(H, W);
  const int seg = blockIdx.x, f = blockIdx.y, t = threadIdx.x;
  const int y0 = seg * g.rows, nrows = min(g.rows, H - y0);
  const int S = nrows * g.L;
  const bool final_seg = seg == g.nseg - 1;
  uint8_t* filt = smem;
  const int filt_bytes = (g.smax + 15) & ~15;
  uint32_t* outw = reinterpret_cast<uint32_t*>(smem + filt_bytes);
  const int out_words = (int)(g.cap / 4);
  uint32_t* scratch = outw + out_words;                     // 4 * kThreads words
  const uint8_t* frame = frames + (int64_t)f * sf;

  for (int i = t; i < out_words; i += kThreads) outw[i] = 0;

  // ---- filter: one row at a time, the five candidates scored by the whole block
  for (int r = 0; r < nrows; ++r) {
    const int y = y0 + r;
    uint32_t sum[5] = {0, 0, 0, 0, 0};
    for (int pass = 0; pass < 2; ++pass) {
      int ft = 0;
      if (pass == 1) {
        uint32_t* part = scratch + (r & 1) * 5 * (kThreads / 32);
        uint32_t best = 0xffffffffu;
        for (int k = 0; k < 5; ++k) {
          uint32_t s = 0;
          for (int w = 0; w < kThreads / 32; ++w) s += part[k * (kThreads / 32) + w];
          if (s < best) {
            best = s;
            ft = k;
          }
        }
        if (t == 0) filt[r * g.L] = (uint8_t)ft;
      }
      for (int x = t; x < W; x += kThreads) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const uint8_t* row = frame + c * sc + (int64_t)y * sy;
          const int v = __ldg(row + x);
          const int a = x > 0 ? __ldg(row + x - 1) : 0;
          const int b = y > 0 ? __ldg(row - sy + x) : 0;
          const int cc = (x > 0 && y > 0) ? __ldg(row - sy + x - 1) : 0;
          const int fv[5] = {v, v - a, v - b, v - ((a + b) >> 1), v - paeth(a, b, cc)};
          if (pass == 0) {
#pragma unroll
            for (int k = 0; k < 5; ++k) sum[k] += sabs(fv[k] & 255);
          } else {
            filt[r * g.L + 1 + 3 * x + c] = (uint8_t)fv[ft];
          }
        }
      }
      if (pass == 0) {
        uint32_t* part = scratch + (r & 1) * 5 * (kThreads / 32);
#pragma unroll
        for (int k = 0; k < 5; ++k) {
          uint32_t s = sum[k];
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
          if ((t & 31) == 0) part[k * (kThreads / 32) + (t >> 5)] = s;
        }
        __syncthreads();
      }
    }
  }
  __syncthreads();

  // ---- LZ77 + fixed Huffman: size first, then emit when the fixed block is not larger than the stored one
  const int sub = (S + kThreads - 1) / kThreads;
  const int b0 = min(S, t * sub), b1 = min(S, b0 + sub);
  uint32_t s1 = 0, s2 = 0;
  for (int i = b0; i < b1; ++i) {
    s1 += filt[i];
    s2 += s1;
  }
  const uint32_t my_bits = parse<false>(filt, b0, b1, g.L, nullptr);
  uint32_t body = 0;
  const uint32_t start = block_scan(my_bits, scratch + 4 * kThreads - 32, &body);
  // header (3 bits), body, end of block (7 zero bits); non-final: empty stored block header (3 zero bits), pad, 00 00 FF FF
  const uint32_t fixed_len = final_seg ? (10 + body + 7) / 8 : (13 + body + 7) / 8 + 4;
  const uint32_t stored_len = (uint32_t)S + 5;
  const bool fixed = fixed_len <= stored_len;
  const uint32_t len = fixed ? fixed_len : stored_len;
  uint8_t* outb = reinterpret_cast<uint8_t*>(outw);
  if (fixed) {
    BitWriter bw(outw, 3 + (int64_t)start);
    parse<true>(filt, b0, b1, g.L, &bw);
    bw.flush();
    if (t == 0) atomicOr(&outw[0], (final_seg ? 1u : 0u) | 2u);
    __syncthreads();
    if (t == 0 && !final_seg) {
      outb[len - 4] = 0;
      outb[len - 3] = 0;
      outb[len - 2] = 0xFF;
      outb[len - 1] = 0xFF;
    }
  } else {
    if (t == 0) {
      outb[0] = final_seg ? 1 : 0;
      outb[1] = (uint8_t)S;
      outb[2] = (uint8_t)(S >> 8);
      outb[3] = (uint8_t)~S;
      outb[4] = (uint8_t)(~S >> 8);
    }
    for (int i = t; i < S; i += kThreads) outb[5 + i] = filt[i];
  }
  __syncthreads();

  // ---- checksums: per-thread pieces, combined pairwise in a tree
  const int piece = ((int)len + kThreads - 1) / kThreads;
  const int c0 = min((int)len, t * piece), c1 = min((int)len, c0 + piece);
  uint32_t crc = 0xffffffffu;
  for (int i = c0; i < c1; ++i) {
    crc ^= outb[i];
#pragma unroll
    for (int k = 0; k < 8; ++k) crc = (crc & 1) ? (crc >> 1) ^ 0xEDB88320u : crc >> 1;
  }
  crc = ~crc;
  uint32_t* t_crc = scratch;
  uint32_t* t_len = scratch + kThreads;
  uint32_t* t_s1 = scratch + 2 * kThreads;
  uint32_t* t_s2 = scratch + 3 * kThreads;
  t_crc[t] = crc;
  t_len[t] = c1 - c0;
  t_s1[t] = s1 % kAdlerMod;
  t_s2[t] = s2 % kAdlerMod;
  __syncthreads();
  for (int step = 1; step < kThreads; step <<= 1) {
    if ((t & (2 * step - 1)) == 0) {
      const int u = t + step;
      t_crc[t] = crc_combine(t_crc[t], t_crc[u], t_len[u]);
      t_len[t] += t_len[u];
      // Adler sums of A || B: s1 = s1A + s1B, s2 = s2A + nB s1A + s2B (nB = B's filtered bytes)
      const int nb = min(S, u * sub + step * sub) - min(S, u * sub);
      t_s2[t] = (uint32_t)((t_s2[t] + (uint64_t)nb * t_s1[t] + t_s2[u]) % kAdlerMod);
      t_s1[t] = (t_s1[t] + t_s1[u]) % kAdlerMod;
    }
    __syncthreads();
  }

  // ---- out: coded bytes (whole words; the workspace slot is a multiple of 16 bytes) and the segment's record
  SegMeta* meta = reinterpret_cast<SegMeta*>(ws) + (int64_t)f * g.nseg + seg;
  uint32_t* dst = reinterpret_cast<uint32_t*>(ws + (int64_t)gridDim.y * g.nseg * sizeof(SegMeta) +
                                              ((int64_t)f * g.nseg + seg) * g.cap);
  for (int i = t; i < ((int)len + 3) / 4; i += kThreads) dst[i] = outw[i];
  if (t == 0) *meta = SegMeta{len, t_crc[0], t_s1[0], t_s2[0]};
}

// grid (nseg, F): segment s of frame f becomes IDAT chunk s of PNG f
__global__ void __launch_bounds__(kThreads) png_assemble_kernel(const uint8_t* __restrict__ ws, int F, int H, int W,
                                                                uint8_t* __restrict__ out, int64_t out_stride,
                                                                int64_t* __restrict__ out_sizes) {
  __shared__ int64_t s_data;   // byte offset of the segment's coded bytes in the PNG
  __shared__ unsigned long long s_before;   // coded bytes of segments 0..s-1
  const Geo g = geometry(H, W);
  const int seg = blockIdx.x, f = blockIdx.y, t = threadIdx.x;
  const bool first = seg == 0, last = seg == g.nseg - 1;
  const SegMeta* meta = reinterpret_cast<const SegMeta*>(ws) + (int64_t)f * g.nseg;
  const uint8_t* src = ws + (int64_t)F * g.nseg * sizeof(SegMeta) + ((int64_t)f * g.nseg + seg) * g.cap;
  uint8_t* png = out + (int64_t)f * out_stride;
  if (t == 0) s_before = 0;
  __syncthreads();
  unsigned long long part = 0;
  for (int k = t; k < seg; k += kThreads) part += meta[k].len;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
  if ((t & 31) == 0 && part) atomicAdd(&s_before, part);
  __syncthreads();
  if (t == 0) {
    // chunk s starts behind the signature, IHDR and chunks 0..s-1 (12 bytes of framing each; zlib header in chunk 0)
    const int64_t at = 8 + 25 + 12LL * seg + (seg > 0 ? 2 : 0) + (int64_t)s_before;
    const uint32_t dlen = meta[seg].len + (first ? 2 : 0) + (last ? 4 : 0);
    uint8_t* chunk = png + at;
    put_be32(chunk, dlen);
    chunk[4] = 'I';
    chunk[5] = 'D';
    chunk[6] = 'A';
    chunk[7] = 'T';
    if (first) {
      chunk[8] = 0x78;
      chunk[9] = 0x01;
    }
    uint32_t crc = crc_bytes(0, chunk + 4, first ? 6 : 4);
    crc = crc_combine(crc, meta[seg].crc, meta[seg].len);
    if (last) {
      // zlib trailer: Adler-32 of all filtered bytes, folded segment by segment
      uint64_t s1 = 0, s2 = 0;
      for (int k = 0; k < g.nseg; ++k) {
        const uint64_t n = (uint64_t)min(g.rows, H - k * g.rows) * g.L;
        s2 = (s2 + n % kAdlerMod * s1 + meta[k].s2) % kAdlerMod;
        s1 = (s1 + meta[k].s1) % kAdlerMod;
      }
      const uint32_t a = (uint32_t)((1 + s1) % kAdlerMod);
      const uint32_t b = (uint32_t)(((uint64_t)H * g.L % kAdlerMod + s2) % kAdlerMod);
      uint8_t* trailer = chunk + 8 + (first ? 2 : 0) + meta[seg].len;
      put_be32(trailer, b << 16 | a);
      crc = crc_bytes(crc, trailer, 4);
      uint8_t* iend = chunk + 8 + dlen + 4;
      put_be32(chunk + 8 + dlen, crc);
      const uint8_t kIend[12] = {0, 0, 0, 0, 'I', 'E', 'N', 'D', 0xAE, 0x42, 0x60, 0x82};
      for (int i = 0; i < 12; ++i) iend[i] = kIend[i];
      out_sizes[f] = at + 12 + dlen + 12;
    } else {
      put_be32(chunk + 8 + dlen, crc);
    }
    if (first) {
      const uint8_t kSig[8] = {0x89, 'P', 'N', 'G', 0x0D, 0x0A, 0x1A, 0x0A};
      for (int i = 0; i < 8; ++i) png[i] = kSig[i];
      uint8_t* ihdr = png + 8;
      put_be32(ihdr, 13);
      ihdr[4] = 'I';
      ihdr[5] = 'H';
      ihdr[6] = 'D';
      ihdr[7] = 'R';
      put_be32(ihdr + 8, (uint32_t)W);
      put_be32(ihdr + 12, (uint32_t)H);
      ihdr[16] = 8;    // bit depth
      ihdr[17] = 2;    // truecolour
      ihdr[18] = ihdr[19] = ihdr[20] = 0;   // deflate, adaptive filtering, no interlace
      put_be32(ihdr + 21, crc_bytes(0, ihdr + 4, 17));
    }
    s_data = at + 8 + (first ? 2 : 0);
  }
  __syncthreads();
  uint8_t* dst = png + s_data;
  const int n = (int)meta[seg].len;
  for (int i = t; i < n; i += kThreads) dst[i] = src[i];
}

// The library's error text lives in pnp_api.cu: pnp_last_error() hands out this thread's buffer, g_err, whose size this
// must not exceed.
constexpr size_t kErrBytes = 512;

int png_fail(const char* fmt, ...) {
  char* buf = const_cast<char*>(pnp_last_error());
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, kErrBytes, fmt, ap);
  va_end(ap);
  return PNP_ERR_ARG;
}

bool bad_size(int H, int W) { return H < 1 || W < 1 || W > kMaxW; }

}  // namespace

extern "C" {

int64_t pnp_png_frame_bound(int H, int W) {
  if (bad_size(H, W)) return png_fail("pnp_png_frame_bound: bad size %d x %d (H >= 1, 1 <= W <= %d)", H, W, kMaxW);
  return frame_bound(H, W);
}

int64_t pnp_png_workspace_bytes(int F, int H, int W) {
  if (F < 1 || F > 65535 || bad_size(H, W))
    return png_fail("pnp_png_workspace_bytes: bad size F=%d %d x %d (1 <= F <= 65535, H >= 1, 1 <= W <= %d)", F, H, W,
                    kMaxW);
  const Geo g = geometry(H, W);
  return (int64_t)F * g.nseg * (int64_t)(sizeof(SegMeta) + g.cap);
}

int pnp_png_encode(const uint8_t* frames, int64_t sf, int64_t sc, int64_t sy, int F, int H, int W, uint8_t* out,
                   int64_t out_frame_stride, int64_t* out_sizes, void* workspace, int64_t workspace_bytes,
                   void* stream) {
  if (!frames || !out || !out_sizes || !workspace) return png_fail("pnp_png_encode: null pointer");
  if (F < 1 || F > 65535 || bad_size(H, W))
    return png_fail("pnp_png_encode: bad size F=%d %d x %d (1 <= F <= 65535, H >= 1, 1 <= W <= %d)", F, H, W, kMaxW);
  const int64_t bound = frame_bound(H, W);
  if (F > 1 && out_frame_stride < bound)
    return png_fail("pnp_png_encode: out_frame_stride %lld is shorter than the frame bound %lld",
                    (long long)out_frame_stride, (long long)bound);
  const int64_t need = pnp_png_workspace_bytes(F, H, W);
  if (workspace_bytes < need)
    return png_fail("pnp_png_encode: workspace of %lld bytes, %lld needed", (long long)workspace_bytes, (long long)need);
  if (reinterpret_cast<uintptr_t>(workspace) & 15) return png_fail("pnp_png_encode: workspace must be 16-byte aligned");
  const int rc = pnp_device_check();
  if (rc) return rc;
  const Geo g = geometry(H, W);
  const size_t smem = (size_t)((g.smax + 15) & ~15) + (size_t)g.cap + 4 * kThreads * sizeof(uint32_t);
  cudaError_t e = cudaFuncSetAttribute(png_segment_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  const cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  if (e == cudaSuccess) {
    png_segment_kernel<<<dim3(g.nseg, F), kThreads, smem, st>>>(frames, sf, sc, sy, H, W, ws);
    png_assemble_kernel<<<dim3(g.nseg, F), kThreads, 0, st>>>(ws, F, H, W, out, out_frame_stride, out_sizes);
    e = cudaGetLastError();
  }
  if (e != cudaSuccess) {
    char* buf = const_cast<char*>(pnp_last_error());
    snprintf(buf, kErrBytes, "pnp_png_encode: %s", cudaGetErrorString(e));
    return PNP_ERR_CUDA;
  }
  return PNP_OK;
}

}  // extern "C"
