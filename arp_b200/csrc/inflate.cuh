#pragma once
// zlib (RFC 1950 framing around RFC 1951 DEFLATE) inflate on the device, one stream per dataset row.
//
// The recorder stores `ob` as gzip chunks of one row each; HDF5's deflate filter writes a plain zlib stream per chunk.
// inflate_rows_kernel decodes n such streams from one buffer of concatenated chunks into whole rows of row_bytes bytes
// (row r at out + r * row_bytes), so the existing decode kernel reads the scored frame with the strided-row contract of
// arp_label: pointer row 0 + (F-1) * frame, stride row_bytes.
//
// Layout: one warp per stream, INF_WARPS streams per CTA. The Huffman decode is serial per stream; every lane of the warp
// runs it on the same data (warp-uniform control flow, broadcast loads), lane 0 writes literals, the lanes copy matches
// and fill the lookup tables in parallel, and the Adler-32 of the inflated row is a warp reduction. Tables live in shared
// memory (3.6 KB per warp): puff-style canonical count / symbol arrays plus a FAST_BITS-bit direct lookup; codes longer
// than FAST_BITS take the canonical walk.
//
// Malformed input never faults: every source read is checked against the row's src_bytes, every back-reference against
// the output position and every write against row_bytes. The first violation stops the row and sets status[row] to an
// ArpInflateStatus; no check traps.
#include <cstdint>

namespace arp_inflate {

constexpr int INF_WARPS = 4;
constexpr int FAST_BITS = 9;
constexpr uint32_t ADLER_MOD = 65521;

struct Huff {
  uint16_t count[16];               // codes of each length (count[0]: unused symbols)
  uint16_t sym[288];                // symbols in canonical code order
  uint16_t fast[1 << FAST_BITS];    // next FAST_BITS input bits -> (symbol << 4) | length; 0: longer code or none
};

struct WarpSmem {
  Huff lit, dist;
  uint8_t lens[320];                // code lengths of a dynamic block's two codes (HLIT + HDIST <= 316)
};

__constant__ uint16_t kLenBase[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31,
                                      35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
__constant__ uint8_t kLenExtra[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
__constant__ uint16_t kDistBase[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769,
                                       1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
__constant__ uint8_t kDistExtra[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11,
                                       12, 12, 13, 13};
__constant__ uint8_t kClenOrder[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

// LSB-first bit reader over one stream; bits above cnt are zero
struct Bits {
  const uint8_t* src;
  int64_t n, pos;                   // stream bytes, next byte not yet in buf
  uint64_t buf;
  int cnt;
  __device__ void refill() {
    while (cnt <= 56 && pos < n) { buf |= static_cast<uint64_t>(__ldg(src + pos)) << cnt; ++pos; cnt += 8; }
  }
  __device__ bool need(int k) { if (cnt < k) refill(); return cnt >= k; }
  __device__ uint32_t peek(int k) const { return static_cast<uint32_t>(buf & ((1ull << k) - 1)); }
  __device__ void drop(int k) { buf >>= k; cnt -= k; }
  // to the next byte boundary, handing the whole bytes still in buf back to the source
  __device__ void align() { drop(cnt & 7); pos -= cnt >> 3; buf = 0; cnt = 0; }
};

enum { SYM_BAD = -1, SYM_EOF = -2 };

// canonical walk of the first `max_len` bits of `bits` (puff.c's decode); SYM_BAD when no code of that length matches
__device__ __forceinline__ int walk(const Huff& h, uint32_t bits, int max_len, int* len_out) {
  int code = 0, first = 0, index = 0;
  for (int len = 1; len <= max_len; ++len) {
    code |= (bits >> (len - 1)) & 1;
    const int count = h.count[len];
    if (code - count < first) { *len_out = len; return h.sym[index + (code - first)]; }
    index += count;
    first = (first + count) << 1;
    code <<= 1;
  }
  return SYM_BAD;
}

__device__ __forceinline__ int decode(Bits& b, const Huff& h) {
  b.refill();
  const uint32_t e = h.fast[b.peek(FAST_BITS)];
  int len = e & 15, sym = static_cast<int>(e >> 4);
  if (!e) {
    sym = walk(h, static_cast<uint32_t>(b.buf), 15, &len);
    if (sym < 0) return b.cnt < 15 ? SYM_EOF : SYM_BAD;
  }
  if (len > b.cnt) return SYM_EOF;
  b.drop(len);
  return sym;
}

// builds h from n code lengths (lens in shared memory, written before the call); false when over-subscribed.
// Incomplete codes are accepted: their unused codes decode as SYM_BAD.
__device__ bool build(Huff& h, const uint8_t* lens, int n, int lane) {
  __syncwarp();                     // every lane is done with the previous table and lens is written
  if (lane == 0) {
    uint16_t offs[16];
    for (int i = 0; i < 16; ++i) h.count[i] = 0;
    for (int s = 0; s < n; ++s) h.count[lens[s]]++;
    offs[1] = 0;
    for (int len = 1; len < 15; ++len) offs[len + 1] = offs[len] + h.count[len];
    for (int s = 0; s < n; ++s)
      if (lens[s]) h.sym[offs[lens[s]]++] = static_cast<uint16_t>(s);
  }
  __syncwarp();
  int left = 1;
  for (int len = 1; len <= 15; ++len) {
    left = (left << 1) - h.count[len];
    if (left < 0) return false;
  }
  for (int j = lane; j < (1 << FAST_BITS); j += 32) {
    int len = 0;
    const int sym = walk(h, static_cast<uint32_t>(j), FAST_BITS, &len);
    h.fast[j] = sym < 0 ? 0 : static_cast<uint16_t>((sym << 4) | len);
  }
  __syncwarp();
  return true;
}

// Adler-32 of out[0, n) as a warp reduction: a = 1 + sum x_i, b = n + sum (n - i) x_i  (mod 65521)
__device__ uint32_t adler32_warp(const uint8_t* out, int64_t n, int lane) {
  uint64_t sa = 0, sb = 0;
  int64_t w = (n - lane) % ADLER_MOD;         // (n - i) mod 65521 for i = lane, lane + 32, ...
  for (int64_t i = lane; i < n; i += 32) {
    const uint32_t x = out[i];
    sa += x;
    sb += static_cast<uint64_t>(w) * x;
    w -= 32;
    if (w < 0) w += ADLER_MOD;
  }
  for (int o = 16; o; o >>= 1) {
    sa += __shfl_xor_sync(0xffffffffu, sa, o);
    sb += __shfl_xor_sync(0xffffffffu, sb, o);
  }
  const uint32_t a = static_cast<uint32_t>((1 + sa) % ADLER_MOD);
  const uint32_t bb = static_cast<uint32_t>((static_cast<uint64_t>(n % ADLER_MOD) + sb) % ADLER_MOD);
  return (bb << 16) | a;
}

// one zlib stream src[0, nsrc) -> out[0, cap); returns an ArpInflateStatus. Warp-uniform: every lane returns the same.
__device__ int inflate_stream(const uint8_t* src, int64_t nsrc, uint8_t* out, int64_t cap, WarpSmem& s, int lane) {
  if (nsrc < 2) return ARP_INFLATE_TRUNCATED;
  const uint32_t cmf = __ldg(src), flg = __ldg(src + 1);
  if ((cmf & 15) != 8 || (cmf >> 4) > 7 || ((cmf << 8) | flg) % 31 != 0 || (flg & 0x20)) return ARP_INFLATE_BAD_HEADER;
  Bits b{src, nsrc, 2, 0, 0};
  int64_t pos = 0;
  bool last = false;
  while (!last) {
    if (!b.need(3)) return ARP_INFLATE_TRUNCATED;
    last = b.peek(1);
    const int type = (b.buf >> 1) & 3;
    b.drop(3);
    if (type == 3) return ARP_INFLATE_BAD_BLOCK;
    if (type == 0) {                                   // stored
      b.align();
      if (b.pos + 4 > nsrc) return ARP_INFLATE_TRUNCATED;
      const uint32_t len = __ldg(src + b.pos) | (__ldg(src + b.pos + 1) << 8);
      const uint32_t nlen = __ldg(src + b.pos + 2) | (__ldg(src + b.pos + 3) << 8);
      if ((len ^ 0xffffu) != nlen) return ARP_INFLATE_BAD_BLOCK;
      b.pos += 4;
      if (b.pos + len > nsrc) return ARP_INFLATE_TRUNCATED;
      if (pos + len > cap) return ARP_INFLATE_TOO_LONG;
      for (uint32_t i = lane; i < len; i += 32) out[pos + i] = __ldg(src + b.pos + i);
      b.pos += len;
      pos += len;
      continue;
    }
    if (type == 1) {                                   // fixed Huffman codes
      __syncwarp();
      if (lane == 0) {
        for (int i = 0; i < 288; ++i) s.lens[i] = i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : 8;
        for (int i = 0; i < 30; ++i) s.lens[288 + i] = 5;
      }
      build(s.lit, s.lens, 288, lane);
      build(s.dist, s.lens + 288, 30, lane);
    } else {                                           // dynamic Huffman codes
      if (!b.need(14)) return ARP_INFLATE_TRUNCATED;
      const int hlit = b.peek(5) + 257, hdist = ((b.buf >> 5) & 31) + 1, hclen = ((b.buf >> 10) & 15) + 4;
      b.drop(14);
      if (hlit > 286 || hdist > 30) return ARP_INFLATE_BAD_CODE;
      __syncwarp();
      for (int i = 0; i < 19; ++i) {
        uint32_t l = 0;
        if (i < hclen) {
          if (!b.need(3)) return ARP_INFLATE_TRUNCATED;
          l = b.peek(3);
          b.drop(3);
        }
        if (lane == 0) s.lens[kClenOrder[i]] = static_cast<uint8_t>(l);
      }
      if (!build(s.dist, s.lens, 19, lane)) return ARP_INFLATE_BAD_CODE;   // the code-length code, in the dist slot
      __syncwarp();
      int k = 0, prev = -1;
      while (k < hlit + hdist) {
        const int sym = decode(b, s.dist);
        if (sym < 0) return sym == SYM_EOF ? ARP_INFLATE_TRUNCATED : ARP_INFLATE_BAD_CODE;
        int rep = 1, val = sym;
        if (sym >= 16) {
          const int nb = sym == 16 ? 2 : sym == 17 ? 3 : 7;
          if (!b.need(nb)) return ARP_INFLATE_TRUNCATED;
          rep = (sym == 16 ? 3 : sym == 17 ? 3 : 11) + static_cast<int>(b.peek(nb));
          b.drop(nb);
          if (sym == 16) {
            if (prev < 0) return ARP_INFLATE_BAD_CODE;
            val = prev;
          } else {
            val = 0;
          }
        }
        if (k + rep > hlit + hdist) return ARP_INFLATE_BAD_CODE;
        if (lane == 0)
          for (int r = 0; r < rep; ++r) s.lens[k + r] = static_cast<uint8_t>(val);
        k += rep;
        prev = val;
      }
      __syncwarp();
      if (s.lens[256] == 0) return ARP_INFLATE_BAD_CODE;                // no end-of-block code
      // build() writes s.dist, which the lengths were just decoded with: its leading __syncwarp orders that
      if (!build(s.lit, s.lens, hlit, lane)) return ARP_INFLATE_BAD_CODE;
      if (!build(s.dist, s.lens + hlit, hdist, lane)) return ARP_INFLATE_BAD_CODE;
    }
    for (;;) {
      int sym = decode(b, s.lit);
      if (sym < 0) return sym == SYM_EOF ? ARP_INFLATE_TRUNCATED : ARP_INFLATE_BAD_CODE;
      if (sym < 256) {
        if (pos >= cap) return ARP_INFLATE_TOO_LONG;
        if (lane == 0) out[pos] = static_cast<uint8_t>(sym);
        ++pos;
        continue;
      }
      if (sym == 256) break;
      sym -= 257;
      if (sym >= 29) return ARP_INFLATE_BAD_CODE;
      const int le = kLenExtra[sym];
      if (!b.need(le)) return ARP_INFLATE_TRUNCATED;
      const int len = kLenBase[sym] + static_cast<int>(b.peek(le));
      b.drop(le);
      const int dsym = decode(b, s.dist);
      if (dsym < 0) return dsym == SYM_EOF ? ARP_INFLATE_TRUNCATED : ARP_INFLATE_BAD_CODE;
      if (dsym >= 30) return ARP_INFLATE_BAD_CODE;
      const int de = kDistExtra[dsym];
      if (!b.need(de)) return ARP_INFLATE_TRUNCATED;
      const int dist = kDistBase[dsym] + static_cast<int>(b.peek(de));
      b.drop(de);
      if (dist > pos) return ARP_INFLATE_DISTANCE_TOO_FAR;
      if (pos + len > cap) return ARP_INFLATE_TOO_LONG;
      __syncwarp();                                    // the bytes this match reads were written by any lane
      // out[pos + i] = out[pos + i - dist], unrolled: every source byte lies before pos, so lanes copy independently
      for (int i = lane; i < len; i += 32) out[pos + i] = out[pos - dist + (i < dist ? i : i % dist)];
      pos += len;
    }
  }
  b.align();
  if (b.pos + 4 > nsrc) return ARP_INFLATE_TRUNCATED;
  if (pos != cap) return ARP_INFLATE_TOO_SHORT;
  const uint32_t want = (static_cast<uint32_t>(__ldg(src + b.pos)) << 24) | (static_cast<uint32_t>(__ldg(src + b.pos + 1)) << 16) |
                        (static_cast<uint32_t>(__ldg(src + b.pos + 2)) << 8) | __ldg(src + b.pos + 3);
  __syncwarp();
  return adler32_warp(out, cap, lane) == want ? ARP_INFLATE_OK : ARP_INFLATE_BAD_ADLER;
}

// row r: the zlib stream src[src_off[r], src_off[r] + src_bytes[r]) -> out[r * row_bytes, (r + 1) * row_bytes),
// status[r] = ArpInflateStatus. A negative offset or size is reported as a truncated stream.
__global__ void __launch_bounds__(INF_WARPS * 32)
inflate_rows_kernel(const uint8_t* __restrict__ src, const int64_t* __restrict__ src_off,
                    const int64_t* __restrict__ src_bytes, int n, int64_t row_bytes, uint8_t* __restrict__ out,
                    int* __restrict__ status) {
  __shared__ WarpSmem smem[INF_WARPS];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row = blockIdx.x * INF_WARPS + w;
  if (row >= n) return;
  const int64_t off = src_off[row], nb = src_bytes[row];
  const int st = off < 0 || nb < 0 ? ARP_INFLATE_TRUNCATED
                                   : inflate_stream(src + off, nb, out + static_cast<int64_t>(row) * row_bytes, row_bytes,
                                                    smem[w], lane);
  if (lane == 0) status[row] = st;
}

}  // namespace arp_inflate
