// Replay checkpoints as blocked gzip, compressed and inflated on the device.
//
// A store column's checkpoint file (circular_replay_buffer.py: save / load) is a sequence of
// independent gzip members (RFC 1952 allows any number; gzip.GzipFile reads them as one
// stream).  Member 0 holds the .npy header and is written by the host; member k >= 1 holds
// column bytes [(k-1) * 65280, k * 65280).  Every member carries the BGZF extra field
// (subfield 'B' 'C', BSIZE = member size - 1), so a reader finds every member from the
// headers alone, and its body is raw deflate (RFC 1951) of fixed-Huffman or stored blocks
// whose matches stay inside the member.  Each member is therefore compressed, and later
// inflated, by one CTA of its own, and a 65280-byte slice always fits one stored block:
// a member never exceeds 18 + 5 + 65280 + 8 = 65311 bytes, under BSIZE's 64 KB.
//
// Compress (one CTA per member): the slice is staged into shared memory by one bulk copy,
// every position is entered in a shared hash table per 8160-byte epoch, and each of the 128
// threads parses its own 510-byte sub-range greedily, with candidates from that table (the
// latest earlier occurrence in its own epoch and the two before it) and the run at distance
// 1.  A block scan of the threads' bit counts places every thread's codes; the member is
// assembled in shared memory and written out whole.  The CRC-32 is computed per thread
// slice and combined with GF(2) multiplications by x^(8n).  When the fixed-Huffman body
// would be larger than one stored block, the stored block is written.  A second kernel
// compacts the window's members into one contiguous stream for the copy to the host.
//
// Inflate (one CTA per member): warp 0 decodes into shared memory (every lane runs the same
// bit reader; matches and stored blocks are copied by all 32 lanes), then the CTA checks
// the CRC-32 and ISIZE and only then writes the slice into the column.  Every read of the
// compressed window and every write of the slice is bounds-checked; a malformed member
// sets its status word and the CTA returns normally.
//
// Scratch is a fixed window of kWindow members, double-buffered on both sides, so the host's
// file I/O for one window overlaps the device work on the next.
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <cerrno>
#include <algorithm>
#include <climits>
#include <vector>

#include "common.cuh"
#include "replay.cuh"

namespace b2r {
namespace {

constexpr int kSlice = 65280;           // column bytes per member
constexpr int kSlot = 65536;            // bytes a member may take (BSIZE is 16 bits)
constexpr int kHeader = 18;             // gzip header with the 6-byte 'BC' extra field
constexpr int kTrailer = 8;             // CRC-32, ISIZE
constexpr int kWindow = 1024;           // members per window (64 MB of column bytes)
constexpr int kThreads = 128;           // compress / inflate CTA
constexpr int kSub = kSlice / kThreads; // 510 bytes parsed by one thread
constexpr int kEpochs = 8;
constexpr int kEpoch = kSlice / kEpochs;  // 8160 bytes
constexpr int kHashBits = 11;
constexpr int kHashSize = 1 << kHashBits;
constexpr int kMaxMatch = 258;
constexpr int kMaxDist = 32768;
constexpr uint32_t kCrcPoly = 0xEDB88320u;  // reflected CRC-32 (RFC 1952)

// Per-member status of the inflate kernel (0 = the member is good).
enum : int32_t {
  kBadHeader = 1, kBadBlockType, kBadCode, kBadDistance, kOutputOverrun, kInputOverrun,
  kBadStored, kBadEnd, kBadSize, kBadCrc, kMismatch,
};
const char *status_text(int32_t s) {
  switch (s) {
    case kBadHeader: return "bad member header";
    case kBadBlockType: return "block type other than stored or fixed Huffman";
    case kBadCode: return "invalid fixed-Huffman code";
    case kBadDistance: return "match distance reaches before the member";
    case kOutputOverrun: return "member inflates past its slice";
    case kInputOverrun: return "deflate stream runs past the member";
    case kBadStored: return "stored block length check failed";
    case kBadEnd: return "deflate stream does not end at the trailer";
    case kBadSize: return "ISIZE / inflated size differs from the slice";
    case kBadCrc: return "CRC-32 mismatch";
    case kMismatch: return "inflated member differs from the column";
    default: return "unknown status";
  }
}

// Deflate's length and distance tables (RFC 1951 3.2.5).
__constant__ uint16_t c_len_base[29] = {3,  4,  5,  6,  7,  8,  9,  10, 11,  13,
                                        15, 17, 19, 23, 27, 31, 35, 43, 51,  59,
                                        67, 83, 99, 115, 131, 163, 195, 227, 258};
__constant__ uint8_t c_len_extra[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2,
                                        2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
__constant__ uint16_t c_dist_base[30] = {1,    2,    3,    4,    5,    7,     9,     13,
                                         17,   25,   33,   49,   65,   97,    129,   193,
                                         257,  385,  513,  769,  1025, 1537,  2049,  3073,
                                         4097, 6145, 8193, 12289, 16385, 24577};
__constant__ uint8_t c_dist_extra[30] = {0, 0, 0, 0, 1, 1, 2, 2,  3,  3,  4,  4,  5,  5,  6,
                                         6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};

// ---- CRC-32 ------------------------------------------------------------------------------
__device__ void crc_table_init(uint32_t *table) {
  for (int i = threadIdx.x; i < 256; i += blockDim.x) {
    uint32_t c = (uint32_t)i;
    for (int k = 0; k < 8; ++k) c = c & 1 ? (c >> 1) ^ kCrcPoly : c >> 1;
    table[i] = c;
  }
}
// a * b modulo the CRC polynomial, reflected bit order (zlib's multmodp).
__device__ __forceinline__ uint32_t multmodp(uint32_t a, uint32_t b) {
  uint32_t m = 1u << 31, p = 0;
  for (;;) {
    if (a & m) {
      p ^= b;
      if ((a & (m - 1)) == 0) break;
    }
    m >>= 1;
    b = b & 1 ? (b >> 1) ^ kCrcPoly : b >> 1;
  }
  return p;
}
// x^(8 * n) modulo the polynomial: the operator that appends n zero bytes.
__device__ uint32_t x8nmodp(uint32_t n) {
  uint32_t p = 1u << 31;   // x^0
  uint32_t sq = 1u << 23;  // x^8
  while (n) {
    if (n & 1) p = multmodp(sq, p);
    sq = multmodp(sq, sq);
    n >>= 1;
  }
  return p;
}
// CRC-32 of buf[0, n) computed by the whole CTA: every thread takes one contiguous slice,
// its standard CRC is shifted past the bytes that follow the slice, and the shifted values
// XOR together (crc(A || B) = crc(A) * x^(8|B|) ^ crc(B)).  `red`: kThreads / 32 words.
__device__ uint32_t block_crc32(const uint8_t *buf, int n, const uint32_t *table,
                                uint32_t *red) {
  const int per = (n + kThreads - 1) / kThreads;
  const int lo = min(n, (int)threadIdx.x * per), hi = min(n, lo + per);
  uint32_t c = 0xFFFFFFFFu;
  for (int i = lo; i < hi; ++i) c = table[(c ^ buf[i]) & 0xFF] ^ (c >> 8);
  uint32_t part = hi > lo ? multmodp(x8nmodp((uint32_t)(n - hi)), ~c) : 0u;
  for (int o = 16; o; o >>= 1) part ^= __shfl_xor_sync(0xFFFFFFFFu, part, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = part;
  __syncthreads();
  uint32_t all = 0;
  for (int w = 0; w < kThreads / 32; ++w) all ^= red[w];
  __syncthreads();
  return all;  // CRC-32 of the empty string is 0, which no thread adds
}

// ---- compress ----------------------------------------------------------------------------
__device__ __forceinline__ uint32_t hash3(const uint8_t *p) {
  const uint32_t v = (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16);
  return (v * 2654435761u) >> (32 - kHashBits);
}

struct Token {
  int len;   // 0: literal
  int dist;
};

// The longest match for position p (end: the thread's sub-range end); len 0 when none.
__device__ __forceinline__ Token find_match(const uint8_t *data, int p, int end,
                                            const uint32_t *table) {
  Token best = {0, 0};
  const int limit = min(kMaxMatch, end - p);
  if (limit < 3) return best;
  const int e = p / kEpoch;
  const uint32_t h = hash3(data + p);
  int cand[4];
  cand[0] = p - 1;
  cand[1] = (int)table[e * kHashSize + h] - 1;
  cand[2] = e >= 1 ? (int)table[(e - 1) * kHashSize + h] - 1 : -1;
  cand[3] = e >= 2 ? (int)table[(e - 2) * kHashSize + h] - 1 : -1;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int c = cand[k];
    if (c < 0 || c >= p || p - c > kMaxDist) continue;
    int l = 0;
    while (l < limit && data[c + l] == data[p + l]) ++l;
    if (l > best.len) {
      best.len = l;
      best.dist = p - c;
    }
  }
  if (best.len < 3) best.len = 0;
  return best;
}

// Fixed-Huffman code fields of a token: calls put(value, bits) in stream order.
template <typename Put>
__device__ __forceinline__ void emit_literal(uint32_t lit, Put &put) {
  if (lit < 144) put(__brev(0x30u + lit) >> 24, 8);
  else put(__brev(0x190u + lit - 144) >> 23, 9);
}
template <typename Put>
__device__ __forceinline__ void emit_match(int len, int dist, Put &put) {
  int code, extra_bits = 0, extra = 0;
  const int ll = len - 3;
  if (len == 258) {
    code = 285;
  } else if (ll < 8) {
    code = 257 + ll;
  } else {
    const int nb = 31 - __clz(ll);
    code = 257 + 4 * (nb - 1) + ((ll >> (nb - 2)) & 3);
    extra_bits = nb - 2;
    extra = ll & ((1 << extra_bits) - 1);
  }
  if (code <= 279) put(__brev((uint32_t)(code - 256)) >> 25, 7);
  else put(__brev(0xC0u + (uint32_t)(code - 280)) >> 24, 8);
  if (extra_bits) put((uint32_t)extra, extra_bits);
  const int dd = dist - 1;
  int dcode, dbits = 0, dextra = 0;
  if (dd < 4) {
    dcode = dd;
  } else {
    const int nb = 31 - __clz(dd);
    dcode = 2 * nb + ((dd >> (nb - 1)) & 1);
    dbits = nb - 1;
    dextra = dd & ((1 << dbits) - 1);
  }
  put(__brev((uint32_t)dcode) >> 27, 5);
  if (dbits) put((uint32_t)dextra, dbits);
}

// Greedy parse of data[lo, hi) (matches end at hi): put() receives the codes.
template <typename Put>
__device__ void parse_range(const uint8_t *data, int lo, int hi, const uint32_t *table,
                            Put &put) {
  int p = lo;
  while (p < hi) {
    const Token t = find_match(data, p, hi, table);
    if (t.len) {
      emit_match(t.len, t.dist, put);
      p += t.len;
    } else {
      emit_literal(data[p], put);
      ++p;
    }
  }
}

struct BitCounter {
  int64_t bits = 0;
  __device__ __forceinline__ void operator()(uint32_t, int n) { bits += n; }
};

// Writes bits LSB-first into shared words starting at an arbitrary bit; the first and last
// words are shared with the neighbouring threads, hence atomicOr.
struct BitWriter {
  uint32_t *words;
  int word;
  int nbits;
  uint64_t acc;
  __device__ BitWriter(uint32_t *w, int64_t bitpos)
      : words(w), word((int)(bitpos >> 5)), nbits((int)(bitpos & 31)), acc(0) {}
  __device__ __forceinline__ void operator()(uint32_t v, int n) {
    acc |= (uint64_t)v << nbits;
    nbits += n;
    if (nbits >= 32) {
      atomicOr(&words[word++], (uint32_t)acc);
      acc >>= 32;
      nbits -= 32;
    }
  }
  __device__ __forceinline__ void finish() {
    if (nbits > 0) atomicOr(&words[word], (uint32_t)acc);
  }
};

constexpr size_t kDeflateSmem = (size_t)kSlice + 16 + kSlot +
                                (size_t)kEpochs * kHashSize * 4 + 256 * 4;

// One CTA per member: column bytes [(first + blockIdx.x) * kSlice, ...) -> a complete gzip
// member at scratch + blockIdx.x * kSlot, its size in sizes[blockIdx.x].
__global__ void __launch_bounds__(kThreads)
ckpt_deflate_kernel(const uint8_t *__restrict__ col, int64_t col_bytes, int64_t first,
                    uint8_t *__restrict__ scratch, int32_t *__restrict__ sizes) {
  extern __shared__ __align__(128) uint8_t smem[];
  uint8_t *data = smem;                                          // kSlice + 16
  uint8_t *out = smem + kSlice + 16;                             // kSlot (member image)
  uint32_t *out_words = reinterpret_cast<uint32_t *>(out);
  uint32_t *table = reinterpret_cast<uint32_t *>(out + kSlot);   // kEpochs x kHashSize
  uint32_t *crc_tab = table + kEpochs * kHashSize;               // 256
  __shared__ __align__(8) uint64_t bar;
  __shared__ int64_t s_scan[kThreads / 32];
  __shared__ uint32_t s_red[kThreads / 32];

  const int64_t start = (first + blockIdx.x) * (int64_t)kSlice;
  const int n = (int)min((int64_t)kSlice, col_bytes - start);
  const uint8_t *src = col + start;
  const int bulk = n & ~15;
  const bool use_bulk = ((uintptr_t)src & 15) == 0 && bulk > 0;
  if (threadIdx.x == 0 && use_bulk) {
    mbar_init(&bar, 1);
    mbar_arrive_expect(&bar, (uint32_t)bulk);
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
        ::"r"(smem_u32(data)), "l"(src), "r"((uint32_t)bulk), "r"(smem_u32(&bar))
        : "memory");
  }
  for (int i = (use_bulk ? bulk : 0) + threadIdx.x; i < n + 16; i += kThreads)
    data[i] = i < n ? src[i] : 0;
  for (int i = threadIdx.x; i < kSlot / 4; i += kThreads) out_words[i] = 0;
  for (int i = threadIdx.x; i < kEpochs * kHashSize; i += kThreads) table[i] = 0;
  crc_table_init(crc_tab);
  __syncthreads();
  if (use_bulk) mbar_wait(&bar, 0);

  // every position with three bytes left, latest one per hash and epoch
  for (int p = threadIdx.x; p + 3 <= n; p += kThreads)
    atomicMax(&table[(p / kEpoch) * kHashSize + hash3(data + p)], (uint32_t)(p + 1));
  __syncthreads();

  const int lo = min(n, (int)threadIdx.x * kSub), hi = min(n, lo + kSub);
  BitCounter count;
  parse_range(data, lo, hi, table, count);
  // exclusive scan of the threads' bit counts
  int64_t incl = count.bits;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int o = 1; o < 32; o <<= 1) {
    const int64_t v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) s_scan[warp] = incl;
  __syncthreads();
  int64_t before = 0, total = 0;
  for (int w = 0; w < kThreads / 32; ++w) {
    if (w < warp) before += s_scan[w];
    total += s_scan[w];
  }
  const int64_t excl = before + incl - count.bits;
  const int64_t body_bits = 3 + total + 7;  // block header, codes, end of block
  const int fixed_bytes = (int)((body_bits + 7) >> 3);
  const int stored_bytes = 5 + n;
  const bool fixed = fixed_bytes <= stored_bytes;
  const int body = fixed ? fixed_bytes : stored_bytes;

  if (fixed) {
    BitWriter wr(out_words, (int64_t)kHeader * 8 + 3 + excl);
    parse_range(data, lo, hi, table, wr);
    wr.finish();
    if (threadIdx.x == 0) atomicOr(&out_words[kHeader / 4], 3u << ((kHeader % 4) * 8));
    // (BFINAL = 1, BTYPE = 01; the end-of-block code is seven zero bits)
  } else {
    for (int i = threadIdx.x; i < n; i += kThreads) out[kHeader + 5 + i] = data[i];
  }
  const uint32_t crc = block_crc32(data, n, crc_tab, s_red);  // (has __syncthreads)
  const int size = kHeader + body + kTrailer;
  if (threadIdx.x == 0) {
    const uint8_t head[kHeader] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 255, 6, 0, 'B', 'C', 2, 0,
                                   (uint8_t)(size - 1), (uint8_t)((size - 1) >> 8)};
    for (int i = 0; i < kHeader; ++i) out[i] = head[i];
    if (!fixed) {
      out[kHeader] = 1;  // BFINAL = 1, BTYPE = 00
      out[kHeader + 1] = (uint8_t)n;
      out[kHeader + 2] = (uint8_t)(n >> 8);
      out[kHeader + 3] = (uint8_t)~n;
      out[kHeader + 4] = (uint8_t)(~n >> 8);
    }
    uint8_t *t = out + kHeader + body;
    for (int i = 0; i < 4; ++i) t[i] = (uint8_t)(crc >> (8 * i));
    for (int i = 0; i < 4; ++i) t[4 + i] = (uint8_t)((uint32_t)n >> (8 * i));
    sizes[blockIdx.x] = size;
  }
  __syncthreads();
  uint4 *dst = reinterpret_cast<uint4 *>(scratch + (int64_t)blockIdx.x * kSlot);
  const uint4 *img = reinterpret_cast<const uint4 *>(out);
  for (int i = threadIdx.x; i < (size + 15) / 16; i += kThreads) dst[i] = img[i];
}

// Member b of the window moves from its slot to offsets[b] = sizes[0] + ... + sizes[b-1]
// of one contiguous stream; the last CTA also writes the stream's length.
__global__ void __launch_bounds__(256)
ckpt_compact_kernel(const uint8_t *__restrict__ scratch, const int32_t *__restrict__ sizes,
                    uint8_t *__restrict__ stream, int64_t *__restrict__ offsets,
                    int64_t *__restrict__ total) {
  __shared__ int64_t s_red[8];
  int64_t part = 0;
  for (int i = threadIdx.x; i < (int)blockIdx.x; i += 256) part += sizes[i];
  for (int o = 16; o; o >>= 1) part += __shfl_xor_sync(0xFFFFFFFFu, part, o);
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = part;
  __syncthreads();
  int64_t off = 0;
  for (int w = 0; w < 8; ++w) off += s_red[w];
  const int size = sizes[blockIdx.x];
  const uint8_t *src = scratch + (int64_t)blockIdx.x * kSlot;
  uint8_t *dst = stream + off;
  for (int i = threadIdx.x; i < size; i += 256) dst[i] = src[i];
  if (threadIdx.x == 0) {
    offsets[blockIdx.x] = off;
    if (blockIdx.x == gridDim.x - 1) *total = off + size;
  }
}

// ---- inflate -----------------------------------------------------------------------------
// LSB-first bit reader over in[pos, end); every lane of the decoding warp runs one.
struct BitReader {
  const uint8_t *in;
  int64_t pos, end;
  uint64_t buf;
  int avail;
  __device__ __forceinline__ void refill() {
    while (avail <= 56 && pos < end) {
      buf |= (uint64_t)in[pos++] << avail;
      avail += 8;
    }
  }
  // next n bits (n <= 16) without consuming; missing bits read as zero
  __device__ __forceinline__ uint32_t peek(int n) {
    refill();
    return (uint32_t)(buf & ((1ull << n) - 1));
  }
  __device__ __forceinline__ bool drop(int n) {  // false: the stream ran out
    if (n > avail) return false;
    buf >>= n;
    avail -= n;
    return true;
  }
  __device__ __forceinline__ bool bits(int n, uint32_t *v) {
    *v = peek(n);
    return drop(n);
  }
  // byte position of the next unread whole byte (after aligning to a byte boundary)
  __device__ __forceinline__ int64_t align() {
    const int skip = avail & 7;
    buf >>= skip;
    avail -= skip;
    return pos - avail / 8;
  }
  __device__ __forceinline__ void seek(int64_t p) {
    pos = p;
    buf = 0;
    avail = 0;
  }
};

// Inflates in[lo, hi) (a member's deflate body) into out (cap bytes) with the 32 lanes of
// one warp.  Returns 0 and sets *out_len / *end_pos, or a status.
__device__ int32_t inflate_warp(const uint8_t *in, int64_t lo, int64_t hi, uint8_t *out,
                                int cap, int *out_len, int64_t *end_pos) {
  const int lane = threadIdx.x & 31;
  BitReader br = {in, lo, hi, 0, 0};
  int o = 0;
  for (;;) {
    uint32_t head;
    if (!br.bits(3, &head)) return kInputOverrun;
    const uint32_t type = head >> 1;
    if (type == 0) {
      const int64_t p = br.align();
      if (p + 4 > hi) return kInputOverrun;
      const uint32_t len = in[p] | (in[p + 1] << 8);
      const uint32_t nlen = in[p + 2] | (in[p + 3] << 8);
      if ((len ^ nlen) != 0xFFFFu) return kBadStored;
      if (p + 4 + len > hi) return kInputOverrun;
      if (o + (int)len > cap) return kOutputOverrun;
      for (uint32_t i = lane; i < len; i += 32) out[o + i] = in[p + 4 + i];
      __syncwarp();
      o += (int)len;
      br.seek(p + 4 + len);
    } else if (type == 1) {
      for (;;) {
        const uint32_t code9 = __brev(br.peek(9)) >> 23;  // first nine code bits, MSB first
        uint32_t sym;
        int nb;
        if ((code9 >> 2) <= 23) {
          sym = 256 + (code9 >> 2), nb = 7;
        } else if ((code9 >> 1) <= 191) {
          sym = (code9 >> 1) - 48, nb = 8;
        } else if ((code9 >> 1) <= 199) {
          sym = 280 + (code9 >> 1) - 192, nb = 8;
        } else {
          sym = 144 + code9 - 400, nb = 9;
        }
        if (!br.drop(nb)) return kInputOverrun;
        if (sym < 256) {
          if (o >= cap) return kOutputOverrun;
          if (lane == 0) out[o] = (uint8_t)sym;
          __syncwarp();
          ++o;
          continue;
        }
        if (sym == 256) break;
        if (sym > 285) return kBadCode;
        uint32_t x;
        if (!br.bits(c_len_extra[sym - 257], &x)) return kInputOverrun;
        const int len = c_len_base[sym - 257] + (int)x;
        const uint32_t dcode = __brev(br.peek(5)) >> 27;
        if (!br.drop(5)) return kInputOverrun;
        if (dcode > 29) return kBadCode;
        if (!br.bits(c_dist_extra[dcode], &x)) return kInputOverrun;
        const int dist = c_dist_base[dcode] + (int)x;
        if (dist > o) return kBadDistance;
        if (o + len > cap) return kOutputOverrun;
        // out[o + i] = out[o + i - dist], unrolled: every byte comes from before o
        for (int i = lane; i < len; i += 32) out[o + i] = out[o - dist + (i < dist ? i : i % dist)];
        __syncwarp();
        o += len;
      }
    } else {
      return kBadBlockType;
    }
    if (head & 1) break;
  }
  *out_len = o;
  *end_pos = br.align();
  return 0;
}

constexpr size_t kInflateSmem = (size_t)kSlice + 256 * 4;

// mode: 0 write the slice into the column, 1 check only, 2 compare with the column.
// in / in_bytes: the window's compressed bytes; member b is in[offsets[b], + sizes[b]) and
// covers column bytes [(first + b) * kSlice, ...).
__global__ void __launch_bounds__(kThreads)
ckpt_inflate_kernel(const uint8_t *__restrict__ in, int64_t in_bytes,
                    const int64_t *__restrict__ offsets, const int32_t *__restrict__ sizes,
                    int64_t first, uint8_t *__restrict__ col, int64_t col_bytes, int mode,
                    int32_t *__restrict__ status) {
  extern __shared__ __align__(128) uint8_t smem[];
  uint8_t *out = smem;
  uint32_t *crc_tab = reinterpret_cast<uint32_t *>(smem + kSlice);
  __shared__ int32_t s_status, s_len;
  __shared__ uint32_t s_red[kThreads / 32];
  crc_table_init(crc_tab);
  const int64_t start = (first + blockIdx.x) * (int64_t)kSlice;
  const int n = (int)min((int64_t)kSlice, col_bytes - start);
  const int64_t off = offsets[blockIdx.x];
  const int64_t size = sizes[blockIdx.x];
  if (threadIdx.x < 32) {
    int32_t st = 0;
    int len = 0;
    int64_t end = 0;
    if (off < 0 || size < kHeader + kTrailer || off + size > in_bytes) {
      st = kBadHeader;
    } else {
      const uint8_t *m = in + off;
      if (m[0] != 0x1f || m[1] != 0x8b || m[2] != 8 || m[3] != 4 || m[10] != 6 || m[11] != 0 ||
          m[12] != 'B' || m[13] != 'C' || m[14] != 2 || m[15] != 0 ||
          (int64_t)(m[16] | (m[17] << 8)) != size - 1)
        st = kBadHeader;
      else
        st = inflate_warp(in, off + kHeader, off + size - kTrailer, out, n, &len, &end);
      if (st == 0 && end != off + size - kTrailer) st = kBadEnd;
      if (st == 0) {
        const uint8_t *t = in + off + size - kTrailer;
        const uint32_t isize = t[4] | (t[5] << 8) | (t[6] << 16) | ((uint32_t)t[7] << 24);
        if (len != n || isize != (uint32_t)n) st = kBadSize;
      }
    }
    if (threadIdx.x == 0) {
      s_status = st;
      s_len = len;
    }
  }
  __syncthreads();
  int32_t st = s_status;
  if (st == 0) {
    const uint8_t *t = in + off + size - kTrailer;
    const uint32_t want = t[0] | (t[1] << 8) | (t[2] << 16) | ((uint32_t)t[3] << 24);
    if (block_crc32(out, s_len, crc_tab, s_red) != want) st = kBadCrc;
  }
  if (st == 0 && mode == 0) {
    uint8_t *dst = col + start;
    for (int i = threadIdx.x; i < n; i += kThreads) dst[i] = out[i];
  } else if (st == 0 && mode == 2) {
    __shared__ int s_diff;
    if (threadIdx.x == 0) s_diff = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += kThreads)
      if (out[i] != col[start + i]) s_diff = 1;
    __syncthreads();
    if (s_diff) st = kMismatch;
  }
  if (threadIdx.x == 0) status[blockIdx.x] = st;
}

// ---- host side ---------------------------------------------------------------------------
// (per call: the attribute belongs to the current device)
int set_smem_limits() {
  B2R_TRY(allow_dynamic_smem(ckpt_deflate_kernel, (int)kDeflateSmem));
  return allow_dynamic_smem(ckpt_inflate_kernel, (int)kInflateSmem);
}

// Device and pinned allocations of one call, released on every return path.
struct Scratch {
  std::vector<void *> dev, host;
  std::vector<cudaEvent_t> events;
  cudaStream_t copy = nullptr;
  ~Scratch() {
    if (copy) cudaStreamSynchronize(copy);
    for (cudaEvent_t e : events) cudaEventSynchronize(e);
    for (void *p : dev) cudaFree(p);
    for (void *p : host) cudaFreeHost(p);
    for (cudaEvent_t e : events) cudaEventDestroy(e);
    if (copy) cudaStreamDestroy(copy);
  }
  template <typename T>
  int device(T **p, size_t bytes) {
    B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(p), bytes));
    dev.push_back(*p);
    return B2R_OK;
  }
  template <typename T>
  int pinned(T **p, size_t bytes) {
    B2R_CUDA(cudaHostAlloc(reinterpret_cast<void **>(p), bytes, cudaHostAllocDefault));
    host.push_back(*p);
    return B2R_OK;
  }
  int event(cudaEvent_t *e) {
    B2R_CUDA(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
    events.push_back(*e);
    return B2R_OK;
  }
};

int check_statuses(const int32_t *st, int count, int64_t first) {
  for (int i = 0; i < count; ++i)
    if (st[i] != 0)
      return fail(B2R_ERR_INVALID_ARGUMENT, "checkpoint member %lld: %s",
                  (long long)(first + i + 1), status_text(st[i]));
  return B2R_OK;
}

int write_all(int fd, const uint8_t *p, int64_t n) {
  while (n > 0) {
    const ssize_t w = ::write(fd, p, (size_t)n);
    if (w < 0) {
      if (errno == EINTR) continue;
      return fail(B2R_ERR_INVALID_ARGUMENT, "checkpoint write failed: %s", strerror(errno));
    }
    p += w;
    n -= w;
  }
  return B2R_OK;
}

int64_t read_at(int fd, uint8_t *p, int64_t n, int64_t at) {
  int64_t got = 0;
  while (got < n) {
    const ssize_t r = ::pread(fd, p + got, (size_t)(n - got), (off_t)(at + got));
    if (r < 0) {
      if (errno == EINTR) continue;
      return -1;
    }
    if (r == 0) break;
    got += r;
  }
  return got;
}

int column_of(b2r_buffer *b, int32_t column, uint8_t **dev, int64_t *bytes) {
  if (column < 0 || column >= b->num_columns)
    return fail(B2R_ERR_INVALID_ARGUMENT, "no store column %d", column);
  *dev = b->col[column].dev;
  *bytes = b->cfg.capacity * b->col[column].row_bytes;
  return B2R_OK;
}

}  // namespace
}  // namespace b2r

using b2r::fail;

int b2r_ckpt_save_column(b2r_buffer *b, int32_t column, int32_t fd, int32_t verify_only,
                         int64_t *bytes_out, b2r_stream stream) {
  using namespace b2r;
  uint8_t *col;
  int64_t col_bytes;
  B2R_TRY(column_of(b, column, &col, &col_bytes));
  if (!verify_only && fd < 0) return fail(B2R_ERR_INVALID_ARGUMENT, "bad file descriptor");
  cudaStream_t s = as_stream(stream);
  B2R_TRY(flush_queue(b, s));
  B2R_TRY(set_smem_limits());
  const int64_t members = (col_bytes + kSlice - 1) / kSlice;
  const int win = (int)std::min<int64_t>(kWindow, std::max<int64_t>(members, 1));
  Scratch sc;
  uint8_t *slots, *dstream[2], *hstream[2] = {nullptr, nullptr};
  int32_t *sizes, *dstatus[2], *hstatus[2];
  int64_t *offsets[2], *dtotal[2], *htotal[2];
  cudaEvent_t ev_done[2];
  B2R_TRY(sc.device(&slots, (size_t)win * kSlot));
  B2R_TRY(sc.device(&sizes, (size_t)win * 4));
  B2R_CUDA(cudaStreamCreateWithFlags(&sc.copy, cudaStreamNonBlocking));
  for (int k = 0; k < 2; ++k) {
    B2R_TRY(sc.device(&dstream[k], (size_t)win * kSlot));
    B2R_TRY(sc.device(&offsets[k], (size_t)win * 8));
    B2R_TRY(sc.device(&dtotal[k], 8));
    B2R_TRY(sc.device(&dstatus[k], (size_t)win * 4));
    B2R_TRY(sc.pinned(&htotal[k], 8));
    B2R_TRY(sc.pinned(&hstatus[k], (size_t)win * 4));
    if (!verify_only) B2R_TRY(sc.pinned(&hstream[k], (size_t)win * kSlot));
    B2R_TRY(sc.event(&ev_done[k]));
  }
  const int64_t windows = (members + win - 1) / win;
  int64_t written = 0;
  // window j's stream is ready on the device: copy it out beside the next window's kernels
  // and append it to the file
  auto finish = [&](int64_t j) -> int {
    const int k = (int)(j & 1);
    const int count = (int)std::min<int64_t>(win, members - j * win);
    B2R_CUDA(cudaEventSynchronize(ev_done[k]));
    const int64_t n = *htotal[k];
    if (verify_only) {
      B2R_TRY(check_statuses(hstatus[k], count, j * win));
    } else {
      B2R_CUDA(cudaMemcpyAsync(hstream[k], dstream[k], (size_t)n, cudaMemcpyDeviceToHost,
                               sc.copy));
      B2R_CUDA(cudaStreamSynchronize(sc.copy));
      B2R_TRY(write_all(fd, hstream[k], n));
    }
    written += n;
    return B2R_OK;
  };
  for (int64_t w = 0; w < windows; ++w) {
    const int k = (int)(w & 1);
    const int count = (int)std::min<int64_t>(win, members - w * win);
    ckpt_deflate_kernel<<<count, kThreads, kDeflateSmem, s>>>(col, col_bytes, w * win, slots,
                                                               sizes);
    B2R_LAUNCHED();
    ckpt_compact_kernel<<<count, 256, 0, s>>>(slots, sizes, dstream[k], offsets[k],
                                               dtotal[k]);
    B2R_LAUNCHED();
    if (verify_only) {
      // inflate the stream just made and compare it with the column
      ckpt_inflate_kernel<<<count, kThreads, kInflateSmem, s>>>(
          dstream[k], (int64_t)win * kSlot, offsets[k], sizes, w * win, col, col_bytes, 2,
          dstatus[k]);
      B2R_LAUNCHED();
      B2R_CUDA(cudaMemcpyAsync(hstatus[k], dstatus[k], (size_t)count * 4,
                               cudaMemcpyDeviceToHost, s));
    }
    B2R_CUDA(cudaMemcpyAsync(htotal[k], dtotal[k], 8, cudaMemcpyDeviceToHost, s));
    B2R_CUDA(cudaEventRecord(ev_done[k], s));
    if (w >= 1) B2R_TRY(finish(w - 1));
  }
  if (windows >= 1) B2R_TRY(finish(windows - 1));
  if (bytes_out) *bytes_out = written;
  return B2R_OK;
}

int b2r_ckpt_load_column(b2r_buffer *b, int32_t column, int32_t fd, int64_t offset,
                         int32_t verify_only, b2r_stream stream) {
  using namespace b2r;
  uint8_t *col;
  int64_t col_bytes;
  B2R_TRY(column_of(b, column, &col, &col_bytes));
  if (fd < 0 || offset < 0) return fail(B2R_ERR_INVALID_ARGUMENT, "bad file descriptor");
  struct stat stbuf;
  if (fstat(fd, &stbuf) != 0)
    return fail(B2R_ERR_INVALID_ARGUMENT, "checkpoint stat failed: %s", strerror(errno));
  const int64_t file_bytes = (int64_t)stbuf.st_size;
  cudaStream_t s = as_stream(stream);
  B2R_TRY(flush_queue(b, s));
  B2R_TRY(set_smem_limits());
  const int64_t members = (col_bytes + kSlice - 1) / kSlice;
  const int win = (int)std::min<int64_t>(kWindow, std::max<int64_t>(members, 1));
  const int64_t chunk = (int64_t)win * kSlot;  // a window of the largest members
  Scratch sc;
  uint8_t *din[2], *hin[2];
  int64_t *doff[2], *hoff[2];
  int32_t *dsize[2], *hsize[2], *dstatus[2], *hstatus[2];
  cudaEvent_t ev_done[2];
  int64_t win_first[2] = {0, 0};
  int win_count[2] = {0, 0};
  for (int k = 0; k < 2; ++k) {
    B2R_TRY(sc.device(&din[k], (size_t)chunk));
    B2R_TRY(sc.device(&doff[k], (size_t)win * 8));
    B2R_TRY(sc.device(&dsize[k], (size_t)win * 4));
    B2R_TRY(sc.device(&dstatus[k], (size_t)win * 4));
    B2R_TRY(sc.pinned(&hin[k], (size_t)chunk));
    B2R_TRY(sc.pinned(&hoff[k], (size_t)win * 8));
    B2R_TRY(sc.pinned(&hsize[k], (size_t)win * 4));
    B2R_TRY(sc.pinned(&hstatus[k], (size_t)win * 4));
    B2R_TRY(sc.event(&ev_done[k]));
  }
  bool pending[2] = {false, false};
  auto retire = [&](int k) -> int {
    if (!pending[k]) return B2R_OK;
    B2R_CUDA(cudaEventSynchronize(ev_done[k]));
    pending[k] = false;
    return check_statuses(hstatus[k], win_count[k], win_first[k]);
  };
  int64_t pos = offset, done = 0;
  for (int64_t w = 0; done < members; ++w) {
    const int k = (int)(w & 1);
    B2R_TRY(retire(k));  // the pinned buffers of window w - 2 are free again
    const int64_t got = read_at(fd, hin[k], std::min(chunk, file_bytes - pos), pos);
    if (got < 0) return fail(B2R_ERR_INVALID_ARGUMENT, "checkpoint read failed: %s",
                             strerror(errno));
    // walk the BGZF headers: whole members of this chunk
    int count = 0;
    int64_t q = 0;
    while (count < win && done + count < members) {
      if (q + kHeader > got) break;
      const uint8_t *m = hin[k] + q;
      if (m[0] != 0x1f || m[1] != 0x8b || m[2] != 8 || m[3] != 4 || m[10] != 6 || m[11] != 0 ||
          m[12] != 'B' || m[13] != 'C' || m[14] != 2 || m[15] != 0)
        return fail(B2R_ERR_INVALID_ARGUMENT, "checkpoint member %lld: %s",
                    (long long)(done + count + 1), status_text(kBadHeader));
      const int64_t size = (int64_t)(m[16] | (m[17] << 8)) + 1;
      if (size < kHeader + kTrailer)
        return fail(B2R_ERR_INVALID_ARGUMENT, "checkpoint member %lld: %s",
                    (long long)(done + count + 1), status_text(kBadHeader));
      if (q + size > got) break;
      hoff[k][count] = q;
      hsize[k][count] = (int32_t)size;
      ++count;
      q += size;
    }
    if (count == 0)
      return fail(B2R_ERR_INVALID_ARGUMENT,
                  "checkpoint truncated: %lld of %lld data members present",
                  (long long)done, (long long)members);
    B2R_CUDA(cudaMemcpyAsync(din[k], hin[k], (size_t)q, cudaMemcpyHostToDevice, s));
    B2R_CUDA(cudaMemcpyAsync(doff[k], hoff[k], (size_t)count * 8, cudaMemcpyHostToDevice, s));
    B2R_CUDA(cudaMemcpyAsync(dsize[k], hsize[k], (size_t)count * 4, cudaMemcpyHostToDevice, s));
    ckpt_inflate_kernel<<<count, kThreads, kInflateSmem, s>>>(
        din[k], q, doff[k], dsize[k], done, col, col_bytes, verify_only ? 1 : 0, dstatus[k]);
    B2R_LAUNCHED();
    B2R_CUDA(cudaMemcpyAsync(hstatus[k], dstatus[k], (size_t)count * 4,
                             cudaMemcpyDeviceToHost, s));
    B2R_CUDA(cudaEventRecord(ev_done[k], s));
    pending[k] = true;
    win_first[k] = done;
    win_count[k] = count;
    done += count;
    pos += q;
  }
  B2R_TRY(retire(0));
  B2R_TRY(retire(1));
  if (pos != file_bytes)
    return fail(B2R_ERR_INVALID_ARGUMENT, "checkpoint has %lld bytes after its last member",
                (long long)(file_bytes - pos));
  if (!verify_only && column == B2R_COL_TERMINAL && b->cfg.capacity > 0)
    B2R_TRY(refresh_terminal_mirror(b, 0, b->cfg.capacity, s));
  return B2R_OK;
}
