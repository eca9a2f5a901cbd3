// Baseline JPEG encoding on the device (sm_100a): uint8 RGB [H, W, 3] -> one complete JFIF file (SOI ... EOI) and its
// byte count, both in device memory.  The format (ITU T.81):
//   SOF0, 8-bit, 3 components, YCbCr 4:2:0 (Y 2x2, Cb and Cr 1x1): one MCU is 16x16 pixels, blocks Y00 Y01 Y10 Y11 Cb Cr;
//   the Annex K.1 quantisation tables scaled by the IJG quality rule, the Annex K.3 Huffman tables, and a restart
//   marker (RST0..RST7 cycling) after every KP_JPEG_RESTART_MCUS MCUs, declared by DRI.
// The integer stages are libjpeg's: jccolor.c's 16-bit fixed-point RGB -> YCbCr, right / bottom edges replicated up to
// a whole MCU, h2v2_downsample with its rounding bias alternating 1, 2 along each chroma row.  The DCT is an fp32
// separable DCT-II of the level-shifted samples; each coefficient is quantised as roundf(coef / Q) (half away from 0).
//
// Restart markers make the scan's segments independent (the DC predictors reset at each), which is what lets the
// entropy coding run in parallel.  Three launches, no host synchronisation, no allocation (graph-capturable):
//   1. segment: one block per segment of R MCUs.  Colour conversion, downsampling, DCT and quantisation into shared
//               memory; one thread per 8x8 block counts its code length, a prefix sum gives each block its bit
//               offset, every block writes its bits into the segment's shared bit buffer, the tail is padded with
//               1-bits to a byte and the bytes go to the segment's fixed-size scratch slot with their 0xFF count;
//   2. scan:    one block: exclusive prefix sum of the stuffed segment sizes (+ 2 marker bytes each but the last),
//               the header copied in front, EOI behind, the file length;
//   3. pack:    one warp per segment: copies its bytes to their place, a 0x00 after every 0xFF, then its RSTm marker.
#include <algorithm>

#include "common.cuh"

namespace kp {

constexpr int kJpegR = KP_JPEG_RESTART_MCUS;
constexpr int kSegBlocks = 6 * kJpegR;    // 8x8 blocks per segment
constexpr int kSegThreads = 8 * kSegBlocks;  // one thread per block row (and column) in the DCT
constexpr int kPackThreads = 256;
constexpr int kScanThreads = 1024;

// Worst case of one block's entropy-coded bits.  DC: the longest DC code of K.3 for category 11 (the largest DC
// difference of 8-bit data, |diff| <= 2047) is 11 bits (chrominance; luminance 9), plus 11 magnitude bits = 22.  AC:
// at most 63 codes (each run/size code consumes at least one of the 63 AC coefficients, a ZRL consumes 16, an EOB is
// only sent when at least one trailing coefficient is zero and ends the block); each code is at most 16 bits (the
// longest K.3 code) plus at most 10 magnitude bits (|AC| <= 1023 for 8-bit data; the orthonormal DCT of level-shifted
// samples gives |AC| <= 128 * 8 * max_u(sum_x |cos((2x+1)u pi/16)|) / 8 < 930 even at Q = 1) = 26 bits.
constexpr int kMaxBlockBits = 22 + 63 * 26;
// A segment's bytes before stuffing: its bits rounded up to a byte (the 1-bit padding never adds a byte past that).
constexpr int kSegBytes = (kJpegR * 6 * kMaxBlockBits + 7) / 8;
constexpr int kSegWords = (kSegBytes + 3) / 4;  // the per-segment scratch slot and shared bit buffer
// Stuffing adds at most one 0x00 per byte, and every segment but the last is followed by a 2-byte RSTm marker, so a
// segment occupies at most 2 * kSegBytes + 2 bytes of the file.
constexpr int64_t kSegMaxFileBytes = 2 * (int64_t)kSegBytes + 2;

// ---- Annex K.3 Huffman tables (BITS: codes per length 1..16, HUFFVAL) and the derived code / length per symbol ----
constexpr uint8_t kDcLumBits[16] = {0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0};
constexpr uint8_t kDcChrBits[16] = {0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0};
constexpr uint8_t kDcVals[12] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11};
constexpr uint8_t kAcLumBits[16] = {0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d};
constexpr uint8_t kAcLumVals[162] = {
    0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71, 0x14,
    0x32, 0x81, 0x91, 0xa1, 0x08, 0x23, 0x42, 0xb1, 0xc1, 0x15, 0x52, 0xd1, 0xf0, 0x24, 0x33, 0x62, 0x72, 0x82, 0x09,
    0x0a, 0x16, 0x17, 0x18, 0x19, 0x1a, 0x25, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x34, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a,
    0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64, 0x65,
    0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88,
    0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9,
    0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca,
    0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe1, 0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea,
    0xf1, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa};
constexpr uint8_t kAcChrBits[16] = {0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77};
constexpr uint8_t kAcChrVals[162] = {
    0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22, 0x32,
    0x81, 0x08, 0x14, 0x42, 0x91, 0xa1, 0xb1, 0xc1, 0x09, 0x23, 0x33, 0x52, 0xf0, 0x15, 0x62, 0x72, 0xd1, 0x0a, 0x16,
    0x24, 0x34, 0xe1, 0x25, 0xf1, 0x17, 0x18, 0x19, 0x1a, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x35, 0x36, 0x37, 0x38, 0x39,
    0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64,
    0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x82, 0x83, 0x84, 0x85, 0x86,
    0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7,
    0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8,
    0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9,
    0xea, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa};

struct HuffCodes {
  uint16_t code[2][2][256];  // [dc / ac][luminance / chrominance][symbol]
  uint8_t len[2][2][256];
};

// T.81 Annex C: codes of increasing length, consecutive within a length, in HUFFVAL order
constexpr void derive_codes(HuffCodes& h, int kind, int tab, const uint8_t* bits, const uint8_t* vals) {
  int code = 0, k = 0;
  for (int l = 1; l <= 16; ++l) {
    for (int i = 0; i < bits[l - 1]; ++i, ++k, ++code) {
      h.code[kind][tab][vals[k]] = (uint16_t)code;
      h.len[kind][tab][vals[k]] = (uint8_t)l;
    }
    code <<= 1;
  }
}

constexpr HuffCodes make_codes() {
  HuffCodes h{};
  derive_codes(h, 0, 0, kDcLumBits, kDcVals);
  derive_codes(h, 0, 1, kDcChrBits, kDcVals);
  derive_codes(h, 1, 0, kAcLumBits, kAcLumVals);
  derive_codes(h, 1, 1, kAcChrBits, kAcChrVals);
  return h;
}

__constant__ HuffCodes c_huff = make_codes();

// zigzag position -> natural (row-major) index (T.81 Figure A.6)
constexpr uint8_t kNatural[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                  41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                  30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
// natural index -> zigzag position (its inverse)
__constant__ uint8_t c_zigzag[64] = {0,  1,  5,  6,  14, 15, 27, 28, 2,  4,  7,  13, 16, 26, 29, 42, 3,  8,  12, 17, 25, 30,
                                     41, 43, 9,  11, 18, 24, 31, 40, 44, 53, 10, 19, 23, 32, 39, 45, 52, 54, 20, 22, 33, 38,
                                     46, 51, 55, 60, 21, 34, 37, 47, 50, 56, 59, 61, 35, 36, 48, 49, 57, 58, 62, 63};

// the orthonormal 8-point DCT-II: c[u][x] = a(u) cos((2x+1) u pi / 16), a(0) = sqrt(1/8), a(u > 0) = 1/2
__constant__ float c_dct[64] = {
    3.535533906e-01f, 3.535533906e-01f,  3.535533906e-01f,  3.535533906e-01f,  3.535533906e-01f,  3.535533906e-01f,  3.535533906e-01f,  3.535533906e-01f,
    4.903926402e-01f, 4.157348062e-01f,  2.777851165e-01f,  9.754516101e-02f,  -9.754516101e-02f, -2.777851165e-01f, -4.157348062e-01f, -4.903926402e-01f,
    4.619397663e-01f, 1.913417162e-01f,  -1.913417162e-01f, -4.619397663e-01f, -4.619397663e-01f, -1.913417162e-01f, 1.913417162e-01f,  4.619397663e-01f,
    4.157348062e-01f, -9.754516101e-02f, -4.903926402e-01f, -2.777851165e-01f, 2.777851165e-01f,  4.903926402e-01f,  9.754516101e-02f,  -4.157348062e-01f,
    3.535533906e-01f, -3.535533906e-01f, -3.535533906e-01f, 3.535533906e-01f,  3.535533906e-01f,  -3.535533906e-01f, -3.535533906e-01f, 3.535533906e-01f,
    2.777851165e-01f, -4.903926402e-01f, 9.754516101e-02f,  4.157348062e-01f,  -4.157348062e-01f, -9.754516101e-02f, 4.903926402e-01f,  -2.777851165e-01f,
    1.913417162e-01f, -4.619397663e-01f, 4.619397663e-01f,  -1.913417162e-01f, -1.913417162e-01f, 4.619397663e-01f,  -4.619397663e-01f, 1.913417162e-01f,
    9.754516101e-02f, -2.777851165e-01f, 4.157348062e-01f,  -4.903926402e-01f, 4.903926402e-01f,  -4.157348062e-01f, 2.777851165e-01f,  -9.754516101e-02f};

// Annex K.1 quantisation tables, natural order
constexpr uint8_t kStdQuant[2][64] = {
    {16, 11, 10, 16, 24,  40,  51,  61,  12, 12, 14, 19, 26,  58,  60,  55,  14, 13, 16, 24, 40,  57,  69,  56,
     14, 17, 22, 29, 51,  87,  80,  62,  18, 22, 37, 56, 68,  109, 103, 77,  24, 35, 55, 64, 81,  104, 113, 92,
     49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99},
    {17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99, 99, 99, 47, 66, 99, 99,
     99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99,
     99, 99, 99, 99, 99, 99, 99, 99}};

// where the two quantisation tables (zigzag order) sit in the header kp_jpeg_header writes
constexpr int kDqtTable0 = 2 + 18 + 5;
constexpr int kDqtTable1 = kDqtTable0 + 65;

// bits of the magnitude category of v (0 for v == 0)
__device__ __forceinline__ int category(int v) { return v == 0 ? 0 : 32 - __clz(abs(v)); }

// Walks one block's Huffman codes in order: emit(code, length) for each code and each magnitude field.
template <typename Emit>
__device__ __forceinline__ void code_block(const int16_t* zz, int diff, int tab, Emit emit) {
  const int dcs = category(diff);
  emit(c_huff.code[0][tab][dcs], c_huff.len[0][tab][dcs]);
  if (dcs) emit((diff < 0 ? diff - 1 : diff) & ((1 << dcs) - 1), dcs);
  int run = 0;
  for (int k = 1; k < 64; ++k) {
    const int v = zz[k];
    if (v == 0) {
      ++run;
      continue;
    }
    for (; run >= 16; run -= 16) emit(c_huff.code[1][tab][0xF0], c_huff.len[1][tab][0xF0]);  // ZRL
    const int s = category(v);
    const int sym = run << 4 | s;
    emit(c_huff.code[1][tab][sym], c_huff.len[1][tab][sym]);
    emit((v < 0 ? v - 1 : v) & ((1 << s) - 1), s);
    run = 0;
  }
  if (run > 0) emit(c_huff.code[1][tab][0x00], c_huff.len[1][tab][0x00]);  // EOB
}

// ORs n <= 16 bits of v, most significant first, into a big-endian bit buffer of 32-bit words at bit position pos
__device__ __forceinline__ void put_bits(uint32_t* words, int pos, uint32_t v, int n) {
  const int w = pos >> 5, off = pos & 31;
  const uint64_t x = (uint64_t)v << (64 - n - off);
  atomicOr(words + w, (uint32_t)(x >> 32));
  if (off + n > 32) atomicOr(words + w + 1, (uint32_t)x);
}

__device__ __forceinline__ int ycc_y(int r, int g, int b) { return (19595 * r + 38470 * g + 7471 * b + 32768) >> 16; }
__device__ __forceinline__ int ycc_cb(int r, int g, int b) { return (-11059 * r - 21709 * g + 32768 * b + (128 << 16) + 32767) >> 16; }
__device__ __forceinline__ int ycc_cr(int r, int g, int b) { return (32768 * r - 27439 * g - 5329 * b + (128 << 16) + 32767) >> 16; }

__global__ void __launch_bounds__(kSegThreads) jpeg_segment_kernel(const uint8_t* __restrict__ img, int H, int W, int mcus_x,
                                                                   int n_mcus, const uint8_t* __restrict__ header,
                                                                   uint32_t* __restrict__ slots, int2* __restrict__ seg_len) {
  __shared__ float s_q[2][64];                 // quantiser, zigzag order (as the header's DQT holds it)
  __shared__ float s_blk[kSegBlocks][64];      // level-shifted samples, then the row transforms
  __shared__ int16_t s_zz[kSegBlocks][64];     // quantised coefficients, zigzag order
  __shared__ uint32_t s_bits[kSegWords];
  __shared__ int s_off[kSegBlocks + 1];
  __shared__ int s_ff;
  const int tid = threadIdx.x;
  const int seg = blockIdx.x;
  const int m0 = seg * kJpegR;
  const int n_mcu = min(kJpegR, n_mcus - m0);
  const int nb = 6 * n_mcu;
  for (int i = tid; i < 128; i += kSegThreads) s_q[i >> 6][i & 63] = (float)__ldg(header + (i < 64 ? kDqtTable0 : kDqtTable1 - 64) + i);
  for (int i = tid; i < kSegWords; i += kSegThreads) s_bits[i] = 0;
  if (tid == 0) s_ff = 0;

  // colour conversion and 2x2 downsampling: one thread per 2x2 pixel quad of an MCU
  for (int q = tid; q < n_mcu * 64; q += kSegThreads) {
    const int k = q >> 6, qy = (q >> 3) & 7, qx = q & 7;
    const int m = m0 + k, my = m / mcus_x, mx = m - my * mcus_x;
    int cb = 0, cr = 0;
#pragma unroll
    for (int d = 0; d < 4; ++d) {
      const int ly = 2 * qy + (d >> 1), lx = 2 * qx + (d & 1);
      const int gy = min(16 * my + ly, H - 1), gx = min(16 * mx + lx, W - 1);  // edge replication to a whole MCU
      const uint8_t* p = img + ((int64_t)gy * W + gx) * 3;
      const int r = __ldg(p), g = __ldg(p + 1), b = __ldg(p + 2);
      s_blk[6 * k + 2 * (ly >> 3) + (lx >> 3)][(ly & 7) * 8 + (lx & 7)] = (float)(ycc_y(r, g, b) - 128);
      cb += ycc_cb(r, g, b);
      cr += ycc_cr(r, g, b);
    }
    const int bias = 1 + (qx & 1);  // h2v2_downsample: 1, 2, 1, 2, ... along the row (MCUs start at even columns)
    s_blk[6 * k + 4][qy * 8 + qx] = (float)(((cb + bias) >> 2) - 128);
    s_blk[6 * k + 5][qy * 8 + qx] = (float)(((cr + bias) >> 2) - 128);
  }
  __syncthreads();

  // separable DCT: thread (b, r) transforms row r of block b in place, then column r, and quantises that column
  const int b = tid >> 3, r = tid & 7;
  if (b < nb) {
    float x[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) x[i] = s_blk[b][r * 8 + i];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      float t = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) t = fmaf(c_dct[u * 8 + i], x[i], t);
      s_blk[b][r * 8 + u] = t;
    }
  }
  __syncthreads();
  if (b < nb) {
    const int comp = (b % 6) < 4 ? 0 : 1;
    float x[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) x[i] = s_blk[b][i * 8 + r];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      float t = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) t = fmaf(c_dct[u * 8 + i], x[i], t);
      const int z = c_zigzag[u * 8 + r];
      s_zz[b][z] = (int16_t)roundf(__fdiv_rn(t, s_q[comp][z]));  // roundf: half away from zero
    }
  }
  __syncthreads();

  // entropy coding: code lengths, their prefix sum, then the bits
  int diff = 0, tab = 0;
  if (tid < nb) {
    const int k = tid / 6, j = tid - 6 * k;
    tab = j < 4 ? 0 : 1;
    int prev = 0;  // the DC predictors reset at each restart
    if (j >= 1 && j <= 3) prev = s_zz[tid - 1][0];
    else if (k > 0) prev = s_zz[j == 0 ? tid - 3 : tid - 6][0];
    diff = s_zz[tid][0] - prev;
  }
  if (tid < 32) {
    int len = 0;
    if (tid < nb) code_block(s_zz[tid], diff, tab, [&](uint32_t, int n) { len += n; });
    int incl = len;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, incl, o);
      if (tid >= o) incl += v;
    }
    if (tid <= kSegBlocks) s_off[tid] = incl - len;  // s_off[kSegBlocks]: the segment's bits (blocks >= nb add 0)
  }
  __syncthreads();
  const int total_bits = s_off[kSegBlocks];
  if (tid < nb) {
    int pos = s_off[tid];
    code_block(s_zz[tid], diff, tab, [&](uint32_t v, int n) {
      if (n) put_bits(s_bits, pos, v, n);
      pos += n;
    });
  }
  const int pad = (8 - (total_bits & 7)) & 7;
  if (tid == kSegThreads - 1 && pad) put_bits(s_bits, total_bits, (1u << pad) - 1, pad);  // fill the last byte with 1s
  __syncthreads();

  const int n_bytes = (total_bits + pad) >> 3;
  uint32_t* slot = slots + (int64_t)seg * kSegWords;
  int ff = 0;
  for (int w = tid; w < (n_bytes + 3) >> 2; w += kSegThreads) {
    const uint32_t v = s_bits[w];
#pragma unroll
    for (int i = 0; i < 4; ++i) ff += (4 * w + i < n_bytes) && ((v >> (24 - 8 * i)) & 0xFF) == 0xFF;
    slot[w] = __byte_perm(v, 0, 0x0123);  // big-endian bit order -> bytes in file order
  }
  if (ff) atomicAdd(&s_ff, ff);
  __syncthreads();
  if (tid == 0) seg_len[seg] = make_int2(n_bytes, n_bytes + s_ff + (seg + 1 < gridDim.x ? 2 : 0));
}

__global__ void __launch_bounds__(kScanThreads) jpeg_scan_kernel(const int2* __restrict__ seg_len, int S, const uint8_t* __restrict__ header,
                                                                 int header_len, int64_t* __restrict__ seg_off, uint8_t* __restrict__ out,
                                                                 int64_t* __restrict__ length) {
  __shared__ int64_t s_warp[kScanThreads / 32];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  for (int i = tid; i < header_len; i += kScanThreads) out[i] = header[i];
  const int chunk = (S + kScanThreads - 1) / kScanThreads;
  const int lo = min(S, tid * chunk), hi = min(S, lo + chunk);
  int64_t sum = 0;
  for (int i = lo; i < hi; ++i) sum += seg_len[i].y;
  int64_t incl = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int64_t v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) s_warp[wid] = incl;
  __syncthreads();
  if (wid == 0) {
    int64_t w = s_warp[lane], wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int64_t v = __shfl_up_sync(0xffffffffu, wi, o);
      if (lane >= o) wi += v;
    }
    s_warp[lane] = wi - w;
  }
  __syncthreads();
  int64_t run = header_len + s_warp[wid] + incl - sum;
  for (int i = lo; i < hi; ++i) {
    seg_off[i] = run;
    run += seg_len[i].y;
  }
  if (tid == kScanThreads - 1) {  // the last thread's running offset is the end of the scan
    out[run] = 0xFF;
    out[run + 1] = 0xD9;  // EOI
    *length = run + 2;
  }
}

__global__ void __launch_bounds__(kPackThreads) jpeg_pack_kernel(const uint32_t* __restrict__ slots, const int2* __restrict__ seg_len,
                                                                 const int64_t* __restrict__ seg_off, int S, uint8_t* __restrict__ out) {
  const int seg = (int)(((int64_t)blockIdx.x * kPackThreads + threadIdx.x) >> 5);
  const int lane = threadIdx.x & 31;
  if (seg >= S) return;
  const uint8_t* src = reinterpret_cast<const uint8_t*>(slots + (int64_t)seg * kSegWords);
  const int n = seg_len[seg].x;
  uint8_t* dst = out + seg_off[seg];
  int o = 0;
  for (int i0 = 0; i0 < n; i0 += 32) {
    const int i = i0 + lane;
    const uint8_t v = i < n ? src[i] : 0;
    const bool ff = i < n && v == 0xFF;
    const uint32_t mask = __ballot_sync(0xffffffffu, ff);
    if (i < n) {
      const int p = o + lane + __popc(mask & ((1u << lane) - 1));
      dst[p] = v;
      if (ff) dst[p + 1] = 0x00;  // byte stuffing
    }
    o += min(32, n - i0) + __popc(mask);
  }
  if (lane == 0 && seg + 1 < S) {
    dst[o] = 0xFF;
    dst[o + 1] = (uint8_t)(0xD0 + (seg & 7));  // RSTm
  }
}

static int64_t jpeg_segments(int H, int W) { return ceil_div(ceil_div(H, 16) * ceil_div(W, 16), kJpegR); }

static int64_t align256(int64_t n) { return (n + 255) & ~(int64_t)255; }

// ---- the header: SOI, APP0 (JFIF 1.01), DQT (both tables), SOF0, DHT (four tables), DRI, SOS ----
struct ByteWriter {
  uint8_t* p;
  int n = 0;
  void u8(int v) { p[n++] = (uint8_t)v; }
  void u16(int v) { u8(v >> 8), u8(v & 0xFF); }
  void huff(int tc_th, const uint8_t* bits, const uint8_t* vals) {
    u8(tc_th);
    int nv = 0;
    for (int i = 0; i < 16; ++i) u8(bits[i]), nv += bits[i];
    for (int i = 0; i < nv; ++i) u8(vals[i]);
  }
};

}  // namespace kp

using namespace kp;

extern "C" int64_t kp_jpeg_encode_capacity(int H, int W) {
  if (H <= 0 || W <= 0) return 0;
  return KP_JPEG_HEADER_BYTES + jpeg_segments(H, W) * kSegMaxFileBytes + 2;
}

extern "C" int64_t kp_jpeg_encode_scratch_bytes(int H, int W) {
  if (H <= 0 || W <= 0) return 0;
  const int64_t S = jpeg_segments(H, W);
  return align256(S * kSegWords * 4) + align256(S * (int64_t)sizeof(int2)) + S * (int64_t)sizeof(int64_t);
}

extern "C" int kp_jpeg_header(int H, int W, int quality, uint8_t* header) {
  KP_CHECK(header, "jpeg_header: NULL argument");
  KP_CHECK(H >= 1 && H <= 65535 && W >= 1 && W <= 65535, "jpeg_header: %dx%d image (1..65535 each)", H, W);
  KP_CHECK(quality >= 1 && quality <= 100, "jpeg_header: quality %d (1..100)", quality);
  ByteWriter w{header};
  w.u16(0xFFD8);  // SOI
  w.u16(0xFFE0), w.u16(16);  // APP0: JFIF 1.01, no units, 1:1 aspect, no thumbnail
  for (char c : {'J', 'F', 'I', 'F', '\0'}) w.u8(c);
  w.u8(1), w.u8(1), w.u8(0), w.u16(1), w.u16(1), w.u8(0), w.u8(0);
  w.u16(0xFFDB), w.u16(2 + 2 * 65);  // DQT: the IJG quality scaling of the K.1 tables (jcparam.c), baseline-clamped
  const int scale = quality < 50 ? 5000 / quality : 200 - 2 * quality;
  for (int t = 0; t < 2; ++t) {
    w.u8(t);
    for (int z = 0; z < 64; ++z) w.u8(std::min(255, std::max(1, (kStdQuant[t][kNatural[z]] * scale + 50) / 100)));
  }
  w.u16(0xFFC0), w.u16(17), w.u8(8), w.u16(H), w.u16(W), w.u8(3);  // SOF0
  w.u8(1), w.u8(0x22), w.u8(0);  // Y: 2x2, table 0
  w.u8(2), w.u8(0x11), w.u8(1);  // Cb
  w.u8(3), w.u8(0x11), w.u8(1);  // Cr
  w.u16(0xFFC4), w.u16(2 + 2 * (17 + 12) + 2 * (17 + 162));  // DHT
  w.huff(0x00, kDcLumBits, kDcVals);
  w.huff(0x10, kAcLumBits, kAcLumVals);
  w.huff(0x01, kDcChrBits, kDcVals);
  w.huff(0x11, kAcChrBits, kAcChrVals);
  w.u16(0xFFDD), w.u16(4), w.u16(kJpegR);  // DRI
  w.u16(0xFFDA), w.u16(12), w.u8(3);  // SOS
  w.u8(1), w.u8(0x00), w.u8(2), w.u8(0x11), w.u8(3), w.u8(0x11);
  w.u8(0), w.u8(63), w.u8(0);
  KP_CHECK(w.n == KP_JPEG_HEADER_BYTES, "jpeg_header: wrote %d bytes, expected %d", w.n, KP_JPEG_HEADER_BYTES);
  return 0;
}

extern "C" int kp_jpeg_encode(const uint8_t* image, int H, int W, const uint8_t* header, void* scratch, uint8_t* out,
                              int64_t* length, void* stream) {
  KP_CHECK(image && header && scratch && out && length, "jpeg_encode: NULL argument");
  KP_CHECK(H >= 1 && H <= 65535 && W >= 1 && W <= 65535, "jpeg_encode: %dx%d image (1..65535 each)", H, W);
  const int64_t S = jpeg_segments(H, W);
  const int mcus_x = (int)ceil_div(W, 16);
  const int n_mcus = (int)(ceil_div(H, 16) * mcus_x);
  uint8_t* base = static_cast<uint8_t*>(scratch);
  uint32_t* slots = reinterpret_cast<uint32_t*>(base);
  int2* seg_len = reinterpret_cast<int2*>(base + align256(S * kSegWords * 4));
  int64_t* seg_off = reinterpret_cast<int64_t*>(base + align256(S * kSegWords * 4) + align256(S * (int64_t)sizeof(int2)));
  cudaStream_t st = as_stream(stream);
  jpeg_segment_kernel<<<(unsigned)S, kSegThreads, 0, st>>>(image, H, W, mcus_x, n_mcus, header, slots, seg_len);
  KP_LAUNCH_CHECK("jpeg_encode(segment)");
  jpeg_scan_kernel<<<1, kScanThreads, 0, st>>>(seg_len, (int)S, header, KP_JPEG_HEADER_BYTES, seg_off, out, length);
  KP_LAUNCH_CHECK("jpeg_encode(scan)");
  jpeg_pack_kernel<<<(unsigned)ceil_div(S * 32, kPackThreads), kPackThreads, 0, st>>>(slots, seg_len, seg_off, (int)S, out);
  KP_LAUNCH_CHECK("jpeg_encode(pack)");
  return 0;
}
