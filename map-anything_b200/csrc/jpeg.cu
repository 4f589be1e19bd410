// Baseline JPEG decoding on the GPU, bit for bit the frame libjpeg-turbo's default decode gives Pillow (JDCT_ISLOW,
// fancy upsampling, table-driven YCbCr -> RGB).
//   * ma_jpeg_parse (host, no CUDA): markers, Huffman / quantisation tables, byte stuffing removed, restart intervals
//     and fixed-size subsequences recorded; everything is packed into one self-contained blob per frame that is
//     uploaded as is (the compressed stream: a 1080p q95 frame is about a sixth of its RGB bytes).
//   * jpeg_sync_kernel: parallel Huffman decoding by self-synchronisation (Weissenberger & Schmidt, ICPP 2018).  The
//     unstuffed stream of each restart interval is cut into MA_JPEG_SUBSEQ_BYTES subsequences; round 0 decodes every
//     subsequence from a guessed state (its first bit, first block of an MCU, DC coefficient) and records the state it
//     ends in as the next subsequence's entry.  Later rounds re-decode the subsequences whose entry changed; a thread
//     whose exit differs from the recorded entry writes it and continues into the following subsequences until its
//     state equals the one recorded there.  The state (bit position, block in MCU, zig-zag index) determines
//     everything after it, so once no entry changes every entry is the true one.
//   * jpeg_scan_check_kernel: per frame, the prefix sum of the blocks each subsequence starts (its first block), and
//     the checks that every restart interval holds exactly its MCUs.
//   * jpeg_write_kernel: the final pass, coefficients in natural order (DC as a difference).
//   * jpeg_dc_kernel: DC prediction, a segmented prefix sum per component and restart interval.
//   * jpeg_idct_kernel: dequantisation + jidctint.c's islow IDCT + the post-IDCT range-limit table, into planes.
//   * jpeg_color_kernel: fancy upsampling (jdsample.c) + jdcolor.c's fixed-point YCbCr -> RGB + EXIF orientation as an
//     index map, packed RGB straight into the caller's frame slot.
// A frame whose stream breaks a rule (invalid code, wrong block count, no convergence) or whose coefficients leave the
// range in which libjpeg-turbo's C and SIMD IDCTs agree gets a nonzero status; the caller decodes it with Pillow.
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "host_common.h"

namespace ma {
namespace {

constexpr int kMaxRounds = 24;  // synchronisation rounds; a frame still changing after them is reported, not guessed
constexpr int kMaxChase = 16;   // subsequences one thread follows past its own in one round

struct HuffTab {
  uint16_t lut[512];   // 9-bit lookahead: (length << 8) | symbol, 0 = longer code
  int32_t maxcode[18];  // largest code of each length, -1 if none
  int32_t valoff[18];   // symbol index of a code of that length = code + valoff
  uint8_t vals[256];
};

struct JpegHdr {
  int32_t width, height, ncomp, hmax, vmax, mcus_x, mcus_y, bpm, restart, nseg, nsub, pad0;
  int32_t bw[3], bh[3];          // block grid of each component's plane
  int32_t dw[3], dh[3];          // downsampled width / height of each component
  int32_t blk_comp[10], blk_dx[10], blk_dy[10];
  int64_t nblocks, plane_off[3];  // plane offsets inside the frame's plane area
  int64_t seg_off, sub_off, data_off, data_bytes;
  uint16_t qt[3][64];  // natural order
  HuffTab dc[3], ac[3];
};
// blob: JpegHdr | data (unstuffed) + 16 zero bytes | uint32 seg_first_sub[nseg + 1] |
//       uint32 sub[nsub][3] (start byte, end byte, segment end byte)

struct FrameDesc {
  const uint8_t* blob;
  uint8_t* planes;
  uint8_t* out;
  int64_t sub_base, blk_base;
  int32_t orient, pad;
};

constexpr int ZZ[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                        41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                        30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
__constant__ uint8_t c_zz[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                 41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

constexpr int32_t ST_ENTROPY = 1, ST_SYNC = 2, ST_RANGE = 4;

// ------------------------------------------------------------------------------------------------ host parser
static bool build_huff(const uint8_t* counts, const uint8_t* vals, int nvals, bool dc, HuffTab* t) {
  memset(t, 0, sizeof(*t));
  int32_t code = 0, k = 0;
  for (int l = 1; l <= 16; ++l) {
    t->maxcode[l] = -1;
    if (counts[l - 1]) {
      t->valoff[l] = k - code;
      for (int i = 0; i < counts[l - 1]; ++i, ++k, ++code) {
        if (code >= (1 << l)) return false;  // over-full: more codes of this length than fit (checked before any write)
        if (l <= 9)
          for (int f = 0; f < (1 << (9 - l)); ++f) t->lut[(code << (9 - l)) | f] = (uint16_t)((l << 8) | vals[k]);
      }
      t->maxcode[l] = code - 1;
    }
    if (code >= (1 << l)) return false;  // jdhuff.c: no code may consist of all 1-bits
    code <<= 1;
  }
  for (int i = 0; i < nvals; ++i) {
    if (dc && vals[i] > 15) return false;
    t->vals[i] = vals[i];
  }
  return true;
}

}  // namespace
}  // namespace ma

using namespace ma;

extern "C" int ma_jpeg_parse(const uint8_t* file_host, int64_t size, ma_jpeg_info* info, uint8_t* blob_host,
                             int64_t blob_capacity) {
  MA_REQUIRE(file_host && info && size >= 0, "ma_jpeg_parse: file_host and info must be non-NULL, size >= 0");
  const uint8_t* f = file_host;
  MA_REQUIRE(size >= 4 && f[0] == 0xFF && f[1] == 0xD8, "ma_jpeg_parse: no SOI marker");
  uint16_t q[4][64];
  bool have_q[4] = {}, have_dc[4] = {}, have_ac[4] = {};
  static thread_local HuffTab dct[4], act[4];
  int W = 0, H = 0, nc = 0, cid[3] = {}, ch[3] = {}, cv[3] = {}, ctq[3] = {}, ctd[3] = {}, cta[3] = {};
  int restart = 0, adobe_transform = -1;
  bool jfif = false, sof = false;
  int64_t p = 2;
  for (;;) {
    while (p + 1 < size && f[p] == 0xFF && f[p + 1] == 0xFF) ++p;  // fill bytes
    MA_REQUIRE(p + 4 <= size, "ma_jpeg_parse: truncated before the scan");
    MA_REQUIRE(f[p] == 0xFF, "ma_jpeg_parse: marker expected at byte %lld", (long long)p);
    const int m = f[p + 1];
    const int L = (f[p + 2] << 8) | f[p + 3];
    MA_REQUIRE(L >= 2 && p + 2 + L <= size, "ma_jpeg_parse: truncated segment (marker 0x%02X)", m);
    const uint8_t* s = f + p + 4;
    const int n = L - 2;
    p += 2 + L;
    if (m == 0xDB) {
      for (int i = 0; i < n;) {
        const int pq = s[i] >> 4, tq = s[i] & 15;
        MA_REQUIRE(pq <= 1 && tq < 4 && i + 1 + 64 * (pq + 1) <= n, "ma_jpeg_parse: bad DQT segment");
        for (int k = 0; k < 64; ++k) q[tq][ZZ[k]] = pq ? (uint16_t)((s[i + 1 + 2 * k] << 8) | s[i + 2 + 2 * k]) : s[i + 1 + k];
        have_q[tq] = true;
        i += 1 + 64 * (pq + 1);
      }
    } else if (m == 0xC4) {
      for (int i = 0; i < n;) {
        MA_REQUIRE(i + 17 <= n, "ma_jpeg_parse: truncated DHT segment");
        const int tc = s[i] >> 4, th = s[i] & 15;
        MA_REQUIRE(tc <= 1 && th < 4, "ma_jpeg_parse: bad Huffman table class / index %d/%d", tc, th);
        int nv = 0;
        for (int k = 0; k < 16; ++k) nv += s[i + 1 + k];
        MA_REQUIRE(nv <= 256 && i + 17 + nv <= n, "ma_jpeg_parse: truncated or oversized Huffman table");
        MA_REQUIRE(build_huff(s + i + 1, s + i + 17, nv, tc == 0, tc ? &act[th] : &dct[th]),
                   "ma_jpeg_parse: Huffman table %d/%d is not a valid prefix code", tc, th);
        (tc ? have_ac : have_dc)[th] = true;
        i += 17 + nv;
      }
    } else if (m == 0xDD) {
      MA_REQUIRE(n == 2, "ma_jpeg_parse: bad DRI segment");
      restart = (s[0] << 8) | s[1];
    } else if (m == 0xE0) {
      if (n >= 14 && !memcmp(s, "JFIF\0", 5)) jfif = true;  // jdmarker.c examine_app0: APP0_DATA_LEN
    } else if (m == 0xEE) {
      if (n >= 12 && !memcmp(s, "Adobe", 5)) adobe_transform = s[11];
    } else if (m == 0xC0 || m == 0xC1) {
      MA_REQUIRE(!sof && n >= 6, "ma_jpeg_parse: bad or repeated SOF segment");
      MA_REQUIRE(s[0] == 8, "ma_jpeg_parse: %d-bit precision (8-bit only)", s[0]);
      H = (s[1] << 8) | s[2];
      W = (s[3] << 8) | s[4];
      nc = s[5];
      MA_REQUIRE(W > 0 && H > 0, "ma_jpeg_parse: frame size %dx%d", W, H);
      MA_REQUIRE(nc == 1 || nc == 3, "ma_jpeg_parse: %d components (1 or 3 only)", nc);
      MA_REQUIRE(n == 6 + 3 * nc, "ma_jpeg_parse: bad SOF length");
      for (int c = 0; c < nc; ++c) {
        cid[c] = s[6 + 3 * c];
        ch[c] = s[7 + 3 * c] >> 4;
        cv[c] = s[7 + 3 * c] & 15;
        ctq[c] = s[8 + 3 * c];
        MA_REQUIRE(ch[c] >= 1 && ch[c] <= 4 && cv[c] >= 1 && cv[c] <= 4 && ctq[c] < 4,
                   "ma_jpeg_parse: bad sampling factors or table index of component %d", c);
      }
      if (nc == 3) {
        MA_REQUIRE(ch[1] == 1 && cv[1] == 1 && ch[2] == 1 && cv[2] == 1 &&
                       ((ch[0] == 1 || ch[0] == 2) && (cv[0] == 1 || cv[0] == 2)),
                   "ma_jpeg_parse: sampling %dx%d,%dx%d,%dx%d (4:4:4, 4:2:2, 4:2:0, 4:4:0 only)", ch[0], cv[0], ch[1],
                   cv[1], ch[2], cv[2]);
      } else {
        ch[0] = cv[0] = 1;  // a single-component scan is not interleaved: one block per MCU
      }
      sof = true;
    } else if (m >= 0xC2 && m <= 0xCF && m != 0xC4 && m != 0xC8 && m != 0xCC) {
      MA_REQUIRE(false, "ma_jpeg_parse: SOF%d frame (baseline / extended sequential Huffman only)", m - 0xC0);
    } else if (m == 0xDA) {
      MA_REQUIRE(sof, "ma_jpeg_parse: scan before the frame header");
      MA_REQUIRE(n >= 1 && s[0] == nc && n == 4 + 2 * nc, "ma_jpeg_parse: the scan does not cover the frame");
      for (int c = 0; c < nc; ++c) {
        MA_REQUIRE(s[1 + 2 * c] == cid[c], "ma_jpeg_parse: scan components not in frame order");
        ctd[c] = s[2 + 2 * c] >> 4;
        cta[c] = s[2 + 2 * c] & 15;
        MA_REQUIRE(ctd[c] < 4 && cta[c] < 4 && have_dc[ctd[c]] && have_ac[cta[c]] && have_q[ctq[c]],
                   "ma_jpeg_parse: component %d refers to a missing table", c);
      }
      MA_REQUIRE(s[1 + 2 * nc] == 0 && s[2 + 2 * nc] == 63 && s[3 + 2 * nc] == 0,
                 "ma_jpeg_parse: spectral selection / approximation of a non-sequential scan");
      break;
    } else {
      MA_REQUIRE(m >= 0xE0 || m == 0xFE, "ma_jpeg_parse: unsupported marker 0x%02X", m);
    }
  }
  if (nc == 3) {
    const bool rgb = jfif ? false : adobe_transform >= 0 ? adobe_transform != 1 : (cid[0] == 'R' && cid[1] == 'G' && cid[2] == 'B');
    MA_REQUIRE(!rgb, "ma_jpeg_parse: components are not YCbCr");
  }
  const int hmax = ch[0], vmax = cv[0];
  const int mcus_x = nc == 1 ? (W + 7) / 8 : (W + 8 * hmax - 1) / (8 * hmax);
  const int mcus_y = nc == 1 ? (H + 7) / 8 : (H + 8 * vmax - 1) / (8 * vmax);
  const int64_t nmcu = (int64_t)mcus_x * mcus_y;
  const int bpm = nc == 1 ? 1 : hmax * vmax + 2;
  const int64_t want_seg = restart ? (nmcu + restart - 1) / restart : 1;

  // entropy-coded data: unstuff, split at RSTn (in sequence), end at EOI.  One pass: the unstuffed bytes go straight to
  // the blob's data area when the caller's blob can hold every remaining byte of the file (they never exceed that).
  constexpr int64_t data_off = (sizeof(JpegHdr) + 15) & ~(int64_t)15;
  std::vector<uint32_t> seg_start(1, 0);
  const int64_t data0 = p;
  uint8_t* dst = blob_host && blob_capacity >= data_off + (size - data0) + 16 ? blob_host + data_off : nullptr;
  auto unstuff = [&](uint8_t* out, bool record) -> int64_t {  // bytes written, or -1 with the error set
    int64_t i = data0, o = 0;
    int next_rst = 0;
    for (;;) {
      if (i >= size || (f[i] == 0xFF && i + 1 >= size)) {
        ma::set_last_error("ma_jpeg_parse: entropy-coded data not terminated by EOI");
        return -1;
      }
      if (f[i] != 0xFF) {
        if (out) out[o] = f[i];
        ++o, ++i;
        continue;
      }
      const int b = f[i + 1];
      if (b == 0x00) {
        if (out) out[o] = 0xFF;
        ++o, i += 2;
      } else if (b == 0xFF) {
        ++i;
      } else if (b >= 0xD0 && b <= 0xD7) {
        if (record) {
          if (!restart || b - 0xD0 != next_rst) {
            ma::set_last_error("ma_jpeg_parse: unexpected restart marker RST%d", b - 0xD0);
            return -1;
          }
          if ((int64_t)seg_start.size() >= want_seg) {
            ma::set_last_error("ma_jpeg_parse: more restart intervals than MCUs");
            return -1;
          }
          next_rst = (next_rst + 1) & 7;
          seg_start.push_back((uint32_t)o);
        }
        i += 2;
      } else if (b == 0xD9) {
        return o;
      } else {
        ma::set_last_error("ma_jpeg_parse: marker 0x%02X after the scan (one baseline scan only)", b);
        return -1;
      }
      if (o >= (int64_t)1 << 31) {
        ma::set_last_error("ma_jpeg_parse: entropy-coded data too large");
        return -1;
      }
    }
  };
  const int64_t unstuffed = unstuff(dst, true);
  if (unstuffed < 0) return MA_ERR_INVALID;
  MA_REQUIRE((int64_t)seg_start.size() == want_seg, "ma_jpeg_parse: %lld restart intervals for %lld MCUs (interval %d)",
             (long long)seg_start.size(), (long long)nmcu, restart);
  const int nseg = (int)seg_start.size();
  seg_start.push_back((uint32_t)unstuffed);
  std::vector<uint32_t> first_sub(nseg + 1);
  int64_t nsub = 0;
  for (int k = 0; k < nseg; ++k) {
    first_sub[k] = (uint32_t)nsub;
    const int64_t bytes = seg_start[k + 1] - seg_start[k];
    nsub += bytes ? (bytes + MA_JPEG_SUBSEQ_BYTES - 1) / MA_JPEG_SUBSEQ_BYTES : 1;
  }
  first_sub[nseg] = (uint32_t)nsub;

  JpegHdr h_;
  memset(&h_, 0, sizeof(h_));
  JpegHdr* h = &h_;
  h->width = W, h->height = H, h->ncomp = nc, h->hmax = hmax, h->vmax = vmax, h->mcus_x = mcus_x, h->mcus_y = mcus_y;
  h->bpm = bpm, h->restart = restart, h->nseg = nseg, h->nsub = (int32_t)nsub;
  int64_t plane = 0;
  for (int c = 0; c < nc; ++c) {
    h->bw[c] = mcus_x * ch[c];
    h->bh[c] = mcus_y * cv[c];
    h->dw[c] = (int)(((int64_t)W * ch[c] + hmax - 1) / hmax);
    h->dh[c] = (int)(((int64_t)H * cv[c] + vmax - 1) / vmax);
    h->plane_off[c] = plane;
    plane += (int64_t)h->bw[c] * h->bh[c] * 64;
    memcpy(h->qt[c], q[ctq[c]], sizeof(h->qt[c]));
    h->dc[c] = dct[ctd[c]];
    h->ac[c] = act[cta[c]];
  }
  for (int c = 0, b = 0; c < nc; ++c)
    for (int v = 0; v < cv[c]; ++v)
      for (int u = 0; u < ch[c]; ++u, ++b) h->blk_comp[b] = c, h->blk_dx[b] = u, h->blk_dy[b] = v;
  h->nblocks = nmcu * bpm;
  h->data_off = data_off;
  h->data_bytes = unstuffed;
  h->seg_off = (data_off + unstuffed + 16 + 15) & ~(int64_t)15;  // 16 zero bytes after the data: bit-buffer refills
  h->sub_off = (h->seg_off + 4 * (nseg + 1) + 15) & ~(int64_t)15;
  const int64_t blob_bytes = (h->sub_off + 12 * nsub + 15) & ~(int64_t)15;

  info->width = W, info->height = H, info->ncomp = nc, info->h_samp = hmax, info->v_samp = vmax;
  info->restart_interval = restart, info->nsegments = nseg, info->nsubseq = (int32_t)nsub;
  info->nblocks = h->nblocks, info->plane_bytes = plane, info->blob_bytes = blob_bytes;
  if (!blob_host) return MA_OK;
  MA_REQUIRE(blob_capacity >= blob_bytes, "ma_jpeg_parse: blob_capacity %lld < %lld bytes", (long long)blob_capacity,
             (long long)blob_bytes);
  if (!dst) unstuff(blob_host + data_off, false);  // the capacity did not cover the whole remaining file
  memcpy(blob_host, h, sizeof(JpegHdr));
  memset(blob_host + sizeof(JpegHdr), 0, data_off - sizeof(JpegHdr));
  memset(blob_host + data_off + unstuffed, 0, h->seg_off - (data_off + unstuffed));
  memcpy(blob_host + h->seg_off, first_sub.data(), 4 * (nseg + 1));
  memset(blob_host + h->seg_off + 4 * (nseg + 1), 0, h->sub_off - (h->seg_off + 4 * (nseg + 1)));
  uint32_t* sub = reinterpret_cast<uint32_t*>(blob_host + h->sub_off);
  for (int k = 0; k < nseg; ++k) {
    for (uint32_t j = first_sub[k]; j < first_sub[k + 1]; ++j) {
      const uint32_t st = seg_start[k] + (j - first_sub[k]) * MA_JPEG_SUBSEQ_BYTES;
      sub[3 * j] = st;
      sub[3 * j + 1] = st + MA_JPEG_SUBSEQ_BYTES < seg_start[k + 1] ? st + MA_JPEG_SUBSEQ_BYTES : seg_start[k + 1];
      sub[3 * j + 2] = seg_start[k + 1];
    }
  }
  memset(blob_host + h->sub_off + 12 * nsub, 0, blob_bytes - (h->sub_off + 12 * nsub));
  return MA_OK;
}

// ------------------------------------------------------------------------------------------------ device
namespace ma {
namespace {

// state: bit position << 16 | block in MCU << 8 | zig-zag index
__device__ __forceinline__ uint64_t pack_state(uint64_t pos, int b, int zz) { return pos << 16 | (uint64_t)b << 8 | zz; }

struct BitReader {
  const uint8_t* data;
  uint64_t buf;
  int nb;
  uint64_t byte;
  __device__ void init(const uint8_t* d, uint64_t pos) {
    data = d;
    byte = pos >> 3;
    buf = 0;
    nb = 0;
    fill();
    buf <<= (pos & 7);
    nb -= (int)(pos & 7);
  }
  __device__ __forceinline__ void fill() {
    while (nb <= 56) {
      buf |= (uint64_t)__ldg(data + byte++) << (56 - nb);
      nb += 8;
    }
  }
};

__device__ __forceinline__ int huff_decode(const HuffTab& t, uint32_t peek16, int* len) {
  const uint16_t e = __ldg(&t.lut[peek16 >> 7]);
  if (e) {
    *len = e >> 8;
    return e & 255;
  }
  int l = 10;
  int32_t code = peek16 >> 6;
  while (code > __ldg(&t.maxcode[l])) {
    if (++l > 16) return -1;
    code = peek16 >> (16 - l);
  }
  *len = l;
  return __ldg(&t.vals[code + __ldg(&t.valoff[l])]);
}

__device__ __forceinline__ int extend(int r, int s) { return s && r < (1 << (s - 1)) ? r - (1 << s) + 1 : r; }

// Decodes from `st` while the bit position is below `end`; a symbol that would cross `seg_end` ends the run.
// SYNC: an invalid code restarts speculation one bit further on; WRITE: it is an error.  Returns the exit state,
// counts started blocks in *nblk.
template <bool WRITE>
__device__ uint64_t decode_run(const JpegHdr* h, const uint8_t* data, uint64_t st, uint64_t end, uint64_t seg_end,
                               int* nblk, int16_t* coef, int64_t blk, int64_t nblocks, bool* err) {
  uint64_t pos = st >> 16;
  int b = (st >> 8) & 255, zz = st & 255;
  const int bpm = h->bpm;
  BitReader br;
  br.init(data, pos);
  int cnt = 0;
  while (pos < end) {
    br.fill();
    const int c = h->blk_comp[b];
    int len;
    const int sym = huff_decode(zz == 0 ? h->dc[c] : h->ac[c], (uint32_t)(br.buf >> 48), &len);
    if (sym < 0) {
      if (pos + 16 > seg_end) break;  // the 1-bit padding before a restart marker / EOI: no code is all 1-bits
      if (WRITE) {
        *err = true;
        break;
      }
      pos += 1;
      br.init(data, pos);
      b = 0, zz = 0;
      continue;
    }
    const int s = sym & 15;
    const int total = len + (zz == 0 ? sym : s);
    if (pos + total > seg_end) break;
    const int r = (int)((br.buf << len) >> 32 >> (32 - (zz == 0 ? sym : s)));
    const int val = extend((zz == 0 ? sym : s) ? r : 0, zz == 0 ? sym : s);
    br.buf <<= total;
    br.nb -= total;
    pos += total;
    if (zz == 0) {
      ++cnt;
      ++blk;
      if (WRITE) {
        if (blk < 0 || blk >= nblocks) {
          *err = true;
          break;
        }
        coef[blk * 64] = (int16_t)val;
      }
      zz = 1;
    } else if (s) {
      zz += sym >> 4;
      if (WRITE) {
        if (blk < 0 || blk >= nblocks) {
          *err = true;
          break;
        }
        coef[blk * 64 + c_zz[zz > 63 ? 63 : zz]] = (int16_t)val;  // jpeg_natural_order maps k > 63 to 63
      }
      ++zz;
    } else {
      zz = (sym >> 4) == 15 ? zz + 16 : 64;
    }
    if (zz >= 64) {
      zz = 0;
      b = b + 1 == bpm ? 0 : b + 1;
    }
  }
  *nblk = cnt;
  return pack_state(pos, b, zz);
}

__device__ __forceinline__ int find_frame(const FrameDesc* fr, int n, int64_t idx, bool by_block) {
  int lo = 0, hi = n - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if ((by_block ? fr[mid].blk_base : fr[mid].sub_base) <= idx) lo = mid; else hi = mid - 1;
  }
  return lo;
}

struct Work {
  uint64_t* entry;
  uint64_t* exitst;
  int32_t* dirty;
  int32_t* nblk;
  int32_t* blkstart;
  int32_t* active;
  int16_t* coef;
};

__global__ void jpeg_init_kernel(const FrameDesc* fr, int n, int64_t total_sub, Work w) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j < kMaxRounds + 2) w.active[j] = 0;
  if (j >= total_sub) return;
  const int f = find_frame(fr, n, j, false);
  const JpegHdr* h = reinterpret_cast<const JpegHdr*>(fr[f].blob);
  const uint32_t* sub = reinterpret_cast<const uint32_t*>(fr[f].blob + h->sub_off) + 3 * (j - fr[f].sub_base);
  w.entry[j] = pack_state((uint64_t)sub[0] * 8, 0, 0);
  w.dirty[j] = 0;
}

__global__ void jpeg_sync_kernel(const FrameDesc* fr, int n, int64_t total_sub, Work w, int round) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= total_sub || (round > 0 && __ldcg(&w.active[round]) == 0)) return;
  if (__ldcg(&w.dirty[j]) != round) return;
  const int f = find_frame(fr, n, j, false);
  const uint8_t* blob = fr[f].blob;
  const JpegHdr* h = reinterpret_cast<const JpegHdr*>(blob);
  const uint32_t* subs = reinterpret_cast<const uint32_t*>(blob + h->sub_off);
  const uint8_t* data = blob + h->data_off;
  const int64_t local0 = j - fr[f].sub_base;
  uint64_t st = __ldcg(&w.entry[j]);
  for (int64_t k = local0; k < local0 + 1 + (round > 0 ? kMaxChase : 0) && k < h->nsub; ++k) {
    const uint32_t* sub = subs + 3 * k;
    int cnt;
    bool err = false;
    const uint64_t ex = decode_run<false>(h, data, st, (uint64_t)sub[1] * 8, (uint64_t)sub[2] * 8, &cnt, nullptr, 0, 0, &err);
    const int64_t g = fr[f].sub_base + k;
    w.nblk[g] = cnt;
    w.exitst[g] = ex;
    if (sub[1] == sub[2] || k + 1 >= h->nsub) break;  // the next subsequence starts a restart interval
    if (__ldcg(&w.entry[g + 1]) == ex) break;        // synchronised with what is recorded there
    w.entry[g + 1] = ex;
    __threadfence();
    w.dirty[g + 1] = round + 1;
    atomicAdd(&w.active[round + 1], 1);
    st = ex;
  }
}

// Block-wide inclusive scan of int64 values (blockDim.x = 256).
__device__ int64_t block_scan(int64_t v, int64_t* sh) {
  const int t = threadIdx.x;
  sh[t] = v;
  __syncthreads();
  for (int o = 1; o < 256; o <<= 1) {
    const int64_t a = t >= o ? sh[t - o] : 0;
    __syncthreads();
    sh[t] += a;
    __syncthreads();
  }
  const int64_t r = sh[t];
  __syncthreads();
  return r;
}

__global__ void __launch_bounds__(256) jpeg_scan_check_kernel(const FrameDesc* fr, Work w, int32_t* status) {
  __shared__ int64_t sh[256];
  const FrameDesc& d = fr[blockIdx.x];
  const JpegHdr* h = reinterpret_cast<const JpegHdr*>(d.blob);
  const uint32_t* first_sub = reinterpret_cast<const uint32_t*>(d.blob + h->seg_off);
  int64_t carry = 0;
  int32_t bad = 0;
  for (int64_t j0 = 0; j0 < h->nsub; j0 += 256) {
    const int64_t j = j0 + threadIdx.x;
    const int64_t v = j < h->nsub ? w.nblk[d.sub_base + j] : 0;
    if (j < h->nsub && w.dirty[d.sub_base + j] >= kMaxRounds) bad |= ST_SYNC;
    const int64_t inc = block_scan(v, sh) + carry;
    if (j < h->nsub) w.blkstart[d.sub_base + j] = (int32_t)(inc - v);
    const int64_t tot = sh[255];
    __syncthreads();
    carry += tot;
  }
  __syncthreads();
  const int64_t per_seg = h->restart ? (int64_t)h->restart * h->bpm : h->nblocks;
  for (int k = threadIdx.x; k < h->nseg; k += 256) {
    const int64_t b0 = w.blkstart[d.sub_base + first_sub[k]];
    const int64_t b1 = k + 1 < h->nseg ? w.blkstart[d.sub_base + first_sub[k + 1]] : carry;
    const int64_t want = k + 1 < h->nseg ? per_seg : h->nblocks - per_seg * (h->nseg - 1);
    const uint64_t ex = w.exitst[d.sub_base + first_sub[k + 1] - 1];
    if (b1 - b0 != want || (ex & 0xffff) != 0) bad |= ST_ENTROPY;
  }
  if (bad) atomicOr(&status[blockIdx.x], bad);
}

__global__ void jpeg_write_kernel(const FrameDesc* fr, int n, int64_t total_sub, Work w, int32_t* status) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= total_sub) return;
  const int f = find_frame(fr, n, j, false);
  const uint8_t* blob = fr[f].blob;
  const JpegHdr* h = reinterpret_cast<const JpegHdr*>(blob);
  const uint32_t* sub = reinterpret_cast<const uint32_t*>(blob + h->sub_off) + 3 * (j - fr[f].sub_base);
  int cnt;
  bool err = false;
  decode_run<true>(h, blob + h->data_off, w.entry[j], (uint64_t)sub[1] * 8, (uint64_t)sub[2] * 8, &cnt,
                   w.coef + fr[f].blk_base * 64, (int64_t)w.blkstart[j] - 1, h->nblocks, &err);
  if (err) atomicOr(&status[f], ST_ENTROPY);
}

// DC prediction: per frame, MCUs in chunks of 256, a segmented (restart interval) inclusive scan of each component's
// DC differences.  libjpeg keeps the predictor as an int and stores its low 16 bits.
__global__ void __launch_bounds__(256) jpeg_dc_kernel(const FrameDesc* fr, Work w) {
  __shared__ int32_t sv[3][256];
  __shared__ int32_t sf[256];
  const FrameDesc& d = fr[blockIdx.x];
  const JpegHdr* h = reinterpret_cast<const JpegHdr*>(d.blob);
  const int64_t nmcu = (int64_t)h->mcus_x * h->mcus_y;
  const int bpm = h->bpm, t = threadIdx.x;
  int16_t* coef = w.coef + d.blk_base * 64;
  int32_t carry[3] = {0, 0, 0};
  for (int64_t m0 = 0; m0 < nmcu; m0 += 256) {
    const int64_t m = m0 + t;
    int32_t v[3] = {0, 0, 0};
    int32_t flag = m < nmcu && h->restart && m % h->restart == 0;
    if (m < nmcu)
      for (int b = 0; b < bpm; ++b) v[h->blk_comp[b]] += coef[(m * bpm + b) * 64];
    for (int c = 0; c < 3; ++c) sv[c][t] = v[c];
    sf[t] = flag;
    __syncthreads();
    for (int o = 1; o < 256; o <<= 1) {
      int32_t a[3] = {0, 0, 0}, af = 0;
      const bool take = t >= o && !sf[t];
      if (t >= o) {
        for (int c = 0; c < 3; ++c) a[c] = sv[c][t - o];
        af = sf[t - o];
      }
      __syncthreads();
      if (take)
        for (int c = 0; c < 3; ++c) sv[c][t] += a[c];
      if (t >= o) sf[t] |= af;
      __syncthreads();
    }
    const bool seen = sf[t];  // a restart interval starts within [m0, m]
    int32_t run[3];
    // exclusive prefix within the current interval: the inclusive scan minus this MCU, plus the carry when no
    // interval started in this chunk up to here
    for (int c = 0; c < 3; ++c) run[c] = (flag ? 0 : sv[c][t] - v[c]) + (seen ? 0 : carry[c]);
    if (m < nmcu)
      for (int b = 0; b < bpm; ++b) {
        const int c = h->blk_comp[b];
        int16_t* p = &coef[(m * bpm + b) * 64];
        run[c] += *p;
        *p = (int16_t)run[c];
      }
    __syncthreads();
    const bool any = sf[255];
    for (int c = 0; c < 3; ++c) carry[c] = sv[c][255] + (any ? 0 : carry[c]);
    __syncthreads();
  }
}

// jidctint.c jpeg_idct_islow (64-bit intermediates like its JLONG), one thread per block.  Reports frames whose
// dequantised coefficients or first-pass outputs leave [-16383, 16383] or whose outputs leave [-512, 511]: there
// libjpeg-turbo's 16-bit SIMD IDCT and its C IDCT can differ, so such a frame is decoded by Pillow instead.
__global__ void __launch_bounds__(128) jpeg_idct_kernel(const FrameDesc* fr, int n, int64_t total_blocks, Work w,
                                                        int32_t* status) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= total_blocks) return;
  const int f = find_frame(fr, n, g, true);
  const JpegHdr* h = reinterpret_cast<const JpegHdr*>(fr[f].blob);
  const int64_t l = g - fr[f].blk_base;
  int c, bx, by;
  if (h->ncomp == 1) {
    c = 0, bx = (int)(l % h->bw[0]), by = (int)(l / h->bw[0]);
  } else {
    const int64_t m = l / h->bpm;
    const int b = (int)(l % h->bpm);
    c = h->blk_comp[b];
    bx = (int)(m % h->mcus_x) * (c ? 1 : h->hmax) + h->blk_dx[b];
    by = (int)(m / h->mcus_x) * (c ? 1 : h->vmax) + h->blk_dy[b];
  }
  const int4* src = reinterpret_cast<const int4*>(w.coef + g * 64);
  int32_t in[64];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int4 v = __ldg(src + i);
    const int32_t words[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      in[8 * i + 2 * k] = (int16_t)(words[k] & 0xffff);
      in[8 * i + 2 * k + 1] = (int16_t)((uint32_t)words[k] >> 16);
    }
  }
  const uint16_t* qt = h->qt[c];
  bool bad = false;
#pragma unroll
  for (int i = 0; i < 64; ++i) {
    const int64_t v = (int64_t)in[i] * __ldg(qt + i);
    bad |= v > 16383 || v < -16383;
    in[i] = (int32_t)v;
  }
  constexpr int CB = 13, P1 = 2;
  auto idct1 = [](int64_t v0, int64_t v1, int64_t v2, int64_t v3, int64_t v4, int64_t v5, int64_t v6, int64_t v7,
                  int64_t* o) {
    int64_t z2 = v2, z3 = v6;
    int64_t z1 = (z2 + z3) * 4433;
    const int64_t tmp2 = z1 + z3 * -15137, tmp3 = z1 + z2 * 6270;
    const int64_t t0 = (v0 + v4) * (1 << CB), t1 = (v0 - v4) * (1 << CB);
    const int64_t t10 = t0 + tmp3, t13 = t0 - tmp3, t11 = t1 + tmp2, t12 = t1 - tmp2;
    int64_t a0 = v7, a1 = v5, a2 = v3, a3 = v1;
    z1 = a0 + a3, z2 = a1 + a2, z3 = a0 + a2;
    int64_t z4 = a1 + a3;
    const int64_t z5 = (z3 + z4) * 9633;
    a0 *= 2446, a1 *= 16819, a2 *= 25172, a3 *= 12299;
    z1 *= -7373, z2 *= -20995, z3 = z3 * -16069 + z5, z4 = z4 * -3196 + z5;
    a0 += z1 + z3, a1 += z2 + z4, a2 += z2 + z3, a3 += z1 + z4;
    o[0] = t10 + a3, o[7] = t10 - a3, o[1] = t11 + a2, o[6] = t11 - a2;
    o[2] = t12 + a1, o[5] = t12 - a1, o[3] = t13 + a0, o[4] = t13 - a0;
  };
  int32_t ws[64];
#pragma unroll
  for (int col = 0; col < 8; ++col) {
    int64_t o[8];
    idct1(in[col], in[8 + col], in[16 + col], in[24 + col], in[32 + col], in[40 + col], in[48 + col], in[56 + col], o);
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      const int64_t v = (o[r] + (1 << (CB - P1 - 1))) >> (CB - P1);
      bad |= v > 16383 || v < -16383;
      ws[8 * r + col] = (int32_t)v;
    }
  }
  uint8_t* plane = fr[f].planes + h->plane_off[c];
  const int pw = h->bw[c] * 8;
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    int64_t o[8];
    idct1(ws[8 * r], ws[8 * r + 1], ws[8 * r + 2], ws[8 * r + 3], ws[8 * r + 4], ws[8 * r + 5], ws[8 * r + 6],
          ws[8 * r + 7], o);
    uint32_t lo = 0, hi = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int64_t x = (o[k] + ((int64_t)1 << (CB + P1 + 2))) >> (CB + P1 + 3);
      bad |= x > 511 || x < -512;
      const int v = (int)(x & 1023);  // jdmaster.c post-IDCT range-limit table
      const uint32_t s = v < 128 ? v + 128 : v < 512 ? 255 : v < 896 ? 0 : v - 896;
      if (k < 4) lo |= s << (8 * k); else hi |= s << (8 * (k - 4));
    }
    *reinterpret_cast<uint2*>(plane + (int64_t)(by * 8 + r) * pw + bx * 8) = make_uint2(lo, hi);
  }
  if (bad) atomicOr(&status[f], ST_RANGE);
}

// jdsample.c for one output sample of component c at (x, y) of the full-size frame.
__device__ __forceinline__ int upsampled(const JpegHdr* h, const uint8_t* p, int c, int x, int y) {
  const int pw = h->bw[c] * 8, dw = h->dw[c], dh = h->dh[c];
  const int hf = h->hmax / (c ? 1 : h->hmax), vf = h->vmax / (c ? 1 : h->vmax);
  auto at = [&](int yy, int xx) { return (int)p[(int64_t)yy * pw + xx]; };
  if (hf == 1 && vf == 1) return at(y, x);
  if (hf == 2 && vf == 1) {
    const int i = x >> 1;
    if (dw <= 2) return at(y, i);
    if (!(x & 1)) return i == 0 ? at(y, 0) : (3 * at(y, i) + at(y, i - 1) + 1) >> 2;
    return i == dw - 1 ? at(y, i) : (3 * at(y, i) + at(y, i + 1) + 2) >> 2;
  }
  const int j = y >> 1;
  const int nj = (y & 1) ? (j + 1 < dh ? j + 1 : dh - 1) : (j > 0 ? j - 1 : 0);
  if (hf == 1) return (3 * at(j, x) + at(nj, x) + ((y & 1) ? 2 : 1)) >> 2;
  const int i = x >> 1;
  if (dw <= 2) return at(j, i);
  const int cs = 3 * at(j, i) + at(nj, i);
  if (!(x & 1)) return i == 0 ? (cs * 4 + 8) >> 4 : (3 * cs + 3 * at(j, i - 1) + at(nj, i - 1) + 8) >> 4;
  return i == dw - 1 ? (cs * 4 + 7) >> 4 : (3 * cs + 3 * at(j, i + 1) + at(nj, i + 1) + 7) >> 4;
}

__device__ __forceinline__ uint8_t clamp255(int v) { return (uint8_t)(v < 0 ? 0 : v > 255 ? 255 : v); }

// One thread per output pixel of the ORIENTED frame (grid.y = frame).  (ox, oy) -> source (x, y) as PIL's
// exif_transpose: 2 FLIP_LEFT_RIGHT, 3 ROTATE_180, 4 FLIP_TOP_BOTTOM, 5 TRANSPOSE, 6 ROTATE_270, 7 TRANSVERSE, 8 ROTATE_90.
__global__ void jpeg_color_kernel(const FrameDesc* fr) {
  const FrameDesc& d = fr[blockIdx.y];
  const JpegHdr* h = reinterpret_cast<const JpegHdr*>(d.blob);
  const int W = h->width, H = h->height, o = d.orient;
  const bool swap = o >= 5 && o <= 8;
  const int Wo = swap ? H : W, Ho = swap ? W : H;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (int64_t)Wo * Ho; i += (int64_t)gridDim.x * blockDim.x) {
    const int ox = (int)(i % Wo), oy = (int)(i / Wo);
    int x = ox, y = oy;
    switch (o) {
      case 2: x = W - 1 - ox; break;
      case 3: x = W - 1 - ox, y = H - 1 - oy; break;
      case 4: y = H - 1 - oy; break;
      case 5: x = oy, y = ox; break;
      case 6: x = oy, y = H - 1 - ox; break;
      case 7: x = W - 1 - oy, y = H - 1 - ox; break;
      case 8: x = W - 1 - oy, y = ox; break;
      default: break;
    }
    uint8_t* out = d.out + i * 3;
    const int Y = upsampled(h, d.planes + h->plane_off[0], 0, x, y);
    if (h->ncomp == 1) {
      out[0] = out[1] = out[2] = (uint8_t)Y;
      continue;
    }
    const int cb = upsampled(h, d.planes + h->plane_off[1], 1, x, y) - 128;
    const int cr = upsampled(h, d.planes + h->plane_off[2], 2, x, y) - 128;
    out[0] = clamp255(Y + ((91881 * cr + 32768) >> 16));
    out[1] = clamp255(Y + ((-22554 * cb + 32768 - 46802 * cr) >> 16));
    out[2] = clamp255(Y + ((116130 * cb + 32768) >> 16));
  }
}

struct Layout {
  int64_t desc, entry, exitst, dirty, nblk, blkstart, active, coef, planes, total;
};

static Layout layout(const ma_jpeg_info* infos, int n, int64_t* subs, int64_t* blocks) {
  int64_t S = 0, B = 0, P = 0;
  for (int i = 0; i < n; ++i) S += infos[i].nsubseq, B += infos[i].nblocks, P += (infos[i].plane_bytes + 15) & ~15;
  Layout L;
  auto al = [](int64_t v) { return (v + 255) & ~(int64_t)255; };
  L.desc = 0;
  L.entry = al(L.desc + (int64_t)sizeof(FrameDesc) * n);
  L.exitst = al(L.entry + 8 * S);
  L.dirty = al(L.exitst + 8 * S);
  L.nblk = al(L.dirty + 4 * S);
  L.blkstart = al(L.nblk + 4 * S);
  L.active = al(L.blkstart + 4 * S);
  L.coef = al(L.active + 4 * (kMaxRounds + 2));
  L.planes = al(L.coef + 128 * B);
  L.total = al(L.planes + P);
  *subs = S, *blocks = B;
  return L;
}

}  // namespace
}  // namespace ma

extern "C" int ma_jpeg_workspace(const ma_jpeg_info* infos, int n, int64_t* bytes) {
  MA_REQUIRE(infos && bytes && n > 0, "ma_jpeg_workspace: infos and bytes must be non-NULL, n > 0");
  int64_t S, B;
  *bytes = layout(infos, n, &S, &B).total;
  return MA_OK;
}

extern "C" int ma_jpeg_decode(const uint8_t* blobs, const int64_t* blob_offsets_host, const ma_jpeg_info* infos_host,
                              int n, uint8_t* const* out_host, const int32_t* orientation_host, void* workspace,
                              int64_t workspace_bytes, int32_t* status, void* stream) {
  MA_REQUIRE(blobs && blob_offsets_host && infos_host && out_host && orientation_host && workspace && status && n > 0,
             "ma_jpeg_decode: NULL argument or n <= 0");
  MA_REQUIRE((reinterpret_cast<uintptr_t>(blobs) & 15) == 0 && (reinterpret_cast<uintptr_t>(workspace) & 255) == 0 &&
                 (reinterpret_cast<uintptr_t>(status) & 3) == 0,
             "ma_jpeg_decode: blobs must be 16-byte, workspace 256-byte and status 4-byte aligned");
  MA_REQUIRE(n <= 65535, "ma_jpeg_decode: at most 65535 frames per call");
  int64_t S, B;
  const Layout L = layout(infos_host, n, &S, &B);
  MA_REQUIRE(workspace_bytes >= L.total, "ma_jpeg_decode: workspace of %lld bytes, %lld needed",
             (long long)workspace_bytes, (long long)L.total);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  std::vector<FrameDesc> fr(n);
  int64_t sb = 0, bb = 0, pb = 0, max_px = 0;
  for (int i = 0; i < n; ++i) {
    MA_REQUIRE((blob_offsets_host[i] & 15) == 0 && out_host[i], "ma_jpeg_decode: frame %d: blob offset not 16-byte aligned or out NULL", i);
    fr[i] = FrameDesc{blobs + blob_offsets_host[i], ws + L.planes + pb, out_host[i], sb, bb, orientation_host[i], 0};
    sb += infos_host[i].nsubseq, bb += infos_host[i].nblocks, pb += (infos_host[i].plane_bytes + 15) & ~15;
    max_px = max_px > (int64_t)infos_host[i].width * infos_host[i].height ? max_px
                                                                         : (int64_t)infos_host[i].width * infos_host[i].height;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  FrameDesc* d_fr = reinterpret_cast<FrameDesc*>(ws + L.desc);
  MA_CHECK_CUDA(cudaMemcpyAsync(d_fr, fr.data(), sizeof(FrameDesc) * n, cudaMemcpyHostToDevice, st));
  MA_CHECK_CUDA(cudaMemsetAsync(ws + L.coef, 0, 128 * B, st));
  MA_CHECK_CUDA(cudaMemsetAsync(status, 0, 4 * n, st));
  Work w{reinterpret_cast<uint64_t*>(ws + L.entry), reinterpret_cast<uint64_t*>(ws + L.exitst),
         reinterpret_cast<int32_t*>(ws + L.dirty),  reinterpret_cast<int32_t*>(ws + L.nblk),
         reinterpret_cast<int32_t*>(ws + L.blkstart), reinterpret_cast<int32_t*>(ws + L.active),
         reinterpret_cast<int16_t*>(ws + L.coef)};
  const int T = 128;
  const unsigned gs = (unsigned)((S + kMaxRounds + 2 + T - 1) / T);
  jpeg_init_kernel<<<gs, T, 0, st>>>(d_fr, n, S, w);
  for (int r = 0; r < kMaxRounds; ++r) jpeg_sync_kernel<<<(unsigned)((S + T - 1) / T), T, 0, st>>>(d_fr, n, S, w, r);
  jpeg_scan_check_kernel<<<n, 256, 0, st>>>(d_fr, w, status);
  jpeg_write_kernel<<<(unsigned)((S + T - 1) / T), T, 0, st>>>(d_fr, n, S, w, status);
  jpeg_dc_kernel<<<n, 256, 0, st>>>(d_fr, w);
  jpeg_idct_kernel<<<(unsigned)((B + 127) / 128), 128, 0, st>>>(d_fr, n, B, w, status);
  const int64_t gx = (max_px + 255) / 256;
  jpeg_color_kernel<<<dim3((unsigned)(gx < 4096 ? gx : 4096), n), 256, 0, st>>>(d_fr);
  MA_CHECK_CUDA(cudaGetLastError());
  return MA_OK;
}
