// encode.cuh -- compress side.
//
//   pass A  k_encode_stats : per chunk, per byte-group: four per-stream 256-bin histograms,
//                            then (one warp per group) the reference's block decisions --
//                            RLE / "not compressible" early-outs, length-limited Huffman
//                            code lengths, table description, exact compressed size,
//                            threshold -> type byte + payload size + saved code lengths.
//   scan    k_encode_scan  : per group inclusive prefix sums of payload sizes -> the
//                            stream's cumulative table, group bases, item offsets, total
//                            length, python header.
//   pass B  k_encode_write : per (chunk, group): raw planes copied, Huffman blocks
//                            bit-packed (per-thread runs, block-wide exclusive scan of bit
//                            lengths, OR into a shared bit buffer, word-coalesced flush)
//                            straight to their final position in the stream.
//
// Replaces reference csrc/zipnn_core.c:294-390 (compression_worker), :105-244
// (prepare_python_return_buffer), hist.c, huf_compress.c:215-724, and the split halves of
// data_manipulation_dtype16.c:64-138 / data_manipulation_dtype32.c:78-133.
#pragma once
#include "common.cuh"
#include "stage1.cuh"

namespace zb {

// Saved per item by pass A for pass B.
struct EncSave {
  uint8_t nb[256];      // code length per symbol (0 = absent)
  uint8_t hdr[128];     // table description (RLE: hdr[0] = the byte)
  uint32_t hsize;       // table description bytes
  uint32_t sbytes[4];   // byte size of each of the 4 bitstreams
  uint32_t lg;          // table log
  uint32_t pad[2];
};
static_assert(sizeof(EncSave) == 416, "EncSave layout");

constexpr int kEncThreads = 256;

// A byte of the (rotated) chunk at byte position pos; words [0, rot_words) are rotated.
template <int G>
__device__ __forceinline__ uint32_t rot_byte_at(const uint8_t* __restrict__ in_c, uint32_t chunk_len, uint32_t rot_words,
                                                uint32_t pos) {
  const uint32_t wi = pos >> 2;
  if (wi >= rot_words) return in_c[pos];
  (void)chunk_len;
  const uint32_t w = rot_word<G>(__ldg(reinterpret_cast<const uint32_t*>(in_c) + wi));
  return (w >> (8 * (pos & 3))) & 0xFFu;
}

// =====================================================================================
// pass A1: histograms.  Pure streaming: every input byte is read once (128-bit loads, four in
// flight per thread), rotated, and counted with one shared-memory atomic.
//
// Counter layout rep[bin][g][col], col = lane % R, 32-bit counters: a warp's 32 atomics go to
// 32 / (32/R) distinct columns, so two lanes can only collide when they hold the same byte
// value.  For G = 2 and 4 a bin's row is 256 bytes, so the counter's byte offset bin << 8 |
// (g * R + col) * 4 is ONE PRMT of the loaded word with a per-lane, per-plane register: two
// instructions per byte with the atomic.  G = 1 (128-byte rows) forms it with one multiply-add,
// which keeps its footprint at 32 KiB.  Per pair of stream quarters the columns are folded
// into hist[item][stream][256] (u16) in global memory for pass A2.
// =====================================================================================
// Columns per bin.  32 = one per lane: no two lanes of a warp ever meet in a bank (1 wavefront per
// atomic instead of 2), at 32 KiB of counters per plane; fp32 has four planes and keeps 16.
// Measured on 16 GiB bf16: 16 columns 5.84 ms, 32 columns 5.07 ms, + two quarters per fold 4.61 ms.
template <int G>
struct HistCfg {
  static constexpr int R = (G == 4) ? 16 : 32;
};

template <int G>
struct HistSmem {
  uint32_t rep[256][G][HistCfg<G>::R];
};
static_assert(sizeof(HistSmem<2>) == 256 * 256 && sizeof(HistSmem<4>) == 256 * 256, "PRMT address form needs 256-byte bin rows");

template <int G>
__global__ void __launch_bounds__(kEncThreads) k_encode_hist(const uint8_t* __restrict__ in, uint64_t n, uint32_t chunk,
                                                             uint64_t K, int bits_mode, uint16_t* __restrict__ hist) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  HistSmem<G>& S = *reinterpret_cast<HistSmem<G>*>(smem_raw);
  constexpr int R = HistCfg<G>::R;
  const int tid = threadIdx.x, lane = tid & 31;
  unsigned char* const rep_b = reinterpret_cast<unsigned char*>(&S.rep[0][0][0]);
  // byte offset of this lane's column of plane g within a bin row (< 256)
  uint32_t col_b[G];
#pragma unroll
  for (int g = 0; g < G; g++) col_b[g] = (uint32_t)(g * R + lane % R) * 4;
  for (int i = tid; i < 256 * G * R; i += kEncThreads) (&S.rep[0][0][0])[i] = 0;
  __syncthreads();
  for (uint64_t c = blockIdx.x; c < K; c += gridDim.x) {
    const uint8_t* in_c = in + c * (uint64_t)chunk;
    const uint32_t chunk_len = (c == K - 1) ? (uint32_t)(n - c * (uint64_t)chunk) : chunk;
    const uint32_t rot_words = (bits_mode == 1 && G > 1) ? (chunk_len >> 2) : 0;
    const bool fast = (chunk_len % 64u) == 0;
    const uint32_t sign_m = rot_words ? ((G == 2) ? 0x00800080u : 0x00800000u) : 0u;  // where the sign bits go
    const uint32_t exp_sh = rot_words ? 1u : 0u;
    for (int q = 0; q < 4; q++) {
      // Two stream quarters share one fold: quarter q counts in the low (q even) or high (q odd) half
      // of the 32-bit counters.  A column receives at most 8 threads x 128 bytes = 1024 per quarter,
      // and a bin at most 32768 in total, so neither half overflows.
      const uint32_t inc = (q & 1) ? 0x10000u : 1u;
      if (fast) {
        const uint32_t qbytes = chunk_len >> 2;  // bytes of input per stream quarter
        const uint4* src = reinterpret_cast<const uint4*>(in_c + (uint64_t)q * qbytes);
        const uint32_t nvec = qbytes >> 4;
        // double-buffered: the next four vectors are in flight while the current four are counted
        uint4 v[4], nv[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
          const uint32_t u = k * kEncThreads + tid;
          nv[k] = (u < nvec) ? __ldg(src + u) : make_uint4(0, 0, 0, 0);
        }
        for (uint32_t u0 = 0; u0 < nvec; u0 += 4 * kEncThreads) {
#pragma unroll
          for (int k = 0; k < 4; k++) v[k] = nv[k];
#pragma unroll
          for (int k = 0; k < 4; k++) {
            const uint32_t u = u0 + (4 + k) * kEncThreads + tid;
            if (u < nvec) nv[k] = __ldg(src + u);
          }
#pragma unroll
          for (int k = 0; k < 4; k++) {
            if (u0 + k * kEncThreads + tid < nvec) {
              uint32_t w[4] = {v[k].x, v[k].y, v[k].z, v[k].w};
#pragma unroll
              for (int i = 0; i < 4; i++) {
                // The sign-bit rotation (rot_word) never builds the rotated word: the exponent bytes are
                // bytes of w << 1, and the sign | mantissa bytes are bytes of one bit-select of w and w >> 8
                // (3 instructions per word instead of 5).
                // Branch-free: without the rotation sign_m = 0 and exp_sh = 0 leave both equal to w.
                uint32_t lo_w, hi_w = w[i] << exp_sh;
                asm("lop3.b32 %0, %1, %2, %3, 0xD8;" : "=r"(lo_w) : "r"(w[i]), "r"(w[i] >> 8), "r"(sign_m));  // sign_m ? b : a
#pragma unroll
                for (int b = 0; b < 4; b++) {
                  const uint32_t g = (4 * i + b) % G;
                  const bool exp_byte = (G == 2 && (b & 1)) || (G == 4 && b == 3);
                  uint32_t off;
                  if constexpr (G == 1) {
                    // extract (PRMT with zeros), then bin * 128 + column on the FMA pipe
                    off = __byte_perm(w[i], 0u, 0x4440u | (uint32_t)b) * (uint32_t)(R * 4) + col_b[0];
                  } else {
                    // bytes (column, byte b, 0, 0): the counter's offset bin << 8 | column in one PRMT
                    off = __byte_perm(exp_byte ? hi_w : lo_w, col_b[g], 0x6504u | ((uint32_t)b << 4));
                  }
                  atomicAdd(reinterpret_cast<uint32_t*>(rep_b + off), inc);
                }
              }
            }
          }
        }
      } else {
        for (int g = 0; g < G; g++) {
          const uint32_t pl = plane_len(chunk_len, G, g);
          const uint32_t seg = (pl + 3) >> 2;
          const uint32_t j0 = min(pl, (uint32_t)q * seg), j1 = (q == 3) ? pl : min(pl, j0 + seg);
          for (uint32_t j = j0 + tid; j < j1; j += kEncThreads)
            atomicAdd(&S.rep[rot_byte_at<G>(in_c, chunk_len, rot_words, j * G + g)][g][lane % R], inc);
        }
      }
      if ((q & 1) == 0) continue;
      __syncthreads();
      // fold the columns of each bin (and clear them); thread t owns bin t of every group.  128-bit
      // accesses, rotated by thread so the eight lanes of an access phase hit distinct banks (G = 4:
      // lanes 4..7 of each phase take the neighbouring plane for the same reason).
      for (int g0 = 0; g0 < G; g0++) {
        const int g = (G == 4) ? (g0 ^ ((tid >> 2) & 1)) : g0;
        uint4* row = reinterpret_cast<uint4*>(&S.rep[tid][g][0]);
        uint32_t sum = 0;
#pragma unroll
        for (int r = 0; r < R / 4; r++) {
          const int rr = (r + tid) % (R / 4);
          const uint4 x = row[rr];
          sum += x.x + x.y + x.z + x.w;
          row[rr] = make_uint4(0, 0, 0, 0);
        }
        uint16_t* h = hist + (((uint64_t)g * K + c) * 4 + (q - 1)) * 256 + tid;
        h[0] = (uint16_t)(sum & 0xFFFFu);
        h[256] = (uint16_t)(sum >> 16);
      }
      __syncthreads();
    }
  }
}

// =====================================================================================
// pass A2: one warp per (group, chunk) item: everything the reference does per block after
// the histogram (huf_compress.c:671-724 + csrc/zipnn_core.c:371-385).
// =====================================================================================
constexpr uint64_t kScanItems = 2048;  // chunks of one group per k_encode_scan CTA

struct __align__(16) TableWarp {
  uint32_t total[256];
  uint8_t nb[256];
  uint8_t nzsym[256];
  TreeScratch tree;
};
constexpr int kTableWarps = 4;

// tANS bytes of the weights T.weight[0..n) (huf_pack_weights' encoder, lines after fse_write_ncount), one warp.
// E.norm holds the normalised counts of the weights 0..max_w at table log lgf (5 or 6).  The spread, the
// next-state table and the per-symbol deltas are built by lane (fse_build_enc), the two interleaved state
// chains run on lane 0 over per-position deltas prepared by lane, and the emitted bits are placed by a warp
// prefix sum.  Scratch: T.cnt (per-position deltas), T.parent (emissions), T.depth (bit words).  Returns the
// byte count written to dst; every lane gets it.
__device__ int warp_fse_encode(TreeScratch& T, int n, int max_w, int lgf, uint8_t* dst) {
  const int lane = threadIdx.x & 31;
  const unsigned full = 0xffffffffu, lt = (1u << lane) - 1u;
  FseEnc& E = T.fse;
  const uint32_t size = 1u << lgf, mask = size - 1, step = (size >> 1) + (size >> 3) + 3;
  // ---- per symbol (lane s <= max_w <= 12): cumul, place of the low-probability symbols, deltas
  const bool is_sym = lane <= max_w;
  const int nrm = is_sym ? E.norm[lane] : 0;
  const uint32_t slots = nrm == -1 ? 1u : (nrm > 0 ? (uint32_t)nrm : 0u);  // cumul increment
  const uint32_t occ = nrm > 0 ? (uint32_t)nrm : 0u;                      // slots taken by the spread walk
  uint32_t cum = slots, pstart = occ;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t a = __shfl_up_sync(full, cum, o), b = __shfl_up_sync(full, pstart, o);
    if (lane >= o) { cum += a; pstart += b; }
  }
  cum -= slots;
  pstart -= occ;
  const uint32_t low = __ballot_sync(full, is_sym && nrm == -1);
  const uint32_t high = size - 1 - __popc(low);
  if (is_sym && nrm == -1) E.spread[size - 1 - __popc(low & lt)] = (uint8_t)lane;
  uint32_t db = 0;
  int32_t df = 0;
  if (nrm == 0) {
    db = ((uint32_t)(lgf + 1) << 16) - size;
  } else if (nrm == -1 || nrm == 1) {
    db = ((uint32_t)lgf << 16) - size;
    df = (int32_t)cum - 1;
  } else {
    const uint32_t max_out = (uint32_t)lgf - (uint32_t)hb32((uint32_t)(nrm - 1));
    db = (max_out << 16) - ((uint32_t)nrm << max_out);
    df = (int32_t)cum - nrm;
  }
  // ---- spread: the positions j * step & mask (j = 0, 1, ..) that are <= high take the positive symbols'
  // slots in symbol order, which is the walk of fse_build_enc with its skips
  uint32_t before = 0;
  for (uint32_t j0 = 0; j0 < size; j0 += 32) {
    const uint32_t u = ((j0 + lane) * step) & mask;
    const bool valid = u <= high;
    const uint32_t vm = __ballot_sync(full, valid);
    const uint32_t r = before + __popc(vm & lt);
    before += __popc(vm);
    int sym = 0;
    for (int s = 0; s <= max_w; s++) {
      const uint32_t ps = __shfl_sync(full, pstart, s), pc = __shfl_sync(full, occ, s);
      if (r >= ps && r < ps + pc) sym = s;
    }
    if (valid) E.spread[u] = (uint8_t)sym;
  }
  if (is_sym) E.cumul[lane] = cum;
  if (lane < 16) E.count[lane] = 0;  // reused: occurrences of each symbol in spread[0, 32)
  __syncwarp();
  // ---- next_state[cumul[s] + k] = size + u for the k-th u with spread[u] = s
  {
    const uint32_t s0 = E.spread[lane];
    const uint32_t m0 = __match_any_sync(full, s0);
    E.next_state[E.cumul[s0] + __popc(m0 & lt)] = (uint16_t)(size + lane);
    if (size > 32) {
      E.count[s0] = __popc(m0);
      __syncwarp();
      const uint32_t s1 = E.spread[32 + lane];
      const uint32_t m1 = __match_any_sync(full, s1);
      E.next_state[E.cumul[s1] + E.count[s1] + __popc(m1 & lt)] = (uint16_t)(size + 32 + lane);
    }
  }
  // ---- the deltas of the weight at every position
  uint32_t* pdb = T.cnt;
  int32_t* pdf = reinterpret_cast<int32_t*>(T.cnt + 256);
  for (int i0 = 0; i0 < n; i0 += 32) {
    const int i = i0 + lane;
    const int w = i < n ? T.weight[i] : 0;
    const uint32_t a = __shfl_sync(full, db, w);
    const int32_t b = __shfl_sync(full, df, w);
    if (i < n) {
      pdb[i] = a;
      pdf[i] = b;
    }
  }
  __syncwarp();
  // ---- the two state chains (huf_pack_weights' order): emissions value | nbits << 8
  uint16_t* em = T.parent;
  int nem = 0;
  if (lane == 0) {
    const uint16_t* ns = E.next_state;
    auto seed = [&](int i) {
      const uint32_t d = pdb[i], nb = (d + (1u << 15)) >> 16;
      return (uint32_t)ns[(int32_t)((((nb << 16) - d)) >> nb) + pdf[i]];
    };
    auto emit = [&](uint32_t st, int i) {
      const uint32_t nb = (st + pdb[i]) >> 16;
      em[nem++] = (uint16_t)((st & ((1u << nb) - 1u)) | (nb << 8));
      return (uint32_t)ns[(int32_t)(st >> nb) + pdf[i]];
    };
    int ip = n;
    uint32_t s1, s2;
    if (n & 1) {
      s1 = seed(--ip);
      s2 = seed(--ip);
      s1 = emit(s1, --ip);
    } else {
      s2 = seed(--ip);
      s1 = seed(--ip);
    }
    while (ip > 0) {
      s2 = emit(s2, --ip);
      s1 = emit(s1, --ip);
    }
    em[nem++] = (uint16_t)((s2 & mask) | ((uint32_t)lgf << 8));
    em[nem++] = (uint16_t)((s1 & mask) | ((uint32_t)lgf << 8));
    em[nem++] = (uint16_t)(1u | (1u << 8));  // end mark
  }
  nem = __shfl_sync(full, nem, 0);
  // ---- place the emissions LSB first: warp prefix sum of their lengths, OR into words
  uint32_t* words = reinterpret_cast<uint32_t*>(T.depth);
  for (int i = lane; i < 128; i += 32) words[i] = 0;
  __syncwarp();
  uint32_t at = 0;
  for (int e0 = 0; e0 < nem; e0 += 32) {
    const uint32_t v = (e0 + lane < nem) ? em[e0 + lane] : 0u;
    const uint32_t len = v >> 8;
    uint32_t x = len;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t y = __shfl_up_sync(full, x, o);
      if (lane >= o) x += y;
    }
    const uint32_t off = at + x - len, bits = v & 0xFFu;
    if (len) {
      atomicOr(&words[off >> 5], bits << (off & 31));
      if ((off & 31) + len > 32) atomicOr(&words[(off >> 5) + 1], bits >> (32 - (off & 31)));
    }
    at += __shfl_sync(full, x, 31);
  }
  __syncwarp();
  const int bytes = (int)((at + 7) >> 3);
  for (int i = lane; i < bytes; i += 32) dst[i] = (uint8_t)(words[i >> 2] >> (8 * (i & 3)));
  __syncwarp();
  return bytes;
}

// Table description from the code lengths nb[256], one warp: the bytes of huf_write_table (huf_serial.cuh,
// which the host tests fuzz against the oracle), with the weights, their histogram, the tANS tables and
// the nibble form built by lane.  Writes T.hdr; returns its size or -1 (block kept raw), on every lane.
__device__ int warp_write_table(TreeScratch& T, const uint8_t* nb, int max_sym, int lg) {
  const int lane = threadIdx.x & 31;
  const unsigned full = 0xffffffffu;
  FseEnc& E = T.fse;
  const int n = max_sym;  // weights of symbols 0..max_sym-1 are sent, the last one is implied
  if (lane < 16) E.count[lane] = 0;
  __syncwarp();
  int max_w = 0;
  for (int s = lane; s <= n; s += 32) {
    const uint32_t w = (s < n && nb[s]) ? (uint32_t)(lg + 1 - nb[s]) : 0u;
    T.weight[s] = (uint8_t)w;  // weight[max_sym] = 0 pads the nibble form
    if (s < n) {
      atomicAdd(&E.count[w], 1u);
      max_w = max(max_w, (int)w);
    }
  }
  max_w = __reduce_max_sync(full, max_w);
  __syncwarp();
  // ---- huf_pack_weights' decisions; h = its return value
  int h = 0;
  if (n > 1) {
    const uint32_t top = __reduce_max_sync(full, lane <= max_w ? E.count[lane] : 0u);
    if (top == (uint32_t)n) {
      h = 1;
    } else if (top > 1) {
      const int lgf = fse_pick_log(6, (uint32_t)n, (uint32_t)max_w, 2);
      int hn = -1;
      if (lane == 0 && fse_normalize(E.norm, lgf, E.count, (uint32_t)n, max_w) == 0)
        hn = fse_write_ncount(T.hdr + 1, E.norm, max_w, lgf);
      hn = __shfl_sync(full, hn, 0);
      __syncwarp();
      if (hn < 0) {
        h = -1;
      } else if (n <= 2) {
        h = 0;
      } else if (hn + 1 >= max_sym / 2) {
        h = hn + 1;  // the bitstream adds at least one byte, so the nibble form (or raw) is chosen anyway
      } else {
        h = hn + warp_fse_encode(T, n, max_w, lgf, T.hdr + 1 + hn);
      }
    }
  }
  if (h < 0) return -1;
  if (h > 1 && h < max_sym / 2) {
    if (lane == 0) T.hdr[0] = (uint8_t)h;
    __syncwarp();
    return h + 1;
  }
  if (max_sym > 128) return -1;
  if (lane == 0) T.hdr[0] = (uint8_t)(128 + (max_sym - 1));
  for (int s = 2 * lane; s < max_sym; s += 64) T.hdr[(s / 2) + 1] = (uint8_t)((T.weight[s] << 4) + T.weight[s + 1]);
  __syncwarp();
  return ((max_sym + 1) / 2) + 1;
}

// hist = this item's four per-stream histograms, u16[4][256] in global memory (read twice: totals, exact sizes)
__device__ void warp_block_decision(TableWarp& S, const uint16_t* __restrict__ hist, uint32_t plen, double thr, uint8_t* type_out,
                                    uint32_t* size_out, EncSave* save) {
  const int lane = threadIdx.x & 31;
  uint32_t* total = S.total;
  uint32_t largest = 0;
  int max_sym = -1;
  for (int s = lane; s < 256; s += 32) {
    const uint32_t t = (uint32_t)__ldg(hist + s) + __ldg(hist + 256 + s) + __ldg(hist + 512 + s) + __ldg(hist + 768 + s);
    total[s] = t;
    largest = max(largest, t);
    if (t) max_sym = s;
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    largest = max(largest, __shfl_xor_sync(0xffffffffu, largest, o));
    max_sym = max(max_sym, __shfl_xor_sync(0xffffffffu, max_sym, o));
  }
  __syncwarp();
  uint8_t type = 0;
  uint32_t size = plen;
  bool huf = false;
  if (plen == 0 || plen > (uint32_t)kHufBlockMax) {
    // empty plane, or HUF_compress rejects > 128 KiB (huf_compress.c:658) -> raw
  } else if (largest == plen) {
    if (1.0 < (double)plen * thr) {  // RLE block of 1 byte (huf_compress.c:673)
      type = 1;
      size = 1;
      if (lane == 0) {
        save->hdr[0] = (uint8_t)max_sym;
        save->hsize = 0;
      }
    }
  } else if (largest <= (plen >> 7) + 4) {
    // heuristic "probably not compressible" (huf_compress.c:674)
  } else {
    huf = true;
  }
  if (huf) {
    // ---- order the present symbols: count descending, symbol ascending ----
    TreeScratch& T = S.tree;
    uint8_t* nz = S.nzsym;
    int k = 0;
    for (int base = 0; base < 256; base += 32) {
      const int s = base + lane;
      const bool p = total[s] != 0;
      const uint32_t m = __ballot_sync(0xffffffffu, p);
      if (p) nz[k + __popc(m & ((1u << lane) - 1u))] = (uint8_t)s;
      k += __popc(m);
    }
    __syncwarp();
    for (int i = lane; i < k; i += 32) {
      const uint32_t c = total[nz[i]];
      int rank = 0;
      for (int j = 0; j < k; j++) {
        const uint32_t cj = total[nz[j]];
        rank += (cj > c) || (cj == c && j < i);
      }
      T.cnt[rank] = c;
      T.sym[rank] = nz[i];
    }
    __syncwarp();
    int lg = 0;
    if (lane == 0) lg = huf_tree_depths(T, k - 1, fse_pick_log(kHufLogDefault, plen, (uint32_t)max_sym, 1));
    for (int s = lane; s < 256; s += 32) S.nb[s] = 0;
    lg = __shfl_sync(0xffffffffu, lg, 0);
    __syncwarp();
    for (int i = lane; i < k; i += 32) S.nb[T.sym[i]] = T.depth[i];
    __syncwarp();
    const int hsize = warp_write_table(T, S.nb, max_sym, lg);
    if (hsize > 0 && (uint32_t)hsize + 12 < plen && plen >= 12) {
      uint32_t bits[4] = {0, 0, 0, 0};
      for (int s = lane; s <= max_sym; s += 32) {
        const uint32_t l = S.nb[s];
#pragma unroll
        for (int q = 0; q < 4; q++) bits[q] += (uint32_t)__ldg(hist + 256 * q + s) * l;
      }
#pragma unroll
      for (int q = 0; q < 4; q++)
#pragma unroll
        for (int o = 16; o; o >>= 1) bits[q] += __shfl_xor_sync(0xffffffffu, bits[q], o);
      uint32_t sb[4], csize = (uint32_t)hsize + 6;
#pragma unroll
      for (int q = 0; q < 4; q++) {
        sb[q] = (bits[q] >> 3) + 1;  // ceil((bits + end mark) / 8), bitstream.h:254-260
        csize += sb[q];
      }
      // (the reference's dst capacity, = chunk, can only bind when the block is kept raw anyway)
      if (csize < plen - 1 && (double)csize < (double)plen * thr) {  // huf_compress.c:625, zipnn_core.c:371-373
        type = 1;
        size = csize;
        for (int s = lane; s < 256; s += 32) save->nb[s] = S.nb[s];
        for (int i = lane; i < hsize; i += 32) save->hdr[i] = T.hdr[i];
        if (lane == 0) {
          save->hsize = (uint32_t)hsize;
          save->lg = (uint32_t)lg;
#pragma unroll
          for (int q = 0; q < 4; q++) save->sbytes[q] = sb[q];
        }
      }
    }
  }
  if (lane == 0) {
    *type_out = type;
    *size_out = size;
  }
}

template <int G>
__global__ void __launch_bounds__(kTableWarps * 32) k_encode_table(const uint16_t* __restrict__ hist, uint64_t n, uint32_t chunk,
                                                                   uint64_t K, double thr, uint8_t* types, uint32_t* sizes,
                                                                   EncSave* saves, unsigned long long* partials) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  TableWarp& S = reinterpret_cast<TableWarp*>(smem_raw)[threadIdx.x >> 5];
  const int lane = threadIdx.x & 31;
  const uint64_t nitems = (uint64_t)G * K;
  for (uint64_t item = (uint64_t)blockIdx.x * kTableWarps + (threadIdx.x >> 5); item < nitems;
       item += (uint64_t)gridDim.x * kTableWarps) {
    const int g = (int)(item / K);
    const uint64_t c = item - (uint64_t)g * K;
    const uint32_t chunk_len = (c == K - 1) ? (uint32_t)(n - c * (uint64_t)chunk) : chunk;
    warp_block_decision(S, hist + item * 1024, plane_len(chunk_len, G, g), thr, types + item, sizes + item, saves + item);
    __syncwarp();
    // payload bytes of this group per block of kScanItems chunks: lets the scan run on many CTAs
    if (lane == 0) atomicAdd(partials + (uint64_t)g * ((K + kScanItems - 1) / kScanItems) + c / kScanItems, (unsigned long long)sizes[item]);
  }
}

// =====================================================================================
// scan: sizes -> cumulative table (written into the stream), bases, item offsets, header.
// =====================================================================================
constexpr int kScanThreads = 256;
// (kScanItems = kScanThreads * 8 chunks of one group per CTA, declared above k_encode_table)

// One CTA per (group, block of kScanItems chunks).  The table kernel left the payload bytes of every
// such block in partials[g][blk]; a CTA adds up what lies in front of it (all blocks of the groups
// before, the earlier blocks of its own group), scans its own 2048 sizes (8 per thread) and writes its
// slice of the cumulative table, the item offsets and the type bytes.  CTA 0 also writes the header.
__global__ void __launch_bounds__(kScanThreads) k_encode_scan(const uint32_t* __restrict__ sizes, const uint8_t* __restrict__ types,
                                                              int G, uint64_t K, const uint8_t* __restrict__ hdr_dev,
                                                              uint32_t hdr_len, uint8_t* out, uint64_t* item_off, Ctrl* ctrl,
                                                              const unsigned long long* __restrict__ partials) {
  __shared__ uint64_t warp_tot[kScanThreads / 32];
  __shared__ uint64_t red[kScanThreads / 32][3];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint64_t nitems = (uint64_t)G * K;
  const uint64_t nblk = (K + kScanItems - 1) / kScanItems;
  const int g = (int)(blockIdx.x / nblk);
  const uint64_t blk = blockIdx.x - (uint64_t)g * nblk;
  // ---- what lies in front of this CTA: whole earlier groups, earlier blocks of this group, everything
  uint64_t s_groups = 0, s_blocks = 0, s_all = 0;
  for (uint64_t i = tid; i < (uint64_t)G * nblk; i += kScanThreads) {
    const uint64_t v = partials[i];
    const uint64_t gi = i / nblk;
    s_all += v;
    if (gi < (uint64_t)g) s_groups += v;
    if (gi == (uint64_t)g && i - gi * nblk < blk) s_blocks += v;
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    s_groups += __shfl_xor_sync(0xffffffffu, s_groups, o);
    s_blocks += __shfl_xor_sync(0xffffffffu, s_blocks, o);
    s_all += __shfl_xor_sync(0xffffffffu, s_all, o);
  }
  if (lane == 0) { red[warp][0] = s_groups; red[warp][1] = s_blocks; red[warp][2] = s_all; }
  __syncthreads();
  s_groups = s_blocks = s_all = 0;
  for (int w = 0; w < kScanThreads / 32; w++) { s_groups += red[w][0]; s_blocks += red[w][1]; s_all += red[w][2]; }
  const uint64_t payload0 = (uint64_t)hdr_len + 9 * nitems;
  const uint64_t base = payload0 + s_groups;  // first payload byte of group g
  // ---- this CTA's chunks: 8 consecutive ones per thread
  const uint64_t c_first = blk * kScanItems + (uint64_t)tid * 8;
  uint32_t v[8];
  uint64_t run = 0;
#pragma unroll
  for (int j = 0; j < 8; j++) {
    v[j] = (c_first + j < K) ? sizes[(uint64_t)g * K + c_first + j] : 0u;
    run += v[j];
  }
  uint64_t x = run;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint64_t y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) warp_tot[warp] = x;
  __syncthreads();
  uint64_t pre = s_blocks + x - run;
  for (int w = 0; w < warp; w++) pre += warp_tot[w];
  uint8_t* cum_out = out + hdr_len + nitems;
#pragma unroll
  for (int j = 0; j < 8; j++) {
    const uint64_t c = c_first + j;
    if (c < K) {
      const uint64_t i = (uint64_t)g * K + c;
      item_off[i] = base + pre;
      pre += v[j];
      st_u64_bytes(cum_out + 8 * i, pre);  // inclusive, counted from the start of the group
      out[hdr_len + i] = types[i];
    }
  }
  if (blk == 0 && tid == 0) {
    ctrl->base[g] = base;
    uint64_t tot = 0;
    for (uint64_t j = 0; j < nblk; j++) tot += partials[(uint64_t)g * nblk + j];
    ctrl->group_total[g] = tot;
  }
  if (blockIdx.x == 0) {
    // python header with the total length patched in (csrc/zipnn_core.c:121)
    const uint64_t total = payload0 + s_all;
    for (uint32_t i = tid; i < hdr_len; i += kScanThreads) {
      uint8_t b = hdr_dev[i];
      if (i >= 24 && i < 32) b = (uint8_t)(total >> (8 * (i - 24)));
      out[i] = b;
    }
    if (tid == 0) ctrl->total_len = total;
  }
}

// =====================================================================================
// pass B
// =====================================================================================
constexpr uint32_t kEncTile = kEncThreads * 16;             // plane bytes per tile (4096)
constexpr uint32_t kBitBufWords = (kEncTile * 11) / 32 + 8;  // worst-case tile bits + carry

struct WriteSmem {
  __align__(16) uint8_t tile[kEncTile + 16];
  uint32_t bitbuf[kBitBufWords];
  uint32_t code[256];  // val | nb << 16
  uint32_t warp_sum[kEncThreads / 32];
  EncSave save;
};

// Fill S.tile[0..cnt) with bytes [p0, p0+cnt) of plane g of the (rotated) chunk.
template <int G>
__device__ __forceinline__ void stage_tile(uint8_t* tile, const uint8_t* __restrict__ in_c, uint32_t chunk_len,
                                           uint32_t rot_words, int g, uint32_t p0, uint32_t cnt) {
  const int tid = threadIdx.x;
  const bool fast = ((p0 * G) % 16u) == 0 && (cnt % 16u) == 0 && ((p0 + cnt) * (uint32_t)G <= (chunk_len & ~3u));
  if (fast) {
    for (uint32_t u = tid; u < (cnt >> 4); u += kEncThreads) {
      const uint4* src = reinterpret_cast<const uint4*>(in_c + (uint64_t)(p0 + 16 * u) * G);
      uint32_t w[4 * G];
#pragma unroll
      for (int i = 0; i < G; i++) {
        const uint4 v = __ldg(src + i);
        w[4 * i] = v.x; w[4 * i + 1] = v.y; w[4 * i + 2] = v.z; w[4 * i + 3] = v.w;
      }
      if (rot_words) {
#pragma unroll
        for (int i = 0; i < 4 * G; i++) w[i] = rot_word<G>(w[i]);
      }
      uint4 pv[G];
      split16<G>(w, pv);
      uint4 mine = pv[0];
#pragma unroll
      for (int k = 1; k < G; k++)
        if (g == k) mine = pv[k];
      *reinterpret_cast<uint4*>(tile + 16 * u) = mine;
    }
  } else {
    for (uint32_t j = tid; j < cnt; j += kEncThreads)
      tile[j] = (uint8_t)rot_byte_at<G>(in_c, chunk_len, rot_words, (p0 + j) * G + g);
  }
}

// Copy tile[0..cnt) to the (arbitrarily aligned) global address dst.
__device__ __forceinline__ void tile_to_global(const uint8_t* tile, uint8_t* dst, uint32_t cnt) {
  const int tid = threadIdx.x;
  const uint32_t head = min(cnt, (uint32_t)((16 - ((uintptr_t)dst & 15)) & 15));
  if ((uint32_t)tid < head) dst[tid] = tile[tid];
  const uint32_t nvec = (cnt - head) >> 4;
  const uint32_t* t32 = reinterpret_cast<const uint32_t*>(tile);
  for (uint32_t v = tid; v < nvec; v += kEncThreads) {
    const uint32_t o = head + 16 * v;
    const uint32_t sh = (o & 3) * 8;
    const uint32_t* p = t32 + (o >> 2);
    const uint32_t a0 = p[0], a1 = p[1], a2 = p[2], a3 = p[3], a4 = p[4];  // tile has 16 B of slack
    *reinterpret_cast<uint4*>(dst + o) = make_uint4(__funnelshift_r(a0, a1, sh), __funnelshift_r(a1, a2, sh),
                                                    __funnelshift_r(a2, a3, sh), __funnelshift_r(a3, a4, sh));
  }
  const uint32_t done = head + 16 * nvec;
  if ((uint32_t)tid < cnt - done) dst[done + tid] = tile[done + tid];
}

// Canonical code values from lengths, one warp (huf_compress.c:390-407).  Entry formats:
//   kLeftAligned = false: val | nb << 16 (k_encode_write);
//   kLeftAligned = true : val << (32 - nb) | nb, 0 for an absent symbol (k_encode_write_warp).  The value sits at
//                         the top of the word and the length in bits 0..4 (bits 5..20 are zero), so a wrapping
//                         funnel shift by the entry itself appends the code to a run in one instruction, and sums
//                         of entries carry the exact sum of lengths in their low 21 bits (see wb_run).
template <bool kLeftAligned>
__device__ __forceinline__ void warp_build_codes(const uint8_t* nb, int lg, uint32_t* code) {
  const int lane = threadIdx.x & 31;
  uint32_t per_len[kHufLogMax + 1];
#pragma unroll
  for (int l = 0; l <= kHufLogMax; l++) per_len[l] = 0;
  for (int base = 0; base < 256; base += 32) {
    const int mine = nb[base + lane];
#pragma unroll
    for (int l = 1; l <= kHufLogMax; l++) per_len[l] += __popc(__ballot_sync(0xffffffffu, mine == l));
  }
  uint32_t start[kHufLogMax + 1];
  {
    uint32_t v = 0;
#pragma unroll
    for (int l = kHufLogMax; l >= 1; l--) {
      if (l <= lg) {
        start[l] = v;
        v = (v + per_len[l]) >> 1;
      } else {
        start[l] = 0;
      }
    }
  }
  for (int base = 0; base < 256; base += 32) {
    const int mine = nb[base + lane];
    uint32_t val = 0;
#pragma unroll
    for (int l = 1; l <= kHufLogMax; l++) {
      const uint32_t m = __ballot_sync(0xffffffffu, mine == l);
      if (mine == l) val = start[l] + __popc(m & ((1u << lane) - 1u));
      start[l] += __popc(m);
    }
    code[base + lane] = kLeftAligned ? (mine ? (val << (32 - mine)) | (uint32_t)mine : 0u) : (val | ((uint32_t)mine << 16));
  }
}

template <int G>
__global__ void __launch_bounds__(kEncThreads) k_encode_write(const uint8_t* __restrict__ in, uint64_t n, uint32_t chunk, uint64_t K,
                                                              int bits_mode, const uint8_t* __restrict__ types,
                                                              const uint32_t* __restrict__ sizes, const EncSave* __restrict__ saves,
                                                              const uint64_t* __restrict__ item_off, uint8_t* out,
                                                              int only_ragged) {
  __shared__ WriteSmem S;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint64_t nitems = (uint64_t)G * K;
  // only_ragged: just the G items of the last chunk (launched with G blocks)
  const uint64_t first = only_ragged ? (uint64_t)blockIdx.x * K + (K - 1) : blockIdx.x;
  const uint64_t step = only_ragged ? nitems : gridDim.x;
  for (uint64_t item = first; item < nitems; item += step) {
    const int g = (int)(item / K);
    const uint64_t c = item - (uint64_t)g * K;
    const uint8_t* in_c = in + c * (uint64_t)chunk;
    const uint32_t chunk_len = (c == K - 1) ? (uint32_t)(n - c * (uint64_t)chunk) : chunk;
    if (only_ragged && chunk_len % (64u * G) == 0) continue;  // k_encode_write_warp takes those
    const uint32_t rot_words = (bits_mode == 1 && G > 1) ? (chunk_len >> 2) : 0;
    const uint32_t plen = plane_len(chunk_len, G, g);
    uint8_t* dest = out + item_off[item];
    const uint8_t type = types[item];
    const uint32_t size = sizes[item];
    if (plen == 0) continue;
    __syncthreads();
    if (type == 0) {
      for (uint32_t p0 = 0; p0 < plen; p0 += kEncTile) {
        const uint32_t cnt = min(kEncTile, plen - p0);
        stage_tile<G>(S.tile, in_c, chunk_len, rot_words, g, p0, cnt);
        __syncthreads();
        tile_to_global(S.tile, dest + p0, cnt);
        __syncthreads();
      }
      continue;
    }
    if (size == 1) {
      if (tid == 0) dest[0] = saves[item].hdr[0];
      continue;
    }
    // ---- Huffman block: table description, jump table, 4 bitstreams ----
    {
      const uint32_t* sv = reinterpret_cast<const uint32_t*>(saves + item);
      uint32_t* dv = reinterpret_cast<uint32_t*>(&S.save);
      for (int i = tid; i < (int)(sizeof(EncSave) / 4); i += kEncThreads) dv[i] = sv[i];
    }
    __syncthreads();
    const uint32_t hsize = S.save.hsize;
    if (warp == 0) warp_build_codes<false>(S.save.nb, (int)S.save.lg, S.code);
    if (warp == 1) {
      for (uint32_t i = lane; i < hsize; i += 32) dest[i] = S.save.hdr[i];
      if (lane < 3) {
        dest[hsize + 2 * lane] = (uint8_t)S.save.sbytes[lane];
        dest[hsize + 2 * lane + 1] = (uint8_t)(S.save.sbytes[lane] >> 8);
      }
    }
    __syncthreads();
    const uint32_t seg = (plen + 3) >> 2;
    uint32_t stream_at = hsize + 6;
    for (int i = 0; i < 4; i++) {
      const uint32_t s_begin = (uint32_t)i * seg;
      const uint32_t s_end = (i == 3) ? plen : s_begin + seg;
      uint8_t* gaddr = dest + stream_at;
      const uint32_t sbytes = S.save.sbytes[i];
      stream_at += sbytes;
      const uint32_t a = (uint32_t)((uintptr_t)gaddr & 3);
      uint32_t* gword = reinterpret_cast<uint32_t*>(gaddr - a);
      uint32_t B = 8 * a;       // bits placed so far, counted from the aligned word base
      uint32_t flushed = 0;     // whole words already written to global
      for (uint32_t w = tid; w < kBitBufWords; w += kEncThreads) S.bitbuf[w] = 0;
      __syncthreads();
      for (uint32_t p1 = s_end; p1 > s_begin;) {
        const uint32_t p0 = (p1 - s_begin > kEncTile) ? p1 - kEncTile : s_begin;
        const uint32_t cnt = p1 - p0;
        stage_tile<G>(S.tile, in_c, chunk_len, rot_words, g, p0, cnt);
        __syncthreads();
        // ---- this thread's 16 symbols, in emission order (last plane byte first) ----
        const uint32_t e0 = 16u * tid;
        const int nvalid = (int)min(16u, cnt > e0 ? cnt - e0 : 0u);
        uint64_t v[4] = {0, 0, 0, 0};
        uint32_t l[4] = {0, 0, 0, 0};
        if (nvalid == 16 && (cnt & 15u) == 0) {
          const uint4 q = *reinterpret_cast<const uint4*>(S.tile + (cnt - 16 - e0));
          const uint32_t wv[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
          for (int k = 0; k < 16; k++) {
            const uint32_t sym = (wv[(15 - k) >> 2] >> (8 * ((15 - k) & 3))) & 0xFFu;
            const uint32_t cd = S.code[sym];
            v[k >> 2] |= (uint64_t)(cd & 0xFFFFu) << l[k >> 2];
            l[k >> 2] += cd >> 16;
          }
        } else {
          for (int k = 0; k < nvalid; k++) {
            const uint32_t cd = S.code[S.tile[cnt - 1 - (e0 + k)]];
            v[k >> 2] |= (uint64_t)(cd & 0xFFFFu) << l[k >> 2];
            l[k >> 2] += cd >> 16;
          }
        }
        const uint32_t mine = l[0] + l[1] + l[2] + l[3];
        // ---- block-wide exclusive scan of bit lengths ----
        uint32_t x = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
          if (lane >= o) x += y;
        }
        if (lane == 31) S.warp_sum[warp] = x;
        __syncthreads();
        uint32_t pre = 0, tile_bits = 0;
#pragma unroll
        for (int w = 0; w < kEncThreads / 32; w++) {
          const uint32_t t = S.warp_sum[w];
          if (w < warp) pre += t;
          tile_bits += t;
        }
        uint32_t off = (B - 32 * flushed) + pre + x - mine;
#pragma unroll
        for (int r = 0; r < 4; r++) {
          if (l[r]) {
            const uint32_t sh = off & 31, wi = off >> 5;
            const uint32_t lo32 = (uint32_t)v[r], hi32 = (uint32_t)(v[r] >> 32);
            const uint32_t w0 = lo32 << sh;
            const uint32_t w1 = __funnelshift_l(lo32, hi32, sh);
            const uint32_t w2 = sh ? (hi32 >> (32 - sh)) : 0u;
            if (w0) atomicOr(&S.bitbuf[wi], w0);
            if (w1) atomicOr(&S.bitbuf[wi + 1], w1);
            if (w2) atomicOr(&S.bitbuf[wi + 2], w2);
            off += l[r];
          }
        }
        __syncthreads();
        B += tile_bits;
        // ---- flush the words that are complete ----
        const uint32_t complete = (B >> 5) - flushed;
        for (uint32_t w = tid; w < complete; w += kEncThreads) {
          const uint32_t val = S.bitbuf[w];
          if (flushed + w == 0 && a != 0) {
            for (uint32_t bb = a; bb < 4; bb++) gaddr[bb - a] = (uint8_t)(val >> (8 * bb));
          } else {
            gword[flushed + w] = val;
          }
        }
        const uint32_t carry = S.bitbuf[complete];
        __syncthreads();
        for (uint32_t w = tid; w <= complete + 1 && w < kBitBufWords; w += kEncThreads) S.bitbuf[w] = 0;
        __syncthreads();
        if (tid == 0) S.bitbuf[0] = carry;
        flushed += complete;
        p1 = p0;
        __syncthreads();
      }
      // ---- end mark + the last (partial) bytes ----
      if (tid == 0) S.bitbuf[(B - 32 * flushed) >> 5] |= 1u << (B & 31);
      __syncthreads();
      {
        const uint32_t first_byte = max(4 * flushed, a);   // relative to the aligned base
        const uint32_t end_byte = a + sbytes;              // exclusive
        for (uint32_t bb = first_byte + tid; bb < end_byte; bb += kEncThreads) {
          const uint32_t rel = bb - 4 * flushed;
          gaddr[bb - a] = (uint8_t)(S.bitbuf[rel >> 2] >> (8 * (rel & 3)));
        }
      }
      __syncthreads();
    }
  }
}

// =====================================================================================
// pass B, regular chunks (chunk_len % (64*G) == 0): one CTA of 4 warps per chunk, warp s owns
// the s-th quarter of every byte plane -- exactly one huff0 bitstream of each coded plane
// (huf_compress.c:552-603) and a contiguous quarter of each raw plane.  The chunk is read
// once (128-bit loads, the next tile prefetched), split in registers, and every plane is
// finished by the same warp: no block-wide synchronisation after the per-chunk setup.
// A warp step covers H halves of 512 plane bytes; a lane holds 16 bytes of each half.
//   coded plane: 16 symbols per lane and half -> 4 runs of <= 44 bits each, ONE warp suffix
//                scan of the bit lengths of all halves (the last symbol is emitted first,
//                huf_compress.c:474-499), OR into a warp-private bit buffer whose words are
//                aligned with the destination's 32-bit words, coalesced flush of the completed
//                words;
//   raw plane  : the step's bytes staged in shared memory, written with aligned 128-bit stores
//                (funnel-shifted to the destination's alignment), byte stores at the edges.
// =====================================================================================
constexpr int kWbWarps = 4;

// H = 2 (32 symbols per lane per step) pays the scan, the flush, the loop head and the raw plane's
// edge bytes once per 1024 plane bytes.  fp32's four planes keep H = 1: its step already needs
// about 120 registers.
template <int G>
struct WbCfg {
  static constexpr int H = (G == 4) ? 1 : 2;
  static constexpr uint32_t kTile = 512u * H;                    // plane bytes per warp step
  // CTAs per SM the register budget has to allow: G = 1 72 registers, G = 2 96, G = 4 121 (sm_100a, no spills)
  static constexpr int kMinBlocks = (G == 4) ? 4 : (G == 2 ? 5 : 7);
  // worst case: 11-bit codes on every symbol, behind a carry of < 32 bits; the last run's third word
  // lies at most two words past the word holding its first bit
  static constexpr uint32_t kBitWords = (kTile * 11 + 31) / 32 + 3;
};

// The four symbols of plane word w, byte 3 first (emission order), as one run of <= 44 bits (lo, hi).
// Entries are left-aligned (warp_build_codes<true>): __funnelshift_l(e, x, e) = x << n | code, so a
// pair costs two funnel shifts and needs no field extraction.  len holds the run's bit length in its
// low 21 bits; the bits above are garbage from the code values (every consumer masks or uses only
// the low 5 bits through a wrapping shift).
__device__ __forceinline__ void wb_run(const unsigned char* code, uint32_t w, uint32_t& lo, uint32_t& hi, uint32_t& len) {
  const uint32_t e3 = *reinterpret_cast<const uint32_t*>(code + ((w >> 22) & 0x3FCu));
  const uint32_t e2 = *reinterpret_cast<const uint32_t*>(code + ((w >> 14) & 0x3FCu));
  const uint32_t e1 = *reinterpret_cast<const uint32_t*>(code + ((w >> 6) & 0x3FCu));
  const uint32_t e0 = *reinterpret_cast<const uint32_t*>(code + ((w << 2) & 0x3FCu));
  const uint32_t pa = __funnelshift_l(e3, __funnelshift_l(e2, 0u, e2), e3);  // code3 | code2 << n3
  const uint32_t pb = __funnelshift_l(e1, __funnelshift_l(e0, 0u, e0), e1);  // code1 | code0 << n1
  const uint32_t la = e3 + e2;                                               // n3 + n2 (2..22) in the low bits
  lo = pa | __funnelshift_l(0u, pb, la);
  hi = __funnelshift_l(pb, 0u, la);
  len = la + e1 + e0;
}

// OR a run of <= 44 bits into the bit buffer at bit offset off (garbage above bit 20 allowed): three
// unconditional reductions, the words that receive no bits get an OR of zero.
__device__ __forceinline__ void wb_place(uint32_t bitbuf_s, uint32_t off, uint32_t lo, uint32_t hi) {
  const uint32_t sa = bitbuf_s + ((off >> 3) & 0xFFFCu);
  const uint32_t w0 = __funnelshift_l(0u, lo, off);  // lo << s
  const uint32_t w1 = __funnelshift_l(lo, hi, off);  // hi << s | lo >> (32 - s); hi when s = 0
  const uint32_t w2 = __funnelshift_l(hi, 0u, off);  // hi >> (32 - s); 0 when s = 0
  asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(sa), "r"(w0) : "memory");
  asm volatile("red.shared.or.b32 [%0+4], %1;" ::"r"(sa), "r"(w1) : "memory");
  asm volatile("red.shared.or.b32 [%0+8], %1;" ::"r"(sa), "r"(w2) : "memory");
}

// (lo, hi) = 4 bytes each of the two top byte planes of 4 elements; the element-level rotation
// [sign][exp8][mant] -> [exp8][sign][mant] (data_manipulation_dtype16.c:10-20, dtype32.c:39-49) becomes
// hi' = exp8 = hi << 1 | lo >> 7, lo' = sign | low 7 bits, per byte.
__device__ __forceinline__ void rotate_planes(uint32_t& lo, uint32_t& hi) {
  const uint32_t l = lo, h = hi;
  hi = ((h << 1) & 0xFEFEFEFEu) | ((l >> 7) & 0x01010101u);
  lo = (h & 0x80808080u) | (l & 0x7F7F7F7Fu);
}

struct WbItem {
  uint8_t* dest;
  uint32_t size;
  uint32_t hsize;
  uint32_t sbytes[4];
  uint32_t lg;
  uint32_t type;  // 0 raw, 1 coded (size 1 = RLE)
};

template <int G>
struct WbSmem {
  uint32_t code[G][256];                       // val << (32 - nb) | nb (warp_build_codes<true>)
  WbItem item[G];
  __align__(16) uint8_t nb[G][256];
  uint32_t bitbuf[kWbWarps][G][WbCfg<G>::kBitWords];
  __align__(16) uint8_t stage[kWbWarps][WbCfg<G>::kTile + 32];
};
static_assert(WbCfg<2>::kBitWords * 4 <= 0xFFFCu, "wb_place masks the word offset to 16 bits");
// Pass B relies on codes of at most 11 bits: the left-aligned entries keep bits 5..20 clear (so sums of
// entries carry exact lengths in bits 0..20) and kBitWords is sized for 11 bits per symbol.  Pass A's table
// log is fse_pick_log(kHufLogDefault, ...), which is at most max(kHufLogDefault, 9) for byte symbols (the
// minimum log for 256 symbols is 9), and the code lengths are limited to it.  kHufLogMax (12) is only what
// the format allows a decoder to meet.
static_assert(kHufLogDefault <= 11, "k_encode_write_warp's entry format and bit buffer assume codes of <= 11 bits");

// Per-stream bit writer state kept in registers by every lane of the warp (uniform values).
struct WbStream {
  uint8_t* gaddr;    // first byte of the bitstream in the output
  uint32_t a;        // gaddr & 3
  uint32_t B;        // bits placed so far, counted from the aligned word below gaddr
  uint32_t flushed;  // whole words already written
};

__device__ __forceinline__ void wb_flush(uint32_t* bitbuf, WbStream& st, int lane) {
  uint32_t* gword = reinterpret_cast<uint32_t*>(st.gaddr - st.a);
  const uint32_t complete = (st.B >> 5) - st.flushed;
  // a stream that starts in the middle of a word: bytes [a, 4) of its first word go out one by one
  const bool split_first = (st.flushed == 0 && st.a != 0);
  if (split_first && lane == 0 && complete > 0) {
    const uint32_t val = bitbuf[0];
    for (uint32_t bb = st.a; bb < 4; bb++) st.gaddr[bb - st.a] = (uint8_t)(val >> (8 * bb));
  }
  for (uint32_t w = lane; w < complete; w += 32) {
    const uint32_t val = bitbuf[w];
    bitbuf[w] = 0;  // cleared as it leaves; only lane 0 touches word 0 and word `complete` below
    if (!(split_first && w == 0)) gword[st.flushed + w] = val;
  }
  if (lane == 0 && complete > 0) {  // the partial word becomes word 0 of the next tile (after lane 0 cleared word 0 above)
    bitbuf[0] = bitbuf[complete];
    bitbuf[complete] = 0;
  }
  st.flushed += complete;
  __syncwarp();
}

template <int G>
__global__ void __launch_bounds__(kWbWarps * 32, WbCfg<G>::kMinBlocks) k_encode_write_warp(const uint8_t* __restrict__ in, uint64_t n, uint32_t chunk,
                                                                     uint64_t K, int bits_mode, const uint8_t* __restrict__ types,
                                                                     const uint32_t* __restrict__ sizes,
                                                                     const EncSave* __restrict__ saves,
                                                                     const uint64_t* __restrict__ item_off, uint8_t* out) {
  __shared__ WbSmem<G> S;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (uint64_t c = blockIdx.x; c < K; c += gridDim.x) {
    const uint32_t chunk_len = (c == K - 1) ? (uint32_t)(n - c * (uint64_t)chunk) : chunk;
    if (chunk_len % (64u * G) != 0) continue;  // ragged tail: k_encode_write
    const uint8_t* in_c = in + c * (uint64_t)chunk;
    const uint32_t plen = chunk_len / G;
    const uint32_t seg = plen >> 2;
    const bool rot = (bits_mode == 1 && G > 1);
    __syncthreads();
    // ---- per-chunk setup: warp g prepares group g ----
    if (warp < G) {
      const int g = warp;
      const uint64_t item = (uint64_t)g * K + c;
      WbItem it;
      it.dest = out + item_off[item];
      it.type = types[item];
      it.size = sizes[item];
      it.hsize = 0;
      it.lg = 0;
      it.sbytes[0] = it.sbytes[1] = it.sbytes[2] = it.sbytes[3] = 0;
      if (it.type == 1 && it.size == 1) {
        if (lane == 0) it.dest[0] = saves[item].hdr[0];
      } else if (it.type == 1) {
        const EncSave* sv = saves + item;
        it.hsize = sv->hsize;
        it.lg = sv->lg;
#pragma unroll
        for (int q = 0; q < 4; q++) it.sbytes[q] = sv->sbytes[q];
        reinterpret_cast<uint2*>(S.nb[g])[lane] = reinterpret_cast<const uint2*>(sv->nb)[lane];
        __syncwarp();
        warp_build_codes<true>(S.nb[g], (int)it.lg, S.code[g]);
        for (uint32_t i = lane; i < it.hsize; i += 32) it.dest[i] = sv->hdr[i];
        if (lane < 3) {
          it.dest[it.hsize + 2 * lane] = (uint8_t)it.sbytes[lane];
          it.dest[it.hsize + 2 * lane + 1] = (uint8_t)(it.sbytes[lane] >> 8);
        }
      }
      if (lane == 0) S.item[g] = it;
    }
    __syncthreads();

    // ---- warp `warp` = stream index ----
    using Cfg = WbCfg<G>;
    constexpr int H = Cfg::H;
    constexpr uint32_t kTile = Cfg::kTile;
    const int s = warp;
    WbStream st[G];
    uint32_t raw_shift[G];  // destination misalignment of the raw plane quarter (bytes, mod 16)
    uint32_t kind[G];       // what the tile loop does with plane g: 0 raw, 1 coded, 2 nothing (RLE)
#pragma unroll
    for (int g = 0; g < G; g++) {
      const WbItem& it = S.item[g];
      st[g].gaddr = it.dest;
      st[g].a = st[g].B = st[g].flushed = 0;
      raw_shift[g] = 0;
      kind[g] = it.type == 0 ? 0u : (it.size > 1 ? 1u : 2u);
      if (kind[g] == 1) {
        uint32_t at = it.hsize + 6;
        for (int q = 0; q < s; q++) at += it.sbytes[q];
        st[g].gaddr = it.dest + at;
        st[g].a = (uint32_t)((uintptr_t)st[g].gaddr & 3);
        st[g].B = 8 * st[g].a;
        for (uint32_t w = lane; w < Cfg::kBitWords; w += 32) S.bitbuf[warp][g][w] = 0;
      } else if (kind[g] == 0) {
        st[g].gaddr = it.dest + (uint64_t)s * seg;
        raw_shift[g] = (uint32_t)((uintptr_t)st[g].gaddr & 15);
      }
    }
    __syncwarp();

    // Lane `lane` holds plane bytes [512 h + 16 lane, +16) of the tile, h < H.
    const uint8_t* src_s = in_c + (uint64_t)s * seg * G;
    const uint32_t ntiles = (seg + kTile - 1) / kTile;
    uint4 cur[H][G], nxt[H][G];
    {
      const uint32_t t0 = (ntiles - 1) * kTile;
#pragma unroll
      for (int h = 0; h < H; h++) {
        if (t0 + 512u * h + 16 * lane < seg) {
          const uint4* p = reinterpret_cast<const uint4*>(src_s + (uint64_t)(t0 + 512u * h + 16 * lane) * G);
#pragma unroll
          for (int i = 0; i < G; i++) nxt[h][i] = __ldg(p + i);
        }
      }
    }
    // Tiles run from the end of the stream to its start (huff0 emits the last symbol first); only the
    // first one processed can be partial, so the others are compiled with `have` known to be true.
    auto do_tile = [&](auto full_tag, const uint32_t ti) {
      constexpr bool kFull = decltype(full_tag)::value;
      const uint32_t t0 = ti * kTile;
      const uint32_t cnt = kFull ? kTile : min(kTile, seg - t0);  // multiple of 16
      bool have[H];
#pragma unroll
      for (int h = 0; h < H; h++) have[h] = kFull ? true : (512u * h + 16u * lane < cnt);
#pragma unroll
      for (int h = 0; h < H; h++)
#pragma unroll
        for (int i = 0; i < G; i++) cur[h][i] = nxt[h][i];
      if (ti > 0) {  // prefetch the next (lower) tile, always full
#pragma unroll
        for (int h = 0; h < H; h++) {
          const uint4* p = reinterpret_cast<const uint4*>(src_s + (uint64_t)(t0 - kTile + 512u * h + 16 * lane) * G);
#pragma unroll
          for (int i = 0; i < G; i++) nxt[h][i] = __ldg(p + i);
        }
      }
      uint4 pv[H][G];
#pragma unroll
      for (int h = 0; h < H; h++) {
        if (have[h]) {
          uint32_t w[4 * G];
#pragma unroll
          for (int i = 0; i < G; i++) {
            w[4 * i] = cur[h][i].x; w[4 * i + 1] = cur[h][i].y; w[4 * i + 2] = cur[h][i].z; w[4 * i + 3] = cur[h][i].w;
          }
          split16<G>(w, pv[h]);
          if (rot) {  // sign-bit rotation at plane level: 4 operations per 4 elements instead of 5 per word
            rotate_planes(pv[h][(G - 2) % G].x, pv[h][G - 1].x);
            rotate_planes(pv[h][(G - 2) % G].y, pv[h][G - 1].y);
            rotate_planes(pv[h][(G - 2) % G].z, pv[h][G - 1].z);
            rotate_planes(pv[h][(G - 2) % G].w, pv[h][G - 1].w);
          }
        }
      }
#pragma unroll
      for (int g = 0; g < G; g++) {
        if (kind[g] == 0) {
          // ---- raw plane: 16 bytes per lane and half -> dest + t0 .. ----
          uint8_t* D = st[g].gaddr + t0;
          const uint32_t m = raw_shift[g];
          if (m == 0) {
#pragma unroll
            for (int h = 0; h < H; h++)
              if (have[h]) *reinterpret_cast<uint4*>(D + 512u * h + 16 * lane) = pv[h][g];
          } else {
            uint8_t* stg = S.stage[warp];
#pragma unroll
            for (int h = 0; h < H; h++)
              if (have[h]) *reinterpret_cast<uint4*>(stg + 512u * h + 16 * lane) = pv[h][g];
            __syncwarp();
            const uint32_t head = 16 - m;  // bytes before the first aligned destination block
            const uint32_t nblk = (cnt - head) >> 4;
            const uint32_t bs = (head & 3) * 8;
#pragma unroll
            for (int h = 0; h < H; h++) {
              // every lane computes (the stage has 32 spare bytes behind the tile); only the store is conditional
              const uint32_t blk = 32u * h + (uint32_t)lane;
              const uint4 a4 = *reinterpret_cast<const uint4*>(stg + 16 * blk);
              const uint4 b4 = *reinterpret_cast<const uint4*>(stg + 16 * blk + 16);
              const uint32_t wv[8] = {a4.x, a4.y, a4.z, a4.w, b4.x, b4.y, b4.z, b4.w};
              // 16 bytes starting `head` bytes into (a4, b4): the word part of the shift is uniform over
              // the warp, so it is a 4-way switch (4 funnel shifts) rather than 7 shifts + 9 selects
              uint32_t o[4];
              switch (head >> 2) {
                case 0:
#pragma unroll
                  for (int i = 0; i < 4; i++) o[i] = __funnelshift_r(wv[i], wv[i + 1], bs);
                  break;
                case 1:
#pragma unroll
                  for (int i = 0; i < 4; i++) o[i] = __funnelshift_r(wv[i + 1], wv[i + 2], bs);
                  break;
                case 2:
#pragma unroll
                  for (int i = 0; i < 4; i++) o[i] = __funnelshift_r(wv[i + 2], wv[i + 3], bs);
                  break;
                default:
#pragma unroll
                  for (int i = 0; i < 4; i++) o[i] = __funnelshift_r(wv[i + 3], wv[i + 4], bs);
                  break;
              }
              if (blk < nblk) *reinterpret_cast<uint4*>(D + head + 16 * blk) = make_uint4(o[0], o[1], o[2], o[3]);
            }
            if (kFull) {  // the 16 bytes around the aligned blocks: head bytes in front, 16 - head behind
              if (lane < 16) {
                const uint32_t idx = (uint32_t)lane < head ? (uint32_t)lane : (kTile - 16u + (uint32_t)lane);
                D[idx] = stg[idx];
              }
            } else {
              if ((uint32_t)lane < head) D[lane] = stg[lane];
              const uint32_t done = head + 16 * nblk;
              if ((uint32_t)lane < cnt - done) D[done + lane] = stg[done + lane];
            }
            __syncwarp();
          }
        } else if (kind[g] == 1) {
          // ---- coded plane: this lane's 16 symbols of each half, last byte first ----
          // Run r of half h = symbols 4r..4r+3 = bytes 3,2,1,0 of word 3-r (wb_run).  Half H-1 is
          // emitted before half H-2, so ONE suffix scan over the lanes of the halves' lengths packed in
          // 16-bit fields (<= 512 * 11 bits per half) places all of them.
          const unsigned char* code = reinterpret_cast<const unsigned char*>(S.code[g]);
          uint32_t lo[H][4], hi[H][4], len[H][4], mine[H];
#pragma unroll
          for (int h = 0; h < H; h++) {
            if (have[h]) {
              const uint32_t wv[4] = {pv[h][g].x, pv[h][g].y, pv[h][g].z, pv[h][g].w};
#pragma unroll
              for (int r = 0; r < 4; r++) wb_run(code, wv[3 - r], lo[h][r], hi[h][r], len[h][r]);
              mine[h] = (len[h][0] + len[h][1] + len[h][2] + len[h][3]) & 0x1FFFFFu;
            } else {  // an idle lane of the partial tile ORs zeros at a valid offset
#pragma unroll
              for (int r = 0; r < 4; r++) lo[h][r] = hi[h][r] = len[h][r] = 0;
              mine[h] = 0;
            }
          }
          const uint32_t packed = (H == 2) ? (mine[H - 1] | (mine[0] << 16)) : mine[0];
          uint32_t x = packed;  // suffix sum over lanes: lane 31 is emitted first
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_down_sync(0xffffffffu, x, o);
            if (lane + o < 32) x += y;
          }
          const uint32_t tot = __shfl_sync(0xffffffffu, x, 0);
          const uint32_t ex = x - packed;  // the fields never borrow: each is >= this lane's part
          uint32_t* bitbuf = S.bitbuf[warp][g];
          const uint32_t bitbuf_s = (uint32_t)__cvta_generic_to_shared(bitbuf);
          const uint32_t base = st[g].B - 32 * st[g].flushed;
          uint32_t off[H], tile_bits;
          if constexpr (H == 2) {
            off[H - 1] = base + (ex & 0xFFFFu);
            off[0] = base + (tot & 0xFFFFu) + (ex >> 16);
            tile_bits = (tot & 0xFFFFu) + (tot >> 16);
          } else {
            off[0] = base + ex;
            tile_bits = tot;
          }
#pragma unroll
          for (int h = 0; h < H; h++) {
            uint32_t o = off[h];
#pragma unroll
            for (int r = 0; r < 4; r++) {
              wb_place(bitbuf_s, o, lo[h][r], hi[h][r]);
              o += len[h][r];
            }
          }
          __syncwarp();
          st[g].B += tile_bits;
          wb_flush(bitbuf, st[g], lane);
        }
      }
    };
    do_tile(std::false_type{}, ntiles - 1);
    for (uint32_t ti = ntiles - 1; ti-- > 0;) do_tile(std::true_type{}, ti);
    // ---- end marks and the last partial bytes of every bitstream ----
#pragma unroll
    for (int g = 0; g < G; g++) {
      if (kind[g] == 1) {
        uint32_t* bitbuf = S.bitbuf[warp][g];
        if (lane == 0) bitbuf[(st[g].B - 32 * st[g].flushed) >> 5] |= 1u << (st[g].B & 31);
        __syncwarp();
        const uint32_t first_byte = max(4 * st[g].flushed, st[g].a);
        const uint32_t end_byte = st[g].a + S.item[g].sbytes[s];
        for (uint32_t bb = first_byte + lane; bb < end_byte; bb += 32) {
          const uint32_t rel = bb - 4 * st[g].flushed;
          st[g].gaddr[bb - st[g].a] = (uint8_t)(bitbuf[rel >> 2] >> (8 * (rel & 3)));
        }
        __syncwarp();
      }
    }
  }
}

}  // namespace zb
