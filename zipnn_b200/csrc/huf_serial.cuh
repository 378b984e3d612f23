// huf_serial.cuh -- the small serial pieces of the huff0 block format, written so
// that one GPU thread (or a host unit test) can run them:
//   * encoder: code lengths from a histogram (length-limited to 11 bits exactly as the
//     reference does), canonical code values, and the table description header
//     (weights compressed with a 2-state tANS coder, or raw nibbles);
//   * decoder: table description header -> weights.
// Everything here is O(alphabet) work per 64-128 KiB byte plane; the O(bytes) work
// (histogram, bit-pack, bit-unpack, byte-group split/regroup) lives in the kernels.
//
// Format references (reference checkout, for parity review):
//   include/FiniteStateEntropy/lib/huf_compress.c:63-147, 215-410
//   include/FiniteStateEntropy/lib/fse_compress.c:66-169, 192-285, 316-494, 554-611
//   include/FiniteStateEntropy/lib/entropy_common.c:41-215
//   include/FiniteStateEntropy/lib/fse_decompress.c:71-133, 178-238
#pragma once
#include <stdint.h>
#include <stddef.h>

#if defined(__CUDACC__)
#define ZB_HD __host__ __device__
#else
#define ZB_HD
#endif

namespace zb {

constexpr int kHufLogMax = 12;      // largest table log the format allows
constexpr int kHufLogDefault = 11;  // what HUF_compress() asks for
constexpr int kHufBlockMax = 128 * 1024;

ZB_HD inline int hb32(uint32_t v) {
#if defined(__CUDA_ARCH__)
  return 31 - __clz((int)v);
#else
  return 31 - __builtin_clz(v);
#endif
}

// ---------------------------------------------------------------------------------
// LSB-first bit sink over a byte buffer (tiny outputs only: table headers).
// ---------------------------------------------------------------------------------
struct BitSink {
  uint8_t* p;
  uint8_t* begin;
  uint64_t acc;
  int fill;
  ZB_HD void init(uint8_t* dst) {
    p = begin = dst;
    acc = 0;
    fill = 0;
  }
  ZB_HD void put(uint32_t v, int nbits) {  // nbits <= 32, fill < 8 on entry
    acc |= (uint64_t)v << fill;
    fill += nbits;
    while (fill >= 8) {
      *p++ = (uint8_t)acc;
      acc >>= 8;
      fill -= 8;
    }
  }
  ZB_HD uint32_t finish() {  // end mark, then pad the last byte
    put(1, 1);
    if (fill > 0) *p++ = (uint8_t)acc;
    return (uint32_t)(p - begin);
  }
};

// ---------------------------------------------------------------------------------
// tANS for the weight table: table log <= 6, alphabet <= 13 on the encode side.
// ---------------------------------------------------------------------------------
ZB_HD inline int fse_min_log(uint32_t n, uint32_t max_sym) {
  int a = hb32(n) + 1, b = hb32(max_sym) + 2;
  return a < b ? a : b;
}

ZB_HD inline int fse_pick_log(int want, uint32_t n, uint32_t max_sym, int minus) {
  int by_src = hb32(n - 1) - minus;
  int lg = want;
  int need = fse_min_log(n, max_sym);
  if (by_src < lg) lg = by_src;
  if (need > lg) lg = need;
  if (lg < 5) lg = 5;
  if (lg > 12) lg = 12;
  return lg;
}

struct FseEnc {
  uint32_t count[16];
  int16_t norm[16];
  uint32_t cumul[18];
  uint8_t spread[64];
  uint16_t next_state[64];
  int32_t delta_find[16];
  uint32_t delta_bits[16];
};

// Fallback normalisation, used when rounding gave away too many slots.
ZB_HD inline int fse_normalize_slow(int16_t* norm, int lg, const uint32_t* count, uint32_t total, int max_sym) {
  const int16_t kPending = -2;
  uint32_t given = 0;
  const uint32_t low_thr = total >> lg;
  uint32_t low_one = (uint32_t)(((uint64_t)total * 3) >> (lg + 1));
  for (int s = 0; s <= max_sym; s++) {
    uint32_t c = count[s];
    if (c == 0) {
      norm[s] = 0;
    } else if (c <= low_thr) {
      norm[s] = -1;
      given++;
      total -= c;
    } else if (c <= low_one) {
      norm[s] = 1;
      given++;
      total -= c;
    } else {
      norm[s] = kPending;
    }
  }
  uint32_t todo = (1u << lg) - given;
  if (todo == 0) return 0;
  if (total / todo > low_one) {
    low_one = (uint32_t)(((uint64_t)total * 3) / ((uint64_t)todo * 2));
    for (int s = 0; s <= max_sym; s++)
      if (norm[s] == kPending && count[s] <= low_one) {
        norm[s] = 1;
        given++;
        total -= count[s];
      }
    todo = (1u << lg) - given;
  }
  if (given == (uint32_t)max_sym + 1) {
    int best = 0;
    uint32_t best_c = 0;
    for (int s = 0; s <= max_sym; s++)
      if (count[s] > best_c) {
        best = s;
        best_c = count[s];
      }
    norm[best] = (int16_t)(norm[best] + (int16_t)todo);
    return 0;
  }
  if (total == 0) {
    for (int s = 0; todo > 0; s = (s + 1) % (max_sym + 1))
      if (norm[s] > 0) {
        todo--;
        norm[s]++;
      }
    return 0;
  }
  const int vlog = 62 - lg;
  const uint64_t mid = (1ull << (vlog - 1)) - 1;
  const uint64_t rstep = (((1ull << vlog) * todo) + mid) / total;
  uint64_t acc = mid;
  for (int s = 0; s <= max_sym; s++)
    if (norm[s] == kPending) {
      uint64_t end = acc + (uint64_t)count[s] * rstep;
      uint32_t w = (uint32_t)(end >> vlog) - (uint32_t)(acc >> vlog);
      if (w < 1) return -1;
      norm[s] = (int16_t)w;
      acc = end;
    }
  return 0;
}

ZB_HD inline int fse_normalize(int16_t* norm, int lg, const uint32_t* count, uint32_t total, int max_sym) {
  const uint32_t kRestToBeat[8] = {0, 473195, 504333, 520860, 550000, 700000, 750000, 830000};
  if (lg < 5 || lg > 12) return -1;
  if (lg < fse_min_log(total, (uint32_t)max_sym)) return -1;
  const int scale = 62 - lg;
  const uint64_t step = (1ull << 62) / total;
  const uint64_t vstep = 1ull << (scale - 20);
  int left = 1 << lg;
  int largest = 0;
  int16_t largest_p = 0;
  const uint32_t low_thr = total >> lg;
  for (int s = 0; s <= max_sym; s++) {
    uint32_t c = count[s];
    if (c == total) return 0;
    if (c == 0) {
      norm[s] = 0;
      continue;
    }
    if (c <= low_thr) {
      norm[s] = -1;
      left--;
    } else {
      int16_t p = (int16_t)(((uint64_t)c * step) >> scale);
      if (p < 8) {
        uint64_t beat = vstep * kRestToBeat[p];
        if (((uint64_t)c * step) - ((uint64_t)p << scale) > beat) p++;
      }
      if (p > largest_p) {
        largest_p = p;
        largest = s;
      }
      norm[s] = p;
      left -= p;
    }
  }
  if (-left >= (norm[largest] >> 1)) return fse_normalize_slow(norm, lg, count, total, max_sym);
  norm[largest] = (int16_t)(norm[largest] + left);
  return 0;
}

// Normalised-count header.  Returns bytes written or -1.
ZB_HD inline int fse_write_ncount(uint8_t* out, const int16_t* norm, int max_sym, int lg) {
  uint8_t* p = out;
  int remaining = (1 << lg) + 1;
  int threshold = 1 << lg;
  int nbits = lg + 1;
  uint32_t acc = (uint32_t)(lg - 5);
  int cnt = 4;
  int sym = 0;
  const int alphabet = max_sym + 1;
  bool prev0 = false;
  while (sym < alphabet && remaining > 1) {
    if (prev0) {
      int start = sym;
      while (sym < alphabet && norm[sym] == 0) sym++;
      if (sym == alphabet) break;
      while (sym >= start + 24) {
        start += 24;
        acc += 0xFFFFu << cnt;
        p[0] = (uint8_t)acc;
        p[1] = (uint8_t)(acc >> 8);
        p += 2;
        acc >>= 16;
      }
      while (sym >= start + 3) {
        start += 3;
        acc += 3u << cnt;
        cnt += 2;
      }
      acc += (uint32_t)(sym - start) << cnt;
      cnt += 2;
      if (cnt > 16) {
        p[0] = (uint8_t)acc;
        p[1] = (uint8_t)(acc >> 8);
        p += 2;
        acc >>= 16;
        cnt -= 16;
      }
    }
    int c = norm[sym++];
    const int max = (2 * threshold - 1) - remaining;
    remaining -= c < 0 ? -c : c;
    c++;
    if (c >= threshold) c += max;
    acc += (uint32_t)c << cnt;
    cnt += nbits;
    cnt -= (c < max) ? 1 : 0;
    prev0 = (c == 1);
    if (remaining < 1) return -1;
    while (remaining < threshold) {
      nbits--;
      threshold >>= 1;
    }
    if (cnt > 16) {
      p[0] = (uint8_t)acc;
      p[1] = (uint8_t)(acc >> 8);
      p += 2;
      acc >>= 16;
      cnt -= 16;
    }
  }
  if (remaining != 1) return -1;
  p[0] = (uint8_t)acc;
  p[1] = (uint8_t)(acc >> 8);
  p += (cnt + 7) / 8;
  return (int)(p - out);
}

ZB_HD inline void fse_build_enc(FseEnc& E, int max_sym, int lg) {
  const uint32_t size = 1u << lg, mask = size - 1;
  const uint32_t step = (size >> 1) + (size >> 3) + 3;
  uint32_t high = size - 1;
  E.cumul[0] = 0;
  for (int u = 1; u <= max_sym + 1; u++) {
    if (E.norm[u - 1] == -1) {
      E.cumul[u] = E.cumul[u - 1] + 1;
      E.spread[high--] = (uint8_t)(u - 1);
    } else {
      E.cumul[u] = E.cumul[u - 1] + (uint32_t)E.norm[u - 1];
    }
  }
  uint32_t pos = 0;
  for (int s = 0; s <= max_sym; s++)
    for (int i = 0; i < E.norm[s]; i++) {
      E.spread[pos] = (uint8_t)s;
      pos = (pos + step) & mask;
      while (pos > high) pos = (pos + step) & mask;
    }
  for (uint32_t u = 0; u < size; u++) {
    int s = E.spread[u];
    E.next_state[E.cumul[s]++] = (uint16_t)(size + u);
  }
  uint32_t total = 0;
  for (int s = 0; s <= max_sym; s++) {
    int n = E.norm[s];
    if (n == 0) {
      E.delta_bits[s] = ((uint32_t)(lg + 1) << 16) - size;
      E.delta_find[s] = 0;
    } else if (n == -1 || n == 1) {
      E.delta_bits[s] = ((uint32_t)lg << 16) - size;
      E.delta_find[s] = (int32_t)total - 1;
      total++;
    } else {
      uint32_t max_out = (uint32_t)lg - (uint32_t)hb32((uint32_t)(n - 1));
      uint32_t min_plus = (uint32_t)n << max_out;
      E.delta_bits[s] = (max_out << 16) - min_plus;
      E.delta_find[s] = (int32_t)total - n;
      total += (uint32_t)n;
    }
  }
}

ZB_HD inline uint32_t fse_seed_state(const FseEnc& E, int sym) {
  uint32_t nb = (E.delta_bits[sym] + (1u << 15)) >> 16;
  uint32_t v = (nb << 16) - E.delta_bits[sym];
  return E.next_state[(int32_t)(v >> nb) + E.delta_find[sym]];
}

ZB_HD inline uint32_t fse_step(BitSink& w, const FseEnc& E, uint32_t state, int sym) {
  uint32_t nb = (state + E.delta_bits[sym]) >> 16;
  w.put(state & ((1u << nb) - 1u), (int)nb);
  return E.next_state[(int32_t)(state >> nb) + E.delta_find[sym]];
}

// Weights -> tANS bytes.  0 = "do not use" (too few / all distinct), 1 = all equal, -1 = error.
ZB_HD inline int huf_pack_weights(uint8_t* dst, const uint8_t* w, int n, FseEnc& E) {
  if (n <= 1) return 0;
  for (int i = 0; i < 16; i++) E.count[i] = 0;
  int max_w = 0;
  for (int i = 0; i < n; i++) {
    E.count[w[i]]++;
    if (w[i] > max_w) max_w = w[i];
  }
  uint32_t top = 0;
  for (int s = 0; s <= max_w; s++)
    if (E.count[s] > top) top = E.count[s];
  if (top == (uint32_t)n) return 1;
  if (top == 1) return 0;
  const int lg = fse_pick_log(6, (uint32_t)n, (uint32_t)max_w, 2);
  if (fse_normalize(E.norm, lg, E.count, (uint32_t)n, max_w) != 0) return -1;
  int h = fse_write_ncount(dst, E.norm, max_w, lg);
  if (h < 0) return -1;
  fse_build_enc(E, max_w, lg);
  if (n <= 2) return 0;
  BitSink bw;
  bw.init(dst + h);
  int ip = n;
  uint32_t s1, s2;
  if (n & 1) {
    s1 = fse_seed_state(E, w[--ip]);
    s2 = fse_seed_state(E, w[--ip]);
    s1 = fse_step(bw, E, s1, w[--ip]);
  } else {
    s2 = fse_seed_state(E, w[--ip]);
    s1 = fse_seed_state(E, w[--ip]);
  }
  while (ip > 0) {
    s2 = fse_step(bw, E, s2, w[--ip]);
    s1 = fse_step(bw, E, s1, w[--ip]);
  }
  bw.put(s2 & ((1u << lg) - 1u), lg);
  bw.put(s1 & ((1u << lg) - 1u), lg);
  return h + (int)bw.finish();
}

// ---------------------------------------------------------------------------------
// Code lengths.
// ---------------------------------------------------------------------------------
struct TreeScratch {
  uint32_t cnt[512];    // [0,256): leaves in sorted order; [256,512): internal nodes
  uint16_t parent[512];
  uint8_t depth[512];
  uint8_t sym[256];     // symbol of sorted leaf i
  uint8_t weight[256];
  uint8_t hdr[256];     // table description scratch (tANS output can exceed the 128 kept)
  FseEnc fse;
};

// Cap depths at max_nb and repay the Kraft debt the way the reference does, so the
// resulting lengths (not merely the cost) are identical.
ZB_HD inline int huf_limit_depth(TreeScratch& T, int last, int max_nb) {
  const int deepest = T.depth[last];
  if (deepest <= max_nb) return deepest;
  const uint32_t kNone = 0xF0F0F0F0u;
  int debt = 0;
  const int base = 1 << (deepest - max_nb);
  int n = last;
  while (T.depth[n] > max_nb) {
    debt += base - (1 << (deepest - T.depth[n]));
    T.depth[n] = (uint8_t)max_nb;
    n--;
  }
  while (T.depth[n] == max_nb) n--;
  debt >>= (deepest - max_nb);

  uint32_t rank_last[16];
  for (int i = 0; i < 16; i++) rank_last[i] = kNone;
  {
    int cur = max_nb;
    for (int pos = n; pos >= 0; pos--) {
      if (T.depth[pos] >= cur) continue;
      cur = T.depth[pos];
      rank_last[max_nb - cur] = (uint32_t)pos;
    }
  }
  while (debt > 0) {
    int dec = hb32((uint32_t)debt) + 1;
    for (; dec > 1; dec--) {
      uint32_t hi = rank_last[dec], lo = rank_last[dec - 1];
      if (hi == kNone) continue;
      if (lo == kNone) break;
      if (T.cnt[hi] <= 2 * T.cnt[lo]) break;
    }
    while (dec <= kHufLogMax && rank_last[dec] == kNone) dec++;
    debt -= 1 << (dec - 1);
    if (rank_last[dec - 1] == kNone) rank_last[dec - 1] = rank_last[dec];
    T.depth[rank_last[dec]]++;
    if (rank_last[dec] == 0) {
      rank_last[dec] = kNone;
    } else {
      rank_last[dec]--;
      if (T.depth[rank_last[dec]] != max_nb - dec) rank_last[dec] = kNone;
    }
  }
  while (debt < 0) {
    if (rank_last[1] == kNone) {
      while (T.depth[n] == max_nb) n--;
      T.depth[n + 1]--;
      rank_last[1] = (uint32_t)(n + 1);
      debt++;
      continue;
    }
    T.depth[rank_last[1] + 1]--;
    rank_last[1]++;
    debt++;
  }
  return max_nb;
}

// Input: T.cnt[0..last], T.sym[0..last] = the symbols with non-zero count ordered by
// (count descending, symbol ascending); last >= 1.  Output: T.depth[0..last], the code length
// of sorted leaf n.  Returns the table log (largest code length).
ZB_HD inline int huf_tree_depths(TreeScratch& T, int last, int max_nb) {
  const int kFirst = 256;
  const uint32_t kWall = 0x80000000u;
  int low_leaf = last, low_int = kFirst, next = kFirst;
  const int root = kFirst + last - 1;
  T.cnt[next] = T.cnt[low_leaf] + T.cnt[low_leaf - 1];
  T.parent[low_leaf] = T.parent[low_leaf - 1] = (uint16_t)next;
  next++;
  low_leaf -= 2;
  for (int n = next; n <= root; n++) T.cnt[n] = 1u << 30;
  while (next <= root) {
    uint32_t cl = low_leaf >= 0 ? T.cnt[low_leaf] : kWall;
    int a = (cl < T.cnt[low_int]) ? low_leaf-- : low_int++;
    cl = low_leaf >= 0 ? T.cnt[low_leaf] : kWall;
    int b = (cl < T.cnt[low_int]) ? low_leaf-- : low_int++;
    T.cnt[next] = T.cnt[a] + T.cnt[b];
    T.parent[a] = T.parent[b] = (uint16_t)next;
    next++;
  }
  T.depth[root] = 0;
  for (int n = root - 1; n >= kFirst; n--) T.depth[n] = (uint8_t)(T.depth[T.parent[n]] + 1);
  for (int n = 0; n <= last; n++) T.depth[n] = (uint8_t)(T.depth[T.parent[n]] + 1);
  return huf_limit_depth(T, last, max_nb);
}

// huf_tree_depths, then nb_out[256] by symbol.
ZB_HD inline int huf_lengths_from_sorted(TreeScratch& T, int last, int max_nb, uint8_t* nb_out) {
  const int lg = huf_tree_depths(T, last, max_nb);
  for (int s = 0; s < 256; s++) nb_out[s] = 0;
  for (int n = 0; n <= last; n++) nb_out[T.sym[n]] = T.depth[n];
  return lg;
}

// Serial ordering step (the kernels compute the same ranks in parallel).
ZB_HD inline int huf_sort_serial(TreeScratch& T, const uint32_t* count, int max_sym) {
  int k = 0;
  for (int s = 0; s <= max_sym; s++) {
    uint32_t c = count[s];
    if (c == 0) continue;
    int pos = k++;
    while (pos > 0 && c > T.cnt[pos - 1]) {
      T.cnt[pos] = T.cnt[pos - 1];
      T.sym[pos] = T.sym[pos - 1];
      pos--;
    }
    T.cnt[pos] = c;
    T.sym[pos] = (uint8_t)s;
  }
  return k - 1;  // index of the last non-zero leaf
}

// Canonical values: within a length, symbols in increasing order; lengths laid out
// longest-first from value 0.
ZB_HD inline void huf_assign_values(const uint8_t* nb, int max_sym, int lg, uint16_t* val) {
  uint16_t per_len[kHufLogMax + 2], start[kHufLogMax + 2];
  for (int i = 0; i < kHufLogMax + 2; i++) per_len[i] = start[i] = 0;
  for (int s = 0; s <= max_sym; s++) per_len[nb[s]]++;
  per_len[0] = 0;
  uint16_t v = 0;
  for (int l = lg; l > 0; l--) {
    start[l] = v;
    v = (uint16_t)(v + per_len[l]);
    v >>= 1;
  }
  for (int s = 0; s <= max_sym; s++) val[s] = nb[s] ? start[nb[s]]++ : 0;
}

// Table description.  Writes into T.hdr; returns its size, or -1 when the block must
// be stored raw (alphabet too large for the nibble form and tANS did not pay off).
// The encode kernel writes the same bytes with a whole warp (warp_write_table, encode.cuh).
ZB_HD inline int huf_write_table(TreeScratch& T, const uint8_t* nb, int max_sym, int lg) {
  for (int s = 0; s < max_sym; s++) T.weight[s] = nb[s] ? (uint8_t)(lg + 1 - nb[s]) : 0;
  int h = huf_pack_weights(T.hdr + 1, T.weight, max_sym, T.fse);
  if (h < 0) return -1;
  if (h > 1 && h < max_sym / 2) {
    T.hdr[0] = (uint8_t)h;
    return h + 1;
  }
  if (max_sym > 128) return -1;
  T.hdr[0] = (uint8_t)(128 + (max_sym - 1));
  T.weight[max_sym] = 0;
  for (int s = 0; s < max_sym; s += 2) T.hdr[(s / 2) + 1] = (uint8_t)((T.weight[s] << 4) + T.weight[s + 1]);
  return ((max_sym + 1) / 2) + 1;
}

// ---------------------------------------------------------------------------------
// Decoder: table description -> weights.
// ---------------------------------------------------------------------------------
// NSYM = how many distinct weight values the tANS header may declare.  The format allows 256;
// every header the reference encoder writes declares at most 13 (weights 0..12), so the fused
// decode kernel uses a 16-symbol scratch and hands anything larger to the general kernel.
template <int NSYM>
struct FseDecT {
  int16_t norm[NSYM];
  uint16_t next[NSYM];
  uint16_t new_state[64];
  uint8_t sym[64];
  uint8_t nb[64];
  static constexpr int kSymbols = NSYM;
};
using FseDec = FseDecT<256>;
using FseDecSmall = FseDecT<16>;

// Forward LSB-first peek of n <= 16 bits at bit offset pos; zeros past the end.
ZB_HD inline uint32_t peek_fwd(const uint8_t* src, uint32_t size, uint32_t pos, int n) {
  uint32_t byte = pos >> 3;
  uint32_t v = 0;
  for (int i = 0; i < 4; i++)
    if (byte + i < size) v |= (uint32_t)src[byte + i] << (8 * i);
  return (v >> (pos & 7)) & ((1u << n) - 1u);
}

// Returns bytes consumed, or -1.  *max_sym_io: in = capacity-1, out = last symbol.
ZB_HD inline int fse_read_ncount(int16_t* norm, int* max_sym_io, int* lg_out, const uint8_t* src, uint32_t size) {
  uint8_t pad[4] = {0, 0, 0, 0};
  uint32_t true_size = size;
  if (size < 4) {
    for (uint32_t i = 0; i < size; i++) pad[i] = src[i];
    src = pad;
    size = 4;
  }
  const int max_sym = *max_sym_io;
  for (int i = 0; i <= max_sym; i++) norm[i] = 0;
  uint32_t pos = 0;
  int nbits = (int)peek_fwd(src, size, pos, 4) + 5;
  pos += 4;
  if (nbits > 15) return -1;
  *lg_out = nbits;
  int remaining = (1 << nbits) + 1;
  int threshold = 1 << nbits;
  nbits++;
  int sym = 0;
  bool prev0 = false;
  while (remaining > 1 && sym <= max_sym) {
    if (prev0) {
      int n0 = sym;
      while (peek_fwd(src, size, pos, 16) == 0xFFFFu) {
        n0 += 24;
        pos += 16;
        if (pos > 8 * size + 64) return -1;
      }
      while (peek_fwd(src, size, pos, 2) == 3u) {
        n0 += 3;
        pos += 2;
        if (pos > 8 * size + 64) return -1;
      }
      n0 += (int)peek_fwd(src, size, pos, 2);
      pos += 2;
      if (n0 > max_sym) return -1;
      while (sym < n0) norm[sym++] = 0;
    }
    const int max = (2 * threshold - 1) - remaining;
    int c;
    uint32_t lowv = peek_fwd(src, size, pos, nbits - 1);
    if ((int)lowv < max) {
      c = (int)lowv;
      pos += (uint32_t)(nbits - 1);
    } else {
      c = (int)peek_fwd(src, size, pos, nbits);
      if (c >= threshold) c -= max;
      pos += (uint32_t)nbits;
    }
    c--;
    remaining -= c < 0 ? -c : c;
    norm[sym++] = (int16_t)c;
    prev0 = (c == 0);
    while (remaining < threshold) {
      nbits--;
      threshold >>= 1;
    }
  }
  if (remaining != 1) return -1;
  if (pos > 8 * size) return -1;
  *max_sym_io = sym - 1;
  int used = (int)((pos + 7) >> 3);
  if ((uint32_t)used > true_size) return -1;
  return used;
}

template <class DEC>
ZB_HD inline int fse_build_dec(DEC& D, int max_sym, int lg) {
  const uint32_t size = 1u << lg, mask = size - 1;
  const uint32_t step = (size >> 1) + (size >> 3) + 3;
  uint32_t high = size - 1;
  for (int s = 0; s <= max_sym; s++) {
    if (D.norm[s] == -1) {
      D.sym[high--] = (uint8_t)s;
      D.next[s] = 1;
    } else {
      D.next[s] = (uint16_t)D.norm[s];
    }
  }
  uint32_t pos = 0;
  for (int s = 0; s <= max_sym; s++)
    for (int i = 0; i < D.norm[s]; i++) {
      D.sym[pos] = (uint8_t)s;
      pos = (pos + step) & mask;
      while (pos > high) pos = (pos + step) & mask;
    }
  if (pos != 0) return -1;
  for (uint32_t u = 0; u < size; u++) {
    uint32_t ns = D.next[D.sym[u]]++;
    int nb = lg - hb32(ns);
    D.nb[u] = (uint8_t)nb;
    D.new_state[u] = (uint16_t)((ns << nb) - size);
  }
  return 0;
}

// Backward reader over a tiny buffer: g = bits consumed from the top.
struct BackBits {
  const uint8_t* p;
  uint32_t total;
  uint32_t g;
  ZB_HD int init(const uint8_t* src, uint32_t size) {
    if (size < 1) return -1;
    uint8_t lastb = src[size - 1];
    if (lastb == 0) return -1;
    p = src;
    total = 8 * size;
    g = 8u - (uint32_t)hb32(lastb);
    return 0;
  }
  ZB_HD uint32_t take(int n) {  // n <= 16; zeros below bit 0
    uint32_t v = 0;
    if (n > 0 && g < total) {
      // bits [total-g-n, total-g) of the little-endian integer
      int lo = (int)total - (int)g - n;
      uint32_t acc = 0;
      int lo_c = lo < 0 ? 0 : lo;
      uint32_t byte = (uint32_t)lo_c >> 3;
      for (int i = 0; i < 4; i++)
        if (byte + i < (total >> 3)) acc |= (uint32_t)p[byte + i] << (8 * i);
      acc >>= (lo_c & 7);
      int have = n - (lo_c - lo);
      acc &= (1u << have) - 1u;
      v = acc << (lo_c - lo);
    }
    g += (uint32_t)n;
    return v;
  }
};

// Two interleaved tANS states; the stream ends when an update reads below bit 0.
// Returns the number of symbols written to dst (<= cap), or -1.
template <class DEC>
ZB_HD inline int fse_unpack(uint8_t* dst, int cap, const uint8_t* src, uint32_t size, int max_log, DEC& D) {
  int max_sym = DEC::kSymbols - 1, lg = 0;
  int h = fse_read_ncount(D.norm, &max_sym, &lg, src, size);
  if (h < 0) return -1;
  if (lg > max_log) return -1;
  if (fse_build_dec(D, max_sym, lg) != 0) return -1;
  BackBits r;
  if (r.init(src + h, size - (uint32_t)h) != 0) return -1;
  uint32_t s1 = r.take(lg);
  uint32_t s2 = r.take(lg);
  int n = 0;
  for (;;) {
    if (n + 2 > cap) return -1;
    dst[n++] = D.sym[s1];
    s1 = (uint32_t)D.new_state[s1] + r.take(D.nb[s1]);
    if (r.g > r.total) {
      dst[n++] = D.sym[s2];
      break;
    }
    if (n + 2 > cap) return -1;
    dst[n++] = D.sym[s2];
    s2 = (uint32_t)D.new_state[s2] + r.take(D.nb[s2]);
    if (r.g > r.total) {
      dst[n++] = D.sym[s1];
      break;
    }
  }
  return n;
}

// Table description -> weights[0..nsym).  Returns header size in bytes, or -1.
template <class DEC>
ZB_HD inline int huf_read_weights(uint8_t* weights /*256*/, int* nsym, int* lg_out, const uint8_t* src, uint32_t size,
                                  DEC& D) {
  if (size == 0) return -1;
  uint32_t isize = src[0];
  int osize;
  if (isize >= 128) {
    osize = (int)isize - 127;
    isize = (uint32_t)(osize + 1) / 2;
    if (isize + 1 > size) return -1;
    for (int n = 0; n < osize; n += 2) {
      uint8_t b = src[1 + n / 2];
      weights[n] = b >> 4;
      weights[n + 1] = b & 15;  // n+1 <= 129
    }
  } else {
    if (isize + 1 > size) return -1;
    osize = fse_unpack(weights, 255, src + 1, isize, 6, D);
    if (osize < 0) return -1;
  }
  uint32_t total = 0;
  uint32_t rank1 = 0;
  for (int n = 0; n < osize; n++) {
    uint32_t w = weights[n];
    if (w >= (uint32_t)kHufLogMax) return -1;
    if (w == 1) rank1++;
    total += (1u << w) >> 1;
  }
  if (total == 0) return -1;
  const int lg = hb32(total) + 1;
  if (lg > kHufLogMax) return -1;
  const uint32_t rest = (1u << lg) - total;
  if ((1u << hb32(rest)) != rest) return -1;
  const int lastw = hb32(rest) + 1;
  weights[osize] = (uint8_t)lastw;
  if (lastw == 1) rank1++;
  if (rank1 < 2 || (rank1 & 1)) return -1;
  *nsym = osize + 1;
  *lg_out = lg;
  return (int)isize + 1;
}

}  // namespace zb
