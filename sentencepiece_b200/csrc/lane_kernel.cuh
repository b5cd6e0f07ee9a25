// lane_kernel.cuh -- unigram fast path: one sentence per LANE (32 sentences per warp).
//
// Measured motivation (profiles/r01_v1_*): with one sentence per warp the kernel is
// instruction-issue bound and ~65 % of the issued instructions are the ORDERED fold of
// Viterbi edges, where 31 of 32 lanes repeat the same scalar work.  The reference
// algorithm (src/unigram_model.cc:889-1020) is a short sequential state machine per
// sentence; running it one sentence per lane makes every instruction do 32 sentences'
// worth of work (~4x fewer issued instructions per sentence, profiles/r01_v2_*).
//
// Per lane, per sentence:
//   K1  Normalizer::Normalize / NormalizePrefix, sequentially (src/normalizer.cc:71-253).
//       Input bytes stream through a 32-byte register window (aligned 16-byte loads, next
//       chunk prefetched); the ASCII fast-path tables of the charsmap sit in shared
//       memory; normalized text goes to a per-lane slab in HBM/L2 with words interleaved
//       by lane.
//   K2  EncodeOptimized as a flat state machine: each loop trip is ONE trie transition
//       for every lane (hot trie prefix in shared memory, rest L2).  The text is read
//       through a 16-byte register window anchored at the current start (next word
//       prefetched at each start transition).  best_path_ends_at[] only ever needs the
//       positions [s, s + max_piece_len], so it lives in a per-lane RING in shared memory
//       laid out [slot][lane] (bank == lane: conflict free).  When a position becomes a
//       start its final back-pointer is appended to a per-lane LOG (entry t of every lane
//       shares a cache line), so the back-trace is a coalesced backward scan.
//   K4  back-trace + id path of PopulateSentencePieceText: two backward scans of the log
//       (count, then write) around one warp-aggregated claim of output space.
// Exactly the reference's relaxation order and mixed float/double comparison.
#ifndef SPM_B200_LANE_KERNEL_CUH_
#define SPM_B200_LANE_KERNEL_CUH_

#include "kernels.cuh"
#include "drain.cuh"

namespace spm_b200 {

constexpr uint32_t kLaneUnk = 0x3FFFFFu;  // 22-bit trie-unit field: UNK piece

// slab geometry: per warp [text words: cap/4 + 12][32] u32, then [log: cap + 4][32] u32
constexpr uint32_t kLaneTextSlack = 12;  // window loads may run a few words past the text
__host__ __device__ inline unsigned long long lane_slab_bytes(uint32_t cap) {
  return (static_cast<unsigned long long>(cap / 4 + kLaneTextSlack) + (cap + 4)) * 32ull * 4ull;
}
// shared memory for the normalizer's fast-path tables
constexpr uint32_t kLaneTableBytes = 32 + 4096 + 512 + 16 + 16;  // cm_lead[8] + cm_pair[1024] + cm_solo[128] + plain[4] + plain_or_space[4]

// Fills the normalizer's fast-path tables in shared memory (all threads of the CTA; caller synchronizes).
__device__ __forceinline__ void fill_lane_tables(const KModel &M, uint32_t *s_tab) {
  const bool has_cm = M.flags & kFlagHasCharsmap;
  for (uint32_t i = threadIdx.x; i < 8 + 1024 + 128 + 4; i += blockDim.x) {
    uint32_t v;
    if (i < 8) v = M.cm_lead[i];
    else if (i < 8 + 1024) v = M.cm_pair[i - 8];
    else if (i < 8 + 1024 + 128) v = static_cast<uint32_t>(M.cm_solo[i - 8 - 1024]);
    else {  // plain ASCII bytes: no charsmap rule starts with them and they are not the space
      const uint32_t wq = i - (8 + 1024 + 128);
      v = ~(has_cm ? M.cm_lead[wq] : 0u);
      if (wq == 1) v &= ~1u;  // ' ' = 0x20
    }
    s_tab[i] = v;
  }
  // "simple" ASCII bytes (space included): followed by another ASCII byte they are always their own chunk -- no
  // rule is the byte alone or the byte + an ASCII byte.  (nmt_nfkc has letter + combining-mark compositions, so
  // most letters DO start rules; those need a non-ASCII second byte, which the caller excludes.)
  for (uint32_t wq = threadIdx.x >> 5; wq < 4; wq += blockDim.x >> 5) {
    const uint32_t ch = wq * 32 + (threadIdx.x & 31);
    bool simple = true;
    if (has_cm && ((M.cm_lead[wq] >> (ch & 31u)) & 1u)) {
      simple = M.cm_solo[ch] < 0;
      for (uint32_t q = 0; q < 4; ++q) simple = simple && M.cm_pair[((ch * 256u) >> 5) + q] == 0u;
    }
    const uint32_t word = __ballot_sync(0xFFFFFFFFu, simple);
    if ((threadIdx.x & 31) == 0) s_tab[8 + 1024 + 128 + 4 + wq] = word;
  }
}

// Streamed host batches (engine.cu, encode_host_streamed): the batch arrives in pieces of 2^piece_shift
// sentences and *B.ready counts the sentences whose bytes are in HBM.  Lane 0 of a warp waits for the piece
// that holds its group; the wait is bounded so that a stalled copy can never hang the GPU.
__device__ __forceinline__ void lane_wait_input(const KBatch &B, uint32_t first, uint32_t lane) {
  if (!B.ready) return;
  if (lane == 0) {
    uint32_t need = ((first >> B.piece_shift) + 1u) << B.piece_shift;
    if (need > B.n) need = B.n;
    need += B.ready_base;
    const volatile uint32_t *r = B.ready;
    if (B.kstats) atomicAdd(B.kstats + 3, 1ull);
    if (*r < need) {
      const long long t0 = clock64();
      while (*r < need) {
        __nanosleep(200);
        if (clock64() - t0 > 6000000000ll || (*reinterpret_cast<const volatile uint32_t *>(B.status + 1) & 2u)) {
          atomicOr(B.status + 1, 2u);  // ~3 s without progress: give up (the host reports the error)
          break;
        }
      }
      if (B.kstats) atomicAdd(B.kstats, static_cast<unsigned long long>(clock64() - t0));
    }
    // No fence here: __threadfence() is MEMBAR.SC + CCTL.IVALL on sm_100, and wiping the SM's L1 twice per group made
    // the whole kernel 1.4x slower on the mixed-script corpus (profiles/README.md).  The input loads below are issued
    // after this load has returned (the loop's exit depends on it), and they cannot hit a stale L1 line: a line of
    // the input is first touched by a sentence of the piece it arrived with (copies are cut at 128-byte lines).
  }
  __syncwarp();
}

struct LaneCtx {
  uint32_t *text_w;  // + word*32 (already offset by lane)
  uint32_t *log;     // + t*32    (already offset by lane)
  float *rs;         // ring scores, + slot*32 (already offset by lane)
  uint32_t *rb;      // ring back-pointers (plen<<24 | unit), 0 = unset
  const uint32_t *s_lead, *s_pair;
  const int32_t *s_solo;
  const uint32_t *s_plain;  // bit b: ASCII byte b is copied verbatim (no rule starts with it, not a space)
  const uint32_t *s_plainsp;  // bit b: ASCII byte b followed by an ASCII byte is always its own chunk (space included)
  unsigned long long pol;     // L2 cache policy of the slab accesses (slab_policy())
};

// The per-lane slabs (normalized text, back-pointer log) are written and read back within one group: ~12 KB per
// resident warp, ~40 MB per GPU, which fits L2 -- but only stays there if the batch's streamed input and ids do not
// push it out.  Every slab access carries an L2 eviction-priority hint (evict_last); the once-read input and the
// once-written ids use the streaming forms (__ldcs / __stcs).
__device__ __forceinline__ unsigned long long slab_policy(uint32_t mode) {
  unsigned long long pol;
  if (mode == 1u) asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  else if (mode == 2u) asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  else asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ uint32_t slab_ld(const uint32_t *p, unsigned long long pol) {
  uint32_t v;
  asm volatile("ld.global.L2::cache_hint.u32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol) : "memory");
  return v;
}
__device__ __forceinline__ void slab_st(uint32_t *p, uint32_t v, unsigned long long pol) {
  asm volatile("st.global.L2::cache_hint.u32 [%0], %1, %2;" :: "l"(p), "r"(v), "l"(pol) : "memory");
}
// End of a group: the rows of the warp's slab that the group used are dead.  Without a hint L2 keeps them as dirty
// lines: they are written back to HBM when they are finally evicted (traffic for nothing) and, until then, they take
// the place of the rows that are still live in other warps.  discard.L2 drops a line without write-back.  Warp-
// collective; row r of a slab is one 128-byte line (32 lanes x 4 bytes).  The barriers order the group's last reads
// before the discards and the discards before the next group's first writes (other lanes' words of the same line).
__device__ __forceinline__ void slab_discard(const LaneCtx &c, uint32_t lane, uint32_t text_rows, uint32_t log_rows) {
  __syncwarp();
  const uint8_t *tb = reinterpret_cast<const uint8_t *>(c.text_w - lane);
  for (uint32_t r = lane; r < text_rows; r += 32)
    asm volatile("discard.global.L2 [%0], 128;" :: "l"(tb + static_cast<size_t>(r) * 128) : "memory");
  const uint8_t *lb = reinterpret_cast<const uint8_t *>(c.log - lane);
  for (uint32_t r = lane; r < log_rows; r += 32)
    asm volatile("discard.global.L2 [%0], 128;" :: "l"(lb + static_cast<size_t>(r) * 128) : "memory");
  __syncwarp();
}

// Sequential byte stream over a lane's input: 16-byte aligned chunks (next chunk prefetched)
// feed a 64-bit shift register that always exposes the next >= 4 bytes.  The aligned chunks
// over-read into the neighbouring sentences by up to 15 bytes; a streamed host batch (engine.cu)
// therefore cuts its copies at 128-byte lines, so that every line a sentence touches has landed
// completely before the sentence's piece is announced.
struct ByteStream {
  const uint4 *cp;      // chunk that `nxt` was loaded from, + 1
  const uint4 *cend;    // first chunk past the sentence
  uint4 cur, nxt;
  uint32_t wi;          // next word of `cur` to feed (0..3)
  unsigned long long win;
  uint32_t have;        // valid bytes in win
  __device__ __forceinline__ uint32_t next_word() {
    const uint32_t w = wi == 0 ? cur.x : (wi == 1 ? cur.y : (wi == 2 ? cur.z : cur.w));
    if (++wi == 4) {
      wi = 0;
      cur = nxt;
      nxt = cp < cend ? __ldcs(cp) : make_uint4(0, 0, 0, 0);
      ++cp;
    }
    return w;
  }
  __device__ __forceinline__ void init(const uint8_t *p, const uint8_t *hi) {
    const uintptr_t a = reinterpret_cast<uintptr_t>(p);
    const uint4 *c0 = reinterpret_cast<const uint4 *>(a & ~static_cast<uintptr_t>(15));
    cend = reinterpret_cast<const uint4 *>((reinterpret_cast<uintptr_t>(hi) + 15) & ~static_cast<uintptr_t>(15));
    cur = __ldcs(c0);  // streaming (evict-first) loads: the input is read once and must not push the slabs out of L2
    nxt = c0 + 1 < cend ? __ldcs(c0 + 1) : make_uint4(0, 0, 0, 0);
    cp = c0 + 2;
    wi = static_cast<uint32_t>((a & 15) >> 2);
    const uint32_t mis = static_cast<uint32_t>(a & 3);
    const uint32_t w = next_word();
    win = static_cast<unsigned long long>(w >> (8 * mis));
    have = 4 - mis;
    win |= static_cast<unsigned long long>(next_word()) << (8 * have);
    have += 4;
  }
  __device__ __forceinline__ uint32_t peek(uint32_t i) const { return static_cast<uint32_t>(win >> (8 * i)) & 0xFFu; }
  __device__ __forceinline__ void consume(uint32_t c) {  // c <= 4
    win >>= 8 * c;
    have -= c;
    if (have <= 4) {
      win |= static_cast<unsigned long long>(next_word()) << (8 * have);
      have += 4;
    }
  }
};

// Sequential normalizer for one lane.  Returns the normalized length, or 0xFFFFFFFF if
// it exceeds `cap` (the caller defers the sentence).
__device__ __forceinline__ uint32_t lane_normalize(const KModel &M, const uint8_t *in, uint32_t len, const LaneCtx &c,
                                                   uint32_t cap) {
  const bool rm = M.flags & kFlagRemoveExtraWs;
  const bool esc = M.flags & kFlagEscapeWs;
  const bool suffix = M.flags & kFlagWsSuffix;
  const bool addp = M.flags & kFlagAddDummyPrefix;
  const bool has_user = M.flags & kFlagHasUserSymbols;
  const bool has_cm = M.flags & kFlagHasCharsmap;
  if (len == 0) return 0;
  ByteStream S;
  S.init(in, in + len);
  uint32_t out = 0;  // normalized bytes produced
  uint32_t acc = 0;  // partial word
  bool overflow = false;
  auto put = [&](uint32_t ch) {
    acc |= ch << ((out & 3u) * 8u);
    if ((out & 3u) == 3u) {
      if (out < cap) slab_st(c.text_w + static_cast<size_t>(out >> 2) * 32, acc, c.pol); else overflow = true;
      acc = 0;
    }
    ++out;
  };
  auto put_ws = [&]() {
    if (esc) { put(0xE2); put(0x96); put(0x81); } else { put(' '); }
  };
  uint32_t pos = 0;
  bool is_prev_space = rm;  // normalizer.cc:130
  bool started = !rm;       // the heading-space loop (:86-95) is over
  if (started && addp && !suffix) put_ws();  // dummy prefix (:128); with the heading loop it is emitted when that ends
  // One chunk of NormalizePrefix (normalizer.cc:195-253) + the emit logic of Normalize (:131-163)
  while (pos < len) {
    const uint32_t rem = len - pos;
    // ---- fast path: four ASCII bytes at once, each "simple" (its own chunk when an ASCII byte follows) and with
    //      an ASCII byte (or the end of the sentence) after the window.  Branch-free restatement of :131-163 for
    //      such chunks: a space after a space is dropped (remove_extra_whitespaces), otherwise it becomes U+2581 or
    //      stays ' '; the <= 8 output bytes are appended with at most two word stores. ----
    if (started && !has_user && rem >= 4) {
      const uint32_t w4 = static_cast<uint32_t>(S.win);
      const uint32_t c0 = w4 & 0xFFu, c1 = (w4 >> 8) & 0xFFu, c2 = (w4 >> 16) & 0xFFu, c3 = w4 >> 24;
      if (!(w4 & 0x80808080u) && ((c.s_plainsp[c0 >> 5] >> (c0 & 31u)) & (c.s_plainsp[c1 >> 5] >> (c1 & 31u)) &
                                  (c.s_plainsp[c2 >> 5] >> (c2 & 31u)) & (c.s_plainsp[c3 >> 5] >> (c3 & 31u)) & 1u) &&
          (rem == 4 || S.peek(4) < 0x80u)) {
        unsigned long long chunk = 0;
        uint32_t clen = 0;
        bool prev = is_prev_space;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const uint32_t ch = (w4 >> (8 * i)) & 0xFFu;
          const bool sp = ch == ' ';
          const bool emit = !(sp && prev);
          const uint32_t bytes = (sp && esc) ? 0x8196E2u : ch;  // U+2581 = E2 96 81
          const uint32_t blen = emit ? ((sp && esc) ? 3u : 1u) : 0u;
          chunk |= static_cast<unsigned long long>(emit ? bytes : 0u) << (8u * clen);
          clen += blen;
          prev = sp && rm;
        }
        is_prev_space = prev;
        const uint32_t r8 = (out & 3u) * 8u;
        const unsigned long long lo = static_cast<unsigned long long>(acc) | (chunk << r8);
        const uint32_t hi = r8 ? static_cast<uint32_t>(chunk >> (64u - r8)) : 0u;
        const uint32_t nw = ((out & 3u) + clen) >> 2;  // full words completed: 0..2
        if (out <= cap) {
          uint32_t *wp = c.text_w + static_cast<size_t>(out >> 2) * 32;
          if (nw >= 1) slab_st(wp + 0, static_cast<uint32_t>(lo), c.pol);
          if (nw >= 2) slab_st(wp + 32, static_cast<uint32_t>(lo >> 32), c.pol);
        }
        acc = nw == 0 ? static_cast<uint32_t>(lo) : (nw == 1 ? static_cast<uint32_t>(lo >> 32) : hi);
        out += clen;
        if (out > cap) overflow = true;
        pos += 4;
        S.consume(4);
        continue;
      }
    }
    const uint32_t b = S.peek(0);
    uint32_t consumed = 1;
    // replacement string: kind + (pointer | inline bytes)
    uint32_t kind = kChunkChar, spl = 1;
    const uint8_t *sp = nullptr;
    bool generic = false;
    if (has_user) {
      const uint32_t ul = user_longest(M, in + pos, rem);
      if (ul) { consumed = ul; spl = ul; kind = kChunkVerbatim; sp = in + pos; generic = true; }
    }
    if (!generic) {
      uint32_t longest = 0, value = 0;
      if (has_cm && ((c.s_lead[b >> 5] >> (b & 31u)) & 1u)) {
        if (b < 0x80u) {
          bool cont = false;
          if (rem > 1) {
            const uint32_t c2 = S.peek(1);
            cont = (c.s_pair[(b * 256u + c2) >> 5] >> (c2 & 31u)) & 1u;
          }
          if (cont) longest = charsmap_longest_win(M, S.win, S.have, in + pos, rem, &value);
          else {
            const int32_t so = c.s_solo[b];
            if (so >= 0) { longest = 1; value = static_cast<uint32_t>(so); }
          }
        } else {
          longest = charsmap_longest_win(M, S.win, S.have, in + pos, rem, &value);
        }
      }
      if (longest) {
        consumed = longest; kind = kChunkTarget; sp = M.cm_targets + value; generic = true;
        spl = 0;
        while (__ldg(sp + spl) != 0) ++spl;
      } else if (b < 0x80u) {
        // ---- fast path: one ASCII byte that is not a rule ----
        if (!started) {
          if (b == ' ') { ++pos; S.consume(1); continue; }  // heading space
          started = true;
          if (addp && !suffix) put_ws();
        }
        if (b == ' ') {
          if (!is_prev_space) { put_ws(); is_prev_space = rm; }
        } else {
          put(b);
          is_prev_space = false;
        }
        ++pos;
        S.consume(1);
        continue;
      } else {
        // DecodeUTF8 / IsValidDecodeUTF8 (util.cc:51-84) on the stream's look-ahead bytes
        uint32_t l = 0;
        const uint32_t b1 = S.peek(1), b2 = S.peek(2), b3 = S.peek(3);
        if (rem >= 2 && (b & 0xE0u) == 0xC0u) {
          if (is_trail(b1) && (((b & 0x1Fu) << 6) | (b1 & 0x3Fu)) >= 0x80u) l = 2;
        } else if (rem >= 3 && (b & 0xF0u) == 0xE0u) {
          const uint32_t cp = ((b & 0x0Fu) << 12) | ((b1 & 0x3Fu) << 6) | (b2 & 0x3Fu);
          if (is_trail(b1) && is_trail(b2) && cp >= 0x800u && (cp < 0xD800u || cp >= 0xE000u)) l = 3;
        } else if (rem >= 4 && (b & 0xF8u) == 0xF0u) {
          const uint32_t cp = ((b & 0x07u) << 18) | ((b1 & 0x3Fu) << 12) | ((b2 & 0x3Fu) << 6) | (b3 & 0x3Fu);
          if (is_trail(b1) && is_trail(b2) && is_trail(b3) && cp >= 0x10000u && cp <= 0x10FFFFu) l = 4;
        }
        if (!started) { started = true; if (addp && !suffix) put_ws(); }
        if (l) {  // a valid multi-byte character: never a space
          put(b); put(b1);
          if (l > 2) put(b2);
          if (l > 3) put(b3);
          consumed = l;
        } else {  // malformed: one byte -> U+FFFD (normalizer.cc:231-244)
          put(0xEF); put(0xBF); put(0xBD);
          consumed = 1;
        }
        is_prev_space = false;
        pos += consumed;
        S.consume(consumed);
        continue;
      }
    }
    // ---- generic path: rule targets and verbatim user symbols ----
    auto sp_byte = [&](uint32_t i) -> uint32_t { return __ldg(sp + i); };
    if (!started) {
      if (spl == 1 && sp_byte(0) == ' ') {  // a chunk that is exactly " " during the heading loop
        pos += consumed;
        if (consumed <= 4) S.consume(consumed); else S.init(in + pos, in + len);
        continue;
      }
      started = true;
      if (addp && !suffix) put_ws();
    }
    {
      uint32_t i0 = 0;
      while (is_prev_space && i0 < spl && sp_byte(i0) == ' ') ++i0;  // :137-138
      if (i0 < spl) {
        uint32_t last = 0;
        for (uint32_t i = i0; i < spl; ++i) {
          last = sp_byte(i);
          if (last == ' ' && esc) { put(0xE2); put(0x96); put(0x81); } else put(last);
        }
        is_prev_space = last == ' ';
      }
      if (!rm) is_prev_space = false;
    }
    pos += consumed;
    if (consumed <= 4) S.consume(consumed); else S.init(in + pos, in + len);
  }
  if (!started) return 0;  // all chars are whitespace (:97-100)
  if (overflow || out > cap) return 0xFFFFFFFFu;
  // flush the partial word, then strip trailing spaces on the escaped output (:166-176)
  slab_st(c.text_w + static_cast<size_t>(out >> 2) * 32, acc, c.pol);
  if (rm) {
    auto byte_at = [&](uint32_t k) -> uint32_t {
      return (slab_ld(c.text_w + static_cast<size_t>(k >> 2) * 32, c.pol) >> ((k & 3u) * 8u)) & 0xFFu;
    };
    if (esc) {
      while (out >= 3 && byte_at(out - 3) == 0xE2 && byte_at(out - 2) == 0x96 && byte_at(out - 1) == 0x81) out -= 3;
    } else {
      while (out >= 1 && byte_at(out - 1) == ' ') out -= 1;
    }
  }
  if (suffix && addp) {  // :179
    if (out + 3 > cap) return 0xFFFFFFFFu;
    acc = (out & 3u) ? (slab_ld(c.text_w + static_cast<size_t>(out >> 2) * 32, c.pol) & ((1u << ((out & 3u) * 8u)) - 1u)) : 0u;
    put_ws();
    slab_st(c.text_w + static_cast<size_t>(out >> 2) * 32, acc, c.pol);
  }
  return out;
}

// K4: back-trace + id path of PopulateSentencePieceText (sentencepiece_processor.cc:547-636) over a lane's
// back-pointer log: two coalesced backward scans (count, then write) around one warp-aggregated claim of output space.
// entry t (t = 0..nlog-1) = plen (6 bits) << 24 | (previous char length - 1) << 22 | trie unit (kLaneUnk: UNK piece);
// bit 31 (lane2 whole-word entries): the previous logged position is plen bytes back.
__device__ __forceinline__ void lane_finish(const KModel &M, const KBatch &B, const LaneCtx &c, uint32_t n, uint32_t nlog,
                                            uint32_t lane, bool have, bool defer, uint32_t sent, bool bf) {
  // ---------------- K4: coalesced backward scans of the log ----------------
  // entry t (t = 0..nlog-1) belongs to the (t+1)-th character boundary p_t; the character
  // before p_t has (entry>>22 & 3) + 1 bytes, so positions are recovered going backwards.
  const uint32_t max_log = __reduce_max_sync(0xFFFFFFFFu, nlog);
  uint32_t count = 0;
  {
    uint32_t pos_b = n, want = n;
    bool prev_unk = false;
    for (uint32_t tb = (max_log + 3u) & ~3u; tb > 0; tb -= 4) {
      uint32_t ev[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {  // four independent, coalesced loads per trip
        const uint32_t t = tb - 1 - j;
        ev[j] = t < nlog ? slab_ld(c.log + static_cast<size_t>(t) * 32, c.pol) : 0u;
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint32_t t = tb - 1 - j;
        if (t < nlog) {
          const uint32_t e = ev[j];
          if (pos_b == want) {
            const uint32_t plen = (e >> 24) & 63u;
            const bool isunk = (e & 0x3FFFFFu) == kLaneUnk;
            if (bf) count += isunk ? plen : 1u;
            else count += !(isunk && prev_unk);
            prev_unk = isunk;
            want -= plen;
          }
          pos_b -= (e >> 31) ? ((e >> 24) & 63u) : ((e >> 22) & 3u) + 1u;  // whole-word entries (lane2) step back plen bytes
        }
      }
    }
    if (n && want != 0) { atomicOr(B.status + 1, 1u); count = 0; }
  }
  // one claim of output space per warp
  uint32_t incl = count;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, d);
    if (lane >= static_cast<uint32_t>(d)) incl += t;
  }
  const uint32_t total = __shfl_sync(0xFFFFFFFFu, incl, 31);
  unsigned long long pos = 0;
  if (lane == 0 && total) {
    pos = atomicAdd(B.cursor, static_cast<unsigned long long>(total));
    if (pos + total > B.tmp_cap) atomicOr(B.status + 2, 1u);
  }
  pos = __shfl_sync(0xFFFFFFFFu, pos, 0);
  const bool room = pos + total <= B.tmp_cap;
  pos += incl - count;
  if (have && !defer) {
    B.sent_start[sent] = pos;
    B.sent_count[sent] = room ? count : 0u;
  }
  // second backward scan: write ids from the end
  if (room) {
    uint32_t pos_b = n, want = n, w = count;
    bool prev_unk = false;
    for (uint32_t tb = (max_log + 3u) & ~3u; tb > 0; tb -= 4) {
      uint32_t ev[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint32_t t = tb - 1 - j;
        ev[j] = t < nlog ? slab_ld(c.log + static_cast<size_t>(t) * 32, c.pol) : 0u;
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
      const uint32_t t = tb - 1 - j;
      if (t < nlog && w > 0) {
        const uint32_t e = ev[j];
        if (pos_b == want) {
          const uint32_t plen = (e >> 24) & 63u;
          const uint32_t idx = e & 0x3FFFFFu;
          const bool isunk = idx == kLaneUnk;
          if (isunk) {
            if (bf) {
              for (uint32_t i = 0; i < plen; ++i) {
                const uint32_t kk = want - 1 - i;
                const uint32_t ch = (slab_ld(c.text_w + static_cast<size_t>(kk >> 2) * 32, c.pol) >> ((kk & 3u) * 8u)) & 0xFFu;
                __stcs(B.tmp_ids + pos + (--w), __ldg(M.byte_to_id + ch));
              }
            } else if (!prev_unk) {
              __stcs(B.tmp_ids + pos + (--w), M.unk_id);
            }
          } else {
            __stcs(B.tmp_ids + pos + (--w), __ldg(M.trie_id + idx));  // streaming store
          }
          prev_unk = isunk;
          want -= plen;
        }
        pos_b -= (e >> 31) ? ((e >> 24) & 63u) : ((e >> 22) & 3u) + 1u;  // whole-word entries (lane2) step back plen bytes
      }
      }
    }
  }
  if (B.slab_discard) slab_discard(c, lane, (__reduce_max_sync(0xFFFFFFFFu, n) >> 2) + 4u, max_log);
}

// shared memory per warp: ring of R slots, each {score f32, back-pointer u32, position tag u16} x 32 lanes
__host__ __device__ inline uint32_t lane_ring_bytes(uint32_t R) { return R * 32u * (4u + 4u + 2u); }

// The reference's candidate score for a piece edge (unigram_model.cc:960-993) and whether it beats the value stored at
// the target: `sc_bits` = the piece's score (NORMAL) or unused (USER_DEFINED: plen * max_score - 0.1).  Exact float
// formulation of the mixed double comparison (Q1) when base_regular: with |score|, |base| in {0} U [2^-10, 2^18) the
// double sum a + b is exact, so (float)cand == fl(a + b) and cand > cur <=> ns > cur || (ns == cur && err > 0), err
// being the exact rounding error of the float add (Knuth two-sum).
__device__ __forceinline__ bool lane_candidate(uint32_t kind, uint32_t sc_bits, uint32_t plen, float base, bool base_regular,
                                               float curs, bool unset, float max_score, float *ns) {
  if (kind == kKindNormal && base_regular) {
    const float a = __uint_as_float(sc_bits);
    *ns = __fadd_rn(a, base);
    const float bb = __fsub_rn(*ns, a);
    const float err = __fadd_rn(__fsub_rn(a, __fsub_rn(*ns, bb)), __fsub_rn(base, bb));
    return unset || *ns > curs || (*ns == curs && err > 0.f);
  }
  const double sc = kind == kKindNormal ? static_cast<double>(__uint_as_float(sc_bits))
                                        : static_cast<double>(__fmul_rn(static_cast<float>(plen), max_score)) - 0.1;
  const double cand = sc + static_cast<double>(base);
  *ns = static_cast<float>(cand);
  return unset || cand > static_cast<double>(curs);
}

constexpr uint32_t kLogWordStep = 1u << 31;  // log entry: the previous logged position is plen bytes back (whole word)
constexpr uint32_t kWsWord = 0x8196E2u;      // U+2581 as the low three bytes of a little-endian word

// Whole-word shortcut (kFlagFastWords; engine.cu upload_word_safe has the proof): when no piece contains U+2581
// past its first byte, every segmentation has a token boundary in front of every U+2581, so the Viterbi problem of
// a word [b, e) (U+2581 + the characters up to the next U+2581) only sees the rest of the sentence through the
// float best_path_score at b.  If the word IS a piece P whose score beats the best split of the word by more than
// the rounding noise the float recurrence can accumulate up to position e (M.word_safe[unit] = the largest such e),
// the reference necessarily ends the word with P alone.  The walk from b reaches e on P's node, P has just been
// relaxed into e exactly as the reference relaxes it (first candidate of e), and the starts inside the word are
// skipped: 73 % of the words of the English corpus, half of all character starts.
// U+2581 step: every walk from a U+2581 starts with root -> E2 -> E2 96 -> U+2581, and the first two are no pieces
// (KModel::ws_unit).  The start transition onto a U+2581 therefore puts the walk on that node at once, 3 bytes in,
// relaxing the piece "U+2581" as the walk would: 3 of the trips of every word (~60 of 272 per English sentence) go.
__global__ void __launch_bounds__(1024, 1) encode_unigram_lane_kernel(const KModel M, const KBatch B, uint8_t *slabs,
                                                                       uint32_t cap, uint32_t R) {
  extern __shared__ __align__(128) uint8_t smem[];
  uint32_t *s_tab = reinterpret_cast<uint32_t *>(smem);
  uint8_t *rings = smem + kLaneTableBytes;
  fill_lane_tables(M, s_tab);
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t warp_in_cta = threadIdx.x >> 5;
  const uint32_t warp_global = blockIdx.x * (blockDim.x >> 5) + warp_in_cta;
  LaneCtx c;
  c.pol = slab_policy(B.slab_l2);
  uint16_t *rp;  // ring position tags: a slot belongs to position p iff rp == p (no clearing, skipped positions
                 // of whole words leave stale slots behind that simply fail the test)
  {
    uint8_t *ring = rings + static_cast<size_t>(warp_in_cta) * lane_ring_bytes(R);
    c.rs = reinterpret_cast<float *>(ring) + lane;
    c.rb = reinterpret_cast<uint32_t *>(ring + R * 32 * 4) + lane;
    rp = reinterpret_cast<uint16_t *>(ring + R * 32 * 8) + lane;
    uint8_t *slab = slabs + static_cast<size_t>(warp_global) * lane_slab_bytes(cap);
    c.text_w = reinterpret_cast<uint32_t *>(slab) + lane;
    c.log = reinterpret_cast<uint32_t *>(slab) + static_cast<size_t>(cap / 4 + kLaneTextSlack) * 32 + lane;
    c.s_lead = s_tab;
    c.s_pair = s_tab + 8;
    c.s_solo = reinterpret_cast<const int32_t *>(s_tab + 8 + 1024);
    c.s_plain = s_tab + 8 + 1024 + 128;
    c.s_plainsp = c.s_plain + 4;
  }
  const uint4 *node4 = M.trie_node4;
  const uint32_t root = __ldg(&node4[0]).x;
  const bool bf = M.flags & kFlagByteFallback;
  const bool regular = M.flags & kFlagRegularScores;
  const bool fastwords = M.flags & kFlagFastWords;
  const uint32_t r_wrap = R * 32;

  for (;;) {
    uint32_t first = 0;
    if (lane == 0) first = atomicAdd(B.work_counter, 32u);
    first = __shfl_sync(0xFFFFFFFFu, first, 0);
    if (first >= B.n) break;
    const bool tst = B.kstats != nullptr;  // trace / kstats mode: phase clocks (lane 0)
    const uint32_t t_g0 = tst ? static_cast<uint32_t>(clock64()) : 0u;
    lane_wait_input(B, first, lane);
    const bool have = first + lane < B.n;
    const uint32_t sent = have && B.order ? B.order[first + lane] : first + lane;
    // ---------------- K1 ----------------
    uint32_t n = 0;
    bool defer = false;
    if (have) {
      const unsigned long long off = B.offsets[sent];
      const unsigned long long len64 = B.offsets[sent + 1] - off;
      if (len64 > 4ull * cap || len64 > 0xFFF0ull || off < B.off_lo || off + len64 > B.off_hi) defer = true;
      else {
        n = lane_normalize(M, B.bytes + off, static_cast<uint32_t>(len64), c, cap);
        if (n == 0xFFFFFFFFu || n >= 0xFFF0u) { defer = true; n = 0; }  // (positions are 16-bit ring tags)
      }
      if (defer) {
        const uint32_t slot = atomicAdd(B.status, 1u);
        B.deferred[2 * slot] = sent;
        B.deferred[2 * slot + 1] = 0;
        B.sent_count[sent] = 0;  // until a later pass encodes it
      }
    }
    __syncwarp();
    const uint32_t t_g1 = tst ? static_cast<uint32_t>(clock64()) : 0u;
    // ---------------- K2: flat state machine, one trie transition per trip ----------------
    // text window: words w0..w3 = bytes [4*aw, 4*aw+16), aw = s >> 2; `cur` streams the bytes
    // from the walk position k (low byte first).  ss = ring slot of s, times 32.
    uint32_t s = 0, ss = 0, k = 0, l = root, lsafe = 0, mblen = 1, nlog = 0;
    bool has_single = false, done = n == 0;
    bool wstart = true;  // s is the first character of a word (text start or U+2581)
    float base = 0.f;
    bool base_regular = regular;  // base == 0
    uint32_t w0 = 0, w1 = 0, w2 = 0, w3 = 0;
    unsigned long long cur = 0;
    auto window_low = [&]() -> unsigned long long {  // bytes s .. s+7
      const uint32_t sh = (s & 3u) * 8u;
      return static_cast<unsigned long long>(__funnelshift_r(w0, w1, sh)) |
             (static_cast<unsigned long long>(__funnelshift_r(w1, w2, sh)) << 32);
    };
    auto window_high = [&]() -> unsigned long long {  // bytes s+8 .. (at least s+12)
      const uint32_t sh = (s & 3u) * 8u;
      return static_cast<unsigned long long>(__funnelshift_r(w2, w3, sh)) |
             (static_cast<unsigned long long>(w3 >> sh) << 32);
    };
    // relaxes the piece at trie unit v (kind, score bits) from s into s + plen
    auto relax = [&](uint32_t kind, uint32_t sc_bits, uint32_t v, uint32_t plen) {
      const uint32_t pos = s + plen;
      uint32_t sl = ss + plen * 32u;
      if (sl >= r_wrap) sl -= r_wrap;
      float ns;
      if (lane_candidate(kind, sc_bits, plen, base, base_regular, c.rs[sl], rp[sl] != pos, M.max_score, &ns)) {
        c.rs[sl] = ns;
        c.rb[sl] = (plen << 24) | v;
        rp[sl] = static_cast<uint16_t>(pos);
      }
    };
    // s is a U+2581 (s + 3 <= n, mblen == 3) and nothing has been walked from it: start on the node of U+2581
    auto ws_step = [&]() {
      k = s + 3u;
      l = M.ws_link;
      lsafe = M.ws_safe;
      cur >>= 24;
      const uint32_t kind = (M.ws_link >> kLinkKindShift) & 3u;
      if (kind == kKindNormal || kind == kKindUserDefined) {
        relax(kind, M.ws_score, M.ws_unit, 3u);
        has_single = true;
      }
    };
    const bool ws_on = M.ws_unit != kNoUnit;
    if (!done) {
      for (uint32_t r = 0; r < R; ++r) rp[r * 32] = 0xFFFFu;  // no slot belongs to a position of this sentence
      c.rs[0] = 0.f;
      w0 = slab_ld(c.text_w + 0, c.pol); w1 = slab_ld(c.text_w + 32, c.pol); w2 = slab_ld(c.text_w + 64, c.pol); w3 = slab_ld(c.text_w + 96, c.pol);
      mblen = one_char_len(w0 & 0xFFu);
      if (mblen > n) mblen = n;
      cur = window_low();
      if (ws_on && n >= 3u && (w0 & 0xFFFFFFu) == kWsWord) ws_step();
    }
    // optional counters (engine: SPM_B200_KSTATS; device-resident path only): [8] warp trips, [9] lane trips,
    // [10] starts retired, [11] whole words, [12] groups, [13] normalized bytes
    const bool kst = B.kstats != nullptr && B.seg_done == nullptr;
    uint32_t st_trips = 0, st_lane = 0, st_starts = 0, st_fast = 0;
    while (__any_sync(0xFFFFFFFFu, !done)) {
      if (kst) { ++st_trips; st_lane += !done; }
      if (!done) {
        bool end_walk = true;
        if (k < n) {
          const uint32_t d = k - s;
          uint32_t ch;
          if (d >= 13u) {  // beyond the register window: long piece, rare
            ch = (slab_ld(c.text_w + static_cast<size_t>(k >> 2) * 32, c.pol) >> ((k & 3u) * 8u)) & 0xFFu;
          } else {
            if (d == 8u) cur = window_high();
            ch = static_cast<uint32_t>(cur) & 0xFFu;
            cur >>= 8;
          }
          const uint32_t v = (l >> kLinkBaseShift) ^ ch;
          const uint4 nd = __ldg(&node4[v]);  // {link, child mask, score, word_safe}: one 16-byte load (L1/L2)
          if ((nd.x & kLinkLabelMask) == ch) {
            ++k;
            l = nd.x;
            lsafe = nd.w;
            const uint32_t kind = (nd.x >> kLinkKindShift) & 3u;
            if (kind == kKindNormal || kind == kKindUserDefined) {
              const uint32_t plen = k - s;
              relax(kind, nd.z, v, plen);
              has_single |= plen == mblen;
            }
            // early termination: if the node has no child on the next byte the failing
            // probe (and its cold miss) is skipped and the start transition happens now
            if (k < n) {
              uint32_t nb;
              const uint32_t d2 = k - s;
              if (d2 >= 13u) nb = (slab_ld(c.text_w + static_cast<size_t>(k >> 2) * 32, c.pol) >> ((k & 3u) * 8u)) & 0xFFu;
              else nb = d2 == 8u ? static_cast<uint32_t>(window_high()) & 0xFFu : static_cast<uint32_t>(cur) & 0xFFu;
              end_walk = !((nd.y >> (nb & 31u)) & 1u);
            }
          }
        }
        if (end_walk) {
          // the walk from s is over (traverse() == -2, or end of text)
          bool fast = false;
          if (fastwords && wstart && k > s && ((l >> kLinkKindShift) & 3u) == kKindNormal) {
            // the walk covered [s, k) and ended on a NORMAL piece: is k the end of the word, early enough to be safe?
            bool wend = k >= n;
            if (!wend && k + 3u <= n) {
              const uint32_t o = k - ((s >> 2) << 2);
              uint32_t b3;
              if (o <= 13u) {
                const uint32_t wi = o >> 2;
                const uint32_t lo = wi == 0u ? w0 : (wi == 1u ? w1 : (wi == 2u ? w2 : w3));
                const uint32_t hi = wi == 0u ? w1 : (wi == 1u ? w2 : (wi == 2u ? w3 : 0u));
                b3 = __funnelshift_r(lo, hi, (o & 3u) * 8u) & 0xFFFFFFu;
              } else {
                b3 = 0;
                for (uint32_t i = 0; i < 3u; ++i)
                  b3 |= ((slab_ld(c.text_w + static_cast<size_t>((k + i) >> 2) * 32, c.pol) >> (((k + i) & 3u) * 8u)) & 0xFFu) << (8u * i);
              }
              wend = b3 == kWsWord;
            }
            fast = wend && k <= lsafe;
          }
          const uint32_t s_old = s;
          uint32_t steplog;
          if (kst) { ++st_starts; st_fast += fast; }
          if (fast) {
            // the piece was relaxed into k when the walk stepped onto its node; nothing else can win there
            ss += (k - s) * 32u;
            s = k;
            steplog = kLogWordStep;
          } else {
            uint32_t sl = ss + mblen * 32u;
            if (sl >= r_wrap) sl -= r_wrap;
            if (!has_single) {  // UNK edge, unigram_model.cc:995-1005
              const float cand = __fadd_rn(M.unk_score, base);
              if (rp[sl] != s + mblen || cand > c.rs[sl]) {
                c.rs[sl] = cand;
                c.rb[sl] = (mblen << 24) | kLaneUnk;
                rp[sl] = static_cast<uint16_t>(s + mblen);
              }
            }
            ss = sl;
            s += mblen;
            steplog = (mblen - 1u) << 22;
          }
          if (ss >= r_wrap) ss -= r_wrap;
          // position s is final: append (plen | previous char length or whole-word step | unit) to the log
          slab_st(c.log + static_cast<size_t>(nlog) * 32, c.rb[ss] | steplog, c.pol);
          ++nlog;
          if (s >= n) {
            done = true;
          } else {
            base = c.rs[ss];
            base_regular = regular && (base == 0.f || (fabsf(base) >= 0.0009765625f && fabsf(base) < 262144.f));
            // slide the text window so that it is anchored at s; prefetch the new tail word
            const uint32_t jw = (s >> 2) - (s_old >> 2);
            if (jw == 1u) {
              w0 = w1; w1 = w2; w2 = w3;
              w3 = slab_ld(c.text_w + static_cast<size_t>((s >> 2) + 3) * 32, c.pol);
            } else if (jw == 2u) {
              w0 = w2; w1 = w3;
              w2 = slab_ld(c.text_w + static_cast<size_t>((s >> 2) + 2) * 32, c.pol);
              w3 = slab_ld(c.text_w + static_cast<size_t>((s >> 2) + 3) * 32, c.pol);
            } else if (jw != 0u) {
              const uint32_t *tw = c.text_w + static_cast<size_t>(s >> 2) * 32;
              w0 = slab_ld(tw + 0, c.pol); w1 = slab_ld(tw + 32, c.pol); w2 = slab_ld(tw + 64, c.pol); w3 = slab_ld(tw + 96, c.pol);
            }
            cur = window_low();
            wstart = (static_cast<uint32_t>(cur) & 0xFFFFFFu) == kWsWord;
            mblen = one_char_len(static_cast<uint32_t>(cur) & 0xFFu);
            if (mblen > n - s) mblen = n - s;
            k = s;
            l = root;
            has_single = false;
            if (ws_on && wstart && s + 3u <= n) ws_step();
          }
        }
      }
    }
    if (kst) {
      typedef unsigned long long ull;
      uint32_t nb = n;
      for (int d = 16; d > 0; d >>= 1) {
        st_lane += __shfl_xor_sync(0xFFFFFFFFu, st_lane, d);
        st_starts += __shfl_xor_sync(0xFFFFFFFFu, st_starts, d);
        st_fast += __shfl_xor_sync(0xFFFFFFFFu, st_fast, d);
        nb += __shfl_xor_sync(0xFFFFFFFFu, nb, d);
      }
      if (lane == 0) {
        atomicAdd(B.kstats + 8, ull(st_trips)); atomicAdd(B.kstats + 9, ull(st_lane)); atomicAdd(B.kstats + 10, ull(st_starts));
        atomicAdd(B.kstats + 11, ull(st_fast)); atomicAdd(B.kstats + 12, ull(1)); atomicAdd(B.kstats + 13, ull(nb));
      }
    }
    const uint32_t t_g2 = tst ? static_cast<uint32_t>(clock64()) : 0u;
    lane_finish(M, B, c, n, nlog, lane, have, defer, sent, bf);  // K4
    const uint32_t t_g3 = tst ? static_cast<uint32_t>(clock64()) : 0u;
    lane_drain(B, sent, have, lane);  // K6 (fused host path only)
    __syncwarp();
    if (tst && lane == 0) {
      typedef unsigned long long ull;
      atomicAdd(B.kstats + 4, ull(static_cast<uint32_t>(clock64()) - t_g0)); atomicAdd(B.kstats + 5, ull(t_g1 - t_g0));
      atomicAdd(B.kstats + 6, ull(t_g2 - t_g1)); atomicAdd(B.kstats + 7, ull(t_g3 - t_g2));
    }
  }
}

// The same kernel without the whole-word shortcut: the round-1 state machine (8-byte {link, child mask} nodes, score
// lookup on a match, cleared ring slots instead of position tags).  Text with few space-separated words -- CJK, the
// byte-fallback / mixed-script configuration -- gains nothing from the shortcut and would only pay for its bookkeeping
// (7.6 vs 6.5 ms per 1M mixed sentences), so the engine picks this instantiation for such batches (engine.cu,
// `pick_fast_words`); ring geometry R * 32 * 8 bytes per warp.
__global__ void __launch_bounds__(1024, 1) encode_unigram_lane_plain_kernel(const KModel M, const KBatch B, uint8_t *slabs,
                                                                       uint32_t cap, uint32_t R) {
  extern __shared__ __align__(128) uint8_t smem[];
  uint32_t *s_tab = reinterpret_cast<uint32_t *>(smem);
  uint8_t *rings = smem + kLaneTableBytes;
  fill_lane_tables(M, s_tab);
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t warp_in_cta = threadIdx.x >> 5;
  const uint32_t warp_global = blockIdx.x * (blockDim.x >> 5) + warp_in_cta;
  LaneCtx c;
  c.pol = slab_policy(B.slab_l2);
  {
    uint8_t *ring = rings + static_cast<size_t>(warp_in_cta) * (R * 32 * 8);
    c.rs = reinterpret_cast<float *>(ring) + lane;
    c.rb = reinterpret_cast<uint32_t *>(ring + R * 32 * 4) + lane;
    uint8_t *slab = slabs + static_cast<size_t>(warp_global) * lane_slab_bytes(cap);
    c.text_w = reinterpret_cast<uint32_t *>(slab) + lane;
    c.log = reinterpret_cast<uint32_t *>(slab) + static_cast<size_t>(cap / 4 + kLaneTextSlack) * 32 + lane;
    c.s_lead = s_tab;
    c.s_pair = s_tab + 8;
    c.s_solo = reinterpret_cast<const int32_t *>(s_tab + 8 + 1024);
    c.s_plain = s_tab + 8 + 1024 + 128;
    c.s_plainsp = c.s_plain + 4;
  }
  const uint2 *node2 = M.trie_node2;
  const uint32_t root = __ldg(&node2[0]).x;
  const bool bf = M.flags & kFlagByteFallback;
  const bool regular = M.flags & kFlagRegularScores;

  for (;;) {
    uint32_t first = 0;
    if (lane == 0) first = atomicAdd(B.work_counter, 32u);
    first = __shfl_sync(0xFFFFFFFFu, first, 0);
    if (first >= B.n) break;
    const bool tst = B.kstats != nullptr;  // trace / kstats mode: phase clocks (lane 0)
    const uint32_t t_g0 = tst ? static_cast<uint32_t>(clock64()) : 0u;
    lane_wait_input(B, first, lane);
    const bool have = first + lane < B.n;
    const uint32_t sent = have && B.order ? B.order[first + lane] : first + lane;
    // ---------------- K1 ----------------
    uint32_t n = 0;
    bool defer = false;
    if (have) {
      const unsigned long long off = B.offsets[sent];
      const unsigned long long len64 = B.offsets[sent + 1] - off;
      if (len64 > 4ull * cap || off < B.off_lo || off + len64 > B.off_hi) defer = true;
      else {
        n = lane_normalize(M, B.bytes + off, static_cast<uint32_t>(len64), c, cap);
        if (n == 0xFFFFFFFFu) { defer = true; n = 0; }
      }
      if (defer) {
        const uint32_t slot = atomicAdd(B.status, 1u);
        B.deferred[2 * slot] = sent;
        B.deferred[2 * slot + 1] = 0;
        B.sent_count[sent] = 0;  // until a later pass encodes it
      }
    }
    __syncwarp();
    const uint32_t t_g1 = tst ? static_cast<uint32_t>(clock64()) : 0u;
    // ---------------- K2: flat state machine, one trie transition per trip ----------------
    // text window: words w0..w3 = bytes [4*aw, 4*aw+16), aw = s >> 2; `cur` streams the bytes
    // from the walk position k (low byte first).
    uint32_t s = 0, ss = 0 /* ring slot of s */, k = 0, l = root, mblen = 1, nlog = 0;
    bool has_single = false, done = n == 0;
    float base = 0.f;
    bool base_regular = regular;  // base == 0
    uint32_t w0 = 0, w1 = 0, w2 = 0, w3 = 0;
    unsigned long long cur = 0;
    auto window_low = [&]() -> unsigned long long {  // bytes s .. s+7
      const uint32_t sh = (s & 3u) * 8u;
      return static_cast<unsigned long long>(__funnelshift_r(w0, w1, sh)) |
             (static_cast<unsigned long long>(__funnelshift_r(w1, w2, sh)) << 32);
    };
    auto window_high = [&]() -> unsigned long long {  // bytes s+8 .. (at least s+12)
      const uint32_t sh = (s & 3u) * 8u;
      return static_cast<unsigned long long>(__funnelshift_r(w2, w3, sh)) |
             (static_cast<unsigned long long>(w3 >> sh) << 32);
    };
    if (!done) {
      for (uint32_t r = 0; r < R; ++r) c.rb[r * 32] = 0u;  // all positions unset
      c.rs[0] = 0.f;
      w0 = slab_ld(c.text_w + 0, c.pol); w1 = slab_ld(c.text_w + 32, c.pol); w2 = slab_ld(c.text_w + 64, c.pol); w3 = slab_ld(c.text_w + 96, c.pol);
      mblen = one_char_len(w0 & 0xFFu);
      if (mblen > n) mblen = n;
      cur = window_low();
    }
    while (__any_sync(0xFFFFFFFFu, !done)) {
      if (!done) {
        bool end_walk = true;
        if (k < n) {
          const uint32_t d = k - s;
          uint32_t ch;
          if (d >= 13u) {  // beyond the register window: long piece, rare
            ch = (slab_ld(c.text_w + static_cast<size_t>(k >> 2) * 32, c.pol) >> ((k & 3u) * 8u)) & 0xFFu;
          } else {
            if (d == 8u) cur = window_high();
            ch = static_cast<uint32_t>(cur) & 0xFFu;
            cur >>= 8;
          }
          const uint32_t v = (l >> kLinkBaseShift) ^ ch;
          const uint2 nd = __ldg(&node2[v]);  // {link, child mask}: one 8-byte load (L1/L2)
          if ((nd.x & kLinkLabelMask) == ch) {
            ++k;
            l = nd.x;
            const uint32_t kind = (nd.x >> kLinkKindShift) & 3u;
            if (kind == kKindNormal || kind == kKindUserDefined) {
              const uint32_t plen = k - s;
              uint32_t sl = ss + plen;
              if (sl >= R) sl -= R;
              sl *= 32;
              const float curs = c.rs[sl];
              const bool unset = c.rb[sl] == 0u;
              float ns;
              bool better;
              if (kind == kKindNormal && base_regular) {
                // Exact float formulation of the reference's double comparison (Q1).  With
                // |score|, |base| in {0} U [2^-10, 2^18) the double sum a + b is exact, so
                // (float)cand == fl(a + b) and cand > cur <=> ns > cur || (ns == cur && err > 0),
                // err being the exact rounding error of the float add (Knuth two-sum).
                const float a = __uint_as_float(__ldg(M.trie_val + v));
                ns = __fadd_rn(a, base);
                const float bb = __fsub_rn(ns, a);
                const float err = __fadd_rn(__fsub_rn(a, __fsub_rn(ns, bb)), __fsub_rn(base, bb));
                better = unset || ns > curs || (ns == curs && err > 0.f);
              } else {
                const double sc = kind == kKindNormal
                                      ? static_cast<double>(__uint_as_float(__ldg(M.trie_val + v)))
                                      : static_cast<double>(__fmul_rn(static_cast<float>(plen), M.max_score)) - 0.1;
                const double cand = sc + static_cast<double>(base);
                better = unset || cand > static_cast<double>(curs);
                ns = static_cast<float>(cand);
              }
              if (better) {
                c.rs[sl] = ns;
                c.rb[sl] = (plen << 24) | v;
              }
              has_single |= plen == mblen;
            }
            // early termination: if the node has no child on the next byte the failing
            // probe (and its cold miss) is skipped and the start transition happens now
            if (k < n) {
              uint32_t nb;
              const uint32_t d2 = k - s;
              if (d2 >= 13u) nb = (slab_ld(c.text_w + static_cast<size_t>(k >> 2) * 32, c.pol) >> ((k & 3u) * 8u)) & 0xFFu;
              else nb = d2 == 8u ? static_cast<uint32_t>(window_high()) & 0xFFu : static_cast<uint32_t>(cur) & 0xFFu;
              end_walk = !((nd.y >> (nb & 31u)) & 1u);
            }
          }
        }
        if (end_walk) {
          // the walk from s is over (traverse() == -2, or end of text)
          uint32_t sl = ss + mblen;
          if (sl >= R) sl -= R;
          if (!has_single) {  // UNK edge, unigram_model.cc:995-1005
            const float cand = __fadd_rn(M.unk_score, base);
            if (c.rb[sl * 32] == 0u || cand > c.rs[sl * 32]) {
              c.rs[sl * 32] = cand;
              c.rb[sl * 32] = (mblen << 24) | kLaneUnk;
            }
          }
          // position s leaves the window; only character starts are ever targets, so its
          // slot is the only one that has to be cleared for position s + R
          c.rb[ss * 32] = 0u;
          s += mblen;
          ss = sl;
          // position s is final: append (plen | previous char length | unit) to the log
          slab_st(c.log + static_cast<size_t>(nlog) * 32, c.rb[ss * 32] | ((mblen - 1u) << 22), c.pol);
          ++nlog;
          if (s >= n) {
            done = true;
          } else {
            base = c.rs[ss * 32];
            base_regular = regular && (base == 0.f || (fabsf(base) >= 0.0009765625f && fabsf(base) < 262144.f));
            // slide the text window so that it is anchored at s; prefetch the new tail word
            if ((s >> 2) != ((s - mblen) >> 2)) {
              w0 = w1; w1 = w2; w2 = w3;
              w3 = slab_ld(c.text_w + static_cast<size_t>((s >> 2) + 3) * 32, c.pol);
            }
            cur = window_low();
            mblen = one_char_len(static_cast<uint32_t>(cur) & 0xFFu);
            if (mblen > n - s) mblen = n - s;
            k = s;
            l = root;
            has_single = false;
          }
        }
      }
    }
    const uint32_t t_g2 = tst ? static_cast<uint32_t>(clock64()) : 0u;
    lane_finish(M, B, c, n, nlog, lane, have, defer, sent, bf);  // K4
    const uint32_t t_g3 = tst ? static_cast<uint32_t>(clock64()) : 0u;
    lane_drain(B, sent, have, lane);  // K6 (fused host path only)
    __syncwarp();
    if (tst && lane == 0) {
      typedef unsigned long long ull;
      atomicAdd(B.kstats + 4, ull(static_cast<uint32_t>(clock64()) - t_g0)); atomicAdd(B.kstats + 5, ull(t_g1 - t_g0));
      atomicAdd(B.kstats + 6, ull(t_g2 - t_g1)); atomicAdd(B.kstats + 7, ull(t_g3 - t_g2));
    }
  }
}


}  // namespace spm_b200
#endif
