// engine.cu -- host side of the engine and the extern "C" boundary (include/spm_b200.h).
//
// Mirrors what SentencePieceProcessor::Load builds on the CPU
// (src/sentencepiece_processor.cc:242-281; ModelInterface::InitializePieces
// src/model_interface.cc:63-151; unigram::Model ctor src/unigram_model.cc:652-670;
// Normalizer::Init src/normalizer.cc:47-69) as flat device tables, and drives the
// kernels of kernels.cuh / bpe_kernel.cuh for a packed batch of sentences.
//
// There is no CPU fallback anywhere in this file: without a CUDA device
// spm_engine_create fails.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cfloat>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <random>
#include <thread>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/spm_b200.h"
#include "bpe_kernel.cuh"
#include "bpe_lane_kernel.cuh"
#include "bpe_lane2_kernel.cuh"
#include "device_model.h"
#include "kernels.cuh"
#include "lane_kernel.cuh"
#include "model_reader.h"
#include "order_kernel.cuh"
#include "decode_kernel.cuh"
#include "nbest_kernel.cuh"
#include "lattice_kernel.cuh"
#include "trie_builder.h"
#include "unigram_warp.cuh"

using namespace spm_b200;

namespace {

std::string g_create_error;
std::mutex g_create_mu;

#define CUDA_TRY(expr)                                                                          \
  do {                                                                                          \
    cudaError_t err__ = (expr);                                                                 \
    if (err__ != cudaSuccess) {                                                                 \
      set_error(std::string(#expr) + ": " + cudaGetErrorString(err__));                         \
      return SPM_ERR_CUDA;                                                                      \
    }                                                                                           \
  } while (0)

template <typename T>
struct DevBuf {
  T *p = nullptr;
  size_t cap = 0;  // elements
  cudaError_t ensure(size_t n, bool keep = false) {
    if (n <= cap) return cudaSuccess;
    size_t want = std::max(n, cap + cap / 2);
    T *np = nullptr;
    cudaError_t e = cudaMalloc(&np, want * sizeof(T) + 256);
    if (e != cudaSuccess) return e;
    if (keep && p && cap) cudaMemcpy(np, p, cap * sizeof(T), cudaMemcpyDeviceToDevice);
    if (p) cudaFree(p);
    p = np;
    cap = want;
    return cudaSuccess;
  }
  cudaError_t upload(const std::vector<T> &v) {
    cudaError_t e = ensure(v.size() ? v.size() : 1);
    if (e != cudaSuccess) return e;
    if (!v.empty()) e = cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

template <typename T>
struct PinBuf {
  T *p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t n) {
    if (n <= cap) return cudaSuccess;
    size_t want = std::max(n, cap + cap / 2);
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
    cudaError_t e = cudaMallocHost(&p, want * sizeof(T) + 64);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

bool valid_utf8(const char *s, size_t n) {
  size_t i = 0;
  const unsigned char *b = reinterpret_cast<const unsigned char *>(s);
  while (i < n) {
    const unsigned c = b[i];
    size_t l = c < 0x80 ? 1 : (c & 0xE0) == 0xC0 ? 2 : (c & 0xF0) == 0xE0 ? 3 : (c & 0xF8) == 0xF0 ? 4 : 0;
    if (!l || i + l > n) return false;
    uint32_t cp = l == 1 ? c : l == 2 ? c & 0x1F : l == 3 ? c & 0x0F : c & 0x07;
    for (size_t k = 1; k < l; ++k) {
      if ((b[i + k] & 0xC0) != 0x80) return false;
      cp = (cp << 6) | (b[i + k] & 0x3F);
    }
    if ((l == 2 && cp < 0x80) || (l == 3 && cp < 0x800) || (l == 4 && cp < 0x10000) || cp > 0x10FFFF ||
        (cp >= 0xD800 && cp < 0xE000))
      return false;
    i += l;
  }
  return true;
}

}  // namespace

struct spm_engine {
  int device = 0;
  int sm_count = 0;
  size_t smem_optin = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  std::mutex mu;
  mutable std::string err;

  ModelData model;
  DeviceTrie trie, user_trie;
  float min_score = 0.f, max_score = 0.f;
  int32_t unk_id = -1;
  uint32_t max_expand_num = 3, max_expand_den = 1;  // worst-case normalized bytes per input byte
  uint32_t charsmap_units = 0;
  bool bpe_word_split = false;

  // device tables
  DevBuf<uint32_t> d_link, d_val, d_user_link, d_cm_units, d_cm_lead, d_cm_pair, d_node2;
  DevBuf<int32_t> d_id, d_cm_solo, d_byte_to_id;
  DevBuf<uint8_t> d_cm_targets, d_types;
  DevBuf<float> d_scores;
  DevBuf<uint16_t> d_word_safe;
  DevBuf<uint4> d_node4;
  DevBuf<uint32_t> d_word_fast;
  DevBuf<uint4> d_bpe_cache;
  // SPM_B200_BPE_CACHE: log2 of the word-cache entries (64 bytes each), 0 = no cache.  Measured per 1M English
  // sentences (profiles/README.md): none 6.58 ms, 2^16 6.57, 2^18 5.45, 2^20 4.66, 2^21 4.43, 2^22 4.16 ms (256 MB of HBM)
  int bpe_cache_log2 = 22;
  int bpe_lane_version = 2;  // SPM_B200_BPE_LANE_V
  bool fast_words = true;  // SPM_B200_FASTWORDS
  int upload_word_safe();
  KModel km{};

  // tuning
  int G = 1;  // 1: lane kernel (sentence per lane); 32: warp kernel; 4/8/16: tile kernel; 64: tile kernel, 32 lanes
  int threads = 1024;
  uint32_t ncap = 256;
  uint32_t slab_discard = 1;  // SPM_B200_SLAB_DISCARD=0 turns it off (KBatch::slab_discard)
  uint32_t slab_l2 = 0;    // SPM_B200_SLAB_L2: L2 eviction priority of the slab accesses (KBatch::slab_l2)
  uint32_t lane_cap = 512;  // normalized-byte capacity per sentence of the lane kernel's slabs
  int ctas_per_sm = 1;

  // per-call buffers (grow only)
  DevBuf<uint8_t> d_bytes, d_tmp_norm, d_norm, d_long_scratch, d_lane_slabs, d_bpe_long;
  DevBuf<uint64_t> d_offsets;
  DevBuf<int32_t> d_tmp_ids, d_ids;
  DevBuf<uint32_t> d_tmp_tok_end, d_tok_end, d_tmp_n2o, d_n2o, d_sent_count, d_norm_len, d_deferred, d_deferred2, d_long_list, d_ctrl32;
  DevBuf<unsigned long long> d_sent_start, d_norm_start, d_id_offsets, d_norm_offsets, d_n2o_offsets, d_block_sums,
      d_ctrl64, d_long_off;
  PinBuf<int32_t> h_ids;
  PinBuf<uint32_t> h_tok_end, h_n2o, h_ctrl32, h_deferred;
  PinBuf<uint64_t> h_id_offsets, h_norm_offsets;
  PinBuf<unsigned long long> h_ctrl64;
  PinBuf<uint8_t> h_norm;
  // pipelined host API: two input slots, two output slots, copy streams
  DevBuf<uint8_t> p_bytes[2];
  DevBuf<uint64_t> p_offsets[2];
  DevBuf<int32_t> p_ids[2];
  DevBuf<unsigned long long> p_id_offsets[2];
  cudaStream_t s_h2d = nullptr, s_d2h = nullptr;
  cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_out[2] = {nullptr, nullptr}, ev_d2h[2] = {nullptr, nullptr};
  size_t pipeline_min_sentences = 300000, pipeline_chunk_sentences = 65536;
  DevBuf<uint32_t> d_order, d_order_hist;  // K0: length-bucketed processing order
  int build_order(const uint64_t *d_offs, size_t n, cudaStream_t st, const uint32_t **order, uint32_t seg);
  bool sort_by_length = true;
  DevBuf<unsigned long long> d_kstats;  // SPM_B200_KSTATS: in-kernel counters of the unigram lane kernel -> stderr
  bool kstats = false;
  // streamed host batches (encode_host_streamed): set around run_device calls
  const uint32_t *cur_ready = nullptr;
  unsigned long long cur_off_lo = 0, cur_off_hi = ~0ull;  // valid offset range of the batch run_device is given
  uint32_t cur_ready_base = 0, cur_piece_shift = 0;
  DevBuf<uint8_t> s_bytes;
  DevBuf<uint64_t> s_offsets;
  DevBuf<uint32_t> d_ready;
  PinBuf<uint32_t> h_marks;
  PinBuf<unsigned long long> h_progress;
  cudaEvent_t ev_offs = nullptr;
  int encode_host_streamed(const char *bytes, const uint64_t *offsets, size_t n, const int32_t **ids,
                           const uint64_t **id_offsets);
  int encode_host_fused(const char *bytes, const uint64_t *offsets, size_t n, const int32_t **ids, const uint64_t **id_offsets);
  bool fused_host_path = true;
  uint64_t fused_fallbacks = 0;
  int fused_skip = 0, fused_backoff = 8;
  DevBuf<uint32_t> d_seg_done, d_sent_rel;
  DevBuf<unsigned long long> d_seg_words;
  // Launch geometry of the lane kernels for an ids-only batch; ok == false: the model / tuning is outside the lane
  // kernels (the tile, warp or general BPE kernels take the batch).  Shared memory per warp grows with the longest
  // piece (ring of max piece length + 2 slots), so the warps per CTA shrink until the rings fit.
  struct LaneGeom {
    bool ok = false;
    int version = 1;       // BPE: 1 = encode_bpe_lane_kernel (sentence per lane), 2 = encode_bpe_lane2_kernel (word lists)
    int threads = 0;
    uint32_t R = 0, smem = 0;
  };
  // unigram: which instantiation takes the next batch -- the whole-word shortcut pays on text made of space-separated
  // words and only costs on text without them (CJK, mixed script).  Decided per call from a sample of the batch's bytes
  // (pick_fast_words); SPM_B200_FASTWORDS=0/1 forces it.
  bool batch_fast_words = true;
  int force_fast_words = -1;
  DevBuf<unsigned long long> d_sample;
  bool pick_fast_words_host(const char *bytes, const uint64_t *offsets, size_t n) const;
  int pick_fast_words_device(const uint8_t *d_bytes_base, const uint64_t *d_offs, size_t n, cudaStream_t st, bool *fast);
  bool any_user_defined = false;
  LaneGeom lane_geometry() const {
    LaneGeom g;
    if (G != 1) return g;
    const size_t avail = smem_optin > kLaneTableBytes ? smem_optin - kLaneTableBytes : 0;
    if (model.model_type == SPM_BPE) {
      if (!((km.flags & kFlagBpeWordSplit) && (km.flags & kFlagEscapeWs) && !(km.flags & (kFlagHasUserSymbols | kFlagHasUnused))))
        return g;
      g.version = bpe_lane_version == 2 ? 2 : 1;
      const size_t per_warp = g.version == 2 ? kBpeLane2WarpBytes : kBpeLaneWarpBytes;
      // (launch bounds: 704 threads for lane2 -- 22 warps is what the shared-memory arrays allow -- 768 for lane v1)
      const int warps = static_cast<int>(std::min<size_t>(std::min(threads, g.version == 2 ? 704 : 768) / 32, avail / per_warp));
      if (warps < 4) return g;
      g.ok = true;
      g.threads = warps * 32;
      g.smem = static_cast<uint32_t>(kLaneTableBytes + static_cast<size_t>(warps) * per_warp);
      return g;
    }
    if (trie.max_key_len > 62) return g;
    g.R = trie.max_key_len + 2;
    g.version = ((km.flags & kFlagFastWords) && batch_fast_words) ? 2 : 1;  // 2: whole-word shortcut, 1: plain
    const size_t ring = g.version == 2 ? lane_ring_bytes(g.R) : static_cast<size_t>(g.R) * 32 * 8;
    const int warps = static_cast<int>(std::min<size_t>(threads / 32, avail / ring));
    if (warps < 4) return g;
    g.ok = true;
    g.threads = warps * 32;
    g.smem = static_cast<uint32_t>(kLaneTableBytes + static_cast<size_t>(warps) * ring);
    return g;
  }
  bool uses_lane_kernel() const { return lane_geometry().ok; }
  // Decode (K7): per-id decoded strings, built on first use
  DevBuf<uint32_t> d_dec_off, d_dec_info;
  DevBuf<uint8_t> d_dec_bytes, d_dec_tmp, d_dec_text;
  DevBuf<int32_t> d_dec_ids;
  DevBuf<unsigned long long> d_dec_text_offsets;
  PinBuf<char> h_dec_text;
  PinBuf<uint64_t> h_dec_text_offsets;
  bool dec_ready = false;
  int ensure_decode_tables();
  // large host batches: chunked three-stage pipeline (staged H2D of the ids / decode kernels / D2H of the text)
  DevBuf<int32_t> p_dec_ids[2];
  DevBuf<uint8_t> p_dec_text[2];
  DevBuf<unsigned long long> p_dec_toff[2];
  PinBuf<uint8_t> h_stage[2];
  int decode_host_pipelined(const int32_t *ids, const uint64_t *id_offsets, size_t n, const char **text,
                            const uint64_t **text_offsets);
  // n-best / sampling
  DevBuf<uint8_t> d_nb_scratch;
  DevBuf<unsigned long long> d_cand_start, d_cand_offsets;
  DevBuf<uint32_t> d_cand_count, d_n_cands, d_picks;
  DevBuf<float> d_cand_score;
  PinBuf<float> h_cand_score;
  PinBuf<uint32_t> h_n_cands, h_picks;
  PinBuf<uint64_t> h_cand_offsets;
  std::mt19937 rng{5489u};
  // full-lattice operations (lattice_kernel.cuh): exported lattices of one chunk of sentences
  DevBuf<uint8_t> d_lat_scratch;
  DevBuf<uint4> d_lat_nodes;
  DevBuf<uint2> d_lat_pos;
  DevBuf<unsigned long long> d_lat_node_start, d_lat_pos_start;
  DevBuf<uint32_t> d_lat_nchars;
  DevBuf<float> d_lat_entropy;
  PinBuf<uint4> h_lat_nodes;
  PinBuf<uint2> h_lat_pos;
  PinBuf<unsigned long long> h_lat_node_start, h_lat_pos_start;
  PinBuf<uint32_t> h_lat_nchars;
  PinBuf<float> h_lat_entropy;
  std::vector<int32_t> byte_to_id_host;
  std::vector<int32_t> lat_ids;          // results of the last lattice sampling call
  std::vector<uint64_t> lat_offsets;
  std::vector<float> lat_scores;
  // mode 0: samples >= 1 draws per sentence from the lattice (ids, offsets[n*samples+1], scores); mode 1: entropy
  int run_lattice(const char *bytes, const uint64_t *offsets, size_t n, float inv_theta, int mode, int samples);
  int run_nbest(const char *bytes, const uint64_t *offsets, size_t n, uint32_t nbest, uint64_t *tmp_total);

  // stats of the last call
  uint64_t last_launches = 0, last_h2d = 0, last_d2h = 0, last_deferred = 0;
  float last_ms = 0.f, last_main_ms = 0.f;

  void set_error(const std::string &m) const { err = m; }
  int build_tables();
  int upload_types();
  int upload_node2();
  int configure_kernel_attrs();
  int run_device(const uint8_t *d_bytes_base, const uint64_t *d_offs, size_t n, uint64_t total_bytes, bool spans,
                 int32_t *user_ids, uint64_t user_ids_cap, unsigned long long *user_id_offsets, uint64_t *total_ids,
                 uint64_t *total_norm, cudaStream_t st, DevBuf<int32_t> *out_ids = nullptr,
                 DevBuf<unsigned long long> *out_offs = nullptr, unsigned long long off_base = 0);
  int encode_host_pipelined(const char *bytes, const uint64_t *offsets, size_t n, const int32_t **ids,
                            const uint64_t **id_offsets);
};

// ---------------------------------------------------------------- model ----

namespace {

// ModelInterface::PieceToId for byte pieces (model_interface.cc:51-61,210-212)
int32_t piece_to_id(const std::unordered_map<std::string, int32_t> &reserved,
                    const std::unordered_map<std::string, int32_t> &pieces, int32_t unk, const std::string &p) {
  auto it = reserved.find(p);
  if (it != reserved.end()) return it->second;
  auto it2 = pieces.find(p);
  if (it2 != pieces.end()) return it2->second;
  return unk;
}

}  // namespace

int spm_engine::build_tables() {
  ModelData &m = model;
  if (m.model_type != SPM_UNIGRAM && m.model_type != SPM_BPE) {
    set_error("only UNIGRAM and BPE models are on the accelerated path (model_factory.cc:25-48)");
    return SPM_ERR_UNSUPPORTED;
  }
  const int V = m.vocab_size();
  // ---- InitializePieces (model_interface.cc:63-151) ----
  std::unordered_map<std::string, int32_t> pieces, reserved;
  std::vector<bool> byte_found(256, false);
  unk_id = -1;
  for (int i = 0; i < V; ++i) {
    const std::string p(m.piece(i), m.piece_len(i));
    if (p.empty()) { set_error("piece must not be empty."); return SPM_ERR_MODEL; }
    const uint8_t t = m.types[i];
    const bool normal = t == SPM_NORMAL || t == SPM_USER_DEFINED || t == SPM_UNUSED;
    if (!(normal ? pieces : reserved).emplace(p, i).second) { set_error(p + " is already defined."); return SPM_ERR_MODEL; }
    if (t == SPM_UNKNOWN) {
      if (unk_id >= 0) { set_error("unk is already defined."); return SPM_ERR_MODEL; }
      unk_id = i;
    }
    if (t == SPM_BYTE) {
      if (!m.byte_fallback) { set_error("byte piece " + p + " is found although `byte_fallback` is false."); return SPM_ERR_MODEL; }
      int b = -1;
      if (p.size() == 6) {
        char canon[8];
        for (int v = 0; v < 256 && b < 0; ++v) {
          snprintf(canon, sizeof canon, "<0x%02X>", v);
          if (p == canon) b = v;
        }
      }
      if (b < 0) { set_error("byte piece " + p + " is invalid."); return SPM_ERR_MODEL; }
      byte_found[b] = true;
    }
  }
  if (unk_id < 0) { set_error("unk is not defined."); return SPM_ERR_MODEL; }
  if (m.byte_fallback && std::find(byte_found.begin(), byte_found.end(), false) != byte_found.end()) {
    set_error("there are not 256 byte pieces although `byte_fallback` is true.");
    return SPM_ERR_MODEL;
  }
  // ---- unigram::Model ctor (unigram_model.cc:657-664): max starts at FLT_MIN (quirk Q3) ----
  min_score = FLT_MAX;
  max_score = FLT_MIN;
  for (int i = 0; i < V; ++i)
    if (m.types[i] == SPM_NORMAL) {
      min_score = std::min(min_score, m.scores[i]);
      max_score = std::max(max_score, m.scores[i]);
    }
  // ---- piece trie over pieces_ (unigram_model.cc:608-650 / bpe pieces_.find) ----
  std::vector<TrieKey> keys, user_keys;
  bool ws_only_at_front = true;
  for (int i = 0; i < V; ++i) {
    const uint8_t t = m.types[i];
    if (!(t == SPM_NORMAL || t == SPM_USER_DEFINED || t == SPM_UNUSED)) continue;
    const float s = m.scores[i];
    const float w = m.model_type == SPM_UNIGRAM ? std::exp(s) : 1.0f / (1.0f + std::fabs(s));
    const uint32_t kind = t == SPM_NORMAL ? kKindNormal : (t == SPM_USER_DEFINED ? kKindUserDefined : kKindUnused);
    keys.push_back({m.piece(i), static_cast<uint32_t>(m.piece_len(i)), i, s, w, kind});
    if (t == SPM_USER_DEFINED) user_keys.push_back({m.piece(i), static_cast<uint32_t>(m.piece_len(i)), i, 0.f, 1.f, kKindNormal});
    if (!valid_utf8(m.piece(i), m.piece_len(i))) {
      set_error("pieces that are not valid UTF-8 are not supported by the device path");
      return SPM_ERR_UNSUPPORTED;
    }
    // U+2581 anywhere but at byte 0 defeats the per-word BPE decomposition
    const std::string p(m.piece(i), m.piece_len(i));
    if (p.find("\xE2\x96\x81", 1) != std::string::npos) ws_only_at_front = false;
  }
  bpe_word_split = ws_only_at_front;
  std::string e;
  if (!BuildDeviceTrie(keys, V, &trie, &e)) { set_error(e); return SPM_ERR_MODEL; }
  if (trie.max_key_len > 255) { set_error("pieces longer than 255 bytes are not supported by the device path"); return SPM_ERR_UNSUPPORTED; }
  if (!user_keys.empty() && !BuildDeviceTrie(user_keys, V, &user_trie, &e)) { set_error(e); return SPM_ERR_MODEL; }

  // ---- byte fallback ids (sentencepiece_processor.cc:587-588) ----
  std::vector<int32_t> byte_to_id(256, unk_id);
  for (int b = 0; b < 256; ++b) {
    char bp[8];
    snprintf(bp, sizeof bp, "<0x%02X>", b);
    byte_to_id[b] = piece_to_id(reserved, pieces, unk_id, bp);
  }

  // ---- precompiled charsmap (normalizer.cc:274-309) + fast-path tables ----
  std::vector<uint32_t> cm_units, cm_lead(8, 0), cm_pair(128 * 256 / 32, 0);
  std::vector<int32_t> cm_solo(128, -1);
  std::vector<uint8_t> cm_targets(1, 0);
  max_expand_num = m.escape_whitespaces ? 3 : 1;
  max_expand_den = 1;
  if (!m.charsmap.empty()) {
    const std::string &blob = m.charsmap;
    uint32_t trie_bytes = 0;
    if (blob.size() <= 4) { set_error("Blob for normalization rule is broken."); return SPM_ERR_MODEL; }
    memcpy(&trie_bytes, blob.data(), 4);
    if (trie_bytes >= blob.size() - 4 + 4 || trie_bytes + 4 > blob.size()) { set_error("Trie data size exceeds the input blob size."); return SPM_ERR_MODEL; }
    cm_units.resize(trie_bytes / 4);
    memcpy(cm_units.data(), blob.data() + 4, cm_units.size() * 4);
    cm_targets.assign(blob.begin() + 4 + trie_bytes, blob.end());
    cm_targets.push_back(0);  // the blob's last target is NUL-terminated already; be safe
    const size_t NU = cm_units.size();
    auto off = [](uint32_t u) { return (u >> 10) << ((u & (1u << 9)) >> 6); };
    auto label = [](uint32_t u) { return u & ((1u << 31) | 0xFFu); };
    if (NU == 0) { set_error("Blob for normalization rule is broken."); return SPM_ERR_MODEL; }
    // enumerate all keys by DFS over the double array: (node after the step, depth)
    struct Fr { uint32_t node; uint32_t depth; uint32_t first; };
    std::vector<Fr> stack;
    const uint32_t root_next = 0 ^ off(cm_units[0]);
    stack.push_back({root_next, 0, 256});
    while (!stack.empty()) {
      const Fr f = stack.back();
      stack.pop_back();
      for (uint32_t c = 0; c < 256; ++c) {
        const uint32_t node = f.node ^ c;
        if (node >= NU) continue;
        const uint32_t unit = cm_units[node];
        if (label(unit) != c) continue;
        const uint32_t first = f.depth == 0 ? c : f.first;
        if (f.depth == 0) cm_lead[c >> 5] |= 1u << (c & 31);
        if (f.depth == 1 && f.first < 128) cm_pair[(f.first * 256 + c) >> 5] |= 1u << (c & 31);
        const uint32_t nxt = node ^ off(unit);
        if ((unit >> 8) & 1u) {
          if (nxt >= NU) { set_error("charsmap trie is malformed"); return SPM_ERR_MODEL; }
          const uint32_t value = cm_units[nxt] & 0x7FFFFFFFu;
          if (value >= cm_targets.size()) { set_error("charsmap target offset out of range"); return SPM_ERR_MODEL; }
          const size_t tl = strlen(reinterpret_cast<const char *>(cm_targets.data()) + value);
          if (!valid_utf8(reinterpret_cast<const char *>(cm_targets.data()) + value, tl)) {
            set_error("charsmap targets that are not valid UTF-8 are not supported by the device path");
            return SPM_ERR_UNSUPPORTED;
          }
          if (f.depth == 0 && c < 128) cm_solo[c] = static_cast<int32_t>(value);
          // expansion: every target byte may be a space that escapes to 3 bytes
          size_t nsp = 0;
          for (size_t k = 0; k < tl; ++k) nsp += cm_targets[value + k] == ' ';
          const uint64_t out_bytes = tl + (m.escape_whitespaces ? 2 * nsp : 0);
          const uint64_t klen = f.depth + 1;
          if (out_bytes * max_expand_den > static_cast<uint64_t>(max_expand_num) * klen) {
            max_expand_num = static_cast<uint32_t>(out_bytes);
            max_expand_den = static_cast<uint32_t>(klen);
          }
        }
        if (f.depth < 64) stack.push_back({nxt, f.depth + 1, first});
      }
    }
  }
  // malformed bytes expand 1 -> 3 (U+FFFD)
  if (static_cast<uint64_t>(3) * max_expand_den > max_expand_num) { max_expand_num = 3; max_expand_den = 1; }
  charsmap_units = static_cast<uint32_t>(cm_units.size());

  // ---- upload ----
  if (cudaSetDevice(device) != cudaSuccess) { set_error("cudaSetDevice failed"); return SPM_ERR_CUDA; }
  CUDA_TRY(d_link.upload(trie.link));
  CUDA_TRY(d_val.upload(trie.val));
  CUDA_TRY(d_id.upload(trie.id));
  if (!user_trie.link.empty()) CUDA_TRY(d_user_link.upload(user_trie.link));
  if (cm_units.empty()) cm_units.push_back(0);
  CUDA_TRY(d_cm_units.upload(cm_units));
  CUDA_TRY(d_cm_targets.upload(cm_targets));
  CUDA_TRY(d_cm_lead.upload(cm_lead));
  CUDA_TRY(d_cm_pair.upload(cm_pair));
  CUDA_TRY(d_cm_solo.upload(cm_solo));
  CUDA_TRY(d_byte_to_id.upload(byte_to_id));
  byte_to_id_host = byte_to_id;
  CUDA_TRY(d_scores.upload(m.scores));
  CUDA_TRY(d_types.upload(m.types));

  { const int rc2 = upload_node2(); if (rc2) return rc2; }
  km.trie_link = d_link.p;
  km.trie_val = d_val.p;
  km.trie_id = d_id.p;
  km.trie_units = static_cast<uint32_t>(trie.link.size());
  km.match_slots = trie.max_matches_per_start + 1;
  km.user_link = d_user_link.p;
  km.cm_units = d_cm_units.p;
  km.cm_nunits = charsmap_units;
  km.cm_targets = d_cm_targets.p;
  km.cm_lead = d_cm_lead.p;
  km.cm_pair = d_cm_pair.p;
  km.cm_solo = d_cm_solo.p;
  km.byte_to_id = d_byte_to_id.p;
  km.scores = d_scores.p;
  km.types = d_types.p;
  km.unk_id = unk_id;
  km.unk_score = min_score - 10.0f;  // kUnkPenalty, unigram_model.cc:955
  km.max_score = max_score;
  km.model_type = m.model_type;
  km.flags = (m.add_dummy_prefix ? kFlagAddDummyPrefix : 0) | (m.remove_extra_whitespaces ? kFlagRemoveExtraWs : 0) |
             (m.escape_whitespaces ? kFlagEscapeWs : 0) | (m.treat_whitespace_as_suffix ? kFlagWsSuffix : 0) |
             (m.byte_fallback ? kFlagByteFallback : 0) | (!user_trie.link.empty() ? kFlagHasUserSymbols : 0) |
             (charsmap_units ? kFlagHasCharsmap : 0) | (bpe_word_split ? kFlagBpeWordSplit : 0);
  any_user_defined = false;
  for (uint8_t t : m.types) {
    if (t == SPM_UNUSED) km.flags |= kFlagHasUnused;
    if (t == SPM_USER_DEFINED) any_user_defined = true;
  }
  {
    bool regular = true;
    for (const TrieKey &k : keys) {
      const float a = std::fabs(k.score);
      if (!(k.score == 0.f || (a >= 0.0009765625f && a <= 1024.f))) regular = false;
    }
    if (regular) km.flags |= kFlagRegularScores;
  }
  return upload_word_safe();
}

// whole-word shortcut of the unigram lane kernel (lane_kernel.cuh): for every NORMAL piece P, seen as a word of its own, the largest
// normalized end position e up to which EncodeOptimized (unigram_model.cc:889-1020) is CERTAIN to encode the word
// as P alone, whatever precedes it.
//
// Setting: no piece contains U+2581 past byte 0 and whitespace is escaped, so a word [b, e) -- U+2581 (or the text
// start) up to the next U+2581 -- is only entered through position b and only left through e: the recurrence inside
// the word depends on the rest of the sentence through B = best_path_score[b] alone.  Let S_P be P's score and
// S_alt the best exact (real-number) score of any OTHER segmentation of the word into pieces / UNK edges, built
// with the reference's edge rules (has_single_node, UNUSED skipped, unk_score = min_score - 10).  The reference
// relaxes the whole-word edge first (start b is the earliest start of any edge into e), storing fl(S_P + B).  Every
// float it stores for a position inside the word is within (characters so far) roundings of B + (exact best), and
// every rounding is at most ulp(Vmax) with Vmax >= any |partial score| <= e * maxabs (at most one edge per byte,
// each of magnitude <= maxabs).  So a later candidate into e is at most B + S_alt + c * ulp(Vmax) and cannot
// exceed the stored value (>= B + S_P - ulp(Vmax)) when  S_P - S_alt > (c + 1) * ulp(Vmax).  The table stores the
// largest e for which that holds with a further factor of two of slack on both the margin and Vmax.
int spm_engine::upload_word_safe() {
  std::vector<uint16_t> safe(trie.link.size(), 0);
  const bool eligible = fast_words && model.model_type == SPM_UNIGRAM && bpe_word_split && model.escape_whitespaces &&
                        !model.treat_whitespace_as_suffix && !any_user_defined && trie.max_key_len <= 62;
  km.flags &= ~kFlagFastWords;
  if (eligible) {
    const int V = model.vocab_size();
    const double unk = static_cast<double>(min_score - 10.0f);
    double maxabs = std::fabs(unk);
    for (int i = 0; i < V; ++i)
      if (model.types[i] == SPM_NORMAL) maxabs = std::max(maxabs, static_cast<double>(std::fabs(model.scores[i])));
    maxabs = std::max(maxabs, 1e-3);
    const double kNegInf = -1e300;
    std::vector<double> E;
    for (int i = 0; i < V; ++i) {
      if (model.types[i] != SPM_NORMAL) continue;
      const uint32_t unit = trie.unit_of_id[i];
      if (unit == 0xFFFFFFFFu) continue;
      const unsigned char *p = reinterpret_cast<const unsigned char *>(model.piece(i));
      const uint32_t L = static_cast<uint32_t>(model.piece_len(i));
      E.assign(L + 1, kNegInf);
      E[0] = 0.0;
      uint32_t chars = 0;
      for (uint32_t st = 0; st < L;) {
        static const uint8_t kLen[16] = {1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 2, 2, 3, 4};  // OneCharLen, util.h:151-153
        const uint32_t mb = std::min<uint32_t>(kLen[p[st] >> 4], L - st);
        ++chars;
        if (E[st] > kNegInf) {
          bool has_single = false;
          uint32_t l = trie.link[0];
          for (uint32_t k = st; k < L; ++k) {
            const uint32_t v = (l >> kLinkBaseShift) ^ p[k];
            if (v >= trie.link.size() || (trie.link[v] & kLinkLabelMask) != p[k]) break;
            l = trie.link[v];
            const uint32_t kind = (l >> kLinkKindShift) & 3u;
            if (kind != kKindNormal && kind != kKindUserDefined) continue;
            const uint32_t len = k + 1 - st;
            if (len == mb) has_single = true;
            if (st == 0 && len == L) continue;  // the whole-word edge itself
            float sc;
            memcpy(&sc, &trie.val[v], 4);
            E[st + len] = std::max(E[st + len], E[st] + static_cast<double>(sc));
          }
          if (!has_single) E[st + mb] = std::max(E[st + mb], E[st] + unk);
        }
        st += mb;
      }
      const double margin = E[L] > kNegInf ? static_cast<double>(model.scores[i]) - E[L] : 1e300;
      if (!(margin > 0.0)) continue;
      // (chars + 1) * 2^(kk - 23) < margin / 2   with   Vmax < 2^(kk + 1)
      const double x = margin / (2.0 * (chars + 1));
      const int kk = std::min(40, std::ilogb(x) + 22);
      if (kk < -40) continue;
      const double vmax = std::ldexp(1.0, kk + 1) / (2.0 * maxabs);  // largest admissible e (Vmax = e * maxabs, 2x slack)
      const double e_max = std::floor(vmax) - 1.0;
      if (e_max >= L) safe[unit] = static_cast<uint16_t>(std::min(65535.0, e_max));
    }
    km.flags |= kFlagFastWords;
  }
  // BPE (bpe_lane2_kernel.cuh): word_fast[unit] = id of the piece when the reference's merge loop
  // (bpe_model.cc:38-203: best score, leftmost on ties; candidates are string members of pieces_) run on the piece's
  // own characters ends with the piece as its only symbol; such a word needs no merge loop on the device.
  std::vector<uint32_t> fastw(trie.link.size(), 0xFFFFFFFFu);
  if (model.model_type == SPM_BPE && bpe_word_split && model.escape_whitespaces && !any_user_defined &&
      !(km.flags & kFlagHasUnused)) {
    static const uint8_t kLen[16] = {1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 2, 2, 3, 4};
    auto find = [&](const unsigned char *p, uint32_t len) -> uint32_t {  // exact match: unit of the piece, or ~0
      uint32_t l = trie.link[0], v = 0xFFFFFFFFu;
      for (uint32_t k = 0; k < len; ++k) {
        v = (l >> kLinkBaseShift) ^ p[k];
        if (v >= trie.link.size() || (trie.link[v] & kLinkLabelMask) != p[k]) return 0xFFFFFFFFu;
        l = trie.link[v];
      }
      return ((l >> kLinkKindShift) & 3u) != kKindNone ? v : 0xFFFFFFFFu;
    };
    std::vector<std::pair<uint32_t, uint32_t>> sy;  // (start, length) of the live symbols
    for (int i = 0; i < model.vocab_size(); ++i) {
      const uint32_t unit = trie.unit_of_id[i];
      if (unit == 0xFFFFFFFFu) continue;
      const unsigned char *p = reinterpret_cast<const unsigned char *>(model.piece(i));
      const uint32_t L = static_cast<uint32_t>(model.piece_len(i));
      sy.clear();
      for (uint32_t st = 0; st < L;) {
        const uint32_t mb = std::min<uint32_t>(kLen[p[st] >> 4], L - st);
        sy.emplace_back(st, mb);
        st += mb;
      }
      while (sy.size() > 1) {
        int bi = -1;
        float best = 0.f;
        for (size_t j = 0; j + 1 < sy.size(); ++j) {
          const uint32_t u = find(p + sy[j].first, sy[j].second + sy[j + 1].second);
          if (u == 0xFFFFFFFFu) continue;
          float sc;
          memcpy(&sc, &trie.val[u], 4);
          if (bi < 0 || sc > best) { best = sc; bi = static_cast<int>(j); }
        }
        if (bi < 0) break;
        sy[bi].second += sy[bi + 1].second;
        sy.erase(sy.begin() + bi + 1);
      }
      if (sy.size() == 1) fastw[unit] = static_cast<uint32_t>(i);
    }
  }
  CUDA_TRY(cudaSetDevice(device));
  CUDA_TRY(d_word_safe.upload(safe));
  CUDA_TRY(d_word_fast.upload(fastw));
  km.word_safe = d_word_safe.p;
  km.word_fast = d_word_fast.p;
  // word cache of the BPE lane2 kernel: emptied whenever the tables change (the ids of a word are a function of the
  // vocabulary and the live piece types)
  km.bpe_cache = nullptr;
  km.bpe_cache_mask = 0;
  if (model.model_type == SPM_BPE && bpe_cache_log2 > 0) {
    const size_t entries = size_t{1} << bpe_cache_log2;
    CUDA_TRY(d_bpe_cache.ensure(entries * 4));
    CUDA_TRY(cudaMemset(d_bpe_cache.p, 0, entries * 64));
    CUDA_TRY(cudaDeviceSynchronize());
    km.bpe_cache = d_bpe_cache.p;
    km.bpe_cache_mask = static_cast<uint32_t>(entries - 1);
  }
  {
    std::vector<uint4> n4(trie.link.size());
    for (size_t u = 0; u < trie.link.size(); ++u) n4[u] = make_uint4(trie.link[u], trie.cmask[u], trie.val[u], safe[u]);
    CUDA_TRY(d_node4.upload(n4));
    km.trie_node4 = d_node4.p;
  }
  // Every walk of the unigram lane kernel from a U+2581 passes root -> E2 -> E2 96 -> U+2581.  When neither of the
  // first two nodes is a piece (E2 and E2 96 are not UTF-8, so only a malformed vocabulary has them) the walk skips
  // nothing by starting on the node of U+2581 with the piece "U+2581" relaxed, 3 bytes in (lane_kernel.cuh).
  km.ws_unit = kNoUnit;
  km.ws_link = km.ws_score = km.ws_safe = 0;
  if (km.flags & kFlagFastWords) {
    static const uint8_t kWs[3] = {0xE2, 0x96, 0x81};
    uint32_t l = trie.link[0], v = kNoUnit;
    for (int i = 0; i < 3; ++i) {
      v = (l >> kLinkBaseShift) ^ kWs[i];
      if (v >= trie.link.size() || (trie.link[v] & kLinkLabelMask) != kWs[i]) { v = kNoUnit; break; }
      l = trie.link[v];
      const uint32_t kind = (l >> kLinkKindShift) & 3u;
      if (i < 2 && (kind == kKindNormal || kind == kKindUserDefined)) { v = kNoUnit; break; }
    }
    if (v != kNoUnit) {
      km.ws_unit = v;
      km.ws_link = trie.link[v];
      km.ws_score = trie.val[v];
      km.ws_safe = safe[v];
    }
  }
  return SPM_OK;
}

// {link, child mask} pairs for the lane kernel.
int spm_engine::upload_node2() {
  std::vector<uint32_t> n2(trie.link.size() * 2);
  for (size_t u = 0; u < trie.link.size(); ++u) { n2[2 * u] = trie.link[u]; n2[2 * u + 1] = trie.cmask[u]; }
  CUDA_TRY(d_node2.upload(n2));
  km.trie_node2 = reinterpret_cast<const uint2 *>(d_node2.p);
  return SPM_OK;
}

// Live piece types -> trie link words (kind bits) + types array.
int spm_engine::upload_types() {
  for (int i = 0; i < model.vocab_size(); ++i) {
    const uint32_t u = trie.unit_of_id[i];
    if (u == 0xFFFFFFFFu) continue;
    const uint8_t t = model.types[i];
    const uint32_t kind = t == SPM_NORMAL ? kKindNormal : (t == SPM_USER_DEFINED ? kKindUserDefined : kKindUnused);
    trie.link[u] = (trie.link[u] & ~(3u << kLinkKindShift)) | (kind << kLinkKindShift);
  }
  bool any_unused = false;
  any_user_defined = false;
  for (uint8_t t : model.types) { any_unused |= t == SPM_UNUSED; any_user_defined |= t == SPM_USER_DEFINED; }
  km.flags = (km.flags & ~kFlagHasUnused) | (any_unused ? kFlagHasUnused : 0u);
  CUDA_TRY(cudaSetDevice(device));
  CUDA_TRY(d_link.upload(trie.link));
  CUDA_TRY(d_types.upload(model.types));
  { const int rc = upload_node2(); if (rc) return rc; }
  return upload_word_safe();
}

// -------------------------------------------------------------- launches ---

namespace {

struct LaunchGeom {
  uint32_t hot_link, hot_val, tile_bytes, smem_bytes, tiles;
};

// Shared memory split: tiles first (threads/G of them), the rest goes to the hot
// trie prefix (3:1 link:val, both multiples of 4 units for the 16-byte bulk copy).
LaunchGeom plan_geometry(const spm_engine &e, bool spans, int G, int threads, uint32_t ncap, uint32_t K) {
  LaunchGeom g{};
  g.tiles = static_cast<uint32_t>(threads / G);
  g.tile_bytes = tile_bytes_for(ncap, G, K, spans);
  const size_t budget = e.smem_optin / std::max(1, e.ctas_per_sm) - (e.ctas_per_sm > 1 ? 1024 : 0);
  const size_t fixed = 16 + static_cast<size_t>(g.tiles) * g.tile_bytes + 128;
  size_t hot = budget > fixed ? budget - fixed : 0;
  if (const char *lim = getenv("SPM_B200_HOT_LIMIT")) hot = std::min<size_t>(hot, strtoull(lim, nullptr, 10));  // experiments
  const uint32_t units = e.km.trie_units;
  uint32_t hl = static_cast<uint32_t>(std::min<size_t>(units, (hot * 3 / 4) / 4)) & ~3u;
  uint32_t hv = static_cast<uint32_t>(std::min<size_t>(units, (hot - static_cast<size_t>(hl) * 4) / 4)) & ~3u;
  // if the whole link array fits, give the remainder to val
  g.hot_link = hl;
  g.hot_val = hv;
  g.smem_bytes = static_cast<uint32_t>(16 + static_cast<size_t>(hl + hv) * 4 + static_cast<size_t>(g.tiles) * g.tile_bytes);
  return g;
}

template <typename KernelT>
cudaError_t set_smem(KernelT k, size_t bytes) {
  return cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bytes));
}

}  // namespace

int spm_engine::configure_kernel_attrs() {
  const size_t mx = smem_optin;
  CUDA_TRY(set_smem(encode_unigram_kernel<4, false>, mx));
  CUDA_TRY(set_smem(encode_unigram_kernel<8, false>, mx));
  CUDA_TRY(set_smem(encode_unigram_kernel<16, false>, mx));
  CUDA_TRY(set_smem(encode_unigram_kernel<32, false>, mx));
  CUDA_TRY(set_smem(encode_unigram_kernel<8, true>, mx));
  CUDA_TRY(set_smem(encode_unigram_kernel<32, true>, mx));
  CUDA_TRY(set_smem(encode_unigram_long_kernel<false>, mx));
  CUDA_TRY(set_smem(encode_unigram_long_kernel<true>, mx));
  CUDA_TRY(set_smem(encode_unigram_lane_kernel, mx));
  CUDA_TRY(set_smem(encode_unigram_lane_plain_kernel, mx));
  CUDA_TRY(set_smem(encode_bpe_lane_kernel, mx));
  CUDA_TRY(set_smem(encode_bpe_lane2_kernel, mx));
  CUDA_TRY(set_smem(nbest_lane_kernel<kNbestTop, 1024>, mx));
  CUDA_TRY(set_smem(lattice_lane_kernel, mx));
  CUDA_TRY(set_smem(encode_unigram_warp_kernel<512>, mx));
  CUDA_TRY(set_smem(encode_unigram_warp_kernel<1024>, mx));
  CUDA_TRY(set_smem(encode_bpe_kernel<false>, mx));
  CUDA_TRY(set_smem(encode_bpe_kernel<true>, mx));
  CUDA_TRY(set_smem(encode_bpe_long_kernel<false>, mx));
  CUDA_TRY(set_smem(encode_bpe_long_kernel<true>, mx));
  return SPM_OK;
}

// Which instantiation of the unigram lane kernel takes this batch: the whole-word shortcut wants text made of
// space-separated words.  A sample of the batch's bytes decides (one space per <= 16 bytes: words of <= 15 bytes on
// average); results never depend on the choice, only the speed does.
bool spm_engine::pick_fast_words_host(const char *bytes, const uint64_t *offsets, size_t n) const {
  if (force_fast_words >= 0) return force_fast_words != 0;
  if (!(km.flags & kFlagFastWords) || !bytes || n == 0) return true;
  const uint64_t lo = offsets[0], hi = offsets[n];
  if (hi <= lo + 64) return true;
  const uint64_t total = hi - lo, win = std::min<uint64_t>(total, 4096);
  uint64_t spaces = 0, seen = 0;
  for (int w = 0; w < 16; ++w) {
    const uint64_t start = lo + (total - win) * static_cast<uint64_t>(w) / 15;
    for (uint64_t k = 0; k < win; ++k) spaces += bytes[start + k] == ' ';
    seen += win;
  }
  return spaces * 16 >= seen;
}

int spm_engine::pick_fast_words_device(const uint8_t *d_bytes_base, const uint64_t *d_offs, size_t n, cudaStream_t st, bool *fast) {
  *fast = true;
  if (force_fast_words >= 0) { *fast = force_fast_words != 0; return SPM_OK; }
  if (!(km.flags & kFlagFastWords) || n == 0) return SPM_OK;
  CUDA_TRY(d_sample.ensure(2));
  CUDA_TRY(h_ctrl64.ensure(8));
  CUDA_TRY(cudaMemsetAsync(d_sample.p, 0, 2 * sizeof(unsigned long long), st));
  sample_spaces_kernel<<<16, 256, 0, st>>>(d_bytes_base, d_offs, static_cast<uint32_t>(n), d_sample.p);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpyAsync(h_ctrl64.p + 6, d_sample.p, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  const unsigned long long spaces = h_ctrl64.p[6], seen = h_ctrl64.p[7];
  *fast = seen < 64 || spaces * 16 >= seen;
  return SPM_OK;
}

// K0: sentence indices sorted by byte length, longest first, within segments of `seg` sentences (order_kernel.cuh;
// seg = 0: the whole batch is one segment); *order = null for tiny batches
int spm_engine::build_order(const uint64_t *d_offs, size_t n, cudaStream_t st, const uint32_t **order, uint32_t seg) {
  *order = nullptr;
  if (!sort_by_length || n <= 64) return SPM_OK;
  const uint32_t n32 = static_cast<uint32_t>(n);
  if (seg == 0 || seg > n32) seg = n32;
  const uint32_t segs = (n32 + seg - 1) / seg;
  CUDA_TRY(d_order.ensure(n));
  CUDA_TRY(d_order_hist.ensure(static_cast<size_t>(segs) * kOrderBuckets));
  CUDA_TRY(cudaMemsetAsync(d_order_hist.p, 0, static_cast<size_t>(segs) * kOrderBuckets * sizeof(uint32_t), st));
  const uint32_t per_block = kOrderThreads * kOrderPerThread;
  const dim3 grid((seg + per_block - 1) / per_block, segs);
  order_hist_kernel<<<grid, kOrderThreads, 0, st>>>(d_offs, n32, seg, d_order_hist.p);
  order_scan_kernel<<<segs, kOrderBuckets, 0, st>>>(d_order_hist.p);
  order_scatter_kernel<<<grid, kOrderThreads, 0, st>>>(d_offs, n32, seg, d_order_hist.p, d_order.p);
  CUDA_TRY(cudaGetLastError());
  last_launches += 3;
  *order = d_order.p;
  return SPM_OK;
}

// Encodes a device-resident batch.  Outputs: ids (+offsets) either into the
// engine's buffers (user_ids == nullptr) or the caller's.
int spm_engine::run_device(const uint8_t *d_bytes_base, const uint64_t *d_offs, size_t n, uint64_t total_bytes,
                           bool spans, int32_t *user_ids, uint64_t user_ids_cap, unsigned long long *user_id_offsets,
                           uint64_t *total_ids, uint64_t *total_norm, cudaStream_t st, DevBuf<int32_t> *out_ids,
                           DevBuf<unsigned long long> *out_offs, unsigned long long off_base) {
  last_launches = 0;
  last_deferred = 0;
  const uint32_t n32 = static_cast<uint32_t>(n);
  const bool bpe = model.model_type == SPM_BPE;
  const int tileG = (G == 4 || G == 8 || G == 16) ? G : 32;
  const int useG = bpe ? 32 : ((spans && tileG != 32) ? 8 : tileG);
  const int tile_threads = std::min(threads, 512);
  const uint32_t K = km.match_slots;
  LaunchGeom geom = plan_geometry(*this, spans, useG, tile_threads, ncap, K);
  // fast paths: sentence per lane (lane kernels), or warp per sentence with a register-resident Viterbi window
  const LaneGeom lg = spans ? LaneGeom{} : lane_geometry();
  const bool lane_path = !bpe && lg.ok;
  const bool bpe_lane_path = bpe && lg.ok;
  const bool warp_path = !bpe && !spans && trie.max_key_len <= 32 && G == 32;
  const int launch_threads = warp_path ? threads : tile_threads;
  if (bpe || warp_path) {
    // these kernels own a warp per sentence and their own scratch layout
    geom.tiles = launch_threads / 32;
    geom.tile_bytes = bpe ? bpe_tile_bytes(ncap, spans) : warp_bytes_for(ncap, K);
    const size_t fixed = 16 + static_cast<size_t>(geom.tiles) * geom.tile_bytes + 128;
    const size_t hot = smem_optin > fixed ? smem_optin - fixed : 0;
    geom.hot_link = static_cast<uint32_t>(std::min<size_t>(km.trie_units, (hot * 3 / 4) / 4)) & ~3u;
    geom.hot_val = static_cast<uint32_t>(std::min<size_t>(km.trie_units, (hot - static_cast<size_t>(geom.hot_link) * 4) / 4)) & ~3u;
    geom.smem_bytes = static_cast<uint32_t>(16 + static_cast<size_t>(geom.hot_link + geom.hot_val) * 4 +
                                            static_cast<size_t>(geom.tiles) * geom.tile_bytes);
  }
  if (lane_path || bpe_lane_path) {
    geom.tiles = lg.threads / 32;
    geom.tile_bytes = bpe ? (lg.version == 2 ? kBpeLane2WarpBytes : kBpeLaneWarpBytes)
                          : (lg.version == 2 ? lane_ring_bytes(lg.R) : lg.R * 32 * 8);
    geom.hot_link = geom.hot_val = 0;  // the lane kernels read the trie through L1: rings / word arrays get the shared memory
    geom.smem_bytes = lg.smem;
    const size_t warps_total = static_cast<size_t>(sm_count) * ctas_per_sm * geom.tiles;
    CUDA_TRY(d_lane_slabs.ensure(warps_total * lane_slab_bytes(lane_cap) + 256));
    if (bpe) CUDA_TRY(d_bpe_long.ensure(warps_total * bpe_long_bytes(lane_cap)));
  }
  if (geom.smem_bytes > smem_optin) { set_error("shared-memory geometry does not fit; lower smem_norm_cap"); return SPM_ERR_ARG; }
  KModel M = km;
  M.hot_link = geom.hot_link;
  M.hot_val = geom.hot_val;

  // capacities: ids <= normalized bytes; start with one id per input byte (+slack) and
  // retry with the exact requirement when a pathological batch overflows.
  unsigned long long tmp_cap = total_bytes + 4ull * n + 1024;
  unsigned long long norm_cap = spans ? (total_bytes * 2 + 8ull * n + 1024) : 0;
  CUDA_TRY(d_sent_start.ensure(n));
  CUDA_TRY(d_sent_count.ensure(n));
  CUDA_TRY(d_deferred.ensure(2 * n + 2));
  CUDA_TRY(d_ctrl32.ensure(16));
  CUDA_TRY(d_deferred2.ensure(2 * n + 2));
  CUDA_TRY(d_ctrl64.ensure(4));
  CUDA_TRY(h_ctrl32.ensure(16));
  CUDA_TRY(h_ctrl64.ensure(4));
  if (spans) {
    CUDA_TRY(d_norm_start.ensure(n));
    CUDA_TRY(d_norm_len.ensure(n));
  }

  const int grid = sm_count * ctas_per_sm;
  for (int attempt = 0; attempt < 3; ++attempt) {
    CUDA_TRY(d_tmp_ids.ensure(tmp_cap));
    if (spans) {
      CUDA_TRY(d_tmp_tok_end.ensure(tmp_cap));
      CUDA_TRY(d_tmp_norm.ensure(norm_cap));
      CUDA_TRY(d_tmp_n2o.ensure(norm_cap));
    }
    CUDA_TRY(cudaMemsetAsync(d_ctrl32.p, 0, 16 * sizeof(uint32_t), st));
    CUDA_TRY(cudaMemsetAsync(d_ctrl64.p, 0, 4 * sizeof(unsigned long long), st));
    KBatch B{};
    B.slab_l2 = slab_l2; B.slab_discard = slab_discard;
    B.bytes = d_bytes_base;
    B.offsets = d_offs;
    B.n = n32;
    B.off_lo = cur_off_lo;
    B.off_hi = cur_off_hi;
    B.tmp_ids = d_tmp_ids.p;
    B.tmp_tok_end = d_tmp_tok_end.p;
    B.tmp_cap = tmp_cap;
    B.cursor = d_ctrl64.p;
    B.sent_start = d_sent_start.p;
    B.sent_count = d_sent_count.p;
    B.tmp_norm = d_tmp_norm.p;
    B.tmp_n2o = d_tmp_n2o.p;
    B.tmp_norm_cap = norm_cap;
    B.norm_start = d_norm_start.p;
    B.norm_len = d_norm_len.p;
    B.work_counter = d_ctrl32.p + 4;
    B.deferred = d_deferred.p;
    B.status = d_ctrl32.p;
    B.ncap = ncap;
    B.tile_bytes = geom.tile_bytes;

    CUDA_TRY(cudaEventRecord(ev[0], st));
    if (kstats) {
      CUDA_TRY(d_kstats.ensure(16));
      CUDA_TRY(cudaMemsetAsync(d_kstats.p, 0, 16 * sizeof(unsigned long long), st));
      B.kstats = d_kstats.p;
    }
    if (lane_path || bpe_lane_path) {
      uint32_t seg = cur_ready ? (1u << cur_piece_shift) : 0u;
      if (const char *v = getenv("SPM_B200_SORT_SEG")) seg = static_cast<uint32_t>(atoi(v));  // experiment knob
      const int rc = build_order(d_offs, n, st, &B.order, seg);
      if (rc) return rc;
      B.ready = cur_ready;
      B.ready_base = cur_ready_base;
      B.piece_shift = cur_piece_shift;
    }
    if (bpe_lane_path && lg.version == 2) {
      encode_bpe_lane2_kernel<<<grid, lg.threads, geom.smem_bytes, st>>>(M, B, d_lane_slabs.p, lane_cap, d_bpe_long.p);
    } else if (bpe_lane_path) {
      encode_bpe_lane_kernel<<<grid, lg.threads, geom.smem_bytes, st>>>(M, B, d_lane_slabs.p, lane_cap);
    } else if (bpe) {
      if (spans) encode_bpe_kernel<true><<<grid, tile_threads, geom.smem_bytes, st>>>(M, B);
      else encode_bpe_kernel<false><<<grid, tile_threads, geom.smem_bytes, st>>>(M, B);
    } else if (lane_path && lg.version == 2) {
      encode_unigram_lane_kernel<<<grid, lg.threads, geom.smem_bytes, st>>>(M, B, d_lane_slabs.p, lane_cap, lg.R);
    } else if (lane_path) {
      encode_unigram_lane_plain_kernel<<<grid, lg.threads, geom.smem_bytes, st>>>(M, B, d_lane_slabs.p, lane_cap, lg.R);
    } else if (warp_path) {
      if (threads <= 512) encode_unigram_warp_kernel<512><<<grid, threads, geom.smem_bytes, st>>>(M, B);
      else encode_unigram_warp_kernel<1024><<<grid, threads, geom.smem_bytes, st>>>(M, B);
    } else if (spans) {
      if (useG == 32) encode_unigram_kernel<32, true><<<grid, tile_threads, geom.smem_bytes, st>>>(M, B);
      else encode_unigram_kernel<8, true><<<grid, tile_threads, geom.smem_bytes, st>>>(M, B);
    } else {
      switch (useG) {
        case 4: encode_unigram_kernel<4, false><<<grid, tile_threads, geom.smem_bytes, st>>>(M, B); break;
        case 8: encode_unigram_kernel<8, false><<<grid, tile_threads, geom.smem_bytes, st>>>(M, B); break;
        case 16: encode_unigram_kernel<16, false><<<grid, tile_threads, geom.smem_bytes, st>>>(M, B); break;
        default: encode_unigram_kernel<32, false><<<grid, tile_threads, geom.smem_bytes, st>>>(M, B); break;
      }
    }
    CUDA_TRY(cudaGetLastError());
    ++last_launches;
    CUDA_TRY(cudaEventRecord(ev[1], st));
    CUDA_TRY(cudaMemcpyAsync(h_ctrl32.p, d_ctrl32.p, 16 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(h_ctrl64.p, d_ctrl64.p, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (kstats) {
      unsigned long long ks[16];
      CUDA_TRY(cudaMemcpy(ks, d_kstats.p, sizeof ks, cudaMemcpyDeviceToHost));
      if (ks[12])
        fprintf(stderr, "[kstats] groups %llu: warp trips/group %.1f, lane trips/sentence %.1f (lane utilisation of K2 %.3f), starts/sentence "
                "%.1f (whole words %.1f), normalized bytes/sentence %.1f\n", ks[12], double(ks[8]) / ks[12], double(ks[9]) / n,
                double(ks[9]) / (32.0 * ks[8]), double(ks[10]) / n, double(ks[11]) / n, double(ks[13]) / n);
      if (ks[4]) {
        const double w = 1e-6 / (static_cast<double>(grid) * geom.tiles);
        fprintf(stderr, "[kstats] M cycles per warp (lane 0): group loop %.2f = K1 %.2f, K2 %.2f, K4 %.2f, rest %.2f\n", ks[4] * w,
                ks[5] * w, ks[6] * w, ks[7] * w, (ks[4] - ks[5] - ks[6] - ks[7]) * w);
      }
    }
    uint32_t n_def = h_ctrl32.p[0];
    const uint32_t *def_list = d_deferred.p;
    if (n_def && (lane_path || bpe_lane_path)) {
      // ---- second chance: the sentences a lane kernel could not take (long words, long
      //      sentences) go through the shared-memory warp kernels before the HBM-scratch path ----
      last_deferred = n_def;
      LaunchGeom g2{};
      g2.tiles = tile_threads / 32;
      g2.tile_bytes = bpe ? bpe_tile_bytes(ncap, false) : tile_bytes_for(ncap, 32, K, false);
      const size_t fixed2 = 16 + static_cast<size_t>(g2.tiles) * g2.tile_bytes + 128;
      const size_t hot2 = smem_optin > fixed2 ? smem_optin - fixed2 : 0;
      KModel M2 = km;
      M2.hot_link = static_cast<uint32_t>(std::min<size_t>(km.trie_units, (hot2 * 3 / 4) / 4)) & ~3u;
      M2.hot_val = static_cast<uint32_t>(std::min<size_t>(km.trie_units, (hot2 - static_cast<size_t>(M2.hot_link) * 4) / 4)) & ~3u;
      const uint32_t smem2 = static_cast<uint32_t>(16 + static_cast<size_t>(M2.hot_link + M2.hot_val) * 4 +
                                                   static_cast<size_t>(g2.tiles) * g2.tile_bytes);
      KBatch B2 = B;
      B2.sub_list = d_deferred.p;
      B2.sub_n = n_def;
      B2.deferred = d_deferred2.p;
      B2.status = d_ctrl32.p + 8;
      B2.work_counter = d_ctrl32.p + 12;
      B2.ncap = ncap;
      B2.tile_bytes = g2.tile_bytes;
      const int grid2 = static_cast<int>(std::min<uint32_t>(static_cast<uint32_t>(grid), (n_def + g2.tiles - 1) / g2.tiles));
      if (bpe) encode_bpe_kernel<false><<<grid2, tile_threads, smem2, st>>>(M2, B2);
      else encode_unigram_kernel<32, false><<<grid2, tile_threads, smem2, st>>>(M2, B2);
      CUDA_TRY(cudaGetLastError());
      ++last_launches;
      CUDA_TRY(cudaMemcpyAsync(h_ctrl32.p, d_ctrl32.p, 16 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
      CUDA_TRY(cudaMemcpyAsync(h_ctrl64.p, d_ctrl64.p, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
      CUDA_TRY(cudaStreamSynchronize(st));
      n_def = h_ctrl32.p[8];
      h_ctrl32.p[1] |= h_ctrl32.p[9];
      h_ctrl32.p[2] |= h_ctrl32.p[10];
      def_list = d_deferred2.p;
      M.hot_link = M2.hot_link;  // the long kernels stage the same hot prefix
      M.hot_val = M2.hot_val;
    }
    if (n_def) {
      // ---- long sentences: warp per sentence, scratch slab in HBM ----
      last_deferred = std::max<uint64_t>(last_deferred, n_def);
      CUDA_TRY(h_deferred.ensure(2 * static_cast<size_t>(n_def)));
      CUDA_TRY(cudaMemcpyAsync(h_deferred.p, def_list, 2ull * n_def * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
      // lengths of the deferred sentences whose normalized size is unknown
      std::vector<uint64_t> two(2);
      std::vector<unsigned long long> offs(n_def + 1, 0);
      CUDA_TRY(cudaStreamSynchronize(st));
      for (uint32_t k = 0; k < n_def; ++k) {
        uint32_t need = h_deferred.p[2 * k + 1];
        if (need == 0) {
          const uint32_t s = h_deferred.p[2 * k];
          CUDA_TRY(cudaMemcpy(two.data(), d_offs + s, 16, cudaMemcpyDeviceToHost));
          const uint64_t len = two[1] - two[0];
          const uint64_t bound = (len * max_expand_num + max_expand_den - 1) / max_expand_den + 8;
          if (bound > 0x7FFFFF00ull) { set_error("sentence too long for the device path"); return SPM_ERR_UNSUPPORTED; }
          need = static_cast<uint32_t>(bound);
        }
        need += 8;
        h_deferred.p[2 * k + 1] = need;
        const uint32_t lk = bpe ? 1 : K;
        const unsigned long long bytes = bpe ? bpe_tile_bytes(need, spans) : tile_bytes_for(need, 32, lk, spans);
        offs[k + 1] = offs[k] + ((bytes + 255ull) & ~255ull);
      }
      CUDA_TRY(d_long_scratch.ensure(offs[n_def] + 256));
      CUDA_TRY(d_long_list.ensure(2 * static_cast<size_t>(n_def)));
      CUDA_TRY(d_long_off.ensure(n_def + 1));
      CUDA_TRY(cudaMemcpyAsync(d_long_list.p, h_deferred.p, 2ull * n_def * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
      CUDA_TRY(cudaMemcpyAsync(d_long_off.p, offs.data(), (n_def + 1) * sizeof(unsigned long long), cudaMemcpyHostToDevice, st));
      B.long_list = d_long_list.p;
      B.long_n = n_def;
      B.long_scratch = d_long_scratch.p;
      B.long_scratch_off = d_long_off.p;
      const int lgrid = static_cast<int>(std::min<uint32_t>((n_def + 7) / 8, static_cast<uint32_t>(sm_count) * 4));
      const uint32_t lsmem = 16 + (M.hot_link + M.hot_val) * 4;
      if (bpe) {
        if (spans) encode_bpe_long_kernel<true><<<lgrid, 256, lsmem, st>>>(M, B);
        else encode_bpe_long_kernel<false><<<lgrid, 256, lsmem, st>>>(M, B);
      } else {
        if (spans) encode_unigram_long_kernel<true><<<lgrid, 256, lsmem, st>>>(M, B);
        else encode_unigram_long_kernel<false><<<lgrid, 256, lsmem, st>>>(M, B);
      }
      CUDA_TRY(cudaGetLastError());
      ++last_launches;
      CUDA_TRY(cudaMemcpyAsync(h_ctrl32.p, d_ctrl32.p, 16 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
      CUDA_TRY(cudaMemcpyAsync(h_ctrl64.p, d_ctrl64.p, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
      CUDA_TRY(cudaStreamSynchronize(st));
      h_ctrl32.p[1] |= h_ctrl32.p[9];
      h_ctrl32.p[2] |= h_ctrl32.p[10];
    }
    if (h_ctrl32.p[1]) {
      if (h_ctrl32.p[1] & 2u) set_error("encode failed: the host-to-device copy of a streamed batch made no progress for 3 s");
      else set_error("encode failed: internal consistency check (status " + std::to_string(h_ctrl32.p[1]) + ")");
      return SPM_ERR_ENCODE;
    }
    if (h_ctrl32.p[2]) {  // temporary buffers too small: cursors hold the exact requirement
      tmp_cap = h_ctrl64.p[0] + 1024;
      norm_cap = spans ? h_ctrl64.p[1] + 1024 : 0;
      continue;
    }
    break;
  }
  if (h_ctrl32.p[2]) { set_error("temporary buffer overflow persisted"); return SPM_ERR_CAPACITY; }
  // ---- offsets (exclusive scan) + compaction into sentence order ----
  const uint32_t nb = (n32 + kScanChunk - 1) / kScanChunk;
  CUDA_TRY(d_block_sums.ensure(nb + 1));
  scan_block_sums_kernel<<<nb, 256, 0, st>>>(d_sent_count.p, n32, d_block_sums.p, 0);
  scan_block_prefix_kernel<<<1, 1024, 0, st>>>(d_block_sums.p, nb, d_ctrl64.p + 2);
  CUDA_TRY(cudaMemcpyAsync(h_ctrl64.p, d_ctrl64.p, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  const unsigned long long tot = h_ctrl64.p[2];  // the cursor over-counts (chunked claims); the scan is exact
  *total_ids = tot;
  if (total_norm) *total_norm = spans ? h_ctrl64.p[1] : 0;
  int32_t *ids_out = user_ids;
  unsigned long long *off_out = user_id_offsets;
  if (!user_ids) {
    DevBuf<int32_t> &ib = out_ids ? *out_ids : d_ids;
    DevBuf<unsigned long long> &ob = out_offs ? *out_offs : d_id_offsets;
    CUDA_TRY(ib.ensure(tot + 1));
    CUDA_TRY(ob.ensure(n + 1));
    ids_out = ib.p;
    off_out = ob.p;
    user_ids_cap = ib.cap;
    if (spans) CUDA_TRY(d_tok_end.ensure(tot + 1));
  } else if (tot > user_ids_cap) {
    set_error("ids_capacity too small: need " + std::to_string(tot));
    return SPM_ERR_CAPACITY;
  }
  scan_write_gather_kernel<int32_t><<<nb, 256, 0, st>>>(d_sent_count.p, n32, d_block_sums.p, off_out, d_sent_start.p,
                                                        d_tmp_ids.p, ids_out,
                                                        spans ? d_tmp_tok_end.p : nullptr, spans ? d_tok_end.p : nullptr,
                                                        user_ids_cap, 0, off_base);
  last_launches += 3;
  if (spans) {
    const unsigned long long tn = h_ctrl64.p[1];  // sum(n_i + 1)
    CUDA_TRY(d_norm.ensure(tn + 1));
    CUDA_TRY(d_n2o.ensure(tn + 1));
    CUDA_TRY(d_norm_offsets.ensure(n + 1));
    CUDA_TRY(d_n2o_offsets.ensure(n + 1));
    scan_block_sums_kernel<<<nb, 256, 0, st>>>(d_norm_len.p, n32, d_block_sums.p, 0);
    scan_block_prefix_kernel<<<1, 1024, 0, st>>>(d_block_sums.p, nb, d_ctrl64.p + 3);
    scan_write_gather_kernel<uint8_t><<<nb, 256, 0, st>>>(d_norm_len.p, n32, d_block_sums.p, d_norm_offsets.p,
                                                          d_norm_start.p, d_tmp_norm.p, d_norm.p, nullptr, nullptr,
                                                          d_norm.cap, 0, 0ull);
    // norm_to_orig has n_i + 1 entries per sentence: block sums of (len + 1)
    scan_block_sums_kernel<<<nb, 256, 0, st>>>(d_norm_len.p, n32, d_block_sums.p, 1);
    scan_block_prefix_kernel<<<1, 1024, 0, st>>>(d_block_sums.p, nb, d_ctrl64.p + 3);
    scan_write_gather_kernel<uint32_t><<<nb, 256, 0, st>>>(d_norm_len.p, n32, d_block_sums.p, d_n2o_offsets.p,
                                                           d_norm_start.p, d_tmp_n2o.p, d_n2o.p, nullptr, nullptr,
                                                           d_n2o.cap, 1, 0ull);
    last_launches += 6;
  }
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaEventRecord(ev[2], st));
  return SPM_OK;
}

// Large host batches: chunked three-stage pipeline.  H2D of chunk c+1 and D2H of chunk c-1
// run on their own streams while chunk c is being encoded; inputs and outputs are double
// buffered, the temporary buffers are only ever touched by the (serial) compute stream.
int spm_engine::encode_host_pipelined(const char *bytes, const uint64_t *offsets, size_t n, const int32_t **ids,
                                      const uint64_t **id_offsets) {
  CUDA_TRY(cudaSetDevice(device));
  for (size_t i = 0; i < n; ++i)
    if (offsets[i + 1] < offsets[i]) { set_error("offsets must be non-decreasing"); return SPM_ERR_ARG; }
  if (!s_h2d) {
    CUDA_TRY(cudaStreamCreateWithFlags(&s_h2d, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&s_d2h, cudaStreamNonBlocking));
    for (int k = 0; k < 2; ++k) {
      CUDA_TRY(cudaEventCreateWithFlags(&ev_in[k], cudaEventDisableTiming));
      CUDA_TRY(cudaEventCreateWithFlags(&ev_out[k], cudaEventDisableTiming));
      CUDA_TRY(cudaEventCreateWithFlags(&ev_d2h[k], cudaEventDisableTiming));
    }
  }
  // one sentence group (32 sentences) per resident warp and chunk: a launch cannot finish faster than
  // one group, so smaller chunks would only add idle warps (measured: 8 x 131k chunks cost 9.2 ms of
  // kernels against 6.5 ms for one launch)
  const bool is_bpe = model.model_type == SPM_BPE;
  const LaneGeom lgw = lane_geometry();
  const size_t warps = static_cast<size_t>(sm_count) * ctas_per_sm * ((lgw.ok ? lgw.threads : std::min(threads, 512)) / 32);
  size_t groups_per_warp = is_bpe ? 2 : 1;
  if (const char *v = getenv("SPM_B200_CHUNK_GROUPS")) groups_per_warp = std::max(1, atoi(v));
  const bool trace = getenv("SPM_B200_TRACE") != nullptr;
  const auto t_begin = std::chrono::steady_clock::now();
  auto now_ms = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count(); };
  const size_t chunk = std::max<size_t>(pipeline_chunk_sentences, warps * 32 * groups_per_warp);
  const size_t C = (n + chunk - 1) / chunk;
  const uint64_t total_bytes = offsets[n] - offsets[0];
  CUDA_TRY(h_id_offsets.ensure(n + 1));
  // ids are not known in advance: start from the running average (or 1 id per 3 bytes) and grow
  CUDA_TRY(h_ids.ensure(std::max<size_t>(h_ids.cap, total_bytes / 3 + 2 * n + 4096)));
  uint64_t max_chunk_bytes = 0;
  for (size_t c = 0; c < C; ++c) {
    const size_t lo = c * chunk, hi = std::min(n, lo + chunk);
    max_chunk_bytes = std::max<uint64_t>(max_chunk_bytes, offsets[hi] - offsets[lo]);
  }
  for (int k = 0; k < 2; ++k) {
    CUDA_TRY(p_bytes[k].ensure(max_chunk_bytes + 64));
    CUDA_TRY(p_offsets[k].ensure(chunk + 1));
  }
  auto issue_h2d = [&](size_t c) -> int {
    const int k = static_cast<int>(c & 1);
    const size_t lo = c * chunk, hi = std::min(n, lo + chunk);
    if (c >= 2) CUDA_TRY(cudaStreamWaitEvent(s_h2d, ev_out[k], 0));  // the slot's previous chunk has been encoded
    const uint64_t nb = offsets[hi] - offsets[lo];
    if (nb) CUDA_TRY(cudaMemcpyAsync(p_bytes[k].p, bytes + offsets[lo], nb, cudaMemcpyHostToDevice, s_h2d));
    CUDA_TRY(cudaMemcpyAsync(p_offsets[k].p, offsets + lo, (hi - lo + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, s_h2d));
    CUDA_TRY(cudaEventRecord(ev_in[k], s_h2d));
    return SPM_OK;
  };
  uint64_t launches = 0, deferred = 0;
  float main_ms = 0.f, all_ms = 0.f;
  unsigned long long id_base = 0;
  if (trace) fprintf(stderr, "[trace] setup done at %.3f ms\n", now_ms());
  { const int rc = issue_h2d(0); if (rc) return rc; }
  for (size_t c = 0; c < C; ++c) {
    const int k = static_cast<int>(c & 1);
    const size_t lo = c * chunk, hi = std::min(n, lo + chunk);
    if (c + 1 < C) { const int rc = issue_h2d(c + 1); if (rc) return rc; }
    CUDA_TRY(cudaStreamWaitEvent(stream, ev_in[k], 0));
    if (c >= 2) CUDA_TRY(cudaStreamWaitEvent(stream, ev_d2h[k], 0));  // the slot's previous results have left the GPU
    uint64_t tot = 0;
    const int rc = run_device(p_bytes[k].p - offsets[lo], p_offsets[k].p, hi - lo, offsets[hi] - offsets[lo], false, nullptr, 0,
                              nullptr, &tot, nullptr, stream, &p_ids[k], &p_id_offsets[k], id_base);
    if (rc) { cudaDeviceSynchronize(); return rc; }
    const double t_ret = trace ? now_ms() : 0.0;
    CUDA_TRY(cudaEventRecord(ev_out[k], stream));
    launches += last_launches;
    deferred += last_deferred;
    if (id_base + tot + 1 > h_ids.cap) {  // grow the pinned result buffer (rare): keep what has already arrived
      CUDA_TRY(cudaStreamSynchronize(s_d2h));
      PinBuf<int32_t> bigger;
      const double per_sent = static_cast<double>(id_base + tot) / static_cast<double>(hi);
      CUDA_TRY(bigger.ensure(static_cast<size_t>(per_sent * 1.25 * n) + tot + 4096));
      if (id_base) memcpy(bigger.p, h_ids.p, id_base * sizeof(int32_t));
      h_ids.release();
      h_ids = bigger;
    }
    CUDA_TRY(cudaStreamWaitEvent(s_d2h, ev_out[k], 0));
    if (tot) CUDA_TRY(cudaMemcpyAsync(h_ids.p + id_base, p_ids[k].p, tot * sizeof(int32_t), cudaMemcpyDeviceToHost, s_d2h));
    CUDA_TRY(cudaMemcpyAsync(h_id_offsets.p + lo, p_id_offsets[k].p, (hi - lo + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, s_d2h));
    CUDA_TRY(cudaEventRecord(ev_d2h[k], s_d2h));
    float a = 0.f;
    if (cudaEventElapsedTime(&a, ev[0], ev[1]) == cudaSuccess) { main_ms += a; all_ms += a; }
    if (trace) fprintf(stderr, "[trace] chunk %zu: run_device returned at %.3f ms (encode kernel %.3f ms), D2H issued at %.3f ms\n", c,
                       t_ret, a, now_ms());
    id_base += tot;
  }
  if (trace) fprintf(stderr, "[trace] all chunks issued at %.3f ms\n", now_ms());
  CUDA_TRY(cudaStreamSynchronize(s_d2h));
  if (trace) fprintf(stderr, "[trace] results on host at %.3f ms (%zu chunks of %zu)\n", now_ms(), C, chunk);
  last_launches = launches;
  last_deferred = deferred;
  last_main_ms = main_ms;
  last_ms = all_ms;
  last_h2d = total_bytes + (n + C) * sizeof(uint64_t);
  last_d2h = id_base * sizeof(int32_t) + (n + C) * sizeof(uint64_t);
  *ids = h_ids.p;
  *id_offsets = h_id_offsets.p;
  return SPM_OK;
}

// Large host batches through the lane kernels: streamed input.  Every H2D copy of the batch is queued up front in
// pieces of 32k sentences, each followed by a 4-byte copy that advances a device-side watermark; the encode kernels
// cover a few large chunks (>= 2 sentence groups per resident warp, so that the length-ordered dynamic schedule can
// balance them) and their warps wait on the watermark for the piece that holds their group.  The kernel of a chunk
// therefore starts as soon as its first piece has landed instead of after the whole chunk, and the D2H of chunk c
// overlaps the encode of chunk c + 1.
int spm_engine::encode_host_streamed(const char *bytes, const uint64_t *offsets, size_t n, const int32_t **ids,
                                     const uint64_t **id_offsets) {
  CUDA_TRY(cudaSetDevice(device));
  if (!s_h2d) {
    CUDA_TRY(cudaStreamCreateWithFlags(&s_h2d, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&s_d2h, cudaStreamNonBlocking));
    for (int k = 0; k < 2; ++k) {
      CUDA_TRY(cudaEventCreateWithFlags(&ev_in[k], cudaEventDisableTiming));
      CUDA_TRY(cudaEventCreateWithFlags(&ev_out[k], cudaEventDisableTiming));
      CUDA_TRY(cudaEventCreateWithFlags(&ev_d2h[k], cudaEventDisableTiming));
    }
  }
  if (!ev_offs) CUDA_TRY(cudaEventCreateWithFlags(&ev_offs, cudaEventDisableTiming));
  const bool trace = getenv("SPM_B200_TRACE") != nullptr;
  const auto t_begin = std::chrono::steady_clock::now();
  auto now_ms = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count(); };
  constexpr uint32_t kPieceShift = 15;
  constexpr size_t kPiece = size_t{1} << kPieceShift;
  const size_t P = (n + kPiece - 1) / kPiece;
  const bool is_bpe = model.model_type == SPM_BPE;
  const LaneGeom lgw = lane_geometry();
  const size_t warps = static_cast<size_t>(sm_count) * ctas_per_sm * ((lgw.ok ? lgw.threads : std::min(threads, 512)) / 32);
  size_t groups_per_warp = is_bpe ? 4 : 2;
  if (const char *v = getenv("SPM_B200_CHUNK_GROUPS")) groups_per_warp = std::max(1, atoi(v));
  const size_t min_chunk = std::max<size_t>(kPiece, warps * 32 * groups_per_warp);
  const size_t want_chunks = std::max<size_t>(1, n / min_chunk);
  const size_t chunk = ((P + want_chunks - 1) / want_chunks) * kPiece;
  const size_t C = (n + chunk - 1) / chunk;
  const uint64_t total_bytes = offsets[n] - offsets[0];
  CUDA_TRY(s_bytes.ensure(total_bytes + 64));
  CUDA_TRY(s_offsets.ensure(n + 1));
  CUDA_TRY(d_ready.ensure(4));
  CUDA_TRY(h_marks.ensure(P + 1));
  CUDA_TRY(h_id_offsets.ensure(n + 1));
  CUDA_TRY(h_ids.ensure(std::max<size_t>(h_ids.cap, total_bytes / 3 + 2 * n + 4096)));
  // ---- queue the whole input ----
  CUDA_TRY(cudaMemsetAsync(d_ready.p, 0, sizeof(uint32_t), s_h2d));
  CUDA_TRY(cudaMemcpyAsync(s_offsets.p, offsets, (n + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, s_h2d));
  CUDA_TRY(cudaEventRecord(ev_offs, s_h2d));
  {
    uint64_t bad = 0;  // checked while the offsets are on their way
    for (size_t i = 0; i < n; ++i) bad |= static_cast<uint64_t>(offsets[i + 1] < offsets[i]);
    if (bad) {
      cudaStreamSynchronize(s_h2d);
      set_error("offsets must be non-decreasing");
      return SPM_ERR_ARG;
    }
  }
  // The copies are issued by a helper thread so that the first encode kernel is launched right away.  Cuts between
  // the copies sit on 128-byte lines of the device buffer (ByteStream in lane_kernel.cuh over-reads within a line).
  std::atomic<int> feed_rc{0};
  std::thread feeder([&]() {
    if (cudaSetDevice(device) != cudaSuccess) { feed_rc = 1; return; }
    uint64_t done_bytes = 0;
    for (size_t p = 0; p < P; ++p) {
      const size_t hi = std::min(n, (p + 1) * kPiece);
      uint64_t cut = offsets[hi] - offsets[0];
      cut = hi == n ? total_bytes : std::min<uint64_t>(total_bytes, (cut + 127u) & ~uint64_t{127});
      if (cut > done_bytes &&
          cudaMemcpyAsync(s_bytes.p + done_bytes, bytes + offsets[0] + done_bytes, cut - done_bytes, cudaMemcpyHostToDevice,
                          s_h2d) != cudaSuccess) { feed_rc = 1; return; }
      done_bytes = std::max(done_bytes, cut);
      h_marks.p[p] = static_cast<uint32_t>(hi);
      if (cudaMemcpyAsync(d_ready.p, h_marks.p + p, sizeof(uint32_t), cudaMemcpyHostToDevice, s_h2d) != cudaSuccess) {
        feed_rc = 1;
        return;
      }
    }
  });
  struct Joiner { std::thread &t; ~Joiner() { if (t.joinable()) t.join(); } } joiner{feeder};
  CUDA_TRY(cudaStreamWaitEvent(stream, ev_offs, 0));
  uint64_t launches = 0, deferred = 0;
  float main_ms = 0.f, all_ms = 0.f;
  unsigned long long id_base = 0;
  for (size_t c = 0; c < C; ++c) {
    const int k = static_cast<int>(c & 1);
    const size_t lo = c * chunk, hi = std::min(n, lo + chunk);
    if (c >= 2) CUDA_TRY(cudaStreamWaitEvent(stream, ev_d2h[k], 0));  // the slot's previous results have left the GPU
    uint64_t tot = 0;
    cur_ready = d_ready.p;
    cur_ready_base = static_cast<uint32_t>(lo);
    cur_piece_shift = kPieceShift;
    const int rc = run_device(s_bytes.p - offsets[0], s_offsets.p + lo, hi - lo, offsets[hi] - offsets[lo], false, nullptr, 0,
                              nullptr, &tot, nullptr, stream, &p_ids[k], &p_id_offsets[k], id_base);
    cur_ready = nullptr;
    if (rc) { cudaDeviceSynchronize(); return rc; }
    const double t_ret = trace ? now_ms() : 0.0;
    CUDA_TRY(cudaEventRecord(ev_out[k], stream));
    launches += last_launches;
    deferred += last_deferred;
    if (id_base + tot + 1 > h_ids.cap) {  // grow the pinned result buffer (rare): keep what has already arrived
      CUDA_TRY(cudaStreamSynchronize(s_d2h));
      PinBuf<int32_t> bigger;
      const double per_sent = static_cast<double>(id_base + tot) / static_cast<double>(hi);
      CUDA_TRY(bigger.ensure(static_cast<size_t>(per_sent * 1.25 * n) + tot + 4096));
      if (id_base) memcpy(bigger.p, h_ids.p, id_base * sizeof(int32_t));
      h_ids.release();
      h_ids = bigger;
    }
    CUDA_TRY(cudaStreamWaitEvent(s_d2h, ev_out[k], 0));
    if (tot) CUDA_TRY(cudaMemcpyAsync(h_ids.p + id_base, p_ids[k].p, tot * sizeof(int32_t), cudaMemcpyDeviceToHost, s_d2h));
    CUDA_TRY(cudaMemcpyAsync(h_id_offsets.p + lo, p_id_offsets[k].p, (hi - lo + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, s_d2h));
    CUDA_TRY(cudaEventRecord(ev_d2h[k], s_d2h));
    float a = 0.f;
    if (cudaEventElapsedTime(&a, ev[0], ev[1]) == cudaSuccess) { main_ms += a; all_ms += a; }
    if (trace) fprintf(stderr, "[trace] chunk %zu (%zu sentences): run_device returned at %.3f ms (encode kernel %.3f ms)\n", c,
                       hi - lo, t_ret, a);
    id_base += tot;
  }
  feeder.join();
  if (feed_rc) { cudaDeviceSynchronize(); set_error("host-to-device copy of a streamed batch failed"); return SPM_ERR_CUDA; }
  CUDA_TRY(cudaStreamSynchronize(s_d2h));
  if (trace) fprintf(stderr, "[trace] results on host at %.3f ms\n", now_ms());
  last_launches = launches;
  last_deferred = deferred;
  last_main_ms = main_ms;
  last_ms = all_ms;
  last_h2d = total_bytes + (n + 1) * sizeof(uint64_t) + P * sizeof(uint32_t);
  last_d2h = id_base * sizeof(int32_t) + (n + C) * sizeof(uint64_t);
  *ids = h_ids.p;
  *id_offsets = h_id_offsets.p;
  return SPM_OK;
}

// Large host batches, fused: ONE launch of a lane kernel for the whole batch.  Input streams in as in
// encode_host_streamed; the results are compacted segment by segment inside the kernel (drain.cuh) straight into the
// pinned host buffers, so the transfer of the ids overlaps the encode and nothing is left to do after the kernel but
// read the status words.  Batches the kernel cannot finish on its own (a sentence deferred to the long path, result
// buffer too small) are redone through encode_host_streamed.
int spm_engine::encode_host_fused(const char *bytes, const uint64_t *offsets, size_t n, const int32_t **ids,
                                  const uint64_t **id_offsets) {
  CUDA_TRY(cudaSetDevice(device));
  if (!s_h2d) {
    CUDA_TRY(cudaStreamCreateWithFlags(&s_h2d, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&s_d2h, cudaStreamNonBlocking));
    for (int k = 0; k < 2; ++k) {
      CUDA_TRY(cudaEventCreateWithFlags(&ev_in[k], cudaEventDisableTiming));
      CUDA_TRY(cudaEventCreateWithFlags(&ev_out[k], cudaEventDisableTiming));
      CUDA_TRY(cudaEventCreateWithFlags(&ev_d2h[k], cudaEventDisableTiming));
    }
  }
  if (!ev_offs) CUDA_TRY(cudaEventCreateWithFlags(&ev_offs, cudaEventDisableTiming));
  const bool trace = getenv("SPM_B200_TRACE") != nullptr;
  const auto t_begin = std::chrono::steady_clock::now();
  auto now_ms = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count(); };
  uint32_t kPieceShift = 15;
  uint32_t kSegShift = 10;
  if (const char *v = getenv("SPM_B200_SEG_SHIFT")) kSegShift = std::min<uint32_t>(kPieceShift, std::max(8, atoi(v)));  // experiment knob
  if (const char *v = getenv("SPM_B200_PIECE_SHIFT")) kPieceShift = std::min(20, std::max(10, atoi(v)));
  // experiment knobs (profiles/README.md, "fused path: what the kernel loses against the device-resident one"): bit 0 no
  // D2H copies while the kernel runs, bit 1 id_offsets to device memory + one copy at the end, bit 2 the whole input is
  // staged before the launch, bit 3 input order instead of the segment-sorted one.  All give correct results.
  int fx = 0;
  if (const char *v = getenv("SPM_B200_FUSED_X")) fx = atoi(v);
  const size_t kPiece = size_t{1} << kPieceShift;
  const size_t P = (n + kPiece - 1) / kPiece;
  const size_t S = (n + (size_t{1} << kSegShift) - 1) >> kSegShift;
  const uint32_t n32 = static_cast<uint32_t>(n);
  const bool bpe = model.model_type == SPM_BPE;
  const uint64_t total_bytes = offsets[n] - offsets[0];
  cudaStream_t st = stream;
  // ---- buffers ----
  CUDA_TRY(s_bytes.ensure(total_bytes + 64));
  CUDA_TRY(s_offsets.ensure(n + 1));
  CUDA_TRY(d_ready.ensure(4));
  CUDA_TRY(h_marks.ensure(P + 1));
  CUDA_TRY(h_id_offsets.ensure(n + 1));
  CUDA_TRY(h_ids.ensure(std::max<size_t>(h_ids.cap, total_bytes / 2 + 2 * n + 4096)));
  const unsigned long long tmp_cap = total_bytes + 4ull * n + 1024;
  CUDA_TRY(d_tmp_ids.ensure(tmp_cap));
  CUDA_TRY(d_sent_start.ensure(n));
  CUDA_TRY(d_sent_count.ensure(n));
  CUDA_TRY(d_sent_rel.ensure(n));
  CUDA_TRY(d_deferred.ensure(2 * n + 2));
  CUDA_TRY(d_ctrl32.ensure(16));
  CUDA_TRY(d_ctrl64.ensure(16));
  CUDA_TRY(h_ctrl32.ensure(16));
  CUDA_TRY(h_ctrl64.ensure(16));
  CUDA_TRY(d_seg_done.ensure(2 * S + 4));   // groups finished [S], copied flags [S], drained counter
  CUDA_TRY(d_seg_words.ensure(2 * S));
  CUDA_TRY(d_ids.ensure(h_ids.cap));
  CUDA_TRY(h_progress.ensure(8));
  *reinterpret_cast<volatile unsigned long long *>(h_progress.p) = 0;
  // ---- launch geometry of the lane kernels (as in run_device) ----
  const LaneGeom lg = lane_geometry();
  if (!lg.ok) { set_error("fused path: the model is outside the lane kernels"); return SPM_ERR_ARG; }
  const int lane_threads = lg.threads;
  const uint32_t smem = lg.smem;
  const int grid = sm_count * ctas_per_sm;
  CUDA_TRY(d_lane_slabs.ensure(static_cast<size_t>(grid) * (lane_threads / 32) * lane_slab_bytes(lane_cap) + 256));
  if (bpe) CUDA_TRY(d_bpe_long.ensure(static_cast<size_t>(grid) * (lane_threads / 32) * bpe_long_bytes(lane_cap)));
  // ---- queue the whole input ----
  CUDA_TRY(cudaMemsetAsync(d_ready.p, 0, sizeof(uint32_t), s_h2d));
  CUDA_TRY(cudaMemcpyAsync(s_offsets.p, offsets, (n + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, s_h2d));
  CUDA_TRY(cudaEventRecord(ev_offs, s_h2d));
  if (offsets[n] < offsets[0]) { cudaStreamSynchronize(s_h2d); set_error("offsets must be non-decreasing"); return SPM_ERR_ARG; }
  std::atomic<int> feed_rc{0};
  std::thread feeder([&]() {
    if (cudaSetDevice(device) != cudaSuccess) { feed_rc = 1; return; }
    uint64_t done_bytes = 0;
    for (size_t p = 0; p < P; ++p) {
      const size_t hi = std::min(n, (p + 1) * kPiece);
      uint64_t cut = offsets[hi] - offsets[0];
      cut = hi == n ? total_bytes : std::min<uint64_t>(total_bytes, (cut + 127u) & ~uint64_t{127});
      if (cut > done_bytes &&
          cudaMemcpyAsync(s_bytes.p + done_bytes, bytes + offsets[0] + done_bytes, cut - done_bytes, cudaMemcpyHostToDevice,
                          s_h2d) != cudaSuccess) { feed_rc = 1; return; }
      done_bytes = std::max(done_bytes, cut);
      h_marks.p[p] = static_cast<uint32_t>(hi);
      if (cudaMemcpyAsync(d_ready.p, h_marks.p + p, sizeof(uint32_t), cudaMemcpyHostToDevice, s_h2d) != cudaSuccess) {
        feed_rc = 1;
        return;
      }
    }
  });
  struct Joiner { std::thread &t; ~Joiner() { if (t.joinable()) t.join(); } } joiner{feeder};
  if (fx & 4) { feeder.join(); CUDA_TRY(cudaStreamSynchronize(s_h2d)); }
  // ---- one launch ----
  last_launches = 0;
  last_deferred = 0;
  CUDA_TRY(cudaStreamWaitEvent(st, ev_offs, 0));
  CUDA_TRY(cudaMemsetAsync(d_ctrl32.p, 0, 16 * sizeof(uint32_t), st));
  CUDA_TRY(cudaMemsetAsync(d_ctrl64.p, 0, 16 * sizeof(unsigned long long), st));
  CUDA_TRY(cudaMemsetAsync(d_seg_done.p, 0, (2 * S + 4) * sizeof(uint32_t), st));
  CUDA_TRY(cudaMemsetAsync(d_seg_words.p, 0, 2 * S * sizeof(unsigned long long), st));
  KModel M = km;
  M.hot_link = M.hot_val = 0;
  KBatch B{};
  B.slab_l2 = slab_l2; B.slab_discard = slab_discard;
  B.bytes = s_bytes.p - offsets[0];
  B.offsets = s_offsets.p;
  B.n = n32;
  B.off_lo = offsets[0];
  B.off_hi = offsets[n];
  B.tmp_ids = d_tmp_ids.p;
  B.tmp_cap = tmp_cap;
  B.cursor = d_ctrl64.p;
  B.sent_start = d_sent_start.p;
  B.sent_count = d_sent_count.p;
  B.work_counter = d_ctrl32.p + 4;
  B.deferred = d_deferred.p;
  B.status = d_ctrl32.p;
  B.ready = d_ready.p;
  B.ready_base = 0;
  B.piece_shift = kPieceShift;
  B.seg_shift = kSegShift;
  B.seg_done = d_seg_done.p;
  B.seg_total = d_seg_words.p;
  B.seg_prefix = d_seg_words.p + S;
  B.sent_rel = d_sent_rel.p;
  {
    void *dp = nullptr;
    CUDA_TRY(cudaHostGetDevicePointer(&dp, h_id_offsets.p, 0));
    B.out_offsets = static_cast<unsigned long long *>(dp);
    if (fx & 2) { CUDA_TRY(d_id_offsets.ensure(n + 1)); B.out_offsets = d_id_offsets.p; }
    CUDA_TRY(cudaHostGetDevicePointer(&dp, h_progress.p, 0));
    B.host_progress = static_cast<unsigned long long *>(dp);
  }
  B.out_ids = d_ids.p;
  B.seg_copied = d_seg_done.p + S;
  B.drained_upto = d_seg_done.p + 2 * S;
  B.out_cap = std::min<unsigned long long>(h_ids.cap, d_ids.cap);
  B.out_off_base = 0;
  B.kstats = trace ? d_ctrl64.p + 4 : nullptr;
  CUDA_TRY(cudaEventRecord(ev[0], st));
  // processing order: sorted within blocks of 2^sort_shift sentences (drain segment <= block <= input piece); the
  // completion of a drain segment is counted per sentence (drain.cuh), so the two granularities are independent.
  // Measured (profiles/README.md): sorting whole pieces makes all 32 segments of a piece finish in the same last few
  // groups, whose warps then compact them one after the other -- e2e 192 -> 81 M sentences/s; the default stays at
  // the segment size.
  uint32_t sort_shift = kSegShift;
  if (const char *v = getenv("SPM_B200_SORT_SHIFT")) sort_shift = std::min<uint32_t>(kPieceShift, std::max<uint32_t>(kSegShift, atoi(v)));
  const bool fused_sort = !(fx & 8);  // bit 3: input order (completion is counted per sentence: any order drains)
  if (fused_sort) {
    const int rc = build_order(s_offsets.p, n, st, &B.order, 1u << sort_shift);
    if (rc) return rc;
    if (!B.order) { set_error("fused path needs the segment order"); return SPM_ERR_ARG; }
  }
  if (bpe && lg.version == 2) encode_bpe_lane2_kernel<<<grid, lane_threads, smem, st>>>(M, B, d_lane_slabs.p, lane_cap, d_bpe_long.p);
  else if (bpe) encode_bpe_lane_kernel<<<grid, lane_threads, smem, st>>>(M, B, d_lane_slabs.p, lane_cap);
  else if (lg.version == 2) encode_unigram_lane_kernel<<<grid, lane_threads, smem, st>>>(M, B, d_lane_slabs.p, lane_cap, lg.R);
  else encode_unigram_lane_plain_kernel<<<grid, lane_threads, smem, st>>>(M, B, d_lane_slabs.p, lane_cap, lg.R);
  CUDA_TRY(cudaGetLastError());
  ++last_launches;
  CUDA_TRY(cudaEventRecord(ev[1], st));
  CUDA_TRY(cudaEventRecord(ev[2], st));
  CUDA_TRY(cudaMemcpyAsync(h_ctrl32.p, d_ctrl32.p, 16 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  if (trace) CUDA_TRY(cudaMemcpyAsync(h_ctrl64.p, d_ctrl64.p, 16 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
  if (trace) fprintf(stderr, "[trace] fused kernel launched at %.3f ms\n", now_ms());
  // the offsets are checked while the GPU works (a decreasing pair only makes the kernels defer that sentence: the
  // lengths are taken as unsigned); a bad batch is reported after the launch has drained
  uint64_t bad = 0;
  for (size_t i = 0; i < n; ++i) bad |= static_cast<uint64_t>(offsets[i + 1] < offsets[i]);
  // fetch the finished prefix of the ids with the copy engine while the kernel is still encoding
  CUDA_TRY(cudaEventRecord(ev_offs, st));  // (reused) kernel + status copy done
  unsigned long long seen = 0, copied = 0;
  const unsigned long long min_copy = 1ull << 20;  // ids per copy: 4 MB
  for (;;) {
    const cudaError_t q = cudaEventQuery(ev_offs);
    if (q != cudaSuccess && q != cudaErrorNotReady) CUDA_TRY(q);
    const unsigned long long pr = *reinterpret_cast<volatile unsigned long long *>(h_progress.p);
    if (pr > seen && pr <= h_ids.cap) seen = pr;
    if (!(fx & 1) && seen - copied >= min_copy) {
      CUDA_TRY(cudaMemcpyAsync(h_ids.p + copied, d_ids.p + copied, (seen - copied) * sizeof(int32_t), cudaMemcpyDeviceToHost, s_d2h));
      copied = seen;
    }
    if (q == cudaSuccess) break;
  }
  CUDA_TRY(cudaStreamSynchronize(st));
  if (feeder.joinable()) feeder.join();
  if (fx & 2) CUDA_TRY(cudaMemcpy(h_id_offsets.p, d_id_offsets.p, (n + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost));
  if (trace) fprintf(stderr, "[trace] fused kernel done at %.3f ms; warp-cycles: input wait %.1f M, compaction %.1f M (look-back %.1f M), "
                     "%llu groups on %d warps\n", now_ms(), h_ctrl64.p[4] * 1e-6, h_ctrl64.p[5] * 1e-6, h_ctrl64.p[6] * 1e-6,
                     static_cast<unsigned long long>(h_ctrl64.p[7]), grid * (lane_threads / 32));
  if (trace) {
    float km = 0.f;
    cudaEventElapsedTime(&km, ev[0], ev[1]);
    const double w = 1e-6 / (grid * (lane_threads / 32));  // M cycles per warp
    fprintf(stderr, "[trace] kernel %.3f ms on the device; M cycles per warp (lane 0): group loop %.2f = K1 + input wait %.2f, K2 %.2f, "
                    "K4 %.2f, drain %.2f\n", km, h_ctrl64.p[8] * w, h_ctrl64.p[9] * w, h_ctrl64.p[10] * w, h_ctrl64.p[11] * w,
            (h_ctrl64.p[8] - h_ctrl64.p[9] - h_ctrl64.p[10] - h_ctrl64.p[11]) * w);
  }
  if (bad) { cudaDeviceSynchronize(); set_error("offsets must be non-decreasing"); return SPM_ERR_ARG; }
  if (feed_rc) { cudaDeviceSynchronize(); set_error("host-to-device copy of a streamed batch failed"); return SPM_ERR_CUDA; }
  if (h_ctrl32.p[1] & 2u) { set_error("encode failed: the host-to-device copy of a streamed batch made no progress for 3 s"); return SPM_ERR_CUDA; }
  if (h_ctrl32.p[1] & 4u) { set_error("encode failed: the in-kernel compaction waited 3 s for an earlier segment"); return SPM_ERR_ENCODE; }
  if (h_ctrl32.p[1]) { set_error("encode failed: internal consistency check (status " + std::to_string(h_ctrl32.p[1]) + ")"); return SPM_ERR_ENCODE; }
  if (h_ctrl32.p[0] || h_ctrl32.p[2]) {
    // deferred sentences or a buffer that was too small: the chunked path has the second-chance and retry logic
    if (trace) fprintf(stderr, "[trace] fused path incomplete (deferred %u, overflow %u): redoing the batch in chunks\n",
                       h_ctrl32.p[0], h_ctrl32.p[2]);
    CUDA_TRY(cudaStreamSynchronize(s_d2h));
    fused_fallbacks++;
    // data like this (long words, very long lines) tends to come in runs: go chunked for a while, longer each time
    fused_skip = fused_backoff;
    fused_backoff = std::min(fused_backoff * 4, 1 << 16);
    return encode_host_streamed(bytes, offsets, n, ids, id_offsets);
  }
  fused_backoff = 8;
  const uint64_t tot = h_id_offsets.p[n];
  if (tot > copied) CUDA_TRY(cudaMemcpyAsync(h_ids.p + copied, d_ids.p + copied, (tot - copied) * sizeof(int32_t), cudaMemcpyDeviceToHost, s_d2h));
  CUDA_TRY(cudaStreamSynchronize(s_d2h));
  if (trace) fprintf(stderr, "[trace] ids on host at %.3f ms (%llu of %llu fetched while encoding)\n", now_ms(),
                     static_cast<unsigned long long>(copied), static_cast<unsigned long long>(tot));
  float a = 0.f;
  if (cudaEventElapsedTime(&a, ev[0], ev[1]) != cudaSuccess) a = 0.f;
  last_main_ms = a;
  last_ms = a;
  last_h2d = total_bytes + (n + 1) * sizeof(uint64_t) + P * sizeof(uint32_t);
  last_d2h = tot * sizeof(int32_t) + (n + 1) * sizeof(uint64_t);  // written by the kernel over PCIe
  *ids = h_ids.p;
  *id_offsets = h_id_offsets.p;
  return SPM_OK;
}

// ---- Decode (K7): per-id decoded strings + info words (decode_kernel.cuh) ----
int spm_engine::ensure_decode_tables() {
  if (dec_ready) return SPM_OK;
  const int V = model.vocab_size();
  std::vector<uint32_t> off(V + 1, 0), info(V, 0);
  std::string bytes;
  static const char kSpace[] = "\xE2\x96\x81";
  for (int i = 0; i < V; ++i) {
    const char *p = model.piece(i);
    const size_t len = model.piece_len(i);
    const uint8_t t = model.types[i];
    off[i] = static_cast<uint32_t>(bytes.size());
    if (t == SPM_CONTROL) {
      info[i] = kDecKindControl;
    } else if (t == SPM_UNKNOWN) {
      info[i] = kDecKindUnknown;
      bytes.append(model.unk_surface.c_str());  // the reference takes c_str() (:772-773)
    } else if (t == SPM_BYTE) {
      // PieceToByte (model_interface.cc:214-230): exactly "<0xXX>", upper-case hex
      int v = -1;
      if (len == 6 && p[0] == '<' && p[1] == '0' && p[2] == 'x' && p[5] == '>') {
        auto hex = [](char ch) { return ch >= '0' && ch <= '9' ? ch - '0' : (ch >= 'A' && ch <= 'F' ? ch - 'A' + 10 : -1); };
        const int hi = hex(p[3]), lo = hex(p[4]);
        if (hi >= 0 && lo >= 0) v = hi * 16 + lo;
      }
      info[i] = kDecKindByte | (v < 0 ? kDecBadByte : (static_cast<uint32_t>(v) << kDecByteShift));
      bytes.push_back(static_cast<char>(v < 0 ? 0 : v));
    } else {  // NORMAL, USER_DEFINED, UNUSED: U+2581 -> ' ' (StrReplaceAll, :809)
      info[i] = kDecKindNormal | ((len >= 3 && memcmp(p, kSpace, 3) == 0) ? kDecLeadWs : 0u);
      for (size_t k = 0; k < len;) {
        if (k + 3 <= len && memcmp(p + k, kSpace, 3) == 0) { bytes.push_back(' '); k += 3; }
        else { bytes.push_back(p[k]); k += 1; }
      }
    }
  }
  off[V] = static_cast<uint32_t>(bytes.size());
  std::vector<uint8_t> b(bytes.begin(), bytes.end());
  b.push_back(0);
  CUDA_TRY(d_dec_off.upload(off));
  CUDA_TRY(d_dec_info.upload(info));
  CUDA_TRY(d_dec_bytes.upload(b));
  dec_ready = true;
  return SPM_OK;
}

// Host-to-device copy of caller memory: pinned memory goes straight to the copy engine; pageable memory is first
// copied into a pinned staging buffer by a few host threads (the driver's own staging of pageable memory is
// single-threaded and synchronous), then handed to the copy engine.
namespace {
bool is_pinned(const void *p) {
  cudaPointerAttributes a{};
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { (void)cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost;
}
void parallel_memcpy(void *dst, const void *src, size_t bytes) {
  const size_t T = bytes < (4u << 20) ? 1 : std::min<size_t>(8, std::max<size_t>(1, std::thread::hardware_concurrency() / 2));
  if (T == 1) { memcpy(dst, src, bytes); return; }
  std::vector<std::thread> th;
  const size_t per = ((bytes + T - 1) / T + 63) & ~size_t{63};
  for (size_t t = 1; t < T; ++t) {
    const size_t lo = std::min(bytes, t * per), hi = std::min(bytes, (t + 1) * per);
    if (hi > lo) th.emplace_back([=]() { memcpy(static_cast<char *>(dst) + lo, static_cast<const char *>(src) + lo, hi - lo); });
  }
  memcpy(dst, src, std::min(bytes, per));
  for (auto &t : th) t.join();
}
}  // namespace

// Decode of a large host batch: chunks of id lists flow through H2D (staged when the caller's memory is pageable),
// decode + scan + gather, and D2H of the text on three streams; inputs and outputs are double buffered.
int spm_engine::decode_host_pipelined(const int32_t *ids, const uint64_t *id_offsets, size_t n, const char **text,
                                      const uint64_t **text_offsets) {
  if (!s_h2d) {
    CUDA_TRY(cudaStreamCreateWithFlags(&s_h2d, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&s_d2h, cudaStreamNonBlocking));
    for (int k = 0; k < 2; ++k) {
      CUDA_TRY(cudaEventCreateWithFlags(&ev_in[k], cudaEventDisableTiming));
      CUDA_TRY(cudaEventCreateWithFlags(&ev_out[k], cudaEventDisableTiming));
      CUDA_TRY(cudaEventCreateWithFlags(&ev_d2h[k], cudaEventDisableTiming));
    }
  }
  cudaStream_t st = stream;
  const bool trace = getenv("SPM_B200_TRACE") != nullptr;
  const auto t_begin = std::chrono::steady_clock::now();
  auto now_ms = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count(); };
  const size_t chunk = 131072;
  const size_t C = (n + chunk - 1) / chunk;
  const bool pinned_in = is_pinned(ids);
  uint64_t max_ids = 0;
  for (size_t c = 0; c < C; ++c) max_ids = std::max<uint64_t>(max_ids, id_offsets[std::min(n, (c + 1) * chunk)] - id_offsets[c * chunk]);
  const uint64_t total_ids = id_offsets[n] - id_offsets[0];
  for (int k = 0; k < 2; ++k) {
    CUDA_TRY(p_dec_ids[k].ensure(max_ids + 1));
    CUDA_TRY(p_offsets[k].ensure(chunk + 1));
    CUDA_TRY(p_dec_toff[k].ensure(chunk + 1));
    if (!pinned_in) CUDA_TRY(h_stage[k].ensure(max_ids * sizeof(int32_t) + 64));
  }
  CUDA_TRY(h_dec_text_offsets.ensure(n + 1));
  CUDA_TRY(h_dec_text.ensure(std::max<size_t>(h_dec_text.cap, total_ids * 5 + 16 * n + 4096)));
  CUDA_TRY(d_sent_start.ensure(chunk));
  CUDA_TRY(d_sent_count.ensure(chunk));
  CUDA_TRY(d_ctrl32.ensure(16));
  CUDA_TRY(d_ctrl64.ensure(8));
  CUDA_TRY(h_ctrl32.ensure(16));
  CUDA_TRY(h_ctrl64.ensure(8));
  const uint32_t nb_max = (static_cast<uint32_t>(chunk) + kScanChunk - 1) / kScanChunk;
  CUDA_TRY(d_block_sums.ensure(nb_max + 1));
  auto issue_h2d = [&](size_t c) -> int {
    const int k = static_cast<int>(c & 1);
    const size_t lo = c * chunk, hi = std::min(n, lo + chunk);
    const uint64_t cnt = id_offsets[hi] - id_offsets[lo];
    if (c >= 2) {
      CUDA_TRY(cudaStreamWaitEvent(s_h2d, ev_out[k], 0));  // the slot's previous chunk has been decoded
      if (!pinned_in) CUDA_TRY(cudaEventSynchronize(ev_in[k]));  // ... and its staging buffer has been read
    }
    const void *src = ids + id_offsets[lo];
    if (cnt && !pinned_in) {
      parallel_memcpy(h_stage[k].p, src, cnt * sizeof(int32_t));
      src = h_stage[k].p;
    }
    if (cnt) CUDA_TRY(cudaMemcpyAsync(p_dec_ids[k].p, src, cnt * sizeof(int32_t), cudaMemcpyHostToDevice, s_h2d));
    CUDA_TRY(cudaMemcpyAsync(p_offsets[k].p, id_offsets + lo, (hi - lo + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, s_h2d));
    CUDA_TRY(cudaEventRecord(ev_in[k], s_h2d));
    return SPM_OK;
  };
  uint64_t launches = 0;
  float main_ms = 0.f, all_ms = 0.f;  // decode kernels; scan + gather kernels
  unsigned long long text_base = 0;
  { const int rc = issue_h2d(0); if (rc) return rc; }
  for (size_t c = 0; c < C; ++c) {
    const int k = static_cast<int>(c & 1);
    const size_t lo = c * chunk, hi = std::min(n, lo + chunk);
    const uint32_t m = static_cast<uint32_t>(hi - lo);
    const uint64_t cnt = id_offsets[hi] - id_offsets[lo];
    CUDA_TRY(cudaStreamWaitEvent(st, ev_in[k], 0));
    if (c >= 2) CUDA_TRY(cudaStreamWaitEvent(st, ev_d2h[k], 0));  // the slot's previous text has left the GPU
    unsigned long long tmp_cap = cnt * 6 + 16ull * m + (1u << 20);
    unsigned long long tot = 0;
    bool staged_next = false;
    for (int attempt = 0; attempt < 3; ++attempt) {
      CUDA_TRY(d_dec_tmp.ensure(tmp_cap));
      CUDA_TRY(cudaMemsetAsync(d_ctrl32.p, 0, 16 * sizeof(uint32_t), st));
      CUDA_TRY(cudaMemsetAsync(d_ctrl64.p, 0, 8 * sizeof(unsigned long long), st));
      KDecode D{};
      D.ids = p_dec_ids[k].p - id_offsets[lo];
      D.id_offsets = reinterpret_cast<const unsigned long long *>(p_offsets[k].p);
      D.n = m;
      D.vocab = model.vocab_size();
      D.dec_off = d_dec_off.p;
      D.dec_bytes = d_dec_bytes.p;
      D.dec_info = d_dec_info.p;
      D.strip = (model.add_dummy_prefix || model.remove_extra_whitespaces) ? 1u : 0u;
      D.rm = model.remove_extra_whitespaces ? 1u : 0u;
      D.tmp = d_dec_tmp.p;
      D.tmp_cap = tmp_cap;
      D.cursor = d_ctrl64.p;
      D.sent_start = d_sent_start.p;
      D.sent_count = d_sent_count.p;
      D.status = d_ctrl32.p;
      CUDA_TRY(cudaEventRecord(ev[0], st));
      const int grid = static_cast<int>(std::min<size_t>(static_cast<size_t>(sm_count) * 8, (m + 7) / 8));
      decode_warp_kernel<<<grid, 256, 0, st>>>(D);
      CUDA_TRY(cudaGetLastError());
      CUDA_TRY(cudaEventRecord(ev[1], st));
      ++launches;
      CUDA_TRY(cudaMemcpyAsync(h_ctrl32.p, d_ctrl32.p, 16 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
      CUDA_TRY(cudaMemcpyAsync(h_ctrl64.p, d_ctrl64.p, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
      // the next chunk's ids are staged / queued while this chunk's kernel runs
      if (!staged_next && c + 1 < C) { const int rc = issue_h2d(c + 1); if (rc) { cudaDeviceSynchronize(); return rc; } }
      staged_next = true;
      CUDA_TRY(cudaStreamSynchronize(st));
      float a = 0.f;
      if (cudaEventElapsedTime(&a, ev[0], ev[1]) == cudaSuccess) main_ms += a;
      if (trace) fprintf(stderr, "[trace] decode chunk %zu: kernel done at %.3f ms (kernel %.3f ms, input %s)\n", c, now_ms(), a,
                         pinned_in ? "pinned" : "pageable, staged");
      if (h_ctrl32.p[1] == 2u) {  // :915-918
        cudaDeviceSynchronize();
        set_error("Invalid id: " + std::to_string(static_cast<int32_t>(h_ctrl32.p[3])));
        return SPM_ERR_ARG;
      }
      if (h_ctrl32.p[1] == 1u) {
        cudaDeviceSynchronize();
        set_error("Decode: byte piece of id " + std::to_string(h_ctrl32.p[3]) + " is not of the form <0xXX>");
        return SPM_ERR_ENCODE;
      }
      tot = h_ctrl64.p[0];
      if (h_ctrl32.p[2]) { tmp_cap = tot + 1024; continue; }
      break;
    }
    if (h_ctrl32.p[2]) { cudaDeviceSynchronize(); set_error("Decode: temporary buffer overflow persisted"); return SPM_ERR_CAPACITY; }
    const uint32_t nb = (m + kScanChunk - 1) / kScanChunk;
    CUDA_TRY(p_dec_text[k].ensure(tot + 16));
    if (c > 0) {  // the previous chunk's scan + gather finished before this chunk's kernel did
      float g = 0.f;
      if (cudaEventElapsedTime(&g, ev[2], ev[3]) == cudaSuccess) all_ms += g;
    }
    CUDA_TRY(cudaEventRecord(ev[2], st));
    scan_block_sums_kernel<<<nb, 256, 0, st>>>(d_sent_count.p, m, d_block_sums.p, 0);
    scan_block_prefix_kernel<<<1, 1024, 0, st>>>(d_block_sums.p, nb, d_ctrl64.p + 2);
    scan_write_gather_kernel<uint8_t><<<nb, 256, 0, st>>>(d_sent_count.p, m, d_block_sums.p, p_dec_toff[k].p, d_sent_start.p,
                                                          d_dec_tmp.p, p_dec_text[k].p, nullptr, nullptr, p_dec_text[k].cap, 0,
                                                          text_base);
    CUDA_TRY(cudaGetLastError());
    launches += 3;
    CUDA_TRY(cudaEventRecord(ev[3], st));
    CUDA_TRY(cudaEventRecord(ev_out[k], st));
    if (text_base + tot + 1 > h_dec_text.cap) {  // grow the pinned result buffer (rare): keep what has already arrived
      CUDA_TRY(cudaStreamSynchronize(s_d2h));
      PinBuf<char> bigger;
      CUDA_TRY(bigger.ensure(static_cast<size_t>(static_cast<double>(text_base + tot) / static_cast<double>(hi) * 1.25 * n) + tot + 4096));
      if (text_base) memcpy(bigger.p, h_dec_text.p, text_base);
      h_dec_text.release();
      h_dec_text = bigger;
    }
    CUDA_TRY(cudaStreamWaitEvent(s_d2h, ev_out[k], 0));
    if (tot) CUDA_TRY(cudaMemcpyAsync(h_dec_text.p + text_base, p_dec_text[k].p, tot, cudaMemcpyDeviceToHost, s_d2h));
    CUDA_TRY(cudaMemcpyAsync(h_dec_text_offsets.p + lo, p_dec_toff[k].p, (m + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, s_d2h));
    CUDA_TRY(cudaEventRecord(ev_d2h[k], s_d2h));
    text_base += tot;
  }
  CUDA_TRY(cudaStreamSynchronize(s_d2h));
  if (trace) fprintf(stderr, "[trace] decode: text on host at %.3f ms (%zu chunks)\n", now_ms(), C);
  {
    float g = 0.f;
    if (cudaEventElapsedTime(&g, ev[2], ev[3]) == cudaSuccess) all_ms += g;
  }
  h_dec_text.p[text_base] = 0;
  last_launches = launches;
  last_main_ms = main_ms;
  last_ms = main_ms + all_ms;
  last_h2d = total_ids * sizeof(int32_t) + (n + C) * sizeof(uint64_t);
  last_d2h = text_base + (n + C) * sizeof(uint64_t);
  *text = h_dec_text.p;
  *text_offsets = h_dec_text_offsets.p;
  return SPM_OK;
}

// ---- n-best (K5): lattice + A* per sentence on the GPU; leaves candidates in the temporary buffers ----
int spm_engine::run_nbest(const char *bytes, const uint64_t *offsets, size_t n, uint32_t nbest, uint64_t *tmp_total) {
  cudaStream_t st = stream;
  const uint64_t base = offsets[0];
  const uint64_t total_bytes = offsets[n] - base;
  CUDA_TRY(d_bytes.ensure(total_bytes + 64));
  CUDA_TRY(d_offsets.ensure(n + 1));
  if (total_bytes) CUDA_TRY(cudaMemcpyAsync(d_bytes.p, bytes + base, total_bytes, cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(d_offsets.p, offsets, (n + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
  last_h2d = total_bytes + (n + 1) * sizeof(uint64_t);
  NbestGeom G{};
  G.cap = lane_cap;
  G.node_cap = std::min<uint32_t>(65535u, 4 * lane_cap + 64);
  G.hyp_cap = 6144 + nbest * 64;   // typical need: ~60 hypotheses per result; retried with 8x on overflow
  G.heap_cap = 10000 + 1024 + 512;  // even: keeps the child pairs of the agenda 16-byte aligned
  // 32 warps per SM (64 registers per lane): the search is bound by L2 / HBM transactions on the per-lane agendas, and
  // measured throughput still rises from 16 to 32 warps (188 -> 157 ms for 256k sentences, nbest 64)
  const size_t groups = std::max<size_t>(1, (n + 31) / 32);   // one group of 32 sentences per warp pass
  int ctas = static_cast<int>(std::min<size_t>(sm_count, groups));
  int warps_per_cta = static_cast<int>(std::min<size_t>(32, (groups + ctas - 1) / ctas));
  size_t warps_total = static_cast<size_t>(ctas) * warps_per_cta;
  CUDA_TRY(d_lane_slabs.ensure(warps_total * lane_slab_bytes(lane_cap) + 256));
  CUDA_TRY(d_nb_scratch.ensure(warps_total * 32 * nbest_lane_bytes(G) + 256));
  bool grown = false;
  const size_t nc = n * static_cast<size_t>(nbest);
  CUDA_TRY(d_cand_start.ensure(nc));
  CUDA_TRY(d_cand_count.ensure(nc));
  CUDA_TRY(d_cand_score.ensure(nc));
  CUDA_TRY(d_n_cands.ensure(n));
  CUDA_TRY(d_ctrl32.ensure(16));
  CUDA_TRY(d_ctrl64.ensure(4));
  CUDA_TRY(h_ctrl32.ensure(16));
  CUDA_TRY(h_ctrl64.ensure(4));
  // candidates: at most one id per normalized byte each; start from 2 ids per input byte per 8 candidates
  unsigned long long tmp_cap = std::max<unsigned long long>(1u << 20, total_bytes * nbest / 3 + 64ull * n);
  for (int attempt = 0; attempt < 4; ++attempt) {
    CUDA_TRY(d_tmp_ids.ensure(tmp_cap));
    CUDA_TRY(cudaMemsetAsync(d_ctrl32.p, 0, 16 * sizeof(uint32_t), st));
    CUDA_TRY(cudaMemsetAsync(d_ctrl64.p, 0, 4 * sizeof(unsigned long long), st));
    KBatch B{};
    B.slab_l2 = slab_l2; B.slab_discard = slab_discard;
    B.bytes = d_bytes.p - base;
    B.offsets = d_offsets.p;
    B.n = static_cast<uint32_t>(n);
    B.off_lo = 0;
    B.off_hi = ~0ull;
    B.work_counter = d_ctrl32.p + 4;
    B.status = d_ctrl32.p;
    NbestOut O{};
    O.tmp_ids = d_tmp_ids.p;
    O.tmp_cap = tmp_cap;
    O.cursor = d_ctrl64.p;
    O.cand_start = d_cand_start.p;
    O.cand_count = d_cand_count.p;
    O.cand_score = d_cand_score.p;
    O.n_cands = d_n_cands.p;
    O.status = d_ctrl32.p;
    CUDA_TRY(cudaEventRecord(ev[0], st));
    { const int rc = build_order(d_offsets.p, n, st, &B.order, 0); if (rc) return rc; }
    nbest_lane_kernel<kNbestTop, 1024><<<ctas, warps_per_cta * 32, nbest_smem_bytes<kNbestTop>(warps_per_cta), st>>>(
        km, B, O, d_lane_slabs.p, d_nb_scratch.p, G, nbest);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(ev[1], st));
    ++last_launches;
    CUDA_TRY(cudaMemcpyAsync(h_ctrl32.p, d_ctrl32.p, 16 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(h_ctrl64.p, d_ctrl64.p, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (h_ctrl32.p[3] && !grown) {
      // some sentence needs a larger lattice / hypothesis pool: rerun the batch with roomy slabs on fewer warps
      grown = true;
      G.hyp_cap = std::min<uint32_t>(1u << 20, 8 * G.hyp_cap);
      G.node_cap = 65535u;
      G.cap = std::max<uint32_t>(G.cap, 8192u);  // long sentences: text and per-position arrays in roomy slabs
      warps_per_cta = G.hyp_cap > (1u << 17) ? 1 : 2;
      ctas = sm_count;
      warps_total = static_cast<size_t>(ctas) * warps_per_cta;
      CUDA_TRY(d_lane_slabs.ensure(warps_total * lane_slab_bytes(G.cap) + 256));
      CUDA_TRY(d_nb_scratch.ensure(warps_total * 32 * nbest_lane_bytes(G) + 256));
      continue;
    }
    if (h_ctrl32.p[3]) {
      set_error("n-best: a sentence exceeds the device path's capacity (normalized length > " + std::to_string(G.cap) +
                " bytes, lattice or hypothesis pool too large)");
      return SPM_ERR_UNSUPPORTED;
    }
    if (h_ctrl32.p[1]) { set_error("n-best: internal consistency check failed"); return SPM_ERR_ENCODE; }
    if (h_ctrl32.p[2]) { tmp_cap = h_ctrl64.p[0] + 1024; continue; }
    *tmp_total = h_ctrl64.p[0];
    return SPM_OK;
  }
  set_error("n-best: temporary buffer overflow persisted");
  return SPM_ERR_CAPACITY;
}

// ---- full-lattice operations (SURVEY 8f item 1): lattice + forward algorithm on the GPU (lattice_kernel.cuh), in
//      chunks of sentences; mode 0 then draws on the host exactly as Lattice::Sample (unigram_model.cc:511-542) does
//      -- std::exp in double, std::discrete_distribution<int> over float probabilities, this engine's std::mt19937 --
//      for the sentences in order, which reproduces the reference's single-threaded stream under a seed ----
int spm_engine::run_lattice(const char *bytes, const uint64_t *offsets, size_t n, float inv_theta, int mode, int samples) {
  cudaStream_t st = stream;
  lat_ids.clear();
  lat_scores.clear();
  lat_offsets.assign(1, 0);
  CUDA_TRY(d_ctrl32.ensure(16));
  CUDA_TRY(d_ctrl64.ensure(4));
  CUDA_TRY(h_ctrl32.ensure(16));
  CUDA_TRY(h_ctrl64.ensure(4));
  LatticeGeom G{};
  G.cap = lane_cap;
  G.node_cap = lane_cap * (trie.max_matches_per_start + 1) + 64;
  constexpr size_t kChunk = 32768;
  int warps_per_cta = 8;
  last_launches = 0;
  last_h2d = last_d2h = 0;
  float main_ms = 0.f;
  if (mode == 1) CUDA_TRY(h_lat_entropy.ensure(n + 1));
  std::vector<float> probs;
  std::vector<uint32_t> path;
  for (size_t lo = 0; lo < n; lo += kChunk) {
    const size_t m = std::min(kChunk, n - lo);
    const uint64_t base = offsets[lo];
    const uint64_t chunk_bytes = offsets[lo + m] - base;
    CUDA_TRY(d_bytes.ensure(chunk_bytes + 64));
    CUDA_TRY(d_offsets.ensure(m + 1));
    if (chunk_bytes) CUDA_TRY(cudaMemcpyAsync(d_bytes.p, bytes + base, chunk_bytes, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(d_offsets.p, offsets + lo, (m + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    last_h2d += chunk_bytes + (m + 1) * sizeof(uint64_t);
    const size_t groups = (m + 31) / 32;
    int ctas = static_cast<int>(std::min<size_t>(sm_count, (groups + warps_per_cta - 1) / warps_per_cta));
    size_t warps_total = static_cast<size_t>(ctas) * warps_per_cta;
    CUDA_TRY(d_lane_slabs.ensure(warps_total * lane_slab_bytes(G.cap) + 256));
    CUDA_TRY(d_lat_scratch.ensure(warps_total * 32 * lattice_lane_bytes(G) + 256));
    CUDA_TRY(d_lat_node_start.ensure(m));
    CUDA_TRY(d_lat_pos_start.ensure(m));
    CUDA_TRY(d_lat_nchars.ensure(m));
    CUDA_TRY(d_lat_entropy.ensure(m));
    // a sentence of b normalized bytes has at most b + 2 position records; nodes: start from 3 per input byte
    unsigned long long node_cap = mode == 0 ? 3ull * chunk_bytes + 64ull * m + 1024 : 1;
    const unsigned long long pos_cap = mode == 0 ? (chunk_bytes * max_expand_num) / max_expand_den + 16ull * m + 1024 : 1;
    for (int attempt = 0;; ++attempt) {
      CUDA_TRY(d_lat_nodes.ensure(node_cap));
      CUDA_TRY(d_lat_pos.ensure(pos_cap));
      CUDA_TRY(cudaMemsetAsync(d_ctrl32.p, 0, 16 * sizeof(uint32_t), st));
      CUDA_TRY(cudaMemsetAsync(d_ctrl64.p, 0, 4 * sizeof(unsigned long long), st));
      KBatch B{};
      B.slab_l2 = slab_l2; B.slab_discard = slab_discard;
      B.bytes = d_bytes.p - base;
      B.offsets = d_offsets.p;
      B.n = static_cast<uint32_t>(m);
      B.off_lo = 0;
      B.off_hi = ~0ull;
      B.work_counter = d_ctrl32.p + 4;
      B.status = d_ctrl32.p;
      LatticeOut O{};
      O.nodes = d_lat_nodes.p;
      O.pos = d_lat_pos.p;
      O.node_cap = node_cap;
      O.pos_cap = pos_cap;
      O.cursor = d_ctrl64.p;
      O.node_start = d_lat_node_start.p;
      O.pos_start = d_lat_pos_start.p;
      O.n_chars = d_lat_nchars.p;
      O.entropy = d_lat_entropy.p;
      O.status = d_ctrl32.p;
      CUDA_TRY(cudaEventRecord(ev[0], st));
      lattice_lane_kernel<<<ctas, warps_per_cta * 32, kLaneTableBytes, st>>>(km, B, O, d_lane_slabs.p, d_lat_scratch.p, G,
                                                                            inv_theta, mode);
      CUDA_TRY(cudaGetLastError());
      CUDA_TRY(cudaEventRecord(ev[1], st));
      ++last_launches;
      CUDA_TRY(cudaMemcpyAsync(h_ctrl32.p, d_ctrl32.p, 16 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
      CUDA_TRY(cudaMemcpyAsync(h_ctrl64.p, d_ctrl64.p, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
      CUDA_TRY(cudaStreamSynchronize(st));
      float a = 0.f;
      if (cudaEventElapsedTime(&a, ev[0], ev[1]) == cudaSuccess) main_ms += a;
      if (h_ctrl32.p[3] && G.cap < 8192u) {
        // a long sentence: this and the later chunks run with roomy per-lane slabs on fewer warps
        G.cap = 8192u;
        G.node_cap = G.cap * (trie.max_matches_per_start + 1) + 64;
        warps_per_cta = 2;
        ctas = static_cast<int>(std::min<size_t>(sm_count, (groups + warps_per_cta - 1) / warps_per_cta));
        warps_total = static_cast<size_t>(ctas) * warps_per_cta;
        CUDA_TRY(d_lane_slabs.ensure(warps_total * lane_slab_bytes(G.cap) + 256));
        CUDA_TRY(d_lat_scratch.ensure(warps_total * 32 * lattice_lane_bytes(G) + 256));
        --attempt;
        continue;
      }
      if (h_ctrl32.p[3]) {
        set_error("lattice: a sentence exceeds the device path's capacity (normalized length > " + std::to_string(G.cap) + " bytes)");
        return SPM_ERR_UNSUPPORTED;
      }
      if (h_ctrl32.p[2] && attempt == 0) { node_cap = h_ctrl64.p[0] + 1024; continue; }
      if (h_ctrl32.p[2]) { set_error("lattice: output buffer overflow persisted"); return SPM_ERR_CAPACITY; }
      break;
    }
    if (mode == 1) {
      CUDA_TRY(cudaMemcpyAsync(h_lat_entropy.p + lo, d_lat_entropy.p, m * sizeof(float), cudaMemcpyDeviceToHost, st));
      CUDA_TRY(cudaStreamSynchronize(st));
      last_d2h += m * sizeof(float);
      continue;
    }
    const unsigned long long tot_nodes = h_ctrl64.p[0], tot_pos = h_ctrl64.p[1];
    CUDA_TRY(h_lat_nodes.ensure(tot_nodes + 1));
    CUDA_TRY(h_lat_pos.ensure(tot_pos + 1));
    CUDA_TRY(h_lat_node_start.ensure(m));
    CUDA_TRY(h_lat_pos_start.ensure(m));
    CUDA_TRY(h_lat_nchars.ensure(m));
    if (tot_nodes) CUDA_TRY(cudaMemcpyAsync(h_lat_nodes.p, d_lat_nodes.p, tot_nodes * sizeof(uint4), cudaMemcpyDeviceToHost, st));
    if (tot_pos) CUDA_TRY(cudaMemcpyAsync(h_lat_pos.p, d_lat_pos.p, tot_pos * sizeof(uint2), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(h_lat_node_start.p, d_lat_node_start.p, m * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(h_lat_pos_start.p, d_lat_pos_start.p, m * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(h_lat_nchars.p, d_lat_nchars.p, m * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    last_d2h += tot_nodes * sizeof(uint4) + tot_pos * sizeof(uint2) + m * 20;
    // ---- Lattice::Sample per sentence, in order, on one generator ----
    const bool bf = model.byte_fallback;
    for (size_t i = 0; i < m; ++i) {
      const uint32_t L = h_lat_nchars.p[i];
      const uint4 *nodes = h_lat_nodes.p + h_lat_node_start.p[i];
      const uint2 *pos = h_lat_pos.p + h_lat_pos_start.p[i];
      for (int sidx = 0; sidx < samples; ++sidx) {
        float score = 0.f;
        if (L) {
          auto A = [&](uint32_t p) { float f; memcpy(&f, &pos[p].x, 4); return f; };
          path.clear();
          float Z = A(L);
          uint32_t p = L;
          while (p != 0) {  // at position 0 the only candidate is BOS: no draw (a one-weight distribution)
            const uint32_t q0 = pos[p].y, q1 = pos[p + 1].y;
            probs.clear();
            for (uint32_t q = q0; q < q1; ++q) {
              float sc; memcpy(&sc, &nodes[q].y, 4);
              const float arg = A(nodes[q].z & 0xFFFFu) + inv_theta * sc - Z;   // float expression (:528-529)
              probs.push_back(static_cast<float>(std::exp(static_cast<double>(arg))));
            }
            std::discrete_distribution<int> dist(probs.begin(), probs.end());
            const uint32_t q = q0 + static_cast<uint32_t>(dist(rng));
            path.push_back(q);
            p = nodes[q].z & 0xFFFFu;
            Z = A(p);
          }
          // id path of PopulateSentencePieceText over the sampled nodes, left to right
          bool prev_unk = false;
          for (size_t k = path.size(); k-- > 0;) {
            const uint4 nd = nodes[path[k]];
            float sc; memcpy(&sc, &nd.y, 4);
            score += inv_theta * sc;   // (:846-847)
            const int32_t id = static_cast<int32_t>(nd.x);
            const bool isunk = id == unk_id;
            if (isunk && bf) {
              const uint32_t first = nd.w & 0xFFu;
              static const uint8_t kLen[16] = {1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 2, 2, 3, 4};
              uint32_t cl = kLen[first >> 4];
              // the node covers one character of the normalized text; its byte count is the span of the character
              // (a truncated character at the end of the text has fewer bytes: the bytes above it are zero and a
              //  zero byte never follows a multi-byte lead in normalized text)
              for (uint32_t bq = 0; bq < cl; ++bq) {
                const uint32_t bv = (nd.w >> (8 * bq)) & 0xFFu;
                if (bq > 0 && bv == 0) break;
                lat_ids.push_back(byte_to_id_host[bv]);
              }
            } else if (!(isunk && prev_unk)) {
              lat_ids.push_back(id);
            }
            prev_unk = isunk;
          }
          score -= A(L);  // - marginal (:853)
        }
        lat_offsets.push_back(lat_ids.size());
        lat_scores.push_back(score);
      }
    }
  }
  last_main_ms = main_ms;
  last_ms = main_ms;
  return SPM_OK;
}

// ---------------------------------------------------------------- C ABI ----

extern "C" {

const char *spm_last_error(const spm_engine *e) {
  if (e) return e->err.c_str();
  return g_create_error.c_str();
}

static int create_common(spm_engine *e, int device, spm_engine **out) {
  auto fail = [&](int code, const std::string &msg) {
    std::lock_guard<std::mutex> lk(g_create_mu);
    g_create_error = msg;
    delete e;
    return code;
  };
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(SPM_ERR_CUDA, "no CUDA device available: this engine has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(SPM_ERR_ARG, "invalid device ordinal");
  e->device = device;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return fail(SPM_ERR_CUDA, "cudaGetDeviceProperties failed");
  if (prop.major < 10) return fail(SPM_ERR_CUDA, "this build targets sm_100a (B200); found compute capability " +
                                                      std::to_string(prop.major) + "." + std::to_string(prop.minor));
  e->sm_count = prop.multiProcessorCount;
  if (const char *v = getenv("SPM_B200_SORT")) e->sort_by_length = atoi(v) != 0;  // A/B knob for profiles/
  if (const char *v = getenv("SPM_B200_FUSED")) e->fused_host_path = atoi(v) != 0;
  if (const char *v = getenv("SPM_B200_FASTWORDS")) e->force_fast_words = atoi(v) != 0 ? 1 : 0;
  if (const char *v = getenv("SPM_B200_KSTATS")) e->kstats = atoi(v) != 0;
  if (const char *v = getenv("SPM_B200_BPE_CACHE")) e->bpe_cache_log2 = std::min(24, std::max(0, atoi(v)));
  if (const char *v = getenv("SPM_B200_SLAB_DISCARD")) e->slab_discard = static_cast<uint32_t>(atoi(v));
  if (const char *v = getenv("SPM_B200_SLAB_L2")) e->slab_l2 = static_cast<uint32_t>(atoi(v));
  if (const char *v = getenv("SPM_B200_LANE_CAP")) e->lane_cap = std::min(1020, std::max(64, atoi(v))) & ~3;
  if (const char *v = getenv("SPM_B200_BPE_LANE_V")) e->bpe_lane_version = atoi(v);
  e->smem_optin = prop.sharedMemPerBlockOptin;
  if (cudaSetDevice(device) != cudaSuccess) return fail(SPM_ERR_CUDA, "cudaSetDevice failed");
  int rc = e->build_tables();
  if (rc) return fail(rc, e->err);
  if (cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking) != cudaSuccess) return fail(SPM_ERR_CUDA, "stream creation failed");
  for (auto &ev : e->ev)
    if (cudaEventCreate(&ev) != cudaSuccess) return fail(SPM_ERR_CUDA, "event creation failed");
  rc = e->configure_kernel_attrs();
  if (rc) return fail(rc, e->err);
  *out = e;
  return SPM_OK;
}

int spm_engine_create(const spm_model_desc *d, int device, spm_engine **out) {
  if (!d || !out || d->vocab_size <= 0 || !d->piece_bytes || !d->piece_off || !d->scores || !d->types) {
    std::lock_guard<std::mutex> lk(g_create_mu);
    g_create_error = "spm_engine_create: null or empty model description";
    return SPM_ERR_ARG;
  }
  spm_engine *e = new spm_engine();
  ModelData &m = e->model;
  m.model_type = d->model_type;
  m.piece_off.assign(d->piece_off, d->piece_off + d->vocab_size + 1);
  m.piece_bytes.assign(d->piece_bytes, d->piece_off[d->vocab_size]);
  m.scores.assign(d->scores, d->scores + d->vocab_size);
  m.types.assign(d->types, d->types + d->vocab_size);
  m.byte_fallback = d->byte_fallback;
  m.treat_whitespace_as_suffix = d->treat_whitespace_as_suffix;
  m.add_dummy_prefix = d->add_dummy_prefix;
  m.remove_extra_whitespaces = d->remove_extra_whitespaces;
  m.escape_whitespaces = d->escape_whitespaces;
  if (d->charsmap && d->charsmap_bytes) m.charsmap.assign(static_cast<const char *>(d->charsmap), d->charsmap_bytes);
  return create_common(e, device, out);
}

int spm_engine_create_from_serialized(const void *model_proto, size_t len, int device, spm_engine **out) {
  if (!model_proto || !len || !out) {
    std::lock_guard<std::mutex> lk(g_create_mu);
    g_create_error = "spm_engine_create_from_serialized: null argument";
    return SPM_ERR_ARG;
  }
  spm_engine *e = new spm_engine();
  std::string err;
  if (!ParseModelProto(model_proto, len, &e->model, &err)) {
    std::lock_guard<std::mutex> lk(g_create_mu);
    g_create_error = err;
    delete e;
    return SPM_ERR_MODEL;
  }
  return create_common(e, device, out);
}

void spm_engine_destroy(spm_engine *e) {
  if (!e) return;
  cudaSetDevice(e->device);
  if (e->stream) cudaStreamSynchronize(e->stream);
  e->d_link.release(); e->d_val.release(); e->d_user_link.release(); e->d_cm_units.release(); e->d_cm_lead.release();
  e->d_cm_pair.release(); e->d_id.release(); e->d_cm_solo.release(); e->d_byte_to_id.release(); e->d_cm_targets.release();
  e->d_types.release(); e->d_scores.release(); e->d_word_safe.release(); e->d_node4.release(); e->d_word_fast.release(); e->d_bpe_cache.release(); e->d_kstats.release(); e->d_sample.release(); e->d_bytes.release(); e->d_tmp_norm.release(); e->d_norm.release();
  e->d_long_scratch.release(); e->d_offsets.release(); e->d_tmp_ids.release(); e->d_ids.release();
  e->d_tmp_tok_end.release(); e->d_tok_end.release(); e->d_tmp_n2o.release(); e->d_n2o.release();
  e->d_sent_count.release(); e->d_norm_len.release(); e->d_deferred.release(); e->d_deferred2.release(); e->d_long_list.release();
  e->d_ctrl32.release(); e->d_sent_start.release(); e->d_norm_start.release(); e->d_id_offsets.release();
  e->d_norm_offsets.release(); e->d_n2o_offsets.release(); e->d_block_sums.release(); e->d_ctrl64.release();
  e->d_long_off.release();
  e->d_lane_slabs.release(); e->d_bpe_long.release();
  e->d_node2.release();
  e->d_lat_scratch.release(); e->d_lat_nodes.release(); e->d_lat_pos.release(); e->d_lat_node_start.release();
  e->d_lat_pos_start.release(); e->d_lat_nchars.release(); e->d_lat_entropy.release(); e->h_lat_nodes.release();
  e->h_lat_pos.release(); e->h_lat_node_start.release(); e->h_lat_pos_start.release(); e->h_lat_nchars.release();
  e->h_lat_entropy.release();
  e->d_nb_scratch.release(); e->d_cand_start.release(); e->d_cand_offsets.release(); e->d_cand_count.release();
  e->d_n_cands.release(); e->d_picks.release(); e->d_cand_score.release(); e->h_cand_score.release();
  e->h_n_cands.release(); e->h_picks.release(); e->h_cand_offsets.release();
  for (int k = 0; k < 2; ++k) {
    e->p_bytes[k].release(); e->p_offsets[k].release(); e->p_ids[k].release(); e->p_id_offsets[k].release();
    if (e->ev_in[k]) cudaEventDestroy(e->ev_in[k]);
    if (e->ev_out[k]) cudaEventDestroy(e->ev_out[k]);
    if (e->ev_d2h[k]) cudaEventDestroy(e->ev_d2h[k]);
  }
  e->s_bytes.release(); e->s_offsets.release(); e->d_ready.release(); e->h_marks.release(); e->h_progress.release();
  e->d_dec_off.release(); e->d_dec_info.release(); e->d_dec_bytes.release(); e->d_dec_tmp.release(); e->d_dec_text.release();
  e->d_dec_ids.release(); e->d_dec_text_offsets.release(); e->h_dec_text.release(); e->h_dec_text_offsets.release();
  for (int k = 0; k < 2; ++k) { e->p_dec_ids[k].release(); e->p_dec_text[k].release(); e->p_dec_toff[k].release(); e->h_stage[k].release(); }
  e->d_order.release(); e->d_order_hist.release(); e->d_seg_done.release(); e->d_sent_rel.release(); e->d_seg_words.release();
  if (e->ev_offs) cudaEventDestroy(e->ev_offs);
  if (e->s_h2d) cudaStreamDestroy(e->s_h2d);
  if (e->s_d2h) cudaStreamDestroy(e->s_d2h);
  e->h_ids.release(); e->h_tok_end.release(); e->h_n2o.release(); e->h_ctrl32.release(); e->h_deferred.release();
  e->h_id_offsets.release(); e->h_norm_offsets.release(); e->h_ctrl64.release(); e->h_norm.release();
  for (auto &ev : e->ev) if (ev) cudaEventDestroy(ev);
  if (e->stream) cudaStreamDestroy(e->stream);
  delete e;
}

int spm_engine_set_types(spm_engine *e, const uint8_t *types) {
  if (!e || !types) return SPM_ERR_ARG;
  std::lock_guard<std::mutex> lk(e->mu);
  // the kinds CONTROL/UNKNOWN/BYTE never change (sentencepiece_processor.cc:311-316)
  for (int i = 0; i < e->model.vocab_size(); ++i) {
    const uint8_t o = e->model.types[i], t = types[i];
    const bool on = o == SPM_NORMAL || o == SPM_USER_DEFINED || o == SPM_UNUSED;
    const bool tn = t == SPM_NORMAL || t == SPM_USER_DEFINED || t == SPM_UNUSED;
    if (on != tn || (!on && o != t)) { e->set_error("spm_engine_set_types: piece class changes are not allowed"); return SPM_ERR_ARG; }
  }
  e->model.types.assign(types, types + e->model.vocab_size());
  return e->upload_types();
}

int spm_engine_cache_reset(spm_engine *e) {
  if (!e) return SPM_ERR_ARG;
  std::lock_guard<std::mutex> lk(e->mu);
  if (e->km.bpe_cache_mask) {
    // (the engine's streams do not synchronize with the legacy stream: the fill runs on the engine's own stream and is
    // complete when the call returns, whatever stream the next batch uses)
    if (cudaSetDevice(e->device) != cudaSuccess ||
        cudaMemsetAsync(e->d_bpe_cache.p, 0, (static_cast<size_t>(e->km.bpe_cache_mask) + 1) * 64, e->stream) != cudaSuccess ||
        cudaStreamSynchronize(e->stream) != cudaSuccess) {
      e->set_error("spm_engine_cache_reset: cudaMemset failed");
      return SPM_ERR_CUDA;
    }
  }
  return SPM_OK;
}

static void finish_timing(spm_engine *e);

int spm_engine_set_unk_surface(spm_engine *e, const char *surface, size_t bytes) {
  if (!e || (!surface && bytes)) return SPM_ERR_ARG;
  std::lock_guard<std::mutex> lk(e->mu);
  e->model.unk_surface.assign(surface ? surface : "", bytes);
  e->dec_ready = false;
  return SPM_OK;
}

int spm_decode_ids(spm_engine *e, const int32_t *ids, const uint64_t *id_offsets, size_t n, const char **text,
                   const uint64_t **text_offsets) {
  if (!e || !id_offsets || !text || !text_offsets) return SPM_ERR_ARG;
  std::lock_guard<std::mutex> lk(e->mu);
  auto set_error = [&](const std::string &m) { e->set_error(m); };
  if (n >= 0xFFFFFFF0ull) { set_error("too many id lists in one call"); return SPM_ERR_ARG; }
  for (size_t i = 0; i < n; ++i)
    if (id_offsets[i + 1] < id_offsets[i]) { set_error("id_offsets must be non-decreasing"); return SPM_ERR_ARG; }
  const uint64_t base = id_offsets[0];
  const uint64_t total_ids = id_offsets[n] - base;
  if (total_ids && !ids) return SPM_ERR_ARG;
  if (!e->model.denormalizer_charsmap.empty()) {
    set_error("Decode: models with a denormalizer_spec are not on the device path");
    return SPM_ERR_UNSUPPORTED;
  }
  CUDA_TRY(cudaSetDevice(e->device));
  { const int rc = e->ensure_decode_tables(); if (rc) return rc; }
  if (n >= e->pipeline_min_sentences) return e->decode_host_pipelined(ids, id_offsets, n, text, text_offsets);
  cudaStream_t st = e->stream;
  e->last_launches = 0;
  CUDA_TRY(e->h_dec_text_offsets.ensure(n + 1));
  if (n == 0) {
    CUDA_TRY(e->h_dec_text.ensure(1));
    e->h_dec_text_offsets.p[0] = 0;
    *text = e->h_dec_text.p;
    *text_offsets = e->h_dec_text_offsets.p;
    return SPM_OK;
  }
  CUDA_TRY(e->d_dec_ids.ensure(total_ids + 1));
  CUDA_TRY(e->d_offsets.ensure(n + 1));
  CUDA_TRY(e->d_sent_start.ensure(n));
  CUDA_TRY(e->d_sent_count.ensure(n));
  CUDA_TRY(e->d_ctrl32.ensure(16));
  CUDA_TRY(e->d_ctrl64.ensure(8));
  CUDA_TRY(e->h_ctrl32.ensure(16));
  CUDA_TRY(e->h_ctrl64.ensure(8));
  CUDA_TRY(e->d_dec_text_offsets.ensure(n + 1));
  if (total_ids) CUDA_TRY(cudaMemcpyAsync(e->d_dec_ids.p, ids + base, total_ids * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(e->d_offsets.p, id_offsets, (n + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
  e->last_h2d = total_ids * sizeof(int32_t) + (n + 1) * sizeof(uint64_t);
  const uint32_t n32 = static_cast<uint32_t>(n);
  unsigned long long tmp_cap = total_ids * 6 + 16ull * n + (1u << 20);  // retried with the exact size on overflow
  unsigned long long tot = 0;
  for (int attempt = 0; attempt < 3; ++attempt) {
    CUDA_TRY(e->d_dec_tmp.ensure(tmp_cap));
    CUDA_TRY(cudaMemsetAsync(e->d_ctrl32.p, 0, 16 * sizeof(uint32_t), st));
    CUDA_TRY(cudaMemsetAsync(e->d_ctrl64.p, 0, 8 * sizeof(unsigned long long), st));
    KDecode D{};
    D.ids = e->d_dec_ids.p - base;
    D.id_offsets = reinterpret_cast<const unsigned long long *>(e->d_offsets.p);
    D.n = n32;
    D.vocab = e->model.vocab_size();
    D.dec_off = e->d_dec_off.p;
    D.dec_bytes = e->d_dec_bytes.p;
    D.dec_info = e->d_dec_info.p;
    D.strip = (e->model.add_dummy_prefix || e->model.remove_extra_whitespaces) ? 1u : 0u;
    D.rm = e->model.remove_extra_whitespaces ? 1u : 0u;
    D.tmp = e->d_dec_tmp.p;
    D.tmp_cap = tmp_cap;
    D.cursor = e->d_ctrl64.p;
    D.sent_start = e->d_sent_start.p;
    D.sent_count = e->d_sent_count.p;
    D.status = e->d_ctrl32.p;
    CUDA_TRY(cudaEventRecord(e->ev[0], st));
    const int grid = static_cast<int>(std::min<size_t>(static_cast<size_t>(e->sm_count) * 8, (n + 7) / 8));
    decode_warp_kernel<<<grid, 256, 0, st>>>(D);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(e->ev[1], st));
    ++e->last_launches;
    CUDA_TRY(cudaMemcpyAsync(e->h_ctrl32.p, e->d_ctrl32.p, 16 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(e->h_ctrl64.p, e->d_ctrl64.p, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (e->h_ctrl32.p[1] == 2u) {  // :915-918
      set_error("Invalid id: " + std::to_string(static_cast<int32_t>(e->h_ctrl32.p[3])));
      return SPM_ERR_ARG;
    }
    if (e->h_ctrl32.p[1] == 1u) {
      set_error("Decode: byte piece of id " + std::to_string(e->h_ctrl32.p[3]) + " is not of the form <0xXX>");
      return SPM_ERR_ENCODE;
    }
    tot = e->h_ctrl64.p[0];
    if (e->h_ctrl32.p[2]) { tmp_cap = tot + 1024; continue; }
    break;
  }
  if (e->h_ctrl32.p[2]) { set_error("Decode: temporary buffer overflow persisted"); return SPM_ERR_CAPACITY; }
  // offsets (exclusive scan) + gather into list order: the kernels of the encode path
  const uint32_t nb = (n32 + kScanChunk - 1) / kScanChunk;
  CUDA_TRY(e->d_block_sums.ensure(nb + 1));
  CUDA_TRY(e->d_dec_text.ensure(tot + 16));
  scan_block_sums_kernel<<<nb, 256, 0, st>>>(e->d_sent_count.p, n32, e->d_block_sums.p, 0);
  scan_block_prefix_kernel<<<1, 1024, 0, st>>>(e->d_block_sums.p, nb, e->d_ctrl64.p + 2);
  scan_write_gather_kernel<uint8_t><<<nb, 256, 0, st>>>(e->d_sent_count.p, n32, e->d_block_sums.p, e->d_dec_text_offsets.p,
                                                        e->d_sent_start.p, e->d_dec_tmp.p, e->d_dec_text.p, nullptr, nullptr,
                                                        e->d_dec_text.cap, 0, 0ull);
  CUDA_TRY(cudaGetLastError());
  e->last_launches += 3;
  CUDA_TRY(cudaEventRecord(e->ev[2], st));
  CUDA_TRY(e->h_dec_text.ensure(tot + 1));
  if (tot) CUDA_TRY(cudaMemcpyAsync(e->h_dec_text.p, e->d_dec_text.p, tot, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaMemcpyAsync(e->h_dec_text_offsets.p, e->d_dec_text_offsets.p, (n + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  e->last_d2h = tot + (n + 1) * sizeof(uint64_t);
  finish_timing(e);
  e->h_dec_text.p[tot] = 0;
  *text = e->h_dec_text.p;
  *text_offsets = e->h_dec_text_offsets.p;
  return SPM_OK;
}

void *spm_host_alloc(size_t bytes) {
  void *p = nullptr;
  if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) return nullptr;
  return p;
}
void spm_host_free(void *p) { if (p) cudaFreeHost(p); }

int spm_engine_get_info(const spm_engine *e, spm_engine_info *info) {
  if (!e || !info) return SPM_ERR_ARG;
  memset(info, 0, sizeof *info);
  info->device = e->device;
  info->sm_count = e->sm_count;
  info->model_type = e->model.model_type;
  info->vocab_size = e->model.vocab_size();
  info->unk_id = e->unk_id;
  info->min_score = e->min_score;
  info->max_score = e->max_score;
  info->trie_units = e->km.trie_units;
  const LaunchGeom g = plan_geometry(*e, false, e->G, e->threads, e->ncap, e->km.match_slots);
  info->trie_hot_units = g.hot_link;
  info->charsmap_units = e->charsmap_units;
  info->last_kernel_launches = e->last_launches;
  info->last_kernel_ms = e->last_ms;
  info->last_main_kernel_ms = e->last_main_ms;
  info->last_h2d_bytes = e->last_h2d;
  info->last_d2h_bytes = e->last_d2h;
  info->last_deferred = e->last_deferred;
  return SPM_OK;
}

int spm_engine_set_tuning(spm_engine *e, int lanes, int cap, int ctas) {
  if (!e) return SPM_ERR_ARG;
  std::lock_guard<std::mutex> lk(e->mu);
  if (lanes) {
    if (lanes != 1 && lanes != 4 && lanes != 8 && lanes != 16 && lanes != 32 && lanes != 64) { e->set_error("lanes_per_sentence must be 1, 4, 8, 16, 32 or 64"); return SPM_ERR_ARG; }
    e->G = lanes;
  }
  if (cap) {
    if (cap < 64 || cap > 8192) { e->set_error("smem_norm_cap out of range"); return SPM_ERR_ARG; }
    e->ncap = static_cast<uint32_t>(cap + 15) & ~15u;
  }
  if (ctas) {
    // encoded as threads per CTA when >= 32
    if (ctas >= 32) {
      if (ctas % 32 || ctas > 1024) { e->set_error("threads per CTA must be a multiple of 32, <= 1024"); return SPM_ERR_ARG; }
      e->threads = ctas;
    } else {
      e->ctas_per_sm = ctas;
    }
  }
  return SPM_OK;
}

static void finish_timing(spm_engine *e) {
  float a = 0.f, b = 0.f;
  if (cudaEventElapsedTime(&a, e->ev[0], e->ev[1]) == cudaSuccess) e->last_main_ms = a;
  if (cudaEventElapsedTime(&b, e->ev[0], e->ev[2]) == cudaSuccess) e->last_ms = b;
  else e->last_ms = e->last_main_ms;
  (void)cudaGetLastError();  // an unrecorded event must not leave a stale error behind
}

int spm_encode_ids_device(spm_engine *e, const char *d_bytes, const uint64_t *d_offsets, size_t n, uint64_t total_bytes,
                          int32_t *d_ids, uint64_t ids_capacity, uint64_t *d_id_offsets, uint64_t *total_ids,
                          void *stream) {
  if (!e) return SPM_ERR_ARG;
  std::lock_guard<std::mutex> lk(e->mu);
  auto set_error = [&](const std::string &m) { e->set_error(m); };
  if (!d_offsets || !d_id_offsets || !total_ids || (n && !d_bytes && total_bytes)) { e->set_error("null argument"); return SPM_ERR_ARG; }
  if (n >= 0xFFFFFFF0ull) { e->set_error("too many sentences in one call"); return SPM_ERR_ARG; }
  CUDA_TRY(cudaSetDevice(e->device));
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : e->stream;
  *total_ids = 0;
  if (n == 0) {
    CUDA_TRY(cudaMemsetAsync(d_id_offsets, 0, sizeof(uint64_t), st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return SPM_OK;
  }
  e->last_h2d = e->last_d2h = 0;
  if (e->model.model_type == SPM_UNIGRAM) {
    const int rc0 = e->pick_fast_words_device(reinterpret_cast<const uint8_t *>(d_bytes), d_offsets, n, st, &e->batch_fast_words);
    if (rc0) return rc0;
  }
  const int rc = e->run_device(reinterpret_cast<const uint8_t *>(d_bytes), d_offsets, n, total_bytes, false, d_ids,
                               ids_capacity, reinterpret_cast<unsigned long long *>(d_id_offsets), total_ids, nullptr, st);
  if (rc) return rc;
  CUDA_TRY(cudaStreamSynchronize(st));
  finish_timing(e);
  return SPM_OK;
}

static int encode_host_locked(spm_engine *e, const char *bytes, const uint64_t *offsets, size_t n, bool spans,
                              const int32_t **ids, const uint32_t **tok_end, const uint64_t **id_offsets,
                              const char **normalized, const uint64_t **norm_offsets, const uint32_t **n2o) {
  auto set_error = [&](const std::string &m) { e->set_error(m); };
  if (!offsets || !ids || !id_offsets || (n && !bytes && offsets[n] != offsets[0])) { e->set_error("null argument"); return SPM_ERR_ARG; }
  if (n >= 0xFFFFFFF0ull) { e->set_error("too many sentences in one call"); return SPM_ERR_ARG; }
  CUDA_TRY(cudaSetDevice(e->device));
  cudaStream_t st = e->stream;
  CUDA_TRY(e->h_id_offsets.ensure(n + 1));
  CUDA_TRY(e->h_ids.ensure(1));
  if (n == 0) {
    e->h_id_offsets.p[0] = 0;
    *ids = e->h_ids.p;
    *id_offsets = e->h_id_offsets.p;
    if (spans) {
      CUDA_TRY(e->h_norm_offsets.ensure(1)); CUDA_TRY(e->h_norm.ensure(1)); CUDA_TRY(e->h_tok_end.ensure(1)); CUDA_TRY(e->h_n2o.ensure(1));
      e->h_norm_offsets.p[0] = 0;
      *tok_end = e->h_tok_end.p; *normalized = reinterpret_cast<const char *>(e->h_norm.p);
      *norm_offsets = e->h_norm_offsets.p; *n2o = e->h_n2o.p;
    }
    return SPM_OK;
  }
  for (size_t i = 0; i < n; ++i)
    if (offsets[i + 1] < offsets[i]) { e->set_error("offsets must be non-decreasing"); return SPM_ERR_ARG; }
  const uint64_t base = offsets[0];
  const uint64_t total_bytes = offsets[n] - base;
  CUDA_TRY(e->d_bytes.ensure(total_bytes + 64));
  CUDA_TRY(e->d_offsets.ensure(n + 1));
  if (total_bytes) CUDA_TRY(cudaMemcpyAsync(e->d_bytes.p, bytes + base, total_bytes, cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(e->d_offsets.p, offsets, (n + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
  e->last_h2d = total_bytes + (n + 1) * sizeof(uint64_t);
  uint64_t tot = 0, totn = 0;
  const int rc = e->run_device(e->d_bytes.p - base, e->d_offsets.p, n, total_bytes, spans, nullptr, 0, nullptr, &tot, &totn, st);
  if (rc) return rc;
  CUDA_TRY(e->h_ids.ensure(tot + 1));
  if (tot) CUDA_TRY(cudaMemcpyAsync(e->h_ids.p, e->d_ids.p, tot * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaMemcpyAsync(e->h_id_offsets.p, e->d_id_offsets.p, (n + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
  e->last_d2h = tot * sizeof(int32_t) + (n + 1) * sizeof(uint64_t);
  if (spans) {
    CUDA_TRY(e->h_tok_end.ensure(tot + 1));
    CUDA_TRY(e->h_norm.ensure(totn + 1));
    CUDA_TRY(e->h_n2o.ensure(totn + 1));
    CUDA_TRY(e->h_norm_offsets.ensure(n + 1));
    if (tot) CUDA_TRY(cudaMemcpyAsync(e->h_tok_end.p, e->d_tok_end.p, tot * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(e->h_norm.p, e->d_norm.p, totn, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(e->h_n2o.p, e->d_n2o.p, totn * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(e->h_norm_offsets.p, e->d_norm_offsets.p, (n + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    e->last_d2h += tot * 4 + totn * 5 + (n + 1) * 8;
  }
  CUDA_TRY(cudaStreamSynchronize(st));
  finish_timing(e);
  *ids = e->h_ids.p;
  *id_offsets = e->h_id_offsets.p;
  if (spans) {
    *tok_end = e->h_tok_end.p;
    *normalized = reinterpret_cast<const char *>(e->h_norm.p);
    *norm_offsets = e->h_norm_offsets.p;
    *n2o = e->h_n2o.p;
  }
  return SPM_OK;
}

static int encode_host_locked(spm_engine *e, const char *bytes, const uint64_t *offsets, size_t n, bool spans,
                              const int32_t **ids, const uint32_t **tok_end, const uint64_t **id_offsets,
                              const char **normalized, const uint64_t **norm_offsets, const uint32_t **n2o);

// spm_encode_ids with e->mu already held (also used by the n-best / sampling entry points for nbest_size <= 1)
static int encode_ids_locked(spm_engine *e, const char *bytes, const uint64_t *offsets, size_t n, const int32_t **ids,
                             const uint64_t **id_offsets) {
  if (offsets && bytes && e->model.model_type == SPM_UNIGRAM && n < 0xFFFFFFF0ull && offsets[n] >= offsets[0])
    e->batch_fast_words = e->pick_fast_words_host(bytes, offsets, n);
  if (offsets && ids && id_offsets && bytes && n >= e->pipeline_min_sentences && n < 0xFFFFFFF0ull) {
    if (e->uses_lane_kernel() && e->sort_by_length && e->fused_host_path) {
      if (e->fused_skip > 0) --e->fused_skip;
      else return e->encode_host_fused(bytes, offsets, n, ids, id_offsets);
    }
    if (e->uses_lane_kernel()) return e->encode_host_streamed(bytes, offsets, n, ids, id_offsets);
    return e->encode_host_pipelined(bytes, offsets, n, ids, id_offsets);
  }
  return encode_host_locked(e, bytes, offsets, n, false, ids, nullptr, id_offsets, nullptr, nullptr, nullptr);
}

int spm_encode_ids(spm_engine *e, const char *bytes, const uint64_t *offsets, size_t n, const int32_t **ids,
                   const uint64_t **id_offsets) {
  if (!e) return SPM_ERR_ARG;
  std::lock_guard<std::mutex> lk(e->mu);
  return encode_ids_locked(e, bytes, offsets, n, ids, id_offsets);
}

static int nbest_args_ok(spm_engine *e, const char *bytes, const uint64_t *offsets, size_t n) {
  if (e->model.model_type != SPM_UNIGRAM) {
    e->set_error("NBestEncode is not available for the current model.");  // sentencepiece_processor.cc:662-663
    return SPM_ERR_UNSUPPORTED;
  }
  if (!offsets || (n && !bytes && offsets[n] != offsets[0]) || n >= 0x7FFFFFF0ull) { e->set_error("bad argument"); return SPM_ERR_ARG; }
  for (size_t i = 0; i < n; ++i)
    if (offsets[i + 1] < offsets[i]) { e->set_error("offsets must be non-decreasing"); return SPM_ERR_ARG; }
  if (e->trie.max_key_len > 255) { e->set_error("pieces too long for the n-best device path"); return SPM_ERR_UNSUPPORTED; }
  return SPM_OK;
}

int spm_set_random_seed(spm_engine *e, uint32_t seed) {
  if (!e) return SPM_ERR_ARG;
  std::lock_guard<std::mutex> lk(e->mu);
  e->rng.seed(seed);
  return SPM_OK;
}

int spm_nbest_encode(spm_engine *e, const char *bytes, const uint64_t *offsets, size_t n, int nbest_size,
                     const int32_t **ids, const uint64_t **cand_offsets, const float **scores, const uint32_t **n_cands) {
  if (!e || !ids || !cand_offsets || !scores || !n_cands) return SPM_ERR_ARG;
  std::lock_guard<std::mutex> lk(e->mu);
  auto set_error = [&](const std::string &m) { e->set_error(m); };
  { const int rc = nbest_args_ok(e, bytes, offsets, n); if (rc) return rc; }
  CUDA_TRY(cudaSetDevice(e->device));
  const uint32_t K = static_cast<uint32_t>(std::max(1, std::min(nbest_size, 1024)));  // unigram_model.cc:701
  cudaStream_t st = e->stream;
  const size_t nc = n * static_cast<size_t>(K);
  if (nc >= 0xFFFFFFF0ull) { e->set_error("n-best: sentences x nbest_size must stay below 2^32; split the batch"); return SPM_ERR_ARG; }
  CUDA_TRY(e->h_cand_offsets.ensure(nc + 1));
  CUDA_TRY(e->h_cand_score.ensure(nc + 1));
  CUDA_TRY(e->h_n_cands.ensure(n + 1));
  CUDA_TRY(e->h_ids.ensure(1));
  *ids = e->h_ids.p; *cand_offsets = e->h_cand_offsets.p; *scores = e->h_cand_score.p; *n_cands = e->h_n_cands.p;
  e->h_cand_offsets.p[0] = 0;
  if (n == 0) return SPM_OK;
  e->last_launches = 0;
  if (K == 1) {
    // nbest_size <= 1: {Encode(normalized), 0.0} (unigram_model.cc:703-705)
    const int32_t *pid; const uint64_t *poff;
    const int rc = encode_ids_locked(e, bytes, offsets, n, &pid, &poff);
    if (rc) return rc;
    for (size_t i = 0; i <= n; ++i) e->h_cand_offsets.p[i] = poff[i];
    for (size_t i = 0; i < n; ++i) { e->h_cand_score.p[i] = 0.f; e->h_n_cands.p[i] = 1; }
    *ids = pid;
    return SPM_OK;
  }
  uint64_t tmp_total = 0;
  { const int rc = e->run_nbest(bytes, offsets, n, K, &tmp_total); if (rc) return rc; }
  // candidate-major compaction: the shared scan + gather over n*K counts
  const uint32_t nc32 = static_cast<uint32_t>(nc);
  const uint32_t nb = (nc32 + kScanChunk - 1) / kScanChunk;
  CUDA_TRY(e->d_block_sums.ensure(nb + 1));
  CUDA_TRY(e->d_cand_offsets.ensure(nc + 1));
  CUDA_TRY(e->d_ids.ensure(tmp_total + 1));
  scan_block_sums_kernel<<<nb, 256, 0, st>>>(e->d_cand_count.p, nc32, e->d_block_sums.p, 0);
  scan_block_prefix_kernel<<<1, 1024, 0, st>>>(e->d_block_sums.p, nb, e->d_ctrl64.p + 2);
  scan_write_gather_kernel<int32_t><<<nb, 256, 0, st>>>(e->d_cand_count.p, nc32, e->d_block_sums.p, e->d_cand_offsets.p,
                                                        e->d_cand_start.p, e->d_tmp_ids.p, e->d_ids.p, nullptr, nullptr,
                                                        e->d_ids.cap, 0, 0ull);
  CUDA_TRY(cudaGetLastError());
  e->last_launches += 3;
  CUDA_TRY(e->h_ids.ensure(tmp_total + 1));
  if (tmp_total) CUDA_TRY(cudaMemcpyAsync(e->h_ids.p, e->d_ids.p, tmp_total * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaMemcpyAsync(e->h_cand_offsets.p, e->d_cand_offsets.p, (nc + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaMemcpyAsync(e->h_cand_score.p, e->d_cand_score.p, nc * sizeof(float), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaMemcpyAsync(e->h_n_cands.p, e->d_n_cands.p, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaEventRecord(e->ev[2], st));
  CUDA_TRY(cudaStreamSynchronize(st));
  e->last_d2h = tmp_total * 4 + (nc + 1) * 8 + nc * 4 + n * 4;
  finish_timing(e);
  *ids = e->h_ids.p;
  return SPM_OK;
}

int spm_sample_encode_ids(spm_engine *e, const char *bytes, const uint64_t *offsets, size_t n, int nbest_size,
                          float alpha, const int32_t **ids, const uint64_t **id_offsets) {
  if (!e || !ids || !id_offsets) return SPM_ERR_ARG;
  std::lock_guard<std::mutex> lk(e->mu);
  if (nbest_size > 512) { e->set_error("nbest_size must be nbest_size <= 512"); return SPM_ERR_ARG; }  // :683
  if (e->model.model_type != SPM_UNIGRAM) {
    // models without NBestEncode go to Model::SampleEncode(normalized, alpha) whatever nbest_size is (:689-693): for
    // BPE that is BPE-dropout, which equals Encode only for alpha <= 0 (bpe_model.cc:132-139)
    if (alpha > 0.f) {
      e->set_error("SampleEncode: BPE-dropout (alpha > 0) is not on the accelerated path");
      return SPM_ERR_UNSUPPORTED;
    }
    return encode_ids_locked(e, bytes, offsets, n, ids, id_offsets);
  }
  if (nbest_size < 0) {
    // forward-filtering / backward-sampling over the whole lattice (unigram_model.cc:511-542)
    { const int rc = nbest_args_ok(e, bytes, offsets, n); if (rc) return rc; }
    if (cudaSetDevice(e->device) != cudaSuccess) { e->set_error("cudaSetDevice failed"); return SPM_ERR_CUDA; }
    const int rc = e->run_lattice(bytes, offsets, n, alpha, 0, 1);
    if (rc) return rc;
    if (e->lat_ids.empty()) e->lat_ids.reserve(1);
    *ids = e->lat_ids.data();
    *id_offsets = e->lat_offsets.data();
    return SPM_OK;
  }
  if (nbest_size <= 1) return encode_ids_locked(e, bytes, offsets, n, ids, id_offsets);  // :695-698
  auto set_error = [&](const std::string &m) { e->set_error(m); };
  { const int rc = nbest_args_ok(e, bytes, offsets, n); if (rc) return rc; }
  CUDA_TRY(cudaSetDevice(e->device));
  cudaStream_t st = e->stream;
  const uint32_t K = static_cast<uint32_t>(nbest_size);
  CUDA_TRY(e->h_id_offsets.ensure(n + 1));
  CUDA_TRY(e->h_ids.ensure(1));
  *ids = e->h_ids.p; *id_offsets = e->h_id_offsets.p;
  e->h_id_offsets.p[0] = 0;
  if (n == 0) return SPM_OK;
  e->last_launches = 0;
  uint64_t tmp_total = 0;
  { const int rc = e->run_nbest(bytes, offsets, n, K, &tmp_total); if (rc) return rc; }
  const size_t nc = n * static_cast<size_t>(K);
  CUDA_TRY(e->h_cand_score.ensure(nc + 1));
  CUDA_TRY(e->h_n_cands.ensure(n + 1));
  CUDA_TRY(e->h_picks.ensure(n + 1));
  CUDA_TRY(cudaMemcpyAsync(e->h_cand_score.p, e->d_cand_score.p, nc * sizeof(float), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaMemcpyAsync(e->h_n_cands.p, e->d_n_cands.p, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  // ---- the draw (sentencepiece_processor.cc:703-718) ----
  // The uniform of sentence i is generate_canonical<double,53>(mt) exactly as
  // std::discrete_distribution::operator() takes it; a sentence with fewer than two candidates
  // draws nothing.  Generated in sentence order on one generator, then the (independent)
  // log-sum-exp / cumulative tables are evaluated by all host threads.
  std::vector<double> u(n, 0.0);
  for (size_t i = 0; i < n; ++i)
    if (e->h_n_cands.p[i] >= 2) u[i] = std::generate_canonical<double, std::numeric_limits<double>::digits>(e->rng);
  const float *sc = e->h_cand_score.p;
  const uint32_t *kc = e->h_n_cands.p;
  uint32_t *picks = e->h_picks.p;
  auto work = [&](size_t lo, size_t hi) {
    std::vector<double> lp(K), cp(K);
    for (size_t i = lo; i < hi; ++i) {
      const uint32_t k = kc[i];
      if (k < 2) { picks[i] = 0; continue; }
      const float *s = sc + i * K;
      for (uint32_t c = 0; c < k; ++c) lp[c] = alpha * s[c];  // float product, widened (:705-706)
      double Z = lp[0];                                       // log_domain::LogSum, util.cc:278-294
      for (uint32_t c = 1; c < k; ++c) {
        double xa = Z, xb = lp[c];
        if (xa > xb) std::swap(xa, xb);
        Z = xb + std::log1p(std::exp(xa - xb));
      }
      double sum = 0.0;
      for (uint32_t c = 0; c < k; ++c) { lp[c] = std::exp(lp[c] - Z); sum += lp[c]; }
      double run = 0.0;  // discrete_distribution::param_type::_M_initialize
      for (uint32_t c = 0; c < k; ++c) { run += lp[c] / sum; cp[c] = run; }
      cp[k - 1] = 1.0;
      picks[i] = static_cast<uint32_t>(std::lower_bound(cp.begin(), cp.begin() + k, u[i]) - cp.begin());
    }
  };
  {
    const size_t T = std::max<size_t>(1, std::min<size_t>(std::thread::hardware_concurrency(), n / 2048 + 1));
    std::vector<std::thread> th;
    const size_t per = (n + T - 1) / T;
    for (size_t t = 1; t < T; ++t) th.emplace_back(work, std::min(n, t * per), std::min(n, (t + 1) * per));
    work(0, std::min(n, per));
    for (auto &t : th) t.join();
  }
  // ---- gather the picked candidates into sentence order ----
  CUDA_TRY(e->d_picks.ensure(n));
  CUDA_TRY(e->d_sent_start.ensure(n));
  CUDA_TRY(e->d_sent_count.ensure(n));
  CUDA_TRY(e->d_id_offsets.ensure(n + 1));
  CUDA_TRY(cudaMemcpyAsync(e->d_picks.p, picks, n * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
  const uint32_t n32 = static_cast<uint32_t>(n);
  pick_candidates_kernel<<<(n32 + 255) / 256, 256, 0, st>>>(e->d_picks.p, n32, K, e->d_cand_start.p, e->d_cand_count.p,
                                                           e->d_sent_start.p, e->d_sent_count.p);
  const uint32_t nb = (n32 + kScanChunk - 1) / kScanChunk;
  CUDA_TRY(e->d_block_sums.ensure(nb + 1));
  scan_block_sums_kernel<<<nb, 256, 0, st>>>(e->d_sent_count.p, n32, e->d_block_sums.p, 0);
  scan_block_prefix_kernel<<<1, 1024, 0, st>>>(e->d_block_sums.p, nb, e->d_ctrl64.p + 2);
  CUDA_TRY(cudaMemcpyAsync(e->h_ctrl64.p, e->d_ctrl64.p, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  const unsigned long long tot = e->h_ctrl64.p[2];
  CUDA_TRY(e->d_ids.ensure(tot + 1));
  scan_write_gather_kernel<int32_t><<<nb, 256, 0, st>>>(e->d_sent_count.p, n32, e->d_block_sums.p, e->d_id_offsets.p,
                                                        e->d_sent_start.p, e->d_tmp_ids.p, e->d_ids.p, nullptr, nullptr,
                                                        e->d_ids.cap, 0, 0ull);
  CUDA_TRY(cudaGetLastError());
  e->last_launches += 4;
  CUDA_TRY(e->h_ids.ensure(tot + 1));
  if (tot) CUDA_TRY(cudaMemcpyAsync(e->h_ids.p, e->d_ids.p, tot * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaMemcpyAsync(e->h_id_offsets.p, e->d_id_offsets.p, (n + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaEventRecord(e->ev[2], st));
  CUDA_TRY(cudaStreamSynchronize(st));
  e->last_d2h = nc * 4 + n * 4 + tot * 4 + (n + 1) * 8;
  finish_timing(e);
  *ids = e->h_ids.p;
  *id_offsets = e->h_id_offsets.p;
  return SPM_OK;
}

int spm_calculate_entropy(spm_engine *e, const char *bytes, const uint64_t *offsets, size_t n, float alpha,
                          const float **entropy) {
  if (!e || !entropy) return SPM_ERR_ARG;
  std::lock_guard<std::mutex> lk(e->mu);
  if (e->model.model_type != SPM_UNIGRAM) {
    e->set_error("CalculateEntropy is not available for the current model.");  // sentencepiece_processor.cc:750-751
    return SPM_ERR_UNSUPPORTED;
  }
  { const int rc = nbest_args_ok(e, bytes, offsets, n); if (rc) return rc; }
  if (cudaSetDevice(e->device) != cudaSuccess) { e->set_error("cudaSetDevice failed"); return SPM_ERR_CUDA; }
  if (e->h_lat_entropy.ensure(n + 1) != cudaSuccess) { e->set_error("pinned allocation failed"); return SPM_ERR_CUDA; }
  *entropy = e->h_lat_entropy.p;
  if (n == 0) return SPM_OK;
  return e->run_lattice(bytes, offsets, n, alpha, 1, 1);
}

int spm_sample_encode_and_score(spm_engine *e, const char *bytes, const uint64_t *offsets, size_t n, int num_samples,
                                float alpha, int wor, int include_best, const int32_t **ids, const uint64_t **cand_offsets,
                                const float **scores) {
  if (!e || !ids || !cand_offsets || !scores) return SPM_ERR_ARG;
  std::lock_guard<std::mutex> lk(e->mu);
  if (e->model.model_type != SPM_UNIGRAM) {
    e->set_error("SampleEncodeAndScore is not available for the current model.");  // sentencepiece_processor.cc:726-727
    return SPM_ERR_UNSUPPORTED;
  }
  if (wor || include_best) {
    // sampling without replacement runs Lattice::NBest with Gumbel-perturbed scores (unigram_model.cc:770-832)
    e->set_error("SampleEncodeAndScore: wor / include_best are not on the accelerated path");
    return SPM_ERR_UNSUPPORTED;
  }
  if (num_samples < 1 || num_samples > 4096) { e->set_error("num_samples must be in [1, 4096]"); return SPM_ERR_ARG; }
  { const int rc = nbest_args_ok(e, bytes, offsets, n); if (rc) return rc; }
  if (cudaSetDevice(e->device) != cudaSuccess) { e->set_error("cudaSetDevice failed"); return SPM_ERR_CUDA; }
  const int rc = e->run_lattice(bytes, offsets, n, alpha, 0, num_samples);
  if (rc) return rc;
  if (e->lat_ids.empty()) e->lat_ids.reserve(1);
  if (e->lat_scores.empty()) e->lat_scores.reserve(1);
  *ids = e->lat_ids.data();
  *cand_offsets = e->lat_offsets.data();
  *scores = e->lat_scores.data();
  return SPM_OK;
}

int spm_encode_spans(spm_engine *e, const char *bytes, const uint64_t *offsets, size_t n, const int32_t **ids,
                     const uint32_t **tok_end, const uint64_t **id_offsets, const char **normalized,
                     const uint64_t **norm_offsets, const uint32_t **n2o) {
  if (!e || !tok_end || !normalized || !norm_offsets || !n2o) return SPM_ERR_ARG;
  std::lock_guard<std::mutex> lk(e->mu);
  return encode_host_locked(e, bytes, offsets, n, true, ids, tok_end, id_offsets, normalized, norm_offsets, n2o);
}

}  // extern "C"
