// device_model.h -- POD views shared by the host engine and the kernels.
#ifndef SPM_B200_DEVICE_MODEL_H_
#define SPM_B200_DEVICE_MODEL_H_

#include <cstdint>

#include <vector_types.h>

namespace spm_b200 {

// flags of KModel::flags
enum : uint32_t {
  kFlagAddDummyPrefix = 1u << 0,   // NormalizerSpec.add_dummy_prefix
  kFlagRemoveExtraWs = 1u << 1,    // NormalizerSpec.remove_extra_whitespaces
  kFlagEscapeWs = 1u << 2,         // NormalizerSpec.escape_whitespaces
  kFlagWsSuffix = 1u << 3,         // TrainerSpec.treat_whitespace_as_suffix
  kFlagByteFallback = 1u << 4,     // TrainerSpec.byte_fallback
  kFlagHasUserSymbols = 1u << 5,   // PrefixMatcher trie is non-empty
  kFlagHasCharsmap = 1u << 6,
  kFlagBpeWordSplit = 1u << 7,     // no piece has U+2581 past byte 0 (SURVEY 7 "exact decomposition")
  kFlagHasUnused = 1u << 8,        // some piece is currently UNUSED (SetVocabulary)
  kFlagFastWords = 1u << 10,       // KModel::word_safe is valid (whole-word shortcut of the unigram lane kernel)
  kFlagRegularScores = 1u << 9,    // every piece score is 0 or has 2^-10 <= |score| <= 2^10 (exact float fold)
};

constexpr uint32_t kValUserDefined = 0xFFFFFFFEu;  // match-buffer marker: USER_DEFINED piece
constexpr uint32_t kValUnk = 0xFFFFFFFDu;          // match-buffer marker: UNK edge
constexpr uint32_t kIdxUnk = 0xFFFFFFFFu;          // DP back-pointer marker: UNK piece
constexpr uint32_t kNoUnit = 0xFFFFFFFFu;          // KModel::ws_unit: no such trie unit

// Read-only model tables resident in HBM (all L2-resident after first touch:
// ~1 MB per model).  Pointers are device pointers.
struct KModel {
  // piece trie (trie_builder.h format)
  const uint32_t *trie_link;
  const uint32_t *trie_val;
  const int32_t *trie_id;
  const uint2 *trie_node2;  // {link, child mask} interleaved (one 8-byte load per transition)
  // {link, child mask, score bits, word_safe} (unigram lane kernel: one 16-byte load per transition brings the piece
  // score and the whole-word limit along, so neither costs a second dependent lookup)
  const uint4 *trie_node4;
  uint32_t trie_units;
  uint32_t hot_link;   // units of trie_link staged into shared memory by each CTA (multiple of 4)
  uint32_t hot_val;    // units of trie_val staged (multiple of 4)
  uint32_t match_slots;  // K: match-buffer slots per lane = max prefixes per start + 1 (UNK edge)
  // user-defined-symbol matcher (PrefixMatcher, normalizer.cc:311-346), same link format
  const uint32_t *user_link;
  // precompiled charsmap: Darts units verbatim + NUL-separated targets (normalizer.cc:274-309)
  const uint32_t *cm_units;
  uint32_t cm_nunits;
  const uint8_t *cm_targets;
  // ASCII fast path tables derived from the charsmap at load:
  //   cm_lead[b>>5] bit (b&31): the charsmap root has a transition on byte b
  //   cm_pair[(b*256+c)>>5] bit: root->b->c exists, for b < 128
  //   cm_solo[b]: target offset of the rule whose key is exactly the byte b (b < 128), or -1
  const uint32_t *cm_lead;
  const uint32_t *cm_pair;
  const int32_t *cm_solo;
  const int32_t *byte_to_id;  // [256] PieceToId(ByteToPiece(b)), sentencepiece_processor.cc:587-588
  const float *scores;        // [vocab] (BPE: score of a piece id)
  const uint8_t *types;       // [vocab] live piece types
  // [trie_units] whole-word shortcut (lane_kernel.cuh): a word that is exactly the piece at this unit and ends at a normalized
  // byte position <= word_safe[unit] is certain to be encoded as that piece alone (0 = never); see engine.cu
  const uint16_t *word_safe;
  // unigram lane kernel: trie unit of the piece path "U+2581" and its node4 entry {link, score bits, word_safe} when a
  // walk from a U+2581 may start on that node (the nodes of E2 and E2 96 are no pieces); ws_unit = kNoUnit otherwise
  uint32_t ws_unit, ws_link, ws_score, ws_safe;
  // [trie_units] BPE lane2 kernel: vocab id of the piece at this unit when a word that is exactly the piece encodes
  // to that single id (its merge sequence reproduces it), else 0xFFFFFFFF
  const uint32_t *word_fast;
  // BPE lane2 kernel: word cache in HBM (bpe_lane2_kernel.cuh, "word cache"): bpe_cache_mask + 1 entries of 64 bytes,
  // filled by the kernels themselves; mask 0 = no cache
  uint4 *bpe_cache;
  uint32_t bpe_cache_mask;
  int32_t unk_id;
  float unk_score;  // min_score_ - kUnkPenalty, unigram_model.cc:955
  float max_score;  // unigram_model.cc:658-663 (FLT_MIN quirk)
  uint32_t flags;
  int32_t model_type;
};

// One batch.
struct KBatch {
  const uint8_t *bytes;
  const uint64_t *offsets;  // [n+1]
  uint32_t n;
  // sentences whose [offset, offset + length) does not lie inside [off_lo, off_hi] are not touched by the lane
  // kernels (deferred; the host validates the offsets and reports the error): a batch with broken offsets must
  // not make the kernel read outside the batch's buffer
  unsigned long long off_lo, off_hi;
  const uint32_t *order;    // lane kernels: processing order (a permutation of 0..n-1), or null = input order
  // streamed host batches: *ready = sentences of the whole batch whose bytes have arrived (input order);
  // this launch covers sentences ready_base .. ready_base + n, which arrive in pieces of 2^piece_shift
  const uint32_t *ready;
  uint32_t ready_base, piece_shift;
  // fused host path (drain.cuh): segments of 2^seg_shift sentences are compacted by the warp that finishes them
  uint32_t seg_shift;
  uint32_t *seg_done;                 // [segments] groups finished, or null = no in-kernel compaction
  unsigned long long *seg_total;      // [segments] flag | ids of the segment
  unsigned long long *seg_prefix;     // [segments] flag | ids up to and including the segment
  uint32_t *sent_rel;                 // [n] scratch: offset of a sentence's ids inside its segment
  int32_t *out_ids;                   // result buffers (pinned host memory in the fused path)
  unsigned long long *out_offsets;    // [n+1]
  unsigned long long out_cap, out_off_base;
  // progress of the compaction for the host's DMA loop: segments [0, *drained_upto) are final in out_ids; the warp
  // that advances the counter stores the id count of that prefix to *host_progress (pinned host memory)
  uint32_t *seg_copied;               // [segments]
  uint32_t *drained_upto;
  unsigned long long *host_progress;
  uint32_t slab_discard;              // lane kernels: discard.L2 the used slab rows at the end of a group (lane_kernel.cuh)
  uint32_t slab_l2;                   // L2 eviction priority of the lane kernels' slab accesses: 0 normal, 1 evict_last, 2 evict_first
  unsigned long long *kstats;         // [4] cycles (lane 0 of each warp): input wait, compaction, look-back wait, groups; or null
  // outputs of the encode kernel
  int32_t *tmp_ids;              // ids in completion order
  uint32_t *tmp_tok_end;         // (spans) token end offsets in normalized text, same positions
  unsigned long long tmp_cap;
  unsigned long long *cursor;    // [0] ids cursor, [1] normalized-bytes cursor
  unsigned long long *sent_start;  // [n] start of sentence i's ids in tmp_ids
  uint32_t *sent_count;          // [n]
  uint8_t *tmp_norm;             // (spans) normalized text in completion order
  uint32_t *tmp_n2o;             // (spans) norm_to_orig, (len+1) entries per sentence
  unsigned long long tmp_norm_cap;
  unsigned long long *norm_start;  // (spans) [n]
  uint32_t *norm_len;            // (spans) [n]
  uint32_t *work_counter;
  uint32_t *deferred;            // list of sentence indices that did not fit shared memory
  uint32_t *status;              // [0] deferred count, [1] error flag, [2] overflow flag
  // long-sentence path: sentence list + per-entry scratch slab
  // second-chance pass over the sentences a lane kernel deferred: (sentence, need) pairs
  const uint32_t *sub_list;
  uint32_t sub_n;
  const uint32_t *long_list;
  uint32_t long_n;
  uint8_t *long_scratch;
  const unsigned long long *long_scratch_off;  // [long_n+1]
  // shared-memory geometry
  uint32_t ncap;        // normalized-byte capacity per tile
  uint32_t tile_bytes;  // bytes of scratch per tile
};

}  // namespace spm_b200
#endif
