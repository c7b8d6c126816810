// Host-side parsers for the two model artefacts of the hot path (SURVEY.md rows a17, a18):
//   * the HuggingFace `tokenizers` JSON written by the reference's scripts/train_bpe.py:68-98
//   * the SentencePiece ModelProto written by scripts/train_spm.py:80-108
// They replace Tokenizer.from_file / SentencePieceProcessor.Load (reference tokenizer.py:88-98) for the CUDA path
// and produce flat tables ready for upload.  No third-party library is used.
#pragma once
#include <stdint.h>
#include <string>
#include <vector>

struct AkBpeHost {
    std::vector<std::string> id_to_token;          // indexed by id ("" where unused)
    std::vector<uint8_t> is_special;               // per id
    std::vector<int32_t> cp_direct;                // [AK_BPE_DIRECT]
    std::vector<uint32_t> cp_keys;
    std::vector<int32_t> cp_ids;
    std::vector<unsigned long long> mkeys, mvals;  // open-addressing table, size 1 << mbits
    uint32_t mbits = 0;
    int32_t bos = -1, eos = -1;
    // pair template `pre $A mid $B post` (post_processor.pair): the ids of each slot; pair_ok = false when the model has
    // a pair template of another shape (then only the pair calls are refused)
    int32_t pair_ids[3][4] = {};
    int pair_n[3] = {0, 0, 0};
    bool pair_ok = true;
    // added tokens (all `special`, matched in the raw text before the normalizer), longest first
    std::vector<uint8_t> sp_bytes;
    std::vector<uint16_t> sp_off;                  // [n + 1]
    std::vector<int32_t> sp_ids;
    int64_t n_merges = 0;
    int vocab_size = 0;
};

struct AkUniHost {
    std::vector<std::string> piece;
    std::vector<float> raw_score;
    std::vector<uint8_t> type;                     // SentencePiece ModelProto.SentencePiece.Type
    std::vector<float> score;                      // effective lattice score per id
    std::vector<uint8_t> usable;
    std::vector<unsigned long long> tkeys, tvals;  // trie edges, size 1 << tbits
    uint32_t tbits = 0;
    int32_t byte_id[256];
    int32_t unk_id = 0;
    float unk_score = 0.f, min_score = 0.f, max_score = 0.f;
    int flags = 0;
    int max_len = 0;
};

// return "" on success, else a one-line description of what is unsupported / malformed
std::string ak_parse_bpe_json(const char* json, size_t len, AkBpeHost& out);
std::string ak_parse_spm_model(const void* proto, size_t len, AkUniHost& out);
