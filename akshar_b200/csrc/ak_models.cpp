// see ak_models.h
#include "ak_models.h"

#include <algorithm>
#include <math.h>
#include <string.h>

#include <map>
#include <memory>
#include <unordered_map>

#define AK_BPE_DIRECT 0x0A00
#define AK_EMPTY_KEY 0xFFFFFFFFFFFFFFFFull
#define AK_MAX_TOKEN_ID (1 << 24)      // ids index host vectors and device tables

namespace {

// ------------------------------------------------------------------------------------------------
// minimal JSON DOM
// ------------------------------------------------------------------------------------------------
struct JVal {
    enum Kind { Null, Bool, Num, Str, Arr, Obj } kind = Null;
    bool b = false;
    double num = 0;
    std::string str;
    std::vector<JVal> arr;
    std::vector<std::pair<std::string, JVal>> obj;
    const JVal* get(const char* key) const {
        if (kind != Obj) return nullptr;
        for (auto& kv : obj)
            if (kv.first == key) return &kv.second;
        return nullptr;
    }
    bool is_null() const { return kind == Null; }
};

struct JParser {
    const char* p;
    const char* end;
    std::string err;
    int depth = 0;

    void ws() { while (p < end && (*p == ' ' || *p == '\n' || *p == '\t' || *p == '\r')) ++p; }
    bool fail(const char* m) { if (err.empty()) err = m; return false; }

    static void put_utf8(std::string& s, uint32_t cp) {
        if (cp < 0x80) s.push_back((char)cp);
        else if (cp < 0x800) { s.push_back((char)(0xC0 | (cp >> 6))); s.push_back((char)(0x80 | (cp & 63))); }
        else if (cp < 0x10000) {
            s.push_back((char)(0xE0 | (cp >> 12))); s.push_back((char)(0x80 | ((cp >> 6) & 63))); s.push_back((char)(0x80 | (cp & 63)));
        } else {
            s.push_back((char)(0xF0 | (cp >> 18))); s.push_back((char)(0x80 | ((cp >> 12) & 63)));
            s.push_back((char)(0x80 | ((cp >> 6) & 63))); s.push_back((char)(0x80 | (cp & 63)));
        }
    }
    bool hex4(uint32_t& v) {
        if (end - p < 4) return fail("bad \\u escape");
        v = 0;
        for (int i = 0; i < 4; ++i) {
            char c = *p++;
            v <<= 4;
            if (c >= '0' && c <= '9') v |= (uint32_t)(c - '0');
            else if (c >= 'a' && c <= 'f') v |= (uint32_t)(c - 'a' + 10);
            else if (c >= 'A' && c <= 'F') v |= (uint32_t)(c - 'A' + 10);
            else return fail("bad \\u escape");
        }
        return true;
    }
    bool string(std::string& s) {
        if (p >= end || *p != '"') return fail("expected string");
        ++p;
        while (p < end && *p != '"') {
            if (*p == '\\') {
                ++p;
                if (p >= end) return fail("bad escape");
                char c = *p++;
                switch (c) {
                    case '"': s.push_back('"'); break;
                    case '\\': s.push_back('\\'); break;
                    case '/': s.push_back('/'); break;
                    case 'b': s.push_back('\b'); break;
                    case 'f': s.push_back('\f'); break;
                    case 'n': s.push_back('\n'); break;
                    case 'r': s.push_back('\r'); break;
                    case 't': s.push_back('\t'); break;
                    case 'u': {
                        uint32_t v;
                        if (!hex4(v)) return false;
                        if (v >= 0xD800 && v < 0xDC00 && end - p >= 6 && p[0] == '\\' && p[1] == 'u') {
                            const char* save = p;
                            p += 2;
                            uint32_t lo;
                            if (!hex4(lo)) return false;
                            if (lo >= 0xDC00 && lo < 0xE000) v = 0x10000 + ((v - 0xD800) << 10) + (lo - 0xDC00);
                            else p = save;
                        }
                        put_utf8(s, v);
                        break;
                    }
                    default: return fail("bad escape");
                }
            } else {
                s.push_back(*p++);
            }
        }
        if (p >= end) return fail("unterminated string");
        ++p;
        return true;
    }
    bool value(JVal& v) {
        if (++depth > 64) return fail("nesting too deep");
        ws();
        if (p >= end) return fail("unexpected end");
        bool ok = true;
        if (*p == '{') {
            v.kind = JVal::Obj;
            ++p;
            ws();
            if (p < end && *p == '}') ++p;
            else {
                for (;;) {
                    ws();
                    std::string k;
                    if (!string(k)) { ok = false; break; }
                    ws();
                    if (p >= end || *p != ':') { ok = fail("expected ':'"); break; }
                    ++p;
                    v.obj.emplace_back(std::move(k), JVal());
                    if (!value(v.obj.back().second)) { ok = false; break; }
                    ws();
                    if (p < end && *p == ',') { ++p; continue; }
                    if (p < end && *p == '}') { ++p; break; }
                    ok = fail("expected ',' or '}'");
                    break;
                }
            }
        } else if (*p == '[') {
            v.kind = JVal::Arr;
            ++p;
            ws();
            if (p < end && *p == ']') ++p;
            else {
                for (;;) {
                    v.arr.emplace_back();
                    if (!value(v.arr.back())) { ok = false; break; }
                    ws();
                    if (p < end && *p == ',') { ++p; continue; }
                    if (p < end && *p == ']') { ++p; break; }
                    ok = fail("expected ',' or ']'");
                    break;
                }
            }
        } else if (*p == '"') {
            v.kind = JVal::Str;
            ok = string(v.str);
        } else if (end - p >= 4 && !memcmp(p, "true", 4)) { v.kind = JVal::Bool; v.b = true; p += 4; }
        else if (end - p >= 5 && !memcmp(p, "false", 5)) { v.kind = JVal::Bool; v.b = false; p += 5; }
        else if (end - p >= 4 && !memcmp(p, "null", 4)) { v.kind = JVal::Null; p += 4; }
        else {
            const char* s = p;
            while (p < end && (*p == '-' || *p == '+' || *p == '.' || *p == 'e' || *p == 'E' || (*p >= '0' && *p <= '9'))) ++p;
            if (p == s) ok = fail("unexpected character");
            else { v.kind = JVal::Num; v.num = strtod(std::string(s, p).c_str(), nullptr); }
        }
        --depth;
        return ok;
    }
};

bool decode_one_cp(const std::string& s, uint32_t& cp) {
    const unsigned char* u = (const unsigned char*)s.data();
    size_t n = s.size();
    if (n == 0) return false;
    size_t need = u[0] < 0x80 ? 1 : u[0] >= 0xF0 ? 4 : u[0] >= 0xE0 ? 3 : u[0] >= 0xC0 ? 2 : 0;
    if (need == 0 || need != n) return false;
    cp = need == 1 ? u[0] : (u[0] & (0xFFu >> (need + 1)));
    for (size_t i = 1; i < need; ++i) cp = (cp << 6) | (u[i] & 0x3Fu);
    return true;
}

inline uint32_t hash64(unsigned long long k, uint32_t bits) {
    return (uint32_t)((k * 0x9E3779B97F4A7C15ull) >> (64 - bits));
}

void table_insert(std::vector<unsigned long long>& keys, std::vector<unsigned long long>& vals, uint32_t bits,
                  unsigned long long key, unsigned long long val) {
    uint32_t mask = (1u << bits) - 1u;
    uint32_t h = hash64(key, bits);
    while (keys[h] != AK_EMPTY_KEY && keys[h] != key) h = (h + 1) & mask;
    keys[h] = key;
    vals[h] = val;
}

const char* type_of(const JVal* v) {
    if (!v || v->is_null()) return "";
    const JVal* t = v->get("type");
    return (t && t->kind == JVal::Str) ? t->str.c_str() : "?";
}

}  // namespace

std::string ak_parse_bpe_json(const char* json, size_t len, AkBpeHost& out) {
    JParser P{json, json + len, "", 0};
    JVal root;
    if (!P.value(root)) return "tokenizer JSON: " + P.err;
    const JVal* model = root.get("model");
    if (!model || strcmp(type_of(model), "BPE")) return "tokenizer JSON: model.type is not BPE";
    // only the configuration scripts/train_bpe.py:68-98 produces is implemented; anything else is refused loudly
    const char* nt = type_of(root.get("normalizer"));
    if (strcmp(nt, "NFKC") && strcmp(nt, "NFC") && strcmp(nt, "")) return std::string("unsupported normalizer ") + nt;
    const char* pt = type_of(root.get("pre_tokenizer"));
    if (strcmp(pt, "Whitespace")) return std::string("unsupported pre_tokenizer '") + pt + "'";
    if (root.get("decoder") && !root.get("decoder")->is_null()) return "unsupported decoder (expected null)";
    for (const char* k : {"unk_token", "dropout", "continuing_subword_prefix", "end_of_word_suffix"}) {
        const JVal* v = model->get(k);
        if (v && !v->is_null() && !(v->kind == JVal::Str && v->str.empty())) return std::string("unsupported model.") + k;
    }
    for (const char* k : {"byte_fallback", "ignore_merges"}) {
        const JVal* v = model->get(k);
        if (v && v->kind == JVal::Bool && v->b) return std::string("unsupported model.") + k;
    }
    const JVal* vocab = model->get("vocab");
    const JVal* merges = model->get("merges");
    if (!vocab || vocab->kind != JVal::Obj || !merges || merges->kind != JVal::Arr) return "tokenizer JSON: vocab / merges missing";
    std::unordered_map<std::string, int32_t> v2i;
    int32_t max_id = -1;
    // ids index host vectors and device tables: integral, non-negative, bounded -- anything else is a malformed model
    auto id_of = [](const JVal& v, int32_t& id) -> bool {
        if (v.kind != JVal::Num || !(v.num >= 0.0) || v.num > (double)AK_MAX_TOKEN_ID || v.num != (double)(int64_t)v.num) return false;
        id = (int32_t)v.num;
        return true;
    };
    for (auto& kv : vocab->obj) {
        int32_t id;
        if (!id_of(kv.second, id)) return "tokenizer JSON: vocab id is not an integer in [0, 2^24]";
        v2i[kv.first] = id;
        if (id > max_id) max_id = id;
    }
    std::vector<std::pair<std::string, int32_t>> specials;
    if (const JVal* added = root.get("added_tokens")) {
        if (added->kind == JVal::Arr)
            for (auto& a : added->arr) {
                const JVal* c = a.get("content");
                const JVal* i = a.get("id");
                int32_t id;
                if (!c || !i || c->kind != JVal::Str || !id_of(*i, id)) return "tokenizer JSON: bad added_tokens entry";
                // the matcher implemented on the device is the plain one: no word-boundary / strip options, raw text
                for (const char* opt : {"single_word", "lstrip", "rstrip", "normalized"}) {
                    const JVal* o = a.get(opt);
                    if (o && o->kind == JVal::Bool && o->b) return std::string("tokenizer JSON: added token option '") + opt + "' is not supported";
                }
                if (c->str.empty() || c->str.size() > 255) return "tokenizer JSON: bad added_tokens content";
                specials.emplace_back(c->str, id);
                const JVal* sp = a.get("special");
                if (sp && sp->kind == JVal::Bool && sp->b) out.special_ids.push_back(id);
                if (id > max_id) max_id = id;
            }
    }
    {
        std::vector<std::pair<std::string, int32_t>> by_len = specials;
        std::stable_sort(by_len.begin(), by_len.end(), [](const std::pair<std::string, int32_t>& x, const std::pair<std::string, int32_t>& y) {
            return x.first.size() > y.first.size();
        });
        out.sp_off.push_back(0);
        for (auto& sp : by_len) {
            out.sp_bytes.insert(out.sp_bytes.end(), sp.first.begin(), sp.first.end());
            out.sp_off.push_back((uint16_t)out.sp_bytes.size());
            out.sp_ids.push_back(sp.second);
        }
        if (out.sp_bytes.size() > 60000 || out.sp_ids.size() > 255) return "tokenizer JSON: too many added tokens";
    }
    out.id_to_token.assign((size_t)max_id + 1, "");
    out.is_special.assign((size_t)max_id + 1, 0);
    for (auto& kv : v2i) out.id_to_token[(size_t)kv.second] = kv.first;
    for (auto& s : specials) { out.id_to_token[(size_t)s.second] = s.first; out.is_special[(size_t)s.second] = 1; }
    {
        std::map<int32_t, int> ids;
        for (auto& kv : v2i) ids[kv.second] = 1;
        for (auto& s : specials) ids[s.second] = 1;
        out.vocab_size = (int)ids.size();
    }
    // single-character tokens
    out.cp_direct.assign(AK_BPE_DIRECT, -1);
    std::map<uint32_t, int32_t> far;
    for (auto& kv : v2i) {
        uint32_t cp;
        if (!decode_one_cp(kv.first, cp)) continue;
        bool special = false;
        for (auto& s : specials) special |= (s.first == kv.first);
        if (special) continue;
        if (cp < AK_BPE_DIRECT) out.cp_direct[cp] = kv.second;
        else far[cp] = kv.second;
    }
    for (auto& kv : far) { out.cp_keys.push_back(kv.first); out.cp_ids.push_back(kv.second); }
    // merges
    size_t nm = merges->arr.size();
    out.n_merges = (int64_t)nm;
    out.mbits = 4;
    while ((1ull << out.mbits) < 2 * nm + 16) ++out.mbits;
    out.mkeys.assign((size_t)1 << out.mbits, AK_EMPTY_KEY);
    out.mvals.assign((size_t)1 << out.mbits, 0);
    for (size_t r = 0; r < nm; ++r) {
        const JVal& m = merges->arr[r];
        std::string a, b;
        if (m.kind == JVal::Str) {
            size_t sp = m.str.find(' ');
            if (sp == std::string::npos) return "tokenizer JSON: bad merge entry";
            a = m.str.substr(0, sp);
            b = m.str.substr(sp + 1);
        } else if (m.kind == JVal::Arr && m.arr.size() == 2 && m.arr[0].kind == JVal::Str && m.arr[1].kind == JVal::Str) {
            a = m.arr[0].str;
            b = m.arr[1].str;
        } else {
            return "tokenizer JSON: bad merge entry";
        }
        auto ia = v2i.find(a), ib = v2i.find(b), ic = v2i.find(a + b);
        if (ia == v2i.end() || ib == v2i.end() || ic == v2i.end()) return "tokenizer JSON: merge refers to a token outside the vocab";
        unsigned long long key = ((unsigned long long)(uint32_t)ia->second << 32) | (uint32_t)ib->second;
        // the first (lowest-rank) entry of a duplicated pair wins, as in HF's HashMap construction order... keep first
        uint32_t mask = (1u << out.mbits) - 1u, h = hash64(key, out.mbits);
        bool dup = false;
        while (out.mkeys[h] != AK_EMPTY_KEY) {
            if (out.mkeys[h] == key) { dup = true; break; }
            h = (h + 1) & mask;
        }
        if (dup) continue;
        table_insert(out.mkeys, out.mvals, out.mbits, key, ((unsigned long long)r << 32) | (uint32_t)ic->second);
    }
    // <s> $A </s> template (scripts/train_bpe.py:87-94)
    const JVal* pp = root.get("post_processor");
    if (pp && !pp->is_null()) {
        if (strcmp(type_of(pp), "TemplateProcessing")) return std::string("unsupported post_processor ") + type_of(pp);
        const JVal* single = pp->get("single");
        const JVal* st = pp->get("special_tokens");
        if (!single || single->kind != JVal::Arr || !st) return "tokenizer JSON: bad TemplateProcessing";
        int seq_at = -1;
        for (size_t i = 0; i < single->arr.size(); ++i)
            if (single->arr[i].get("Sequence")) seq_at = (int)i;
        if (seq_at < 0 || single->arr.size() > 3) return "unsupported TemplateProcessing layout";
        auto special_id = [&](const JVal& item, int32_t& id) -> bool {
            const JVal* sp = item.get("SpecialToken");
            if (!sp) return false;
            const JVal* nm_ = sp->get("id");
            if (!nm_ || nm_->kind != JVal::Str) return false;
            const JVal* ent = st->get(nm_->str.c_str());
            if (!ent) return false;
            const JVal* ids = ent->get("ids");
            if (!ids || ids->kind != JVal::Arr || ids->arr.size() != 1) return false;
            // the template's ids are emitted as they are: they must name tokens of this vocabulary
            if (!id_of(ids->arr[0], id) || id > max_id || out.id_to_token[(size_t)id].empty()) return false;
            return true;
        };
        if (seq_at == 1 && !special_id(single->arr[0], out.bos)) return "unsupported TemplateProcessing layout";
        if (seq_at + 1 < (int)single->arr.size() && !special_id(single->arr[(size_t)seq_at + 1], out.eos))
            return "unsupported TemplateProcessing layout";
        if (seq_at > 1) return "unsupported TemplateProcessing layout";
        // `pre $A mid $B post` pair template: any other shape leaves the model usable for everything but pairs
        const JVal* pair = pp->get("pair");
        int slot = 0;
        out.pair_ok = pair && pair->kind == JVal::Arr;
        for (size_t i = 0; out.pair_ok && i < pair->arr.size(); ++i) {
            const JVal& item = pair->arr[i];
            const JVal* seq = item.get("Sequence");
            int32_t id = -1;
            if (seq) {
                const JVal* nm_ = seq->get("id");
                const char* want = slot == 0 ? "A" : "B";
                out.pair_ok = slot < 2 && nm_ && nm_->kind == JVal::Str && nm_->str == want;
                ++slot;
            } else if (special_id(item, id) && out.pair_n[slot] < 4) {
                out.pair_ids[slot][out.pair_n[slot]++] = id;
            } else {
                out.pair_ok = false;
            }
        }
        if (slot != 2) out.pair_ok = false;
        if (!out.pair_ok) out.pair_n[0] = out.pair_n[1] = out.pair_n[2] = 0;
    }
    return "";
}

// ------------------------------------------------------------------------------------------------
// SentencePiece ModelProto (protobuf wire format, only the fields the encoder needs)
// ------------------------------------------------------------------------------------------------
namespace {
struct PbReader {
    const uint8_t* p;
    const uint8_t* end;
    bool ok = true;
    bool varint(uint64_t& v) {
        v = 0;
        int shift = 0;
        while (p < end && shift < 64) {
            uint8_t b = *p++;
            v |= (uint64_t)(b & 0x7F) << shift;
            shift += 7;
            if (!(b & 0x80)) return true;
        }
        ok = false;
        return false;
    }
    // next field; for wire type 2 sets [s, s + n)
    bool next(uint32_t& fno, uint32_t& wt, uint64_t& val, const uint8_t*& s, size_t& n) {
        if (p >= end) return false;
        uint64_t key;
        if (!varint(key)) return false;
        fno = (uint32_t)(key >> 3);
        wt = (uint32_t)(key & 7);
        s = nullptr;
        n = 0;
        val = 0;
        if (wt == 0) return varint(val);
        if (wt == 1) { if (end - p < 8) { ok = false; return false; } s = p; n = 8; p += 8; return true; }
        if (wt == 5) { if (end - p < 4) { ok = false; return false; } s = p; n = 4; p += 4; return true; }
        if (wt == 2) {
            uint64_t l;
            if (!varint(l) || (uint64_t)(end - p) < l) { ok = false; return false; }
            s = p;
            n = (size_t)l;
            p += l;
            return true;
        }
        ok = false;
        return false;
    }
};
}  // namespace

std::string ak_parse_spm_model(const void* proto, size_t len, AkUniHost& out) {
    PbReader R{(const uint8_t*)proto, (const uint8_t*)proto + len};
    bool add_dummy = true, remove_extra = true, escape = true, byte_fallback = false;
    int model_type = 1;
    std::string norm_name;
    size_t charsmap_len = 0;
    bool treat_ws_suffix = false;
    uint32_t fno, wt;
    uint64_t val;
    const uint8_t* s;
    size_t n;
    int n_top = 0;
    while (R.next(fno, wt, val, s, n)) {
        ++n_top;
        if (fno == 1 && wt == 2) {
            PbReader P{s, s + n};
            std::string piece;
            float score = 0.f;
            int type = 1;
            uint32_t f2, w2;
            uint64_t v2;
            const uint8_t* s2;
            size_t n2;
            while (P.next(f2, w2, v2, s2, n2)) {
                if (f2 == 1 && w2 == 2) piece.assign((const char*)s2, n2);
                else if (f2 == 2 && w2 == 5) memcpy(&score, s2, 4);
                else if (f2 == 3 && w2 == 0) type = (int)v2;
            }
            if (!P.ok) return "SentencePiece model: malformed piece";
            out.piece.push_back(piece);
            out.raw_score.push_back(score);
            out.type.push_back((uint8_t)type);
        } else if (fno == 2 && wt == 2) {
            PbReader P{s, s + n};
            uint32_t f2, w2;
            uint64_t v2;
            const uint8_t* s2;
            size_t n2;
            while (P.next(f2, w2, v2, s2, n2)) {
                if (f2 == 3 && w2 == 0) model_type = (int)v2;
                else if (f2 == 35 && w2 == 0) byte_fallback = v2 != 0;
                else if (f2 == 24 && w2 == 0) treat_ws_suffix = v2 != 0;
            }
            if (!P.ok) return "SentencePiece model: malformed trainer_spec";
        } else if (fno == 3 && wt == 2) {
            PbReader P{s, s + n};
            uint32_t f2, w2;
            uint64_t v2;
            const uint8_t* s2;
            size_t n2;
            while (P.next(f2, w2, v2, s2, n2)) {
                if (f2 == 1 && w2 == 2) norm_name.assign((const char*)s2, n2);
                else if (f2 == 2 && w2 == 2) charsmap_len = n2;
                else if (f2 == 3 && w2 == 0) add_dummy = v2 != 0;
                else if (f2 == 4 && w2 == 0) remove_extra = v2 != 0;
                else if (f2 == 5 && w2 == 0) escape = v2 != 0;
            }
            if (!P.ok) return "SentencePiece model: malformed normalizer_spec";
        }
    }
    if (!R.ok || out.piece.empty()) return "could not parse ModelProto";
    if (model_type != 1) return "SentencePiece model_type is not UNIGRAM";
    // only the configuration scripts/train_spm.py:80-108 produces is implemented (identity normalization)
    if (charsmap_len != 0) return "unsupported SentencePiece normalization rule '" + norm_name + "' (only identity)";
    if (treat_ws_suffix) return "unsupported treat_whitespace_as_suffix";
    out.flags = (add_dummy ? 1 : 0) | (remove_extra ? 2 : 0) | (escape ? 4 : 0) | (byte_fallback ? 8 : 0);
    size_t np = out.piece.size();
    for (int i = 0; i < 256; ++i) out.byte_id[i] = -1;
    bool have_min = false;
    out.max_score = 0.f;
    bool have_max = false;
    out.unk_id = 0;
    for (size_t i = 0; i < np; ++i) {
        int t = out.type[i];
        if (t == 1) {
            float sc = out.raw_score[i];
            if (!have_min || sc < out.min_score) { out.min_score = sc; have_min = true; }
            if (!have_max || sc > out.max_score) { out.max_score = sc; have_max = true; }
        } else if (t == 2) {
            out.unk_id = (int32_t)i;
        } else if (t == 6) {
            const std::string& p = out.piece[i];
            if (p.size() == 6 && p[0] == '<' && p[1] == '0' && p[2] == 'x' && p[5] == '>')
                out.byte_id[strtol(p.substr(3, 2).c_str(), nullptr, 16) & 255] = (int32_t)i;
        }
    }
    if (!have_min) out.min_score = 0.f;
    out.unk_score = out.min_score - 10.0f;
    if (byte_fallback)
        for (int i = 0; i < 256; ++i)
            if (out.byte_id[i] < 0) return "byte_fallback model without all 256 byte pieces";
    // trie over code points of NORMAL / USER_DEFINED / UNUSED pieces
    out.score.assign(np, 0.f);
    out.usable.assign(np, 0);
    std::map<std::pair<uint32_t, uint32_t>, uint32_t> edges;      // (node, cp) -> child
    std::vector<int32_t> node_piece(1, -1);
    out.max_len = 0;
    for (size_t i = 0; i < np; ++i) {
        int t = out.type[i];
        if (t != 1 && t != 4 && t != 5) continue;
        const std::string& p = out.piece[i];
        if (p.empty()) continue;
        uint32_t node = 0;
        int ncp = 0;
        const unsigned char* u = (const unsigned char*)p.data();
        size_t q = 0;
        while (q < p.size()) {
            size_t need = u[q] < 0x80 ? 1 : u[q] >= 0xF0 ? 4 : u[q] >= 0xE0 ? 3 : u[q] >= 0xC0 ? 2 : 1;
            if (q + need > p.size()) need = p.size() - q;
            uint32_t cp = need == 1 ? u[q] : (u[q] & (0xFFu >> (need + 1)));
            for (size_t k = 1; k < need; ++k) cp = (cp << 6) | (u[q + k] & 0x3Fu);
            q += need;
            ++ncp;
            auto key = std::make_pair(node, cp);
            auto it = edges.find(key);
            if (it == edges.end()) {
                uint32_t child = (uint32_t)node_piece.size();
                node_piece.push_back(-1);
                edges[key] = child;
                node = child;
            } else {
                node = it->second;
            }
        }
        if (node_piece[node] < 0) node_piece[node] = (int32_t)i;     // first id wins for duplicated surface forms
        if (ncp > out.max_len) out.max_len = ncp;
        if (t == 1) { out.score[i] = out.raw_score[i]; out.usable[i] = 1; }
        else if (t == 4) return "USER_DEFINED pieces are not supported (scripts/train_spm.py defines none)";
    }
    if (out.max_len >= 62) return "piece longer than 61 code points";
    out.tbits = 4;
    while ((1ull << out.tbits) < 2 * edges.size() + 16) ++out.tbits;
    out.tkeys.assign((size_t)1 << out.tbits, AK_EMPTY_KEY);
    out.tvals.assign((size_t)1 << out.tbits, 0);
    for (auto& e : edges) {
        unsigned long long key = ((unsigned long long)e.first.first << 21) | e.first.second;
        unsigned long long v = ((unsigned long long)e.second << 32) | (uint32_t)(node_piece[e.second] + 1);
        table_insert(out.tkeys, out.tvals, out.tbits, key, v);
    }
    return "";
}
