// ORACLE — TEST INFRASTRUCTURE ONLY (see kzo.hpp). TEXT transform (DICT_TYPE), encoding type 2 — the variant the factory selects
// for the NONE / ANS0 / HUFFMAN / RANGE entropy codecs (v2/transform/Factory.go:100-120), i.e. the one `-l 3`, `-l 4`, `-l 5` use.
// Restated from v2/transform/TextCodec.go:
//   computeTextStats :187-305, detectTextType :307-396, delimiters :408-447, createDictionary :450-489,
//   textCodec2: constructor :1137-1188, reset :1190-1223, Forward :1225-1398, expandDictionary :1400-1413, emitSymbols :1415-1487,
//   emitWordIndex2 :1489-1511, Inverse :1513-1718, MaxEncodedLen :1720-1724; wrapper TextCodec.Forward/Inverse :549-592.
// Encoding type 1 (textCodec1, used with the FPAQ / CM / TPAQ / ANS1 entropy codecs) is not restated.
// The static dictionary (1024 English words, :96-185) is a format constant of the reference: it is written from
// tests/golden/text_dict_en_1024.txt into oracle/_ref/kzo_text_dict.inc at build time (oracle/gen_text_dict.py).
// The dictionary map of the reference holds pointers into dictList; expandDictionary reallocates dictList so the map may point
// to stale copies, but an entry is only modified right after its map slot has been cleared, so index semantics are equivalent.
#include <algorithm>
#include <cstring>
#include <vector>

#include "kzo.hpp"
#include "kzo_transforms.hpp"

#if __has_include("_ref/kzo_text_dict.inc")
#include "_ref/kzo_text_dict.inc"
#define KZO_HAVE_TEXT_DICT 1
#else
#define KZO_HAVE_TEXT_DICT 0
#endif

namespace kzo {

bool text_available() { return KZO_HAVE_TEXT_DICT != 0; }

#if KZO_HAVE_TEXT_DICT
namespace {

const int TC_THRESHOLD1 = 128, TC_THRESHOLD2 = TC_THRESHOLD1 * TC_THRESHOLD1, TC_THRESHOLD3 = 64, TC_THRESHOLD4 = TC_THRESHOLD3 * 128;
const int TC_MAX_DICT_SIZE = 1 << 19, TC_MAX_WORD_LENGTH = 31;
const uint8_t TC_ESCAPE_TOKEN1 = 0x0F;
const uint8_t TC_MASK_FLIP_CASE = 0x80, TC_MASK_NOT_TEXT = 0x80, TC_MASK_CRLF = 0x40, TC_MASK_XML_HTML = 0x20, TC_MASK_DT = 0x0F;
const int32_t TC_MASK_LENGTH = 0x0007FFFF;
const uint32_t TC_HASH1 = 0x7FEB352Du, TC_HASH2 = 0x846CA68Bu;  // int32 arithmetic of the reference = uint32 modulo 2^32
const uint8_t CR = 0x0D, LF = 0x0A;

inline bool is_lower(uint8_t v) { return v >= 'a' && v <= 'z'; }
inline bool is_upper(uint8_t v) { return v >= 'A' && v <= 'Z'; }
inline bool is_text(uint8_t v) { return is_lower(v | 0x20); }
inline bool is_delimiter(uint8_t v) {  // initDelimiterChars :408-447
    if (v >= ' ' && v <= '/') return true;
    if (v >= ':' && v <= '?') return true;
    switch (v) {
        case '\n': case '\r': case '\t': case '_': case '|': case '{': case '}': case '[': case ']': return true;
        default: return false;
    }
}
inline uint32_t hash_step(uint32_t h, uint32_t c) { return (h * TC_HASH1) ^ (c * TC_HASH2); }

struct Entry {
    int32_t hash = 0;
    int32_t data = 0;  // length << 24 | index
    const uint8_t* ptr = nullptr;
};

struct StaticDict {
    std::vector<uint8_t> words;  // lower-cased letters
    std::vector<Entry> entries;
    StaticDict() {  // createDictionary :450-489
        const size_t n = sizeof(KZO_TC_DICT_EN_1024) - 1;
        words.assign(KZO_TC_DICT_EN_1024, KZO_TC_DICT_EN_1024 + n);
        entries.resize(1024);
        size_t anchor = 0;
        uint32_t h = TC_HASH1;
        int nb = 0;
        for (size_t i = 0; i < n && nb < 1024; i++) {
            if (is_upper(words[i])) {
                if (i > anchor) {
                    entries[nb].ptr = words.data() + anchor;
                    entries[nb].hash = int32_t(h);
                    entries[nb].data = int32_t(((i - anchor) << 24) | size_t(nb));
                    nb++;
                    anchor = i;
                    h = TC_HASH1;
                }
                words[i] ^= 0x20;
            }
            h = hash_step(h, words[i]);
        }
        if (nb < 1024) {
            entries[nb].ptr = words.data() + anchor;
            entries[nb].hash = int32_t(h);
            entries[nb].data = int32_t(((n - anchor) << 24) | size_t(nb));
            nb++;
        }
        entries.resize(size_t(nb));
    }
};
const StaticDict& static_dict() {
    static const StaticDict d;
    return d;
}

// detectTextType :307-396
uint8_t detect_text_type(const int* freqs0, const int* freqs1 /*[256][256]*/, int count) {
    const int dt = detect_simple_type(size_t(count), freqs0);
    if (dt != DT_UNDEFINED) return uint8_t(TC_MASK_NOT_TEXT | dt);
    int sum = freqs0[0xC0] + freqs0[0xC1];
    for (int i = 0xF5; i < 256; i++) sum += freqs0[i];
    if (sum != 0) return TC_MASK_NOT_TEXT;
    int sum2 = 0;
    auto f = [&](int a, int b) { return freqs1[(a << 8) | b]; };
    for (int i = 0; i < 256; i++) {
        if (i < 0xA0 || i > 0xBF) sum += f(0xE0, i);
        if (i < 0x80 || i > 0x9F) sum += f(0xED, i);
        if (i < 0x90 || i > 0xBF) sum += f(0xF0, i);
        if (i < 0x80 || i > 0x8F) sum += f(0xF4, i);
        if (i < 0x80 || i > 0xBF) {
            for (int j = 0xC2; j <= 0xDF; j++) sum += f(j, i);
            for (int j = 0xE1; j <= 0xEC; j++) sum += f(j, i);
            sum += f(0xF1, i) + f(0xF2, i) + f(0xF3, i);
            sum += f(0xEE, i);
            sum += f(0xEF, i);
        } else {
            sum2 += freqs0[i];
        }
        if (sum != 0) return TC_MASK_NOT_TEXT;
    }
    return sum2 >= count / 8 ? uint8_t(TC_MASK_NOT_TEXT | DT_UTF8) : TC_MASK_NOT_TEXT;
}

// computeTextStats :187-305 with strict = false
uint8_t compute_text_stats(const uint8_t* block, int count, int* freqs0, int* freqs1) {
    if (get_magic_type(block, size_t(count)) != 0) return TC_MASK_NOT_TEXT;
    std::fill(freqs1, freqs1 + 65536, 0);
    uint8_t prv = 0;
    for (int i = 0; i < count; i++) {
        const uint8_t cur = block[i];
        freqs0[cur]++;
        freqs1[(int(prv) << 8) | cur]++;
        prv = cur;
    }
    int nb_text = freqs0[CR] + freqs0[LF];
    int nb_ascii = 0;
    for (int i = 0; i < 128; i++) {
        if (is_text(uint8_t(i))) nb_text += freqs0[i];
        nb_ascii += freqs0[i];
    }
    const int nb_bin = count - nb_ascii;
    bool not_text;
    if (nb_bin > (count >> 2)) {
        not_text = true;
    } else {
        not_text = nb_text < count / 4;
        not_text = not_text || freqs0[32] < count / 50;
    }
    uint8_t res = 0;
    if (not_text) return uint8_t(res | detect_text_type(freqs0, freqs1, count));
    if (nb_bin <= count - count / 10) {
        const int f1 = freqs0['<'], f2 = freqs0['>'];
        const int f3 = freqs1[('&' << 8) | 'a'] + freqs1[('&' << 8) | 'g'] + freqs1[('&' << 8) | 'l'] + freqs1[('&' << 8) | 'q'];
        int min_freq = (count - nb_bin) >> 9;
        if (min_freq < 2) min_freq = 2;
        if (f1 >= min_freq && f2 >= min_freq && f3 > 0) {
            if (f1 < f2) {
                if (f1 >= f2 - f2 / 100) res |= TC_MASK_XML_HTML;
            } else if (f2 < f1) {
                if (f2 >= f1 - f1 / 100) res |= TC_MASK_XML_HTML;
            } else {
                res |= TC_MASK_XML_HTML;
            }
        }
    }
    if (freqs0[CR] != 0 && freqs0[CR] == freqs0[LF]) {
        bool is_crlf = true;
        for (int i = 0; i < 256; i++) {
            if (i != LF && freqs1[(int(CR) << 8) | i] != 0) {
                is_crlf = false;
                break;
            }
            if (i != CR && freqs1[(i << 8) | LF] != 0) {
                is_crlf = false;
                break;
            }
        }
        if (is_crlf) res |= TC_MASK_CRLF;
    }
    return res;
}

struct TextCodec2 {
    std::vector<int32_t> dict_map;  // slot -> index in dict_list, -1 = nil
    std::vector<Entry> dict_list;
    int static_size = 0, dict_size = 1 << 13;
    uint32_t log_hash = 13;
    uint32_t hash_mask = 0;
    bool is_crlf = false;

    explicit TextCodec2(size_t block_size) {  // newTextCodec2WithCtx :1137-1188 (entropy is never TPAQX here; bsVersion 6)
        uint32_t log = 13;
        if (block_size >= 32) {
            log = log2_floor(uint32_t(block_size / 32));
            log = std::min<uint32_t>(log, 24);
            log = std::max<uint32_t>(log, 13);
        }
        log_hash = log;
        hash_mask = (1u << log_hash) - 1;
        static_size = int(static_dict().entries.size());
    }
    void reset(int count) {  // :1190-1223 (a fresh instance per block: the "already allocated" branches are never taken)
        if (count >= 1024) {
            uint32_t log = log2_floor(uint32_t(count / 128));
            log = std::min<uint32_t>(log, 18);
            log = std::max<uint32_t>(log, 13);
            dict_size = 1 << log;
        }
        dict_map.assign(size_t(1) << log_hash, -1);
        dict_list.assign(size_t(dict_size), Entry());
        const auto& sd = static_dict().entries;
        for (size_t i = 0; i < sd.size() && i < dict_list.size(); i++) dict_list[i] = sd[i];
        for (int i = 0; i < static_size; i++) dict_map[uint32_t(dict_list[size_t(i)].hash) & hash_mask] = i;
        for (int i = static_size; i < dict_size; i++) {
            dict_list[size_t(i)].ptr = nullptr;
            dict_list[size_t(i)].hash = 0;
            dict_list[size_t(i)].data = i;
        }
    }
    bool expand() {  // :1400-1413
        if (dict_size >= TC_MAX_DICT_SIZE) return false;
        dict_list.resize(size_t(dict_size) * 2);
        for (int i = dict_size; i < dict_size * 2; i++) {
            dict_list[size_t(i)].ptr = nullptr;
            dict_list[size_t(i)].hash = 0;
            dict_list[size_t(i)].data = i;
        }
        dict_size <<= 1;
        return true;
    }
    // the shared "word not found: maybe add it" step of Forward (:1302-1324) and Inverse (:1559-1581)
    void add_word(int& words, const uint8_t* p, int32_t length, uint32_t h1) {
        Entry& pe = dict_list[size_t(words)];
        if ((pe.data & TC_MASK_LENGTH) >= static_size) {
            dict_map[uint32_t(pe.hash) & hash_mask] = -1;
            pe.ptr = p;
            pe.hash = int32_t(h1);
            pe.data = (length << 24) | words;
        }
        dict_map[h1 & hash_mask] = words;
        words++;
        if (words >= dict_size) {
            if (!expand()) words = static_size;
        }
    }
    // emitSymbols :1415-1487. dst_len = room left; returns dst_len + 1 on overflow
    int emit_symbols(const uint8_t* src, int len, uint8_t* dst, int dst_len) const {
        int d = 0;
        const bool checked = !(2 * len < dst_len);
        for (int i = 0; i < len; i++) {
            const uint8_t cur = src[i];
            if (cur == TC_ESCAPE_TOKEN1) {
                if (checked && d + 1 >= dst_len) return dst_len + 1;
                dst[d++] = TC_ESCAPE_TOKEN1;
                dst[d++] = TC_ESCAPE_TOKEN1;
            } else if (cur == CR) {
                if (!is_crlf) {
                    if (checked && d >= dst_len) return dst_len + 1;
                    dst[d++] = cur;
                }
            } else {
                if (cur >= 0x80) {
                    if (checked && d >= dst_len) return dst_len + 1;
                    dst[d++] = TC_ESCAPE_TOKEN1;
                }
                if (checked && d >= dst_len) return dst_len + 1;
                dst[d++] = cur;
            }
        }
        return d;
    }
};

int emit_word_index2(uint8_t* dst, int widx) {  // :1489-1511
    widx++;
    if (widx >= TC_THRESHOLD3) {
        if (widx >= TC_THRESHOLD4) {
            dst[0] = uint8_t(0xF0 | (widx >> 16));
            dst[1] = uint8_t(widx >> 8);
            dst[2] = uint8_t(widx);
            return 3;
        }
        dst[0] = uint8_t(0xC0 | (widx >> 8));
        dst[1] = uint8_t(widx);
        return 2;
    }
    dst[0] = uint8_t(0x80 | widx);
    return 1;
}

inline bool same_words(const uint8_t* a, const uint8_t* b, int n) { return n <= 0 || std::memcmp(a, b, size_t(n)) == 0; }

}  // namespace
#endif  // KZO_HAVE_TEXT_DICT

size_t text_max_encoded_len(size_t n) { return n; }  // textCodec2.MaxEncodedLen :1720-1724

bool text_forward(Ctx& ctx, const uint8_t* src, size_t n, uint8_t* dst, size_t cap, size_t* out_n) {
    *out_n = 0;
#if !KZO_HAVE_TEXT_DICT
    (void)ctx; (void)src; (void)n; (void)dst; (void)cap;
    throw Error(ERR_CREATE_CODEC, "TEXT: static dictionary not extracted (oracle/gen_text_dict.py needs the reference tree)");
#else
    if (n == 0) return true;
    if (n < 1024 || n > (size_t(1) << 30)) return false;  // wrapper :549-560
    const int count = int(n);
    if (cap < size_t(count)) return false;
    if (ctx.data_type != DT_UNDEFINED && ctx.data_type != DT_TEXT && ctx.data_type != DT_BIN) return false;  // :1232-1241
    std::vector<int> freqs0(256, 0), stats1(65536, 0);
    const uint8_t mode = compute_text_stats(src, count, freqs0.data(), stats1.data());
    if (mode & TC_MASK_NOT_TEXT) {
        ctx.data_type = mode & TC_MASK_DT;
        return false;
    }
    ctx.data_type = DT_TEXT;
    TextCodec2 tc(ctx.stream_block_size ? ctx.stream_block_size : ctx.block_size);
    tc.reset(count);
    const int src_end = count, dst_end = count, dst_end3 = dst_end - 3;
    int emit_anchor = 0;
    int words = tc.static_size;
    tc.is_crlf = (mode & TC_MASK_CRLF) != 0;
    dst[0] = mode;
    int src_idx = 0, dst_idx = 1;
    while (src_idx < src_end && src[src_idx] == ' ') {
        dst[dst_idx++] = ' ';
        src_idx++;
        emit_anchor++;
    }
    if (src_idx >= src_end) return false;  // the reference would index past the slice (panic -> block error); unreachable for text
    bool err = false;
    int delim_anchor = src_idx;
    if (is_text(src[src_idx])) delim_anchor = src_idx - 1;
    while (src_idx < src_end) {
        if (is_text(src[src_idx])) {
            src_idx++;
            continue;
        }
        if (src_idx > delim_anchor + 2 && is_delimiter(src[src_idx])) {
            const int32_t length = src_idx - delim_anchor - 1;
            if (length <= TC_MAX_WORD_LENGTH) {
                const uint8_t val = src[delim_anchor + 1];
                uint32_t h1 = hash_step(TC_HASH1, val);
                uint32_t h2 = hash_step(TC_HASH1, uint32_t(val) ^ 0x20);
                for (int i = delim_anchor + 2; i < src_idx; i++) {
                    const uint32_t h = uint32_t(src[i]) * TC_HASH2;
                    h1 = (h1 * TC_HASH1) ^ h;
                    h2 = (h2 * TC_HASH1) ^ h;
                }
                int pe = -1;
                const int pe1 = tc.dict_map[h1 & tc.hash_mask];
                if (pe1 >= 0 && tc.dict_list[size_t(pe1)].hash == int32_t(h1) && (tc.dict_list[size_t(pe1)].data >> 24) == length) {
                    pe = pe1;
                } else {
                    const int pe2 = tc.dict_map[h2 & tc.hash_mask];
                    if (pe2 >= 0 && tc.dict_list[size_t(pe2)].hash == int32_t(h2) && (tc.dict_list[size_t(pe2)].data >> 24) == length) pe = pe2;
                }
                if (pe >= 0 && !same_words(tc.dict_list[size_t(pe)].ptr + 1, src + delim_anchor + 2, length - 1)) pe = -1;
                if (pe < 0) {
                    if ((length > 3 || (length == 3 && words < TC_THRESHOLD2)) && pe1 < 0) tc.add_word(words, src + delim_anchor + 1, length, h1);
                } else {
                    if (emit_anchor != delim_anchor || src[delim_anchor] != ' ')
                        dst_idx += tc.emit_symbols(src + emit_anchor, delim_anchor + 1 - emit_anchor, dst + dst_idx, dst_end - dst_idx);
                    if (dst_idx >= dst_end3) {
                        err = true;
                        break;
                    }
                    if (pe != pe1) dst[dst_idx++] = TC_MASK_FLIP_CASE;
                    const Entry& e = tc.dict_list[size_t(pe)];
                    dst_idx += emit_word_index2(dst + dst_idx, int(e.data & TC_MASK_LENGTH));
                    emit_anchor = delim_anchor + 1 + int(e.data >> 24);
                }
            }
        }
        delim_anchor = src_idx;
        src_idx++;
    }
    if (!err) {
        dst_idx += tc.emit_symbols(src + emit_anchor, src_end - emit_anchor, dst + dst_idx, dst_end - dst_idx);
        if (dst_idx > dst_end) err = true;
    }
    if (!err && src_idx != src_end) err = true;
    if (err) return false;
    *out_n = size_t(dst_idx);
    return true;
#endif
}

bool text_inverse(Ctx& ctx, const uint8_t* src, size_t len, uint8_t* dst, size_t cap, size_t* out_n) {
    *out_n = 0;
#if !KZO_HAVE_TEXT_DICT
    (void)ctx; (void)src; (void)len; (void)dst; (void)cap;
    throw Error(ERR_CREATE_CODEC, "TEXT: static dictionary not extracted (oracle/gen_text_dict.py needs the reference tree)");
#else
    if (len == 0 || cap == 0) return true;
    if (len < 2 || len > (size_t(1) << 30)) return false;
    TextCodec2 tc(ctx.stream_block_size ? ctx.stream_block_size : ctx.block_size);
    tc.reset(int(cap));
    int words = tc.static_size;
    bool word_run = false;
    tc.is_crlf = (src[0] & TC_MASK_CRLF) != 0;
    int src_idx = 1, dst_idx = 0;
    const int src_end = int(len), dst_end = int(cap);
    int delim_anchor = src_idx;
    if (is_text(src[src_idx])) delim_anchor = src_idx - 1;
    while (src_idx < src_end && dst_idx < dst_end) {
        uint8_t cur = src[src_idx];
        if (is_text(cur)) {
            dst[dst_idx++] = cur;
            src_idx++;
            continue;
        }
        if (src_idx > delim_anchor + 3 && is_delimiter(cur)) {
            const int32_t length = src_idx - delim_anchor - 1;
            if (length <= TC_MAX_WORD_LENGTH) {
                uint32_t h1 = TC_HASH1;
                for (int i = delim_anchor + 1; i < src_idx; i++) h1 = hash_step(h1, src[i]);
                int pe = -1;
                const int pe1 = tc.dict_map[h1 & tc.hash_mask];
                if (pe1 >= 0) {
                    const Entry& e = tc.dict_list[size_t(pe1)];
                    if (e.hash == int32_t(h1) && (e.data >> 24) == length && same_words(e.ptr + 1, src + delim_anchor + 2, length - 1)) pe = pe1;
                }
                if (pe < 0) {
                    if ((length > 3 || words < TC_THRESHOLD2) && pe1 < 0) tc.add_word(words, src + delim_anchor + 1, length, h1);
                }
            }
        }
        src_idx++;
        uint8_t flip_mask = 0;
        if (cur >= 128) {
            int idx;
            if (cur == TC_MASK_FLIP_CASE) {
                flip_mask = 0x20;
                if (src_idx >= src_end) return false;
                cur = src[src_idx++];
            }
            idx = cur & 0x7F;
            if (idx >= 64) {
                if (idx >= 112) {
                    if (src_idx + 1 >= src_end) return false;
                    idx = ((idx & 0x0F) << 16) | (int(src[src_idx]) << 8) | src[src_idx + 1];
                    src_idx += 2;
                } else {
                    if (src_idx >= src_end) return false;
                    idx = ((idx & 0x1F) << 8) | src[src_idx];
                    src_idx++;
                }
                if (idx > tc.dict_size) return false;
            } else if (idx == 0) {
                return false;
            }
            idx--;
            if (idx < 0 || size_t(idx) >= tc.dict_list.size()) return false;
            const Entry& e = tc.dict_list[size_t(idx)];
            const int length = (e.data >> 24) & 0xFF;
            if (length > 1) {
                if (word_run) dst[dst_idx++] = ' ';
                word_run = true;
                delim_anchor = src_idx;
            } else {
                word_run = false;
                delim_anchor = src_idx - 1;
            }
            if (e.ptr == nullptr || dst_idx + length >= dst_end) return false;
            std::memcpy(dst + dst_idx, e.ptr, size_t(length));
            dst[dst_idx] ^= flip_mask;
            dst_idx += length;
        } else {
            if (cur == TC_ESCAPE_TOKEN1) {
                if (src_idx >= src_end) return false;
                dst[dst_idx++] = src[src_idx++];
            } else {
                if (tc.is_crlf && cur == LF) {
                    dst[dst_idx++] = CR;
                    if (dst_idx >= dst_end) return false;
                }
                dst[dst_idx++] = cur;
            }
            word_run = false;
            delim_anchor = src_idx - 1;
        }
    }
    if (src_idx != src_end) return false;
    *out_n = size_t(dst_idx);
    return true;
#endif
}

}  // namespace kzo
