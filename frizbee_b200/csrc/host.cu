// host.cu — the C ABI (include/frz_cuda.h): host-side mirror of the reference's Matcher / Pattern /
// Config logic for the match_list path, orchestrating the CUDA stages.  No CPU compute fallback.
//
// Reference logic mirrored here (file:line relative to the reference crate):
//   Pattern::parse / parse_query          src/pattern.rs:100-222
//   PatternConfig::resolve                src/pattern.rs:250-262
//   Matcher::build_patterns / compile     src/matcher/mod.rs:178-205
//   Matcher::get_backend                  src/matcher/mod.rs:448-498
//   score_fits_in_u8                      src/smith_waterman/mod.rs:91-116
//   Scoring::guard_against_score_overflow src/lib.rs:506-537
//   Matcher::match_list / match_list_into src/matcher/mod.rs:212-222, 373-392
//   match_list_multi_into                 src/matcher/multi.rs:84-152
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <memory>
#include <mutex>

#include "frz_device.cuh"
#include "frz_host.h"
#include "unicode_needle.h"
#include "indices_path.cuh"

// ------------------------------------------------------------------------------------ errors

static thread_local char g_err[512] = "";

frz_status frz_fail(frz_status s, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return s;
}

extern "C" const char* frz_last_error(void) { return g_err; }
extern "C" int frz_abi_version(void) { return FRZ_ABI_VERSION; }
extern "C" const char* frz_status_str(frz_status s) {
    switch (s) {
        case FRZ_OK: return "ok";
        case FRZ_ERR_INVALID_ARG: return "invalid argument";
        case FRZ_ERR_NEEDLE_TOO_LONG: return "needle too long and could overflow the u16 score";
        case FRZ_ERR_GAP_OVERFLOW: return "gap penalties too large and could overflow the u16 score";
        case FRZ_ERR_TOO_MANY_ITEMS: return "too many items in haystack, will overflow the u32 index";
        case FRZ_ERR_THREADS_ZERO: return "threads must be positive";
        case FRZ_ERR_CAPACITY: return "output capacity too small";
        case FRZ_ERR_CUDA: return "CUDA error";
        case FRZ_ERR_NO_DEVICE: return "no usable CUDA device";
        case FRZ_ERR_UNSUPPORTED: return "not supported on the GPU path";
        case FRZ_ERR_OOM: return "out of device memory";
        case FRZ_ERR_NCCL: return "NCCL error";
    }
    return "?";
}

extern "C" void frz_scoring_default(frz_scoring* s) {
    *s = frz_scoring{12, 6, 5, 1, 12, 4, 4, 8, 4};  // src/const.rs:1-10
}
extern "C" void frz_config_default(frz_config* c) {
    memset(c, 0, sizeof *c);
    c->max_typos = 0;
    c->casing = FRZ_CASE_SMART;
    c->unicode = FRZ_UNICODE_SMART;
    c->matching = FRZ_MATCHING_FUZZY;
    c->sort = FRZ_SORT_SCORE_THEN_INDEX_ASC;
    frz_scoring_default(&c->scoring);
    c->emulate_lanes = 0;
}

static frz_status ensure_device(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        return frz_fail(FRZ_ERR_NO_DEVICE, "no CUDA device available (%s); this library has no CPU fallback",
                        e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    }
    if (device < 0 || device >= n) return frz_fail(FRZ_ERR_INVALID_ARG, "device %d out of range (have %d)", device, n);
    FRZ_CUDA_TRY(cudaSetDevice(device));
    return FRZ_OK;
}

// ----------------------------------------------------------------------------- query parser

struct OwnedPattern {
    std::string needle;
    std::string raw;
    bool negated = false;
    int matching = -1, casing = -1, unicode = -1, max_typos = -1;
    bool has_scoring = false;
    frz_scoring scoring{};
};

struct frz_query {
    std::vector<OwnedPattern> pats;
};

namespace {

// Decodes one UTF-8 scalar starting at s[i] (input is a Rust &str, so valid UTF-8; be lenient).
uint32_t utf8_next(const uint8_t* s, size_t len, size_t* i) {
    uint8_t b = s[*i];
    int extra = b < 0x80 ? 0 : (b >> 5) == 6 ? 1 : (b >> 4) == 14 ? 2 : (b >> 3) == 30 ? 3 : 0;
    uint32_t cp = extra == 0 ? b : extra == 1 ? (b & 0x1f) : extra == 2 ? (b & 0x0f) : (b & 0x07);
    size_t j = *i + 1;
    for (int k = 0; k < extra && j < len; k++, j++) cp = (cp << 6) | (s[j] & 0x3f);
    *i = j;
    return cp;
}
void utf8_push(std::string& out, uint32_t cp) {
    if (cp < 0x80) out.push_back((char)cp);
    else if (cp < 0x800) { out.push_back((char)(0xC0 | (cp >> 6))); out.push_back((char)(0x80 | (cp & 0x3f))); }
    else if (cp < 0x10000) {
        out.push_back((char)(0xE0 | (cp >> 12))); out.push_back((char)(0x80 | ((cp >> 6) & 0x3f))); out.push_back((char)(0x80 | (cp & 0x3f)));
    } else {
        out.push_back((char)(0xF0 | (cp >> 18))); out.push_back((char)(0x80 | ((cp >> 12) & 0x3f)));
        out.push_back((char)(0x80 | ((cp >> 6) & 0x3f))); out.push_back((char)(0x80 | (cp & 0x3f)));
    }
}
// char::is_whitespace (Unicode White_Space)
bool is_ws(uint32_t c) {
    return (c >= 9 && c <= 13) || c == 0x20 || c == 0x85 || c == 0xA0 || c == 0x1680 || (c >= 0x2000 && c <= 0x200A) ||
           c == 0x2028 || c == 0x2029 || c == 0x202F || c == 0x205F || c == 0x3000;
}

// Pattern::parse (src/pattern.rs:100-165)
OwnedPattern parse_atom(const uint8_t* atom, size_t len) {
    struct Tok { uint32_t c; bool escaped; };
    std::vector<Tok> toks;
    size_t i = 0;
    while (i < len) {
        uint32_t c = utf8_next(atom, len, &i);
        if (c == '\\' && i < len) toks.push_back({utf8_next(atom, len, &i), true});
        else toks.push_back({c, false});
    }
    size_t lo = 0, hi = toks.size();
    auto strip_first = [&](uint32_t op) {
        if (lo < hi && !toks[lo].escaped && toks[lo].c == op) { lo++; return true; }
        return false;
    };
    auto strip_last = [&](uint32_t op) {
        if (lo < hi && !toks[hi - 1].escaped && toks[hi - 1].c == op) { hi--; return true; }
        return false;
    };
    OwnedPattern p;
    p.raw.assign((const char*)atom, len);
    p.negated = strip_first('!');
    bool prefix = strip_first('^');
    bool substring = !prefix && strip_first('\'');
    bool suffix = strip_last('$');
    auto is_special = [](uint32_t c) { return c == '!' || c == '^' || c == '\'' || c == '$' || is_ws(c); };
    for (size_t k = lo; k < hi; k++) {
        if (toks[k].escaped && !is_special(toks[k].c)) p.needle.push_back('\\');
        utf8_push(p.needle, toks[k].c);
    }
    if (prefix && suffix) p.matching = FRZ_MATCHING_EXACT;
    else if (prefix) p.matching = FRZ_MATCHING_PREFIX;
    else if (suffix) p.matching = FRZ_MATCHING_SUFFIX;
    else if (substring) p.matching = FRZ_MATCHING_SUBSTRING;
    else if (p.negated) p.matching = FRZ_MATCHING_SUBSTRING;
    else p.matching = -1;
    return p;
}

// Pattern::parse_query (src/pattern.rs:190-222)
std::vector<OwnedPattern> parse_query(const uint8_t* q, size_t len) {
    std::vector<OwnedPattern> out;
    bool have_start = false, escaped = false;
    size_t start = 0;
    auto push = [&](size_t a, size_t b) {
        OwnedPattern p = parse_atom(q + a, b - a);
        if (!p.needle.empty()) out.push_back(std::move(p));
    };
    size_t i = 0;
    while (i < len) {
        size_t at = i;
        uint32_t c = utf8_next(q, len, &i);
        if (escaped) escaped = false;
        else if (c == '\\') { if (!have_start) { have_start = true; start = at; } escaped = true; }
        else if (is_ws(c)) { if (have_start) { push(start, at); have_start = false; } }
        else if (!have_start) { have_start = true; start = at; }
    }
    if (have_start) push(start, len);
    return out;
}

void fill_c_pattern(const OwnedPattern& o, frz_pattern* out) {
    memset(out, 0, sizeof *out);
    out->needle = (const uint8_t*)o.needle.data();
    out->needle_len = o.needle.size();
    out->negated = o.negated;
    out->has_scoring = o.has_scoring;
    out->casing = (int8_t)o.casing;
    out->unicode = (int8_t)o.unicode;
    out->matching = (int8_t)o.matching;
    out->max_typos = o.max_typos;
    out->scoring = o.scoring;
}

}  // namespace

extern "C" frz_status frz_parse_query(const uint8_t* query, size_t len, frz_query** out) {
    if (!out || (!query && len)) return frz_fail(FRZ_ERR_INVALID_ARG, "null argument");
    auto* q = new frz_query();
    q->pats = parse_query(query, len);
    *out = q;
    return FRZ_OK;
}
extern "C" frz_status frz_parse_atom(const uint8_t* atom, size_t len, frz_query** out) {
    if (!out || (!atom && len)) return frz_fail(FRZ_ERR_INVALID_ARG, "null argument");
    auto* q = new frz_query();
    q->pats.push_back(parse_atom(atom, len));
    *out = q;
    return FRZ_OK;
}
extern "C" size_t frz_query_len(const frz_query* q) { return q ? q->pats.size() : 0; }
extern "C" frz_status frz_query_get(const frz_query* q, size_t i, frz_pattern* out) {
    if (!q || !out || i >= q->pats.size()) return frz_fail(FRZ_ERR_INVALID_ARG, "pattern index out of range");
    fill_c_pattern(q->pats[i], out);
    return FRZ_OK;
}
extern "C" void frz_query_destroy(frz_query* q) { delete q; }

// ---------------------------------------------------------------------------------- corpus

extern "C" frz_status frz_corpus_create_device(const uint8_t* d_bytes, const uint64_t* d_offsets, uint64_t n,
                                               uint64_t total_bytes, int device, void* stream, frz_corpus** out) {
    if (!out) return frz_fail(FRZ_ERR_INVALID_ARG, "null out");
    if (n > 0xFFFFFFFFull) return frz_fail(FRZ_ERR_TOO_MANY_ITEMS, "too many items in haystack: %llu", (unsigned long long)n);
    FRZ_TRY(ensure_device(device));
    auto c = std::make_unique<frz_corpus>();
    c->st.device = device;
    frz_status s = frz_pack_corpus_device(d_bytes, d_offsets, 8, n, total_bytes, (cudaStream_t)stream, &c->st);
    if (s != FRZ_OK) { c->st.release(); return s; }
    *out = c.release();
    return FRZ_OK;
}

// Host Arrow buffers (Utf8: 32-bit offsets, LargeUtf8: 64-bit; a sliced array may start at offsets[0] != 0).
extern "C" frz_status frz_corpus_create_arrow(const uint8_t* bytes, const void* offsets, int offset_width, uint64_t n, int device,
                                              frz_corpus** out) {
    if (!out || !offsets) return frz_fail(FRZ_ERR_INVALID_ARG, "null argument");
    if (offset_width != 4 && offset_width != 8) return frz_fail(FRZ_ERR_INVALID_ARG, "offset_width must be 4 or 8");
    if (n > 0xFFFFFFFFull) return frz_fail(FRZ_ERR_TOO_MANY_ITEMS, "too many items in haystack: %llu", (unsigned long long)n);
    FRZ_TRY(ensure_device(device));
    auto c = std::make_unique<frz_corpus>();
    c->st.device = device;
    FrzIngest ing;
    cudaStream_t stream = nullptr;
    frz_status s = frz_ingest_host(ing, bytes, offsets, offset_width, n, stream, &c->st);
    if (s == FRZ_OK && cudaStreamSynchronize(stream) != cudaSuccess)
        s = frz_fail(FRZ_ERR_CUDA, "pack failed: %s", cudaGetErrorString(cudaGetLastError()));
    ing.release();
    if (s != FRZ_OK) { c->st.release(); return s; }
    *out = c.release();
    return FRZ_OK;
}

extern "C" frz_status frz_corpus_create(const uint8_t* bytes, const uint64_t* offsets, uint64_t n, int device, frz_corpus** out) {
    return frz_corpus_create_arrow(bytes, offsets, 8, n, device, out);
}

// Incremental ingestion: the new haystacks get indices [len, len + n_new).  Synchronous; must not overlap a match
// call on the same corpus.
extern "C" frz_status frz_corpus_append(frz_corpus* c, const uint8_t* bytes, const void* offsets, int offset_width, uint64_t n_new) {
    if (!c || (n_new && !offsets)) return frz_fail(FRZ_ERR_INVALID_ARG, "null argument");
    if (offset_width != 4 && offset_width != 8) return frz_fail(FRZ_ERR_INVALID_ARG, "offset_width must be 4 or 8");
    if (n_new == 0) return FRZ_OK;
    FRZ_TRY(ensure_device(c->st.device));
    if (!c->ingest) c->ingest = new FrzIngest();
    cudaStream_t stream = nullptr;
    FRZ_TRY(frz_append_host(*c->ingest, bytes, offsets, offset_width, n_new, stream, &c->st));
    FRZ_CUDA_TRY(cudaStreamSynchronize(stream));
    return FRZ_OK;
}

extern "C" frz_status frz_corpus_create_ptrs(const uint8_t* const* ptrs, const uint32_t* lens, uint64_t n, int device,
                                             frz_corpus** out) {
    if (!out || (n && (!ptrs || !lens))) return frz_fail(FRZ_ERR_INVALID_ARG, "null argument");
    std::vector<uint64_t> off(n + 1, 0);
    for (uint64_t i = 0; i < n; i++) off[i + 1] = off[i] + lens[i];
    std::vector<uint8_t> bytes(off[n] ? off[n] : 1);
    for (uint64_t i = 0; i < n; i++)
        if (lens[i]) memcpy(bytes.data() + off[i], ptrs[i], lens[i]);
    return frz_corpus_create(bytes.data(), off.data(), n, device, out);
}

extern "C" uint64_t frz_corpus_len(const frz_corpus* c) { return c ? c->st.n : 0; }
extern "C" uint64_t frz_corpus_total_bytes(const frz_corpus* c) { return c ? c->st.total_bytes : 0; }
extern "C" uint64_t frz_corpus_device_bytes(const frz_corpus* c) {
    if (!c) return 0;
    const auto& s = c->st;
    return (s.total_units + 1) * 16 + (uint64_t)s.n_tiles * (8 + FRZ_GROUPS_PER_TILE * 16 + FRZ_TILE * (6 + 8));
}
extern "C" int frz_corpus_device(const frz_corpus* c) { return c ? c->st.device : -1; }
extern "C" void frz_corpus_destroy(frz_corpus* c) {
    if (!c) return;
    cudaSetDevice(c->st.device);
    c->st.release();
    if (c->ingest) { c->ingest->release(); delete c->ingest; }
    delete c;
}

// --------------------------------------------------------------------------------- matcher

namespace {

struct CpuIsa {
    bool avx512_pf, avx512_sw, avx512_sw_u8, avx2, sse;
};
CpuIsa detect_isa() {
    CpuIsa r{false, false, false, false, false};
#if defined(__x86_64__)
    __builtin_cpu_init();
    bool f = __builtin_cpu_supports("avx512f"), bw = __builtin_cpu_supports("avx512bw");
    bool bmi1 = __builtin_cpu_supports("bmi"), bmi2 = __builtin_cpu_supports("bmi2");
    bool vbmi = __builtin_cpu_supports("avx512vbmi");
    r.avx512_pf = f && bw && bmi1 && bmi2;       // src/prefilter/backend/avx512.rs:14-19
    r.avx512_sw = f && bw;                       // src/smith_waterman/backend/avx512.rs:44-46
    r.avx512_sw_u8 = f && bw && vbmi;            // src/smith_waterman/backend/avx512.rs:112-116
    r.avx2 = __builtin_cpu_supports("avx2");
    r.sse = __builtin_cpu_supports("sse2") && __builtin_cpu_supports("ssse3") && __builtin_cpu_supports("sse4.1");
#endif
    return r;
}

uint16_t sat_add16(uint32_t a, uint32_t b) { uint32_t r = a + b; return (uint16_t)(r > 0xFFFF ? 0xFFFF : r); }
uint16_t sat_sub16(uint32_t a, uint32_t b) { return (uint16_t)(a > b ? a - b : 0); }

uint32_t max_per_char_bonus(const frz_scoring& s) {  // src/lib.rs:488-494
    uint32_t bonus = std::max(s.delimiter_bonus, s.capitalization_bonus);
    uint32_t amort = std::max((bonus + 1) / 2, bonus > s.gap_open_penalty ? bonus - s.gap_open_penalty : 0u);
    return sat_add16(amort, s.matching_case_bonus);
}
uint32_t max_one_time_bonus(const frz_scoring& s) {  // src/lib.rs:497-503
    uint32_t bonus = std::max(s.delimiter_bonus, s.capitalization_bonus);
    uint32_t amort = std::max((bonus + 1) / 2, bonus > s.gap_open_penalty ? bonus - s.gap_open_penalty : 0u);
    return bonus - amort;
}
bool score_fits_in_u8(size_t needle_len, const frz_scoring& s) {  // src/smith_waterman/mod.rs:91-116
    size_t mc = (size_t)s.match_score + s.mismatch_penalty;
    mc = std::max<size_t>(mc, s.gap_open_penalty);
    mc = std::max<size_t>(mc, s.gap_extend_penalty);
    mc = std::max<size_t>(mc, s.matching_case_bonus);
    mc = std::max<size_t>(mc, s.capitalization_bonus);
    mc = std::max<size_t>(mc, s.delimiter_bonus);
    mc = std::max<size_t>(mc, s.prefix_bonus);
    if (mc > 255) return false;
    if (64 * (size_t)s.gap_extend_penalty + s.gap_open_penalty > 255) return false;
    size_t per_char = (size_t)s.match_score + max_per_char_bonus(s);
    size_t max_matrix = per_char * needle_len + max_one_time_bonus(s) + s.prefix_bonus;
    return max_matrix + s.mismatch_penalty <= 255;
}
// Scoring::guard_against_score_overflow (src/lib.rs:506-537)
frz_status guard_against_score_overflow(const frz_scoring& s, size_t needle_len, uint32_t max_bonus_per_char, uint32_t one_time) {
    uint32_t per_char = sat_add16(s.match_score, max_bonus_per_char);
    if (per_char == 0) return FRZ_OK;
    uint32_t headroom = sat_sub16(sat_sub16(sat_sub16(sat_sub16(0xFFFF, s.prefix_bonus), s.exact_match_bonus), s.mismatch_penalty), one_time);
    uint32_t max_len = headroom / per_char;
    if (needle_len > max_len)
        return frz_fail(FRZ_ERR_NEEDLE_TOO_LONG, "needle too long and could overflow the u16 score: %zu > %u", needle_len, max_len);
    size_t max_gap = 32 * (size_t)s.gap_extend_penalty + s.gap_open_penalty;
    if (max_gap > 0xFFFF)
        return frz_fail(FRZ_ERR_GAP_OVERFLOW, "gap penalties too large and could overflow the u16 score: %zu > 65535", max_gap);
    return FRZ_OK;
}

struct Compiled {
    FrzPatternDev dev;
    bool negated = false;
    bool literal = false;
    bool unicode = false;      // UNICODE = true specialisations (unicode.cu)
    FrzUNeedle un;             // case_needle_unicode (valid when `unicode`)
    FrzUScoring usc;
    uint32_t score_bound = 0;  // host-side upper bound of any score this pattern can emit
};

// Matcher::compile + get_backend (src/matcher/mod.rs:193-205, 448-498) → device pattern
frz_status compile_pattern(const OwnedPattern& src, const frz_config& mcfg, bool* is_none, Compiled* out) {
    *is_none = src.needle.empty();
    if (*is_none) return FRZ_OK;
    // PatternConfig::resolve (src/pattern.rs:250-262)
    const int max_typos = src.max_typos >= 0 ? src.max_typos : mcfg.max_typos;
    const int casing = src.casing >= 0 ? src.casing : mcfg.casing;
    const int unicode = src.unicode >= 0 ? src.unicode : mcfg.unicode;
    const int matching = src.matching >= 0 ? src.matching : mcfg.matching;
    const frz_scoring sc = src.has_scoring ? src.scoring : mcfg.scoring;
    const uint8_t* nd = (const uint8_t*)src.needle.data();
    const size_t n = src.needle.size();
    bool ascii = true;
    size_t nchars = 0;
    for (size_t i = 0; i < n; i++) {
        if (nd[i] >= 0x80) ascii = false;
        if ((nd[i] & 0xC0) != 0x80) nchars++;
    }
    // UnicodeMatching::respects_unicode_for (src/lib.rs:394-401)
    const bool needs_unicode = unicode == FRZ_UNICODE_ALWAYS || (unicode == FRZ_UNICODE_SMART && !ascii);
    // CaseMatching::respects_case_for (src/lib.rs:368-377): needle.chars().any(char::is_uppercase)
    bool case_sensitive;
    if (casing == FRZ_CASE_IGNORE) case_sensitive = false;
    else if (casing == FRZ_CASE_RESPECT) case_sensitive = true;
    else case_sensitive = frz_needle_has_uppercase(nd, n);
    if (n > FRZ_MAX_NEEDLE) return frz_fail(FRZ_ERR_UNSUPPORTED, "needle of %zu bytes exceeds the GPU kernels' limit of %d", n, FRZ_MAX_NEEDLE);

    Compiled c;
    FrzPatternDev& d = c.dev;
    memset(&d, 0, sizeof d);
    c.negated = src.negated;
    c.literal = matching != FRZ_MATCHING_FUZZY;
    c.unicode = needs_unicode;
    if (needs_unicode) {
        if (!frz_build_uneedle(nd, n, case_sensitive, &c.un)) return frz_fail(FRZ_ERR_INVALID_ARG, "the needle is not valid UTF-8");
    } else {
        // byte path: only the byte-level case_needle pairs are used (frz_match_indices); the needle may be any bytes
        memset(&c.un, 0, sizeof c.un);
        c.un.nbytes = (int32_t)n;
        for (size_t i = 0; i < n; i++) {
            const uint8_t ch = nd[i];
            c.un.c[i] = ch;
            c.un.f[i] = ch;
            c.un.bflip[i] = case_sensitive ? ch : (ch >= 'a' && ch <= 'z') ? (uint8_t)(ch - 32) : (ch >= 'A' && ch <= 'Z') ? (uint8_t)(ch + 32) : ch;
        }
    }
    d.n = (int)n;
    d.matching = matching;
    d.case_sensitive = case_sensitive;
    for (size_t i = 0; i < n; i++) {  // case_needle (src/prefilter/mod.rs:49-65)
        uint8_t ch = nd[i], fl;
        if (case_sensitive) fl = ch;
        else if (ch >= 'a' && ch <= 'z') fl = (uint8_t)(ch - 32);
        else if (ch >= 'A' && ch <= 'Z') fl = (uint8_t)(ch + 32);
        else fl = ch;
        d.c[i] = ch; d.flip[i] = fl;
        d.om[i] = fl != ch ? 0x20 : 0;
        d.tg[i] = fl != ch ? (uint8_t)(ch | 0x20) : ch;
    }
    {   // distinct (om, tg) classes
        int nd = 0;
        bool ok = true;
        for (size_t i = 0; i < n && ok; i++) {
            int found = -1;
            for (int k = 0; k < nd; k++) if (d.dc_om[k] == d.om[i] && d.dc_tg[k] == d.tg[i]) { found = k; break; }
            if (found < 0) {
                if (nd == 16) { ok = false; break; }
                d.dc_om[nd] = d.om[i]; d.dc_tg[nd] = d.tg[i]; found = nd++;
            }
            d.cid[i] = (uint8_t)found;
        }
        d.n_distinct = ok ? nd : 0;
    }
    d.raw_match = sc.match_score; d.raw_mismatch = sc.mismatch_penalty; d.raw_gap_open = sc.gap_open_penalty;
    d.raw_gap_extend = sc.gap_extend_penalty; d.raw_prefix = sc.prefix_bonus; d.raw_cap = sc.capitalization_bonus;
    d.raw_case = sc.matching_case_bonus; d.raw_delim = sc.delimiter_bonus; d.exact_bonus = sc.exact_match_bonus;

    const CpuIsa isa = detect_isa();
    const int em = mcfg.emulate_lanes;
    if (em != 0 && em != 16 && em != 32 && em != 64) return frz_fail(FRZ_ERR_INVALID_ARG, "emulate_lanes must be 0, 16, 32 or 64");
    // per-char bound used for the sort's digit width
    const uint32_t maxb = std::max(sc.capitalization_bonus, sc.delimiter_bonus);

    memset(&c.usc, 0, sizeof c.usc);   // untruncated u16 scoring (literal matcher, greedy scorer); lane constants below
    c.usc.raw_match = sc.match_score; c.usc.raw_gap_open = sc.gap_open_penalty; c.usc.raw_gap_extend = sc.gap_extend_penalty;
    c.usc.raw_prefix = sc.prefix_bonus; c.usc.raw_cap = sc.capitalization_bonus; c.usc.raw_case = sc.matching_case_bonus;
    c.usc.raw_delim = sc.delimiter_bonus; c.usc.exact_bonus = sc.exact_match_bonus;
    if (c.literal) {
        // LiteralImpl::guard_against_score_overflow (src/literal/algo.rs:316-324)
        FRZ_TRY(guard_against_score_overflow(sc, n, sat_add16(maxb, sc.matching_case_bonus), 0));
        d.typo_mode = FRZ_T_LITERAL;
        d.min_hay_len = 0;
        {   // a literal match holds every needle byte (either case): signature test with no typo budget
            // (unicode path: only the needle's ASCII scalars count — a non-ASCII scalar and its case flip may differ in
            // every byte, an ASCII scalar is matched by the same letter in either case, which the classes fold)
            uint32_t cnt[32] = {0};
            for (size_t i = 0; i < n; i++)
                if (!needs_unicode || d.c[i] < 0x80) cnt[frz_sig_bucket(d.c[i])]++;
            for (int b2 = 0; b2 < 32; b2++) {
                if (cnt[b2] >= 1) d.sig_need1 |= 1u << b2;
                if (cnt[b2] >= 2) d.sig_need2 |= 1u << b2;
            }
            d.sig_on = 1;
            d.sig_k = 0;
        }
        d.pf_lanes = 64; d.sw_lanes = 64; d.score_bits = 16;
        uint64_t b = (uint64_t)n * ((uint64_t)sc.match_score + sc.matching_case_bonus + maxb) + sc.prefix_bonus + sc.exact_match_bonus;
        c.score_bound = (uint32_t)std::min<uint64_t>(b, 0xFFFF);
        *out = c;
        return FRZ_OK;
    }
    // MatcherImpl::guard_against_score_overflow (src/matcher/algo.rs:311-325): byte length on the ascii path,
    // (needle.chars().count() when the unicode specialisation is selected, algo.rs:318-321)
    const size_t guard_len = needs_unicode ? nchars : n;
    FRZ_TRY(guard_against_score_overflow(sc, guard_len, max_per_char_bonus(sc), max_one_time_bonus(sc)));
    const bool use_u8 = score_fits_in_u8(n, sc);
    int pf_lanes, sw_lanes;
    if (em == 0) {
        if (use_u8) {
            if (isa.avx512_pf && isa.avx512_sw_u8) { pf_lanes = 64; sw_lanes = 64; }
            else if (isa.avx2) { pf_lanes = 32; sw_lanes = 32; }
            else { pf_lanes = 16; sw_lanes = 16; }   // SSE / NEON / scalar
        } else {
            if (isa.avx512_pf && isa.avx512_sw) { pf_lanes = 64; sw_lanes = 32; }
            else if (isa.avx2) { pf_lanes = 32; sw_lanes = 16; }
            else { pf_lanes = 16; sw_lanes = 8; }
        }
    } else {
        pf_lanes = em;
        sw_lanes = use_u8 ? em : em / 2;
    }
    d.pf_lanes = pf_lanes; d.sw_lanes = sw_lanes; d.score_bits = use_u8 ? 8 : 16;
    // constants exactly as the reference splats them (ascii.rs:35-46); `as u8` truncation in the u8 family
    const uint32_t tm = use_u8 ? 0xFF : 0xFFFF;
    d.gap_extend = sc.gap_extend_penalty & tm;
    d.gap_open_x = sat_sub16(sc.gap_open_penalty, sc.gap_extend_penalty) & tm;
    d.match_x = sat_add16(sc.match_score, sc.mismatch_penalty) & tm;
    d.mismatch = sc.mismatch_penalty & tm;
    d.case_bonus = sc.matching_case_bonus & tm;
    d.cap_bonus = sc.capitalization_bonus & tm;
    d.delim_bonus = sc.delimiter_bonus & tm;
    d.prefix_bonus = sc.prefix_bonus & tm;
    c.usc.gex = d.gap_extend; c.usc.gopx = d.gap_open_x; c.usc.match_x = d.match_x; c.usc.mismatch = d.mismatch;
    c.usc.case_bonus = d.case_bonus; c.usc.cap_bonus = d.cap_bonus; c.usc.delim_bonus = d.delim_bonus; c.usc.prefix_bonus = d.prefix_bonus;
    {
        auto sp = [](int v) { return ((uint32_t)v & 0xffffu) * 0x00010001u; };
        for (int k = 0; k < 6; k++) {
            const int sft = 1 << k;
            d.k_pen_a[k] = sp(-(sft * d.gap_extend));
            d.k_pen_b[k] = sp(-(sft * d.gap_extend + d.gap_open_x));
        }
        d.k_neg_mis = sp(-d.mismatch);
        d.k_ex_add = sp(d.case_bonus - d.mismatch);
        d.k_up_plain = sp(-d.gap_extend);
        d.k_up_open = sp(-(d.gap_extend + d.gap_open_x));
        d.k_case = sp(d.case_bonus); d.k_cap = sp(d.cap_bonus); d.k_delim = sp(d.delim_bonus); d.k_base = sp(d.match_x);
        for (size_t i = 0; i < n; i++) { d.om16[i] = sp(d.om[i]); d.tg16[i] = sp(d.tg[i]); d.c16[i] = sp(d.c[i]); }
    }
    // the kernels keep cells in signed 16-bit lanes: every intermediate must stay below 2^15
    const uint64_t cell_bound = (uint64_t)n * ((uint64_t)sc.match_score + maxb + sc.matching_case_bonus) + sc.prefix_bonus +
                                (uint64_t)sc.mismatch_penalty + sc.match_score;
    const uint64_t pen_bound = (uint64_t)sw_lanes * sc.gap_extend_penalty + sc.gap_open_penalty;
    if (!needs_unicode && (cell_bound > 32767 || pen_bound > 32767))   // (the unicode kernel uses true u8/u16 lanes)
        return frz_fail(FRZ_ERR_UNSUPPORTED, "scoring/needle combination exceeds the kernels' signed 16-bit cell range");
    d.wrap8 = use_u8 && cell_bound > 255;  // cannot prove "no u8 add ever wraps" → emulate the wrap
    {   // column-limited SW classes need: padding bytes (0) never match, and plain (non-wrapping) arithmetic
        bool has_nul = false;
        for (int i = 0; i < d.n; i++) has_nul = has_nul || d.c[i] == 0;
        d.col_classes = (!d.wrap8 && !has_nul) ? 1 : 0;
    }
    if (max_typos < 0) d.typo_mode = FRZ_T_NONE;
    else if (max_typos == 0) d.typo_mode = FRZ_T_0;
    else if (max_typos == 1) d.typo_mode = FRZ_T_1;
    else if (max_typos == 2) d.typo_mode = FRZ_T_2;
    else {
        d.typo_mode = FRZ_T_MANY;
        if (max_typos > 15 && (size_t)max_typos < guard_len)
            return frz_fail(FRZ_ERR_UNSUPPORTED, "max_typos > 15 is not on the GPU path yet");
    }
    {   // Phase-A necessary condition on the signature index (frz_device.cuh: frz_sig_bucket).  A haystack accepted with
        // k typos holds a common subsequence of n - k needle bytes (the k >= 1 trackers never accept what LCS rejects,
        // DESIGN.md §2), so per byte class at most k needle bytes in total may lack a partner:
        //     sum_c max(0, m_c - cnt_c) <= k     >=     popc(need1 & ~occurs) + popc(need2 & ~occurs_twice)
        // The unicode trackers are the same trackers over needle SCALARS; there only the ASCII scalars are counted (see the
        // literal branch above), which keeps the sum a lower bound.
        uint32_t cnt[32] = {0};
        for (size_t i = 0; i < n; i++)
            if (!needs_unicode || d.c[i] < 0x80) cnt[frz_sig_bucket(d.c[i])]++;
        d.sig_need1 = d.sig_need2 = 0;
        for (int b2 = 0; b2 < 32; b2++) {
            if (cnt[b2] >= 1) d.sig_need1 |= 1u << b2;
            if (cnt[b2] >= 2) d.sig_need2 |= 1u << b2;
        }
        d.sig_on = max_typos >= 0 ? 1 : 0;                       // NO_PREFILTER scores everything
        d.sig_k = max_typos < 0 ? 0 : std::min<int>(max_typos, 64);
    }
    d.max_typos = max_typos < 0 ? 0 : std::min(max_typos, (int)guard_len);  // budget >= needle length matches everything
    // min_haystack_len (src/matcher/algo.rs:62-65)
    d.min_hay_len = max_typos >= 0 ? (int)(nchars > (size_t)max_typos ? nchars - max_typos : 0) : 0;
    uint64_t b = std::min<uint64_t>(cell_bound, use_u8 ? 255 : 0xFFFF) + sc.exact_match_bonus;
    c.score_bound = (uint32_t)std::min<uint64_t>(b, 0xFFFF);
    *out = c;
    return FRZ_OK;
}

}  // namespace

void FrzWorkspace::release() {
    if (device >= 0) cudaSetDevice(device);
    cudaFree(counters);
    cudaFree(stream_total); stream_total = nullptr;
    if (h_counters) cudaFreeHost(h_counters);
    for (auto& s : survivors) { cudaFree(s); s = nullptr; }
    cudaFree(surv_bitmap); cudaFree(word_prefix); surv_bitmap = nullptr; word_prefix = nullptr;
    cudaFree(tile_count); cudaFree(tile_out_base); cudaFree(matches_a); cudaFree(matches_b); cudaFree(sort_hist); cudaFree(cand_list);
    for (auto& e : ev) { if (e) cudaEventDestroy(e); e = nullptr; }
    if (table_ev) cudaEventDestroy(table_ev);
    table_ev = nullptr;
    counters = nullptr; h_counters = nullptr; tile_count = nullptr; tile_out_base = nullptr; matches_a = matches_b = nullptr;
    sort_hist = nullptr; cand_list = nullptr;
    cudaFree(retain_cnt); cudaFree(retain_base); cudaFree(retain_keep); retain_cnt = nullptr; retain_base = nullptr; retain_keep = nullptr; retain_cap = 0;
    cudaFree(unicode_scratch); unicode_scratch = nullptr; unicode_scratch_cap = 0;
    survivor_cap = match_cap = sort_hist_cap = cand_cap = 0; tiles_cap = 0; device = -1;
}

struct frz_matcher {
    frz_config config;
    std::vector<OwnedPattern> raw;
    std::vector<Compiled> compiled;   // build_patterns: patterns with non-empty needles
    FrzWorkspace ws;
    // end-to-end (host in / host out) staging arena, grow-only: raw Arrow buffers + a reusable packed corpus
    FrzIngest e2e_ingest;     // staging arena + copy stream of frz_match_list_host*
    frz_corpus e2e_corpus;
    FrzMatchDev* multi_a = nullptr;   // multi-pattern candidate ping-pong
    FrzMatchDev* multi_b = nullptr;
    uint64_t multi_cap = 0;
    float last_ms[4] = {0, 0, 0, 0};
    uint64_t last_launches = 0;
    // shard path: the match count is known after the tile scan, long before the scores; it is published there so
    // that the count exchange of match_list_parallel overlaps the Smith-Waterman and sort kernels
    uint64_t* early_count_dst = nullptr;   // device destination of the count (set for the duration of a shard call)
    cudaEvent_t count_ev = nullptr;        // recorded once the count is in early_count_dst
    bool count_published = false;
    bool timings_pending = false;
    uint64_t epoch = 0;                    // identity of the compiled patterns (clones made for another epoch are stale)
    int last_sort_bins = 0;                // bins of the single-pass score sort of the last call (0: none / two passes)
    ~frz_matcher() {
        if (ws.device >= 0) { cudaSetDevice(ws.device); cudaFree(multi_a); cudaFree(multi_b); if (count_ev) cudaEventDestroy(count_ev); }
        if (e2e_ingest.d_bytes || e2e_ingest.copy_stream || e2e_corpus.st.data) {
            cudaSetDevice(e2e_corpus.st.device);
            e2e_ingest.release();
            e2e_corpus.st.release();
        }
        ws.release();
    }
};

namespace {

std::atomic<uint64_t> g_matcher_epoch{1};

frz_status build_patterns(frz_matcher* m) {
    m->epoch = g_matcher_epoch.fetch_add(1);
    std::vector<Compiled> comp;
    for (const auto& p : m->raw) {
        bool none = false;
        Compiled c;
        FRZ_TRY(compile_pattern(p, m->config, &none, &c));
        if (!none) comp.push_back(c);
    }
    m->compiled.swap(comp);
    return FRZ_OK;
}

frz_status validate_config(const frz_config* c) {
    if (!c) return frz_fail(FRZ_ERR_INVALID_ARG, "null config");
    if (c->max_typos < -1 || c->max_typos > 65535) return frz_fail(FRZ_ERR_INVALID_ARG, "max_typos out of range");
    if (c->casing > 2 || c->unicode > 2 || c->matching > 4 || c->sort > 3) return frz_fail(FRZ_ERR_INVALID_ARG, "bad enum value in config");
    return FRZ_OK;
}

}  // namespace

extern "C" frz_status frz_matcher_create(const frz_pattern* patterns, size_t n_patterns, const frz_config* config, frz_matcher** out) {
    if (!out || (n_patterns && !patterns)) return frz_fail(FRZ_ERR_INVALID_ARG, "null argument");
    FRZ_TRY(validate_config(config));
    for (size_t i = 0; i < n_patterns; i++) {   // PatternConfig overrides (src/pattern.rs:230-246): -1 = inherit, else the enum range
        const frz_pattern& p = patterns[i];
        if (p.needle_len && !p.needle) return frz_fail(FRZ_ERR_INVALID_ARG, "pattern %zu: null needle", i);
        if (p.casing < -1 || p.casing > 2 || p.unicode < -1 || p.unicode > 2 || p.matching < -1 || p.matching > 4)
            return frz_fail(FRZ_ERR_INVALID_ARG, "pattern %zu: bad enum value in the per-pattern overrides", i);
        if (p.max_typos < -1 || p.max_typos > 65535) return frz_fail(FRZ_ERR_INVALID_ARG, "pattern %zu: max_typos out of range", i);
    }
    auto m = std::make_unique<frz_matcher>();
    m->config = *config;
    for (size_t i = 0; i < n_patterns; i++) {
        const frz_pattern& p = patterns[i];
        OwnedPattern o;
        o.needle.assign((const char*)p.needle, p.needle_len);
        o.raw = o.needle;
        o.negated = p.negated != 0;
        o.matching = p.matching; o.casing = p.casing; o.unicode = p.unicode; o.max_typos = p.max_typos;
        o.has_scoring = p.has_scoring != 0; o.scoring = p.scoring;
        m->raw.push_back(std::move(o));
    }
    FRZ_TRY(build_patterns(m.get()));
    *out = m.release();
    return FRZ_OK;
}

extern "C" frz_status frz_matcher_from_query(const uint8_t* query, size_t len, const frz_config* config, frz_matcher** out) {
    if (!out || (!query && len)) return frz_fail(FRZ_ERR_INVALID_ARG, "null argument");
    FRZ_TRY(validate_config(config));
    auto m = std::make_unique<frz_matcher>();
    m->config = *config;
    m->raw = parse_query(query, len);
    FRZ_TRY(build_patterns(m.get()));
    *out = m.release();
    return FRZ_OK;
}

extern "C" frz_status frz_matcher_set_config(frz_matcher* m, const frz_config* config) {
    if (!m) return frz_fail(FRZ_ERR_INVALID_ARG, "null matcher");
    FRZ_TRY(validate_config(config));
    if (memcmp(&m->config, config, sizeof *config) == 0) return FRZ_OK;
    frz_config old = m->config;
    m->config = *config;
    frz_status s = build_patterns(m);
    if (s != FRZ_OK) { m->config = old; build_patterns(m); }
    return s;
}

// `Matcher: Clone` (src/matcher/mod.rs:76): same patterns and config, fresh device scratch.  match_list_parallel clones
// the matcher once per worker (src/matcher/parallel.rs:46); frz_match_list_parallel does the same once per GPU.
extern "C" frz_status frz_matcher_clone(const frz_matcher* src, frz_matcher** out) {
    if (!src || !out) return frz_fail(FRZ_ERR_INVALID_ARG, "null argument");
    auto m = std::make_unique<frz_matcher>();
    m->config = src->config;
    m->raw = src->raw;
    FRZ_TRY(build_patterns(m.get()));
    *out = m.release();
    return FRZ_OK;
}
uint64_t frz_matcher_epoch(const frz_matcher* m) { return m ? m->epoch : 0; }
uint8_t frz_matcher_sort(const frz_matcher* m) { return m ? m->config.sort : 0; }
cudaEvent_t frz_matcher_table_event(const frz_matcher* m) { return (m && m->last_sort_bins && m->ws.table_ev_recorded) ? m->ws.table_ev : nullptr; }
const uint32_t* frz_matcher_last_sort_table(const frz_matcher* m, int* bins) {
    if (bins) *bins = m ? m->last_sort_bins : 0;
    return (m && m->last_sort_bins) ? frz_sort_digit_base(m->ws) : nullptr;
}

extern "C" void frz_matcher_destroy(frz_matcher* m) { delete m; }
extern "C" size_t frz_matcher_num_patterns(const frz_matcher* m) { return m ? m->compiled.size() : 0; }
extern "C" frz_status frz_matcher_backend_info(const frz_matcher* m, size_t i, int* lanes, int* score_bits, int* prefilter_lanes, int* is_literal) {
    if (!m || i >= m->compiled.size()) return frz_fail(FRZ_ERR_INVALID_ARG, "pattern index out of range");
    const auto& c = m->compiled[i];
    if (lanes) *lanes = c.dev.sw_lanes;
    if (score_bits) *score_bits = c.dev.score_bits;
    if (prefilter_lanes) *prefilter_lanes = c.dev.pf_lanes;
    if (is_literal) *is_literal = c.literal;
    return FRZ_OK;
}
void collect_timings(frz_matcher* m, const FrzLaunchStats& st);
extern "C" frz_status frz_matcher_last_timings(const frz_matcher* mc, float* ms4, uint64_t* launches) {
    frz_matcher* m = const_cast<frz_matcher*>(mc);
    if (!m) return frz_fail(FRZ_ERR_INVALID_ARG, "null matcher");
    if (m->timings_pending && m->ws.device >= 0) {
        cudaSetDevice(m->ws.device);
        cudaEventSynchronize(m->ws.ev[3]);
        FrzLaunchStats st;
        st.launches = m->last_launches;
        collect_timings(m, st);
        m->timings_pending = false;
    }
    if (ms4) memcpy(ms4, m->last_ms, sizeof m->last_ms);
    if (launches) *launches = m->last_launches;
    return FRZ_OK;
}

// ------------------------------------------------------------------------ small helper kernels

namespace {

__global__ void k_fill_all(FrzMatchDev* out, uint64_t n, uint32_t index_offset, FrzCounters* ctr) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        out[i] = FrzMatchDev{index_offset + (uint32_t)i, 0, 0, 0};
    if (blockIdx.x == 0 && threadIdx.x == 0) ctr->total = n;
}
__global__ void k_reverse(const FrzMatchDev* in, FrzMatchDev* out, const unsigned long long* n_ptr) {
    const unsigned long long n = *n_ptr;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x)
        out[n - 1 - i] = in[i];
}
// candidate bitmap over haystack indices (relative to index_offset)
__global__ void k_bitmap_set(const FrzMatchDev* cand, uint64_t n, uint32_t index_offset, uint32_t* bitmap) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t idx = cand[i].index - index_offset;
        atomicOr(&bitmap[idx >> 5], 1u << (idx & 31));
    }
}
// keep[i] = candidate i is (not) hit; hits are index-ordered → binary search
__device__ __forceinline__ long long find_hit(const FrzMatchDev* hits, uint64_t nh, uint32_t index) {
    uint64_t lo = 0, hi = nh;
    while (lo < hi) {
        uint64_t mid = (lo + hi) >> 1;
        if (hits[mid].index < index) lo = mid + 1; else hi = mid;
    }
    return (lo < nh && hits[lo].index == index) ? (long long)lo : -1;
}
// non-negated extra pattern: every hit is a surviving candidate; add the candidate's score
// (hit.score saturating_add, exact |=; src/matcher/multi.rs:133-147)
__global__ void k_combine_hits(const FrzMatchDev* cand, uint64_t nc, FrzMatchDev* hits, uint64_t nh) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nh; i += (uint64_t)gridDim.x * blockDim.x) {
        FrzMatchDev h = hits[i];
        long long j = find_hit(cand, nc, h.index);
        if (j >= 0) {
            uint32_t s = (uint32_t)h.score + cand[j].score;
            h.score = (uint16_t)(s > 0xFFFF ? 0xFFFF : s);
            h.exact |= cand[j].exact;
        }
        hits[i] = h;
    }
}
// negated extra pattern: retain candidates that were NOT hit (src/matcher/multi.rs:124-132).
// Stable compaction: per-block ballot counts → single-block scan → scatter.
constexpr int kCompactBlock = 1024;
__global__ void __launch_bounds__(kCompactBlock) k_retain_count(const FrzMatchDev* cand, uint64_t nc, const FrzMatchDev* hits, uint64_t nh,
                                                                uint32_t* block_count, uint8_t* keep) {
    __shared__ uint32_t wc[32];
    uint64_t i = (uint64_t)blockIdx.x * kCompactBlock + threadIdx.x;
    bool k = i < nc && find_hit(hits, nh, cand[i].index) < 0;
    if (i < nc) keep[i] = k;
    uint32_t b = __ballot_sync(0xffffffffu, k);
    if ((threadIdx.x & 31) == 0) wc[threadIdx.x >> 5] = __popc(b);
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t s = 0;
        for (int w = 0; w < 32; w++) s += wc[w];
        block_count[blockIdx.x] = s;
    }
}
__global__ void __launch_bounds__(kCompactBlock) k_retain_scatter(const FrzMatchDev* cand, uint64_t nc, const uint8_t* keep,
                                                                  const uint64_t* block_base, FrzMatchDev* out) {
    __shared__ uint32_t wc[32];
    uint64_t i = (uint64_t)blockIdx.x * kCompactBlock + threadIdx.x;
    bool k = i < nc && keep[i];
    uint32_t b = __ballot_sync(0xffffffffu, k);
    uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) wc[warp] = __popc(b);
    __syncthreads();
    uint32_t pre = 0;
    for (uint32_t w = 0; w < warp; w++) pre += wc[w];
    if (k) out[block_base[blockIdx.x] + pre + __popc(b & ((1u << lane) - 1))] = cand[i];
}
__global__ void __launch_bounds__(1024) k_scan_blocks(const uint32_t* cnt, uint64_t* base, uint32_t n, FrzCounters* ctr) {
    __shared__ uint64_t carry;
    __shared__ uint64_t ws[32];
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (uint32_t b0 = 0; b0 < n; b0 += blockDim.x) {
        uint32_t i = b0 + threadIdx.x;
        uint64_t v = i < n ? cnt[i] : 0, x = v;
        for (int d = 1; d < 32; d <<= 1) { uint64_t y = __shfl_up_sync(0xffffffffu, x, d); if ((threadIdx.x & 31) >= (unsigned)d) x += y; }
        if ((threadIdx.x & 31) == 31) ws[threadIdx.x >> 5] = x;
        __syncthreads();
        if (threadIdx.x < 32) {
            uint64_t w = ws[threadIdx.x], xs = w;
            for (int d = 1; d < 32; d <<= 1) { uint64_t y = __shfl_up_sync(0xffffffffu, xs, d); if (threadIdx.x >= (unsigned)d) xs += y; }
            ws[threadIdx.x] = xs - w;
        }
        __syncthreads();
        uint64_t incl = carry + ws[threadIdx.x >> 5] + x;
        if (i < n) base[i] = incl - v;
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) carry = incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) ctr->total = carry;
}

frz_status ensure_workspace(frz_matcher* m, const FrzCorpusStorage& cs, uint64_t survivor_cap) {
    FrzWorkspace& ws = m->ws;
    if (ws.device != cs.device) {
        if (ws.device >= 0) { cudaSetDevice(ws.device); cudaFree(m->multi_a); cudaFree(m->multi_b); m->multi_a = m->multi_b = nullptr; m->multi_cap = 0; }
        ws.release();
        FRZ_CUDA_TRY(cudaSetDevice(cs.device));
        ws.device = cs.device;
        FRZ_CUDA_TRY(cudaMalloc(&ws.counters, sizeof(FrzCounters)));
        FRZ_CUDA_TRY(cudaMalloc(&ws.stream_total, 2 * sizeof(unsigned long long)));   // [0] tile-scan carry, [1] spare count slot
        FRZ_CUDA_TRY(cudaMallocHost(&ws.h_counters, sizeof(FrzCounters)));
        for (auto& e : ws.ev) FRZ_CUDA_TRY(cudaEventCreate(&e));
        FRZ_CUDA_TRY(cudaEventCreateWithFlags(&ws.table_ev, cudaEventDisableTiming));
        FRZ_TRY(frz_sort_hist_alloc(&ws.sort_hist));
        ws.sort_hist_cap = frz_sort_hist_words();
    }
    if (ws.tiles_cap < cs.n_tiles) {
        cudaFree(ws.tile_count); cudaFree(ws.tile_out_base); cudaFree(ws.surv_bitmap); cudaFree(ws.word_prefix);
        ws.tile_count = nullptr; ws.tile_out_base = nullptr; ws.surv_bitmap = nullptr; ws.word_prefix = nullptr; ws.tiles_cap = 0;
        FRZ_CUDA_TRY(cudaMalloc(&ws.surv_bitmap, (size_t)cs.n_tiles * 32 * sizeof(uint32_t)));
        FRZ_CUDA_TRY(cudaMalloc(&ws.word_prefix, (size_t)cs.n_tiles * 32 * sizeof(uint16_t)));
        FRZ_CUDA_TRY(cudaMalloc(&ws.tile_count, (size_t)cs.n_tiles * sizeof(uint32_t)));
        FRZ_CUDA_TRY(cudaMalloc(&ws.tile_out_base, (size_t)cs.n_tiles * sizeof(uint64_t)));
        ws.tiles_cap = cs.n_tiles;
    }
    if (ws.survivor_cap < survivor_cap) {
        for (auto& s : ws.survivors) { cudaFree(s); s = nullptr; }
        ws.survivor_cap = 0;
        for (auto& s : ws.survivors) FRZ_CUDA_TRY(cudaMalloc(&s, (size_t)survivor_cap * sizeof(FrzSurvivor)));
        ws.survivor_cap = survivor_cap;
    }
    if (ws.cand_cap < std::max<uint64_t>(cs.n, 1)) {   // worst case: every haystack passes the signature test
        cudaFree(ws.cand_list); ws.cand_list = nullptr; ws.cand_cap = 0;
        const uint64_t want = std::max<uint64_t>(cs.n, 1);
        FRZ_CUDA_TRY(cudaMalloc(&ws.cand_list, (size_t)want * 16));
        ws.cand_cap = want;
    }
    if (ws.match_cap < cs.n) {
        cudaFree(ws.matches_a); cudaFree(ws.matches_b);
        ws.matches_a = ws.matches_b = nullptr; ws.match_cap = 0;
        FRZ_CUDA_TRY(cudaMalloc(&ws.matches_a, (size_t)std::max<uint64_t>(cs.n, 1) * sizeof(FrzMatchDev)));
        FRZ_CUDA_TRY(cudaMalloc(&ws.matches_b, (size_t)std::max<uint64_t>(cs.n, 1) * sizeof(FrzMatchDev)));
        ws.match_cap = cs.n;
    }
    return FRZ_OK;
}

// multi-pattern candidate ping-pong / two-pass sort scratch: grow-only, always >= n entries after this call
frz_status ensure_multi_buffers(frz_matcher* m, uint64_t n) {
    if (m->multi_a && m->multi_b && m->multi_cap >= std::max<uint64_t>(n, 1)) return FRZ_OK;
    cudaFree(m->multi_a); cudaFree(m->multi_b);
    m->multi_a = m->multi_b = nullptr; m->multi_cap = 0;
    const uint64_t want = std::max<uint64_t>(n, 1);
    FRZ_CUDA_TRY(cudaMalloc(&m->multi_a, (size_t)want * sizeof(FrzMatchDev)));
    FRZ_CUDA_TRY(cudaMalloc(&m->multi_b, (size_t)want * sizeof(FrzMatchDev)));
    m->multi_cap = want;
    return FRZ_OK;
}

uint64_t initial_survivor_cap(const FrzCorpusStorage& cs, const FrzPatternDev& d) {
    if (d.typo_mode == FRZ_T_NONE) return std::max<uint64_t>(cs.n, 1);
    return std::min<uint64_t>(std::max<uint64_t>(cs.n / 4, 1 << 16), std::max<uint64_t>(cs.n, 1));
}

// One pattern over the corpus (optionally restricted to a candidate bitmap) → index-ordered matches in
// d_out (reversed order if `reversed`); the count is left in ws.counters->total (device).
frz_status run_pattern(frz_matcher* m, const FrzCorpusStorage& cs, const Compiled& c, const uint32_t* cand_bitmap,
                       uint32_t index_offset, bool reversed, FrzMatchDev* d_out, cudaStream_t stream, FrzLaunchStats* st,
                       bool record_events, const FrzMatchDev* cand_list = nullptr, uint64_t n_cand = 0) {
    FrzWorkspace& ws = m->ws;
    const FrzCorpusView cv = cs.view();
    uint64_t cap = std::max(ws.survivor_cap, initial_survivor_cap(cs, c.dev));
    FRZ_TRY(ensure_workspace(m, cs, cap));
    FRZ_CUDA_TRY(cudaMemsetAsync(ws.counters, 0, sizeof(FrzCounters), stream));
    if (record_events) { cudaEventRecord(ws.ev[0], stream); ws.ev_rec[0] = true; }
    if (c.unicode) FRZ_TRY(frz_launch_unicode(cv, c.dev, c.un, c.usc, cand_list, n_cand, index_offset, ws, stream, st));
    else if (cand_list) FRZ_TRY(frz_launch_prefilter_list(cv, c.dev, cand_list, n_cand, index_offset, ws, stream, st));
    else FRZ_TRY(frz_launch_prefilter(cv, c.dev, ws, stream, st));
    FRZ_TRY(frz_launch_tile_scan(cv, ws, stream, st));
    if (record_events) { cudaEventRecord(ws.ev[1], stream); ws.ev_rec[1] = true; }
    if (m->early_count_dst && !cand_list && !cand_bitmap && m->compiled.size() == 1) {
        // single pattern: every survivor becomes exactly one match, so the scan total is the final count
        FRZ_CUDA_TRY(cudaMemcpyAsync(m->early_count_dst, &ws.counters->total, sizeof(uint64_t), cudaMemcpyDeviceToDevice, stream));
        FRZ_CUDA_TRY(cudaEventRecord(m->count_ev, stream));
        m->count_published = true;
    }
    // A survivor-list overflow (lists are sized by a heuristic unless the pattern can match everything)
    // only sets a sticky device flag; whoever reads the counters back re-runs with worst-case lists.
    if (c.unicode) {
        // the unicode kernel has already scored its survivors: they travel as literal-style records (score, exact)
        FrzPatternDev emit = c.dev;
        emit.typo_mode = FRZ_T_LITERAL;
        FRZ_TRY(frz_launch_sw(cv, emit, index_offset, reversed, ws, d_out, stream, st));
    } else {
        FRZ_TRY(frz_launch_sw(cv, c.dev, index_offset, reversed, ws, d_out, stream, st));
    }
    if (record_events) { cudaEventRecord(ws.ev[2], stream); ws.ev_rec[2] = true; }
    return FRZ_OK;
}

constexpr frz_status kRetryOverflow = (frz_status)100;

frz_status read_counters(frz_matcher* m, cudaStream_t stream) {
    FrzWorkspace& ws = m->ws;
    FRZ_CUDA_TRY(cudaMemcpyAsync(ws.h_counters, ws.counters, sizeof(FrzCounters), cudaMemcpyDeviceToHost, stream));
    FRZ_CUDA_TRY(cudaStreamSynchronize(stream));
    if (ws.h_counters->error & FRZ_DEVERR_SURVIVOR_OVERFLOW) return kRetryOverflow;
    return FRZ_OK;
}

int grid_for(uint64_t n, int block) {
    uint64_t g = (n + block - 1) / block;
    return (int)std::max<uint64_t>(1, std::min<uint64_t>(g, 148 * 16));
}

// match_list_into over all compiled patterns → index-ordered device list; returns pointer + leaves the
// count in ws.counters->total.  `final_reversed` asks for the list in descending index order.
frz_status match_into_device(frz_matcher* m, const FrzCorpusStorage& cs, uint32_t index_offset, bool final_reversed,
                             FrzMatchDev** d_result, uint32_t* score_bound, cudaStream_t stream, FrzLaunchStats* st,
                             FrzMatchDev* prefer_out = nullptr) {
    FrzWorkspace& ws = m->ws;
    if ((uint64_t)cs.n + index_offset > 0xFFFFFFFFull)
        return frz_fail(FRZ_ERR_TOO_MANY_ITEMS, "too many items in haystack, will overflow the u32 index: %llu > %u (index offset: %u)",
                        (unsigned long long)cs.n + index_offset, 0xFFFFFFFFu, index_offset);
    const auto& pats = m->compiled;
    *score_bound = 0;
    if (pats.empty()) {  // CompiledPatterns::Empty (src/matcher/mod.rs:380-383)
        FRZ_TRY(ensure_workspace(m, cs, 1));
        FRZ_CUDA_TRY(cudaMemsetAsync(ws.counters, 0, sizeof(FrzCounters), stream));
        k_fill_all<<<grid_for(cs.n, 256), 256, 0, stream>>>(ws.matches_a, cs.n, index_offset, ws.counters);
        st->launches++;
        if (final_reversed) {
            k_reverse<<<grid_for(cs.n, 256), 256, 0, stream>>>(ws.matches_a, ws.matches_b, &ws.counters->total);
            st->launches++;
            *d_result = ws.matches_b;
        } else *d_result = ws.matches_a;
        FRZ_CUDA_TRY(cudaGetLastError());
        return FRZ_OK;
    }
    if (pats.size() == 1 && !pats[0].negated) {  // CompiledPatterns::Single
        FRZ_TRY(ensure_workspace(m, cs, initial_survivor_cap(cs, pats[0].dev)));
        FrzMatchDev* dst = prefer_out ? prefer_out : ws.matches_a;
        FRZ_TRY(run_pattern(m, cs, pats[0], nullptr, index_offset, final_reversed, dst, stream, st, true));
        *d_result = dst;
        *score_bound = pats[0].score_bound;
        return FRZ_OK;
    }
    // CompiledPatterns::Multi (src/matcher/multi.rs:84-152).  Counts are read back between patterns.
    FRZ_TRY(ensure_workspace(m, cs, initial_survivor_cap(cs, pats[0].dev)));
    FRZ_TRY(ensure_multi_buffers(m, cs.n));
    int base = -1;
    for (size_t i = 0; i < pats.size(); i++) if (!pats[i].negated) { base = (int)i; break; }
    FrzMatchDev* cand = m->multi_a;
    FrzMatchDev* spare = m->multi_b;
    uint64_t nc = 0;
    uint64_t bound = 0;
    if (base >= 0) {
        FRZ_TRY(run_pattern(m, cs, pats[base], nullptr, index_offset, false, cand, stream, st, true));
        FRZ_TRY(read_counters(m, stream));
        nc = ws.h_counters->total;
        bound = pats[base].score_bound;
    } else {
        FRZ_CUDA_TRY(cudaMemsetAsync(ws.counters, 0, sizeof(FrzCounters), stream));
        k_fill_all<<<grid_for(cs.n, 256), 256, 0, stream>>>(cand, cs.n, index_offset, ws.counters);
        st->launches++;
        nc = cs.n;
    }
    if (ws.retain_cap < cs.n) {
        cudaFree(ws.retain_cnt); cudaFree(ws.retain_base); cudaFree(ws.retain_keep);
        ws.retain_cnt = nullptr; ws.retain_base = nullptr; ws.retain_keep = nullptr; ws.retain_cap = 0;
        const uint32_t nb_max = (uint32_t)((cs.n + kCompactBlock - 1) / kCompactBlock) + 1;
        FRZ_CUDA_TRY(cudaMalloc(&ws.retain_cnt, nb_max * sizeof(uint32_t)));
        FRZ_CUDA_TRY(cudaMalloc(&ws.retain_base, nb_max * sizeof(uint64_t)));
        FRZ_CUDA_TRY(cudaMalloc(&ws.retain_keep, std::max<uint64_t>(cs.n, 1)));
        ws.retain_cap = cs.n;
    }
    uint32_t* d_block_cnt = ws.retain_cnt;
    uint64_t* d_block_base = ws.retain_base;
    uint8_t* d_keep = ws.retain_keep;
    frz_status status = FRZ_OK;
    for (size_t pi = 0; pi < pats.size() && status == FRZ_OK; pi++) {
        if ((int)pi == base || nc == 0) continue;
        status = [&]() -> frz_status {
            // evaluate the pattern on the surviving candidates only; hits land in ws.matches_a, index-ordered,
            // with real indices
            FRZ_TRY(run_pattern(m, cs, pats[pi], nullptr, index_offset, false, ws.matches_a, stream, st, false, cand, nc));
            FRZ_TRY(read_counters(m, stream));
            const uint64_t nh = ws.h_counters->total;
            if (pats[pi].negated) {
                const uint32_t nb = (uint32_t)((nc + kCompactBlock - 1) / kCompactBlock);
                k_retain_count<<<nb, kCompactBlock, 0, stream>>>(cand, nc, ws.matches_a, nh, d_block_cnt, d_keep);
                k_scan_blocks<<<1, 1024, 0, stream>>>(d_block_cnt, d_block_base, nb, ws.counters);
                k_retain_scatter<<<nb, kCompactBlock, 0, stream>>>(cand, nc, d_keep, d_block_base, spare);
                st->launches += 3;
                FRZ_TRY(read_counters(m, stream));
                nc = ws.h_counters->total;
                std::swap(cand, spare);
            } else {
                k_combine_hits<<<grid_for(nh, 256), 256, 0, stream>>>(cand, nc, ws.matches_a, nh);
                st->launches++;
                FRZ_CUDA_TRY(cudaMemcpyAsync(spare, ws.matches_a, nh * sizeof(FrzMatchDev), cudaMemcpyDeviceToDevice, stream));
                std::swap(cand, spare);
                nc = nh;
                bound += pats[pi].score_bound;
            }
            return FRZ_OK;
        }();
    }
    FRZ_TRY(status);
    // publish: count → counters.total, list → matches_a (reversed if asked)
    ws.h_counters->total = nc;
    FRZ_CUDA_TRY(cudaMemcpyAsync(&ws.counters->total, &ws.h_counters->total, sizeof(unsigned long long), cudaMemcpyHostToDevice, stream));
    if (final_reversed) {
        k_reverse<<<grid_for(nc, 256), 256, 0, stream>>>(cand, ws.matches_a, &ws.counters->total);
        st->launches++;
    } else {
        FRZ_CUDA_TRY(cudaMemcpyAsync(ws.matches_a, cand, nc * sizeof(FrzMatchDev), cudaMemcpyDeviceToDevice, stream));
    }
    FRZ_CUDA_TRY(cudaGetLastError());
    *d_result = ws.matches_a;
    *score_bound = (uint32_t)std::min<uint64_t>(bound, 0xFFFF);
    return FRZ_OK;
}

// Matcher::match_list on device: into (+reverse) (+stable score sort).  Result pointer + device count.
__global__ void k_copy_n(const FrzMatchDev* __restrict__ in, FrzMatchDev* __restrict__ out, const unsigned long long* n_ptr) {
    const unsigned long long n = *n_ptr;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x)
        out[i] = in[i];
}

// `final_out` (optional, device, >= corpus length): where the final list must land
frz_status match_list_device(frz_matcher* m, const FrzCorpusStorage& cs, uint32_t index_offset, uint8_t sort,
                             FrzMatchDev** d_result, cudaStream_t stream, FrzLaunchStats* st, FrzMatchDev* final_out = nullptr) {
    FrzWorkspace& ws = m->ws;
    const bool reversed = sort == FRZ_SORT_INDEX_DESC || sort == FRZ_SORT_SCORE_THEN_INDEX_DESC;
    const bool by_score = sort == FRZ_SORT_SCORE_THEN_INDEX_ASC || sort == FRZ_SORT_SCORE_THEN_INDEX_DESC;
    const bool will_sort = by_score && !m->compiled.empty();
    for (bool& f : ws.ev_rec) f = false;
    m->last_sort_bins = 0;
    FrzMatchDev* d_list = nullptr;
    uint32_t bound = 0;
    FRZ_TRY(match_into_device(m, cs, index_offset, reversed, &d_list, &bound, stream, st, will_sort ? nullptr : final_out));
    // `!self.patterns.is_empty() && sort.is_by_score()` (src/matcher/mod.rs:218)
    if (will_sort) {
        FrzMatchDev* other = final_out ? final_out : (d_list == ws.matches_a ? ws.matches_b : ws.matches_a);
        // two-pass sort (score bound >= 1024) needs a scratch list of the corpus size: the multi-pattern ping-pong
        // buffer is free at this point (d_list is never multi_a); grow it whenever THIS corpus is larger
        FrzMatchDev* tmp = nullptr;
        if (bound >= 1024) {
            FRZ_TRY(ensure_multi_buffers(m, cs.n));
            tmp = m->multi_a;
        }
        FRZ_TRY(frz_launch_sort_by_score_dev(d_list, tmp, other, &ws.counters->total, bound, ws, stream, st));
        m->last_sort_bins = frz_sort_single_pass_bins(bound);
        d_list = other;
    } else if (final_out && d_list != final_out) {
        k_copy_n<<<grid_for(cs.n, 256), 256, 0, stream>>>(d_list, final_out, &ws.counters->total);
        st->launches++;
        d_list = final_out;
    }
    cudaEventRecord(ws.ev[3], stream);
    ws.ev_rec[3] = true;
    *d_result = d_list;
    return FRZ_OK;
}

}  // namespace
void collect_timings(frz_matcher* m, const FrzLaunchStats& st) {
    FrzWorkspace& ws = m->ws;
    float a = 0, b = 0, c = 0, t = 0;
    const bool* r = ws.ev_rec;
    if (r[0] && r[1] && cudaEventElapsedTime(&a, ws.ev[0], ws.ev[1]) != cudaSuccess) a = 0;
    if (r[1] && r[2] && cudaEventElapsedTime(&b, ws.ev[1], ws.ev[2]) != cudaSuccess) b = 0;
    if (r[2] && r[3] && cudaEventElapsedTime(&c, ws.ev[2], ws.ev[3]) != cudaSuccess) c = 0;
    if (r[0] && r[3] && cudaEventElapsedTime(&t, ws.ev[0], ws.ev[3]) != cudaSuccess) t = 0;
    cudaGetLastError();
    m->last_ms[0] = a; m->last_ms[1] = b; m->last_ms[2] = c; m->last_ms[3] = t;
    m->last_launches = st.launches;
}
namespace {

frz_status copy_out(frz_matcher* m, FrzMatchDev* d_list, frz_match* out, uint64_t cap, uint64_t* n_out, cudaStream_t stream) {
    FRZ_TRY(read_counters(m, stream));
    const uint64_t n = m->ws.h_counters->total;
    if (n_out) *n_out = n;
    if (n > cap) return frz_fail(FRZ_ERR_CAPACITY, "output capacity %llu < %llu matches", (unsigned long long)cap, (unsigned long long)n);
    if (n) {
        if (!out) return frz_fail(FRZ_ERR_INVALID_ARG, "null out");
        static_assert(sizeof(frz_match) == sizeof(FrzMatchDev), "layout");
        FRZ_CUDA_TRY(cudaMemcpyAsync(out, d_list, n * sizeof(frz_match), cudaMemcpyDeviceToHost, stream));
        FRZ_CUDA_TRY(cudaStreamSynchronize(stream));
    }
    return FRZ_OK;
}

}  // namespace

extern "C" frz_status frz_match_list(frz_matcher* m, const frz_corpus* corpus, frz_match* out, uint64_t cap, uint64_t* n_out) {
    if (!m || !corpus) return frz_fail(FRZ_ERR_INVALID_ARG, "null argument");
    FRZ_TRY(ensure_device(corpus->st.device));
    cudaStream_t stream = nullptr;
    FrzLaunchStats st;
    FrzMatchDev* d_list = nullptr;
    frz_status s = FRZ_OK;
    for (int attempt = 0; attempt < 2; attempt++) {
        s = match_list_device(m, corpus->st, 0, m->config.sort, &d_list, stream, &st);
        if (s == FRZ_OK) s = copy_out(m, d_list, out, cap, n_out, stream);
        if (s != kRetryOverflow) break;
        FRZ_TRY(ensure_workspace(m, corpus->st, std::max<uint64_t>(corpus->st.n, 1)));  // worst-case lists, then once more
    }
    if (s == kRetryOverflow) s = frz_fail(FRZ_ERR_CUDA, "survivor list overflow persisted");
    collect_timings(m, st);
    return s;
}

extern "C" frz_status frz_match_list_into(frz_matcher* m, const frz_corpus* corpus, uint32_t index_offset, frz_match* out,
                                          uint64_t cap, uint64_t* n_out) {
    if (!m || !corpus) return frz_fail(FRZ_ERR_INVALID_ARG, "null argument");
    FRZ_TRY(ensure_device(corpus->st.device));
    cudaStream_t stream = nullptr;
    FrzLaunchStats st;
    FrzMatchDev* d_list = nullptr;
    frz_status s = FRZ_OK;
    for (int attempt = 0; attempt < 2; attempt++) {
        s = match_list_device(m, corpus->st, index_offset, FRZ_SORT_INDEX_ASC, &d_list, stream, &st);
        if (s == FRZ_OK) s = copy_out(m, d_list, out, cap, n_out, stream);
        if (s != kRetryOverflow) break;
        FRZ_TRY(ensure_workspace(m, corpus->st, std::max<uint64_t>(corpus->st.n, 1)));
    }
    if (s == kRetryOverflow) s = frz_fail(FRZ_ERR_CUDA, "survivor list overflow persisted");
    collect_timings(m, st);
    return s;
}

namespace {   // defined with the shard calls below
bool streamed_eligible(const frz_matcher* m, uint64_t n, uint32_t index_offset);
frz_status match_streamed_impl(frz_matcher* m, const uint8_t* bytes, const void* offsets, int offset_width, uint64_t n, int device,
                               uint32_t index_offset, FrzMatchDev* d_out, uint64_t* d_count, cudaStream_t stream, FrzMatchDev** d_result);
}  // namespace

// End to end from host Arrow buffers: streamed H2D + pack (pack.cu: ingest_host_t), match, D2H of the matches.
extern "C" frz_status frz_match_list_host_arrow(frz_matcher* m, const uint8_t* bytes, const void* offsets, int offset_width, uint64_t n,
                                                int device, frz_match* out, uint64_t cap, uint64_t* n_out) {
    if (!m || !offsets) return frz_fail(FRZ_ERR_INVALID_ARG, "null argument");
    if (offset_width != 4 && offset_width != 8) return frz_fail(FRZ_ERR_INVALID_ARG, "offset_width must be 4 or 8");
    if (n > 0xFFFFFFFFull) return frz_fail(FRZ_ERR_TOO_MANY_ITEMS, "too many items in haystack: %llu", (unsigned long long)n);
    if (streamed_eligible(m, n, 0)) {   // the match pipeline runs while the list streams in (frz_match_shard_streamed)
        FrzMatchDev* d_list = nullptr;
        FRZ_TRY(match_streamed_impl(m, bytes, offsets, offset_width, n, device, 0, nullptr, nullptr, nullptr, &d_list));
        const frz_status s = copy_out(m, d_list, out, cap, n_out, nullptr);
        m->timings_pending = false;
        FrzLaunchStats st; st.launches = m->last_launches;
        collect_timings(m, st);
        return s;
    }
    const frz_corpus* c = nullptr;
    FRZ_TRY(frz_matcher_ingest_e2e(m, bytes, offsets, offset_width, n, device, &c));
    return frz_match_list(m, c, out, cap, n_out);
}

// The ingest half of the end-to-end call: host Arrow buffers → the matcher's reusable packed corpus (grow-only staging
// arena, streamed H2D overlapped with the pack kernels; asynchronous on the legacy default stream).
frz_status frz_matcher_ingest_e2e(frz_matcher* m, const uint8_t* bytes, const void* offsets, int offset_width, uint64_t n, int device,
                                  const frz_corpus** out) {
    if (!m || !offsets || !out) return frz_fail(FRZ_ERR_INVALID_ARG, "null argument");
    if (offset_width != 4 && offset_width != 8) return frz_fail(FRZ_ERR_INVALID_ARG, "offset_width must be 4 or 8");
    if (n > 0xFFFFFFFFull) return frz_fail(FRZ_ERR_TOO_MANY_ITEMS, "too many items in haystack: %llu", (unsigned long long)n);
    FRZ_TRY(ensure_device(device));
    cudaStream_t stream = nullptr;
    frz_corpus& c = m->e2e_corpus;
    if (c.st.device != device && (m->e2e_ingest.d_bytes || m->e2e_ingest.copy_stream || c.st.data)) {  // arena lives on another device
        cudaSetDevice(c.st.device);
        m->e2e_ingest.release();
        c.st.release();
        FRZ_CUDA_TRY(cudaSetDevice(device));
    }
    c.st.device = device;
    FRZ_TRY(frz_ingest_host(m->e2e_ingest, bytes, offsets, offset_width, n, stream, &c.st));
    *out = &c;
    return FRZ_OK;
}

extern "C" frz_status frz_match_list_host(frz_matcher* m, const uint8_t* bytes, const uint64_t* offsets, uint64_t n, int device,
                                          frz_match* out, uint64_t cap, uint64_t* n_out) {
    return frz_match_list_host_arrow(m, bytes, offsets, 8, n, device, out, cap, n_out);
}

// Matcher::match_list_indices for chosen haystacks (src/matcher/mod.rs:234-262): Match + matched byte offsets.
namespace {
// one pattern over the chosen rows: match_one_indices_impl (fuzzy / literal), results in host arrays
frz_status match_indices_one(const Compiled& c, const frz_corpus* corpus, const uint32_t* which, uint64_t n, frz_match* out_matches,
                             uint32_t* out_indices, uint32_t stride, uint32_t* out_counts) {
    cudaStream_t stream = nullptr;
    const uint32_t threads = (uint32_t)std::min<uint64_t>(n, 1024);
    const int rows = c.unicode ? c.un.n : c.un.nbytes;
    const uint64_t sstride = c.literal ? 1 : (uint64_t)frzi::indices_scratch_elems(rows, c.dev.sw_lanes);
    uint32_t *d_which = nullptr, *d_idx = nullptr, *d_cnt = nullptr;
    FrzMatchDev* d_m = nullptr;
    uint16_t* d_scratch = nullptr;
    frz_status st = [&]() -> frz_status {
        FRZ_CUDA_TRY(cudaMalloc(&d_which, n * sizeof(uint32_t)));
        FRZ_CUDA_TRY(cudaMalloc(&d_idx, n * (uint64_t)stride * sizeof(uint32_t)));
        FRZ_CUDA_TRY(cudaMalloc(&d_cnt, n * sizeof(uint32_t)));
        FRZ_CUDA_TRY(cudaMalloc(&d_m, n * sizeof(FrzMatchDev)));
        FRZ_CUDA_TRY(cudaMalloc(&d_scratch, (uint64_t)threads * sstride * sizeof(uint16_t)));
        FRZ_CUDA_TRY(cudaMemcpyAsync(d_which, which, n * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
        FRZ_CUDA_TRY(cudaMemsetAsync(d_m, 0, n * sizeof(FrzMatchDev), stream));
        FRZ_TRY(frz_launch_match_indices(corpus->st.view(), c.dev, c.un, c.usc, c.unicode, d_which, n, d_m, d_idx, stride, d_cnt,
                                         d_scratch, sstride, threads, stream));
        FRZ_CUDA_TRY(cudaMemcpyAsync(out_matches, d_m, n * sizeof(FrzMatchDev), cudaMemcpyDeviceToHost, stream));
        FRZ_CUDA_TRY(cudaMemcpyAsync(out_indices, d_idx, n * (uint64_t)stride * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
        FRZ_CUDA_TRY(cudaMemcpyAsync(out_counts, d_cnt, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
        FRZ_CUDA_TRY(cudaStreamSynchronize(stream));
        return FRZ_OK;
    }();
    cudaFree(d_which); cudaFree(d_idx); cudaFree(d_cnt); cudaFree(d_m); cudaFree(d_scratch);
    return st;
}
}  // namespace

extern "C" frz_status frz_match_indices(frz_matcher* m, const frz_corpus* corpus, const uint32_t* which, uint64_t n,
                                        frz_match* out_matches, uint32_t* out_indices, uint32_t stride, uint32_t* out_counts) {
    if (!m || !corpus || (n && (!which || !out_matches || !out_indices || !out_counts)) || stride == 0)
        return frz_fail(FRZ_ERR_INVALID_ARG, "null argument");
    if (m->compiled.empty()) return frz_fail(FRZ_ERR_INVALID_ARG, "the matcher has no pattern");
    if (n == 0) return FRZ_OK;
    FRZ_TRY(ensure_device(corpus->st.device));
    if (m->compiled.size() == 1 && !m->compiled[0].negated)   // CompiledPatterns::Single
        return match_indices_one(m->compiled[0], corpus, which, n, out_matches, out_indices, stride, out_counts);
    // CompiledPatterns::Multi → match_one_indices_multi (src/matcher/multi.rs:56-79): a negated atom that matches drops the
    // row, the others add their scores, OR their exact flags and pool their indices (sorted descending, de-duplicated)
    // every atom yields at most one index per needle scalar (<= FRZ_MAX_NEEDLE): pool with an internal stride that
    // cannot truncate an atom, cut the pooled (sorted, de-duplicated) list at the caller's stride afterwards
    const uint32_t istride = std::max<uint32_t>(stride, FRZ_MAX_NEEDLE);
    std::vector<frz_match> pm(n);
    std::vector<uint32_t> pi((size_t)n * istride), pc(n);
    std::vector<std::vector<uint32_t>> pooled(n);
    std::vector<uint8_t> alive(n, 1);
    for (uint64_t j = 0; j < n; j++) out_matches[j] = frz_match{which[j], 0, 0, 0};
    for (const Compiled& c : m->compiled) {
        FRZ_TRY(match_indices_one(c, corpus, which, n, pm.data(), pi.data(), istride, pc.data()));
        for (uint64_t j = 0; j < n; j++) {
            if (!alive[j]) continue;
            const bool hit = pc[j] != 0xFFFFFFFFu;
            if (c.negated) { if (hit) alive[j] = 0; continue; }
            if (!hit) { alive[j] = 0; continue; }
            const uint32_t sum = (uint32_t)out_matches[j].score + pm[j].score;
            out_matches[j].score = (uint16_t)std::min<uint32_t>(sum, 0xFFFF);
            out_matches[j].exact |= pm[j].exact;
            const size_t got = std::min<size_t>(pc[j], istride);
            pooled[j].insert(pooled[j].end(), pi.begin() + (size_t)j * istride, pi.begin() + (size_t)j * istride + got);
        }
    }
    for (uint64_t j = 0; j < n; j++) {
        if (!alive[j]) { out_counts[j] = 0xFFFFFFFFu; continue; }
        auto& v = pooled[j];
        std::sort(v.begin(), v.end(), [](uint32_t a, uint32_t b) { return a > b; });
        v.erase(std::unique(v.begin(), v.end()), v.end());
        out_counts[j] = (uint32_t)v.size();   // untruncated: a value > stride tells the caller the row was cut
        for (uint32_t k = 0; k < std::min<uint32_t>(out_counts[j], stride); k++) out_indices[(size_t)j * stride + k] = v[k];
    }
    return FRZ_OK;
}

extern "C" frz_status frz_match_shard_device(frz_matcher* m, const frz_corpus* shard, uint32_t index_offset, frz_match* d_out,
                                             uint64_t cap, uint64_t* d_count, void* stream_) {
    if (!m || !shard || !d_out || !d_count) return frz_fail(FRZ_ERR_INVALID_ARG, "null argument");
    FRZ_TRY(ensure_device(shard->st.device));
    cudaStream_t stream = (cudaStream_t)stream_;
    FrzLaunchStats st;
    FrzMatchDev* d_list = nullptr;
    // asynchronous entry point: nobody reads the overflow flag back, so size the lists for the worst case
    FRZ_TRY(ensure_workspace(m, shard->st, std::max<uint64_t>(shard->st.n, 1)));
    // the run can never exceed the shard size; the caller sizes d_out as >= shard length
    if (cap < shard->st.n) return frz_fail(FRZ_ERR_CAPACITY, "d_out must hold the whole shard (%llu)", (unsigned long long)shard->st.n);
    if (!m->count_ev) FRZ_CUDA_TRY(cudaEventCreateWithFlags(&m->count_ev, cudaEventDisableTiming));
    m->early_count_dst = d_count;
    m->count_published = false;
    m->ws.arm_table_ev = true;
    m->ws.table_ev_recorded = false;
    const frz_status ms = match_list_device(m, shard->st, index_offset, m->config.sort, &d_list, stream, &st, reinterpret_cast<FrzMatchDev*>(d_out));
    m->early_count_dst = nullptr;
    m->ws.arm_table_ev = false;
    FRZ_TRY(ms);
    if (!m->count_published) {   // multi-pattern / empty pattern: the count exists only at the end
        FRZ_CUDA_TRY(cudaMemcpyAsync(d_count, &m->ws.counters->total, sizeof(uint64_t), cudaMemcpyDeviceToDevice, stream));
        FRZ_CUDA_TRY(cudaEventRecord(m->count_ev, stream));
    }
    m->last_launches = st.launches;
    m->timings_pending = true;   // events were recorded; frz_matcher_last_timings reads them once the stream is idle
    return FRZ_OK;
}

// Makes `stream` wait until the count of the last frz_match_shard_device call has been written to its d_count
// (which happens before the scoring kernels for a single-pattern matcher).
extern "C" frz_status frz_matcher_wait_count(frz_matcher* m, void* stream) {
    if (!m) return frz_fail(FRZ_ERR_INVALID_ARG, "null matcher");
    if (!m->count_ev) return frz_fail(FRZ_ERR_INVALID_ARG, "no shard call has been made on this matcher");
    FRZ_CUDA_TRY(cudaStreamWaitEvent((cudaStream_t)stream, m->count_ev, 0));
    return FRZ_OK;
}

// ---- streamed shard call: host Arrow buffers in, locally ordered run out, the match pipeline overlapped with the H2D copy ----
// The tiles of a packed corpus are independent, so the pipeline can run on tiles [t0, t1) through a SUB-VIEW of the corpus
// (array pointers advanced to tile t0; unit addresses are absolute) as soon as their H2D chunk has been packed: length gate →
// signature scan → exact windows → tile scan (carrying the running match count, so every range appends to the same
// index-ordered list) → scoring.  Only the score sort waits for the last chunk.  The copy engine stays busy from the first
// byte to the last; what is left after the last chunk lands is one range's pipeline + the sort instead of the whole list's.
namespace {
struct StreamedCtx {
    frz_matcher* m;
    const Compiled* c;
    uint32_t index_offset;
    FrzMatchDev* dst;       // index-ordered matches (pre-sort)
    cudaStream_t stream;
    FrzLaunchStats* st;
    uint32_t pending_t0;    // first tile not yet matched
    int chunks_pending;     // packed chunks since the last range
    int group;              // chunks per range
};
frz_status streamed_range(StreamedCtx& x, uint32_t t0, uint32_t t1, bool last) {
    frz_matcher* m = x.m;
    FrzWorkspace& ws = m->ws;
    const FrzCorpusStorage& cs = m->e2e_corpus.st;
    FrzCorpusView cv = cs.view();
    cv.tile_base += t0;
    cv.groups += (size_t)t0 * FRZ_GROUPS_PER_TILE;
    cv.slot_meta += (size_t)t0 * FRZ_TILE;
    cv.slot_of += (size_t)t0 * FRZ_TILE;
    cv.slot_sig += (size_t)t0 * FRZ_TILE;
    cv.n = std::min<uint64_t>(cs.n, (uint64_t)t1 * FRZ_TILE) - (uint64_t)t0 * FRZ_TILE;
    cv.n_tiles = t1 - t0;
    const uint32_t off = x.index_offset + t0 * FRZ_TILE;
    FRZ_CUDA_TRY(cudaMemsetAsync(ws.counters, 0, sizeof(FrzCounters), x.stream));
    FRZ_TRY(frz_launch_prefilter(cv, x.c->dev, ws, x.stream, x.st));
    FRZ_TRY(frz_launch_tile_scan(cv, ws, x.stream, x.st, ws.stream_total));
    if (last) {
        cudaEventRecord(ws.ev[1], x.stream); ws.ev_rec[1] = true;
        if (m->early_count_dst) {   // the running count is final: publish it before the last range is scored
            FRZ_CUDA_TRY(cudaMemcpyAsync(m->early_count_dst, &ws.counters->total, sizeof(uint64_t), cudaMemcpyDeviceToDevice, x.stream));
            FRZ_CUDA_TRY(cudaEventRecord(m->count_ev, x.stream));
            m->count_published = true;
        }
    }
    FRZ_TRY(frz_launch_sw(cv, x.c->dev, off, false, ws, x.dst, x.stream, x.st));
    return FRZ_OK;
}
frz_status streamed_after_chunk(void* ctx, uint32_t t0, uint32_t t1, bool last) {
    StreamedCtx& x = *static_cast<StreamedCtx*>(ctx);
    (void)t0;
    x.chunks_pending++;
    if (!last && x.chunks_pending < x.group) return FRZ_OK;
    const uint32_t r0 = x.pending_t0;
    x.pending_t0 = t1;
    x.chunks_pending = 0;
    if (t1 <= r0) return FRZ_OK;
    return streamed_range(x, r0, t1, last);
}
}  // namespace

namespace {
bool streamed_eligible(const frz_matcher* m, uint64_t n, uint32_t index_offset) {
    const uint8_t sort = m->config.sort;
    return m->compiled.size() == 1 && !m->compiled[0].negated && !m->compiled[0].unicode &&
           (sort == FRZ_SORT_INDEX_ASC || sort == FRZ_SORT_SCORE_THEN_INDEX_ASC) &&   // reversed lists need the final total per element
           n >= 64 * FRZ_TILE && (uint64_t)n + index_offset <= 0xFFFFFFFFull;
}
}  // namespace
// (match_streamed_impl: d_out == nullptr leaves the list in the matcher's own buffer, returned through d_result;
//  d_count == nullptr uses a spare device slot)

frz_status frz_match_shard_streamed(frz_matcher* m, const uint8_t* bytes, const void* offsets, int offset_width, uint64_t n, int device,
                                    uint32_t index_offset, frz_match* d_out, uint64_t cap, uint64_t* d_count, void* stream_) {
    if (!m || !offsets || !d_out || !d_count) return frz_fail(FRZ_ERR_INVALID_ARG, "null argument");
    if (offset_width != 4 && offset_width != 8) return frz_fail(FRZ_ERR_INVALID_ARG, "offset_width must be 4 or 8");
    if (!streamed_eligible(m, n, index_offset)) {
        const frz_corpus* shard = nullptr;
        FRZ_TRY(frz_matcher_ingest_e2e(m, bytes, offsets, offset_width, n, device, &shard));
        return frz_match_shard_device(m, shard, index_offset, d_out, cap, d_count, stream_);
    }
    if (cap < n) return frz_fail(FRZ_ERR_CAPACITY, "d_out must hold the whole shard (%llu)", (unsigned long long)n);
    return match_streamed_impl(m, bytes, offsets, offset_width, n, device, index_offset, reinterpret_cast<FrzMatchDev*>(d_out), d_count,
                               (cudaStream_t)stream_, nullptr);
}

namespace {
frz_status match_streamed_impl(frz_matcher* m, const uint8_t* bytes, const void* offsets, int offset_width, uint64_t n, int device,
                               uint32_t index_offset, FrzMatchDev* d_out, uint64_t* d_count, cudaStream_t stream, FrzMatchDev** d_result) {
    const uint8_t sort = m->config.sort;
    FRZ_TRY(ensure_device(device));
    frz_corpus& c = m->e2e_corpus;
    if (c.st.device != device && (m->e2e_ingest.d_bytes || m->e2e_ingest.copy_stream || c.st.data)) {  // arena lives on another device
        cudaSetDevice(c.st.device);
        m->e2e_ingest.release();
        c.st.release();
        FRZ_CUDA_TRY(cudaSetDevice(device));
    }
    c.st.device = device;
    c.st.n = n;
    c.st.n_tiles = (uint32_t)((n + FRZ_TILE - 1) / FRZ_TILE);
    FrzWorkspace& ws = m->ws;
    FRZ_TRY(ensure_workspace(m, c.st, std::max<uint64_t>(n, 1)));   // nobody reads the overflow flag back: worst-case lists
    if (!m->count_ev) FRZ_CUDA_TRY(cudaEventCreateWithFlags(&m->count_ev, cudaEventDisableTiming));
    const Compiled& pat = m->compiled[0];
    const bool will_sort = sort == FRZ_SORT_SCORE_THEN_INDEX_ASC;
    FrzMatchDev* final_out = d_out ? d_out : ws.matches_b;
    if (!d_count) d_count = reinterpret_cast<uint64_t*>(ws.stream_total + 1);
    if (d_result) *d_result = final_out;
    FrzLaunchStats st;
    for (bool& f : ws.ev_rec) f = false;
    m->last_sort_bins = 0;
    m->early_count_dst = d_count;
    m->count_published = false;
    ws.arm_table_ev = true;
    ws.table_ev_recorded = false;
    StreamedCtx x;
    x.m = m; x.c = &pat; x.index_offset = index_offset; x.dst = will_sort ? ws.matches_a : final_out; x.stream = stream; x.st = &st;
    x.pending_t0 = 0; x.chunks_pending = 0;
    x.group = 4;   // a range per four H2D chunks (about 1/8 of the list): the tail after the last chunk is one range + the sort
    const frz_status ms = [&]() -> frz_status {
        FRZ_CUDA_TRY(cudaMemsetAsync(ws.stream_total, 0, sizeof(unsigned long long), stream));
        cudaEventRecord(ws.ev[0], stream); ws.ev_rec[0] = true;
        FRZ_TRY(frz_ingest_host(m->e2e_ingest, bytes, offsets, offset_width, n, stream, &c.st, streamed_after_chunk, &x));
        cudaEventRecord(ws.ev[2], stream); ws.ev_rec[2] = true;
        if (will_sort) {
            FrzMatchDev* tmp = nullptr;
            if (pat.score_bound >= 1024) { FRZ_TRY(ensure_multi_buffers(m, n)); tmp = m->multi_a; }
            FRZ_TRY(frz_launch_sort_by_score_dev(ws.matches_a, tmp, final_out, &ws.counters->total, pat.score_bound, ws, stream, &st));
            m->last_sort_bins = frz_sort_single_pass_bins(pat.score_bound);
        }
        cudaEventRecord(ws.ev[3], stream); ws.ev_rec[3] = true;
        return FRZ_OK;
    }();
    m->early_count_dst = nullptr;
    ws.arm_table_ev = false;
    FRZ_TRY(ms);
    if (!m->count_published) {   // (cannot happen with >= 1 chunk; kept for symmetry with frz_match_shard_device)
        FRZ_CUDA_TRY(cudaMemcpyAsync(d_count, &ws.counters->total, sizeof(uint64_t), cudaMemcpyDeviceToDevice, stream));
        FRZ_CUDA_TRY(cudaEventRecord(m->count_ev, stream));
    }
    m->last_launches = st.launches;
    m->timings_pending = true;
    return FRZ_OK;
}
}  // namespace

namespace {
// Run metadata travels BY VALUE as a kernel parameter (1 KB of the 4 KB parameter space): no staging buffer, so
// back-to-back merges with different counts cannot race and the entry point needs no per-call H2D copy.
struct MergeMeta {
    uint64_t counts[FRZ_MERGE_MAX_RUNS];   // valid entries of run r
    uint64_t bases[FRZ_MERGE_MAX_RUNS];    // concatenation offset of the r-th run in merge order
    uint64_t total;
};

__global__ void k_gather_runs(const FrzMatchDev* runs, uint64_t stride, const __grid_constant__ MergeMeta meta, int n_runs,
                              int reverse_runs, FrzMatchDev* out, unsigned long long* d_total) {
    if (blockIdx.x == 0 && threadIdx.x == 0 && d_total) *d_total = meta.total;
    for (int r = 0; r < n_runs; r++) {
        const int src_run = reverse_runs ? n_runs - 1 - r : r;
        const FrzMatchDev* src = runs + (uint64_t)src_run * stride;
        const uint64_t cnt = meta.counts[src_run], base = meta.bases[r];
        for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < cnt; i += (uint64_t)gridDim.x * blockDim.x)
            out[base + i] = src[i];
    }
}

// ---- k-way merge of score-sorted runs (src/k_merge.rs:90-131) without comparing heads -------------------
// Every run is sorted by score descending, so "the elements of run r with score s" is the index range
// [gt[r][s], gt[r][s-1]) where gt[r][s] = #elements of run r with score > s — a binary search per (r, s).
// The merged position of that block is  Σ_r' gt[r'][s]  (everything with a higher score)  +  the sizes of the
// same-score blocks of the runs that come earlier in the merge order; one scatter pass places the elements.
constexpr int kMergeMaxBins = 4096;

__global__ void k_merge_bounds(const FrzMatchDev* __restrict__ runs, uint64_t stride, const __grid_constant__ MergeMeta meta,
                               int n_runs, int bins, uint32_t* __restrict__ gt) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_runs * bins) return;
    const int r = t / bins;
    const uint32_t s = (uint32_t)(t - r * bins);
    const FrzMatchDev* run = runs + (uint64_t)r * stride;
    uint64_t lo = 0, hi = meta.counts[r];   // first index whose score <= s
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if (run[mid].score > s) lo = mid + 1; else hi = mid;
    }
    gt[t] = (uint32_t)lo;
}

// pos0[r][s] = merged position of the first element of run r's score-s block.  One thread per score.
__global__ void k_merge_bases(const uint32_t* __restrict__ gt, const __grid_constant__ MergeMeta meta, int n_runs, int bins,
                              int reverse_runs, uint32_t* __restrict__ pos0) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= bins) return;
    uint32_t higher = 0;
    for (int r = 0; r < n_runs; r++) higher += gt[r * bins + s];
    uint32_t acc = higher;
    for (int k = 0; k < n_runs; k++) {
        const int r = reverse_runs ? n_runs - 1 - k : k;
        pos0[r * bins + s] = acc;
        const uint32_t ge = s == 0 ? (uint32_t)meta.counts[r] : gt[r * bins + s - 1];   // #elements with score >= s
        acc += ge - gt[r * bins + s];
    }
}

// One pass over the gathered runs: gridDim.y = n_runs rows of blocks, one row per run, so every run streams at
// full width (the first version looped over the runs inside one grid: short runs left most blocks idle).
__global__ void __launch_bounds__(256) k_merge_scatter(const FrzMatchDev* __restrict__ runs, uint64_t stride,
                                                       const __grid_constant__ MergeMeta meta, int bins,
                                                       const uint32_t* __restrict__ gt, const uint32_t* __restrict__ pos0,
                                                       FrzMatchDev* __restrict__ out) {
    const int r = blockIdx.y;
    const FrzMatchDev* run = runs + (uint64_t)r * stride;
    const uint64_t cnt = meta.counts[r];
    const uint32_t* gtr = gt + (size_t)r * bins;
    const uint32_t* p0r = pos0 + (size_t)r * bins;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < cnt; i += (uint64_t)gridDim.x * blockDim.x) {
        const FrzMatchDev m = run[i];
        const uint32_t s = min((uint32_t)m.score, (uint32_t)bins - 1);
        out[p0r[s] + ((uint32_t)i - gtr[s])] = m;
    }
}
}  // namespace

// k_merge_matches_by (src/k_merge.rs:90-131).  Runs are index-range shards in rank order, each already
// ordered per `sort`; concatenating them in (reverse) rank order and stable-sorting by score yields
// exactly the reference's k-way merge (ties resolve by index because the shards are index-ordered).
// Debugging / test aid: the compiled device pattern of pattern i (the struct the kernels receive), so that host
// builds of the kernel cores (tests/test_kernel_logic_cpu.py) run with exactly the constants the GPU gets.
extern "C" frz_status frz_matcher_debug_pattern(const frz_matcher* m, size_t i, void* out, size_t out_size) {
    if (!m || !out || i >= m->compiled.size()) return frz_fail(FRZ_ERR_INVALID_ARG, "pattern index out of range");
    if (out_size != sizeof(FrzPatternDev)) return frz_fail(FRZ_ERR_INVALID_ARG, "expected a buffer of %zu bytes", sizeof(FrzPatternDev));
    memcpy(out, &m->compiled[i].dev, sizeof(FrzPatternDev));
    return FRZ_OK;
}

extern "C" uint32_t frz_matcher_score_bound(const frz_matcher* m) {
    if (!m) return 0;
    uint64_t b = 0;
    for (const auto& c : m->compiled) if (!c.negated) b += c.score_bound;
    return (uint32_t)std::min<uint64_t>(b, 0xFFFF);
}

void FrzMergeScratch::release() {
    if (device >= 0) cudaSetDevice(device);
    cudaFree(hist); cudaFree(tables); cudaFree(cat); cudaFree(tmp); cudaFree(d_total);
    hist = tables = nullptr; cat = tmp = nullptr; d_total = nullptr; cap = 0; device = -1;
}

// k_merge_matches_by on `stream` with caller-owned scratch (one per concurrent user; grow-only).
frz_status frz_merge_runs_ex(FrzMergeScratch& ms, const FrzMatchDev* runs, uint64_t run_stride, const uint64_t* run_counts_host,
                             int n_runs, uint8_t sort, uint32_t score_bound_in, FrzMatchDev* d_out, cudaStream_t stream) {
    if (!runs || !run_counts_host || !d_out || n_runs <= 0 || n_runs > FRZ_MERGE_MAX_RUNS) return frz_fail(FRZ_ERR_INVALID_ARG, "bad argument");
    const bool reversed = sort == FRZ_SORT_INDEX_DESC || sort == FRZ_SORT_SCORE_THEN_INDEX_DESC;
    const bool by_score = sort == FRZ_SORT_SCORE_THEN_INDEX_ASC || sort == FRZ_SORT_SCORE_THEN_INDEX_DESC;
    const uint32_t score_bound = score_bound_in ? score_bound_in : 0xFFFF;
    MergeMeta meta;
    memset(&meta, 0, sizeof meta);
    uint64_t total = 0;
    for (int r = 0; r < n_runs; r++) {
        meta.counts[r] = run_counts_host[r];
        const int src_run = reversed ? n_runs - 1 - r : r;
        meta.bases[r] = total;
        total += run_counts_host[src_run];
    }
    meta.total = total;
    if (ms.device < 0) {
        int dev = 0;
        FRZ_CUDA_TRY(cudaGetDevice(&dev));
        FRZ_TRY(frz_sort_hist_alloc(&ms.hist));
        FRZ_CUDA_TRY(cudaMalloc(&ms.tables, (size_t)2 * FRZ_MERGE_MAX_RUNS * kMergeMaxBins * sizeof(uint32_t)));
        FRZ_CUDA_TRY(cudaMalloc(&ms.d_total, sizeof(unsigned long long)));
        ms.device = dev;
    }
    const int bins = (int)std::min<uint32_t>(score_bound, 0xFFFFu) + 1;
    if (total == 0) return FRZ_OK;
    if (by_score && bins <= kMergeMaxBins && total <= 0xFFFFFFFFull) {
        // score-sorted runs: boundaries by binary search, one scatter pass (no concatenation, no re-sort)
        uint32_t* gt = ms.tables;
        uint32_t* pos0 = ms.tables + (size_t)FRZ_MERGE_MAX_RUNS * kMergeMaxBins;
        k_merge_bounds<<<(n_runs * bins + 255) / 256, 256, 0, stream>>>(runs, run_stride, meta, n_runs, bins, gt);
        k_merge_bases<<<(bins + 127) / 128, 128, 0, stream>>>(gt, meta, n_runs, bins, reversed ? 1 : 0, pos0);
        uint64_t longest = 0;
        for (int r = 0; r < n_runs; r++) longest = std::max(longest, run_counts_host[r]);
        const dim3 grid((unsigned)std::max<uint64_t>(1, std::min<uint64_t>((longest + 255) / 256, 148 * 8 / std::max(n_runs, 1) + 1)), (unsigned)n_runs);
        k_merge_scatter<<<grid, 256, 0, stream>>>(runs, run_stride, meta, bins, gt, pos0, d_out);
        FRZ_CUDA_TRY(cudaGetLastError());
        return FRZ_OK;  // asynchronous on `stream`
    }
    if (by_score && ms.cap < total) {
        cudaFree(ms.cat); cudaFree(ms.tmp); ms.cat = ms.tmp = nullptr; ms.cap = 0;
        const uint64_t want = total + total / 4 + 1024;
        FRZ_CUDA_TRY(cudaMalloc(&ms.cat, want * sizeof(FrzMatchDev)));
        FRZ_CUDA_TRY(cudaMalloc(&ms.tmp, want * sizeof(FrzMatchDev)));
        ms.cap = want;
    }
    FrzMatchDev* dst = by_score ? ms.cat : d_out;
    k_gather_runs<<<grid_for(total / std::max(n_runs, 1) + 1, 256), 256, 0, stream>>>(runs, run_stride, meta, n_runs, reversed ? 1 : 0, dst,
                                                                                     ms.d_total);
    if (by_score) {
        FrzWorkspace ws;  // only the sort scratch is used
        ws.sort_hist = ms.hist;
        FRZ_TRY(frz_launch_sort_by_score_dev(ms.cat, ms.tmp, d_out, ms.d_total, score_bound, ws, stream, nullptr));
    }
    FRZ_CUDA_TRY(cudaGetLastError());
    return FRZ_OK;  // asynchronous on `stream`
}

extern "C" frz_status frz_merge_runs_device(const frz_match* d_runs, uint64_t run_stride, const uint64_t* run_counts_host,
                                            int n_runs, uint8_t sort, uint32_t score_bound_in, frz_match* d_out, int device, void* stream_) {
    if (!d_runs || !run_counts_host || !d_out || n_runs <= 0 || n_runs > FRZ_MERGE_MAX_RUNS) return frz_fail(FRZ_ERR_INVALID_ARG, "bad argument");
    FRZ_TRY(ensure_device(device));
    if (device >= 64) return frz_fail(FRZ_ERR_INVALID_ARG, "device index too large");
    // grow-only per-device scratch (tables only: the run metadata travels as kernel parameters).  Calls for one device
    // must be stream-ordered with each other, as documented in the header.
    static FrzMergeScratch scratch[64];
    static std::mutex mu;
    std::lock_guard<std::mutex> lock(mu);
    return frz_merge_runs_ex(scratch[device], reinterpret_cast<const FrzMatchDev*>(d_runs), run_stride, run_counts_host, n_runs, sort,
                             score_bound_in, reinterpret_cast<FrzMatchDev*>(d_out), (cudaStream_t)stream_);
}

extern "C" frz_status frz_radix_sort_matches(frz_match* matches, uint64_t n, int device) {
    if (n == 0) return FRZ_OK;
    if (!matches) return frz_fail(FRZ_ERR_INVALID_ARG, "null matches");
    FRZ_TRY(ensure_device(device));
    FrzMatchDev *d_a = nullptr, *d_b = nullptr, *d_c = nullptr;
    unsigned long long* d_n = nullptr;
    FrzWorkspace ws;
    cudaStream_t stream = nullptr;
    frz_status s = [&]() -> frz_status {
        FRZ_CUDA_TRY(cudaMalloc(&d_a, n * sizeof(FrzMatchDev)));
        FRZ_CUDA_TRY(cudaMalloc(&d_b, n * sizeof(FrzMatchDev)));
        FRZ_CUDA_TRY(cudaMalloc(&d_c, n * sizeof(FrzMatchDev)));
        FRZ_CUDA_TRY(cudaMalloc(&d_n, sizeof(unsigned long long)));
        FRZ_TRY(frz_sort_hist_alloc(&ws.sort_hist));
        unsigned long long hn = n;
        FRZ_CUDA_TRY(cudaMemcpyAsync(d_n, &hn, sizeof hn, cudaMemcpyHostToDevice, stream));
        FRZ_CUDA_TRY(cudaMemcpyAsync(d_a, matches, n * sizeof(FrzMatchDev), cudaMemcpyHostToDevice, stream));
        FRZ_TRY(frz_launch_sort_by_score_dev(d_a, d_b, d_c, d_n, 0xFFFF, ws, stream, nullptr));
        FRZ_CUDA_TRY(cudaMemcpyAsync(matches, d_c, n * sizeof(FrzMatchDev), cudaMemcpyDeviceToHost, stream));
        FRZ_CUDA_TRY(cudaStreamSynchronize(stream));
        return FRZ_OK;
    }();
    cudaFree(d_a); cudaFree(d_b); cudaFree(d_c); cudaFree(d_n); cudaFree(ws.sort_hist);
    return s;
}
