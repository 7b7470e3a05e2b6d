// The text side of `place_sequences`, native and host-only (no CUDA):
//   cls_records_render   cls_result arrays + query headers + the Clade fields of the tree -> the bytes the reference
//                        appends to `<out>.yaml|.jsonl` and `<out>.error`
//                        (core/src/use_cases/place_sequences/mod.rs:160-249; PlacementResponse / PlacementStatus:
//                        domain/dtos/placement_response.rs:7-94; AdherenceTest: adherence_test.rs:6-17; Clade:
//                        clade.rs:18-38; the annotation join along the path to the root: mod.rs:180-224, clade.rs:95-125).
//                        serde_yaml 0.9 block style and serde_json compact style are reproduced for this fixed record
//                        shape: floats as the ryu crate prints them, strings quoted only where libyaml would quote them.
//                        One block of records per task on the host pool, concatenated in input order.
//   cls_filter_sequence  SequenceBody::remove_non_iupac_from_sequence (sequence.rs:47-56)
//   cls_fasta_read       the reader of file_or_stdin.rs:76-116 (chunks of whole lines scanned on the host pool)
//   cls_fastq_read       the FASTQ reader (four-line records; chunks of whole records read on the host pool)
//   cls_sequences_open / cls_sequences_write / cls_place_sequences
//                        the use-case itself (mod.rs:43-270): path handling, reader, cls_place_batch, writer
// The Python mirror (classeq2_b200/placement.py) is the second implementation of all of it; tests hold the two
// byte-identical, and both equal to a reference-written result file.
#include <algorithm>
#include <atomic>
#include <charconv>
#include <cstdio>
#include <stdexcept>
#include <cmath>
#include <cstdlib>
#include <cerrno>
#include <cstring>
#include <future>
#include <memory>
#include <string>
#include <unordered_map>
#include <vector>

#include <sys/stat.h>
#include <sys/types.h>

#include "../../include/classeq_b200.h"
#include "fastq_rules.hpp"
#include "host_pool.hpp"
#include "last_error.hpp"

namespace {

// ---- f64 as serde_yaml / serde_json print it (the ryu crate): shortest round-trip digits, decimal notation for
//      1e-5 <= |x| < 1e16, exponent form outside, a trailing ".0" on integral values in decimal notation ----------
void ryu_float(double x, bool json, std::string &out) {
    if (std::isnan(x)) { out += json ? "null" : ".nan"; return; }
    if (std::isinf(x)) { out += json ? "null" : (x > 0 ? ".inf" : "-.inf"); return; }
    if (x == 0) { out += std::signbit(x) ? "-0.0" : "0.0"; return; }
    if (x < 0) { out += '-'; x = -x; }
    char buf[64];
    auto r = std::to_chars(buf, buf + sizeof buf, x, std::chars_format::scientific);  // d[.ddd]e[+-]XX, shortest round trip
    const char *e = static_cast<const char *>(memchr(buf, 'e', (size_t)(r.ptr - buf)));
    std::string digits;
    for (const char *p = buf; p < e; ++p)
        if (*p != '.') digits += *p;
    while (digits.size() > 1 && digits.back() == '0') digits.pop_back();
    const int exp10 = atoi(std::string(e + 1, static_cast<const char *>(r.ptr)).c_str());
    const int kk = exp10 + 1;  // value = 0.d1d2... * 10^kk
    const int n = (int)digits.size();
    if (0 < kk && kk <= 16) {
        if (n <= kk) { out += digits; out.append((size_t)(kk - n), '0'); out += ".0"; }
        else { out.append(digits, 0, (size_t)kk); out += '.'; out.append(digits, (size_t)kk, std::string::npos); }
    } else if (-5 < kk && kk <= 0) {
        out += "0."; out.append((size_t)(-kk), '0'); out += digits;
    } else {
        out += digits[0];
        if (n > 1) { out += '.'; out.append(digits, 1, std::string::npos); }
        out += 'e'; out += std::to_string(kk - 1);
    }
}

// ---- strings ------------------------------------------------------------------------------------------------
// serde_yaml 0.9 (ser.rs serialize_str -> de.rs visit_untagged_scalar; the crate is not vendored in the reference tree, this
// restates its published source): a string that would read back as null, a boolean, an integer or a finite float under
// the YAML 1.2 core schema - or as digits with a leading zero - is emitted single-quoted; for everything else the style is
// libyaml's choice.
bool reads_as_another_type(const std::string &s) {
    static const char *words[] = {"null", "Null", "NULL", "~", "true", "True", "TRUE", "false", "False", "FALSE"};
    if (s.empty()) return true;
    for (const char *w : words)
        if (s == w) return true;
    for (unsigned char c : s)
        if (c >= 0x80) return false;
    const std::string body = (s[0] == '+' || s[0] == '-') ? s.substr(1) : s;
    auto digit = [](char c) { return c >= '0' && c <= '9'; };
    if (body.size() > 2 && body[0] == '0' && (body[1] == 'x' || body[1] == 'o' || body[1] == 'b')) {   // parse_unsigned_int / parse_negative_int
        const int bits_per = body[1] == 'x' ? 4 : body[1] == 'o' ? 3 : 1;
        bool ok = true;
        size_t first = std::string::npos;   // first non-zero digit
        for (size_t i = 2; i < body.size() && ok; ++i) {
            const char c = body[i];
            const int v = digit(c) ? c - '0' : (c >= 'a' && c <= 'f') ? c - 'a' + 10 : (c >= 'A' && c <= 'F') ? c - 'A' + 10 : 99;
            ok = v < (1 << bits_per);
            if (ok && v && first == std::string::npos) first = i;
        }
        if (ok) {
            if (first == std::string::npos) return true;   // zero
            const char c = body[first];
            const int v = digit(c) ? c - '0' : (c | 0x20) - 'a' + 10;
            int top = 0;
            while ((v >> top) > 1) ++top;                   // bit length of the leading digit - 1
            const size_t bits = (body.size() - first - 1) * (size_t)bits_per + (size_t)top + 1;
            if (bits <= 128) return true;                   // fits u128 (from_str_radix)
        }
    }
    bool all_digits = !body.empty();
    for (char c : body) all_digits = all_digits && digit(c);
    if (all_digits) return true;                            // an integer, or digits_but_not_number (a leading zero)
    std::string unpositive = s;
    if (s[0] == '+') {
        unpositive = s.substr(1);
        if (!unpositive.empty() && (unpositive[0] == '+' || unpositive[0] == '-')) return false;
    }
    if (unpositive == ".inf" || unpositive == ".Inf" || unpositive == ".INF" || s == "-.inf" || s == "-.Inf" || s == "-.INF" ||
        s == ".nan" || s == ".NaN" || s == ".NAN")
        return true;
    // str::parse::<f64>(): [+-]? (digits+ [. digits*] | . digits+) [(e|E) [+-]? digits+], then is_finite()
    size_t i = 0;
    const std::string &u = unpositive;
    if (i < u.size() && (u[i] == '+' || u[i] == '-')) ++i;
    size_t ni = 0, nf = 0;
    while (i < u.size() && digit(u[i])) { ++i; ++ni; }
    if (i < u.size() && u[i] == '.') {
        ++i;
        while (i < u.size() && digit(u[i])) { ++i; ++nf; }
    }
    if (ni + nf == 0) return false;
    if (i < u.size() && (u[i] == 'e' || u[i] == 'E')) {
        ++i;
        if (i < u.size() && (u[i] == '+' || u[i] == '-')) ++i;
        size_t ne = 0;
        while (i < u.size() && digit(u[i])) { ++i; ++ne; }
        if (ne == 0) return false;
    }
    if (i != u.size()) return false;
    return std::isfinite(strtod(u.c_str(), nullptr));
}

// One UTF-8 code point of s starting at byte i (advances i); malformed bytes come back as 0xFFFF'FFFF (treated as special).
uint32_t next_cp(const std::string &s, size_t &i) {
    const unsigned char *p = reinterpret_cast<const unsigned char *>(s.data());
    const size_t n = s.size() - i;
    const unsigned char c = p[i];
    auto cont = [&](size_t k) { return (p[i + k] & 0xC0) == 0x80; };
    if (c < 0x80) { ++i; return c; }
    if ((c & 0xE0) == 0xC0 && n >= 2 && cont(1)) { const uint32_t v = ((c & 0x1Fu) << 6) | (p[i + 1] & 0x3Fu); i += 2; return v; }
    if ((c & 0xF0) == 0xE0 && n >= 3 && cont(1) && cont(2)) {
        const uint32_t v = ((c & 0x0Fu) << 12) | ((p[i + 1] & 0x3Fu) << 6) | (p[i + 2] & 0x3Fu); i += 3; return v;
    }
    if ((c & 0xF8) == 0xF0 && n >= 4 && cont(1) && cont(2) && cont(3)) {
        const uint32_t v = ((c & 0x07u) << 18) | ((p[i + 1] & 0x3Fu) << 12) | ((p[i + 2] & 0x3Fu) << 6) | (p[i + 3] & 0x3Fu); i += 4; return v;
    }
    ++i;
    return 0xFFFFFFFFu;
}

// Outside libyaml's printable set (IS_PRINTABLE: 0x0A, 0x20-0x7E, 0x85, 0xA0-0xD7FF, 0xE000-0xFFFD without the BOM); 0x85
// and the Unicode line separators count as breaks, which a quoted one-line scalar cannot hold unescaped either.
bool yaml_special(uint32_t o) {
    return o < 0x20 || o == 0x7F || (o >= 0x80 && o <= 0x9F) || o == 0x2028 || o == 0x2029 || o == 0xFEFF ||
           (o >= 0xD800 && o <= 0xDFFF) || o >= 0xFFFE;
}
bool has_yaml_special(const std::string &s) {
    for (size_t i = 0; i < s.size();)
        if (yaml_special(next_cp(s, i))) return true;
    return false;
}

// whether libyaml (hence serde_yaml) may emit the string as a plain scalar - or, for text that reads as a number, a
// boolean or null, whether serde_yaml leaves the choice to libyaml at all
bool yaml_plain_ok(const std::string &s) {
    if (reads_as_another_type(s)) return false;                                     // serde_yaml forces single quotes
    if (s.front() == ' ' || s.back() == ' ') return false;                          // libyaml looks at 0x20 only
    if (s.compare(0, 3, "---") == 0 || s.compare(0, 3, "...") == 0) return false;   // document markers
    static const char special[] = "-?:,[]{}#&*!|>'\"%@`";
    if (strchr(special, s[0]) && !(strchr("-?:", s[0]) && s.size() > 1 && s[1] != ' ' && s[1] != '\t')) return false;
    if (s.find(": ") != std::string::npos || s.find(" #") != std::string::npos || s.back() == ':') return false;
    if (has_yaml_special(s)) return false;
    return true;
}

void yaml_string(const std::string &s, int indent, std::string &out) {
    if (s.find('\n') != std::string::npos) {  // literal block scalar, serde_yaml's choice for multi-line strings
        const bool keep = s.back() == '\n';
        const std::string body = keep ? s.substr(0, s.size() - 1) : s;
        out += keep ? "|" : "|-";
        size_t a = 0;
        for (;;) {
            const size_t b = body.find('\n', a);
            const std::string ln = body.substr(a, b == std::string::npos ? std::string::npos : b - a);
            out += '\n';
            if (!ln.empty()) { out.append((size_t)indent, ' '); out += ln; }
            if (b == std::string::npos) break;
            a = b + 1;
        }
        return;
    }
    if (yaml_plain_ok(s)) { out += s; return; }
    // libyaml's choice when a plain scalar is not allowed (yaml_emitter_select_scalar_style): single quotes ('' for an
    // apostrophe) unless the text holds a character outside its printable set - then double quotes with its escapes
    if (!has_yaml_special(s)) {
        out += '\'';
        for (char c : s) { if (c == '\'') out += '\''; out += c; }
        out += '\'';
        return;
    }
    out += '"';
    char buf[16];
    for (size_t i = 0; i < s.size();) {
        const size_t at = i;
        const uint32_t o = next_cp(s, i);
        switch (o) {
            case 0x00: out += "\\0"; continue;
            case 0x07: out += "\\a"; continue;
            case 0x08: out += "\\b"; continue;
            case 0x09: out += "\\t"; continue;
            case 0x0A: out += "\\n"; continue;
            case 0x0B: out += "\\v"; continue;
            case 0x0C: out += "\\f"; continue;
            case 0x0D: out += "\\r"; continue;
            case 0x1B: out += "\\e"; continue;
            case '"': out += "\\\""; continue;
            case '\\': out += "\\\\"; continue;
            case 0x85: out += "\\N"; continue;
            case 0x2028: out += "\\L"; continue;
            case 0x2029: out += "\\P"; continue;
            default: break;
        }
        if (!yaml_special(o)) { out.append(s, at, i - at); continue; }
        const uint32_t v = o == 0xFFFFFFFFu ? (unsigned char)s[at] : o;   // a malformed byte stands for itself
        if (v <= 0xFF) snprintf(buf, sizeof buf, "\\x%02X", v);
        else if (v <= 0xFFFF) snprintf(buf, sizeof buf, "\\u%04X", v);
        else snprintf(buf, sizeof buf, "\\U%08X", v);
        out += buf;
    }
    out += '"';
}

void json_string(const std::string &s, std::string &out) {  // serde_json: raw UTF-8, the short escapes, \u00XX for controls
    out += '"';
    char b[8];
    for (unsigned char c : s) {
        switch (c) {
            case '"': out += "\\\""; break;
            case '\\': out += "\\\\"; break;
            case '\n': out += "\\n"; break;
            case '\r': out += "\\r"; break;
            case '\t': out += "\\t"; break;
            case '\b': out += "\\b"; break;
            case '\f': out += "\\f"; break;
            default:
                if (c < 0x20) { snprintf(b, sizeof b, "\\u%04x", c); out += b; }
                else out += (char)c;
        }
    }
    out += '"';
}

void rust_debug_str(const std::string &s, std::string &out) {  // format!("{:?}", String)
    out += '"';
    char b[16];
    for (unsigned char c : s) {
        if (c == '"') out += "\\\"";
        else if (c == '\\') out += "\\\\";
        else if (c == '\n') out += "\\n";
        else if (c == '\r') out += "\\r";
        else if (c == '\t') out += "\\t";
        else if (c == 0) out += "\\0";
        else if (c < 0x20 || c == 0x7F) { snprintf(b, sizeof b, "\\u{%x}", c); out += b; }
        else out += (char)c;
    }
    out += '"';
}

const char *kind_name(uint8_t k) { return k == CLS_KIND_ROOT ? "ROOT" : k == CLS_KIND_LEAF ? "LEAF" : "NODE"; }

struct TreeView {
    const cls_record_tree *t;
    std::unordered_map<uint64_t, uint64_t> by_id;  // Clade.id -> first node (pre-order) carrying it: get_node_by_id (clade.rs:95-109)
    std::string name(uint64_t i) const { return std::string(t->names + t->name_off[i], t->names + t->name_off[i + 1]); }
};

// One Clade (clade.rs:18-38, serde camelCase, `None` name / support / length / children skipped, parent always present).
// YAML: keys at column `indent`; `first` is what precedes the first key on its line (the padding, or "- " inside a list).
void yaml_clade(const TreeView &tv, uint64_t i, int indent, const std::string &first, std::string &out) {
    const cls_record_tree *t = tv.t;
    const std::string pad((size_t)indent, ' ');
    out += first; out += "id: "; out += std::to_string(t->node_id[i]); out += '\n';
    out += pad; out += "parent: "; out += t->parent_id[i] < 0 ? std::string("null") : std::to_string(t->parent_id[i]); out += '\n';
    out += pad; out += "kind: "; out += kind_name(t->node_kind[i]); out += '\n';
    if (t->has_name[i]) { out += pad; out += "name: "; yaml_string(tv.name(i), indent + 2, out); out += '\n'; }
    if (!std::isnan(t->support[i])) { out += pad; out += "support: "; ryu_float(t->support[i], false, out); out += '\n'; }
    if (!std::isnan(t->length[i])) { out += pad; out += "length: "; ryu_float(t->length[i], false, out); out += '\n'; }
    if (t->children_some[i]) {
        const uint64_t a = t->child_off[i], b = t->child_off[i + 1];
        if (a == b) { out += pad; out += "children: []\n"; }
        else {
            out += pad; out += "children:\n";   // serde_yaml does not indent sequences inside maps
            for (uint64_t j = a; j < b; ++j) yaml_clade(tv, t->child_idx[j], indent + 2, pad + "- ", out);
        }
    }
}

void json_clade(const TreeView &tv, uint64_t i, std::string &out) {
    const cls_record_tree *t = tv.t;
    out += "{\"id\":"; out += std::to_string(t->node_id[i]);
    out += ",\"parent\":"; out += t->parent_id[i] < 0 ? std::string("null") : std::to_string(t->parent_id[i]);
    out += ",\"kind\":\""; out += kind_name(t->node_kind[i]); out += '"';
    if (t->has_name[i]) { out += ",\"name\":"; json_string(tv.name(i), out); }
    if (!std::isnan(t->support[i])) { out += ",\"support\":"; ryu_float(t->support[i], true, out); }
    if (!std::isnan(t->length[i])) { out += ",\"length\":"; ryu_float(t->length[i], true, out); }
    if (t->children_some[i]) {
        out += ",\"children\":[";
        for (uint64_t j = t->child_off[i]; j < t->child_off[i + 1]; ++j) {
            if (j > t->child_off[i]) out += ',';
            json_clade(tv, t->child_idx[j], out);
        }
        out += ']';
    }
    out += '}';
}

// Annotations of the clades on the path to the root (mod.rs:180-224): get_path_to_root (clade.rs:111-125) follows the
// Clade.parent FIELDS from the first pre-order node with that id; records keep their file order among equal clades.
void annotations_for(const TreeView &tv, uint64_t clade_id, std::vector<uint64_t> &picked) {
    picked.clear();
    const cls_record_tree *t = tv.t;
    if (!t->n_annotations) return;
    std::vector<uint64_t> path;
    auto it = tv.by_id.find(clade_id);
    uint64_t hops = 0;
    while (it != tv.by_id.end() && hops <= t->n_nodes) {
        path.push_back(it->first);
        const int64_t p = t->parent_id[it->second];
        if (p < 0) break;
        path.push_back((uint64_t)p);
        it = tv.by_id.find((uint64_t)p);
        ++hops;
    }
    for (uint64_t a = 0; a < t->n_annotations; ++a)
        for (uint64_t id : path)
            if (t->ann_clade[a] == id) { picked.push_back(a); break; }
    std::stable_sort(picked.begin(), picked.end(), [&](uint64_t x, uint64_t y) { return t->ann_clade[x] < t->ann_clade[y]; });
}

const char kErrTooShort[] = "The sequence does not contain enough kmers.";                        // place_sequence.rs:98-102
const char kErrMaxIter[] = "The maximum number of iterations has been reached.";                  // :295-301
const char kErrRootNoChildren[] = "The root node does not have children. This is unexpected.";    // :199-206
const char kErrInvalidBase[] = "Invalid character in sequence";                                   // kmers_map.rs:440 (a panic there)
const char kMsgNoRoot[] = "Query sequence has no overlapping kmers with the reference tree";       // :156-166
const char kMsgNoIntrospection[] =
    "Tree introspection not possible. Query sequence has no overlapping kmers with the reference tree";  // :446-454

// A header that is certainly a plain YAML scalar (and needs no JSON escape): it starts with an ASCII letter, holds only
// [A-Za-z0-9_] and is none of the words serde_yaml quotes - the common shape of a read name; everything else takes the
// general path (yaml_string / json_string), which gives the same text for these.
bool simple_header(const char *p, size_t n) {
    if (n == 0 || !((p[0] >= 'A' && p[0] <= 'Z') || (p[0] >= 'a' && p[0] <= 'z'))) return false;
    bool letters_only = true;
    for (size_t i = 0; i < n; ++i) {
        const unsigned char c = (unsigned char)p[i];
        const bool letter = (c >= 'A' && c <= 'Z') || (c >= 'a' && c <= 'z');
        if (!(letter || (c >= '0' && c <= '9') || c == '_')) return false;
        letters_only = letters_only && letter;
    }
    return !(letters_only && (n == 4 || n == 5));   // null / true / false in their three spellings have 4 or 5 letters
}

// What does not change from record to record, rendered once per call: the `code` line of every status whose text is
// fixed, and the Clade block of every node an IdentityFound record of the batch names (a batch places many reads on few
// clades; the blocks are rendered on the host pool before the records are).
struct Fixed {
    std::string code_yaml[16], code_json[16];   // by status: "\ncode: <scalar>\n" / ",\"code\":<string>"
    std::string incon_yaml, incon_json;         // the Inconclusive code again, as the placement
    std::vector<std::string> clade_text;        // by node index (pre-order); empty = not rendered
};

// The statuses whose `code` text is the same for every record.
bool fixed_code(uint8_t st, std::string *text = nullptr) {
    const char *head = nullptr, *tail = "";
    switch (st) {
        case CLS_STATUS_UNCL_NO_ROOT: head = "Unclassifiable: "; tail = kMsgNoRoot; break;
        case CLS_STATUS_UNCL_NO_INTROSPECTION: head = "Unclassifiable: "; tail = kMsgNoIntrospection; break;
        case CLS_STATUS_MAX_RESOLUTION: head = "MaxResolutionReached: LCA Accepted"; break;
        case CLS_STATUS_IDENTITY_FOUND: head = "IdentityFound"; break;
        case CLS_STATUS_INCONCLUSIVE: head = "Inconclusive: Multiple proposals"; break;
        default: return false;
    }
    if (text) { *text = head; *text += tail; }
    return true;
}

void make_fixed_codes(Fixed &fx) {
    std::string c;
    for (int st = 0; st < 16; ++st)
        if (fixed_code((uint8_t)st, &c)) {
            fx.code_yaml[st] = "\ncode: "; yaml_string(c, 2, fx.code_yaml[st]); fx.code_yaml[st] += '\n';
            fx.code_json[st] = ",\"code\":"; json_string(c, fx.code_json[st]);
        }
    fixed_code(CLS_STATUS_INCONCLUSIVE, &c);
    yaml_string(c, 2, fx.incon_yaml);
    json_string(c, fx.incon_json);
}

void append_u64(std::string &out, uint64_t v) {
    char b[24];
    auto r = std::to_chars(b, b + sizeof b, v);
    out.append(b, (size_t)(r.ptr - b));
}
void append_i64(std::string &out, int64_t v) {
    char b[24];
    auto r = std::to_chars(b, b + sizeof b, v);
    out.append(b, (size_t)(r.ptr - b));
}

// One query: appends its record to `out` or its error text to `err`.  Returns false on an unknown status / node id.
bool render_one(const TreeView &tv, const Fixed &fx, const char *hp, size_t hn, const cls_result *r, uint64_t i, bool yaml,
                std::string &out, std::string &err, std::vector<uint64_t> &scratch, std::string &header, std::string &code) {
    const uint8_t st = r->status[i];
    switch (st) {
        case CLS_STATUS_ERR_TOO_SHORT: err += kErrTooShort; return true;
        case CLS_STATUS_ERR_MAX_ITERATIONS: err += kErrMaxIter; return true;
        case CLS_STATUS_ERR_ROOT_NO_CHILDREN: err += kErrRootNoChildren; return true;
        case CLS_STATUS_ERR_INVALID_BASE: err += kErrInvalidBase; return true;
        case CLS_STATUS_UNCL_NO_MATCH: case CLS_STATUS_UNCL_COVERAGE: case CLS_STATUS_UNCL_NO_ROOT:
        case CLS_STATUS_UNCL_NO_INTROSPECTION: case CLS_STATUS_MAX_RESOLUTION: case CLS_STATUS_IDENTITY_FOUND:
        case CLS_STATUS_INCONCLUSIVE: break;
        default: return false;
    }
    const bool simple = simple_header(hp, hn);
    if (!simple || st == CLS_STATUS_UNCL_NO_MATCH) header.assign(hp, hn);
    const bool fixed = fixed_code(st);
    if (st == CLS_STATUS_UNCL_NO_MATCH) {
        code = "Unclassifiable: Query sequence SequenceHeader("; rust_debug_str(header, code); code += ") may not be related to the phylogeny";
    } else if (st == CLS_STATUS_UNCL_COVERAGE) {
        code = "Unclassifiable: Insufficient kmers coverage: "; append_u64(code, r->n_root_matched ? r->n_root_matched[i] : 0u);
    }
    const bool identity = st == CLS_STATUS_IDENTITY_FOUND, max_res = st == CLS_STATUS_MAX_RESOLUTION;
    uint64_t node = 0;
    if (identity) {
        auto it = tv.by_id.find(r->node_id[i]);
        if (it == tv.by_id.end()) return false;
        node = it->second;
    }
    if (tv.t->has_annotations && (identity || max_res)) annotations_for(tv, r->node_id[i], scratch); else scratch.clear();
    const cls_record_tree *t = tv.t;
    if (yaml) {
        out += "---\nquery: ";
        if (simple) out.append(hp, hn); else yaml_string(header, 2, out);
        if (fixed) out += fx.code_yaml[st];
        else { out += "\ncode: "; yaml_string(code, 2, out); out += '\n'; }
        if (!scratch.empty()) {
            out += "annotations:\n";
            for (uint64_t a : scratch) out.append(t->ann_yaml + t->ann_yaml_off[a], t->ann_yaml + t->ann_yaml_off[a + 1]);
        }
        if (identity) {
            out += "placement:\n  clade:\n";
            out += fx.clade_text[node];
            out += "  one: "; append_i64(out, r->one[i]); out += "\n  rest: "; append_i64(out, r->rest[i]); out += '\n';
        } else if (max_res) {
            out += "placement: "; append_u64(out, r->node_id[i]); out += '\n';
        } else if (st == CLS_STATUS_INCONCLUSIVE) {
            out += "placement: "; out += fx.incon_yaml; out += '\n';
        }
    } else {
        out += "{\"query\":";
        if (simple) { out += '"'; out.append(hp, hn); out += '"'; } else json_string(header, out);
        if (fixed) out += fx.code_json[st];
        else { out += ",\"code\":"; json_string(code, out); }
        if (!scratch.empty()) {
            out += ",\"annotations\":[";
            for (size_t k = 0; k < scratch.size(); ++k) {
                if (k) out += ',';
                out.append(t->ann_json + t->ann_json_off[scratch[k]], t->ann_json + t->ann_json_off[scratch[k] + 1]);
            }
            out += ']';
        }
        if (identity) {
            out += ",\"placement\":{\"clade\":";
            out += fx.clade_text[node];
            out += ",\"one\":"; append_i64(out, r->one[i]); out += ",\"rest\":"; append_i64(out, r->rest[i]); out += '}';
        } else if (max_res) {
            out += ",\"placement\":"; append_u64(out, r->node_id[i]);
        } else if (st == CLS_STATUS_INCONCLUSIVE) {
            out += ",\"placement\":"; out += fx.incon_json;
        }
        out += "}\n";
    }
    return true;
}

// The blocks back to back in one malloc'ed text; copied on the host pool (a fresh gigabyte of pages is faulted in by
// whoever writes it first: one thread would spend longer here than the pool spends rendering).
char *to_malloc(const std::vector<std::string> &parts, uint64_t *len) {
    std::vector<size_t> at(parts.size() + 1, 0);
    for (size_t i = 0; i < parts.size(); ++i) at[i + 1] = at[i] + parts[i].size();
    const size_t n = at.back();
    char *buf = static_cast<char *>(malloc(n + 1));
    if (!buf) return nullptr;
    cls::parallel_for(parts.size(), 1, [&](uint64_t p0, uint64_t p1) {
        for (uint64_t i = p0; i < p1; ++i) memcpy(buf + at[i], parts[i].data(), parts[i].size());
    });
    buf[n] = 0;
    *len = n;
    return buf;
}

// Renders blocks of 2 048 records on the host pool: outs[b] / errs[b] hold the record text / error text of block b.
int render_blocks(const cls_record_tree *tree, uint64_t n, const uint64_t *header_off, const char *headers, const cls_result *res,
                  uint32_t format, std::vector<std::string> &outs, std::vector<std::string> &errs) {
    using cls::set_last_error;
    if (!tree || !res || (n && (!header_off || !headers))) return set_last_error(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (format > 1) return set_last_error(CLS_ERR_INVALID_ARGUMENT, "format must be 0 (yaml) or 1 (jsonl)");
    if (n && (!res->status || !res->node_id || !res->one || !res->rest)) return set_last_error(CLS_ERR_INVALID_ARGUMENT, "result arrays are NULL");
    // the child lists must form a forest (as cls_index_create demands of the same tree): the Clade writers recurse over them
    {
        std::vector<uint8_t> seen(tree->n_nodes, 0);
        std::vector<uint32_t> depth(tree->n_nodes, 0);
        for (uint64_t i = 0; i < tree->n_nodes; ++i) {
            if (tree->child_off[i] > tree->child_off[i + 1]) return set_last_error(CLS_ERR_INVALID_ARGUMENT, "child_off is not non-decreasing");
            for (uint64_t j = tree->child_off[i]; j < tree->child_off[i + 1]; ++j) {
                const uint64_t c = tree->child_idx[j];
                if (c >= tree->n_nodes || c == 0 || seen[c]) return set_last_error(CLS_ERR_INVALID_ARGUMENT, "child lists do not form a tree");
                seen[c] = 1;
                if (c <= i) return set_last_error(CLS_ERR_INVALID_ARGUMENT, "nodes must come in pre-order (children after their parent)");
                depth[c] = depth[i] + 1;
                if (depth[c] > 20000) return set_last_error(CLS_ERR_UNSUPPORTED, "tree deeper than 20 000 levels");
            }
        }
    }
    TreeView tv{tree, {}};
    tv.by_id.reserve(tree->n_nodes * 2);
    for (uint64_t i = 0; i < tree->n_nodes; ++i) tv.by_id.emplace(tree->node_id[i], i);   // emplace keeps the first
    const bool yaml = format == 0;
    constexpr uint64_t kBlock = 2048;
    const uint64_t nblk = (n + kBlock - 1) / kBlock;
    outs.assign(nblk, std::string());
    errs.assign(nblk, std::string());
    std::vector<uint8_t> bad(nblk, 0);
    Fixed fx;
    make_fixed_codes(fx);
    fx.clade_text.assign(tree->n_nodes, std::string());
    // pass 1: the node behind every IdentityFound record (an id that is not in the tree is reported by pass 3), the
    // distinct ones collected per task
    std::vector<uint64_t> wanted;
    {
        std::vector<uint8_t> mark(tree->n_nodes, 0);   // written with 1 only, by any task: relaxed atomics
        cls::parallel_for(n, 16384, [&](uint64_t a, uint64_t b) {
            for (uint64_t i = a; i < b; ++i) {
                if (res->status[i] != CLS_STATUS_IDENTITY_FOUND) continue;
                auto it = tv.by_id.find(res->node_id[i]);
                if (it != tv.by_id.end()) __atomic_store_n(&mark[it->second], (uint8_t)1, __ATOMIC_RELAXED);
            }
        });
        for (uint64_t i = 0; i < tree->n_nodes; ++i)
            if (mark[i]) wanted.push_back(i);
    }
    // pass 2: their Clade blocks, each rendered once (pre-order: the big subtrees come first)
    std::vector<uint8_t> bad2(wanted.size(), 0);
    cls::parallel_for(wanted.size(), 1, [&](uint64_t a, uint64_t b) {
        for (uint64_t w = a; w < b; ++w) {
            try {   // nothing may escape a pool thread
                if (yaml) yaml_clade(tv, wanted[w], 4, "    ", fx.clade_text[wanted[w]]);
                else json_clade(tv, wanted[w], fx.clade_text[wanted[w]]);
            } catch (...) {
                bad2[w] = 1;
            }
        }
    });
    for (uint8_t x : bad2)
        if (x) return set_last_error(CLS_ERR_OUT_OF_MEMORY, "host allocation failed while rendering records");
    // pass 3: the records
    cls::parallel_for(nblk, 1, [&](uint64_t b0, uint64_t b1) {
        std::vector<uint64_t> scratch;
        std::string header, code;
        for (uint64_t b = b0; b < b1; ++b) {
            std::string &o = outs[b], &e = errs[b];
            const uint64_t lo = b * kBlock, hi = std::min(n, (b + 1) * kBlock);
            try {   // nothing may escape a pool thread
                // the block's text in one allocation: Clade blocks + headers + about a hundred bytes of keys per record
                // (annotations, quoted headers and NoMatch codes, which repeat the header, may still grow it)
                size_t est = (hi - lo) * 160 + 2 * (size_t)(header_off[hi] - header_off[lo]);
                for (uint64_t i = lo; i < hi; ++i)
                    if (res->status[i] == CLS_STATUS_IDENTITY_FOUND) {
                        auto it = tv.by_id.find(res->node_id[i]);
                        if (it != tv.by_id.end()) est += fx.clade_text[it->second].size();
                    }
                o.reserve(est);
                for (uint64_t i = lo; i < hi; ++i)
                    if (!render_one(tv, fx, headers + header_off[i], (size_t)(header_off[i + 1] - header_off[i]), res, i, yaml, o, e,
                                    scratch, header, code))
                        bad[b] = 1;
            } catch (...) {
                bad[b] = 2;
            }
        }
    });
    for (uint8_t x : bad) {
        if (x == 2) return set_last_error(CLS_ERR_OUT_OF_MEMORY, "host allocation failed while rendering records");
        if (x) return set_last_error(CLS_ERR_INVALID_ARGUMENT, "unknown status, or a placement node id that is not in the tree");
    }
    return CLS_OK;
}

int render(const cls_record_tree *tree, uint64_t n, const uint64_t *header_off, const char *headers, const cls_result *res,
           uint32_t format, char **out_text, uint64_t *out_len, char **err_text, uint64_t *err_len) {
    using cls::set_last_error;
    if (!out_text || !out_len || !err_text || !err_len) return set_last_error(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    *out_text = *err_text = nullptr;
    *out_len = *err_len = 0;
    std::vector<std::string> outs, errs;
    const int rc = render_blocks(tree, n, header_off, headers, res, format, outs, errs);
    if (rc != CLS_OK) return rc;
    *out_text = to_malloc(outs, out_len);
    *err_text = to_malloc(errs, err_len);
    if (!*out_text || !*err_text) {
        free(*out_text); free(*err_text);
        *out_text = *err_text = nullptr;
        return set_last_error(CLS_ERR_OUT_OF_MEMORY, "host allocation of the rendered records failed");
    }
    return CLS_OK;
}

}  // namespace

extern "C" int cls_records_render(const cls_record_tree *tree, uint64_t n_queries, const uint64_t *header_off, const char *headers,
                                  const cls_result *result, uint32_t format, char **out_text, uint64_t *out_len, char **err_text,
                                  uint64_t *err_len) {
    try {
        return render(tree, n_queries, header_off, headers, result, format, out_text, out_len, err_text, err_len);
    } catch (const std::bad_alloc &) {
        return cls::set_last_error(CLS_ERR_OUT_OF_MEMORY, "host allocation failed while rendering records");
    } catch (const std::exception &e) {
        return cls::set_last_error(CLS_ERR_INVALID_ARGUMENT, std::string("cls_records_render: ") + e.what());
    }
}

extern "C" void cls_text_free(char *p) { free(p); }

extern "C" {
// sequence.rs:47-56: `sequence.to_uppercase().chars().filter(A|C|G|T)`.  Rust upper-cases with the
// full Unicode mapping; the only non-ASCII scalars whose upper-case expansion contains an ASCII
// A/C/G/T are U+1E97 (t with diaeresis -> "T" + U+0308), U+1E9A (a with right half ring -> "A" +
// U+02BE), U+FB05 and U+FB06 (long-s-t / st ligatures -> "ST").  Every other non-ASCII byte
// sequence contributes nothing.
uint64_t cls_filter_sequence(const uint8_t *line, uint64_t len, uint8_t *out, uint64_t cap) {
    uint64_t n = 0;
    auto put = [&](uint8_t c) { if (n < cap && out) out[n] = c; ++n; };
    // upper-cased base for A/C/G/T/a/c/g/t, 0 for every other byte
    static const struct Lut { uint8_t v[256]; Lut() : v{} { for (const char *p = "ACGTacgt"; *p; ++p) v[(uint8_t)*p] = (uint8_t)(*p & 0xDF); } } lut;
    for (uint64_t i = 0; i < len; ++i) {
        // fast path: a stretch of ASCII with room in `out` - one table look-up and a branch-free store per byte
        if (out) {
            while (i < len && line[i] < 0x80 && n < cap) {
                const uint8_t u = lut.v[line[i]];
                out[n] = u;
                n += u != 0;
                ++i;
            }
            if (i >= len) break;
        }
        const uint8_t c = line[i];
        if (c < 0x80) {
            const uint8_t u = (c >= 'a' && c <= 'z') ? (uint8_t)(c - 32) : c;
            if (u == 'A' || u == 'C' || u == 'G' || u == 'T') put(u);
        } else if (c == 0xE1 && i + 2 < len && line[i + 1] == 0xBA && (line[i + 2] == 0x97 || line[i + 2] == 0x9A)) {
            put(line[i + 2] == 0x97 ? 'T' : 'A');
            i += 2;
        } else if (c == 0xEF && i + 2 < len && line[i + 1] == 0xAC && (line[i + 2] == 0x85 || line[i + 2] == 0x86)) {
            put('T');
            i += 2;
        }
    }
    return n;
}
}  // extern "C"

// ---- the reference's FASTA reader on the host (file_or_stdin.rs:76-116 + sequence.rs:47-56), for texts the device ingest
//      does not take (non-ASCII bytes, streams) and for callers without a resident batch.  Same record rules as
//      cls_fasta_upload applies on the device; one pass over the text. ---------------------------------------------
struct cls_fasta_text {
    std::vector<uint64_t> header_begin, header_end, offsets;
    std::unique_ptr<uint8_t[]> bases;   // as long as the text; [0, offsets.back()) is written
};

// str::from_utf8 on one line (BufRead::lines yields Err for a line that is not valid UTF-8: the reader then returns, and
// the caller places what was sent so far, file_or_stdin.rs:85)
static bool valid_utf8(const uint8_t *p, uint64_t n) {
    uint64_t i = 0;
    while (i < n) {
        const uint8_t c = p[i];
        if (c < 0x80) { ++i; continue; }
        uint32_t need, lo = 0x80, hi = 0xBF;
        if (c >= 0xC2 && c <= 0xDF) need = 1;
        else if (c == 0xE0) { need = 2; lo = 0xA0; }
        else if ((c >= 0xE1 && c <= 0xEC) || c == 0xEE || c == 0xEF) need = 2;
        else if (c == 0xED) { need = 2; hi = 0x9F; }
        else if (c == 0xF0) { need = 3; lo = 0x90; }
        else if (c >= 0xF1 && c <= 0xF3) need = 3;
        else if (c == 0xF4) { need = 3; hi = 0x8F; }
        else return false;
        if (i + need >= n) return false;   // truncated sequence
        if (p[i + 1] < lo || p[i + 1] > hi) return false;
        for (uint32_t j = 2; j <= need; ++j)
            if ((p[i + j] & 0xC0) != 0x80) return false;
        i += need + 1;
    }
    return true;
}

// cls_fasta_read works on CHUNKS of whole lines, a wave of them at a time on the host pool: a chunk is scanned without
// knowing the reader's state at its first line - its filtered bases go to a buffer of its own, and every line that the
// state machine has to see (a header line, a line that is not valid UTF-8) becomes an event carrying the number of bases
// the chunk had kept before it.  The reader of file_or_stdin.rs:76-116 then runs over the events alone, in file order
// (a few bytes per record), and the chunks' bases are copied to where that pass says they start.
namespace {

struct FaEvent {
    uint64_t begin, end;   // the line, [begin, end)
    uint64_t kept;         // bases the chunk had kept before this line
    uint8_t kind;          // 0: header line with text, 1: header line of '>' only, 2: a line that is not valid UTF-8
};
struct FaChunk {
    uint64_t a = 0, b = 0;           // whole lines [a, b) of the text
    uint64_t kept = 0;               // filtered bases of the chunk
    std::vector<FaEvent> events;
    std::vector<uint8_t> bases;      // sized to the chunk (reused by the following waves)
};

void fasta_scan_chunk(const uint8_t *text, FaChunk &c) {
    c.events.clear();
    c.kept = 0;
    if (c.bases.size() < c.b - c.a) c.bases.resize(c.b - c.a);
    uint64_t a = c.a;
    while (a < c.b) {
        const uint8_t *nl = static_cast<const uint8_t *>(memchr(text + a, '\n', c.b - a));
        uint64_t b = nl ? (uint64_t)(nl - text) : c.b;              // line = [a, b)
        const uint64_t next = nl ? b + 1 : c.b;
        if (nl && b > a && text[b - 1] == '\r') --b;                // BufRead::lines: "\r\n" is a terminator, a lone "\r" is not
        if (b > a) {                                                // empty lines are skipped (:87-89)
            bool ascii = true;
            for (uint64_t i = a; i < b && ascii; ++i) ascii = text[i] < 0x80;
            if (!ascii && !valid_utf8(text + a, b - a)) {           // `line?`: the reader returns here
                c.events.push_back(FaEvent{a, b, c.kept, 2});
                return;                                             // nothing after it is ever looked at
            }
            if (text[a] == '>') {
                bool nonempty = false;                              // header = the line minus every '>' (:102)
                for (uint64_t i = a; i < b && !nonempty; ++i) nonempty = text[i] != '>';
                c.events.push_back(FaEvent{a, b, c.kept, (uint8_t)(nonempty ? 0 : 1)});
            } else {
                c.kept += cls_filter_sequence(text + a, b - a, c.bases.data() + c.kept, c.bases.size() - c.kept);
            }
        }
        a = next;
    }
}

}  // namespace

extern "C" int cls_fasta_read(const uint8_t *text, uint64_t n_bytes, cls_fasta_text **out, cls_fasta_host_records *rec) {
    using cls::set_last_error;
    if (!out || !rec || (n_bytes && !text)) return set_last_error(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    *out = nullptr;
    memset(rec, 0, sizeof *rec);
    try {
        auto ft = std::make_unique<cls_fasta_text>();
        ft->offsets.push_back(0);
        ft->bases.reset(new uint8_t[n_bytes ? n_bytes : 1]);   // not zero-filled: only [0, offsets.back()) is ever read
        // chunk size: 2 MiB of text (CLS_FASTA_CHUNK bytes: tests run the stitching over chunks of a few lines)
        uint64_t chunk_bytes = 2u << 20;
        if (const char *e = getenv("CLS_FASTA_CHUNK")) { const long long v = atoll(e); if (v > 0) chunk_bytes = (uint64_t)v; }
        const size_t wave = (size_t)std::max(1, cls::host_threads()) * 2;
        std::vector<FaChunk> chunks(wave);
        std::vector<uint64_t> dst(wave);
        uint64_t kept = 0;              // filtered bases sent or pending so far
        uint64_t rec_start = 0;         // first base of the record being read
        bool have_header = false;       // the reader holds a non-empty header
        uint64_t hb = 0, he = 0;        // its line
        bool stop = false;
        uint64_t at = 0;                // first byte of the next chunk (a line start)
        while (at < n_bytes && !stop) {
            size_t nc = 0;
            for (; nc < wave && at < n_bytes; ++nc) {               // cut the wave's chunks at line ends
                uint64_t end = n_bytes;
                if (n_bytes - at > chunk_bytes) {
                    const uint8_t *nl = static_cast<const uint8_t *>(memchr(text + at + chunk_bytes - 1, '\n', n_bytes - (at + chunk_bytes - 1)));
                    if (nl) end = (uint64_t)(nl - text) + 1;
                }
                chunks[nc].a = at; chunks[nc].b = end;
                at = end;
            }
            cls::parallel_for(nc, 1, [&](uint64_t c0, uint64_t c1) {
                for (uint64_t c = c0; c < c1; ++c) fasta_scan_chunk(text, chunks[c]);
            });
            size_t copy_n = 0;                                      // chunks whose bases are kept
            for (size_t c = 0; c < nc && !stop; ++c) {
                const uint64_t base = kept;                         // where the chunk's bases start
                for (const FaEvent &e : chunks[c].events) {
                    kept = base + e.kept;
                    if (e.kind == 2) { stop = true; break; }        // the pending record is not sent
                    if (have_header) {                              // send the previous record, even without sequence (:103-108)
                        ft->header_begin.push_back(hb); ft->header_end.push_back(he);
                        ft->offsets.push_back(kept);
                        rec_start = kept;
                    } else if (kept > rec_start) {                  // sequence without header: the reader errors out (:96-100)
                        stop = true;
                        break;
                    }
                    have_header = e.kind == 0;
                    hb = e.begin; he = e.end;
                }
                dst[c] = base;
                copy_n = c + 1;
                if (!stop) kept = base + chunks[c].kept;
            }
            cls::parallel_for(copy_n, 1, [&](uint64_t c0, uint64_t c1) {
                for (uint64_t c = c0; c < c1; ++c)
                    if (chunks[c].kept) memcpy(ft->bases.get() + dst[c], chunks[c].bases.data(), chunks[c].kept);
            });
        }
        if (stop) kept = rec_start;
        if (!stop && have_header && kept > rec_start) {             // the trailing record needs a sequence (:111-113)
            ft->header_begin.push_back(hb); ft->header_end.push_back(he);
            ft->offsets.push_back(kept);
        }
        rec->n_records = ft->header_begin.size();
        rec->header_begin = ft->header_begin.data();
        rec->header_end = ft->header_end.data();
        rec->offsets = ft->offsets.data();
        rec->bases = ft->bases.get();
        *out = ft.release();
        return CLS_OK;
    } catch (const std::bad_alloc &) {
        return set_last_error(CLS_ERR_OUT_OF_MEMORY, "host allocation failed while reading the FASTA text");
    }
}

extern "C" void cls_fasta_text_destroy(cls_fasta_text *t) { delete t; }

// ---- FASTQ queries (the rules are in include/classeq_b200.h, next to CLS_QUERY_FASTQ).  The reference has no FASTQ
//      reader; these rules make a FASTQ file and its FASTA rendering place identically.  cls_fastq_upload applies the same
//      rules on the device and reports its first bad record through the helpers below. -------------------------------------
namespace cls {

const char *fastq_reason(int code) {
    switch (code) {
    case kFastqBlankLine: return "blank line inside the records";
    case kFastqNoAt: return "title line does not start with '@'";
    case kFastqTruncated: return "truncated record (fewer than four lines)";
    case kFastqNoPlus: return "separator line does not start with '+'";
    case kFastqQualityLength: return "quality length differs from sequence length";
    case kFastqTitleUtf8: return "title is not valid UTF-8";
    default: return "malformed record";
    }
}

int fastq_fail(uint64_t record, int code) {   // record: 0-based
    return set_last_error(CLS_ERR_INVALID_ARGUMENT, "malformed FASTQ record " + std::to_string(record + 1) + ": " + fastq_reason(code));
}

// Records of the text: the records end at the last non-blank line (blank lines may only follow the last record).  A line
// is blank when nothing but its terminator ("\n" or "\r\n") is in it.
uint64_t fastq_n_records(const uint8_t *text, uint64_t n, uint64_t n_newlines) {
    uint64_t e = n, blank = 0;
    while (e > 0 && text[e - 1] == '\n') {
        uint64_t s = e - 1;
        if (s > 0 && text[s - 1] == '\r') --s;
        if (s > 0 && text[s - 1] != '\n') break;   // the terminator of a line with content
        e = s;
        ++blank;
    }
    const uint64_t lines = n_newlines - blank + (e > 0 && text[e - 1] != '\n' ? 1 : 0);   // lines up to the last non-blank one
    return lines ? (lines - 1) / 4 + 1 : 0;
}

// First record r < n_records whose title text[hb[r] .. he[r]) is not valid UTF-8, or n_records.
uint64_t fastq_first_bad_title(const uint8_t *text, const uint64_t *hb, const uint64_t *he, uint64_t n_records) {
    std::atomic<uint64_t> first{n_records};
    parallel_for(n_records, 1 << 14, [&](uint64_t a, uint64_t b) {
        for (uint64_t r = a; r < b && r < first.load(std::memory_order_relaxed); ++r) {
            bool ascii = true;
            for (uint64_t i = hb[r]; i < he[r] && ascii; ++i) ascii = text[i] < 0x80;
            if (!ascii && !valid_utf8(text + hb[r], he[r] - hb[r])) {
                uint64_t cur = first.load();
                while (r < cur && !first.compare_exchange_weak(cur, r)) {}
                break;
            }
        }
    });
    return first.load();
}

}  // namespace cls

// cls_fastq_read: chunks of ~2 MiB cut at line ends; their newlines are counted side by side, which gives the line number
// at every chunk start; each chunk is then moved forward to its first record start (a line number that is a multiple of
// 4), so that every chunk holds whole records and is read without knowing anything about the others.  A wave of chunks
// at a time is read on the host pool into buffers of their own, and appended in file order.
namespace {

struct FqLine {
    uint64_t begin, end, next;   // content [begin, end) ("\n" / "\r\n" excluded); next: the first byte after the terminator
};
FqLine fq_line(const uint8_t *text, uint64_t n, uint64_t a) {
    const uint8_t *nl = static_cast<const uint8_t *>(memchr(text + a, '\n', n - a));
    if (!nl) return FqLine{a, n, n};
    uint64_t e = (uint64_t)(nl - text);
    const uint64_t next = e + 1;
    if (e > a && text[e - 1] == '\r') --e;
    return FqLine{a, e, next};
}

struct FqChunk {
    uint64_t a = 0, b = 0;         // whole records [a, b) of the text
    uint64_t first = 0;            // number of its first record
    uint64_t lines = 0;            // (line counting) newlines in the raw chunk
    std::vector<uint64_t> hb, he, len;
    std::vector<uint8_t> bases;
    uint64_t kept = 0;
    uint64_t bad = ~0ull;          // first bad record, 0-based (~0: none)
    int code = 0;
};

void fastq_read_chunk(const uint8_t *text, uint64_t n, uint64_t n_records, FqChunk &c) {
    c.hb.clear(); c.he.clear(); c.len.clear();
    c.kept = 0;
    c.bad = ~0ull;
    if (c.bases.size() < c.b - c.a) c.bases.resize(c.b - c.a);
    uint64_t at = c.a;
    for (uint64_t r = c.first; at < c.b && r < n_records; ++r) {
        auto fail = [&](int code) { c.bad = r; c.code = code; };
        const FqLine t = fq_line(text, n, at);
        if (t.end == t.begin) { fail(cls::kFastqBlankLine); return; }
        if (text[t.begin] != '@') { fail(cls::kFastqNoAt); return; }
        if (t.next >= n) { fail(cls::kFastqTruncated); return; }
        const FqLine s = fq_line(text, n, t.next);
        if (s.next >= n) { fail(cls::kFastqTruncated); return; }
        const FqLine p = fq_line(text, n, s.next);
        if (p.next >= n) { fail(cls::kFastqTruncated); return; }
        const FqLine q = fq_line(text, n, p.next);
        if (p.end == p.begin || text[p.begin] != '+') { fail(cls::kFastqNoPlus); return; }
        if (q.end - q.begin != s.end - s.begin) { fail(cls::kFastqQualityLength); return; }
        bool ascii = true;
        for (uint64_t i = t.begin + 1; i < t.end && ascii; ++i) ascii = text[i] < 0x80;
        if (!ascii && !valid_utf8(text + t.begin + 1, t.end - t.begin - 1)) { fail(cls::kFastqTitleUtf8); return; }
        c.hb.push_back(t.begin + 1);
        c.he.push_back(t.end);
        uint64_t k = 0;
        uint8_t *out = c.bases.data() + c.kept;
        for (uint64_t i = s.begin; i < s.end; ++i) {   // a byte rule: bytes >= 0x80 are deleted like every non-A/C/G/T byte
            const uint8_t u = text[i] & 0xDFu;
            if (text[i] >= 'A' && text[i] < 0x80 && (u == 'A' || u == 'C' || u == 'G' || u == 'T')) out[k++] = u;
        }
        c.len.push_back(k);
        c.kept += k;
        at = q.next;
    }
}

}  // namespace

extern "C" int cls_fastq_read(const uint8_t *text, uint64_t n_bytes, cls_fasta_text **out, cls_fasta_host_records *rec) {
    using cls::set_last_error;
    if (!out || !rec || (n_bytes && !text)) return set_last_error(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    *out = nullptr;
    memset(rec, 0, sizeof *rec);
    try {
        auto ft = std::make_unique<cls_fasta_text>();
        ft->offsets.push_back(0);
        ft->bases.reset(new uint8_t[n_bytes ? n_bytes : 1]);
        // chunk size: 2 MiB of text (CLS_FASTA_CHUNK bytes: tests put every rule on a chunk boundary)
        uint64_t chunk_bytes = 2u << 20;
        if (const char *e = getenv("CLS_FASTA_CHUNK")) { const long long v = atoll(e); if (v > 0) chunk_bytes = (uint64_t)v; }
        std::vector<FqChunk> raw;                                    // cut at line ends
        for (uint64_t at = 0; at < n_bytes;) {
            uint64_t end = n_bytes;
            if (n_bytes - at > chunk_bytes) {
                const uint8_t *nl = static_cast<const uint8_t *>(memchr(text + at + chunk_bytes - 1, '\n', n_bytes - (at + chunk_bytes - 1)));
                if (nl) end = (uint64_t)(nl - text) + 1;
            }
            raw.emplace_back();
            raw.back().a = at; raw.back().b = end;
            at = end;
        }
        cls::parallel_for(raw.size(), 1, [&](uint64_t c0, uint64_t c1) {
            for (uint64_t c = c0; c < c1; ++c) raw[c].lines = (uint64_t)std::count(text + raw[c].a, text + raw[c].b, '\n');
        });
        uint64_t n_newlines = 0;
        for (FqChunk &c : raw) {                                     // move every chunk start to its first record start
            const uint64_t skip = (4 - (n_newlines & 3)) & 3;
            c.first = (n_newlines + 3) / 4;
            uint64_t a = c.a;
            for (uint64_t j = 0; j < skip && a < n_bytes; ++j) a = fq_line(text, n_bytes, a).next;
            c.a = a;
            n_newlines += c.lines;
        }
        for (size_t c = 0; c < raw.size(); ++c) {
            raw[c].b = c + 1 < raw.size() ? raw[c + 1].a : n_bytes;
            if (raw[c].b < raw[c].a) raw[c].b = raw[c].a;            // a chunk of fewer than four lines holds no record start
        }
        const uint64_t n_records = cls::fastq_n_records(text, n_bytes, n_newlines);
        const size_t wave = (size_t)std::max(1, cls::host_threads()) * 2;
        std::vector<FqChunk> chunks(wave);
        uint64_t kept = 0;
        for (size_t w0 = 0; w0 < raw.size(); w0 += wave) {
            const size_t nc = std::min(wave, raw.size() - w0);
            for (size_t c = 0; c < nc; ++c) { chunks[c].a = raw[w0 + c].a; chunks[c].b = raw[w0 + c].b; chunks[c].first = raw[w0 + c].first; }
            cls::parallel_for(nc, 1, [&](uint64_t c0, uint64_t c1) {
                for (uint64_t c = c0; c < c1; ++c) fastq_read_chunk(text, n_bytes, n_records, chunks[c]);
            });
            std::vector<uint64_t> dst(nc);
            for (size_t c = 0; c < nc; ++c) {
                const FqChunk &ch = chunks[c];
                if (ch.bad != ~0ull) return cls::fastq_fail(ch.bad, ch.code);   // the first bad record of the file: chunks go in order
                dst[c] = kept;
                ft->header_begin.insert(ft->header_begin.end(), ch.hb.begin(), ch.hb.end());
                ft->header_end.insert(ft->header_end.end(), ch.he.begin(), ch.he.end());
                for (uint64_t l : ch.len) ft->offsets.push_back(kept += l);
            }
            cls::parallel_for(nc, 1, [&](uint64_t c0, uint64_t c1) {
                for (uint64_t c = c0; c < c1; ++c)
                    if (chunks[c].kept) memcpy(ft->bases.get() + dst[c], chunks[c].bases.data(), chunks[c].kept);
            });
        }
        rec->n_records = ft->header_begin.size();
        rec->header_begin = ft->header_begin.data();
        rec->header_end = ft->header_end.data();
        rec->offsets = ft->offsets.data();
        rec->bases = ft->bases.get();
        *out = ft.release();
        return CLS_OK;
    } catch (const std::bad_alloc &) {
        return set_last_error(CLS_ERR_OUT_OF_MEMORY, "host allocation failed while reading the FASTQ text");
    }
}


// ---- place_sequences as the reference spells it (core/src/use_cases/place_sequences/mod.rs:43-270): a query FASTA, an
//      output path, the knobs -> result / error files.  cls_sequences_open does the path handling of :73-106 and reads the
//      records (:118-119), cls_sequences_write appends what the closure at :160-249 appends for a batch of results, and
//      cls_place_sequences strings them together around cls_place_batch. -------------------------------------------------
// Bytes of a file in a malloc'ed buffer (not zero-filled first, unlike a std::string that is resized).
struct RawText {
    char *p = nullptr;
    size_t n = 0;
    RawText() = default;
    RawText(const RawText &) = delete;
    RawText &operator=(const RawText &) = delete;
    ~RawText() { free(p); }
    void clear() { n = 0; }
};

struct cls_sequences {
    RawText text;                     // the query file
    cls_fasta_text *records = nullptr;
    cls_fasta_host_records rec{};
    std::vector<uint64_t> header_off; // headers with every '>' removed, back to back
    std::string headers;
    std::string out_path, err_path;
    uint32_t format = 0;
    uint64_t written = 0;             // records handed to cls_sequences_write so far
    ~cls_sequences() { cls_fasta_text_destroy(records); }
};

namespace {

// PathBuf::set_extension(ext): the extension of the FILE NAME is replaced (or appended when there is none; a leading
// dot of the name does not start an extension)
std::string with_extension(const std::string &path, const char *ext) {
    const size_t slash = path.find_last_of('/');
    const size_t name = slash == std::string::npos ? 0 : slash + 1;
    const size_t dot = path.find_last_of('.');
    std::string root = (dot == std::string::npos || dot <= name) ? path : path.substr(0, dot);
    return root + "." + ext;
}

// The whole of `f` (a regular file is read in one piece into a buffer of its size; a pipe grows the buffer as it comes).
bool read_whole(FILE *f, RawText &out) {
    out.n = 0;
    size_t cap = (size_t)1 << 20;
    struct stat st;
    if (fstat(fileno(f), &st) == 0 && S_ISREG(st.st_mode) && st.st_size > 0) cap = (size_t)st.st_size + 1;   // + 1: the read that finds EOF
    for (;;) {
        if (out.n == cap || !out.p) {
            if (out.p) cap += cap / 2;
            char *q = static_cast<char *>(realloc(out.p, cap));
            if (!q) throw std::bad_alloc();
            out.p = q;
        }
        const size_t got = fread(out.p + out.n, 1, cap - out.n, f);
        out.n += got;
        if (got == 0) break;
    }
    return !ferror(f);
}

bool append_blocks(const std::string &path, const std::vector<std::string> &blocks) {
    FILE *f = fopen(path.c_str(), "ab");
    if (!f) return false;
    bool ok = true;
    for (const std::string &b : blocks)
        if (!b.empty() && fwrite(b.data(), 1, b.size(), f) != b.size()) { ok = false; break; }
    return fclose(f) == 0 && ok;
}

bool append_file(const std::string &path, const char *data, uint64_t n) {
    FILE *f = fopen(path.c_str(), "ab");
    if (!f) return false;
    const bool ok = n == 0 || fwrite(data, 1, n, f) == n;
    return fclose(f) == 0 && ok;
}

}  // namespace

extern "C" int cls_sequences_open(const char *query_path, const char *out_file, uint32_t format, uint32_t overwrite,
                                  cls_sequences **out, cls_batch *batch) {
    using cls::set_last_error;
    if (!out_file || !out || !batch) return set_last_error(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    *out = nullptr;
    const bool fastq = (format & CLS_QUERY_FASTQ) != 0;
    format &= ~CLS_QUERY_FASTQ;
    if (format > 1) return set_last_error(CLS_ERR_INVALID_ARGUMENT, "format must be 0 (yaml) or 1 (jsonl), optionally ORed with CLS_QUERY_FASTQ");
    try {
        auto s = std::make_unique<cls_sequences>();
        s->format = format;
        s->out_path = with_extension(out_file, format == 0 ? "yaml" : "jsonl");       // :73-90
        s->err_path = with_extension(out_file, "error");
        const size_t slash = s->out_path.find_last_of('/');
        if (slash != std::string::npos && slash > 0) {
            const std::string dir = s->out_path.substr(0, slash);
            struct stat st;
            if (stat(dir.c_str(), &st) != 0) mkdir(dir.c_str(), 0777);                 // create_dir, its error ignored (:92-94)
        }
        struct stat st;
        if (stat(s->out_path.c_str(), &st) == 0) {
            if (!overwrite) {                                                           // :96-101
                std::string msg = "Could not overwrite existing file ";
                rust_debug_str(s->out_path, msg);
                msg += " when overwrite option is `false`.";
                return set_last_error(CLS_ERR_INVALID_ARGUMENT, msg);
            }
            if (remove(s->out_path.c_str()) != 0)                                        // :103-110
                return set_last_error(CLS_ERR_INVALID_ARGUMENT, std::string("Could not remove file given ") + strerror(errno));
        }
        const bool use_stdin = !query_path || strcmp(query_path, "-") == 0;
        FILE *f = use_stdin ? stdin : fopen(query_path, "rb");
        // a query that cannot be opened or read is NOT an error of the use-case: the reference drops the reader's
        // Result (`let _ = query_sequence.sequence_content_by_channel(sender)`, :119), creates both files and
        // returns Ok with nothing placed
        struct Close { FILE *f; bool own; ~Close() { if (f && own) fclose(f); } } closer{f, !use_stdin};   // also when an allocation throws
        if (!f || !read_whole(f, s->text)) s->text.clear();
        const uint8_t *text = reinterpret_cast<const uint8_t *>(s->text.p);
        const int rc = fastq ? cls_fastq_read(text, s->text.n, &s->records, &s->rec) : cls_fasta_read(text, s->text.n, &s->records, &s->rec);
        if (rc != CLS_OK) return rc;
        s->header_off.assign(s->rec.n_records + 1, 0);
        uint64_t hbytes = 0;
        for (uint64_t i = 0; i < s->rec.n_records; ++i) hbytes += s->rec.header_end[i] - s->rec.header_begin[i];
        s->headers.reserve(hbytes);
        for (uint64_t i = 0; i < s->rec.n_records; ++i) {          // the header line minus every '>' (:102); a FASTQ title as it is
            const char *a = s->text.p + s->rec.header_begin[i], *e = s->text.p + s->rec.header_end[i];
            if (fastq) s->headers.append(a, e);
            while (a < e && !fastq) {
                const char *g = static_cast<const char *>(memchr(a, '>', (size_t)(e - a)));
                if (!g) g = e;
                s->headers.append(a, g);
                a = g + 1;
            }
            s->header_off[i + 1] = s->headers.size();
        }
        if (!append_file(s->out_path, nullptr, 0) || !append_file(s->err_path, nullptr, 0))   // both files exist from here on
            return set_last_error(CLS_ERR_INVALID_ARGUMENT, "cannot create " + s->out_path + " / " + s->err_path);
        batch->n_queries = s->rec.n_records;
        batch->bases = s->rec.bases;
        batch->offsets = s->rec.offsets;
        *out = s.release();
        return CLS_OK;
    } catch (const std::bad_alloc &) {
        return set_last_error(CLS_ERR_OUT_OF_MEMORY, "host allocation failed while opening the query sequences");
    }
}

extern "C" int cls_sequences_write(cls_sequences *s, const cls_record_tree *tree, uint64_t n, const cls_result *result) {
    using cls::set_last_error;
    if (!s || !tree || !result) return set_last_error(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (s->written + n > s->rec.n_records) return set_last_error(CLS_ERR_INVALID_ARGUMENT, "more results than records");
    try {
        std::vector<std::string> outs, errs;
        // header_off is absolute into `headers`: the writer takes the sub-array as it is; the blocks go to the files as
        // they are (no concatenated copy of what can be a gigabyte of text)
        const int rc = render_blocks(tree, n, s->header_off.data() + s->written, s->headers.data(), result, s->format, outs, errs);
        if (rc != CLS_OK) return rc;
        if (!append_blocks(s->out_path, outs) || !append_blocks(s->err_path, errs))
            return set_last_error(CLS_ERR_INVALID_ARGUMENT, "Error writing to file: " + s->out_path);
        s->written += n;
        return CLS_OK;
    } catch (const std::bad_alloc &) {
        return set_last_error(CLS_ERR_OUT_OF_MEMORY, "host allocation failed while writing records");
    }
}

extern "C" void cls_sequences_close(cls_sequences *s) { delete s; }

extern "C" int cls_place_sequences(cls_index *index, const cls_record_tree *tree, const char *query_path, const char *out_file,
                                   const cls_params *params, uint32_t format, uint32_t overwrite, uint64_t *n_placed) {
    using cls::set_last_error;
    if (!index || !tree || !params) return set_last_error(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (n_placed) *n_placed = 0;
    cls_sequences *s = nullptr;
    cls_batch all{};
    int rc = cls_sequences_open(query_path, out_file, format, overwrite, &s, &all);
    if (rc != CLS_OK) return rc;
    std::unique_ptr<cls_sequences> guard(s);
    try {
        // queries per device call: bounds the result arrays (CLS_SEQ_BATCH: smaller batches, for tests of this loop)
        static const uint64_t kBatch = [] { const char *e = getenv("CLS_SEQ_BATCH"); const long v = e ? atol(e) : 0; return v > 0 ? (uint64_t)v : 1ull << 20; }();
        const uint64_t cap = std::min<uint64_t>(all.n_queries, kBatch);
        // Two sets of result arrays: the records of batch i are rendered and appended to the files (host pool + file
        // I/O) on a second thread WHILE batch i + 1 is placed - the writer, not the GPU, sets the pace of a big file
        // otherwise (1.27 GB of YAML per million records).  Writes stay in order: write i + 1 starts after write i ended.
        struct ResultArrays {
            std::vector<uint8_t> status;
            std::vector<uint64_t> node;
            std::vector<int32_t> one, rest;
            std::vector<uint32_t> nq, nm, nr, it;
            cls_result res{};
            explicit ResultArrays(uint64_t c) : status(c), node(c), one(c), rest(c), nq(c), nm(c), nr(c), it(c) {
                res = cls_result{status.data(), node.data(), one.data(), rest.data(), nq.data(), nm.data(), nr.data(), it.data()};
            }
        };
        const bool two = all.n_queries > kBatch;
        ResultArrays buf0(cap), buf1(two ? cap : 0);
        ResultArrays *bufs[2] = {&buf0, two ? &buf1 : &buf0};
        std::future<std::pair<int, std::string>> pending;   // the write of the previous batch (error text: thread-local over there)
        uint64_t pending_n = 0;
        auto finish_write = [&]() -> int {
            if (!pending.valid()) return CLS_OK;
            const std::pair<int, std::string> r = pending.get();
            if (r.first != CLS_OK) return set_last_error(r.first, r.second);
            if (n_placed) *n_placed += pending_n;
            return CLS_OK;
        };
        uint64_t i = 0;
        for (uint64_t a = 0; a < all.n_queries; a += kBatch, ++i) {
            const uint64_t n = std::min<uint64_t>(kBatch, all.n_queries - a);
            const cls_batch part{n, all.bases, all.offsets + a};   // offsets are absolute into `bases`
            ResultArrays *b = bufs[i & 1];                          // last used by write i - 2, which has ended
            rc = cls_place_batch(index, &part, params, &b->res);
            const int wrc = finish_write();                         // write i - 1 (it ran meanwhile)
            if (rc != CLS_OK) return rc;
            if (wrc != CLS_OK) return wrc;
            pending_n = n;
            pending = std::async(std::launch::async, [s, tree, n, b]() {
                const int r = cls_sequences_write(s, tree, n, &b->res);
                return std::make_pair(r, std::string(r == CLS_OK ? "" : cls_last_error()));
            });
        }
        return finish_write();
    } catch (const std::bad_alloc &) {
        return set_last_error(CLS_ERR_OUT_OF_MEMORY, "host allocation failed in cls_place_sequences");
    }
}
