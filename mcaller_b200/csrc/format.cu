// Host-side writer of the `.diffs.<k>` rows (reference extract_contexts.py:216 + writefi :83-86), native and multi-threaded
// (row ranges formatted by host threads into private buffers, then concatenated in row order) so that runs with millions
// of calls are not bound by string formatting.  Floats are printed like str(np.float64) / repr(float):
// the shortest digit string that round-trips (std::to_chars), fixed notation for 1e-4 <= |x| < 1e16, else scientific
// with a two-digit exponent; empty columns print the integer 0; the probability is np.round(p, 2) (rint(p*100)/100).
#include <charconv>
#include <cmath>
#include <cstring>
#include <string>
#include <thread>
#include <vector>
#include "common.cuh"

namespace {

struct Out {
    char *p, *end;
    bool ok = true;
    void put(char c) { if (p < end) *p++ = c; else ok = false; }
    void put(const char *s, size_t n) { if ((size_t)(end - p) >= n) { memcpy(p, s, n); p += n; } else ok = false; }
    void put(const char *s) { put(s, strlen(s)); }
};

void put_repr(Out &o, double v) {
    if (std::isnan(v)) { o.put("nan"); return; }
    if (std::isinf(v)) { o.put(v < 0 ? "-inf" : "inf"); return; }
    if (v == 0.0) { o.put(std::signbit(v) ? "-0.0" : "0.0"); return; }
    char buf[64];
    auto r = std::to_chars(buf, buf + sizeof(buf), v, std::chars_format::scientific);   // shortest round-trip digits
    *r.ptr = 0;
    // parse  [-]d[.ddd]e[+-]XX
    const char *s = buf;
    if (*s == '-') { o.put('-'); ++s; }
    char digits[32];
    int nd = 0;
    digits[nd++] = *s++;
    if (*s == '.') { ++s; while (*s != 'e') digits[nd++] = *s++; }
    ++s;                                   // 'e'
    const int e10 = atoi(s);
    if (e10 >= -4 && e10 < 16) {
        if (e10 >= 0) {
            for (int i = 0; i <= e10; ++i) o.put(i < nd ? digits[i] : '0');
            o.put('.');
            if (nd > e10 + 1) o.put(digits + e10 + 1, (size_t)(nd - e10 - 1)); else o.put('0');
        } else {
            o.put("0.");
            for (int i = 0; i < -e10 - 1; ++i) o.put('0');
            o.put(digits, (size_t)nd);
        }
    } else {
        o.put(digits[0]);
        if (nd > 1) { o.put('.'); o.put(digits + 1, (size_t)(nd - 1)); }
        o.put('e');
        o.put(e10 < 0 ? '-' : '+');
        const int a = e10 < 0 ? -e10 : e10;
        char eb[8];
        const int n = snprintf(eb, sizeof(eb), "%02d", a);
        o.put(eb, (size_t)n);
    }
}

void put_int(Out &o, long long v) {
    char b[32];
    auto r = std::to_chars(b, b + sizeof(b), v);
    o.put(b, (size_t)(r.ptr - b));
}

// the probability column: np.round(p, 2) printed as str(np.float64)
void put_prob(Out &o, double p) { put_repr(o, std::rint(p * 100.0) / 100.0); }

char comp(char c) {
    switch (c) { case 'A': return 'T'; case 'C': return 'G'; case 'G': return 'C'; case 'T': return 'A'; case 'N': return 'N'; case 'M': return 'M'; }
    return 0;
}

}  // namespace

namespace {

struct FormatArgs {
    const mc_call *h_calls;
    const uint8_t *h_text;
    const uint8_t *carry_name;
    int32_t carry_name_len;
    const char *const *contig_names, *const *marked_fwd, *const *marked_rev;
    const int64_t *contig_len;
    int32_t n_contigs, k, with_prob;
    const char *base_label, *mod_label;
};

// rows [lo, hi) appended to `dst`; returns 0 or a negative error code and leaves the failing row / flags in err_*
int64_t format_range(const FormatArgs &A, int64_t lo, int64_t hi, std::string &dst, int64_t &err_row, int &err_flags) {
    char line[4096];
    for (int64_t i = lo; i < hi; ++i) {
        const mc_call &c = A.h_calls[i];
        if (c.kind != MC_CALL || c.close_rec == 0xFFFFFFFFu) continue;
        if (c.err) { err_row = i; err_flags = c.err; return -100 - (int64_t)c.err; }
        if (c.chrom_contig >= A.n_contigs || c.win_contig >= A.n_contigs) { err_row = i; err_flags = -1; return MC_EINVAL; }
        const char *src = c.rev ? A.marked_rev[c.win_contig] : A.marked_fwd[c.win_contig];
        const int64_t a = (int64_t)c.mpos - A.k + 1, b = (int64_t)c.mpos + A.k;
        if (a < 0 || b > A.contig_len[c.win_contig]) { err_row = i; err_flags = -2; return MC_EINVAL; }
        const size_t name_len = strlen(A.contig_names[c.chrom_contig]);
        // the read name: bytes of this chunk's text, or (a window carried over a chunk edge) the name the caller kept
        const char *read = reinterpret_cast<const char *>(A.h_text) + c.read_off;
        size_t read_len = (size_t)c.read_len;
        if (c.read_off >= 0 && !A.h_text) { err_row = i; err_flags = -6; return MC_EINVAL; }
        if (c.read_off < 0) {
            if (!A.carry_name) { err_row = i; err_flags = -4; return MC_EINVAL; }
            read = reinterpret_cast<const char *>(A.carry_name);
            read_len = (size_t)A.carry_name_len;
        }
        if (name_len + read_len + 1024 > sizeof(line)) {                    // unusually long names: straight into the string
            dst.append(A.contig_names[c.chrom_contig], name_len);
            dst.push_back('\t');
            dst.append(read, read_len);
        }
        Out o{line, line + sizeof(line)};
        if (name_len + read_len + 1024 <= sizeof(line)) {
            o.put(A.contig_names[c.chrom_contig], name_len);
            o.put('\t');
            o.put(read, read_len);
        }
        o.put('\t');
        put_int(o, c.mpos);
        o.put('\t');
        // context = revcomp(last_ref[mpos-k+1 : mpos+k], last_rev)   (extract_contexts.py:194)
        for (int64_t j = 0; j < b - a; ++j) {
            const char ch = c.rev ? comp(src[b - 1 - j]) : src[a + j];
            if (ch == 0) { err_row = i; err_flags = -5; return MC_EINVAL; }   // revcomp of a letter outside ACGTNM (:11-15 KeyError)
            o.put(ch);
        }
        o.put('\t');
        for (int j = 0; j <= A.k; ++j) {
            if (j) o.put(',');
            if (j < A.k && ((c.empty_mask >> j) & 1u)) o.put('0'); else put_repr(o, c.feat[j]);
        }
        o.put('\t');
        o.put(c.rev ? '-' : '+');
        if (A.with_prob) {
            o.put('\t');
            o.put(c.prob >= 0.5 ? A.mod_label : A.base_label);
            o.put('\t');
            put_prob(o, c.prob);
        }
        o.put('\n');
        if (!o.ok) { err_row = i; err_flags = -3; return MC_ECAPACITY; }       // cannot happen: labels are short
        dst.append(line, (size_t)(o.p - line));
    }
    return 0;
}

}  // namespace

extern "C" int64_t mc_format_rows(const mc_call *h_calls, int64_t n_calls, const uint8_t *h_text, const uint8_t *carry_name,
                                  int32_t carry_name_len, const char *const *contig_names, const char *const *marked_fwd,
                                  const char *const *marked_rev, const int64_t *contig_len, int32_t n_contigs, int32_t k,
                                  const char *base_label, const char *mod_label, int32_t with_prob, int32_t max_threads, char *out,
                                  int64_t out_cap) {
    if (!h_calls || !contig_names || !marked_fwd || !marked_rev || !contig_len || !out || k < 1 || k > MC_MAXK ||
        !base_label || !mod_label || strlen(base_label) > 256 || strlen(mod_label) > 256) {
        mc_set_error("mc_format_rows: bad argument");
        return MC_EINVAL;
    }
    const FormatArgs A{h_calls, h_text, carry_name, carry_name_len, contig_names, marked_fwd, marked_rev, contig_len, n_contigs, k, with_prob,
                       base_label, mod_label};
    // one host thread per ~2k rows (a thread costs ~20 us to start, 2k rows ~2 ms to render), at most the hardware concurrency
    unsigned hw = std::thread::hardware_concurrency();
    if (hw == 0) hw = 1;
    if (max_threads > 0 && (unsigned)max_threads < hw) hw = (unsigned)max_threads;
    int nt = (int)((n_calls + 2047) / 2048);
    if (nt > (int)hw) nt = (int)hw;
    if (nt < 1) nt = 1;
    std::vector<std::string> parts((size_t)nt);
    std::vector<int64_t> rc((size_t)nt, 0), erow((size_t)nt, -1);
    std::vector<int> eflags((size_t)nt, 0);
    auto work = [&](int t) {
        const int64_t lo = n_calls * t / nt, hi = n_calls * (t + 1) / nt;
        parts[(size_t)t].reserve((size_t)(hi - lo) * 200);
        rc[(size_t)t] = format_range(A, lo, hi, parts[(size_t)t], erow[(size_t)t], eflags[(size_t)t]);
    };
    if (nt == 1) work(0);
    else {
        std::vector<std::thread> th;
        for (int t = 1; t < nt; ++t) th.emplace_back(work, t);
        work(0);
        for (auto &x : th) x.join();
    }
    for (int t = 0; t < nt; ++t) {                                  // the first failing row in row order decides
        if (rc[(size_t)t] == 0) continue;
        if (eflags[(size_t)t] > 0)
            mc_set_error("row %lld (position %d) carries error flags 0x%x", (long long)erow[(size_t)t], h_calls[erow[(size_t)t]].mpos,
                         (unsigned)eflags[(size_t)t]);
        else if (eflags[(size_t)t] == -1) mc_set_error("mc_format_rows: contig index out of range");
        else if (eflags[(size_t)t] == -2) mc_set_error("mc_format_rows: context out of range");
        else if (eflags[(size_t)t] == -4) mc_set_error("mc_format_rows: row %lld was carried over a chunk edge but no read name was given", (long long)erow[(size_t)t]);
        else if (eflags[(size_t)t] == -6) mc_set_error("mc_format_rows: row %lld names its read by offset but no text was given", (long long)erow[(size_t)t]);
        else if (eflags[(size_t)t] == -5)
            mc_set_error("mc_format_rows: the context of row %lld (position %d) covers a reference letter outside ACGTNM", (long long)erow[(size_t)t],
                         h_calls[erow[(size_t)t]].mpos);
        else mc_set_error("mc_format_rows: row too long");
        return rc[(size_t)t];
    }
    int64_t total = 0;
    for (auto &sp : parts) total += (int64_t)sp.size();
    if (total > out_cap) { mc_set_error("mc_format_rows: output buffer too small"); return MC_ECAPACITY; }
    char *p = out;
    for (auto &sp : parts) { memcpy(p, sp.data(), sp.size()); p += sp.size(); }
    return total;
}

extern "C" int64_t mc_format_probs(const double *h_prob, int64_t n, int32_t max_threads, char *out, int64_t out_cap, int64_t *h_offsets) {
    if ((n > 0 && (!h_prob || !out)) || !h_offsets || n < 0) {
        mc_set_error("mc_format_probs: bad argument");
        return MC_EINVAL;
    }
    // a string is at most 24 bytes ("-1.2345678901234567e-05"), so slices of the output fit 32 bytes per value
    if (out_cap < 32 * n) { mc_set_error("mc_format_probs: output buffer too small"); return MC_ECAPACITY; }
    unsigned hw = std::thread::hardware_concurrency();
    if (hw == 0) hw = 1;
    if (max_threads > 0 && (unsigned)max_threads < hw) hw = (unsigned)max_threads;
    int nt = (int)((n + 65535) / 65536);                            // ~65k values per thread (~5 ms of rendering)
    if (nt > (int)hw) nt = (int)hw;
    if (nt < 1) nt = 1;
    // thread t renders values [lo, hi) into out[32 lo, 32 hi) with offsets relative to its slice; then the slices are packed
    std::vector<int64_t> used((size_t)nt, 0);
    auto work = [&](int t) {
        const int64_t lo = n * t / nt, hi = n * (t + 1) / nt;
        Out o{out + 32 * lo, out + 32 * hi};
        for (int64_t i = lo; i < hi; ++i) {
            h_offsets[i] = (int64_t)(o.p - (out + 32 * lo));
            put_prob(o, h_prob[i]);
        }
        used[(size_t)t] = (int64_t)(o.p - (out + 32 * lo));
    };
    if (nt == 1) work(0);
    else {
        std::vector<std::thread> th;
        for (int t = 1; t < nt; ++t) th.emplace_back(work, t);
        work(0);
        for (auto &x : th) x.join();
    }
    int64_t total = 0;
    for (int t = 0; t < nt; ++t) {
        const int64_t lo = n * t / nt, hi = n * (t + 1) / nt;
        if (total != 32 * lo) memmove(out + total, out + 32 * lo, (size_t)used[(size_t)t]);
        for (int64_t i = lo; i < hi; ++i) h_offsets[i] += total;
        total += used[(size_t)t];
    }
    h_offsets[n] = total;
    return total;
}
