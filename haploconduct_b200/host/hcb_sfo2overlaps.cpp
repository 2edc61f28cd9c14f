// hc_sfo2overlaps -- scripts/sfo2overlaps.py of the reference in C++ on all host threads: the output of the
// suffix-filter overlapper (SFO / rust-overlaps: "idA idB ori OHA OHB OLA OLB K" per line) -> the 13-column overlaps file
// EdgeCalculator reads, with the overlaps of the two ends of a paired-end read matched into one paired overlap.
// Same flags, same temporary semantics, same output BYTES as the script run under LC_ALL=C:
//   1. every line gets the two original read ids in front (the two ends of a pair share one, :136-147) and is flipped so
//      that the smaller original id comes first (:38-48, flip_N / flip_I :108-119);
//   2. `sort -k1,1n -k2,2n -k3,3n -k4,4n | uniq` (:51): four numeric keys, ties by the bytes of the whole line (C locale),
//      identical adjacent lines dropped;
//   3. one pass over the sorted lines (:56-100): a line between two single-end reads gives its overlap at once
//      (get_s_s_overlap :150-205); lines that involve a paired-end read are collected per (idA, idB) and matched pairwise when
//      the NEXT such pair shows up (match_candidates / find_paired_overlap / merge_overlaps :208-329) -- so the pairs of the
//      last collected id pair are never written, and a pair's overlaps follow the single-single lines read in between;
//   4. `uniq` on the result (:104).
// The script spends its time in the Python loop and two external sorts; here parsing, flipping, sorting (parallel merge
// sort) and the per-line / per-pair work run on all host threads and the results are stitched in the script's order.
// SURVEY 8f rank 2 (the converter half).  Reference: scripts/sfo2overlaps.py.
// --gpu=true: the same bytes from one hc_sfo2overlaps call (include/hc_b200.h; all of 1-4 on the device).  Input the
// device path does not take (a line this program dies on, or one outside the device's ranges) or a working set that does
// not fit the device is said on stderr and converted here as without the flag; no usable device is an error.
#include <omp.h>

#include "../../include/hc_b200.h"

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

namespace {

[[noreturn]] void die(const std::string& m) {
    std::fprintf(stderr, "%s\n", m.c_str());
    std::exit(1);
}

struct Rec {                 // one line of the temporary file: idA idB sfoA sfoB ori OHA OHB OLA OLB K
    long idA, idB, sfoA, sfoB;
    char ori;
    long OHA, OHB, OLA, OLB;
    const char* text;        // the line as the script writes it (without '\n'): sort's last-resort key, uniq's identity --
    uint32_t text_len;       // bytes in the arena of the thread that parsed the line
};

int text_cmp(const Rec& a, const Rec& b) {                    // bytes as unsigned char, shorter first on a common prefix (LC_ALL=C)
    const uint32_t n = a.text_len < b.text_len ? a.text_len : b.text_len;
    const int c = std::memcmp(a.text, b.text, n);
    if (c) return c;
    return a.text_len < b.text_len ? -1 : (a.text_len > b.text_len ? 1 : 0);
}

bool parse_long(const char* b, const char* e, long& v) {       // Python int() on a whitespace-free token
    if (b == e) return false;
    const char* p = b;
    bool neg = false;
    if (*p == '+' || *p == '-') { neg = *p == '-'; p++; }
    if (p == e) return false;
    long x = 0;
    for (; p < e; p++) {
        if (*p < '0' || *p > '9') return false;
        x = x * 10 + (*p - '0');
    }
    v = neg ? -x : x;
    return true;
}

// str.split(): fields separated by runs of whitespace
int split_ws(const char* b, const char* e, const char* fb[], const char* fe[], int maxf) {
    int n = 0;
    const char* p = b;
    while (p < e) {
        while (p < e && (*p == ' ' || *p == '\t' || *p == '\r' || *p == '\v' || *p == '\f' || *p == '\n')) p++;
        if (p >= e) break;
        const char* s = p;
        while (p < e && !(*p == ' ' || *p == '\t' || *p == '\r' || *p == '\v' || *p == '\f' || *p == '\n')) p++;
        if (n < maxf) { fb[n] = s; fe[n] = p; }
        n++;
    }
    return n;
}

long original_id(long sfo, long ns, long np) {                 // get_original_id :136-147
    if (np == 0) return sfo;
    if (!(sfo >= 0 && sfo < ns + 2 * np)) die("AssertionError: sfo_ID >= 0 and sfo_ID < num_singles + 2*num_pairs");
    return sfo < ns + np ? sfo : sfo - np;
}

bool is_paired(long id, long ns, long np) {                    // :121-133
    if (np == 0) return false;
    if (!(id >= 0 && id < ns + np)) die("AssertionError: ID >= 0 and ID < num_singles + num_pairs");
    return id >= ns;
}

struct SS {                  // get_s_s_overlap :150-205
    long id1, id2, pos1, perc, len1;
    char ori1, ori2;
};

SS s_s_overlap(const Rec& r) {
    SS o;
    const char ori = r.ori == 'N' ? '+' : '-';
    const long ovlen = std::min(r.OLA, r.OLB);
    long lenA, lenB;
    if (r.OHA >= 0) {
        if (r.OHB >= 0) { lenA = r.OLA + r.OHA; lenB = r.OLB + r.OHB; }
        else { lenA = r.OLA + r.OHA - r.OHB; lenB = r.OLB; }
        o.id1 = r.idA; o.id2 = r.idB; o.pos1 = r.OHA; o.ori1 = '+'; o.ori2 = ori;
    } else {
        if (r.OHB >= 0) { lenA = r.OLA; lenB = -r.OHA + r.OLB + r.OHB; }
        else { lenA = r.OLA - r.OHB; lenB = -r.OHA + r.OLB; }
        o.id1 = r.idB; o.id2 = r.idA; o.pos1 = -r.OHA; o.ori1 = ori; o.ori2 = '+';
    }
    const long minlen = std::min(lenA, lenB);
    if (minlen == 0) die("ZeroDivisionError: float division by zero");
    // min(round(100*ovlen/minreadlen), 100): true division, Python 2's round (half away from zero), printed with "{:.0f}"
    const double x = std::round((double)(100 * ovlen) / (double)minlen);
    const double p = std::min(x, 100.0);
    char buf[32];
    std::snprintf(buf, sizeof(buf), "%.0f", p);
    o.perc = std::atol(buf);
    o.len1 = ovlen;
    if (!(minlen > 0)) die("AssertionError: minreadlen > 0");
    return o;
}

void put_long(std::string& b, long v) {
    char tmp[24];
    int k = 24;
    unsigned long u = v < 0 ? 0ul - (unsigned long)v : (unsigned long)v;
    do { tmp[--k] = (char)('0' + u % 10); u /= 10; } while (u);
    if (v < 0) tmp[--k] = '-';
    b.append(tmp + k, (size_t)(24 - k));
}

void put_ss_line(std::string& b, const SS& o) {                // ID1 ID2 POS1 - - ORI1 ORI2 PERC1 - LEN1 - s s
    put_long(b, o.id1); b += '\t'; put_long(b, o.id2); b += '\t'; put_long(b, o.pos1); b += "\t-\t-\t";
    b += o.ori1; b += '\t'; b += o.ori2; b += '\t'; put_long(b, o.perc); b += "\t-\t"; put_long(b, o.len1); b += "\t-\ts\ts\n";
}

// find_paired_overlap + merge_overlaps :226-329; appends the line if the two candidates match
void paired_overlap(std::string& b, const Rec& c1, const Rec& c2, bool typeA, bool typeB) {
    if (c1.ori != c2.ori) return;
    int first = 0;          // 1: (overlap1, overlap2) = (c1, c2); 2: = (c2, c1)
    const bool N = c1.ori == 'N', I = c1.ori == 'I';
    if (typeA && typeB) {
        if (N) { if (c1.sfoA < c2.sfoA && c1.sfoB < c2.sfoB) first = 1; else if (c1.sfoA > c2.sfoA && c1.sfoB > c2.sfoB) first = 2; }
        else if (I) { if (c1.sfoA < c2.sfoA && c1.sfoB > c2.sfoB) first = 1; else if (c1.sfoA > c2.sfoA && c1.sfoB < c2.sfoB) first = 2; }
    } else if (typeA && !typeB) {
        if (N) { if (c1.sfoA < c2.sfoA && c1.OHA < c2.OHA) first = 1; else if (c1.sfoA > c2.sfoA && c1.OHA > c2.OHA) first = 2; }
        else if (I) { if (c1.sfoA < c2.sfoA && c1.OHA > c2.OHA) first = 2; else if (c1.sfoA > c2.sfoA && c1.OHA < c2.OHA) first = 1; }
    } else {
        if (N) { if (c1.sfoB < c2.sfoB && c1.OHA < c2.OHA) first = 1; else if (c1.sfoB > c2.sfoB && c1.OHA > c2.OHA) first = 2; }
        else if (I) { if (c1.sfoB < c2.sfoB && c1.OHA > c2.OHA) first = 2; else if (c1.sfoB > c2.sfoB && c1.OHA < c2.OHA) first = 1; }
    }
    if (!first) return;
    const SS o1 = s_s_overlap(first == 1 ? c1 : c2), o2 = s_s_overlap(first == 1 ? c2 : c1);
    char t1, t2;
    if (o1.id1 == c1.idA) {
        if (o1.id2 != c1.idB) die("AssertionError: overlap1[1] == cand1[1]");
        t1 = typeA ? 'p' : 's'; t2 = typeB ? 'p' : 's';
    } else {
        if (o1.id2 != c1.idA || o1.id1 != c1.idB) die("AssertionError: overlap1[1] == cand1[0]");
        t1 = typeB ? 'p' : 's'; t2 = typeA ? 'p' : 's';
    }
    char ord = '-';
    if (t1 == 'p' && t2 == 'p') {
        if (o1.id1 != o2.id1) {
            if (o1.id1 != o2.id2) die("AssertionError: overlap1[0] == overlap2[1]");
            ord = '2';
        } else {
            ord = '1';
        }
    }
    put_long(b, o1.id1); b += '\t'; put_long(b, o1.id2); b += '\t'; put_long(b, o1.pos1); b += '\t'; put_long(b, o2.pos1); b += '\t';
    b += ord; b += '\t'; b += o1.ori1; b += '\t'; b += o1.ori2; b += '\t'; put_long(b, o1.perc); b += '\t'; put_long(b, o2.perc); b += '\t';
    put_long(b, o1.len1); b += '\t'; put_long(b, o2.len1); b += '\t'; b += t1; b += '\t'; b += t2; b += '\n';
}

bool rec_less(const Rec& a, const Rec& b) {                   // sort -k1,1n -k2,2n -k3,3n -k4,4n, then the whole line (LC_ALL=C)
    if (a.idA != b.idA) return a.idA < b.idA;
    if (a.idB != b.idB) return a.idB < b.idB;
    if (a.sfoA != b.sfoA) return a.sfoA < b.sfoA;
    if (a.sfoB != b.sfoB) return a.sfoB < b.sfoB;
    return text_cmp(a, b) < 0;
}

void parallel_sort(std::vector<Rec>& v) {
    const int T = std::max(1, omp_get_max_threads());
    const size_t n = v.size();
    if (T == 1 || n < 1u << 15) { std::sort(v.begin(), v.end(), rec_less); return; }
    std::vector<size_t> cut(T + 1);
    for (int t = 0; t <= T; t++) cut[t] = n * (size_t)t / (size_t)T;
#pragma omp parallel for schedule(static, 1)
    for (int t = 0; t < T; t++) std::sort(v.begin() + cut[t], v.begin() + cut[t + 1], rec_less);
    for (int w = 1; w < T; w *= 2) {
#pragma omp parallel for schedule(dynamic, 1)
        for (int t = 0; t < T; t += 2 * w) {
            const int m = std::min(t + w, T), e = std::min(t + 2 * w, T);
            if (m < e) std::inplace_merge(v.begin() + cut[t], v.begin() + cut[m], v.begin() + cut[e], rec_less);
        }
    }
}

}  // namespace

static double now_s() { return omp_get_wtime(); }

int main(int argc, char** argv) {
    const bool timing = getenv("HC_TIMING") != nullptr;
    double t_mark = now_s();
    auto mark = [&](const char* what) { if (timing) { const double t = now_s(); std::fprintf(stderr, "[hc_sfo2overlaps] %-28s %8.1f ms\n", what, (t - t_mark) * 1e3); t_mark = t; } };
    std::string in, out;
    long ns = -1, np = -1;
    bool gpu = false;
    for (int i = 1; i < argc; i++) {
        std::string a = argv[i], v;
        const size_t eq = a.find('=');
        if (eq != std::string::npos) { v = a.substr(eq + 1); a = a.substr(0, eq); }
        else if (i + 1 < argc) v = argv[++i];
        if (a == "--in") in = v;
        else if (a == "--out") out = v;
        else if (a == "--num_singles") ns = std::atol(v.c_str());
        else if (a == "--num_pairs") np = std::atol(v.c_str());
        else if (a == "--gpu") gpu = v == "true" || v == "1";
        else { std::fprintf(stderr, "unknown option %s\n", a.c_str()); return 2; }
    }
    if (in.empty() || out.empty() || ns < 0 || np < 0) {
        std::fprintf(stderr, "usage: hc_sfo2overlaps --in SFO --out OVERLAPS --num_singles N --num_pairs N [--gpu=true]\n");
        return 2;
    }
    // ---- the file
    const int fd = open(in.c_str(), O_RDONLY);
    if (fd < 0) die("IOError: [Errno 2] No such file or directory: '" + in + "'");
    struct stat st;
    fstat(fd, &st);
    std::string text((size_t)std::max<off_t>(st.st_size, 0), '\0');
    {
        const size_t blk = 8u << 20, nb = (text.size() + blk - 1) / blk;
#pragma omp parallel for schedule(dynamic, 1)
        for (long b = 0; b < (long)nb; b++) {
            size_t o = (size_t)b * blk;
            const size_t end = std::min(text.size(), o + blk);
            while (o < end) {
                const ssize_t r = pread(fd, &text[o], end - o, (off_t)o);
                if (r <= 0) break;
                o += (size_t)r;
            }
        }
    }
    close(fd);
    mark("file read");
    if (gpu) {
        // the output is rarely more than twice the input; a larger one costs a second call with the exact size
        uint64_t cap = 2 * (uint64_t)text.size() + 4096, n_out = 0;
        hc_sfo_stats st;
        char* buf = (char*)std::malloc(cap);
        if (!buf) die("hc_sfo2overlaps: out of host memory");
        int rc = hc_sfo2overlaps(text.data(), text.size(), ns, np, buf, cap, &n_out, &st, 0);
        if (rc == HC_ERR_CAPACITY) {
            std::free(buf);
            cap = n_out;
            buf = (char*)std::malloc(cap ? cap : 1);
            if (!buf) die("hc_sfo2overlaps: out of host memory");
            rc = hc_sfo2overlaps(text.data(), text.size(), ns, np, buf, cap, &n_out, &st, 0);
        }
        if (rc == HC_OK) {
            mark("device call");
            if (timing)
                std::fprintf(stderr, "[hc_sfo2overlaps]   copy in %.1f ms, device %.1f ms, copy out %.1f ms\n", st.h2d_ms, st.device_ms, st.d2h_ms);
            FILE* fo = std::fopen(out.c_str(), "w");
            if (!fo) die("IOError: cannot write " + out);
            if (std::fwrite(buf, 1, n_out, fo) != n_out || std::fclose(fo) != 0) die("IOError: cannot write " + out);
            std::free(buf);
            mark("write");
            std::printf("total overlap count: %lu\nof which single-single: %lu\n", (unsigned long)(st.s_s_count + st.p_count),
                        (unsigned long)st.s_s_count);
            return 0;
        }
        std::free(buf);
        if (rc != HC_ERR_INPUT && rc != HC_ERR_NOMEM) die(hc_last_error());
        std::fprintf(stderr, "%s; converting on the host\n", hc_last_error());
        mark("device call (not taken)");
    }
    std::vector<size_t> ls(1, 0);                               // line starts
    for (size_t i = 0; i < text.size(); i++) if (text[i] == '\n' && i + 1 < text.size()) ls.push_back(i + 1);
    if (text.empty()) ls.clear();
    const size_t nl = ls.size();
    mark("line starts");
    // ---- 1. original ids in front, smaller one first
    std::vector<Rec> recs(nl);
    // the temporary file's lines live in one arena per thread (a flipped line is at most a few bytes longer than the original
    // plus the two ids in front: 48 bytes of headroom per line)
    const int T = std::max(1, omp_get_max_threads());
    std::vector<std::vector<char>> arena(T);
#pragma omp parallel num_threads(T)
    {
    const int tid = omp_get_thread_num();
    const size_t klo = nl * (size_t)tid / (size_t)T, khi = nl * (size_t)(tid + 1) / (size_t)T;
    const size_t span = klo < khi ? ((khi < nl ? ls[khi] : text.size()) - ls[klo]) : 0;
    std::vector<char>& A = arena[tid];
    A.resize(span + 64 * (khi - klo) + 64);
    char* ap = A.data();
    std::string t;
    for (long k = (long)klo; k < (long)khi; k++) {
        const char* b = text.data() + ls[(size_t)k];
        const char* e = (size_t)k + 1 < nl ? text.data() + ls[(size_t)k + 1] : text.data() + text.size();
        const char* le = e;                                     // the line without its '\n' (line.strip('\n') strips all of them)
        while (le > b && le[-1] == '\n') le--;
        const char *fb[9], *fe[9];
        const int nf = split_ws(b, le, fb, fe, 9);
        if (nf != 8) die("AssertionError: len(sfo_line) == 8");
        Rec& r = recs[(size_t)k];
        long sa, sb, oha, ohb, ola, olb;
        if (!parse_long(fb[0], fe[0], sa) || !parse_long(fb[1], fe[1], sb)) die("ValueError: invalid literal for int()");
        const long na = original_id(sa, ns, np), nb = original_id(sb, ns, np);
        const bool flip = na > nb;
        // the fields 3..6 are only read as numbers in the second pass (int(sfo_line[5..8])) and by flip_N
        if (!parse_long(fb[3], fe[3], oha) || !parse_long(fb[4], fe[4], ohb) || !parse_long(fb[5], fe[5], ola) || !parse_long(fb[6], fe[6], olb))
            die("ValueError: invalid literal for int()");
        const std::string ori(fb[2], fe[2]), K(fb[7], fe[7]);
        t.clear();
        if (flip) {
            long foha = oha, fohb = ohb;
            if (ori == "I") { foha = ohb; fohb = oha; }          // flip_I swaps the overhangs, flip_N negates them
            else { foha = -oha; fohb = -ohb; }
            put_long(t, nb); t += '\t'; put_long(t, na); t += '\t';
            t.append(fb[1], fe[1]); t += '\t'; t.append(fb[0], fe[0]); t += '\t'; t += ori; t += '\t';
            if (ori == "I") { t.append(fb[4], fe[4]); t += '\t'; t.append(fb[3], fe[3]); }   // strings as they are
            else { put_long(t, foha); t += '\t'; put_long(t, fohb); }                        // str(-1 * int(..))
            t += '\t'; t.append(fb[6], fe[6]); t += '\t'; t.append(fb[5], fe[5]); t += '\t'; t += K;
            r.idA = nb; r.idB = na; r.sfoA = sb; r.sfoB = sa; r.OHA = foha; r.OHB = fohb; r.OLA = olb; r.OLB = ola;
        } else {
            put_long(t, na); t += '\t'; put_long(t, nb); t += '\t'; t.append(b, le);      // the original line as it is
            r.idA = na; r.idB = nb; r.sfoA = sa; r.sfoB = sb; r.OHA = oha; r.OHB = ohb; r.OLA = ola; r.OLB = olb;
        }
        r.ori = ori.size() == 1 ? ori[0] : '?';
        if ((size_t)(ap - A.data()) + t.size() > A.size()) die("internal: line arena too small");
        std::memcpy(ap, t.data(), t.size());
        r.text = ap; r.text_len = (uint32_t)t.size();
        ap += t.size();
    }
    }
    std::string().swap(text);
    mark("parse + flip");
    // ---- 2. sort | uniq
    parallel_sort(recs);
    mark("sort");
    {
        size_t w = 0;
        for (size_t k = 0; k < recs.size(); k++)
            if (k == 0 || text_cmp(recs[k], recs[w - 1]) != 0) { if (w != k) recs[w] = recs[k]; w++; }
        recs.resize(w);
    }
    const size_t n = recs.size();
    mark("uniq");
    // ---- 3. the pass: classes of the lines, groups of the lines that involve a paired-end read
    std::vector<unsigned char> kind(n, 0);                      // 0 self-overlap (skipped), 1 single-single, 2 paired involved
#pragma omp parallel for schedule(static)
    for (long k = 0; k < (long)n; k++) {
        const Rec& r = recs[(size_t)k];
        if (r.idA == r.idB) continue;
        const bool pa = is_paired(r.idA, ns, np), pb = is_paired(r.idB, ns, np);
        kind[(size_t)k] = (!pa && !pb) ? 1 : 2;
    }
    // groups: consecutive paired-involved lines (lines of other kinds in between do not end a group) with equal (idA, idB)
    struct Group { size_t first_line, next_first_line; std::vector<size_t> lines; };
    std::vector<Group> groups;
    for (size_t k = 0; k < n; k++) {
        if (kind[k] != 2) continue;
        if (groups.empty() || recs[groups.back().lines[0]].idA != recs[k].idA || recs[groups.back().lines[0]].idB != recs[k].idB) {
            if (!groups.empty()) {
                const Rec& p = recs[groups.back().lines[0]];
                if (!(recs[k].idA >= p.idA) || (recs[k].idA == p.idA && !(recs[k].idB >= p.idB))) die("AssertionError: idA >= int(candidates_ids[0])");
                groups.back().next_first_line = k;
            }
            Group g;
            g.first_line = k; g.next_first_line = (size_t)-1;
            groups.push_back(g);
        }
        groups.back().lines.push_back(k);
    }
    mark("kinds + groups");
    std::vector<std::string> line_out(n), group_out(groups.size());
    long s_s_count = 0, p_count = 0;
#pragma omp parallel for schedule(dynamic, 4096) reduction(+ : s_s_count)
    for (long k = 0; k < (long)n; k++) {
        if (kind[(size_t)k] != 1) continue;
        put_ss_line(line_out[(size_t)k], s_s_overlap(recs[(size_t)k]));
        s_s_count++;
    }
#pragma omp parallel for schedule(dynamic, 256) reduction(+ : p_count)
    for (long g = 0; g < (long)groups.size(); g++) {
        const Group& G = groups[(size_t)g];
        if (G.next_first_line == (size_t)-1 || G.lines.size() < 2) continue;     // the last group is never matched (:84-93 run on a change of ids only)
        // (the script hands match_candidates the paired flags of the line that ENDS the group, i.e. of the next id pair, :84)
        const Rec& f = recs[G.next_first_line];
        const bool ta = is_paired(f.idA, ns, np), tb = is_paired(f.idB, ns, np);
        std::string& b = group_out[(size_t)g];
        for (size_t i = 0; i < G.lines.size(); i++)
            for (size_t j = i + 1; j < G.lines.size(); j++) {
                const size_t before = b.size();
                paired_overlap(b, recs[G.lines[i]], recs[G.lines[j]], ta, tb);
                if (b.size() != before) p_count++;
            }
    }
    mark("overlaps");
    // ---- 4. stitch in the script's order (a group's lines come out when the next group's first line is read), uniq
    FILE* fo = std::fopen(out.c_str(), "w");
    if (!fo) die("IOError: cannot write " + out);
    std::string prev, buf;
    auto emit = [&](const std::string& chunk) {                 // chunk = zero or more complete lines
        size_t p = 0;
        while (p < chunk.size()) {
            const size_t q = chunk.find('\n', p);
            const size_t len = q - p + 1;
            if (prev.size() != len || chunk.compare(p, len, prev) != 0) { buf.append(chunk, p, len); prev.assign(chunk, p, len); }
            p = q + 1;
        }
        if (buf.size() > (4u << 20)) { std::fwrite(buf.data(), 1, buf.size(), fo); buf.clear(); }
    };
    size_t gi = 0;                                              // next group whose output is pending
    for (size_t k = 0; k < n; k++) {
        while (gi < groups.size() && groups[gi].next_first_line == k) { emit(group_out[gi]); gi++; }
        if (kind[k] == 1) emit(line_out[k]);
    }
    std::fwrite(buf.data(), 1, buf.size(), fo);
    std::fclose(fo);
    mark("stitch + write");
    std::printf("total overlap count: %ld\nof which single-single: %ld\n", s_s_count + p_count, s_s_count);
    return 0;
}
