// hc_sam2overlaps -- scripts/sam2overlaps.py of the reference in C++ on all host threads: the overlaps file of the
// reference-guided mode, derived from the alignments of the reads to a reference genome (single-end SAM and / or interleaved
// paired-end SAM).  Same flags, same output BYTES as the script.
//
// The script sorts the alignments of one reference sequence by position, sweeps over them with a list of "active" reads
// (those that still reach the current position by at least min_overlap_len bases, judged on the uncorrected coordinates),
// corrects every (active read, current read) overlap for the indels of both CIGAR strings (compute_overlap_pos :281-330) and
// writes single / paired overlap lines (get_overlaps :372-470).  The active list depends on positions only and positions are
// sorted, so "read j is active when read i arrives" is  i == j + 1  or  len_j - (POS_{i-1} - POS_j) >= min_overlap_len :
// every read i finds its partners by itself and all reads are processed in parallel, the lines stitched in the script's order.
// SURVEY 8f rank 2 (the converter half).  Reference: scripts/sam2overlaps.py.
// --gpu=true: the same bytes and stdout from one hc_sam2overlaps call (include/hc_b200.h; pairing, sort and sweep on the
// device; the FASTA is read here as without the flag).  Input the device path does not take (a line this program dies
// on, or one outside the device's ranges) or a working set that does not fit the device is said on stderr and
// converted here as without the flag; no usable device is an error.
#include <omp.h>

#include "../../include/hc_b200.h"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iterator>
#include <map>
#include <string>
#include <vector>

namespace {

[[noreturn]] void die(const std::string& m) {
    std::fprintf(stderr, "%s\n", m.c_str());
    std::exit(1);
}

struct Aln {                      // what the script keeps of a SAM line and uses: [ID, FLAG, REF, cpos, ., CIGAR, ., ., ., cseq, .]
    std::string id, ref, cigar;
    long flag = 0, pos = 0, len = 0;             // pos = clipping-corrected POS, len = len(cseq)
};
struct Rec {                      // a single-end read, or the two ends of a pair in reference order + "reverse complement"
    Aln a, b;
    bool paired = false, rc = false;
    long pos() const { return a.pos; }
};

long to_long(const std::string& s) {              // Python int()
    if (s.empty()) die("ValueError: invalid literal for int() with base 10: ''");
    size_t i = 0;
    bool neg = false;
    if (s[0] == '+' || s[0] == '-') { neg = s[0] == '-'; i = 1; }
    if (i == s.size()) die("ValueError: invalid literal for int() with base 10: '" + s + "'");
    long v = 0;
    for (; i < s.size(); i++) {
        if (s[i] < '0' || s[i] > '9') die("ValueError: invalid literal for int() with base 10: '" + s + "'");
        v = v * 10 + (s[i] - '0');
    }
    return neg ? -v : v;
}

// ["".join(x) for _, x in itertools.groupby(CIGAR, key=str.isdigit)]: alternating runs of digits and of other characters
std::vector<std::string> cigar_runs(const std::string& c) {
    std::vector<std::string> r;
    for (size_t i = 0; i < c.size();) {
        const bool d = c[i] >= '0' && c[i] <= '9';
        size_t j = i;
        while (j < c.size() && ((c[j] >= '0' && c[j] <= '9') == d)) j++;
        r.push_back(c.substr(i, j - i));
        i = j;
    }
    return r;
}

// one SAM line -> Aln (read_sam_to_list / read_paired_sam_to_list :139-183, :197-226); false if the read is unmapped
bool parse_aln(const std::string& line, Aln& a) {
    std::vector<std::string> f;
    size_t p = 0;
    while (f.size() < 11) {
        const size_t q = line.find('\t', p);
        if (q == std::string::npos) { f.push_back(line.substr(p)); break; }
        f.push_back(line.substr(p, q - p));
        p = q + 1;
    }
    if (f.size() < 11) die("ValueError: need more than " + std::to_string(f.size()) + " values to unpack");
    a.flag = to_long(f[1]);
    if (a.flag & 4) return false;
    a.id = f[0]; a.ref = f[2]; a.cigar = f[5];
    const long POS = to_long(f[3]);
    to_long(f[4]); to_long(f[7]); to_long(f[8]);      // int(MAPQ), int(PNEXT), int(TLEN): only their validity matters
    const std::vector<std::string> c = cigar_runs(f[5]);
    if (c.size() < 2) die("IndexError: list index out of range");
    long len = (long)f[9].size();
    if (c[1] == "S") a.pos = POS - to_long(c[0]);
    else if (c[1] == "H") { a.pos = POS - to_long(c[0]); len += to_long(c[0]); }
    else a.pos = POS;
    if (c.back() == "H") len += to_long(c[c.size() - 2]);
    a.len = len;
    return true;
}

struct Ov { long pos, len; };

// compute_overlap_pos :281-330 (read #2 is in front)
Ov overlap_pos(long pos1, long pos2, long len1, long len2, const std::string& C1, const std::string& C2) {
    const std::vector<std::string> c1 = cigar_runs(C1), c2 = cigar_runs(C2);
    if (c1.size() % 2 || c2.size() % 2) die("IndexError: list index out of range");
    long total_back = 0;
    for (size_t j = 0; j < c1.size(); j += 2) if (c1[j + 1] != "I") total_back += to_long(c1[j]);
    const long max_len = pos1 - pos2 + total_back;
    long front_seq = 0, front_ref = 0, p = 0;
    for (size_t i = 0; i < c2.size(); i += 2) {
        const std::string& t = c2[i + 1];
        const long n = to_long(c2[i]);
        if (p < max_len) {
            if (t != "D") front_seq += std::min(n, max_len - p);
            if (t != "I") { front_ref += std::min(n, max_len - p); p += n; }
        }
    }
    Ov o;
    if (front_ref <= pos1 - pos2) { o.pos = -1; o.len = 0; }
    else {
        const long back_ref = front_ref - (pos1 - pos2);
        long back_seq = 0;
        p = 0;
        for (size_t i = 0; i < c1.size(); i += 2) {
            const std::string& t = c1[i + 1];
            const long n = to_long(c1[i]);
            if (!(n > 0)) die("AssertionError: aln_len > 0");
            if (p < back_ref) {
                if (t != "D") back_seq += std::min(n, back_ref - p);
                if (t != "I") p += n;
            }
        }
        o.pos = (pos1 - pos2) - ((front_ref - front_seq) - (back_ref - back_seq));
        if (o.pos >= 0) o.len = std::min(len2 - o.pos, len1);
        else { o.pos = -1; o.len = 0; }
    }
    return o;
}

struct Line {                    // the thirteen fields of an overlap line, as far as they vary
    const std::string *id1, *id2;
    long pos1, pos2 = 0, perc1, perc2 = 0, len1, len2 = 0;
    char ord = '-', ori1 = '+', ori2 = '+', t1 = 's', t2 = 's';
};

// get_overlap_line :332-366
Line overlap_line(const Aln& r1, const Aln& r2, long pos, long ovlen) {
    Line l;
    l.id1 = &r1.id; l.id2 = &r2.id; l.pos1 = pos; l.len1 = ovlen;
    const long m = std::min(r1.len, r2.len);
    if (m == 0) die("ZeroDivisionError: float division by zero");
    l.perc1 = (long)std::round((double)ovlen / (double)m * 100.0);         // int(round(ovlen / min(..) * 100)), Python 2 round
    if (!(l.perc1 >= 0)) die("AssertionError: perc >= 0");
    if (!(l.perc1 <= 100)) die("AssertionError: perc <= 100");
    return l;
}

// merge_overlaps :368-388
Line merge(Line o1, const Line& o2, char t1, char t2) {
    o1.t1 = t1; o1.t2 = t2;
    if (t1 == 'p' && t2 == 'p') {
        if (*o1.id1 != *o2.id1) {
            if (*o1.id1 != *o2.id2) die("AssertionError: overlap1[0] == overlap2[1]");
            o1.ord = '2';
        } else {
            o1.ord = '1';
        }
    }
    o1.pos2 = o2.pos1; o1.perc2 = o2.perc1; o1.len2 = o2.len1;
    return o1;
}

void put(std::string& b, long v) { char t[24]; b.append(t, (size_t)std::snprintf(t, sizeof(t), "%ld", v)); }

void put_line(std::string& b, const Line& l) {
    b += *l.id1; b += '\t'; b += *l.id2; b += '\t'; put(b, l.pos1); b += '\t'; put(b, l.pos2); b += '\t'; b += l.ord; b += '\t';
    b += l.ori1; b += '\t'; b += l.ori2; b += '\t'; put(b, l.perc1); b += '\t'; put(b, l.perc2); b += '\t'; put(b, l.len1); b += '\t';
    put(b, l.len2); b += '\t'; b += l.t1; b += '\t'; b += l.t2; b += '\n';
}

// one (active read, current record) pair of get_overlaps :384-468; appends at most one line
void pair_overlap(std::string& out, const Rec& read, const Rec& record, long min_ov, long& problems, std::string& warn) {
    const Aln &R = read.a, &C = record.a;
    if (!(C.pos - R.pos >= 0)) die("AssertionError: overlap_pos >= 0");
    const Ov o = overlap_pos(C.pos, R.pos, C.len, R.len, C.cigar, R.cigar);
    if (o.len > std::min(C.len, R.len)) { char t[96]; std::snprintf(t, sizeof(t), "%ld %ld %ld\n", o.len, C.len, R.len); warn += t; }
    if (o.len <= min_ov || o.pos < 0) return;
    auto ori_flag = [](const Aln& a) { return (a.flag & 16) ? '-' : '+'; };
    auto checked = [&](long p1, long p2, const Aln& x, const Aln& y) {       // compute_overlap_pos with its diagnostic print
        const Ov v = overlap_pos(p1, p2, x.len, y.len, x.cigar, y.cigar);
        if (v.len > std::min(x.len, y.len)) { char t[96]; std::snprintf(t, sizeof(t), "%ld %ld %ld\n", v.len, x.len, y.len); warn += t; }
        return v;
    };
    if (!record.paired && !read.paired) {
        Line l = overlap_line(R, C, o.pos, o.len);
        l.ori1 = ori_flag(R); l.ori2 = ori_flag(C);
        put_line(out, l);
    } else if (record.paired && !read.paired) {
        const Line o1 = overlap_line(R, record.a, o.pos, o.len);
        const Ov v = checked(record.b.pos, R.pos, record.b, R);
        const Line o2 = overlap_line(R, record.b, v.pos, v.len);
        Line l = merge(o1, o2, 's', 'p');
        l.ori1 = ori_flag(R); l.ori2 = record.rc ? '-' : '+';
        if (v.len > min_ov && v.pos >= 0) put_line(out, l);
    } else if (!record.paired && read.paired) {
        const Line o1 = overlap_line(read.a, C, o.pos, o.len);
        if (read.b.pos - C.pos < 0) { problems++; return; }
        const Ov v = checked(read.b.pos, C.pos, read.b, C);
        const Line o2 = overlap_line(C, read.b, v.pos, v.len);
        Line l = merge(o1, o2, 's', 'p');
        l.ori1 = read.rc ? '-' : '+'; l.ori2 = ori_flag(C);
        if (v.len > min_ov && v.pos >= 0) put_line(out, l);
    } else {
        const Line o1 = overlap_line(read.a, record.a, o.pos, o.len);
        Ov v;
        Line o2;
        if (record.b.pos - read.b.pos < 0) {
            v = checked(read.b.pos, record.b.pos, read.b, record.b);
            o2 = overlap_line(record.b, read.b, v.pos, v.len);
        } else {
            v = checked(record.b.pos, read.b.pos, record.b, read.b);
            o2 = overlap_line(read.b, record.b, v.pos, v.len);
        }
        Line l = merge(o1, o2, 'p', 'p');
        l.ori1 = read.rc ? '-' : '+'; l.ori2 = record.rc ? '-' : '+';
        if (v.len > min_ov && v.pos >= 0) put_line(out, l);
    }
}

std::vector<std::string> read_lines(const std::string& path) {
    std::ifstream f(path.c_str());
    if (!f.is_open()) die("IOError: [Errno 2] No such file or directory: '" + path + "'");
    std::vector<std::string> v;
    std::string l;
    while (std::getline(f, l)) v.push_back(l);
    return v;
}

}  // namespace

int main(int argc, char** argv) {
    std::string sam_s, sam_p, ref_path, out;
    long min_ov = 0;
    bool verbose = false, gpu = false;
    for (int i = 1; i < argc; i++) {
        std::string a = argv[i], v;
        const size_t eq = a.find('=');
        if (a == "--verbose") { verbose = true; continue; }
        if (eq != std::string::npos) { v = a.substr(eq + 1); a = a.substr(0, eq); }
        else if (i + 1 < argc) v = argv[++i];
        if (a == "--sam_s") sam_s = v;
        else if (a == "--sam_p") sam_p = v;
        else if (a == "--ref") ref_path = v;
        else if (a == "--out") out = v;
        else if (a == "--min_overlap_len") min_ov = std::atol(v.c_str());
        else if (a == "--gpu") gpu = v == "true" || v == "1";
        else { std::fprintf(stderr, "unknown option %s\n", a.c_str()); return 2; }
    }
    if ((sam_s.empty() && sam_p.empty()) || out.empty() || ref_path.empty()) {
        std::fprintf(stderr, "usage: hc_sam2overlaps [--sam_s S.sam] [--sam_p P.sam] --ref REF.fasta --out OVERLAPS [--min_overlap_len N] [--verbose] [--gpu=true]\n");
        return 2;
    }
    std::remove(out.c_str());
    // ---- reference sequences: id -> index, length (:45-76)
    std::vector<long> ref_len;
    std::map<std::string, size_t> ref_idx;
    {
        const std::vector<std::string> lines = read_lines(ref_path);
        if (lines.empty()) { std::printf("empty reference fasta... exiting.\n"); return 1; }
        std::string id;
        long seq = 0;
        bool have_seq = false;
        for (const std::string& l : lines) {
            if (!l.empty() && l[0] == '>') {
                if (have_seq && !id.empty()) { ref_len.push_back(seq); ref_idx[id] = ref_len.size() - 1; seq = 0; have_seq = false; }
                size_t b = 0;
                while (b < l.size() && std::isspace((unsigned char)l[b])) b++;
                size_t e = b;
                while (e < l.size() && !std::isspace((unsigned char)l[e])) e++;
                id = l.substr(b, e - b).substr(1);
            } else {
                seq += (long)l.size();
                if (!l.empty()) have_seq = true;
            }
        }
        if (!have_seq) { std::printf("invalid fasta file... exiting\n"); return 1; }
        ref_len.push_back(seq);
        ref_idx[id] = ref_len.size() - 1;
    }
    if (gpu) {
        std::string text_s, text_p;
        auto slurp = [](const std::string& path, std::string& t) {
            std::ifstream f(path.c_str(), std::ios::binary);
            if (!f.is_open()) return false;
            t.assign(std::istreambuf_iterator<char>(f), std::istreambuf_iterator<char>());
            return true;
        };
        // a file that cannot be read is left to the host path, which says so as without the flag
        if ((sam_s.empty() || slurp(sam_s, text_s)) && (sam_p.empty() || slurp(sam_p, text_p))) {
            std::string names;
            std::vector<uint64_t> name_off(1, 0);
            std::vector<uint32_t> name_idx;
            for (const auto& e : ref_idx) {
                names += e.first;
                name_off.push_back(names.size());
                name_idx.push_back((uint32_t)e.second);
            }
            const uint32_t n_refs = (uint32_t)ref_len.size();
            std::vector<int64_t> rlen(ref_len.begin(), ref_len.end());
            std::vector<hc_sam_ref_stats> rs(n_refs);
            hc_sam_stats st;
            // the file is typically several times the SAM text (tens of lines per alignment); a larger one costs a
            // second call with the exact size
            uint64_t cap = 16 * (uint64_t)(text_s.size() + text_p.size()) + (1u << 20), n_out = 0;
            auto call = [&](char* buf) {
                return hc_sam2overlaps(text_s.data(), text_s.size(), text_p.data(), text_p.size(), names.data(), name_off.data(),
                                       name_idx.data(), (uint32_t)name_idx.size(), rlen.data(), n_refs, min_ov, buf, cap, &n_out,
                                       rs.data(), &st, 0);
            };
            char* buf = (char*)std::malloc(cap);
            if (!buf) die("hc_sam2overlaps: out of host memory");
            int rc = call(buf);
            if (rc == HC_ERR_CAPACITY) {
                std::free(buf);
                cap = n_out;
                buf = (char*)std::malloc(cap ? cap : 1);
                if (!buf) die("hc_sam2overlaps: out of host memory");
                rc = call(buf);
            }
            if (rc == HC_OK) {
                if (std::getenv("HC_TIMING"))
                    std::fprintf(stderr, "[hc_sam2overlaps]   copy in %.1f ms, device %.1f ms, copy out %.1f ms\n", st.h2d_ms, st.device_ms, st.d2h_ms);
                FILE* fo = std::fopen(out.c_str(), "w");
                if (!fo) die("IOError: cannot write " + out);
                if (std::fwrite(buf, 1, n_out, fo) != n_out || std::fclose(fo) != 0) die("IOError: cannot write " + out);
                std::free(buf);
                if (verbose && !sam_s.empty())
                    std::printf("Number of singles unmapped:  %lu\nNumber of singles reversed:  %lu\n", (unsigned long)st.unmapped_s,
                                (unsigned long)st.reverse_s);
                if (verbose && !sam_p.empty())
                    std::printf("Number of read ends discarded:  %lu\nNumber of read ends unmapped:  %lu\nNumber of reverse complements considered:  %lu\n",
                                (unsigned long)st.discarded, (unsigned long)st.unmapped_p, (unsigned long)st.reverse_p);
                for (uint32_t r = 0; r < n_refs && verbose; r++) {
                    const hc_sam_ref_stats& x = rs[r];
                    if (x.n_alignments == 0) continue;
                    std::printf("Total number of alignments:  %lu\n... of which singles:  %lu\n... of which paired:  %lu\n", (unsigned long)x.n_alignments,
                                (unsigned long)x.n_singles, (unsigned long)x.n_paired);
                    if (x.problems > 0) std::printf("# cases where overlap_pos2 < 0:  %lu\n", (unsigned long)x.problems);
                    std::printf("Total number of overlaps found:  %lu\n... of which ++:  %lu\n... of which +-:  %lu\n... of which -+:  %lu\n... of which --:  %lu\n",
                                (unsigned long)x.n_overlaps, (unsigned long)x.types[0], (unsigned long)x.types[1], (unsigned long)x.types[2],
                                (unsigned long)x.types[3]);
                }
                if (st.total_alns == 0) { std::printf("\n\nERROR: No reads could be aligned to reference. Exiting.\n"); return 1; }
                return 0;
            }
            std::free(buf);
            if (rc != HC_ERR_INPUT && rc != HC_ERR_NOMEM) die(hc_last_error());
            std::fprintf(stderr, "%s; converting on the host\n", hc_last_error());
        }
    }
    // ---- alignments (the header is skipped while lines start with '@'; parsing in parallel, pairing in file order)
    auto parse_file = [&](const std::string& path, std::vector<Aln>& alns, std::vector<char>& mapped) {
        const std::vector<std::string> lines = read_lines(path);
        size_t first = 0;
        while (first < lines.size() && !lines[first].empty() && lines[first][0] == '@') first++;
        const size_t n = lines.size() - first;
        alns.assign(n, Aln());
        mapped.assign(n, 0);
#pragma omp parallel for schedule(dynamic, 1024)
        for (long k = 0; k < (long)n; k++) mapped[(size_t)k] = parse_aln(lines[first + (size_t)k], alns[(size_t)k]) ? 1 : 0;
    };
    std::vector<std::vector<Rec>> per_ref_s(ref_len.size()), per_ref_p(ref_len.size());
    long unmapped_s = 0, reverse_s = 0, discarded = 0, unmapped_p = 0, reverse_p = 0;
    auto ref_of = [&](const std::string& r) -> size_t {
        const auto it = ref_idx.find(r);
        if (it == ref_idx.end()) die("KeyError: '" + r + "'");
        return it->second;
    };
    if (!sam_s.empty()) {
        std::vector<Aln> alns;
        std::vector<char> mapped;
        parse_file(sam_s, alns, mapped);
        for (size_t k = 0; k < alns.size(); k++) {
            if (!mapped[k]) { unmapped_s++; continue; }
            if (alns[k].flag & 16) reverse_s++;
            Rec r;
            r.a = alns[k];
            per_ref_s[ref_of(r.a.ref)].push_back(std::move(r));
        }
        if (verbose) std::printf("Number of singles unmapped:  %ld\nNumber of singles reversed:  %ld\n", unmapped_s, reverse_s);
    }
    if (!sam_p.empty()) {
        std::vector<Aln> alns;
        std::vector<char> mapped;
        parse_file(sam_p, alns, mapped);
        std::vector<Aln> pr;                                    // paired_read
        long i = 0;
        for (size_t k = 0; k < alns.size(); k++) {              // :227-257, with its counter i that unmapped and mismatched ends do not advance
            if (!mapped[k]) { unmapped_p++; continue; }
            pr.push_back(alns[k]);
            if (!(pr.size() <= 2)) die("AssertionError: len(paired_read) <= 2");
            if (i % 2 == 1) {
                if (pr.size() == 2) {
                    if (pr[0].id != pr[1].id) { pr.erase(pr.begin()); discarded++; continue; }
                    Rec r;
                    r.paired = true;
                    if (pr[0].pos >= pr[1].pos) {
                        if ((pr[0].flag & 16) && (pr[1].flag & 16)) { r.a = pr[1]; r.b = pr[0]; r.rc = true; reverse_p++; per_ref_p[ref_of(r.a.ref)].push_back(std::move(r)); }
                        else discarded++;
                    } else {
                        if (!(pr[0].flag & 16) && !(pr[1].flag & 16)) { r.a = pr[0]; r.b = pr[1]; r.rc = false; per_ref_p[ref_of(r.a.ref)].push_back(std::move(r)); }
                        else discarded++;
                    }
                } else {
                    discarded++;
                }
                pr.clear();
            }
            i++;
        }
        if (verbose) std::printf("Number of read ends discarded:  %ld\nNumber of read ends unmapped:  %ld\nNumber of reverse complements considered:  %ld\n", discarded, unmapped_p, reverse_p);
    }
    // ---- per reference sequence: sort, merge, sweep (:472-548)
    FILE* fo = std::fopen(out.c_str(), "a");
    if (!fo) die("IOError: cannot write " + out);
    long total_alns = 0;
    for (size_t ri = 0; ri < ref_len.size(); ri++) {
        std::vector<Rec>& S = per_ref_s[ri];
        std::vector<Rec>& P = per_ref_p[ri];
        total_alns += (long)(S.size() + P.size());
        if (S.empty() && P.empty()) continue;
        auto by_pos = [](const Rec& x, const Rec& y) { return x.pos() < y.pos(); };
        std::stable_sort(S.begin(), S.end(), by_pos);
        std::stable_sort(P.begin(), P.end(), by_pos);
        std::vector<const Rec*> M;                               // merged_records: singles first where positions tie
        M.reserve(S.size() + P.size());
        size_t k1 = 0, k2 = 0;
        while (k1 < S.size() && k2 < P.size()) { if (S[k1].pos() <= P[k2].pos()) M.push_back(&S[k1++]); else M.push_back(&P[k2++]); }
        while (k1 < S.size()) M.push_back(&S[k1++]);
        while (k2 < P.size()) M.push_back(&P[k2++]);
        const size_t n = M.size();
        if (verbose) std::printf("Total number of alignments:  %zu\n... of which singles:  %zu\n... of which paired:  %zu\n", n, S.size(), P.size());
        // records processed: the loop runs while the position of the PREVIOUS record (the first one's for i = 0) is inside the reference
        size_t n_proc = 0;
        { long cur = M[0]->pos(); while (n_proc < n && cur < ref_len[ri]) { cur = M[n_proc]->pos(); n_proc++; } }
        long max_len = 0;
        for (size_t k = 0; k < n_proc; k++) max_len = std::max(max_len, M[k]->a.len);
        std::vector<std::string> chunk(n_proc), warn(n_proc);
        long problems = 0;
#pragma omp parallel for schedule(dynamic, 64) reduction(+ : problems)
        for (long i = 0; i < (long)n_proc; i++) {
            if (i == 0) continue;
            const Rec& rec = *M[(size_t)i];
            const long prev_pos = M[(size_t)i - 1]->pos();
            // partners: j < i still active when i arrives; none can start before prev_pos - (max_len - min_ov)
            long j0 = i - 1;
            while (j0 > 0 && M[(size_t)j0 - 1]->pos() >= prev_pos - (max_len - min_ov)) j0--;
            for (long j = j0; j < i; j++) {
                const Rec& rd = *M[(size_t)j];
                if (j != i - 1 && !(rd.a.len - (prev_pos - rd.pos()) >= min_ov)) continue;
                pair_overlap(chunk[(size_t)i], rd, rec, min_ov, problems, warn[(size_t)i]);
            }
        }
        long count = 0, types[4] = {0, 0, 0, 0};
        for (size_t i = 0; i < n_proc; i++) {
            if (!warn[i].empty()) std::fputs(warn[i].c_str(), stdout);
            const std::string& c = chunk[i];
            if (c.empty()) continue;
            std::fwrite(c.data(), 1, c.size(), fo);
            if (verbose) {
                size_t p = 0;
                while (p < c.size()) {
                    const size_t q = c.find('\n', p);
                    int tab = 0;
                    size_t t = p;
                    for (; tab < 5; t++) if (c[t] == '\t') tab++;
                    const char o1 = c[t], o2 = c[t + 2];
                    types[(o1 == '-') * 2 + (o2 == '-')]++;
                    count++;
                    p = q + 1;
                }
            }
        }
        if (problems > 0 && verbose) std::printf("# cases where overlap_pos2 < 0:  %ld\n", problems);
        if (verbose) std::printf("Total number of overlaps found:  %ld\n... of which ++:  %ld\n... of which +-:  %ld\n... of which -+:  %ld\n... of which --:  %ld\n", count, types[0], types[1], types[2], types[3]);
    }
    std::fclose(fo);
    if (total_alns == 0) { std::printf("\n\nERROR: No reads could be aligned to reference. Exiting.\n"); return 1; }
    return 0;
}
