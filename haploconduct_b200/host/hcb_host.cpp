// hcb_host.cpp -- see hcb_host.h.  Host plumbing around the C ABI: FASTQ / overlaps-file parsing,
// id -> index mapping, the ordered graph insert.  No score is computed here.
#include "hcb_host.h"
#include <omp.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <fstream>
#include <iostream>
#include <sstream>
#include <thread>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

namespace hcb {

static double wall_s() {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec + 1e-9 * ts.tv_nsec;
}

void die(const std::string& msg) {
    std::cerr << msg;
    if (msg.empty() || msg.back() != '\n') std::cerr << std::endl;
    std::exit(1);
}

static read_id_t str_to_read_id(const std::string& s) { return strtoul(s.c_str(), NULL, 0); }   // src/Types.h:99-102

// ---------------------------------------------------------------------------------------------- reads
static void slurp_lines(const std::string& path, unsigned long max_reads, std::vector<std::string>& out) {
    std::ifstream f(path.c_str());
    if (!f.is_open()) die("Unable to open fastq file " + path);                   // src/FastqStorage.cpp:54-56
    std::string line;
    unsigned long count = 0;
    while (count < 4 * max_reads && getline(f, line)) { out.push_back(line); count++; }
}

static std::string first_token(const std::string& s) {
    std::stringstream st(s);
    std::string t;
    st >> t;
    return t;
}

void FastqStorage::read_new_ids(const std::string& path) {                        // src/FastqStorage.cpp:60-90
    std::ifstream f(path.c_str());
    if (!f.is_open()) die("Unable to open read-to-overlapID file");
    std::string line;
    while (getline(f, line)) {
        std::stringstream ss(line);
        std::string new_id, old_id;
        getline(ss, new_id, '\t');
        getline(ss, old_id, '\t');
        if (!old_id.empty() && old_id[0] == '>') old_id = old_id.substr(1);
        new_ids_.insert(std::make_pair(old_id, new_id));
    }
    have_new_ids_ = true;
}

void FastqStorage::read_singles(const std::string& path, unsigned long max_reads) {   // src/FastqStorage.cpp:92-152
    std::vector<std::string> lines;
    slurp_lines(path, max_reads, lines);
    Read cur;
    for (size_t k = 0; k < lines.size(); k++) {
        const std::string& l = lines[k];
        switch (k % 4) {
            case 0: {
                if (l.empty() || l[0] != '@') die("Read ID does not start with @. Exiting read_singles.");
                const std::string tok = first_token(l.substr(1));
                cur = Read();
                cur.read_id = have_new_ids_ ? str_to_read_id(new_ids_.at(tok)) : str_to_read_id(tok);
                break;
            }
            case 1:
                cur.seq1 = l;
                for (size_t i = 0; i < cur.seq1.size(); i++) cur.seq1[i] = (char)toupper((unsigned char)cur.seq1[i]);   // :123
                break;
            case 3:
                cur.phred1 = l;
                if (cur.seq1.empty()) die("single read with ID " + std::to_string(cur.read_id) + " has an empty sequence... exiting.");
                cur.is_paired = false;
                m_read_vec.push_back(cur);
                break;
            default: break;
        }
    }
}

void FastqStorage::read_pairs(const std::string& p1, const std::string& p2, unsigned long max_reads) {   // :154-235
    std::vector<std::string> l1, l2;
    slurp_lines(p1, max_reads, l1);
    slurp_lines(p2, max_reads, l2);
    Read cur;
    const size_t n = std::min(l1.size(), l2.size());
    for (size_t k = 0; k < n; k++) {
        switch (k % 4) {
            case 0: {
                if (l1[k].empty() || l1[k][0] != '@') die("Read ID does not start with @. Exiting read_pairs.");
                const std::string t1 = first_token(l1[k].substr(1));
                const std::string t2 = l2[k].empty() ? std::string() : first_token(l2[k].substr(1));
                if (t1 != t2) die("Fastq files /1 /2 are not ordered identically. Exiting read_pairs.");
                cur = Read();
                cur.read_id = have_new_ids_ ? str_to_read_id(new_ids_.at(t1)) : str_to_read_id(t1);
                break;
            }
            case 1:
                cur.seq1 = l1[k];   // pairs are NOT upper-cased by the reference (:196-197)
                cur.seq2 = l2[k];
                break;
            case 3:
                cur.phred1 = l1[k];
                cur.phred2 = l2[k];
                if (cur.seq1.empty() || cur.seq2.empty())
                    die("paired read with ID " + std::to_string(cur.read_id) + " has an empty sequence... exiting.");
                cur.is_paired = true;
                m_read_vec.push_back(cur);
                break;
            default: break;
        }
    }
}

FileBuf& FileBuf::operator=(FileBuf&& o) noexcept {
    if (this != &o) {
        if (data) munmap(data, mapped);
        data = o.data; size = o.size; mapped = o.mapped;
        o.data = nullptr; o.size = o.mapped = 0;
    }
    return *this;
}
FileBuf::~FileBuf() { if (data) munmap(data, mapped); }

bool read_whole_file(const std::string& path, FileBuf& out, int threads) {
    out = FileBuf();
    const int fd = open(path.c_str(), O_RDONLY);
    if (fd < 0) return false;
    struct stat st;
    if (fstat(fd, &st) != 0 || st.st_size <= 0) { close(fd); return true; }      // empty (or not a regular file): no bytes
    const size_t size = (size_t)st.st_size, mapped = (size + (2u << 20)) & ~((size_t)(2u << 20) - 1);
    void* p = mmap(nullptr, mapped, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
    if (p == MAP_FAILED) { close(fd); die("out of memory reading " + path); }
    madvise(p, mapped, MADV_HUGEPAGE);
    out.data = static_cast<char*>(p); out.mapped = mapped;
    const size_t blk = 8u << 20;
    const long long nb = (long long)((size + blk - 1) / blk);
    int T = threads > 0 ? threads : omp_get_max_threads();
    if (T > 16) T = 16;
    size_t got_min = size;
#pragma omp parallel for schedule(dynamic, 1) num_threads(T) reduction(min : got_min)
    for (long long b = 0; b < nb; b++) {
        size_t o = (size_t)b * blk;
        const size_t end = std::min(size, o + blk);
        while (o < end) {
            const ssize_t r = pread(fd, out.data + o, end - o, (off_t)o);
            if (r <= 0) { got_min = std::min(got_min, o); break; }               // shorter than fstat said: keep what is there
            o += (size_t)r;
        }
    }
    close(fd);
    out.size = got_min;
    return true;
}

std::function<void()> FastqStorage::device_ready_hook;

FastqStorage::FastqStorage(const ProgramSettings& ps) {                           // src/FastqStorage.h:58-98
    if (ps.gpu_fastq) {
        // --IDs: the table maps the header token (a string) to the id; the device scan reads ids as numbers, so the tokens are
        // taken from the headers by the host (every fourth line of the singles file and of the first paired file, like
        // :113-121,:186-195) and the ids of the store's reads replaced below
        std::vector<std::string> header_tokens;
        if (!ps.id_correspondence.empty()) {
            read_new_ids(ps.id_correspondence);
            for (const std::string* path : {&ps.singles_file, &ps.paired1_file}) {
                if (path->empty() || *path == "None") continue;
                FileBuf fb;
                if (!read_whole_file(*path, fb)) die("Unable to open fastq file " + *path);
                size_t line = 0, b = 0;
                const size_t max_lines = ps.max_reads > (~0ul) / 4 ? ~0ul : 4 * ps.max_reads;
                std::vector<std::string> toks;
                while (b < fb.size && line < max_lines) {
                    const void* nl = memchr(fb.data + b, '\n', fb.size - b);
                    const size_t e = nl ? (size_t)((const char*)nl - fb.data) : fb.size;
                    if (line % 4 == 0) toks.push_back(first_token(std::string(fb.data + b + (e > b ? 1 : 0), fb.data + e)));
                    line++;
                    b = e + 1;
                }
                toks.resize(line / 4);                          // complete records only
                header_tokens.insert(header_tokens.end(), toks.begin(), toks.end());
            }
        }
        // the files are streamed to the device by the library (pinned ring, several reading threads): no host copy of them
        const double tfr = wall_s();
        t_read_s = 0;
        if (hc_warm_up(ps.first_device) != HC_OK) die(std::string("hc_warm_up: ") + hc_last_error());
        if (device_ready_hook) device_ready_hook();      // e.g. start reading the overlaps file: from here on nothing maps memory at CUDA's pace
        const double tf1 = wall_s();
        t_cuda_init_s = tf1 - tfr;
        first_device_ = ps.first_device;
        store_ = hc_store_create_fastq_files(ps.singles_file.c_str(), ps.paired1_file.c_str(), ps.paired2_file.c_str(), ps.max_reads,
                                             ps.first_device, ps.n_devices);
        if (!store_) die(hc_last_error());                // "Unable to open fastq file ...", src/FastqStorage.cpp:54-56, or what is wrong with a record
        const double tf2 = wall_s();
        t_store_s = tf2 - tf1;
        const uint64_t n = hc_store_n_reads(store_);
        std::vector<uint64_t> ids(n);
        std::vector<uint32_t> lens(2 * n);
        if (hc_store_read_ids(store_, ids.data(), lens.data()) != HC_OK) die(hc_last_error());
        if (have_new_ids_) {
            if (header_tokens.size() < n) die("--IDs: fewer FASTQ headers than reads in the store");
            for (uint64_t i = 0; i < n; i++) {
                const auto it = new_ids_.find(header_tokens[i]);
                if (it == new_ids_.end()) die("read name " + header_tokens[i] + " is not in the read-to-overlapID file");   // std::map::at throws in the reference
                ids[i] = str_to_read_id(it->second);
            }
        }
        m_readcount_single = (unsigned int)hc_store_n_single(store_);
        m_readcount_paired = (unsigned int)(n - m_readcount_single);
        m_read_vec.resize(n);
        mate_len = lens;
        read_ids = ids;
        for (uint64_t i = 0; i < n; i++) {
            m_read_vec[i].read_id = ids[i];
            m_read_vec[i].is_paired = i >= m_readcount_single;
            max_read_len = std::max(max_read_len, std::max(lens[2 * i], lens[2 * i + 1]));
            // with the overlaps file parsed on the device too, nothing on the host looks an id up (the device map does)
            if (!ps.gpu_parse) m_ID_to_index.insert(std::make_pair((read_id_t)ids[i], (unsigned int)i));
        }
        t_index_s = wall_s() - tf2;
        if (ps.verbose) {
            std::cout << "Singles: " << m_readcount_single << std::endl;
            std::cout << "Pairs: " << m_readcount_paired << std::endl;
        }
        return;
    }
    if (!ps.id_correspondence.empty()) read_new_ids(ps.id_correspondence);
    if (!ps.singles_file.empty() && ps.singles_file != "None") read_singles(ps.singles_file, ps.max_reads);
    m_readcount_single = (unsigned int)m_read_vec.size();
    if (!ps.paired1_file.empty() && ps.paired1_file != "None") read_pairs(ps.paired1_file, ps.paired2_file, ps.max_reads);
    m_readcount_paired = (unsigned int)m_read_vec.size() - m_readcount_single;
    if (ps.verbose) {
        std::cout << "Singles: " << m_readcount_single << std::endl;
        std::cout << "Pairs: " << m_readcount_paired << std::endl;
    }
    for (unsigned int i = 0; i < m_read_vec.size(); i++) m_ID_to_index.insert(std::make_pair(m_read_vec[i].read_id, i));
    read_ids.resize(m_read_vec.size());
    for (size_t i = 0; i < m_read_vec.size(); i++) read_ids[i] = m_read_vec[i].read_id;
    if (m_read_vec.empty()) return;
    // ---- device replica: concatenate, describe, hand to the C ABI
    std::vector<hc_read_desc> descs(m_read_vec.size());
    std::string bases, quals;
    size_t total = 0;
    for (auto& r : m_read_vec) total += r.seq1.size() + r.seq2.size();
    bases.reserve(total);
    quals.reserve(total);
    for (size_t i = 0; i < m_read_vec.size(); i++) {
        const Read& r = m_read_vec[i];
        if (r.seq1.size() != r.phred1.size() || r.seq2.size() != r.phred2.size())
            die("read with ID " + std::to_string(r.read_id) + ": sequence and quality lengths differ");   // string::at would throw, :93-94
        max_read_len = std::max(max_read_len, (unsigned int)std::max(r.seq1.size(), r.seq2.size()));
        mate_len.push_back((uint32_t)r.seq1.size());
        mate_len.push_back((uint32_t)r.seq2.size());
        descs[i].seq_off[0] = bases.size();
        descs[i].seq_len[0] = (uint32_t)r.seq1.size();
        bases += r.seq1;
        quals += r.phred1;
        descs[i].seq_off[1] = bases.size();
        descs[i].seq_len[1] = (uint32_t)r.seq2.size();
        bases += r.seq2;
        quals += r.phred2;
    }
    first_device_ = ps.first_device;
    store_ = hc_store_create(descs.data(), descs.size(), m_readcount_single, bases.data(), quals.data(), ps.first_device,
                             ps.n_devices);
    if (!store_) die(std::string("hc_store_create: ") + hc_last_error());
}

FastqStorage::~FastqStorage() {
    hc_idmap_destroy(idmap_);
    hc_store_destroy(store_);
}

hc_idmap* FastqStorage::device_idmap() {
    if (!idmap_) {
        std::vector<uint64_t> ids(m_read_vec.size());
        for (size_t i = 0; i < ids.size(); i++) ids[i] = m_read_vec[i].read_id;
        idmap_ = hc_idmap_create(ids.data(), ids.size(), first_device_);
        if (!idmap_) die(std::string("hc_idmap_create: ") + hc_last_error());
    }
    return idmap_;
}

// ---------------------------------------------------------------------------------------------- Overlap
static std::string strip(const std::string& s, const char* chars) {
    std::string r;
    for (char c : s) if (!strchr(chars, c)) r.push_back(c);
    return r;
}

Overlap Overlap::from_fields(const std::vector<std::string>& f) {                // src/Overlap.h:39-73
    Overlap o;
    o.id1 = str_to_read_id(f[0]);
    o.id2 = str_to_read_id(f[1]);
    o.pos1 = (unsigned int)atoi(f[2].c_str());
    o.pos2 = (unsigned int)atoi(f[3].c_str());
    o.perc1 = (unsigned int)atoi(f[7].c_str());
    o.perc2 = (unsigned int)atoi(f[8].c_str());
    o.len1 = (unsigned int)atoi(f[9].c_str());
    o.len2 = (unsigned int)atoi(f[10].c_str());
    if (f[3] == "-") { o.pos2 = 0; o.perc2 = 0; o.len2 = 0; }                      // :55-59
    if ((int)o.pos1 < 0 || (int)o.pos2 < 0) die("overlap.m_pos < 0; Exiting.");    // :107-112
    std::string ori1 = f[5].size() == 1 ? f[5] : strip(f[5], " "), ori2 = f[6].size() == 1 ? f[6] : strip(f[6], " ");
    if (ori1.size() != 1 || ori2.size() != 1 || (ori1 != "+" && ori1 != "-") || (ori2 != "+" && ori2 != "-"))
        die("overlap.m_ori not of the right format (+, -). Exiting.");              // :125-134
    for (unsigned int p : {o.perc1, o.perc2})
        if ((int)p < 0 || (int)p > 100) die(std::to_string((int)p) + "\noverlap.m_perc not of the right format (0 <= perc <= 100). Exiting.");
    if ((int)o.len1 < 0 || (int)o.len2 < 0) die("overlap.m_len < 0. Exiting.");    // :144-149
    std::string t1 = f[11].size() == 1 ? f[11] : strip(f[11], "\n\t "), t2 = f[12].size() == 1 ? f[12] : strip(f[12], "\n\t ");
    if (t1.size() != 1 || t2.size() != 1) die("overlap type field is not a single character (the reference asserts)");
    if (t1 != "s" && t1 != "p") die(t1 + " not of the form 's' or 'p'. Exiting.");
    if (t2 != "s" && t2 != "p") die(t2 + " not of the form 's' or 'p'. Exiting.");
    std::string ord = f[4].size() == 1 ? f[4] : strip(f[4], " ");
    bool ord_ok = ord.size() == 1 && (ord == "1" || ord == "2" || ord == "-");
    if (ord_ok) ord_ok = (t1 == "s" || t2 == "s") ? ord == "-" : (ord == "1" || ord == "2");   // :114-123
    if (!ord_ok) die("overlap ORD field inconsistent with the read types (the reference asserts, src/Overlap.h:114-123)");
    o.ord = ord[0];
    o.ori1 = ori1[0];
    o.ori2 = ori2[0];
    o.type1 = t1[0];
    o.type2 = t2[0];
    return o;
}

// Overlap::get_overlap_line appended to a buffer without the thirteen std::to_string temporaries
static inline void put_u64(std::string& b, unsigned long v) {
    char tmp[24];
    int k = 0;
    do { tmp[k++] = (char)('0' + v % 10); v /= 10; } while (v);
    while (k) b.push_back(tmp[--k]);
}

void Overlap::append_overlap_line(std::string& b) const {                         // src/Overlap.h:234-237
    put_u64(b, id1); b.push_back('\t'); put_u64(b, id2); b.push_back('\t'); put_u64(b, pos1); b.push_back('\t'); put_u64(b, pos2);
    b.push_back('\t'); b.push_back(ord); b.push_back('\t'); b.push_back(ori1); b.push_back('\t'); b.push_back(ori2); b.push_back('\t');
    put_u64(b, perc1); b.push_back('\t'); put_u64(b, perc2); b.push_back('\t'); put_u64(b, len1); b.push_back('\t'); put_u64(b, len2);
    b.push_back('\t'); b.push_back(type1); b.push_back('\t'); b.push_back(type2); b.push_back('\n');
}

std::string Overlap::get_overlap_line() const {                                   // src/Overlap.h:234-237
    std::string s = std::to_string(id1) + "\t" + std::to_string(id2) + "\t" + std::to_string(pos1) + "\t" +
                    std::to_string(pos2) + "\t";
    s.push_back(ord); s += "\t"; s.push_back(ori1); s += "\t"; s.push_back(ori2);
    s += "\t" + std::to_string(perc1) + "\t" + std::to_string(perc2) + "\t" + std::to_string(len1) + "\t" +
         std::to_string(len2) + "\t";
    s.push_back(type1); s += "\t"; s.push_back(type2); s += "\n";
    return s;
}

// ---------------------------------------------------------------------------------------------- Edge / graph
void Edge::swap_reads() {                                                         // src/Edge.h:74-88
    std::swap(vertex1, vertex2);
    std::swap(ori1, ori2);
    if (ord == '1') ord = '2';
    else if (ord == '2') ord = '1';
    pos3 = -pos3;
    pos4 = -pos4;
}

OverlapGraph::OverlapGraph(unsigned int V) : inclusions(V, 0), adj_out(V) {}

uint64_t OverlapGraph::key(node_id_t a, node_id_t b, bool same_ori) {
    const uint64_t lo = std::min(a, b), hi = std::max(a, b);
    return (lo << 33) | (hi << 1) | (same_ori ? 1u : 0u);
}

node_id_t OverlapGraph::addVertex(read_id_t id) {
    vertex_to_read.push_back(id);
    return vertex_to_read.size() - 1;
}

void OverlapGraph::addEdge(const Edge& e) {
    adj_out[e.vertex1].push_back(e);
    if (!owner_stale_) owner_[key(e.vertex1, e.vertex2, e.ori1 == e.ori2)] = e.vertex1;
    edge_count_++;
}

void OverlapGraph::addEdges(const std::vector<Edge>& es, const unsigned char* keep) {
    const size_t n = es.size(), V = adj_out.size();
    if (n < 4096) { for (size_t k = 0; k < n; k++) if (!keep || keep[k]) addEdge(es[k]); return; }
    // stable counting sort of the kept edges by vertex1 (input order inside a list = the order the reference appends in)
    std::vector<uint32_t> off(V + 1, 0);
    for (size_t k = 0; k < n; k++) if (!keep || keep[k]) off[es[k].vertex1 + 1]++;
    for (size_t v = 0; v < V; v++) off[v + 1] += off[v];
    const size_t kept = off[V];
    std::vector<uint32_t> order(kept), cur(off.begin(), off.end() - 1);
    for (size_t k = 0; k < n; k++) if (!keep || keep[k]) order[cur[es[k].vertex1]++] = (uint32_t)k;
#pragma omp parallel for schedule(dynamic, 4096)
    for (long long v = 0; v < (long long)V; v++) {
        const uint32_t a = off[v], b = off[v + 1];
        if (a == b) continue;
        std::vector<Edge>& lst = adj_out[(size_t)v];
        lst.reserve(lst.size() + (b - a));
        for (uint32_t j = a; j < b; j++) lst.push_back(es[order[j]]);
    }
    edge_count_ += (unsigned int)kept;
    owner_stale_ = true;
    owner_.clear();
}

void OverlapGraph::ensure_owner() const {
    if (!owner_stale_) return;
    owner_.clear();
    owner_.reserve(edge_count_ * 2u);
    for (const auto& lst : adj_out)
        for (const Edge& e : lst) owner_[key(e.vertex1, e.vertex2, e.ori1 == e.ori2)] = e.vertex1;
    owner_stale_ = false;
}

const Edge* OverlapGraph::getEdgeInfoWithOri(node_id_t v, node_id_t w, bool same_ori) const {
    ensure_owner();
    auto it = owner_.find(key(v, w, same_ori));
    if (it == owner_.end()) return nullptr;
    const node_id_t from = it->second, to = from == v ? w : v;
    for (const Edge& e : adj_out[from])
        if (e.vertex2 == to && (e.ori1 == e.ori2) == same_ori) return &e;
    return nullptr;
}

double OverlapGraph::checkEdgeWithOri(node_id_t v, node_id_t w, bool same_ori) const {
    const Edge* e = getEdgeInfoWithOri(v, w, same_ori);
    return e ? e->score : -1;
}

void OverlapGraph::removeEdgeWithOri(node_id_t v, node_id_t w, bool same_ori) {
    ensure_owner();
    std::vector<Edge>& lst = adj_out[v];
    for (size_t i = 0; i < lst.size(); i++) {
        if (lst[i].vertex2 == w && (lst[i].ori1 == lst[i].ori2) == same_ori) {
            lst.erase(lst.begin() + i);
            owner_.erase(key(v, w, same_ori));
            edge_count_--;
            return;
        }
    }
    die("Edge to be removed not found...\n" + std::to_string(v) + " " + std::to_string(w));
}

void OverlapGraph::sortEdges(const std::vector<uint32_t>& read_len, int device) {
    const size_t V = adj_out.size();
    auto nonoverlap = [&](const Edge& e) -> unsigned int {                       // Edge::get_nonoverlap_len, src/Edge.h:58-63
        return (unsigned int)read_len[e.vertex1] + (unsigned int)read_len[e.vertex2] - (unsigned int)(2 * e.overlap_len);
    };
    auto std_sort_list = [&](std::vector<Edge>& lst) {                           // :726-747, the reference's own call
        std::vector<std::pair<Edge, unsigned int>> pairs;
        pairs.reserve(lst.size());
        for (const Edge& e : lst) pairs.push_back(std::make_pair(e, nonoverlap(e)));
        std::sort(pairs.begin(), pairs.end(), [](const std::pair<Edge, unsigned int>& a, const std::pair<Edge, unsigned int>& b) {
            if (a.second == b.second) return a.first.vertex2 < b.first.vertex2;
            return a.second < b.second;
        });
        for (size_t k = 0; k < lst.size(); k++) lst[k] = pairs[k].first;
    };
    bool in_done = false;
    if (device >= 0 && edge_count_ > 0) {
        std::vector<uint64_t> start(V + 1, 0);
        for (size_t v = 0; v < V; v++) start[v + 1] = start[v] + adj_out[v].size();
        const size_t n = start[V];
        std::vector<hc_adj_edge> ae(n);
#pragma omp parallel for schedule(dynamic, 4096)
        for (long long v = 0; v < (long long)V; v++) {
            size_t k = start[(size_t)v];
            for (const Edge& e : adj_out[(size_t)v]) {
                ae[k].vertex1 = (uint32_t)e.vertex1; ae[k].vertex2 = (uint32_t)e.vertex2; ae[k].nonoverlap_len = nonoverlap(e); ae[k].reserved = 0;
                k++;
            }
        }
        std::vector<uint64_t> out_off(V + 1), in_off(V + 1);
        std::vector<uint32_t> perm(n ? n : 1), in_src(n ? n : 1);
        std::vector<uint8_t> ties(V ? V : 1);
        uint64_t kept = 0;
        const int rc = hc_build_adjacency(ae.data(), n, nullptr, V, 1, out_off.data(), perm.data(), in_off.data(), in_src.data(), ties.data(), &kept, device);
        if (rc != HC_OK) die(std::string("hc_build_adjacency: ") + hc_last_error());
        bool any_tie = false;
#pragma omp parallel for schedule(dynamic, 4096) reduction(|| : any_tie)
        for (long long v = 0; v < (long long)V; v++) {
            std::vector<Edge>& lst = adj_out[(size_t)v];
            if (lst.size() < 2) continue;
            if (ties[(size_t)v]) { std_sort_list(lst); any_tie = true; continue; }
            std::vector<Edge> sorted(lst.size());
            const size_t base = start[(size_t)v];                                 // out_off == start: every edge is kept
            for (size_t k = 0; k < lst.size(); k++) sorted[k] = lst[perm[base + k] - base];
            lst.swap(sorted);
        }
        if (!any_tie) {
            adj_in.assign(V, std::vector<node_id_t>());
#pragma omp parallel for schedule(dynamic, 4096)
            for (long long w = 0; w < (long long)V; w++) {
                std::vector<node_id_t>& in = adj_in[(size_t)w];
                in.reserve(in_off[(size_t)w + 1] - in_off[(size_t)w]);
                for (uint64_t k = in_off[(size_t)w]; k < in_off[(size_t)w + 1]; k++) in.push_back(in_src[k]);
            }
            in_done = true;
        }
    } else {
        for (auto& lst : adj_out) if (lst.size() > 1) std_sort_list(lst);
    }
    if (!in_done) {                                                               // :752-763
        adj_in.assign(V, std::vector<node_id_t>());
        for (const auto& lst : adj_out)
            for (const Edge& e : lst) adj_in[e.vertex2].push_back(e.vertex1);
    }
}

void OverlapGraph::writeDiGraphToFile(const std::string& path) const {
    std::ofstream f(path.c_str());
    for (size_t v = 0; v < adj_out.size(); v++)
        for (const Edge& e : adj_out[v]) f << v << "\t" << e.vertex2 << "\n";
}

void OverlapGraph::dumpAdjacency(const std::string& path, bool with_in) const {
    FILE* fo = fopen(path.c_str(), "w");
    if (!fo) die("cannot write " + path);
    fprintf(fo, "#v1\tv2\tscore\tmm_rate\tpos1\tpos2\tpos3\tpos4\tori1\tori2\tord\tperc\tlen1\tlen2\n");
    for (const auto& lst : adj_out)
        for (const Edge& e : lst)
            fprintf(fo, "%lu\t%lu\t%a\t%a\t%d\t%d\t%d\t%d\t%d\t%d\t%c\t%d\t%d\t%d\n", e.vertex1, e.vertex2, e.score,
                    e.mismatch_rate, e.pos1, e.pos2, e.pos3, e.pos4, (int)e.ori1, (int)e.ori2, e.ord, e.overlap_perc,
                    e.overlap_len1, e.overlap_len2);
    for (size_t v = 0; v < inclusions.size(); v++) if (inclusions[v]) fprintf(fo, "#I\t%zu\n", v);
    if (with_in)
        for (size_t v = 0; v < adj_in.size(); v++) {
            if (adj_in[v].empty()) continue;
            fprintf(fo, "#IN\t%zu", v);
            for (node_id_t s : adj_in[v]) fprintf(fo, "\t%lu", s);
            fprintf(fo, "\n");
        }
    fclose(fo);
}

// ---------------------------------------------------------------------------------------------- EdgeCalculator
EdgeCalculator::EdgeCalculator(std::shared_ptr<FastqStorage> fastq, std::shared_ptr<OverlapGraph> graph, const ProgramSettings ps)
    : ps_(ps), fastq_(fastq), graph_(graph) {}

static hc_params to_params(const ProgramSettings& ps) {
    hc_params p;
    memset(&p, 0, sizeof(p));
    p.edge_threshold = ps.edge_threshold;
    p.ov_threshold = ps.ov_threshold;
    p.merge_contigs = ps.merge_contigs;
    p.mismatch = ps.mismatch;
    p.min_read_len = ps.min_read_len;
    p.flags = ps.exact_scores ? HC_FLAG_EXACT_EDGE_SCORES : 0u;
    return p;
}

double EdgeCalculator::phred_to_prob(const int phred) { return hc_phred_to_prob(phred); }

double EdgeCalculator::overlap_score(std::string seq1, std::string seq2, std::string score1, std::string score2,
                                     const unsigned int pos, double& mismatch_rate) {
    const hc_params p = to_params(ps_);
    const double s = hc_overlap_score(seq1.data(), (uint32_t)seq1.size(), seq2.data(), (uint32_t)seq2.size(), score1.data(),
                                      score2.data(), pos, &p, &mismatch_rate);
    if (s < 0) die(std::string("hc_overlap_score: ") + hc_last_error());
    return s;
}

// The body of src/EdgeCalculator.cpp:389-557: score the batch on the device (the omp-parallel
// region), then the serial, ORDER-DEPENDENT graph insert (:429-545) and the non-edge append (:546-555).
void EdgeCalculator::process_overlaps(std::vector<Overlap>& batch) {
    const size_t n = batch.size();
    if (n == 0) return;
    std::vector<hc_candidate> cand(n);
    for (size_t i = 0; i < n; i++) {
        const Overlap& o = batch[i];
        hc_candidate& c = cand[i];
        memset(&c, 0, sizeof(c));
        if (o.idx1 >= 0 && o.idx2 >= 0) {
            c.idx1 = (uint32_t)o.idx1; c.idx2 = (uint32_t)o.idx2;
        } else {
            auto i1 = fastq_->m_ID_to_index.find(o.id1), i2 = fastq_->m_ID_to_index.find(o.id2);
            if (i1 == fastq_->m_ID_to_index.end()) die(std::to_string(o.id1) + "\nread ID of the overlaps file is not in the fastq input");
            if (i2 == fastq_->m_ID_to_index.end()) die(std::to_string(o.id2) + "\nread ID of the overlaps file is not in the fastq input");
            c.idx1 = i1->second; c.idx2 = i2->second;
        }
        c.pos1 = o.pos1; c.pos2 = o.pos2; c.len1 = o.len1; c.len2 = o.len2;
        c.perc1 = (uint8_t)o.perc1; c.perc2 = (uint8_t)o.perc2;
        c.ord = (uint8_t)o.ord; c.ori1 = o.ori1 == '+'; c.ori2 = o.ori2 == '+';
        c.type1 = (uint8_t)o.type1; c.type2 = (uint8_t)o.type2;
    }
    std::unique_ptr<hc_edge[]> edges_buf(new hc_edge[n]);       // written by the call, not zero-initialised here
    std::unique_ptr<uint64_t[]> nonedge_buf(new uint64_t[n]);
    hc_edge* edges = edges_buf.get();
    uint64_t* nonedge = nonedge_buf.get();
    uint64_t ne = 0, nn = 0;
    hc_batch_stats st;
    const hc_params p = to_params(ps_);
    int rc;
    const double ts0 = wall_s();
    bool fits = fastq_->max_read_len < (1u << 14);
    for (size_t i = 0; i < n && fits; i++) fits = cand[i].pos1 < (1u << 14) && cand[i].pos2 < (1u << 14);
    if (fits && fastq_->m_read_vec.size() < (1ull << 31)) {
        // run-encoded 8-byte records: the copy in is what bounds the call, and the overlaps of one read follow each other
        // in the file.  Greedy cut: a run grows while the next candidate still contains one of the reads every
        // candidate of the run has contained so far.
        std::vector<hc_candidate_entry> en(n);
        std::vector<uint32_t> anchor;
        std::vector<uint64_t> start;
        for (size_t i = 0; i < n;) {
            const uint32_t a = cand[i].idx1, b = cand[i].idx2;
            bool a_ok = true, b_ok = true;
            size_t j = i + 1;
            for (; j < n; j++) {
                const bool ha = a_ok && (cand[j].idx1 == a || cand[j].idx2 == a), hb = b_ok && (cand[j].idx1 == b || cand[j].idx2 == b);
                if (!ha && !hb) break;
                a_ok = ha; b_ok = hb;
            }
            const uint32_t anc = a_ok ? a : b;
            start.push_back(i);
            anchor.push_back(anc);
            for (size_t k = i; k < j; k++) {
                const hc_candidate& c = cand[k];
                const uint32_t o = c.ord == '1' ? 1u : (c.ord == '2' ? 2u : 0u);
                en[k].other = c.idx1 == anc ? c.idx2 : (c.idx1 | 0x80000000u);
                en[k].pos = c.pos1 | (c.pos2 << 14) | ((uint32_t)(c.ori1 != 0) << 28) | ((uint32_t)(c.ori2 != 0) << 29) | (o << 30);
            }
            i = j;
        }
        start.push_back(n);
        rc = hc_score_batch_runs(fastq_->device_store(), &p, anchor.data(), start.data(), anchor.size(), en.data(), n, nullptr, edges, n,
                                 &ne, nonedge, n, &nn, &st);
    } else if (fits) {   // 12-byte records
        std::vector<hc_candidate_short> sc(n);
        for (size_t i = 0; i < n; i++) {
            const hc_candidate& c = cand[i];
            const uint32_t o = c.ord == '1' ? 1u : (c.ord == '2' ? 2u : 0u);
            sc[i].idx1 = c.idx1; sc[i].idx2 = c.idx2;
            sc[i].pos = c.pos1 | (c.pos2 << 14) | ((uint32_t)(c.ori1 != 0) << 28) | ((uint32_t)(c.ori2 != 0) << 29) | (o << 30);
        }
        rc = hc_score_batch_short(fastq_->device_store(), &p, sc.data(), n, nullptr, edges, n, &ne, nonedge, n, &nn, &st);
    } else {
        rc = hc_score_batch(fastq_->device_store(), &p, cand.data(), n, nullptr, edges, n, &ne, nonedge, n, &nn, &st);
    }
    if (rc != HC_OK) die(std::string("hc_score_batch: ") + hc_last_error());
    scored_candidates += n;
    device_ms += st.total_ms;
    const double ts1 = wall_s();
    t_score_s += ts1 - ts0;

    unsigned int doubles = 0;
    for (uint64_t k = 0; k < ne; k++) {
        const hc_edge& he = edges[k];
        const Overlap& o = batch[he.cand];
        const hc_candidate& c = cand[he.cand];
        const Read& r1 = fastq_->m_read_vec[c.idx1];
        const Read& r2 = fastq_->m_read_vec[c.idx2];
        Edge e;
        e.score = he.score;
        if (ps_.exact_scores) {   // :138 and :256-261 with the host libm on the reference's own mean logs
            const double ov1 = std::isnan(he.mean_log[0]) ? 0.0 : exp(he.mean_log[0]);
            if (r1.is_paired || r2.is_paired) {
                const double ov2 = std::isnan(he.mean_log[1]) ? 0.0 : exp(he.mean_log[1]);
                e.score = (ov1 > ps_.edge_threshold && ov2 > ps_.edge_threshold) ? 0.5 * (ov1 + ov2) : std::min(ov1, ov2);
            } else {
                e.score = ov1;
            }
        }
        e.pos1 = (int)o.pos1; e.pos2 = (int)o.pos2; e.pos3 = he.pos3; e.pos4 = he.pos4;
        e.ori1 = o.ori1 == '+'; e.ori2 = o.ori2 == '+';
        e.ord = o.ord;
        e.vertex1 = r1.vertex_id; e.vertex2 = r2.vertex_id;
        e.overlap_perc = (int)o.get_perc();
        e.overlap_len1 = (int)o.len1;
        e.overlap_len2 = (r1.is_paired || r2.is_paired) ? (int)o.len2 : 0;       // set_len(len1, 0) for S-S, :227
        e.overlap_len = e.overlap_len1 + e.overlap_len2;
        e.mismatch_rate = he.mismatch_rate;

        if (e.pos1 == 0 && e.vertex1 > e.vertex2) e.swap_reads();                  // :443-448
        if (ps_.gpu_dedup) pending_.push_back(e);
        else insert_edge(e, doubles);
    }
    dup_count += doubles;
    const double ts2 = wall_s();
    t_edges_s += ts2 - ts1;

    std::ofstream out((ps_.output_dir + "nonedge_overlaps.txt").c_str(), std::fstream::out | std::fstream::app);
    std::string buf;
    buf.reserve(1 << 22);
    for (uint64_t k = 0; k < nn; k++) {
        batch[nonedge[k]].append_overlap_line(buf);
        if (buf.size() > (1u << 22) - 256) { out.write(buf.data(), (std::streamsize)buf.size()); buf.clear(); }
    }
    out.write(buf.data(), (std::streamsize)buf.size());
    t_write_s += wall_s() - ts2;
}

// One step of the sequential insert, src/EdgeCalculator.cpp:449-538 (the edge is already normalised).
void EdgeCalculator::insert_edge(Edge& e, unsigned int& doubles) {
    const node_id_t v1 = e.vertex1, v2 = e.vertex2;
    if (e.overlap_perc == 100) inclusion_count++;                              // :449-451
    const bool same_ori = e.ori1 == e.ori2;
    const double have = graph_->checkEdgeWithOri(v1, v2, same_ori);
    if (have < 0) {                                                            // :455-469
        graph_->addEdge(e);
        if (ps_.ignore_inclusions && e.overlap_perc == 100 && e.mismatch_rate < 0.000001 && e.mismatch_rate >= 0) {
            if (e.pos3 < 0) { if (e.pos1 == 0) graph_->inclusions[v1] = 1; }
            else graph_->inclusions[v2] = 1;
        }
    } else if (e.score >= have) {                                              // :470-534
        doubles++;
        const Edge* old = graph_->getEdgeInfoWithOri(v1, v2, same_ori);
        bool keep_old = false;
        if (have == e.score) {   // the reference's deterministic tie-break, one criterion decides
            if (old->overlap_len != e.overlap_len) keep_old = old->overlap_len > e.overlap_len;
            else if (old->mismatch_rate != e.mismatch_rate) keep_old = old->mismatch_rate < e.mismatch_rate;
            else if (old->vertex1 != e.vertex1) keep_old = old->vertex1 < e.vertex1;
            else if (old->ori1 != e.ori1) keep_old = old->ori1;
            else if (old->ori2 != e.ori2) keep_old = old->ori2;
            else if (old->pos1 != e.pos1) keep_old = old->pos1 < e.pos1;
            else if (old->pos2 != e.pos2) keep_old = old->pos2 < e.pos2;
        }
        if (keep_old) return;
        if (old->vertex1 == v1) graph_->removeEdgeWithOri(v1, v2, same_ori);
        else graph_->removeEdgeWithOri(v2, v1, same_ori);
        graph_->addEdge(e);
    } else {
        doubles++;                                                             // :535-538
    }
}

int EdgeCalculator::handle_line(const std::string& line, std::vector<Overlap>& batch, std::vector<Overlap>& filtered) {
    size_t b = 0, e = line.size();
    while (b < e && (line[b] == '\t' || line[b] == ' ')) b++;                      // trim outer tabs/spaces, :584
    while (e > b && (line[e - 1] == '\t' || line[e - 1] == ' ')) e--;
    std::vector<std::string> f;
    std::string cur;
    if (b < e) {
        for (size_t k = b; k < e; k++) {
            const char ch = line[k];
            const bool sep = ps_.allow_spaces ? (ch == '\t' || ch == ' ') : ch == '\t';
            if (sep) {
                f.push_back(cur);
                cur.clear();
                if (ps_.allow_spaces) while (k + 1 < e && (line[k + 1] == '\t' || line[k + 1] == ' ')) k++;   // token_compress_on
            } else cur.push_back(ch);
        }
        f.push_back(cur);
    }
    if (f.size() != 13) { std::cout << "incorrect overlap; skipping" << std::endl; return 0; }   // :600-603
    Overlap o = Overlap::from_fields(f);
    if (o.id1 == o.id2) return 0;                                                  // :605-607
    const bool any_p = o.type1 == 'p' || o.type2 == 'p';
    bool in_band = false;
    if (o.len1 >= ps_.min_overlap_len && o.type1 == 's' && o.type2 == 's') in_band = true;                   // :612-617
    else if (o.len1 >= 0.5 * ps_.min_overlap_len && o.len2 >= 0.5 * ps_.min_overlap_len && any_p) in_band = true;   // :618-624
    else if (ps_.relax_PE_edges && o.len1 + o.len2 >= ps_.min_overlap_len && any_p) in_band = true;          // :626-632
    if (in_band) {
        if (o.get_perc() >= ps_.min_overlap_perc) { batch.push_back(o); return 1; }
        return 0;
    }
    filtered.push_back(o);                                                         // :633-635
    return 2;
}

// The text loop on the device: the file goes to hc_ingest_overlaps in pieces that end at a line end; scored
// candidates arrive with their store indices, pre-filtered overlaps as printable records, both in file order.
void EdgeCalculator::ingest_on_device(std::vector<Overlap>& batch, std::vector<Overlap>& filtered) {
    std::ifstream in(ps_.overlaps_file.c_str(), std::ios::binary);
    if (!in.is_open()) { std::cerr << "Unable to open overlaps file"; std::exit(1); }
    hc_idmap* idmap = fastq_->device_idmap();
    const size_t piece = (size_t)64 << 20;
    std::string buf, carry;
    unsigned long lines_done = 0;
    std::vector<hc_candidate> cand;
    std::vector<hc_overlap_rec> filt;
    while (lines_done < ps_.max_overlaps) {
        buf = carry;
        carry.clear();
        const size_t have = buf.size();
        buf.resize(have + piece);
        in.read(&buf[have], (std::streamsize)piece);
        buf.resize(have + (size_t)in.gcount());
        if (buf.empty()) break;
        if (!in.eof()) {                       // keep the unfinished last line for the next piece
            const size_t nl = buf.rfind('\n');
            if (nl == std::string::npos) { carry.swap(buf); continue; }
            carry = buf.substr(nl + 1);
            buf.resize(nl + 1);
        }
        const size_t cap = (size_t)std::count(buf.begin(), buf.end(), '\n') + 1;
        cand.resize(cap);
        filt.resize(cap);
        hc_ingest_params ip;
        memset(&ip, 0, sizeof(ip));
        ip.max_overlaps = ps_.max_overlaps - lines_done;
        ip.min_overlap_len = ps_.min_overlap_len; ip.min_overlap_perc = ps_.min_overlap_perc;
        ip.relax_PE_edges = ps_.relax_PE_edges; ip.allow_spaces = ps_.allow_spaces;
        hc_ingest_stats st;
        const double ti0 = wall_s();
        const int rc = hc_ingest_overlaps(idmap, buf.data(), buf.size(), &ip, cand.data(), nullptr, cap, filt.data(), nullptr, cap, &st);
        t_ingest_s += wall_s() - ti0;
        if (rc != HC_OK) die(std::string("hc_ingest_overlaps: ") + hc_last_error());
        if (st.first_error_line != ~0ull) {    // the reference ends at this line: let the host parser say why
            std::vector<Overlap> b2, f2;
            handle_line(buf.substr(st.first_error_offset, st.first_error_length), b2, f2);
            if (!b2.empty()) process_overlaps(b2);    // an id that is not in the store
            die("overlaps file: line rejected by the device parser");
        }
        for (uint64_t k = 0; k < st.n_skipped; k++) std::cout << "incorrect overlap; skipping" << std::endl;   // :600-603
        for (uint64_t k = 0; k < st.n_filtered; k++) {
            const hc_overlap_rec& r = filt[k];
            Overlap o;
            o.id1 = r.id1; o.id2 = r.id2; o.pos1 = r.pos1; o.pos2 = r.pos2; o.perc1 = r.perc1; o.perc2 = r.perc2;
            o.len1 = r.len1; o.len2 = r.len2; o.ord = (char)r.ord; o.ori1 = (char)r.ori1; o.ori2 = (char)r.ori2;
            o.type1 = (char)r.type1; o.type2 = (char)r.type2;
            filtered.push_back(o);
        }
        for (uint64_t k = 0; k < st.n_scored; k++) {
            const hc_candidate& c = cand[k];
            Overlap o;
            o.idx1 = c.idx1; o.idx2 = c.idx2;
            o.id1 = fastq_->m_read_vec[c.idx1].read_id; o.id2 = fastq_->m_read_vec[c.idx2].read_id;
            o.pos1 = c.pos1; o.pos2 = c.pos2; o.perc1 = c.perc1; o.perc2 = c.perc2; o.len1 = c.len1; o.len2 = c.len2;
            o.ord = (char)c.ord; o.ori1 = c.ori1 ? '+' : '-'; o.ori2 = c.ori2 ? '+' : '-';
            o.type1 = (char)c.type1; o.type2 = (char)c.type2;
            batch.push_back(o);
            if (batch.size() == 1000000) { process_overlaps(batch); batch.clear(); }   // :636-644
        }
        lines_done += st.n_lines;
        parse_device_ms += st.device_ms;
        if (in.eof() && carry.empty()) break;
    }
}

// ---- the stage on arrays ------------------------------------------------------------------------------------
// What the reference does line by line and object by object (:561-666 with process_overlaps :389-557) on flat arrays:
// the order of everything observable is the file order -- accepted edges are inserted in file order, nonedge_overlaps.txt
// holds the scored non-edges in file order followed by the pre-filtered lines in file order (the batches of 10^6 of :571
// do not change either) -- so one parse call, one scoring call and loops over arrays that every host thread takes a
// share of reproduce it.
namespace {

// the same line through a raw pointer (no capacity check per character; the caller reserves HC_LINE_MAX bytes per line)
#define HC_LINE_MAX 160
inline char* put_u(char* p, unsigned long v) {
    static const char d2[] = "00010203040506070809101112131415161718192021222324252627282930313233343536373839404142434445464748495051525354555657585960616263646566676869707172737475767778798081828384858687888990919293949596979899";
    char tmp[24];
    int k = 24;
    while (v >= 100) { const unsigned long q = v / 100; const unsigned r = (unsigned)(v - q * 100); v = q; tmp[--k] = d2[2 * r + 1]; tmp[--k] = d2[2 * r]; }
    if (v >= 10) { tmp[--k] = d2[2 * v + 1]; tmp[--k] = d2[2 * v]; }
    else tmp[--k] = (char)('0' + v);
    const int n = 24 - k;
    memcpy(p, tmp + k, (size_t)n);
    return p + n;
}
inline char* put_cand_line(char* p, const hc_candidate& c, read_id_t id1, read_id_t id2) {                  // src/Overlap.h:234-237
    p = put_u(p, id1); *p++ = '\t'; p = put_u(p, id2); *p++ = '\t'; p = put_u(p, c.pos1); *p++ = '\t'; p = put_u(p, c.pos2);
    *p++ = '\t'; *p++ = (char)c.ord; *p++ = '\t'; *p++ = c.ori1 ? '+' : '-'; *p++ = '\t'; *p++ = c.ori2 ? '+' : '-'; *p++ = '\t';
    p = put_u(p, c.perc1); *p++ = '\t'; p = put_u(p, c.perc2); *p++ = '\t'; p = put_u(p, c.len1); *p++ = '\t'; p = put_u(p, c.len2);
    *p++ = '\t'; *p++ = (char)c.type1; *p++ = '\t'; *p++ = (char)c.type2; *p++ = '\n';
    return p;
}

inline void put_rec_line(std::string& b, const hc_overlap_rec& r) {
    put_u64(b, r.id1); b.push_back('\t'); put_u64(b, r.id2); b.push_back('\t'); put_u64(b, r.pos1); b.push_back('\t'); put_u64(b, r.pos2);
    b.push_back('\t'); b.push_back((char)r.ord); b.push_back('\t'); b.push_back((char)r.ori1); b.push_back('\t'); b.push_back((char)r.ori2);
    b.push_back('\t');
    put_u64(b, r.perc1); b.push_back('\t'); put_u64(b, r.perc2); b.push_back('\t'); put_u64(b, r.len1); b.push_back('\t'); put_u64(b, r.len2);
    b.push_back('\t'); b.push_back((char)r.type1); b.push_back('\t'); b.push_back((char)r.type2); b.push_back('\n');
}

}  // namespace

bool EdgeCalculator::construct_edges_arrays() {
    // one device: parse and score in one call, no limit on read lengths; more devices: the 8-byte run records, which
    // hc_score_batch_runs_small shards over the devices
    hc_store* const store = fastq_->device_store();
    const bool one_call = hc_store_n_devices(store) == 1;
    if (!one_call && (fastq_->max_read_len >= (1u << 14) || fastq_->m_read_vec.size() >= (1ull << 31))) return false;   // needs the 8-byte records
    const int T = std::max(1, omp_get_max_threads());
    // HC_MIRROR_TIMING=1: wall clock of every step of this function on stderr
    const bool timing = getenv("HC_MIRROR_TIMING") != nullptr;
    double t_mark = wall_s();
    auto mark = [&](const char* what) {
        if (!timing) return;
        const double t = wall_s();
        fprintf(stderr, "[construct_edges] %-34s %8.2f ms\n", what, (t - t_mark) * 1e3);
        t_mark = t;
    };
    // ---- the file, in one read (several threads; or already read by the caller while the read store was built)
    const double t0 = wall_s();
    FileBuf fb;
    if (have_preloaded) { fb = std::move(preloaded_overlaps); have_preloaded = false; }
    else if (!read_whole_file(ps_.overlaps_file, fb)) { std::cerr << "Unable to open overlaps file"; std::exit(1); }
    struct { char* p; char* get() const { return p; } char operator[](long long i) const { return p[i]; } } text{fb.data};
    const size_t got = fb.size;
    const double t0r = wall_s();
    size_t lines = 1;
#pragma omp parallel for schedule(static) reduction(+ : lines)
    for (long long i = 0; i < (long long)got; i++) lines += text[i] == '\n';
    (void)t0r;
    mark("file read + line count");
    hc_ingest_params ip;
    memset(&ip, 0, sizeof(ip));
    ip.max_overlaps = ps_.max_overlaps;
    ip.min_overlap_len = ps_.min_overlap_len; ip.min_overlap_perc = ps_.min_overlap_perc;
    ip.relax_PE_edges = ps_.relax_PE_edges; ip.allow_spaces = ps_.allow_spaces;
    hc_ingest_stats st;
    hc_idmap* idmap = fastq_->device_idmap();
    size_t filt_cap = std::max<size_t>(lines / 8, 4096);
    std::unique_ptr<hc_overlap_rec[]> filt(new hc_overlap_rec[filt_cap]);
    const hc_params p = to_params(ps_);
    const size_t erec = ps_.exact_scores ? sizeof(hc_edge_small_exact) : sizeof(hc_edge_small);
    // what the rest works on: candidates (the edge records' `cand` indexes them), the non-edge bit map over them, edges
    std::unique_ptr<hc_candidate[]> cand;
    std::unique_ptr<uint64_t[]> bits;
    std::unique_ptr<char[]> ebuf;
    size_t n = 0;
    uint64_t ne = 0, nn = 0;
    int rc = HC_OK;
    double t1 = 0;
    if (one_call) {
        // ---- parse + pre-filter + id lookup + scoring on the device; only the candidates scored as edges or non-edges
        // come back (with their class), and the edge records name them
        t_ingest_s += wall_s() - t0;
        t1 = wall_s();
        size_t kcap = std::max<size_t>(lines / 2, 4096), ecap = std::max<size_t>(lines / 8, 1024);
        std::unique_ptr<uint8_t[]> kcls(new uint8_t[kcap]);
        cand.reset(new hc_candidate[kcap]);
        ebuf.reset(new char[ecap * erec]);
        hc_ingest_score_stats ss;
        rc = hc_ingest_score_overlaps(store, idmap, text.get(), got, &ip, &p, cand.get(), nullptr, kcls.get(), kcap, ebuf.get(), ecap,
                                      filt.get(), nullptr, filt_cap, &ss);
        if (rc == HC_ERR_CAPACITY) {
            if (ss.n_kept > kcap) { kcap = ss.n_kept; kcls.reset(new uint8_t[kcap]); cand.reset(new hc_candidate[kcap]); }
            if (ss.score.n_edges > ecap) { ecap = ss.score.n_edges; ebuf.reset(new char[ecap * erec]); }
            if (ss.ingest.n_filtered > filt_cap) { filt_cap = ss.ingest.n_filtered; filt.reset(new hc_overlap_rec[filt_cap]); }
            rc = hc_ingest_score_overlaps(store, idmap, text.get(), got, &ip, &p, cand.get(), nullptr, kcls.get(), kcap, ebuf.get(), ecap,
                                          filt.get(), nullptr, filt_cap, &ss);
        }
        if (rc != HC_OK) die(std::string("hc_ingest_score_overlaps: ") + hc_last_error());
        st = ss.ingest;
        parse_device_ms += st.device_ms;
        if (st.first_error_line != ~0ull) return false;      // the line-by-line path reproduces what the reference does up to that line
        n = ss.n_kept;
        ne = ss.score.n_edges;
        nn = ss.score.n_nonedges;
        bool overflow = false;
#pragma omp parallel for schedule(static) reduction(|| : overflow)
        for (long long k = 0; k < (long long)ne; k++) overflow = overflow || (reinterpret_cast<const hc_edge_small*>(ebuf.get() + (size_t)k * erec)->flags & HC_EDGE_OVERFLOW);
        if (overflow) return false;                          // a window of 65536+ positions: the batch path scores it
        const size_t words = (n + 63) / 64;
        bits.reset(new uint64_t[words + 1]);
#pragma omp parallel for schedule(static)
        for (long long w = 0; w < (long long)words; w++) {
            uint64_t b = 0;
            for (size_t i = (size_t)w * 64; i < std::min(n, (size_t)w * 64 + 64); i++) b |= (uint64_t)(kcls[i] == HC_CLASS_NONEDGE) << (i & 63);
            bits[w] = b;
        }
        scored_candidates += st.n_scored;
        device_ms += ss.score.total_ms;
        for (uint64_t k = 0; k < st.n_skipped; k++) std::cout << "incorrect overlap; skipping" << std::endl;   // :600-603
        mark("hc_ingest_score_overlaps");
    } else {
        cand.reset(new hc_candidate[lines]);
        rc = hc_ingest_overlaps(idmap, text.get(), got, &ip, cand.get(), nullptr, lines, filt.get(), nullptr, filt_cap, &st);
        if (rc == HC_ERR_CAPACITY) {
            filt_cap = st.n_filtered + 1;
            filt.reset(new hc_overlap_rec[filt_cap]);
            rc = hc_ingest_overlaps(idmap, text.get(), got, &ip, cand.get(), nullptr, lines, filt.get(), nullptr, filt_cap, &st);
        }
        if (rc != HC_OK) die(std::string("hc_ingest_overlaps: ") + hc_last_error());
        parse_device_ms += st.device_ms;
        if (st.first_error_line != ~0ull) return false;      // the line-by-line path reproduces what the reference does up to that line
        n = st.n_scored;
        mark("hc_ingest_overlaps");
        t1 = wall_s();
        t_ingest_s += t1 - t0;
        bool fits = true;
#pragma omp parallel for schedule(static) reduction(&& : fits)
        for (long long i = 0; i < (long long)n; i++) fits = fits && cand[i].pos1 < (1u << 14) && cand[i].pos2 < (1u << 14);
        if (!fits) return false;
        for (uint64_t k = 0; k < st.n_skipped; k++) std::cout << "incorrect overlap; skipping" << std::endl;   // :600-603
        // ---- run-encoded records: a run = a stretch of candidates with the same smaller read index (an overlaps file sorted by
        // read gives long runs; any list gives valid ones), cut by every thread in its own share
        std::unique_ptr<hc_candidate_entry[]> en(new hc_candidate_entry[n ? n : 1]);
        std::vector<std::vector<uint64_t>> t_start(T);
        std::vector<uint32_t> anchor;
        std::vector<uint64_t> start;
#pragma omp parallel num_threads(T)
        {
            const int t = omp_get_thread_num();
            const size_t lo = n * (size_t)t / (size_t)T, hi = n * (size_t)(t + 1) / (size_t)T;
            std::vector<uint64_t>& mine = t_start[t];
            for (size_t i = lo; i < hi; i++) {
                const hc_candidate& c = cand[i];
                const uint32_t key = std::min(c.idx1, c.idx2);
                if (i == 0 || key != std::min(cand[i - 1].idx1, cand[i - 1].idx2)) mine.push_back(i);
                const uint32_t o = c.ord == '1' ? 1u : (c.ord == '2' ? 2u : 0u);
                en[i].other = c.idx1 == key ? c.idx2 : (c.idx1 | 0x80000000u);
                en[i].pos = c.pos1 | (c.pos2 << 14) | ((uint32_t)(c.ori1 != 0) << 28) | ((uint32_t)(c.ori2 != 0) << 29) | (o << 30);
            }
        }
        for (int t = 0; t < T; t++) start.insert(start.end(), t_start[t].begin(), t_start[t].end());
        anchor.resize(start.size());
#pragma omp parallel for schedule(static)
        for (long long r = 0; r < (long long)start.size(); r++) anchor[r] = std::min(cand[start[r]].idx1, cand[start[r]].idx2);
        start.push_back(n);
        mark("run-encoded records");
        // ---- scoring: small outputs
        size_t ecap = std::max<size_t>(n / 4, 1024);
        ebuf.reset(new char[ecap * erec]);
        bits.reset(new uint64_t[n / 64 + 2]);
        hc_batch_stats bst;
        memset(&bst, 0, sizeof(bst));
        if (n) {
            rc = hc_score_batch_runs_small(store, &p, anchor.data(), start.data(), anchor.size(), en.get(), n, ebuf.get(), ecap, &ne,
                                           bits.get(), &nn, &bst);
            if (rc == HC_ERR_CAPACITY) {
                ecap = ne;
                ebuf.reset(new char[ecap * erec]);
                rc = hc_score_batch_runs_small(store, &p, anchor.data(), start.data(), anchor.size(), en.get(), n, ebuf.get(), ecap,
                                               &ne, bits.get(), &nn, &bst);
            }
            if (rc != HC_OK) die(std::string("hc_score_batch_runs_small: ") + hc_last_error());
        }
        scored_candidates += n;
        device_ms += bst.total_ms;
        mark("hc_score_batch_runs_small");
    }
    const double t2 = wall_s();
    t_score_s += t2 - t1;
    // ---- nonedge_overlaps.txt: the scored non-edges (bit map) in file order, then the pre-filtered lines (:546-555, :654-660);
    // every thread formats a share of the words into its own buffer; the buffers are written in order by a thread of their own
    // while this one builds the edges (both only read the candidates)
    const size_t words = (n + 63) / 64;
    std::vector<std::unique_ptr<char[]>> part(T);
    std::vector<size_t> part_len(T, 0);
    std::string filt_lines;
    const uint64_t* rid = fastq_->read_ids.data();       // 8 bytes per read instead of a walk over the Read objects
#pragma omp parallel num_threads(T)
    {
        const int t = omp_get_thread_num();
        const size_t lo = words * (size_t)t / (size_t)T, hi = words * (size_t)(t + 1) / (size_t)T;
        size_t mine = 0;
        for (size_t w = lo; w < hi; w++) mine += (size_t)__builtin_popcountll(bits[w]);
        part[t].reset(new char[mine * HC_LINE_MAX + 16]);
        char* p = part[t].get();
        for (size_t w = lo; w < hi; w++) {
            uint64_t m = bits[w];
            while (m) {
                const size_t i = w * 64 + (size_t)__builtin_ctzll(m);
                m &= m - 1;
                const hc_candidate& c = cand[i];
                p = put_cand_line(p, c, rid[c.idx1], rid[c.idx2]);
            }
        }
        part_len[t] = (size_t)(p - part[t].get());
    }
    for (uint64_t k = 0; k < st.n_filtered; k++) put_rec_line(filt_lines, filt[k]);
    bool write_failed = false;
    const std::string nonedge_path = ps_.output_dir + "nonedge_overlaps.txt";
    std::thread writer([&part, &part_len, &filt_lines, &write_failed, &nonedge_path]() {
        FILE* out = std::fopen(nonedge_path.c_str(), "ab");
        if (!out) { write_failed = true; return; }
        for (size_t t = 0; t < part.size(); t++) if (part_len[t]) std::fwrite(part[t].get(), 1, part_len[t], out);
        if (!filt_lines.empty()) std::fwrite(filt_lines.data(), 1, filt_lines.size(), out);
        std::fclose(out);
    });
    mark("non-edge lines formatted");
    const double t2b = wall_s();
    t_write_s += t2b - t2;
    // ---- accepted edges: Edge fields from the candidate + the small record, every thread a share
    std::vector<Edge> es(ne);
    const uint32_t* ml = fastq_->mate_len.data();
    bool overflow = false;
#pragma omp parallel for schedule(static) reduction(|| : overflow)
    for (long long k = 0; k < (long long)ne; k++) {
        const hc_edge_small* hs = reinterpret_cast<const hc_edge_small*>(ebuf.get() + (size_t)k * erec);   // the common head of both records
        const hc_candidate& c = cand[hs->cand];
        const Read& r1 = fastq_->m_read_vec[c.idx1];
        const Read& r2 = fastq_->m_read_vec[c.idx2];
        const bool two = r1.is_paired || r2.is_paired;
        overflow = overflow || (hs->flags & HC_EDGE_OVERFLOW);
        Edge& e = es[(size_t)k];
        if (ps_.exact_scores) {   // :138 and :256-261 with the host libm on the reference's own mean logs
            const hc_edge_small_exact* hx = reinterpret_cast<const hc_edge_small_exact*>(hs);
            const double ov1 = hx->compared[0] ? exp(hx->mean_log[0]) : 0.0;
            if (two) {
                const double ov2 = hx->compared[1] ? exp(hx->mean_log[1]) : 0.0;
                e.score = (ov1 > ps_.edge_threshold && ov2 > ps_.edge_threshold) ? 0.5 * (ov1 + ov2) : std::min(ov1, ov2);
            } else {
                e.score = ov1;
            }
        } else {
            e.score = hs->score;
        }
        double r0 = hs->compared[0] ? (hs->mismatches[0] ? (double)(float)(int)hs->mismatches[0] / (double)hs->compared[0] : 0.0) : 1.0;   // :132
        if (two) {
            const double rb = hs->compared[1] ? (hs->mismatches[1] ? (double)(float)(int)hs->mismatches[1] / (double)hs->compared[1] : 0.0) : 1.0;
            r0 = std::max(r0, rb);                                                                                                         // :254
        }
        e.mismatch_rate = r0;
        int32_t p3, p4;
        hc_edge_extra_pos(c.pos1, c.pos2, (char)c.ord, ml[2 * c.idx1], ml[2 * c.idx1 + 1], ml[2 * c.idx2], ml[2 * c.idx2 + 1], &p3, &p4);
        e.pos1 = (int)c.pos1; e.pos2 = (int)c.pos2; e.pos3 = p3; e.pos4 = p4;
        e.ori1 = c.ori1 != 0; e.ori2 = c.ori2 != 0;
        e.ord = (char)c.ord;
        e.vertex1 = r1.vertex_id; e.vertex2 = r2.vertex_id;
        e.overlap_perc = (int)(c.perc2 > 0 ? (unsigned int)(0.5 * (c.perc1 + c.perc2)) : c.perc1);            // Overlap::get_perc, :203-210
        e.overlap_len1 = (int)c.len1;
        e.overlap_len2 = two ? (int)c.len2 : 0;                                                                // set_len(len1, 0) for S-S, :227
        e.overlap_len = e.overlap_len1 + e.overlap_len2;
        if (e.pos1 == 0 && e.vertex1 > e.vertex2) e.swap_reads();                                              // :443-448
    }
    if (overflow) die("a window of 65536 or more positions: not representable in the small edge records");
    mark("Edge objects");
    unsigned int doubles = 0;
    if (ps_.gpu_dedup && ne) {
        std::vector<hc_dedup_edge> de(ne);
#pragma omp parallel for schedule(static)
        for (long long k = 0; k < (long long)ne; k++) {
            const Edge& e = es[(size_t)k];
            hc_dedup_edge& d = de[(size_t)k];
            memset(&d, 0, sizeof(d));
            d.vertex1 = (uint32_t)e.vertex1; d.vertex2 = (uint32_t)e.vertex2; d.score = e.score; d.mismatch_rate = e.mismatch_rate;
            d.pos1 = e.pos1; d.pos2 = e.pos2; d.pos3 = e.pos3; d.overlap_len = e.overlap_len; d.perc = e.overlap_perc;
            d.ori1 = e.ori1; d.ori2 = e.ori2;
        }
        std::vector<uint8_t> win(ne);
        uint64_t counts[2] = {0, 0};
        rc = hc_dedup_edges(de.data(), de.size(), ps_.ignore_inclusions, win.data(), (uint8_t*)graph_->inclusions.data(),
                            graph_->inclusions.size(), counts, ps_.first_device);
        if (rc != HC_OK) die(std::string("hc_dedup_edges: ") + hc_last_error());
        mark("hc_dedup_edges");
        graph_->addEdges(es, win.data());
        mark("addEdges");
        dup_count += (unsigned int)counts[0];
        inclusion_count += (unsigned int)counts[1];
    } else {
        for (size_t k = 0; k < ne; k++) insert_edge(es[k], doubles);
        dup_count += doubles;
    }
    const double t3 = wall_s();
    t_edges_s += t3 - t2b;
    if (ps_.verbose) {
        std::cout << "Number of self-overlapping reads: " << self_overlap_count << "\n";
        std::cout << "Number of inclusion edges: " << inclusion_count << "\n";
    }
    writer.join();
    if (write_failed) die("Unable to open nonedge_overlaps.txt");
    mark("non-edge file written (join)");
    t_write_s += wall_s() - t3;
    return true;
}

void EdgeCalculator::construct_edges() {                                          // src/EdgeCalculator.cpp:561-666
    if (ps_.add_duplicates) die("add_duplicates=true is not supported by this build (no driver script uses it)");
    std::remove("nonedge_overlaps.txt");                                          // :566 (cwd, like the reference)
    const size_t per_batch = 1000000;                                             // :571
    std::vector<Overlap> batch, filtered;
    batch.reserve(per_batch);
    if (ps_.gpu_parse && construct_edges_arrays()) return;
    if (ps_.gpu_parse) {
        ingest_on_device(batch, filtered);
    } else {
        std::ifstream in(ps_.overlaps_file.c_str());
        if (!in.is_open()) { std::cerr << "Unable to open overlaps file"; std::exit(1); }
        std::string line;
        unsigned long i = 0;
        while (i < ps_.max_overlaps && getline(in, line)) {
            i++;
            handle_line(line, batch, filtered);
            if (batch.size() == per_batch) { process_overlaps(batch); batch.clear(); }
        }
    }
    if (!batch.empty()) { process_overlaps(batch); batch.clear(); }
    if (ps_.gpu_dedup && !pending_.empty()) {
        // all accepted edges of the run at once: the per-key arg-max of hc_dedup_edges equals the sequential
        // replace-if-better fold, and the survivors in input order are the final adjacency lists
        std::vector<hc_dedup_edge> de(pending_.size());
        for (size_t k = 0; k < pending_.size(); k++) {
            const Edge& e = pending_[k];
            hc_dedup_edge& d = de[k];
            memset(&d, 0, sizeof(d));
            d.vertex1 = (uint32_t)e.vertex1; d.vertex2 = (uint32_t)e.vertex2; d.score = e.score; d.mismatch_rate = e.mismatch_rate;
            d.pos1 = e.pos1; d.pos2 = e.pos2; d.pos3 = e.pos3; d.overlap_len = e.overlap_len; d.perc = e.overlap_perc;
            d.ori1 = e.ori1; d.ori2 = e.ori2;
        }
        std::vector<uint8_t> win(pending_.size());
        uint64_t counts[2] = {0, 0};
        const int rc = hc_dedup_edges(de.data(), de.size(), ps_.ignore_inclusions, win.data(), (uint8_t*)graph_->inclusions.data(),
                                      graph_->inclusions.size(), counts, ps_.first_device);
        if (rc != HC_OK) die(std::string("hc_dedup_edges: ") + hc_last_error());
        for (size_t k = 0; k < pending_.size(); k++) if (win[k]) graph_->addEdge(pending_[k]);
        dup_count += (unsigned int)counts[0];
        inclusion_count += (unsigned int)counts[1];
        pending_.clear();
    }
    if (ps_.verbose) {
        std::cout << "Number of self-overlapping reads: " << self_overlap_count << "\n";
        std::cout << "Number of inclusion edges: " << inclusion_count << "\n";
    }
    std::ofstream out((ps_.output_dir + "nonedge_overlaps.txt").c_str(), std::fstream::out | std::fstream::app);   // :654-660
    std::string buf;
    buf.reserve(1 << 22);
    for (const Overlap& o : filtered) {
        o.append_overlap_line(buf);
        if (buf.size() > (1u << 22) - 256) { out.write(buf.data(), (std::streamsize)buf.size()); buf.clear(); }
    }
    out.write(buf.data(), (std::streamsize)buf.size());
}

}  // namespace hcb
