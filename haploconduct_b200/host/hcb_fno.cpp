// hcb_fno.cpp -- SRBuilder::findNextOverlaps / findNextOverlaps3 on the C ABI (hc_fno1 / hc_fno3).
// See hcb_fno.h for what is host code here and why.  Reference: src/FindNextOverlaps.cpp, src/FindNextOverlaps3.cpp.
#include "hcb_fno.h"

#include <algorithm>
#include <cassert>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <memory>
#include <sstream>

namespace hcb {

namespace {

double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// Calls `call(buf, cap, &n_bytes, &n_lines)` into a buffer sized from `guess` lines and, if the text does not fit, once more
// with the exact size; writes the text to `filename` with one write.  Returns the line count; `t_text` is when the text
// had arrived in host memory.
// With input_error, HC_ERR_INPUT sets it and returns 0 without writing the file (the caller takes another path).
template <class Call>
uint64_t write_text(Call call, uint64_t guess, const std::string& filename, const char* what, double& t_text, bool* input_error = nullptr) {
    uint64_t cap = std::min<uint64_t>(guess, 1ull << 24) * 128 + 4096, n_bytes = 0, n_lines = 0;
    std::unique_ptr<char[]> buf(new char[cap]);            // not touched here: only the written pages are committed
    int rc = call(buf.get(), cap, &n_bytes, &n_lines);
    if (rc == HC_ERR_CAPACITY) {
        cap = n_bytes;
        buf.reset(new char[cap]);
        rc = call(buf.get(), cap, &n_bytes, &n_lines);
    }
    if (rc == HC_ERR_INPUT && input_error) { *input_error = true; return 0; }
    if (rc != HC_OK) die(std::string(what) + ": " + hc_last_error());
    t_text = now_s();
    std::ofstream outfile(filename.c_str(), std::ios::binary);
    if (!outfile.is_open()) die("Unable to open " + filename);
    outfile.write(buf.get(), (std::streamsize)n_bytes);
    outfile.close();
    if (!outfile) die("Unable to write " + filename);
    return n_lines;
}

hc_fno_edge to_fno_edge(const Edge& e) {
    hc_fno_edge f;
    std::memset(&f, 0, sizeof(f));
    f.u = (uint32_t)e.vertex1;
    f.v = (uint32_t)e.vertex2;
    f.pos1 = e.pos1;
    f.pos2 = e.pos2;
    f.perc = e.overlap_perc;
    f.len1 = e.overlap_len1;
    f.len2 = e.overlap_len2;
    f.ord = (uint8_t)e.ord;
    f.ori1 = e.ori1 ? 1 : 0;
    f.ori2 = e.ori2 ? 1 : 0;
    f.nonedge = e.score == 0 ? 1 : 0;              // Edge::score == 0 marks a non-edge overlap (:34)
    return f;
}

}  // namespace

SRBuilder::SRBuilder(std::shared_ptr<FastqStorage> fastq, std::shared_ptr<OverlapGraph> graph, const ProgramSettings ps)
    : ps_(ps), fastq_(fastq), graph_(graph) {
    visited.assign(graph ? graph->getVertexCount() : 0, 0);     // src/SRBuilder.h:96-106
}

bool SRBuilder::orientation(node_id_t v) const {
    return v < graph_state.vertex_orientations.size() ? graph_state.vertex_orientations[v] != 0 : true;
}

// OverlapGraph::checkEdge, src/OverlapGraph.cpp:233-259: the score of v->w (or, reverse_allowed, of w->v), -1 if none
double SRBuilder::checkEdge(node_id_t v, node_id_t w, bool reverse_allowed) const {
    for (const Edge& e : graph_->adj_out.at(v)) if (e.vertex2 == w) return e.score;
    if (reverse_allowed) for (const Edge& e : graph_->adj_out.at(w)) if (e.vertex2 == v) return e.score;
    return -1;
}

void SRBuilder::read_lengths(node_id_t index, unsigned long& l1, unsigned long& l2) const {
    if (!read_len1.empty()) {
        l1 = read_len1.at(index);
        l2 = read_len2.at(index);
        return;
    }
    const Read& r = fastq_->m_read_vec.at(index);
    l1 = r.seq1.size();
    l2 = r.is_paired ? r.seq2.size() : 0;
}

// The loop of :635-697 over nonedge_overlaps.txt: every overlap that is not an edge of the graph joins the stream as a
// non-edge (score 0)
void SRBuilder::append_nonedges(std::vector<hc_fno_edge>& stream) {
    const std::string path = ps_.output_dir + "nonedge_overlaps.txt";
    std::ifstream f(path.c_str());
    if (!f.is_open()) die("Unable to open non-edge overlaps file");
    if (fastq_->m_ID_to_index.empty())      // --gpu_fastq with --gpu_parse leaves the host map empty (FastqStorage)
        for (unsigned int i = 0; i < fastq_->m_read_vec.size(); i++) fastq_->m_ID_to_index.insert(std::make_pair(fastq_->m_read_vec[i].read_id, i));
    std::string line, tmp;
    std::vector<std::string> fields;
    unsigned long lines = 0, kept = 0;
    while (std::getline(f, line)) {
        lines++;
        const size_t b = line.find_first_not_of("\t "), e2 = line.find_last_not_of("\t ");
        line = b == std::string::npos ? std::string() : line.substr(b, e2 - b + 1);                          // boost::trim_if, :650
        fields.clear();
        std::stringstream ss(line);
        while (std::getline(ss, tmp, '\t')) fields.push_back(tmp);
        const Overlap ov = Overlap::from_fields(fields);
        const Read& r1 = fastq_->m_read_vec.at(fastq_->m_ID_to_index.at(ov.id1));
        const Read& r2 = fastq_->m_read_vec.at(fastq_->m_ID_to_index.at(ov.id2));
        Edge e;
        e.score = 0;
        e.pos1 = (int)ov.pos1;
        e.pos2 = (int)ov.pos2;
        e.ori1 = ov.ori1 == '+';
        e.ori2 = ov.ori2 == '+';
        e.ord = ov.ord;
        e.overlap_perc = (int)ov.get_perc();
        e.overlap_len1 = (int)ov.len1;
        e.overlap_len2 = (int)ov.len2;
        e.vertex1 = r1.vertex_id;
        e.vertex2 = r2.vertex_id;
        if (checkEdge(e.vertex1, e.vertex2, true) > 0) continue;                                               // :694-696
        stream.push_back(to_fno_edge(e));
        kept++;
    }
    nonedge_lines = lines;
    nonedge_kept = kept;
}

// What hc_fno1_text_nonedges assumes of the graph: vertex i is read i, list v holds the edges out of v (its (u, v) pairs are
// what checkEdge looks up) and every edge score is 0 (non-edge) or positive (edge)
bool SRBuilder::nonedge_device_ok() const {
    const auto& reads = fastq_->m_read_vec;
    if (graph_->adj_out.size() != reads.size()) return false;
    for (size_t i = 0; i < reads.size(); i++) if (reads[i].vertex_id != i) return false;
    for (size_t v = 0; v < graph_->adj_out.size(); v++)
        for (const Edge& e : graph_->adj_out[v]) if (e.vertex1 != v || !(e.score == 0 || e.score > 0)) return false;
    return true;
}

unsigned long SRBuilder::findNextOverlaps() {
    if (ps_.add_duplicates) die("findNextOverlaps: --add_duplicates=true is not supported by the GPU path");
    const size_t V = graph_->getVertexCount();
    if (visited.size() != V) die("findNextOverlaps: visited has not one entry per vertex");
    const double t0 = now_s();
    // ---- new reads: super-reads (single, then paired; src/FindNextOverlaps.cpp:898-913) and the flattened nodes_to_SR
    std::vector<const SuperRead*> srs;
    for (const SuperRead& r : single_SR_vec) srs.push_back(&r);
    for (const SuperRead& r : paired_SR_vec) srs.push_back(&r);
    std::vector<hc_fno_read> superread(srs.size());
    std::vector<uint64_t> sr_off(V + 1, 0);
    for (size_t k = 0; k < srs.size(); k++) {
        superread[k].id = srs[k]->read_id;
        superread[k].len1 = (uint32_t)srs[k]->len1;
        superread[k].len2 = (uint32_t)(srs[k]->is_paired ? srs[k]->len2 : 0);
        for (node_id_t node : srs[k]->sorted_clique) sr_off.at(node + 1)++;
    }
    for (size_t v = 0; v < V; v++) sr_off[v + 1] += sr_off[v];
    std::vector<uint32_t> sr_idx(sr_off[V]);
    std::vector<hc_fno_subread> sr_sub(sr_off[V]);
    {
        std::vector<uint64_t> fill(sr_off.begin(), sr_off.end() - 1);
        for (size_t k = 0; k < srs.size(); k++) {              // push_back order of :901-912 = list order per vertex
            for (node_id_t node : srs[k]->sorted_clique) {
                const uint64_t at = fill[node]++;
                sr_idx[at] = (uint32_t)k;
                const auto it = srs[k]->subread_info.find(node);
                if (it == srs[k]->subread_info.end()) die("findNextOverlaps: a super-read has no sub-read info for a vertex of its clique");
                sr_sub[at].index1 = it->second.index1;
                sr_sub[at].index2 = it->second.index2;
                sr_sub[at].startpos1 = it->second.startpos1;
                sr_sub[at].startpos2 = it->second.startpos2;
            }
        }
    }
    std::vector<uint8_t> vis(V), label(V);
    std::vector<hc_fno_read> vertex_read(V);
    for (size_t v = 0; v < V; v++) {
        vis[v] = visited[v] ? 1 : 0;
        label[v] = orientation(v) ? 1 : 0;
        unsigned long l1, l2;
        read_lengths(v, l1, l2);
        const auto it = nodes_to_new_IDs.find(v);
        vertex_read[v].id = it == nodes_to_new_IDs.end() ? ~0ull : it->second;
        vertex_read[v].len1 = (uint32_t)l1;
        vertex_read[v].len2 = (uint32_t)l2;
    }
    // ---- the edge stream in processing order: head (adjacency lists, branching edges), non-edge lines, tail
    std::vector<hc_fno_edge> stream;
    for (const auto& lst : graph_->adj_out) for (const Edge& e : lst) stream.push_back(to_fno_edge(e));       // :610-623
    const uint64_t n_adjacency = stream.size();
    for (const Edge& e : graph_state.branching_edges) stream.push_back(to_fno_edge(e));                        // :624-630
    const uint64_t n_head = stream.size();
    FileBuf nonedge_text;
    const bool nonedges_on_device = !optimize && ps_.gpu_parse && nonedge_device_ok();
    if (nonedges_on_device) {
        if (!read_whole_file(ps_.output_dir + "nonedge_overlaps.txt", nonedge_text)) die("Unable to open non-edge overlaps file");
    } else if (!optimize) {
        append_nonedges(stream);                                                                               // :635-697
    }
    std::vector<hc_fno_edge> tail;
    for (const auto& edge_list : graph_state.inclusion_edges) {                                                // :816-887
        const size_t l = edge_list.size();
        for (size_t i = 0; i < l; i++) {
            for (size_t j = i + 1; j < l; j++) {
                const Edge &e1 = edge_list[i], &e2 = edge_list[j];
                node_id_t n1, n2;
                int pos1;
                bool o1, o2;
                if (e1.vertex1 == e2.vertex1) continue;
                else if (e1.vertex1 == e2.vertex2) { n1 = e2.vertex1; n2 = e1.vertex2; pos1 = e2.pos1; o1 = e2.ori1; o2 = e1.ori2; }
                else if (e1.vertex2 == e2.vertex1) { n1 = e1.vertex1; n2 = e2.vertex2; pos1 = e1.pos1; o1 = e1.ori1; o2 = e2.ori2; }
                else continue;
                unsigned long a1, a2, b1, b2;
                read_lengths(n1, a1, a2);
                read_lengths(n2, b1, b2);
                if (a2 != 0 || b2 != 0) continue;                                     // paired-end reads: not handled (:860-862)
                const unsigned int len1 = (unsigned int)a1, len2 = (unsigned int)b1;  // Read::get_len(), src/Read.h:203-212
                const int len = (int)std::min(len1 - (unsigned int)pos1, len2);       // unsigned arithmetic as in :863
                const int perc = (int)std::floor((double)((unsigned int)(100 * len) / std::min(len1, len2)));   // :864
                Edge ne;
                ne.score = ps_.edge_threshold;
                ne.pos1 = pos1;
                ne.pos2 = 0;
                ne.ori1 = o1;
                ne.ori2 = o2;
                ne.ord = '-';
                ne.vertex1 = n1;
                ne.vertex2 = n2;
                ne.overlap_perc = perc;
                ne.overlap_len1 = len;
                ne.overlap_len2 = 0;
                if (checkEdge(n1, n2, true) == -1) tail.push_back(to_fno_edge(ne));
            }
        }
    }
    if (!nonedges_on_device) stream.insert(stream.end(), tail.begin(), tail.end());
    const double t1 = now_s();
    // ---- the derivations, on the device
    hc_fno_input in;
    std::memset(&in, 0, sizeof(in));
    in.n_vertices = V;
    in.visited = vis.data();
    in.label = label.data();
    in.vertex_read = vertex_read.data();
    in.sr_off = sr_off.data();
    in.sr_idx = sr_idx.data();
    in.sr_sub = sr_sub.data();
    in.n_superreads = superread.size();
    in.superread = superread.data();
    in.resolve_orientations = ps_.resolve_orientations ? 1 : 0;
    in.no_inclusions = no_inclusions ? 1 : 0;
    // ---- overlaps.txt, formatted, sorted and de-duplicated on the device (the reference's std::set<std::string>, :918,:946-948)
    const int dev = ps_.first_device;
    uint64_t n_records = 0, n_lines = 0;
    double t2 = 0, t_host = t1 - t0, t_call = t1;
    nonedge_on_device = false;
    nonedge_device_ms = 0;
    bool input_error = false;
    if (nonedges_on_device) {
        // the non-edge file is parsed, checked against the adjacency lists and put into the stream on the device; a line the
        // loop below would die on sends the whole file there, so that the messages stay the reference's.  If the guessed
        // text size is too small, write_text's second call repeats the whole device job (copy, parse, probe, derivations):
        // the guess of 128 bytes per stream edge and non-edge line makes that rare
        hc_idmap* idmap = fastq_->device_idmap();
        hc_fno_nonedge_stats st;
        n_lines = write_text([&](char* text, uint64_t cap, uint64_t* n_bytes, uint64_t* n_lines) {
            return hc_fno1_text_nonedges(&in, idmap, stream.data(), n_head, n_adjacency, nonedge_text.data, nonedge_text.size,
                                         tail.data(), tail.size(), text, cap, n_bytes, n_lines, &n_records, &st, dev); },
            n_head + tail.size() + nonedge_text.size / 40, ps_.output_dir + "overlaps.txt", "hc_fno1_text_nonedges", t2, &input_error);
        if (!input_error) {
            nonedge_on_device = true;
            n_stream_edges = st.n_stream;
            nonedge_lines = st.n_lines;
            nonedge_kept = st.n_nonedges;
            nonedge_device_ms = st.device_ms;
        } else {
            append_nonedges(stream);
            stream.insert(stream.end(), tail.begin(), tail.end());
        }
    }
    if (!nonedges_on_device || input_error) {
        t_call = now_s();
        t_host += t_call - t1;       // after an HC_ERR_INPUT: the device attempt and the loop count as stream time
        n_stream_edges = stream.size();
        n_lines = write_text([&](char* text, uint64_t cap, uint64_t* n_bytes, uint64_t* n_lines) {
            return hc_fno1_text(&in, stream.data(), stream.size(), text, cap, n_bytes, n_lines, &n_records, dev); },
            stream.size(), ps_.output_dir + "overlaps.txt", "hc_fno1_text", t2);
    }
    n_device_overlaps = n_records;
    t_stream_s = t_host;
    t_device_s = t2 - t_call;
    t_format_s = now_s() - t2;
    next_overlaps_count = n_lines;
    return n_lines;
}

void SRBuilder::findNextOverlaps3() {
    const double t0 = now_s();
    // ---- original read -> the new reads that contain it, built with the reference's container and insertion sequence
    // (src/FindNextOverlaps3.cpp:26-76), so that the walk below visits the originals in the reference's order (:101)
    std::vector<const SuperRead*> srs;
    for (const SuperRead& r : single_SR_vec) srs.push_back(&r);
    for (const SuperRead& r : paired_SR_vec) srs.push_back(&r);
    for (const SuperRead& r : trivial_SR_vec) srs.push_back(&r);
    std::unordered_map<read_id_t, node_id_t> original_to_index;
    std::vector<std::vector<std::pair<uint32_t, OriginalIndex>>> lists;
    for (size_t k = 0; k < srs.size(); k++) {
        for (const auto& it : srs[k]->original_reads) {
            const auto ex = original_to_index.find(it.first);
            if (ex == original_to_index.end()) {
                original_to_index.insert(std::make_pair(it.first, (node_id_t)lists.size()));
                lists.emplace_back(1, std::make_pair((uint32_t)k, it.second));
            } else {
                lists[ex->second].push_back(std::make_pair((uint32_t)k, it.second));
            }
        }
    }
    const std::unordered_map<read_id_t, node_id_t> by_value(original_to_index);    // nodeDictApproach takes the map by value (:90)
    std::vector<uint64_t> off(1, 0);
    std::vector<uint32_t> sr_idx;
    std::vector<hc_fno3_pos> sr_pos;
    for (const auto& it : by_value) {
        for (const auto& e : lists[it.second]) {
            sr_idx.push_back(e.first);
            hc_fno3_pos p;
            p.index1 = (int32_t)e.second.index1;
            p.index2 = (int32_t)e.second.index2;
            sr_pos.push_back(p);
        }
        off.push_back(sr_idx.size());
    }
    std::vector<hc_fno_read> reads(srs.size());
    for (size_t k = 0; k < srs.size(); k++) {
        reads[k].id = srs[k]->read_id;
        reads[k].len1 = (uint32_t)srs[k]->len1;
        reads[k].len2 = (uint32_t)(srs[k]->is_paired ? srs[k]->len2 : 0);
    }
    const double t1 = now_s();
    uint64_t attempts = 0;
    for (size_t o = 0; o + 1 < off.size(); o++) { const uint64_t c = off[o + 1] - off[o]; attempts += c * (c - 1) / 2; }
    // ---- overlaps.txt in discovery order, not sorted (:139-166), formatted on the device
    const int dev = ps_.first_device, noinc = no_inclusions ? 1 : 0;
    double t2 = 0;
    const uint64_t n_lines = write_text([&](char* text, uint64_t cap, uint64_t* n_bytes, uint64_t* n_lines) {
        return hc_fno3_text(off.size() - 1, off.data(), sr_idx.data(), sr_pos.data(), reads.size(), reads.data(), noinc, text, cap,
                            n_bytes, n_lines, dev); },
        attempts, ps_.output_dir + "overlaps.txt", "hc_fno3_text", t2);
    n_stream_edges = attempts;
    n_device_overlaps = n_lines;
    t_stream_s = t1 - t0;
    t_device_s = t2 - t1;
    t_format_s = now_s() - t2;
    next_overlaps_count += n_lines;
}

}  // namespace hcb
