// hc_fno -- command-line front end of hcb::SRBuilder::findNextOverlaps / findNextOverlaps3 (hcb_fno.h): the step of
// bin/ViralQuasispecies that writes the next iteration's overlaps.txt (src/ViralQuasispecies.cpp:452-463), on the B200
// path.  The graph algorithms and the merging step that precede it are not part of this path, so their result is read
// from a state file (one record per line, tab separated):
//   P  resolve_orientations  no_inclusions  optimize  edge_threshold  n_vertices
//   V  vertex  visited  new_id|-1  label
//   A|B|I  list  vertex1  vertex2  pos1  pos2  ord  ori1  ori2  score  perc  len1  len2
//          A = adjacency lists in order, B = OverlapGraph::branching_edges, I = inclusion_edges[list]
//   S  s|p|t  read_id  len1  len2  node:index1:index2:startpos1:startpos2 ...      a super-read (single / paired / trivial)
//   O  original_id:index1:index2 ...                                              its original reads, reference map order
// nonedge_overlaps.txt is read from, overlaps.txt written to, the output directory.  Prints one JSON summary line.
// --gpu_parse=true (FNO1): nonedge_overlaps.txt is parsed and checked against the adjacency lists on the device.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <sstream>
#include <string>
#include <vector>

#include "hcb_fno.h"

static std::vector<std::string> split(const std::string& s, char sep) {
    std::vector<std::string> out;
    std::string cur;
    std::stringstream ss(s);
    while (std::getline(ss, cur, sep)) out.push_back(cur);
    return out;
}

int main(int argc, char** argv) {
    hcb::ProgramSettings ps;
    std::string state;
    int fno = 1;
    for (int i = 1; i < argc; i++) {
        std::string a = argv[i], v;
        const size_t eq = a.find('=');
        if (eq != std::string::npos) { v = a.substr(eq + 1); a = a.substr(0, eq); }
        else if (i + 1 < argc) v = argv[++i];
        if (a == "--singles" || a == "-s") ps.singles_file = v;
        else if (a == "--paired1") ps.paired1_file = v;
        else if (a == "--paired2") ps.paired2_file = v;
        else if (a == "--output" || a == "-O") ps.output_dir = v;
        else if (a == "--state") state = v;
        else if (a == "--FNO") fno = atoi(v.c_str());
        else if (a == "--gpu_fastq") ps.gpu_fastq = v == "true" || v == "1";
        else if (a == "--gpu_parse") ps.gpu_parse = v == "true" || v == "1";     // FNO1: nonedge_overlaps.txt parsed on the device
        else { fprintf(stderr, "unknown option %s\n", a.c_str()); return 2; }
    }
    if (state.empty()) { fprintf(stderr, "No state file provided.\n"); return 1; }
    std::shared_ptr<hcb::FastqStorage> fastq(new hcb::FastqStorage(ps));
    std::shared_ptr<hcb::OverlapGraph> graph(new hcb::OverlapGraph(fastq->get_readcount()));
    for (auto& r : fastq->m_read_vec) r.vertex_id = graph->addVertex(r.read_id);   // src/ViralQuasispecies.cpp:258-263
    std::ifstream f(state.c_str());
    if (!f.is_open()) { fprintf(stderr, "cannot read %s\n", state.c_str()); return 1; }
    std::unique_ptr<hcb::SRBuilder> srb;
    hcb::SuperRead* last = nullptr;
    std::string line;
    while (std::getline(f, line)) {
        const std::vector<std::string> t = split(line, '\t');
        if (t.empty()) continue;
        if (t[0] == "P") {
            ps.resolve_orientations = atoi(t[1].c_str()) != 0;
            ps.edge_threshold = strtod(t[4].c_str(), NULL);
            srb.reset(new hcb::SRBuilder(fastq, graph, ps));
            srb->no_inclusions = atoi(t[2].c_str()) != 0;
            srb->optimize = atoi(t[3].c_str()) != 0;
            srb->graph_state.vertex_orientations.assign(graph->getVertexCount(), 1);
            if (strtoul(t[5].c_str(), NULL, 10) != graph->getVertexCount()) { fprintf(stderr, "state file and FASTQ files disagree on the number of reads\n"); return 1; }
        } else if (!srb) {
            fprintf(stderr, "state file does not start with a P record\n");
            return 1;
        } else if (t[0] == "V") {
            const unsigned long v = strtoul(t[1].c_str(), NULL, 10);
            srb->visited.at(v) = (char)atoi(t[2].c_str());
            const long nid = atol(t[3].c_str());
            if (nid >= 0) srb->nodes_to_new_IDs[v] = (hcb::read_id_t)nid;
            srb->graph_state.vertex_orientations.at(v) = (char)atoi(t[4].c_str());
        } else if (t[0] == "A" || t[0] == "B" || t[0] == "I") {
            hcb::Edge e;
            e.vertex1 = strtoul(t[2].c_str(), NULL, 10);
            e.vertex2 = strtoul(t[3].c_str(), NULL, 10);
            e.pos1 = atoi(t[4].c_str());
            e.pos2 = atoi(t[5].c_str());
            e.ord = t[6][0];
            e.ori1 = atoi(t[7].c_str()) != 0;
            e.ori2 = atoi(t[8].c_str()) != 0;
            e.score = strtod(t[9].c_str(), NULL);
            e.overlap_perc = atoi(t[10].c_str());
            e.overlap_len1 = atoi(t[11].c_str());
            e.overlap_len2 = atoi(t[12].c_str());
            e.overlap_len = e.overlap_len1 + e.overlap_len2;
            if (t[0] == "A") graph->adj_out.at(e.vertex1).push_back(e);
            else if (t[0] == "B") srb->graph_state.branching_edges.push_back(e);
            else {
                const size_t k = strtoul(t[1].c_str(), NULL, 10);
                if (srb->graph_state.inclusion_edges.size() <= k) srb->graph_state.inclusion_edges.resize(k + 1);
                srb->graph_state.inclusion_edges[k].push_back(e);
            }
        } else if (t[0] == "S") {
            hcb::SuperRead r;
            r.is_paired = t[1] == "p";
            r.read_id = strtoul(t[2].c_str(), NULL, 10);
            r.len1 = strtoul(t[3].c_str(), NULL, 10);
            r.len2 = strtoul(t[4].c_str(), NULL, 10);
            if (r.len2 != 0) r.is_paired = true;           // a trivial super-read keeps the type of its read
            for (size_t k = 5; k < t.size(); k++) {
                const std::vector<std::string> q = split(t[k], ':');
                const hcb::node_id_t node = strtoul(q[0].c_str(), NULL, 10);
                hcb::SubreadInfo si;
                si.index1 = atoi(q[1].c_str()); si.index2 = atoi(q[2].c_str());
                si.startpos1 = atoi(q[3].c_str()); si.startpos2 = atoi(q[4].c_str());
                r.sorted_clique.push_back(node);
                r.subread_info[node] = si;
            }
            std::deque<hcb::SuperRead>& dst = t[1] == "s" ? srb->single_SR_vec : (t[1] == "p" ? srb->paired_SR_vec : srb->trivial_SR_vec);
            dst.push_back(r);
            last = &dst.back();
        } else if (t[0] == "O" && last) {
            for (size_t k = 1; k < t.size(); k++) {
                const std::vector<std::string> q = split(t[k], ':');
                hcb::OriginalIndex oi;
                oi.index1 = atol(q[1].c_str());
                oi.index2 = atol(q[2].c_str());
                last->original_reads.push_back(std::make_pair((hcb::read_id_t)strtoul(q[0].c_str(), NULL, 10), oi));
            }
        }
    }
    if (!srb) { fprintf(stderr, "empty state file\n"); return 1; }
    unsigned long lines = 0;
    if (fno == 3) { srb->findNextOverlaps3(); lines = srb->next_overlaps_count; }
    else lines = srb->findNextOverlaps();
    printf("{\"fno\": %d, \"lines\": %lu, \"stream\": %lu, \"device_overlaps\": %lu, \"t_stream_s\": %.6f, \"t_device_s\": %.6f, \"t_format_s\": %.6f, "
           "\"nonedge_lines\": %lu, \"nonedge_kept\": %lu, \"nonedge_on_device\": %d, \"nonedge_device_ms\": %.3f}\n",
           fno, lines, srb->n_stream_edges, srb->n_device_overlaps, srb->t_stream_s, srb->t_device_s, srb->t_format_s,
           srb->nonedge_lines, srb->nonedge_kept, srb->nonedge_on_device ? 1 : 0, srb->nonedge_device_ms);
    return 0;
}
