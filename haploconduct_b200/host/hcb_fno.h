// hcb_fno.h -- host-side C++ mirror of the FindNextOverlaps interfaces of the reference's SRBuilder
// (src/SRBuilder.h:120-125), written against hc_fno1_text / hc_fno3_text of include/hc_b200.h.
//
//   unsigned long SRBuilder::findNextOverlaps()     src/FindNextOverlaps.cpp:890-958
//   void          SRBuilder::findNextOverlaps3()    src/FindNextOverlaps3.cpp:20-173
//
// What stays host code here is graph code: producing the edge stream in the reference's processing order
// (adjacency lists, removed branching edges :605-631; non-edge overlaps that are not an edge :635-697; edges induced
// through removed inclusion vertices :816-887), flattening nodes_to_SR (:898-913), and for FNO3 the iteration order of
// the reference's std::unordered_map (FindNextOverlaps3.cpp:101, same container, same insertions).  The derivations
// themselves (updateOverlap / computeOverlapData, deduceOverlap) run on the device, and so does the text of
// overlaps.txt: formatted there and, for FNO1, sorted and de-duplicated like the reference's std::set<std::string>
// (:918,:946-948); the host writes the bytes it gets back.  With ps.gpu_parse the non-edge file is parsed on the device as
// well (hc_fno1_text_nonedges): the host reads it into memory and hands over the adjacency and inclusion segments of the
// stream; a line the reference would die on sends the file back to the host loop, for the reference's message.
//
// The merging step that fills the super-read vectors (mergeAlongEdges / cliquesToSuperreads) and the graph algorithms
// that fill branching_edges / inclusion_edges are not part of this path: a host that links this class keeps its own and
// hands their results over through the public members below, which carry the reference's names.
#ifndef HCB_FNO_H_
#define HCB_FNO_H_

#include <deque>
#include <list>
#include <map>
#include <memory>
#include <string>
#include <unordered_map>
#include <vector>

#include "hcb_host.h"

namespace hcb {

struct SubreadInfo { int index1 = 0, index2 = 0, startpos1 = 0, startpos2 = 0; };   // src/Types.h:77-82
struct OriginalIndex { long index1 = 0, index2 = 0; };                               // src/Types.h:84-91 (the fields FNO3 reads)

// What FindNextOverlaps reads of a new read (a super-read Read of src/Read.h): its id, type, sequence lengths, the
// vertices it was merged from (get_sorted_clique, src/Read.h:237-255), where each of them lies inside it
// (get_subread_info, :294-297) and, for FNO3, its original reads (get_original_reads, :274-276).
struct SuperRead {
    read_id_t read_id = 0;
    bool is_paired = false;
    unsigned long len1 = 0, len2 = 0;                              // len2 == 0 for a single-end super-read
    std::list<node_id_t> sorted_clique;                            // get_sorted_clique(0) resp. (1)
    std::map<node_id_t, SubreadInfo> subread_info;
    std::vector<std::pair<read_id_t, OriginalIndex>> original_reads;   // in the iteration order of the reference's map
};

// The graph state FindNextOverlaps reads besides the adjacency lists (src/OverlapGraph.h:48,70-72).
struct FnoGraphState {
    std::vector<Edge> branching_edges;                             // edges removed by tip / branch / cycle removal
    std::vector<std::vector<Edge>> inclusion_edges;                // per removed inclusion vertex
    std::vector<char> vertex_orientations;                         // getOrientation(v); empty = all forward
};

class SRBuilder {
public:
    SRBuilder(std::shared_ptr<FastqStorage> fastq, std::shared_ptr<OverlapGraph> graph, const ProgramSettings ps);

    unsigned long findNextOverlaps();      // writes <output_dir>overlaps.txt, returns the number of lines
    void findNextOverlaps3();              // writes <output_dir>overlaps.txt, adds to next_overlaps_count

    // ---- state left by the merging step, names as in src/SRBuilder.h:43-52,132
    std::deque<SuperRead> single_SR_vec, paired_SR_vec, trivial_SR_vec;
    std::map<node_id_t, read_id_t> nodes_to_new_IDs;
    std::vector<char> visited;
    FnoGraphState graph_state;
    unsigned long next_overlaps_count = 0;
    // settings FindNextOverlaps reads beyond hcb::ProgramSettings (src/Types.h:19-67)
    bool optimize = false;                 // every driver passes --optimize=false: non-edge overlaps are reconsidered
    bool no_inclusions = false;            // ProgramSettings::no_inclusions
    // paired-ness and mate lengths of the ORIGINAL reads when m_read_vec holds no sequences (--gpu_fastq)
    std::vector<uint32_t> read_len1, read_len2;
    // measurements of the last call (not in the reference): n_device_overlaps = records before de-duplication,
    // t_device_s = device call up to the text in host memory, t_format_s = writing overlaps.txt
    unsigned long n_stream_edges = 0, n_device_overlaps = 0;
    double t_stream_s = 0, t_device_s = 0, t_format_s = 0;
    // the non-edge file: lines read, lines that joined the stream, and (ps.gpu_parse) the device time of building the stream
    unsigned long nonedge_lines = 0, nonedge_kept = 0;
    double nonedge_device_ms = 0;
    bool nonedge_on_device = false;        // the last call put the non-edge lines into the stream on the device

private:
    double checkEdge(node_id_t v, node_id_t w, bool reverse_allowed) const;        // src/OverlapGraph.cpp:233-259
    bool orientation(node_id_t v) const;                                           // OverlapGraph::getOrientation
    void read_lengths(node_id_t index, unsigned long& l1, unsigned long& l2) const;
    void append_nonedges(std::vector<hc_fno_edge>& stream);                          // :635-697 on the host
    bool nonedge_device_ok() const;                                                 // the graph hc_fno1_text_nonedges assumes
    ProgramSettings ps_;
    std::shared_ptr<FastqStorage> fastq_;
    std::shared_ptr<OverlapGraph> graph_;
};

}  // namespace hcb
#endif
