// gkd_cli.cpp -- the `gkd` command: C++ mirror of the two reference sub-commands on the hot path,
// with the reference's option names, defaults, validation messages, headers and number format.
//
//   fastaDist  -> FastaDistanceProcessor.java  (options :66-90, validation :93-112, report :134-194)
//   genomes    -> GenomeProcessor.java         (options :54-79, validation :82-116, report :119-150)
//   fastaReps  -> FastaDistanceRepsProcessor.java (options :52-76, validation :78-91, report :110-147);
//   distReps   -> DistanceRepsProcessor.java (options :66-83, validation :154-177, run :180-275);
//                 callers of the same distance(), SURVEY section 8f "next" row 1
//
// Dispatch mirrors App.java:35-111 (args[0] selects the processor).  Reports go to stdout or -o,
// log lines to stderr (logback.xml:4-13).  Every distance comes from libgkd.so; there is no CPU path.
#include <dirent.h>
#include <sys/stat.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstring>
#include <ctime>
#include <fstream>
#include <iostream>
#include <map>
#include <memory>
#include <set>
#include <sstream>

#include "kmers.hpp"

using namespace theseed;

namespace {

void logInfo(const std::string &msg) {
    auto now = std::chrono::system_clock::now();
    std::time_t t = std::chrono::system_clock::to_time_t(now);
    auto ms = std::chrono::duration_cast<std::chrono::milliseconds>(now.time_since_epoch()).count() % 1000;
    char buf[64];
    std::strftime(buf, sizeof(buf), "%Y-%m-%d %H:%M:%S", std::localtime(&t));
    fprintf(stderr, "%s,%03d [main] %s\n", buf, (int)ms, msg.c_str());  // "%date [%thread] %msg%n"
}

std::string javaDouble(double v) {
    char buf[64];
    gkd_format_double(v, buf, sizeof(buf));
    return buf;
}

bool readable(const std::string &p) {
    std::ifstream f(p);
    return f.good();
}
bool exists(const std::string &p) {
    struct stat st;
    return stat(p.c_str(), &st) == 0;
}
bool isDir(const std::string &p) {
    struct stat st;
    return stat(p.c_str(), &st) == 0 && S_ISDIR(st.st_mode);
}

// ---- args4j-style option table -----------------------------------------------------------------
struct OptSpec {
    std::vector<std::string> names;
    bool takesValue;
    std::string usage;
};

struct Parsed {
    std::map<std::string, std::string> values;  // keyed by first name
    std::vector<std::string> positional;
};

Parsed parseOptions(const std::vector<OptSpec> &specs, const std::vector<std::string> &args) {
    Parsed out;
    for (size_t i = 0; i < args.size(); i++) {
        const std::string &a = args[i];
        if (a.size() > 1 && a[0] == '-' && !(a.size() > 1 && (isdigit((unsigned char)a[1]) || a[1] == '.'))) {
            const OptSpec *hit = nullptr;
            for (auto &s : specs)
                for (auto &n : s.names)
                    if (n == a) hit = &s;
            if (!hit) throw ParseFailureException("\"" + a + "\" is not a valid option");
            if (hit->takesValue) {
                if (i + 1 >= args.size()) throw ParseFailureException("Option \"" + a + "\" takes an operand");
                out.values[hit->names[0]] = args[++i];
            } else {
                out.values[hit->names[0]] = "true";
            }
        } else {
            out.positional.push_back(a);
        }
    }
    return out;
}

int toInt(const std::string &name, const std::string &v) {
    try {
        size_t pos = 0;
        int r = std::stoi(v, &pos);
        if (pos != v.size()) throw std::invalid_argument(v);
        return r;
    } catch (...) {
        throw ParseFailureException("\"" + v + "\" is not a valid value for \"" + name + "\"");
    }
}
double toDouble(const std::string &name, const std::string &v) {
    try {
        size_t pos = 0;
        double r = std::stod(v, &pos);
        if (pos != v.size()) throw std::invalid_argument(v);
        return r;
    } catch (...) {
        throw ParseFailureException("\"" + v + "\" is not a valid value for \"" + name + "\"");
    }
}

void printUsage(const std::string &cmd, const std::vector<OptSpec> &specs, const std::string &positional) {
    fprintf(stderr, "usage: gkd %s [options] %s\n", cmd.c_str(), positional.c_str());
    for (auto &s : specs) {
        std::string names;
        for (auto &n : s.names) names += (names.empty() ? "" : ", ") + n;
        fprintf(stderr, "  %-34s %s\n", names.c_str(), s.usage.c_str());
    }
}

// ---- fastaDist -----------------------------------------------------------------------------------
const std::vector<OptSpec> FASTA_OPTS = {
    {{"--input", "-i"}, true, "input FASTA file (if not STDIN)"},
    {{"--kSize", "--kmerSize", "-K"}, true, "kmer size to use; 0 for sequence type default"},
    {{"--batch", "-b"}, true, "batch size for kmer cache and parallelism"},
    {{"--type"}, true, "input sequence type"},
    {{"--output", "-o"}, true, "output file for report (if not STDOUT)"},
    {{"--device"}, true, "CUDA device ordinal (additive option; default 0)"},
    {{"--gpus"}, true, "number of GPUs to shard the pair matrix over (additive option; default 1; needs --input)"},
    {{"--devices"}, true, "explicit comma-separated device ordinals for the group, e.g. 0,1,2,3 (an ordinal may repeat)"},
    {{"--metrics"}, true, "write one JSON line of engine metrics to this file (additive option)"},
    {{"--maxDist"}, true, "report only the pairs with distance <= this (additive option; selected on the GPU)"},
    {{"--nearest"}, true, "report each record's N (1..256) nearest other records within --maxDist (default 1.0), in "
                          "input order, nearest first; a pair can appear twice, once from each end (additive option)"},
    {{"--clusters"}, false, "report each record's single-linkage cluster at --maxDist: the label of the cluster's first "
                            "record (additive option; needs --maxDist)"},
    {{"--linkage"}, false, "report the single-linkage hierarchy up to --maxDist (default 1.0, the whole tree): one line "
                           "per merge of single-linkage agglomeration, in merge order (additive option)"},
    {{"--method"}, true, "linkage method of --linkage and --clusters: single (default), complete or average (UPGMA); a "
                         "complete or average merge line holds the two clusters' first records and the merge height "
                         "(additive option)"},
    {{"--tree"}, false, "write the neighbour-joining tree of all records as one Newick line, rooted at the midpoint of "
                        "its last edge, instead of the report (additive option)"},
    {{"--treeMethod"}, true, "tree method of --tree: nj (default, neighbour joining) or bionj (BIONJ, which weights each "
                             "join by the variances of the distances) (additive option)"},
    {{"--nni"}, false, "refine the tree of --tree by balanced minimum-evolution nearest-neighbour interchanges and give it "
                       "BME branch lengths (additive option)"},
    {{"--help", "-h"}, false, "display command-line usage"},
    {{"--verbose", "-v"}, false, "display more frequent log messages"},
};

// The sets fastaDist reports on: one context, or a group of contexts, one per device, with the pair matrix sharded over
// them (gkd_group_*).  Every report is written once, from these calls.
struct DistSource {
    std::unique_ptr<KmerEngine> engine;  // exactly one of engine and grp is set
    gkd_group *grp = nullptr;
    int gpus = 1;
    uint32_t n = 0;  // sets
    DistSource(KmerType type, int k, int device, const std::vector<int32_t> &devices)
        : gpus(devices.empty() ? 1 : (int)devices.size()) {
        if (devices.empty()) {
            engine.reset(new KmerEngine(type, k, device));
            return;
        }
        gkd_config cfg{};
        cfg.k = k;
        cfg.alphabet = (int)type;
        if (gkd_group_create(&grp, &cfg, devices.data(), (uint32_t)devices.size()) != GKD_OK)
            throw std::runtime_error(gkd_group_last_error(nullptr));
    }
    ~DistSource() {
        if (grp) gkd_group_destroy(grp);
    }
    void check(int rc) const {
        if (engine) return engine->check(rc);
        if (rc == GKD_EIO) throw IOException(gkd_group_last_error(grp));
        if (rc == GKD_EINVAL) throw ParseFailureException(gkd_group_last_error(grp));
        if (rc != GKD_OK) throw std::runtime_error(gkd_group_last_error(grp));
    }
    // every record of a FASTA file as its own set
    void addFasta(const std::string &path) {
        if (engine) n = (uint32_t)engine->addFasta(path).size();
        else check(gkd_group_add_fasta_file(grp, path.c_str(), &n));
    }
    void build() { check(engine ? gkd_build_sets(engine->raw()) : gkd_group_build(grp)); }
    const char *label(size_t i) const {
        return engine ? gkd_label(engine->raw(), (uint32_t)i) : gkd_group_label(grp, (uint32_t)i);
    }
    const char *comment(size_t i) const {
        return engine ? gkd_comment(engine->raw(), (uint32_t)i) : gkd_group_comment(grp, (uint32_t)i);
    }
    // the context whose metrics --metrics writes
    gkd_ctx *metricsCtx() const { return engine ? engine->raw() : gkd_group_member(grp, 0); }
    void allVsAll(double *dist) const {
        check(engine ? gkd_all_vs_all(engine->raw(), nullptr, dist) : gkd_group_all_vs_all(grp, nullptr, dist));
    }
    void nearest(uint32_t k, double maxDist, const gkd_neighbors &nb) const {
        check(engine ? gkd_all_vs_all_nearest(engine->raw(), n, k, maxDist, &nb)
                     : gkd_group_all_vs_all_nearest(grp, k, maxDist, &nb));
    }
    void clusters(double maxDist, uint32_t *label) const {
        check(engine ? gkd_all_vs_all_clusters(engine->raw(), n, maxDist, label, nullptr)
                     : gkd_group_all_vs_all_clusters(grp, maxDist, label, nullptr));
    }
    void linkage(double maxDist, gkd_hits &h) const {
        check(engine ? gkd_all_vs_all_linkage(engine->raw(), n, maxDist, &h) : gkd_group_all_vs_all_linkage(grp, maxDist, &h));
    }
    // The dense call; when complete linkage fails with GKD_ENOMEM before any pair was intersected (its matrix does not
    // fit in device memory), the same merges from the pairs within maxDist, whose memory grows with those pairs only
    void agglomerate(int method, double maxDist, gkd_merges &m) const {
        gkd_metrics before{}, after{};
        gkd_get_metrics(metricsCtx(), &before);
        int rc = engine ? gkd_all_vs_all_agglomerate(engine->raw(), n, method, maxDist, &m)
                        : gkd_group_all_vs_all_agglomerate(grp, method, maxDist, &m);
        gkd_get_metrics(metricsCtx(), &after);
        if (rc == GKD_ENOMEM && method == GKD_LINK_COMPLETE && after.total_pairs == before.total_pairs) {
            logInfo("The complete-linkage matrix does not fit in device memory: merging from the pairs within distance " +
                    javaDouble(maxDist) + " instead.");
            rc = engine ? gkd_all_vs_all_complete_linkage(engine->raw(), n, maxDist, &m)
                        : gkd_group_all_vs_all_complete_linkage(grp, maxDist, &m);
        }
        check(rc);
    }
    void nj(gkd_joins &j) const { check(engine ? gkd_all_vs_all_nj(engine->raw(), n, &j) : gkd_group_all_vs_all_nj(grp, &j)); }
    uint64_t bme(int start, gkd_joins &j) const {
        uint64_t swaps = 0;
        check(engine ? gkd_all_vs_all_bme(engine->raw(), n, start, &j, &swaps) : gkd_group_all_vs_all_bme(grp, start, &j, &swaps));
        return swaps;
    }
    void bionj(gkd_joins &j) const {
        check(engine ? gkd_all_vs_all_bionj(engine->raw(), n, &j) : gkd_group_all_vs_all_bionj(grp, &j));
    }
};

// one report line of fastaDist (:188-192)
void writePairLine(std::ostream &writer, std::string &line, size_t i, size_t j, double dist, const DistSource &src) {
    line.clear();
    line += src.label(i);
    line += '\t';
    line += src.comment(i);
    line += '\t';
    line += src.label(j);
    line += '\t';
    line += src.comment(j);
    line += '\t';
    line += javaDouble(dist);
    line += '\n';
    writer << line;
}

// the report lines of fastaDist (:188-192), in list order
size_t writePairs(std::ostream &writer, const std::vector<double> &dist, const DistSource &src) {
    size_t t = 0;
    std::string line;
    for (size_t i = 0; i < src.n; i++)
        for (size_t j = i + 1; j < src.n; j++, t++) writePairLine(writer, line, i, j, dist[t], src);
    writer.flush();
    return t;
}

// the lines of the full report whose distance is <= maxDist, in the same order: hits of gkd_*_within (a < b)
void writeHits(std::ostream &writer, const uint32_t *a, const uint32_t *b, const double *dist, uint64_t n,
               const DistSource &src) {
    std::string line;
    for (uint64_t t = 0; t < n; t++) writePairLine(writer, line, a[t], b[t], dist[t], src);
}

// the lines of `fastaDist --nearest`: for each record in input order its neighbours (n*k lists of gkd_*_nearest), record
// first, in ascending distance and then input order
uint64_t writeNeighbors(std::ostream &writer, uint32_t k, const uint32_t *pos, const double *dist, const uint32_t *found,
                        const DistSource &src) {
    std::string line;
    uint64_t lines = 0;
    for (size_t i = 0; i < src.n; i++)
        for (uint32_t s = 0; s < found[i]; s++, lines++) writePairLine(writer, line, i, pos[i * k + s], dist[i * k + s], src);
    writer.flush();
    return lines;
}

// the lines of `fastaDist --clusters`: every record in input order with the label of its cluster's first record
uint32_t writeClusters(std::ostream &writer, const uint32_t *cluster, const DistSource &src) {
    std::string line;
    uint32_t clusters = 0;
    writer << "seq\tname\tcluster\n";
    for (size_t i = 0; i < src.n; i++) {
        line.clear();
        line += src.label(i);
        line += '\t';
        line += src.comment(i);
        line += '\t';
        line += src.label(cluster[i]);
        line += '\n';
        writer << line;
        clusters += cluster[i] == i ? 1u : 0u;
    }
    writer.flush();
    return clusters;
}

// a Newick label: single-quoted, with any ' doubled, when it holds whitespace or one of ()[]':;,
std::string newickLabel(const char *label) {
    std::string s(label);
    if (s.find_first_of(" \t\n\v\f\r()[]':;,") == std::string::npos) return s;
    std::string q = "'";
    for (char ch : s) {
        q += ch;
        if (ch == '\'') q += '\'';
    }
    return q + "'";
}

// `fastaDist --tree`: row t of gkd_joins is the node (A:len_a,B:len_b) of the current subtrees of labels a and b; the
// last row's node is the root.  One record: its label.  No records: nothing.
void writeNewick(std::ostream &writer, const gkd_joins &j, const DistSource &src) {
    if (src.n == 0) return;
    std::vector<std::string> sub(src.n);
    for (uint32_t i = 0; i < src.n; i++) sub[i] = newickLabel(src.label(i));
    for (uint64_t t = 0; t < j.n; t++) {
        std::string node = "(" + sub[j.a[t]] + ":" + javaDouble(j.len_a[t]) + "," + sub[j.b[t]] + ":" + javaDouble(j.len_b[t]) + ")";
        sub[j.a[t]].swap(node);
        std::string().swap(sub[j.b[t]]);
    }
    writer << sub[0] << ";\n";
    writer.flush();
}

// pairs per gkd_all_vs_all_range_within call of `fastaDist --maxDist`: host memory stays O(range), not O(n^2)
constexpr uint64_t WITHIN_RANGE = 64ull << 20;

void writeMetrics(const std::string &path, const std::string &command, gkd_ctx *ctx, size_t pairs, int gpus) {
    if (path.empty()) return;
    gkd_metrics m{};
    if (ctx) gkd_get_metrics(ctx, &m);
    std::ofstream f(path);
    if (!f) throw IOException("Cannot open metrics file " + path + ".");
    char buf[1024];
    snprintf(buf, sizeof(buf),
             "{\"command\": \"%s\", \"gpus\": %d, \"pairs\": %zu, \"pack_ms\": %.3f, \"encode_ms\": %.3f, \"sort_ms\": %.3f, "
             "\"unique_ms\": %.3f, \"intersect_ms\": %.3f, \"epilogue_ms\": %.3f, \"residues_packed\": %llu, "
             "\"kmer_positions\": %llu, \"keys_unique\": %llu, \"intersect_bytes\": %llu, \"h2d_bytes\": %llu, "
             "\"d2h_bytes\": %llu, \"launches\": %llu, \"intersect_kernel\": %u, \"scope\": \"%s\"}\n",
             command.c_str(), gpus, pairs, m.pack_ms, m.encode_ms, m.sort_ms, m.unique_ms, m.total_intersect_ms, m.epilogue_ms,
             (unsigned long long)m.residues_packed, (unsigned long long)m.kmer_positions, (unsigned long long)m.keys_unique,
             (unsigned long long)m.total_intersect_bytes, (unsigned long long)m.h2d_bytes, (unsigned long long)m.d2h_bytes,
             (unsigned long long)m.launches, m.intersect_kernel, gpus > 1 ? "member 0 of the group" : "context");
    f << buf;
}

int fastaDist(const std::vector<std::string> &args) {
    Parsed p = parseOptions(FASTA_OPTS, args);
    if (p.values.count("--help")) {
        printUsage("fastaDist", FASTA_OPTS, "");
        return 0;
    }
    // setReporterDefaults (:85-90)
    std::string inFile = p.values.count("--input") ? p.values["--input"] : "";
    int kmerSize = p.values.count("--kSize") ? toInt("--kSize", p.values["--kSize"]) : 0;
    int batchSize = p.values.count("--batch") ? toInt("--batch", p.values["--batch"]) : 20;
    KmerType seqType = p.values.count("--type") ? parseKmerType(p.values["--type"]) : KmerType::DNA;
    int device = p.values.count("--device") ? toInt("--device", p.values["--device"]) : 0;
    // validateReporterParms (:93-112)
    if (kmerSize == 0) kmerSize = kmerTypeDefaultK(seqType);
    if (kmerSize < 2) throw ParseFailureException("Kmer size must be at least 2.");
    if (batchSize < 1) throw ParseFailureException("Batch size must be at least 1.");
    const bool tree = p.values.count("--tree") > 0;
    if (tree)
        for (const char *opt : {"--maxDist", "--nearest", "--clusters", "--linkage", "--method"})
            if (p.values.count(opt)) throw ParseFailureException(std::string("--tree and ") + opt + " cannot be combined.");
    bool bionj = false;
    if (p.values.count("--treeMethod")) {
        const std::string &m = p.values["--treeMethod"];
        if (m == "bionj") bionj = true;
        else if (m != "nj") throw ParseFailureException("Tree method must be nj or bionj.");
        if (!tree) throw ParseFailureException("--treeMethod needs --tree.");
    }
    const bool nni = p.values.count("--nni") > 0;
    if (nni && !tree) throw ParseFailureException("--nni needs --tree.");
    const bool within = p.values.count("--maxDist") > 0;
    const double maxDist = within ? toDouble("--maxDist", p.values["--maxDist"]) : 1.0;
    if (!(maxDist > 0.0 && maxDist <= 1.0)) throw ParseFailureException("Maximum distance must be > 0 and <= 1.");
    const int nearest = p.values.count("--nearest") ? toInt("--nearest", p.values["--nearest"]) : 0;
    if (p.values.count("--nearest") && (nearest < 1 || nearest > 256))
        throw ParseFailureException("Number of neighbors must be between 1 and 256.");
    // single linkage at the default 1.0 would put every record in one cluster
    const bool clusters = p.values.count("--clusters") > 0;
    if (clusters && !within) throw ParseFailureException("--clusters needs --maxDist.");
    if (clusters && nearest) throw ParseFailureException("--clusters and --nearest cannot be combined.");
    const bool linkage = p.values.count("--linkage") > 0;
    if (linkage && nearest) throw ParseFailureException("--linkage and --nearest cannot be combined.");
    if (linkage && clusters) throw ParseFailureException("--linkage and --clusters cannot be combined.");
    // 0 = single linkage (gkd_*_linkage / gkd_*_clusters), else a gkd_link_method
    int method = 0;
    if (p.values.count("--method")) {
        const std::string &m = p.values["--method"];
        if (m == "complete") method = GKD_LINK_COMPLETE;
        else if (m == "average") method = GKD_LINK_AVERAGE;
        else if (m != "single") throw ParseFailureException("Linkage method must be single, complete or average.");
        if (!linkage && !clusters) throw ParseFailureException("--method needs --linkage or --clusters.");
    }
    const char *typeName = seqType == KmerType::DNA ? "DNA" : (seqType == KmerType::RNA ? "RNA" : "PROT");
    if (inFile.empty()) logInfo(std::string("Reading ") + typeName + " sequences from the standard input.");
    else if (!readable(inFile)) throw IOException("Input file " + inFile + " is not found or unreadable.");
    else logInfo(std::string("Reading ") + typeName + " sequences from " + inFile + ".");
    std::ofstream ofile;
    if (p.values.count("--output")) {
        ofile.open(p.values["--output"]);
        if (!ofile) throw IOException("Cannot open output file " + p.values["--output"] + ".");
    }
    std::ostream &writer = p.values.count("--output") ? (std::ostream &)ofile : std::cout;

    int gpus = p.values.count("--gpus") ? toInt("--gpus", p.values["--gpus"]) : 1;
    std::vector<int32_t> deviceList;
    if (p.values.count("--devices")) {
        std::string item;
        for (char ch : p.values["--devices"] + ",") {
            if (ch == ',') {
                if (!item.empty()) deviceList.push_back(toInt("--devices", item));
                item.clear();
            } else item += ch;
        }
        if (deviceList.empty()) throw ParseFailureException("--devices needs at least one ordinal.");
        gpus = (int)deviceList.size();
    }
    const std::string metricsFile = p.values.count("--metrics") ? p.values["--metrics"] : "";
    if (gpus < 1) throw ParseFailureException("Number of GPUs must be at least 1.");
    // more than one GPU, or an explicit device list: the pair matrix sharded over a group, one context per device
    std::vector<int32_t> devices = deviceList;
    if (devices.empty() && gpus > 1)
        for (int d = 0; d < gpus; d++) devices.push_back(device + d);
    if (!devices.empty() && inFile.empty()) throw ParseFailureException("--gpus needs an input file (--input).");
    DistSource src(seqType, kmerSize, device, devices);
    src.addFasta(inFile.empty() ? "-" : inFile);
    logInfo(std::to_string(src.n) + " sequences read from input.");
    // runReporter (:134-165): the batch cache and the per-row parallel streams are what the engine
    // replaces; every pair i<j is computed in one batched launch and printed in list order
    if (!clusters && !tree) writer << "seq1\tname1\tseq2\tname2\tdistance\n";
    src.build();
    logInfo(std::to_string(src.n) + " sequences cached" + (src.grp ? " on " + std::to_string(src.gpus) + " GPUs" : "") +
            ". Computing distances.");
    const uint64_t n = src.n, total = n < 2 ? 0 : n * (n - 1) / 2;
    if (tree) {
        // each pair i < j is intersected once; the tree is joined on the GPU and only its n - 1 rows leave it
        const uint64_t cap = n ? n - 1 : 0;
        std::vector<uint32_t> a(cap), b(cap);
        std::vector<double> la(cap), lb(cap);
        gkd_joins j{a.data(), b.data(), la.data(), lb.data(), cap, 0};
        uint64_t swaps = 0;
        if (nni) swaps = src.bme(bionj ? GKD_TREE_BIONJ : GKD_TREE_NJ, j);
        else if (bionj) src.bionj(j);
        else src.nj(j);
        writeNewick(writer, j, src);
        if (nni)
            logInfo(std::to_string(swaps) + " balanced NNIs applied to the " + (bionj ? "BIONJ" : "neighbor-joining") + " tree" +
                    (swaps > 0 && swaps == GKD_BME_MAX_SWAPS(n) ? "; the search stopped at its cap of " + std::to_string(swaps) + " swaps." : "."));
        logInfo(std::to_string(total) + " pairs computed in 1 batches, " + std::to_string(j.n) + " joins in the " +
                (bionj ? "BIONJ" : "neighbor-joining") + " tree.");
        writeMetrics(metricsFile, "fastaDist", src.metricsCtx(), total, src.gpus);
        return 0;
    }
    if (method && (clusters || linkage)) {
        // each pair i < j is intersected once; the agglomeration runs on the GPU and only its merges (<= n - 1) leave it
        const uint64_t cap = n ? n - 1 : 0;
        std::vector<uint32_t> a(cap), b(cap), size(cap);
        std::vector<double> d(cap);
        gkd_merges m{a.data(), b.data(), d.data(), size.data(), cap, 0};
        src.agglomerate(method, maxDist, m);
        if (linkage) {
            writeHits(writer, a.data(), b.data(), d.data(), m.n, src);
            writer.flush();
            logInfo(std::to_string(total) + " pairs computed in 1 batches, " + std::to_string(m.n) + " merges up to distance " +
                    javaDouble(maxDist) + ".");
        } else {
            // the clusters at maxDist are the components of the merges; each is labelled by its first record
            std::vector<uint32_t> label(n);
            for (uint32_t i = 0; i < n; i++) label[i] = i;
            auto find = [&](uint32_t x) {
                while (label[x] != x) x = label[x];
                return x;
            };
            for (uint64_t t = 0; t < m.n; t++) label[find(b[t])] = find(a[t]);  // a < b are both roots' labels
            for (uint32_t i = 0; i < n; i++) label[i] = find(i);
            const uint32_t found = writeClusters(writer, label.data(), src);
            logInfo(std::to_string(total) + " pairs computed in 1 batches, " + std::to_string(found) + " clusters at distance " +
                    javaDouble(maxDist) + ".");
        }
        writeMetrics(metricsFile, "fastaDist", src.metricsCtx(), total, src.gpus);
        return 0;
    }
    if (clusters) {
        // each pair i < j is intersected once and linked on the GPU; only the n labels leave it
        std::vector<uint32_t> label(n);
        src.clusters(maxDist, label.data());
        const uint32_t found = writeClusters(writer, label.data(), src);
        logInfo(std::to_string(total) + " pairs computed in 1 batches, " + std::to_string(found) + " clusters at distance " +
                javaDouble(maxDist) + ".");
        writeMetrics(metricsFile, "fastaDist", src.metricsCtx(), total, src.gpus);
        return 0;
    }
    if (linkage) {
        // each pair i < j is intersected once; only the spanning forest (<= n - 1 edges) leaves the GPU
        const uint64_t cap = n ? n - 1 : 0;
        std::vector<uint32_t> a(cap), b(cap);
        std::vector<double> d(cap);
        gkd_hits h{a.data(), b.data(), nullptr, d.data(), cap, 0};
        src.linkage(maxDist, h);
        writeHits(writer, a.data(), b.data(), d.data(), h.n, src);
        writer.flush();
        logInfo(std::to_string(total) + " pairs computed in 1 batches, " + std::to_string(h.n) + " merges up to distance " +
                javaDouble(maxDist) + ".");
        writeMetrics(metricsFile, "fastaDist", src.metricsCtx(), total, src.gpus);
        return 0;
    }
    if (nearest) {
        // each pair i < j is intersected once and offered to both rows; only the n*k lists leave the GPU
        const uint32_t k = (uint32_t)nearest;
        std::vector<uint32_t> pos(n * k), found(n);
        std::vector<double> d(n * k);
        const gkd_neighbors nb{pos.data(), nullptr, d.data(), found.data()};
        src.nearest(k, maxDist, nb);
        const uint64_t lines = writeNeighbors(writer, k, pos.data(), d.data(), found.data(), src);
        logInfo(std::to_string(total) + " pairs computed in 1 batches, " + std::to_string(lines) + " neighbor lines.");
        writeMetrics(metricsFile, "fastaDist", src.metricsCtx(), total, src.gpus);
        return 0;
    }
    if (within) {
        // only the pairs within maxDist leave the GPUs
        uint64_t hits = 0;
        if (src.engine) {
            // the triangle in ranges of <= WITHIN_RANGE pairs
            const uint64_t room = std::min(total, WITHIN_RANGE);
            std::unique_ptr<uint32_t[]> a(new uint32_t[room + 1]), b(new uint32_t[room + 1]);
            std::unique_ptr<double[]> d(new double[room + 1]);
            for (uint64_t first = 0; first < total; first += WITHIN_RANGE) {
                const uint64_t cnt = std::min(WITHIN_RANGE, total - first);
                gkd_hits h{a.get(), b.get(), nullptr, d.get(), cnt, 0};
                src.check(gkd_all_vs_all_range_within(src.engine->raw(), src.n, first, cnt, maxDist, &h));
                writeHits(writer, a.get(), b.get(), d.get(), h.n, src);
                hits += h.n;
            }
        } else {
            // every member selects on its device; one call, repeated with the exact capacity if the first was short
            uint64_t cap = std::min<uint64_t>(total, WITHIN_RANGE);
            std::vector<uint32_t> a, b;
            std::vector<double> d;
            gkd_hits h{};
            for (;;) {
                a.resize(cap);
                b.resize(cap);
                d.resize(cap);
                h = gkd_hits{a.data(), b.data(), nullptr, d.data(), cap, 0};
                src.check(gkd_group_all_vs_all_within(src.grp, maxDist, &h));
                if (h.n <= cap) break;
                cap = h.n;
            }
            writeHits(writer, a.data(), b.data(), d.data(), h.n, src);
            hits = h.n;
        }
        writer.flush();
        logInfo(std::to_string(total) + " pairs computed in 1 batches, " + std::to_string(hits) + " within distance " +
                javaDouble(maxDist) + ".");
        writeMetrics(metricsFile, "fastaDist", src.metricsCtx(), total, src.gpus);
        return 0;
    }
    std::vector<double> dist(total);
    src.allVsAll(dist.data());
    const size_t t = writePairs(writer, dist, src);
    logInfo(std::to_string(t) + " pairs computed in 1 batches.");
    writeMetrics(metricsFile, "fastaDist", src.metricsCtx(), t, src.gpus);
    return 0;
}

// ---- fastaReps -----------------------------------------------------------------------------------
const std::vector<OptSpec> REPS_OPTS = {
    {{"--input", "-i"}, true, "input FASTA file (if not STDIN)"},
    {{"--kSize", "--kmerSize", "-K"}, true, "kmer size to use; 0 for sequence type default"},
    {{"--dist", "--maxDist", "-d"}, true, "maximum distance a neighbor can be from a representative"},
    {{"--type"}, true, "input sequence type"},
    {{"--output", "-o"}, true, "output file for report (if not STDOUT)"},
    {{"--device"}, true, "CUDA device ordinal (additive option; default 0)"},
    {{"--help", "-h"}, false, "display command-line usage"},
    {{"--verbose", "-v"}, false, "display more frequent log messages"},
};

int fastaReps(const std::vector<std::string> &args) {
    Parsed p = parseOptions(REPS_OPTS, args);
    if (p.values.count("--help")) {
        printUsage("fastaReps", REPS_OPTS, "");
        return 0;
    }
    // setReporterDefaults (:71-76)
    std::string inFile = p.values.count("--input") ? p.values["--input"] : "";
    int kmerSize = p.values.count("--kSize") ? toInt("--kSize", p.values["--kSize"]) : 0;
    double maxDist = p.values.count("--dist") ? toDouble("--dist", p.values["--dist"]) : 0.97;
    KmerType seqType = p.values.count("--type") ? parseKmerType(p.values["--type"]) : KmerType::DNA;
    int device = p.values.count("--device") ? toInt("--device", p.values["--device"]) : 0;
    // validateReporterParms (:79-91)
    if (kmerSize == 0) kmerSize = kmerTypeDefaultK(seqType);
    if (kmerSize < 2) throw ParseFailureException("Kmer size must be at least 2.");
    if (!inFile.empty() && !readable(inFile)) throw IOException("Input file " + inFile + " is not found or invalid.");
    std::ofstream ofile;
    if (p.values.count("--output")) {
        ofile.open(p.values["--output"]);
        if (!ofile) throw IOException("Cannot open output file " + p.values["--output"] + ".");
    }
    std::ostream &writer = p.values.count("--output") ? (std::ostream &)ofile : std::cout;

    KmerEngine engine(seqType, kmerSize, device);
    std::vector<SequenceKmers> seqs = engine.addFasta(inFile.empty() ? "-" : inFile);
    engine.build();  // every createKmers (:122) in one batched pass
    // runReporter (:110-147): a sequence becomes a representative unless some current representative
    // is within maxDist.  repMap is keyed by label, so a later representative with the same label
    // replaces the earlier one (HashMap.put, :145).
    writer << "seq\tname\n";
    std::vector<std::pair<std::string, uint32_t>> repMap;  // insertion-ordered label -> set handle
    size_t pairCount = 0;
    bool uniqueLabels = true;
    {
        std::set<std::string> seen;
        for (auto &seq : seqs) uniqueLabels = seen.insert(seq.getGenomeId()).second && uniqueLabels;
    }
    if (uniqueLabels) {
        // the whole greedy pass on the device (gkd_greedy_reps): the representative list never leaves HBM and no
        // candidate costs a host round trip
        std::vector<uint32_t> order;
        for (auto &seq : seqs) order.push_back(seq.handle());
        std::vector<uint8_t> isRep(order.size(), 0);
        engine.check(gkd_greedy_reps(engine.raw(), order.data(), (uint32_t)order.size(), maxDist, isRep.data()));
        for (size_t i = 0; i < seqs.size(); i++)
            if (isRep[i]) {
                writer << seqs[i].getGenomeId() << '\t' << seqs[i].getGenomeName() << '\n';
                repMap.emplace_back(seqs[i].getGenomeId(), seqs[i].handle());
            }
    } else {
        // duplicate labels: a later representative replaces the earlier one under the same key (HashMap.put,
        // :145), which changes who is compared -- keep the literal per-candidate loop for that case
        std::vector<uint32_t> a, b;
        std::vector<double> dist;
        for (auto &seq : seqs) {
            bool repFound = false;
            if (!repMap.empty()) {
                a.clear();
                b.clear();
                for (auto &r : repMap) {
                    a.push_back(r.second);        // repKmers.distance(seqKmers) (:128)
                    b.push_back(seq.handle());
                }
                dist.assign(a.size(), 1.0);
                engine.check(gkd_pairs(engine.raw(), a.data(), b.data(), a.size(), nullptr, dist.data()));
                pairCount += a.size();
                for (double d : dist)
                    if (d <= maxDist) repFound = true;
            }
            if (!repFound) {
                writer << seq.getGenomeId() << '\t' << seq.getGenomeName() << '\n';
                bool replaced = false;
                for (auto &r : repMap)
                    if (r.first == seq.getGenomeId()) {
                        r.second = seq.handle();
                        replaced = true;
                    }
                if (!replaced) repMap.emplace_back(seq.getGenomeId(), seq.handle());
            }
        }
    }
    writer.flush();
    logInfo(std::to_string(repMap.size()) + " representatives found for " + std::to_string(seqs.size()) + " sequences.");
    (void)pairCount;
    return 0;
}

// ---- GTO reader (GenomeSource.Type.DIR: a directory of *.gto JSON files) ---------------------------
struct JsonCursor {
    const std::string &s;
    size_t p = 0;
    explicit JsonCursor(const std::string &str) : s(str) {}
    void ws() {
        while (p < s.size() && isspace((unsigned char)s[p])) p++;
    }
    bool eat(char c) {
        ws();
        if (p < s.size() && s[p] == c) {
            p++;
            return true;
        }
        return false;
    }
    std::string str() {
        ws();
        if (p >= s.size() || s[p] != '"') throw IOException("malformed GTO: string expected");
        p++;
        std::string out;
        while (p < s.size() && s[p] != '"') {
            if (s[p] == '\\' && p + 1 < s.size()) {
                char e = s[p + 1];
                p += 2;
                switch (e) {
                case 'n': out += '\n'; break;
                case 't': out += '\t'; break;
                case 'r': out += '\r'; break;
                case 'b': out += '\b'; break;
                case 'f': out += '\f'; break;
                case 'u': {  // \uXXXX (with surrogate pairs) -> UTF-8, the bytes a Java PrintWriter would emit
                    auto hex4 = [&](size_t at, uint32_t &v) {
                        if (at + 4 > s.size()) return false;
                        v = 0;
                        for (size_t i = 0; i < 4; i++) {
                            const char h = s[at + i];
                            v <<= 4;
                            if (h >= '0' && h <= '9') v |= (uint32_t)(h - '0');
                            else if (h >= 'a' && h <= 'f') v |= (uint32_t)(h - 'a' + 10);
                            else if (h >= 'A' && h <= 'F') v |= (uint32_t)(h - 'A' + 10);
                            else return false;
                        }
                        return true;
                    };
                    uint32_t cp = 0, lo = 0;
                    if (!hex4(p, cp)) throw IOException("malformed GTO: bad \\u escape");
                    p += 4;
                    if (cp >= 0xD800 && cp < 0xDC00 && p + 6 <= s.size() && s[p] == '\\' && s[p + 1] == 'u' && hex4(p + 2, lo) &&
                        lo >= 0xDC00 && lo < 0xE000) {
                        cp = 0x10000 + ((cp - 0xD800) << 10) + (lo - 0xDC00);
                        p += 6;
                    }
                    if (cp < 0x80) out += (char)cp;
                    else if (cp < 0x800) {
                        out += (char)(0xC0 | (cp >> 6));
                        out += (char)(0x80 | (cp & 0x3F));
                    } else if (cp < 0x10000) {
                        out += (char)(0xE0 | (cp >> 12));
                        out += (char)(0x80 | ((cp >> 6) & 0x3F));
                        out += (char)(0x80 | (cp & 0x3F));
                    } else {
                        out += (char)(0xF0 | (cp >> 18));
                        out += (char)(0x80 | ((cp >> 12) & 0x3F));
                        out += (char)(0x80 | ((cp >> 6) & 0x3F));
                        out += (char)(0x80 | (cp & 0x3F));
                    }
                    break;
                }
                default: out += e;
                }
            } else out += s[p++];
        }
        p++;
        return out;
    }
    void skip() {
        ws();
        if (p >= s.size()) return;
        char c = s[p];
        if (c == '"') {
            str();
        } else if (c == '{' || c == '[') {
            char close = c == '{' ? '}' : ']';
            p++;
            if (eat(close)) return;
            do {
                if (c == '{') {
                    str();
                    if (!eat(':')) throw IOException("malformed GTO: ':' expected");
                }
                skip();
            } while (eat(','));
            if (!eat(close)) throw IOException("malformed GTO: unbalanced brackets");
        } else {
            while (p < s.size() && s[p] != ',' && s[p] != '}' && s[p] != ']' && !isspace((unsigned char)s[p])) p++;
        }
    }
};

struct GenomeData {
    std::string id, name;
    std::vector<std::string> contigs;
};

GenomeData readGto(const std::string &path) {
    std::ifstream f(path, std::ios::binary);
    if (!f) throw IOException("Cannot read genome file " + path + ".");
    std::stringstream ss;
    ss << f.rdbuf();
    std::string text = ss.str();
    JsonCursor c(text);
    GenomeData g;
    if (!c.eat('{')) throw IOException("malformed GTO " + path);
    if (!c.eat('}')) {
        do {
            std::string key = c.str();
            if (!c.eat(':')) throw IOException("malformed GTO " + path);
            if (key == "id") g.id = c.str();
            else if (key == "scientific_name") g.name = c.str();
            else if (key == "contigs") {
                if (!c.eat('[')) throw IOException("malformed GTO " + path + ": contigs is not a list");
                if (!c.eat(']')) {
                    do {
                        if (!c.eat('{')) throw IOException("malformed GTO " + path + ": contig is not an object");
                        if (!c.eat('}')) {
                            do {
                                std::string ck = c.str();
                                if (!c.eat(':')) throw IOException("malformed GTO " + path);
                                if (ck == "dna") g.contigs.push_back(c.str());
                                else c.skip();
                            } while (c.eat(','));
                            if (!c.eat('}')) throw IOException("malformed GTO " + path);
                        }
                    } while (c.eat(','));
                    if (!c.eat(']')) throw IOException("malformed GTO " + path);
                }
            } else c.skip();
        } while (c.eat(','));
    }
    return g;
}

GenomeData readFastaGenome(const std::string &path, const std::string &stem) {
    std::ifstream f(path);
    if (!f) throw IOException("Cannot read genome file " + path + ".");
    GenomeData g;
    g.id = stem;
    g.name = stem;
    std::string line;
    while (std::getline(f, line)) {
        while (!line.empty() && isspace((unsigned char)line.back())) line.pop_back();
        if (line.empty()) continue;
        if (line[0] == '>') g.contigs.emplace_back();
        else if (!g.contigs.empty()) g.contigs.back() += line;
    }
    return g;
}

// GenomeSource.Type.create(dir): genomes of a source in sorted-name order
std::vector<GenomeData> loadSource(const std::string &type, const std::string &dir) {
    std::vector<std::string> files;
    if (isDir(dir)) {
        DIR *d = opendir(dir.c_str());
        if (!d) throw IOException("Genome source \"" + dir + "\" is not readable.");
        while (dirent *e = readdir(d)) files.push_back(e->d_name);
        closedir(d);
        std::sort(files.begin(), files.end());
    } else {
        files.push_back("");
    }
    std::vector<GenomeData> out;
    for (auto &fn : files) {
        std::string path = fn.empty() ? dir : dir + "/" + fn;
        std::string base = fn.empty() ? dir.substr(dir.find_last_of('/') + 1) : fn;
        size_t dot = base.find_last_of('.');
        std::string ext = dot == std::string::npos ? "" : base.substr(dot);
        std::string stem = dot == std::string::npos ? base : base.substr(0, dot);
        if (type == "DIR") {
            if (ext != ".gto") continue;
            out.push_back(readGto(path));
        } else {
            if (ext != ".fa" && ext != ".fna" && ext != ".fasta") continue;
            out.push_back(readFastaGenome(path, stem));
        }
    }
    return out;
}

const std::vector<OptSpec> GENOME_OPTS = {
    {{"--kmerSize", "-K", "--kmer"}, true, "DNA kmer size"},
    {{"--maxDist", "-m", "--max", "--distance"}, true, "maximum acceptable distance for a neighboring genome"},
    {{"--type", "-t"}, true, "genome source type (DIR = directory of GTO files; FASTA = directory of FASTA files)"},
    {{"--output", "-o"}, true, "output file for report (if not STDOUT)"},
    {{"--device"}, true, "CUDA device ordinal (additive option; default 0)"},
    {{"--nearest"}, true, "report only the N nearest base genomes of each genome within --maxDist (additive option; 1..256)"},
    {{"--help", "-h"}, false, "display usage information"},
    {{"--verbose", "-v"}, false, "show more detail on the log"},
};

int genomes(const std::vector<std::string> &args) {
    Parsed p = parseOptions(GENOME_OPTS, args);
    if (p.values.count("--help")) {
        printUsage("genomes", GENOME_OPTS, "gtoDir gtoDir1 gtoDir2 ...");
        return 0;
    }
    // setReporterDefaults (:75-79)
    int kmerSize = p.values.count("--kmerSize") ? toInt("--kmerSize", p.values["--kmerSize"]) : 21;
    double maxDist = p.values.count("--maxDist") ? toDouble("--maxDist", p.values["--maxDist"]) : 0.9;
    std::string sourceType = p.values.count("--type") ? p.values["--type"] : "DIR";
    int device = p.values.count("--device") ? toInt("--device", p.values["--device"]) : 0;
    if (sourceType != "DIR" && sourceType != "FASTA")
        throw ParseFailureException("\"" + sourceType + "\" is not a valid value for \"--type\"");
    if (p.positional.size() < 1) throw ParseFailureException("Argument \"gtoDir\" is required");
    if (p.positional.size() < 2) throw ParseFailureException("Argument \"gtoDir1 gtoDir2 ...\" is required");
    // validateReporterParms (:82-116)
    if (kmerSize < 4) throw ParseFailureException("Kmer size cannot be less than 4.");
    logInfo("Chosen kmer size is " + std::to_string(kmerSize) + ".");
    if (maxDist <= 0.0 || maxDist > 1.0) throw ParseFailureException("Maximum distance must be > 0 and <= 1.");
    const int nearest = p.values.count("--nearest") ? toInt("--nearest", p.values["--nearest"]) : 0;
    if (p.values.count("--nearest") && (nearest < 1 || nearest > 256))
        throw ParseFailureException("Number of neighbors must be between 1 and 256.");
    const std::string baseDir = p.positional[0];
    if (!exists(baseDir)) throw IOException("Main genome source \"" + baseDir + "\" is not found.");
    for (size_t i = 1; i < p.positional.size(); i++)
        if (!exists(p.positional[i])) throw IOException("Genome source \"" + p.positional[i] + "\" is not found.");
    std::ofstream ofile;
    if (p.values.count("--output")) {
        ofile.open(p.values["--output"]);
        if (!ofile) throw IOException("Cannot open output file " + p.values["--output"] + ".");
    }
    std::ostream &writer = p.values.count("--output") ? (std::ostream &)ofile : std::cout;

    KmerEngine engine(KmerType::DNA, kmerSize, device);
    std::vector<SequenceKmers> mainKmers;
    {
        std::vector<GenomeData> base = loadSource(sourceType, baseDir);
        logInfo("Loading " + std::to_string(base.size()) + " genomes from " + baseDir + ".");
        for (auto &g : base) mainKmers.push_back(engine.genomeKmers(g.contigs, g.id, g.name));
    }
    // runReporter (:119-150): every genome of the other sources against all base genomes; the
    // maxDist option is validated but, as in the reference, never applied to the output (:143-146) -- unless
    // --nearest asks for each genome's N nearest base genomes within maxDist
    writer << "genome1\tgenome2\tdistance\n";
    std::vector<SequenceKmers> queries;
    for (size_t i = 1; i < p.positional.size(); i++) {
        logInfo("Loading genome directory " + p.positional[i] + ".");
        for (auto &g : loadSource(sourceType, p.positional[i])) queries.push_back(engine.genomeKmers(g.contigs, g.id, g.name));
    }
    engine.build();
    std::vector<uint32_t> q, r;
    for (auto &s : queries) q.push_back(s.handle());
    for (auto &s : mainKmers) r.push_back(s.handle());
    size_t compares = 0;
    if (nearest) {
        // selected on the GPU: ascending distance, ties in base load order; only the kept neighbours come back
        const uint64_t k = (uint64_t)nearest;
        std::vector<uint32_t> pos(q.size() * k), found(q.size());
        std::vector<double> nd(q.size() * k);
        engine.check(gkd_query_vs_ref_nearest(engine.raw(), q.data(), (uint32_t)q.size(), r.data(), (uint32_t)r.size(), (uint32_t)k,
                                              maxDist, 0, pos.data(), nullptr, nd.data(), found.data()));
        for (size_t qi = 0; qi < queries.size(); qi++)
            for (uint32_t i = 0; i < found[qi]; i++, compares++)
                writer << queries[qi].getGenomeId() << '\t' << mainKmers[pos[qi * k + i]].getGenomeId() << '\t'
                       << javaDouble(nd[qi * k + i]) << '\n';
        writer.flush();
        logInfo(std::to_string(compares) + " comparisons output.");
        return 0;
    }
    std::vector<double> dist;
    engine.queryVsRef(q, r, dist);
    for (size_t qi = 0; qi < queries.size(); qi++)
        for (size_t ri = 0; ri < mainKmers.size(); ri++, compares++)
            writer << queries[qi].getGenomeId() << '\t' << mainKmers[ri].getGenomeId() << '\t'
                   << javaDouble(dist[qi * mainKmers.size() + ri]) << '\n';
    writer.flush();
    logInfo(std::to_string(compares) + " comparisons output.");
    return 0;
}

// ---- distReps ------------------------------------------------------------------------------------
const std::vector<OptSpec> DISTREPS_OPTS = {
    {{"--kmerSize", "-K", "--kmer"}, true, "kmer size to use for distance computation"},
    {{"--sourceType", "--type", "-t"}, true, "type of genome sources (DIR = directory of GTO files; FASTA = directory of FASTA files)"},
    {{"--dist"}, true, "maximum distance for a representative neighborhood"},
    {{"--outDir", "-D"}, true, "output directory name"},
    {{"--clear"}, false, "erase the output directory before processing"},
    {{"--device"}, true, "CUDA device ordinal (additive option; default 0)"},
    {{"--help", "-h"}, false, "display command-line usage"},
    {{"--verbose", "-v"}, false, "display more frequent log messages"},
};

// DistanceRepsProcessor.java: pass 1 picks representatives greedily (:185-201), pass 2 assigns every
// genome to its closest representative (:220-262) and writes rep%.4f_K%d.list.tbl / .stats.tbl (:212-274)
int distReps(const std::vector<std::string> &args) {
    Parsed p = parseOptions(DISTREPS_OPTS, args);
    if (p.values.count("--help")) {
        printUsage("distReps", DISTREPS_OPTS, "inDir1 inDir2 ...");
        return 0;
    }
    // setMultiReportDefaults (:146-151)
    int kmerSize = p.values.count("--kmerSize") ? toInt("--kmerSize", p.values["--kmerSize"]) : 9;
    double maxDist = p.values.count("--dist") ? toDouble("--dist", p.values["--dist"]) : 0.97;
    std::string sourceType = p.values.count("--sourceType") ? p.values["--sourceType"] : "DIR";
    std::string outDir = p.values.count("--outDir") ? p.values["--outDir"] : "repDb";
    int device = p.values.count("--device") ? toInt("--device", p.values["--device"]) : 0;
    if (sourceType != "DIR" && sourceType != "FASTA")
        throw ParseFailureException("\"" + sourceType + "\" is not a valid value for \"--sourceType\"");
    if (p.positional.empty()) throw ParseFailureException("Argument \"inDir1 inDir2 ...\" is required");
    // validateMultiReportParms (:154-177)
    if (kmerSize < 4) throw ParseFailureException("Kmer size must be at least 4.");
    if (maxDist <= 0.0 || maxDist >= 1.0) throw ParseFailureException("Distance must be strictly between 0 and 1.");
    for (auto &d : p.positional)
        if (!exists(d)) throw IOException("Genome source " + d + " is not found.");
    if (!isDir(outDir)) {
        if (mkdir(outDir.c_str(), 0777) != 0) throw IOException("Cannot create output directory " + outDir + ".");
    } else if (p.values.count("--clear")) {
        // BaseMultiReportProcessor erases the output directory before processing when --clear is given
        logInfo("Erasing output directory " + outDir + ".");
        if (DIR *d = opendir(outDir.c_str())) {
            while (dirent *e = readdir(d)) {
                const std::string name = e->d_name;
                if (name == "." || name == "..") continue;
                const std::string path = outDir + "/" + name;
                struct stat st;
                if (stat(path.c_str(), &st) == 0 && S_ISREG(st.st_mode)) remove(path.c_str());
            }
            closedir(d);
        }
    }

    KmerEngine engine(KmerType::DNA, kmerSize, device);
    std::vector<SequenceKmers> all;
    for (auto &d : p.positional) {
        std::vector<GenomeData> src = loadSource(sourceType, d);
        logInfo(std::to_string(src.size()) + " genomes found in " + d + ".");
        for (auto &g : src) all.push_back(engine.genomeKmers(g.contigs, g.id, g.name));
    }
    logInfo(std::to_string(all.size()) + " total genomes found in all sources.");
    engine.build();
    // pass 1: a genome joins the representative set unless a current representative is within maxDist
    logInfo("Starting first pass to find representatives.");
    std::vector<size_t> reps;            // indices into `all`, in insertion order
    std::vector<char> isRep(all.size(), 0);
    {
        // x.distance(kmers) <= maxDist for any current representative x (:185-201), for every genome in turn, as one
        // device-resident pass (gkd_greedy_reps)
        std::vector<uint32_t> order;
        for (auto &g : all) order.push_back(g.handle());
        std::vector<uint8_t> flags(order.size(), 0);
        if (!order.empty())
            engine.check(gkd_greedy_reps(engine.raw(), order.data(), (uint32_t)order.size(), maxDist, flags.data()));
        for (size_t i = 0; i < all.size(); i++)
            if (flags[i]) {
                reps.push_back(i);
                isRep[i] = 1;
            }
    }
    logInfo(std::to_string(reps.size()) + " total representatives found for " + std::to_string(all.size()) + " genomes.");
    // pass 2: closest representative of every other genome in one batched call; ties keep the
    // representative met first (Result.merge keeps the left operand, :120-122; the reference walks its
    // HashMap, whose order is unspecified, so insertion order is used here)
    std::vector<uint32_t> q, r;
    std::vector<size_t> qIdx;
    for (size_t i = 0; i < all.size(); i++)
        if (!isRep[i]) {
            q.push_back(all[i].handle());
            qIdx.push_back(i);
        }
    for (size_t x : reps) r.push_back(all[x].handle());
    // the nearest representative of every genome is selected on the GPU (k = 1, ties by representative order); only
    // one distance per genome comes back
    std::vector<uint32_t> nearPos(q.size()), nearFound(q.size());
    std::vector<double> nearDist(q.size());
    if (!q.empty())
        engine.check(gkd_query_vs_ref_nearest(engine.raw(), q.data(), (uint32_t)q.size(), r.data(), (uint32_t)r.size(), 1, 1.0, 0,
                                              nearPos.data(), nullptr, nearDist.data(), nearFound.data()));
    std::vector<size_t> bestRep(all.size());
    std::vector<double> bestDist(all.size(), 0.0);
    for (size_t i = 0; i < all.size(); i++) bestRep[i] = i;
    for (size_t qi = 0; qi < qIdx.size(); qi++) {
        // reduce(NULL_RESULT, merge): start from distance 1.0 and replace only on a strictly smaller distance, so the
        // result is the first representative at the smallest distance when that is below 1.0
        double best = 1.0;
        size_t arg = reps[0];  // only kept if no distance is below 1.0, which pass 1 rules out
        if (nearFound[qi] && nearDist[qi] < best) {
            best = nearDist[qi];
            arg = reps[nearPos[qi]];
        }
        bestRep[qIdx[qi]] = arg;
        bestDist[qIdx[qi]] = best;
    }
    char prefix[64];
    snprintf(prefix, sizeof(prefix), "rep%.4f_K%d", maxDist, kmerSize);
    std::map<std::string, long> neighborCounts;
    {
        std::ofstream list(outDir + "/" + prefix + ".list.tbl");
        if (!list) throw IOException("Cannot write to " + outDir + ".");
        list << "genome_id\tgenome_name\trep_id\trep_name\tdistance\n";
        for (size_t i = 0; i < all.size(); i++) {
            const SequenceKmers &rep = all[bestRep[i]];
            list << all[i].getGenomeId() << '\t' << all[i].getGenomeName() << '\t' << rep.getGenomeId() << '\t'
                 << rep.getGenomeName() << '\t' << javaDouble(bestDist[i]) << '\n';
            neighborCounts[rep.getGenomeId()]++;
        }
    }
    logInfo(std::to_string(all.size()) + " total genomes placed.");
    {
        // CountMap.sortedCounts(): largest neighbourhood first (ties by id)
        std::vector<std::pair<std::string, long>> counts(neighborCounts.begin(), neighborCounts.end());
        std::stable_sort(counts.begin(), counts.end(), [](const auto &x, const auto &y) { return x.second > y.second; });
        std::map<std::string, std::string> names;
        for (size_t x : reps) names[all[x].getGenomeId()] = all[x].getGenomeName();
        std::ofstream stats(outDir + "/" + prefix + ".stats.tbl");
        stats << "rep_id\trep_name\tsize\n";
        for (auto &c : counts) stats << c.first << '\t' << names[c.first] << '\t' << c.second << '\n';
    }
    return 0;
}

}  // namespace

int main(int argc, char **argv) {
    if (argc < 2) {
        fprintf(stderr, "usage: gkd <fastaDist|genomes|fastaReps|distReps> [options]\n");
        return 2;
    }
    std::string command = argv[1];
    std::vector<std::string> rest(argv + 2, argv + argc);
    try {
        if (command == "fastaDist") return fastaDist(rest);
        if (command == "genomes") return genomes(rest);
        if (command == "fastaReps") return fastaReps(rest);
        if (command == "distReps") return distReps(rest);
        // App.java:104 -- IllegalArgumentException("Invalid command " + command)
        fprintf(stderr, "Invalid command %s. (gkd implements the k-mer distance hot path: fastaDist, genomes, fastaReps, distReps)\n", command.c_str());
        return 2;
    } catch (const ParseFailureException &e) {
        fprintf(stderr, "%s\n", e.what());  // BaseProcessor prints the message and the usage
        printUsage(command,
                   command == "genomes" ? GENOME_OPTS
                                        : (command == "fastaReps" ? REPS_OPTS : (command == "distReps" ? DISTREPS_OPTS : FASTA_OPTS)),
                   command == "genomes" ? "gtoDir gtoDir1 gtoDir2 ..." : (command == "distReps" ? "inDir1 inDir2 ..." : ""));
        return 1;
    } catch (const IOException &e) {
        fprintf(stderr, "%s\n", e.what());
        return 1;
    } catch (const std::exception &e) {
        fprintf(stderr, "ERROR: %s\n", e.what());
        return 3;
    }
}
