// kj_cli.cpp -- `kaiju-b200`: the reference's command-line surface (src/kaiju.cpp:74-202, usage 430-451) on top of the C ABI.
//   kaiju-b200 -t nodes.dmp -f db.fmi -i reads.fastq [-j reads2.fastq] [-a mem|greedy] [-m -s -e -E -l] [-x|-X] [-o out] [-z N] [-v]
//   kaiju-b200 -M mkfmi -i db.faa -o prefix [-e 3] [-a ALPHABET] [-d N]      (index construction on the GPU)
// Output: "C\t<name>\t<taxid>\n" / "U\t<name>\t0\n" (ConsumerThread.cpp:724-739), in INPUT order.
// Host glue only: option parsing; kj_classify_files() reads FASTA/FASTQ(.gz), parses it on the device with the reference's name
// trimming (kaiju.cpp:318-335) and strip() (util.cpp:26-33), classifies and formats the output.  -z is accepted and ignored (the GPU replaces the consumer threads); -p = protein input; with -v
// all seven columns of the reference's -v output are printed (best length/score, taxon ids, accessions, fragment strings); from a device-native
// index file (no sequence names) -v prints columns 1-5.
#include <getopt.h>
#include <unistd.h>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <mutex>
#include <string>
#include <thread>
#include <vector>
#include <zlib.h>
#include <algorithm>
#include "kaiju_b200.h"

static void die(const std::string& m);

// ---- the name-reporting front-ends kaijux / kaijup (src/kaijux.cpp, kaijup.cpp, ConsumerThreadx.cpp:193-256, ConsumerThreadp.cpp:6-94) ----
// Same kernels: the index view numbers the sequences (seq_taxon[i] = i + 2 under one root), so the "taxon id set" of a read IS the set of
// matching database sequences; params.name_mode selects the front-ends' MEM list order.  The host side here is deliberately plain (a line
// reader and a formatter): these tools are not the throughput path.
namespace {
struct LineReader {
    gzFile f = nullptr; std::string buf;
    bool open(const std::string& p) { f = gzopen(p.c_str(), "rb"); if (f) gzbuffer(f, 1 << 20); return f != nullptr; }
    bool getline(std::string& out) {
        out.clear(); char tmp[1 << 16];
        for (;;) { if (!gzgets(f, tmp, sizeof tmp)) return !out.empty(); out += tmp; if (!out.empty() && out.back() == '\n') { out.pop_back(); return true; } }
    }
    int peek() { const int c = gzgetc(f); if (c >= 0) gzungetc(c, f); return c; }
    void skipline() { std::string t; getline(t); }
    ~LineReader() { if (f) gzclose(f); }
};
void strip_letters(std::string& s) { size_t o = 0; for (char c : s) if ((c >= 'A' && c <= 'Z') || (c >= 'a' && c <= 'z')) s[o++] = c; s.resize(o); }     // util.cpp:25-33
// one record (kaijux.cpp / kaiju.cpp reader rules; trim = cut the name at the first of " /\t\r")
bool next_record(LineReader& in, bool& first, bool& fastq, bool trim, bool skip_empty, const std::string& fname, std::string& name, std::string& seq) {
    std::string line;
    for (;;) { if (!in.getline(line)) return false; if (!line.empty() || !skip_empty) break; }
    if (first) { const char c = line.empty() ? 0 : line[0]; if (c == '@') fastq = true; else if (c != '>') { fprintf(stderr, "Error: Auto-detection of file type for file %s failed.\n", fname.c_str()); exit(EXIT_FAILURE); } first = false; }
    if (!line.empty()) line.erase(line.begin());
    if (trim) { const size_t n = line.find_first_of(" /\t\r"); if (n != std::string::npos) line.erase(n); }
    name = line;
    if (fastq) { in.getline(seq); in.skipline(); in.skipline(); }
    else { seq.clear(); std::string l; while (!(in.peek() == '>' || in.peek() < 0)) { in.getline(l); seq += l; } }
    strip_letters(seq);
    return true;
}
// BLOSUM62 self-scores of the 20 residues (calcScore, ConsumerThread.cpp:397-421), by letter
int self_score(char c) {
    switch (c) { case 'A': return 4; case 'R': return 5; case 'N': return 6; case 'D': return 6; case 'C': return 9; case 'Q': return 5; case 'E': return 5; case 'G': return 6; case 'H': return 8; case 'I': return 4;
                 case 'L': return 4; case 'K': return 5; case 'M': return 5; case 'F': return 6; case 'P': return 7; case 'S': return 4; case 'T': return 5; case 'W': return 11; case 'Y': return 7; case 'V': return 4; default: return 0; }
}
// ConsumerThreadp.cpp:22-63: does the protein read yield any fragment?
bool protein_has_fragment(std::string s, const kj_params& P) {
    for (char& c : s) c = (char)toupper((unsigned char)c);
    size_t start = 0; bool any = false;
    auto piece = [&](size_t b, size_t e) { if (e - b < P.min_fragment_length) return; if (P.mode == 1) { unsigned sc = 0; for (size_t i = b; i < e; i++) sc += (unsigned)self_score(s[i]); if (sc < P.min_score) return; } any = true; };
    for (size_t pos = s.find_first_not_of("ACDEFGHIKLMNPQRSTVWY"); pos != std::string::npos; pos = s.find_first_not_of("ACDEFGHIKLMNPQRSTVWY", pos + 1)) { if (pos - start >= P.min_fragment_length) piece(start, pos); start = pos + 1; }
    piece(start, s.size());
    return any;
}
int run_name_frontend(bool protein, kj_params P, const std::string& fmi_fn, const std::string& in1, const std::string& in2, const std::string& out_fn, int device) {
    kj_fmi* fmi = nullptr; if (kj_fmi_load(fmi_fn.c_str(), &fmi) != KJ_OK) die(kj_last_error());
    kj_index_view iv; kj_fmi_view(fmi, &iv);
    // sequences numbered 2.. under the root 1: the id set of a read = its matching sequences, ascending = the front-ends' output order
    std::vector<uint64_t> st((size_t)iv.nseq), node((size_t)iv.nseq + 1), parent((size_t)iv.nseq + 1, 1);
    node[0] = 1; for (int32_t i = 0; i < iv.nseq; i++) { st[(size_t)i] = (uint64_t)i + 2; node[(size_t)i + 1] = (uint64_t)i + 2; }
    iv.seq_taxon = st.data();
    kj_taxonomy_view tv; tv.n = node.size(); tv.node = node.data(); tv.parent = parent.data();
    P.name_mode = 1; P.input_is_protein = protein ? 1 : 0;
    kj_ctx* ctx = nullptr; if (kj_create(&ctx, device, &P, &iv, &tv) != KJ_OK) die(kj_last_error());
    LineReader r1, r2; const bool paired = !in2.empty();
    if (!r1.open(in1)) die("Could not open file " + in1);
    if (paired && !r2.open(in2)) die("Could not open file " + in2);
    FILE* out = out_fn.empty() ? stdout : fopen(out_fn.c_str(), "w"); if (!out) die("Could not open file " + out_fn + " for writing");
    bool first1 = true, first2 = true, fq1 = false, fq2 = false; const uint32_t m = P.min_fragment_length;
    std::vector<std::string> names; std::string s1, s2; std::vector<uint64_t> o1{0}, o2{0}; std::vector<uint8_t> gate;      // gate: 1 = "U\tname\t0"
    auto flush = [&]() {
        const size_t n = names.size(); if (!n) return;
        std::vector<uint64_t> tax(n), ids(n * KJ_MAX_MATCH_IDS); std::vector<uint32_t> best(n); std::vector<uint8_t> nids(n);
        if (kj_classify_verbose(ctx, s1.data(), o1.data(), paired ? s2.data() : nullptr, paired ? o2.data() : nullptr, n, tax.data(), best.data(), ids.data(), nids.data()) != KJ_OK) die(kj_last_error());
        for (size_t i = 0; i < n; i++) {
            if (gate[i]) { fprintf(out, "U\t%s\t0\n", names[i].c_str()); continue; }
            if (!tax[i] || !nids[i]) { fprintf(out, "U\t%s\n", names[i].c_str()); continue; }
            fprintf(out, "C\t%s\t%u\t", names[i].c_str(), best[i]);
            for (uint8_t k = 0; k < nids[i]; k++) fprintf(out, "%s,", kj_fmi_seq_name(fmi, (int32_t)(ids[i * KJ_MAX_MATCH_IDS + k] - 2)));
            fprintf(out, "\t\n");
        }
        names.clear(); s1.clear(); s2.clear(); o1.assign(1, 0); o2.assign(1, 0); gate.clear();
    };
    std::string name, seq, name2, seq2;
    while (next_record(r1, first1, fq1, !protein, !protein, in1, name, seq)) {
        if (paired) {
            if (!next_record(r2, first2, fq2, true, true, in2, name2, seq2)) die("File " + in1 + " contains more reads then file " + in2);
            if (name != name2) die("Error: Read names are not identical between the two input files. Probably reads are not in the same order in both files.");
        }
        bool g;
        if (protein) g = seq.size() < m || !protein_has_fragment(seq, P);                                     // ConsumerThreadp.cpp:16-20, 66-70
        else g = (!paired && seq.size() < 3u * m) || (paired && seq.size() < 3u * m && seq2.size() < 3u * m);    // ConsumerThreadx.cpp:202-207
        names.push_back(name); gate.push_back(g ? 1 : 0); s1 += seq; o1.push_back(s1.size());
        if (paired) { s2 += seq2; o2.push_back(s2.size()); }
        if (names.size() >= (1u << 18)) flush();
    }
    flush();
    if (out != stdout) fclose(out);
    kj_destroy(ctx); kj_fmi_free(fmi);
    return EXIT_SUCCESS;
}
// `kaiju -v`: all seven columns (ConsumerThread.cpp:527-536, 614-623: best, taxon ids, accessions, fragment strings).  A debugging output in the
// reference too; here it takes the host-side reader and kj_classify_verbose2 rather than the device-side text pipeline.
int run_verbose(kj_ctx* ctx, kj_fmi* fmi, const kj_params& P, const std::string& in1, const std::string& in2, const std::string& out_fn, uint64_t& n_reads, uint64_t& n_class) {
    LineReader r1, r2; const bool paired = !in2.empty(); const bool protein = P.input_is_protein != 0;
    if (!r1.open(in1)) die("Could not open file " + in1);
    if (paired && !r2.open(in2)) die("Could not open file " + in2);
    FILE* out = out_fn.empty() ? stdout : fopen(out_fn.c_str(), "w"); if (!out) die("Could not open file " + out_fn + " for writing");
    bool first1 = true, first2 = true, fq1 = false, fq2 = false;
    std::vector<std::string> names; std::string s1, s2; std::vector<uint64_t> o1{0}, o2{0}; size_t maxlen = 0;
    auto flush = [&]() {
        const size_t n = names.size(); if (!n) return;
        const uint32_t stride = (uint32_t)(32u * ((protein ? maxlen : maxlen / 3u) + 2u) + 64u);
        std::vector<uint64_t> tax(n), ids(n * KJ_MAX_MATCH_IDS); std::vector<uint32_t> best(n), acc(n * KJ_MAX_MATCH_ACC), flen(n); std::vector<uint8_t> nids(n), nacc(n); std::vector<char> frag(n * (size_t)stride);
        if (kj_classify_verbose2(ctx, s1.data(), o1.data(), paired ? s2.data() : nullptr, paired ? o2.data() : nullptr, n, tax.data(), best.data(), ids.data(), nids.data(),
                                 acc.data(), nacc.data(), frag.data(), stride, flen.data()) != KJ_OK) die(kj_last_error());
        for (size_t i = 0; i < n; i++) {
            if (!tax[i]) { fprintf(out, "U\t%s\t0\n", names[i].c_str()); continue; }
            n_class++;
            fprintf(out, "C\t%s\t%llu\t%u\t", names[i].c_str(), (unsigned long long)tax[i], best[i]);
            for (uint8_t k = 0; k < nids[i]; k++) fprintf(out, "%llu,", (unsigned long long)ids[i * KJ_MAX_MATCH_IDS + k]);
            fputc('\t', out);
            for (uint8_t k = 0; k < nacc[i]; k++) fprintf(out, "%s,", kj_fmi_accession(fmi, acc[i * KJ_MAX_MATCH_ACC + k]));
            fputc('\t', out);
            fwrite(frag.data() + i * (size_t)stride, 1, flen[i], out);
            fputc('\n', out);
        }
        n_reads += n; names.clear(); s1.clear(); s2.clear(); o1.assign(1, 0); o2.assign(1, 0); maxlen = 0;
    };
    std::string name, seq, name2, seq2;
    while (next_record(r1, first1, fq1, true, true, in1, name, seq)) {
        if (paired) {
            if (!next_record(r2, first2, fq2, true, true, in2, name2, seq2)) die("File " + in1 + " contains more reads then file " + in2);
            if (name != name2) die("Read names are not identical between the two input files. Probably reads are not in the same order in both files.");
        }
        names.push_back(name); s1 += seq; o1.push_back(s1.size()); maxlen = std::max(maxlen, seq.size());
        if (paired) { s2 += seq2; o2.push_back(s2.size()); maxlen = std::max(maxlen, seq2.size()); }
        if (names.size() >= (1u << 17)) flush();
    }
    flush();
    if (out != stdout) fclose(out);
    return EXIT_SUCCESS;
}
}  // namespace

static void die(const std::string& m) { fprintf(stderr, "Error: %s\n\n", m.c_str()); exit(EXIT_FAILURE); }
// -M mkfmi: protein FASTA -> <prefix>.fmi on the GPU (kj_mkfmi), what `kaiju-mkbwt -a ALPHABET -e E -o prefix db.faa` + `kaiju-mkfmi prefix`
// write; with -w (and -t) the new index is also transcoded into a device-native index file.  Exit status 1 on any error.
static int run_mkfmi(const std::string& in, const std::string& prefix, const char* a_arg, const char* e_arg, const std::string& dev,
                     const std::string& nodes_fn, const std::string& native_out) {
    if (in.empty() || prefix.empty()) die("-M mkfmi needs the protein FASTA (-i) and the output prefix (-o)");
    if (!native_out.empty() && nodes_fn.empty()) die("-w after -M mkfmi needs nodes.dmp (-t)");
    kj_mkfmi_opts o; memset(&o, 0, sizeof o);
    o.chpt_exp = 3; o.alphabet = a_arg;
    if (e_arg) { char* end = nullptr; const long v = strtol(e_arg, &end, 10); if (!*e_arg || *end || v < 0 || v > 16) die("-e (suffix array sampling exponent) must be 0..16"); o.chpt_exp = (int32_t)v; }
    char* end = nullptr; const long d = strtol(dev.c_str(), &end, 10);
    if (dev.empty() || *end || d < 0) die("-M mkfmi takes one device number (-d N)");
    kj_mkfmi_stats st;
    if (kj_mkfmi(in.c_str(), prefix.c_str(), &o, (int)d, &st) != KJ_OK) die(kj_last_error());
    fprintf(stderr, "%s.fmi: %lld rows, %d sequences, %d sort rounds; %.1f ms parse, %.1f ms upload, %.1f ms sort, %.1f ms assembly, %.1f ms write\n",
            prefix.c_str(), (long long)st.bwtlen, st.nseq, st.sort_rounds, st.parse_ms, st.upload_ms, st.sort_ms, st.assemble_ms, st.write_ms);
    if (!native_out.empty()) {
        kj_fmi* fmi = nullptr; kj_nodes* nodes = nullptr;
        if (kj_nodes_load(nodes_fn.c_str(), &nodes) != KJ_OK || kj_fmi_load((prefix + ".fmi").c_str(), &fmi) != KJ_OK) die(kj_last_error());
        kj_index_view iv; kj_taxonomy_view tv; kj_fmi_view(fmi, &iv); kj_nodes_view(nodes, &tv);
        if (kj_native_index_write(&iv, &tv, native_out.c_str()) != KJ_OK) die(kj_last_error());
        kj_fmi_free(fmi); kj_nodes_free(nodes);
    }
    return EXIT_SUCCESS;
}
static void usage(const char* prog) {
    fprintf(stderr, "kaiju-b200 (B200-native classification path of Kaiju)\n\nUsage:\n   %s -t nodes.dmp -f kaiju_db.fmi -i reads.fastq [-j reads2.fastq]\n\n"
                    "Mandatory arguments:\n   -t FILENAME   Name of nodes.dmp file\n   -f FILENAME   Name of database (.fmi) file\n   -i FILENAME   Name of input file containing reads in FASTA or FASTQ format\n\n"
                    "Optional arguments:\n   -j FILENAME   Name of second input file for paired-end reads\n   -o FILENAME   Name of output file. If not specified, output will be printed to STDOUT\n"
                    "   -z INT        accepted for compatibility (ignored: the GPU replaces the worker threads)\n   -a STRING     Run mode, either \"mem\"  or \"greedy\" (default: greedy)\n"
                    "   -e INT        Number of mismatches allowed in Greedy mode (default: 3)\n   -m INT        Minimum match length (default: 11)\n   -s INT        Minimum match score in Greedy mode (default: 65)\n"
                    "   -E FLOAT      Minimum E-value in Greedy mode (default: 0.01)\n   -x            Enable SEG low complexity filter (enabled by default)\n   -X            Disable SEG low complexity filter\n"
                    "   -w FILENAME   Write the device-native index file for -t/-f and exit; such a file can then be given as -f (no -t needed, no transcode at start-up)\n   -T FILENAME   Also write kaiju2table's summary (reads per taxon of rank -r, default species; needs -N names.dmp) from the counts kept on the GPU\n   -p            Input sequences are protein sequences\n   -v            Enable verbose output (adds the match length/score, the matching taxon ids, accession numbers and fragment sequences)\n   -M STRING     front-end: \"kaijux\" (as kaiju, but reports the names of the matching database sequences; no -t) or \"kaijup\" (the same for protein reads),\n                 or \"mkfmi\": build the index <-o>.fmi from the protein FASTA -i on the GPU, as kaiju-mkbwt + kaiju-mkfmi do (no -f; -e = suffix\n                 array sampling exponent, default 3; -a = alphabet, default ACDEFGHIKLMNPQRSTVWY, or \"protein\"; -w FILE -t nodes.dmp also writes a native index)\n   -d LIST       CUDA device ordinal(s): one number, a comma-separated list, or \"all\" (default 0).  With several devices the data sets of the\n                 -i/-j/-o lists are classified in parallel, one context (index replica) per device\n", prog);
    exit(EXIT_FAILURE);
}

int main(int argc, char** argv) {
    kj_params P; P.mode = 1; P.min_fragment_length = 11; P.mismatches = 3; P.min_score = 65; P.seed_length = 7; P.use_evalue = 1; P.min_evalue = 0.01; P.seg = 1; P.input_is_protein = 0; P.name_mode = 0;
    std::string nodes_fn, fmi_fn, in1, in2, out_fn, native_out, table_fn, table_rank = "species", names_fn; bool verbose = false; std::string device_arg = "0", frontend; int c;
    const char* a_arg = nullptr; const char* e_arg = nullptr;       // -a / -e: run mode and mismatches, or with -M mkfmi alphabet and SA exponent
    while ((c = getopt(argc, argv, "a:hd:pxXvn:m:e:E:l:t:f:i:j:s:z:o:w:T:r:N:M:")) != -1) {
        switch (c) {
            case 'a': a_arg = optarg; break;
            case 'h': usage(argv[0]); break;
            case 'd': device_arg = optarg; break;
            case 'v': verbose = true; break;
            case 'p': P.input_is_protein = 1; break;
            case 'x': P.seg = 1; break;
            case 'X': P.seg = 0; break;
            case 'o': out_fn = optarg; break;
            case 'w': native_out = optarg; break;
            case 'T': table_fn = optarg; break;
            case 'r': table_rank = optarg; break;
            case 'N': names_fn = optarg; break;
            case 'f': fmi_fn = optarg; break;
            case 't': nodes_fn = optarg; break;
            case 'i': in1 = optarg; break;
            case 'j': in2 = optarg; break;
            case 'l': { int v = atoi(optarg); if (v < 7) { die("Seed length must be >= 7."); } P.seed_length = (uint32_t)v; break; }
            case 's': { int v = atoi(optarg); if (v <= 0) die("Min Score (-s) must be greater than 0."); P.min_score = (uint32_t)v; break; }
            case 'm': { int v = atoi(optarg); if (v <= 0) die("Min fragment length (-m) must be greater than 0."); P.min_fragment_length = (uint32_t)v; break; }
            case 'e': e_arg = optarg; break;
            case 'E': { P.min_evalue = atof(optarg); if (P.min_evalue <= 0.0) die("E-value threshold must be greater than 0."); break; }
            case 'z': { if (atoi(optarg) <= 0) die("Number of threads (-z) must be greater than 0."); break; }
            case 'n': break;
            case 'M': frontend = optarg; break;
            default: usage(argv[0]);
        }
    }
    if (frontend == "mkfmi") return run_mkfmi(in1, out_fn, a_arg, e_arg, device_arg, nodes_fn, native_out);
    if (a_arg) { if (!strcmp(a_arg, "mem")) { P.mode = 0; P.use_evalue = 0; } else if (!strcmp(a_arg, "greedy")) P.mode = 1; else { fprintf(stderr, "-a must be a valid mode.\n"); usage(argv[0]); } }
    if (e_arg) { int v = atoi(e_arg); if (v < 0) die("Number of mismatches must be >= 0."); P.mismatches = (uint32_t)v; }
    if (fmi_fn.empty()) { fprintf(stderr, "Error: Please specify the location of the FMI file, using the -f option.\n\n"); usage(argv[0]); }
    { const char* b = strrchr(argv[0], '/'); const std::string prog = b ? b + 1 : argv[0]; if (frontend.empty() && (prog == "kaijux" || prog == "kaijup")) frontend = prog; }
    if (!frontend.empty()) {      // -M kaijux | kaijup (or invoked under that name): report the names of the matching database sequences, no taxonomy
        if (frontend != "kaijux" && frontend != "kaijup") die("-M must be kaijux, kaijup or mkfmi");
        if (in1.empty()) { fprintf(stderr, "Error: Please specify the location of the input file, using the -i option.\n\n"); usage(argv[0]); }
        if (frontend == "kaijup" && !in2.empty()) die("kaijup takes one input file");
        return run_name_frontend(frontend == "kaijup", P, fmi_fn, in1, in2, out_fn, atoi(device_arg.c_str()));
    }
    // -f may name a device-native index file (written with -w): it holds the taxonomy too, so -t is not needed then
    bool native_in = false;
    { FILE* f = fopen(fmi_fn.c_str(), "rb"); char m[8] = {0}; if (f) { native_in = fread(m, 1, 8, f) == 8 && memcmp(m, "KJB200IX", 8) == 0; fclose(f); } }
    if (nodes_fn.empty() && !native_in) { fprintf(stderr, "Error: Please specify the location of the nodes.dmp file, using the -t option.\n\n"); usage(argv[0]); }
    if (!native_out.empty()) {              // -w FILE: transcode .fmi + nodes.dmp into the device-native index file and exit (no GPU needed)
        if (native_in) die("-w needs the reference's .fmi as -f");
        kj_fmi* fmi = nullptr; kj_nodes* nodes = nullptr;
        if (kj_nodes_load(nodes_fn.c_str(), &nodes) != KJ_OK || kj_fmi_load(fmi_fn.c_str(), &fmi) != KJ_OK) die(kj_last_error());
        kj_index_view iv; kj_taxonomy_view tv; kj_fmi_view(fmi, &iv); kj_nodes_view(nodes, &tv);
        if (kj_native_index_write(&iv, &tv, native_out.c_str()) != KJ_OK) die(kj_last_error());
        kj_fmi_free(fmi); kj_nodes_free(nodes);
        return EXIT_SUCCESS;
    }
    if (in1.empty()) { fprintf(stderr, "Error: Please specify the location of the input file, using the -i option.\n\n"); usage(argv[0]); }
    const bool paired = !in2.empty();
    if (paired && P.input_is_protein) { fprintf(stderr, "Error: Protein input only supports one input file.\n\n"); usage(argv[0]); }      // kaiju.cpp:201

    auto split = [](const std::string& v) { std::vector<std::string> out; size_t b = 0; while (b <= v.size()) { size_t e = v.find(',', b); if (e == std::string::npos) e = v.size(); if (e > b) out.push_back(v.substr(b, e - b)); b = e + 1; } return out; };
    const std::vector<std::string> l1 = split(in1), l2 = split(in2), lo = split(out_fn);
    if (l1.empty()) die("Please specify the location of the input file, using the -i option.");
    if (paired && l2.size() != l1.size()) die("Length of input file lists differ");                      // kaiju-multi.cpp:255-258
    if (!lo.empty() && lo.size() != l1.size()) die("Length of input and output file lists differ");
    if (lo.empty() && l1.size() > 1) die("Several input files need a list of output files (-o)");

    // devices: one context (index replica) per device; the data sets of the lists are handed out to whichever device is free
    std::vector<int> devices;
    if (device_arg == "all") { const int nd = kj_device_count(); if (nd <= 0) die("no CUDA device available (this program has no CPU fallback)"); for (int d = 0; d < nd; d++) devices.push_back(d); }
    else for (const std::string& t : split(device_arg)) devices.push_back(atoi(t.c_str()));
    if (devices.empty()) devices.push_back(0);
    if (devices.size() > l1.size()) devices.resize(l1.size());                                           // no more contexts than data sets
    if (!table_fn.empty() && (names_fn.empty() || nodes_fn.empty())) die("The summary table (-T) needs names.dmp (-N) and nodes.dmp (-t).");

    kj_fmi* fmi = nullptr; kj_nodes* nodes = nullptr; kj_index_view iv; kj_taxonomy_view tv;
    if (!native_in) {
        if (kj_nodes_load(nodes_fn.c_str(), &nodes) != KJ_OK) die(kj_last_error());
        if (kj_fmi_load(fmi_fn.c_str(), &fmi) != KJ_OK) die(kj_last_error());
        kj_fmi_view(fmi, &iv); kj_nodes_view(nodes, &tv);
    }
    std::vector<kj_ctx*> ctxs(devices.size(), nullptr);
    {
        std::vector<std::thread> th; std::mutex mu; std::string err;
        for (size_t d = 0; d < devices.size(); d++) th.emplace_back([&, d] {
            const int rc = native_in ? kj_create_from_native(&ctxs[d], devices[d], &P, fmi_fn.c_str()) : kj_create(&ctxs[d], devices[d], &P, &iv, &tv);
            if (rc != KJ_OK) { std::lock_guard<std::mutex> lk(mu); if (err.empty()) err = kj_last_error(); }
        });
        for (auto& x : th) x.join();
        if (!err.empty()) die(err);
    }
    if (fmi && !verbose) { kj_fmi_free(fmi); fmi = nullptr; }      // -v prints accession strings: the loader's names stay
    if (nodes) kj_nodes_free(nodes);

    // parsing, classification and output formatting all run on the device; the host moves bytes (kj_ingest.h).
    // Comma-separated lists for -i / -j / -o process several data sets against the index loaded once per device (kaiju-multi.cpp:220-330).
    struct Done { uint64_t n_reads = 0, n_classified = 0; double secs = 0; std::vector<uint64_t> ids, counts; };
    std::vector<Done> done(l1.size()); std::atomic<size_t> next(0); std::mutex mu; std::string err;
    std::vector<std::thread> workers;
    for (size_t d = 0; d < ctxs.size(); d++) workers.emplace_back([&, d] {
        for (;;) {
            const size_t k = next.fetch_add(1); if (k >= l1.size()) return;
            { std::lock_guard<std::mutex> lk(mu); if (!err.empty()) return; }
            Done& r = done[k]; kj_ctx* ctx = ctxs[d]; int rc = KJ_OK;
            if (!table_fn.empty()) rc = kj_counts_reset(ctx);
            const auto t0 = std::chrono::steady_clock::now();
            if (rc == KJ_OK && verbose && fmi) run_verbose(ctx, fmi, P, l1[k], paired ? l2[k] : std::string(), lo.empty() ? std::string() : lo[k], r.n_reads, r.n_classified);
            else if (rc == KJ_OK) rc = kj_classify_files(ctx, l1[k].c_str(), paired ? l2[k].c_str() : nullptr, lo.empty() ? nullptr : lo[k].c_str(), verbose ? 1 : 0, &r.n_reads, &r.n_classified);
            r.secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
            if (rc == KJ_OK && !table_fn.empty()) { r.ids.resize(kj_counts_size(ctx)); r.counts.resize(r.ids.size()); rc = kj_counts_get(ctx, r.ids.data(), r.counts.data()); }
            if (rc != KJ_OK) { std::lock_guard<std::mutex> lk(mu); if (err.empty()) err = kj_last_error(); return; }
        }
    });
    for (auto& x : workers) x.join();
    if (!err.empty()) die(err);
    for (size_t k = 0; k < l1.size(); k++) {
        if (!table_fn.empty()) {     // kaiju2table's report from the per-taxon counts kept in HBM (one block of rows per data set, in list order)
            kj_table_opts to; memset(&to, 0, sizeof to); to.rank = table_rank.c_str();
            const std::string label = lo.empty() ? l1[k] : lo[k];
            if (kj_table_write(done[k].ids.data(), done[k].counts.data(), done[k].ids.size(), nodes_fn.c_str(), names_fn.c_str(), label.c_str(), &to, table_fn.c_str(), k > 0) != KJ_OK) die(kj_last_error());
        }
        if (verbose || getenv("KJ_CLI_TIMING")) fprintf(stderr, "%s: %llu reads, %llu classified, %.4f s from the first byte read to the last byte written\n", l1[k].c_str(), (unsigned long long)done[k].n_reads, (unsigned long long)done[k].n_classified, done[k].secs);
    }
    for (kj_ctx* ctx : ctxs) kj_destroy(ctx);
    if (fmi) kj_fmi_free(fmi);
    return EXIT_SUCCESS;
}
