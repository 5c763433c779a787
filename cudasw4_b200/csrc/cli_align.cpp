// align - drop-in for the reference's search CLI (reference src/main.cu:98-426, src/options.cpp:47-267): same options,
// same plain / TSV result formats, same console messages, driving the B200 engine through the cudasw4::CudaSW4 facade
// (include/cudasw4.cuh -> C ABI -> libsw4b200.so). The GPUs used are all visible ones (CUDA_VISIBLE_DEVICES).
// Unlike the shipped reference binary, --gop/--gex (and the per-matrix defaults) really reach the kernels
// (SURVEY.md 0-1), and the database is always uploaded in full (--uploadFull is accepted and implied).
#include <algorithm>
#include <cctype>
#include <cerrno>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <memory>
#include <sstream>
#include <string>
#include <vector>

#include "blosum_tables.hpp"
#include "cudasw4.cuh"
#include "fasta_reader.hpp"

namespace {

struct Options {
    enum class Output { Plain, TSV };
    bool help = false, uploadFull = false, pseudo = false, printPartitions = false, interactive = false, verbose = false,
         prefetchFile = false, coordinates = false, cigar = false, evalue = false;
    double maxEvalue = INFINITY;  // extension: --maxEvalue (implies --evalue)
    // extension: iterative profile search (--iterations, --inclusionEvalue) and the final PSSMs (--outPssm PREFIX)
    int iterations = 1;
    double inclusionEvalue = 0.002;
    std::string outPssm;
    bool iterative() const { return iterations > 1 || !outPssm.empty(); }
    int top = 10, gop = -11, gex = -1, pseudoLen = 0;
    int batchQueries = 1;  // extension: queries handed to one scanMany call (1 = one scan per query, as the reference)
    size_t pseudoNum = 0;
    cudasw4::BlosumType blosum = cudasw4::BlosumType::BLOSUM62_20;
    cudasw4::KernelTypeConfig kernels;
    cudasw4::MemoryConfig mem;
    Output output = Output::Plain;
    std::string outfile = "/dev/stdout", db;
    std::vector<std::string> queries;
    std::vector<std::string> pssmFiles;  // extension: --pssm, PSI-BLAST ASCII PSSM files (one query each)
};

// One PSSM query: the residue letters of its rows and the [length][21] scores (column 20: the --mat table's `low`).
struct PssmQuery {
    std::string path, letters;
    std::vector<std::int8_t> scores;
};

// PSI-BLAST's ASCII PSSM (-out_ascii_pssm). The header line starts with the 20 letters A R N D C Q E G H I L K M F P S T
// W Y V in this order. Each row that follows is "pos letter s1 ... s20 ...", positions 1, 2, ... without gaps; tokens
// after the 20 scores are ignored. The first line that is not a row ends the matrix.
PssmQuery readAsciiPssm(const std::string& path, int low) {
    std::ifstream in(path);
    if (!in) throw std::runtime_error("cannot open PSSM file " + path);
    static const char* kOrder = "ARNDCQEGHILKMFPSTWYV";
    auto bad = [&](const std::string& why) { return std::runtime_error("PSSM file " + path + ": " + why); };
    auto integer = [](const std::string& t, long& v) {
        if (t.empty()) return false;
        char* end = nullptr;
        errno = 0;
        v = std::strtol(t.c_str(), &end, 10);
        return *end == '\0' && errno == 0;
    };
    PssmQuery q;
    q.path = path;
    std::string line;
    bool header = false;
    while (std::getline(in, line)) {  // the header: the first line that starts with 20 one-letter tokens
        std::istringstream ls(line);
        std::vector<std::string> t;
        for (std::string w; ls >> w;) t.push_back(w);
        if (t.size() < 20 || !std::all_of(t.begin(), t.begin() + 20, [](const std::string& w) {
                return w.size() == 1 && std::isalpha((unsigned char)w[0]);
            }))
            continue;
        for (int k = 0; k < 20; k++)
            if (t[k] != std::string(1, kOrder[k])) throw bad("the header's residue order is not A R N D C Q E G H I L K M F P S T W Y V");
        header = true;
        break;
    }
    if (!header) throw bad("no header line with the residue letters");
    while (std::getline(in, line)) {
        std::istringstream ls(line);
        std::vector<std::string> t;
        for (std::string w; ls >> w;) t.push_back(w);
        long pos = 0;
        if (t.empty() || !integer(t[0], pos)) break;  // not a row: the end of the matrix
        const long want = (long)q.letters.size() + 1;
        if (pos != want) throw bad("row " + t[0] + " where row " + std::to_string(want) + " was expected");
        if (t.size() < 22 || t[1].size() != 1) throw bad("row " + t[0] + " is not 'position letter' and 20 scores");
        q.letters.push_back(t[1][0]);
        for (int k = 0; k < 20; k++) {
            long v = 0;
            if (!integer(t[2 + k], v)) throw bad("row " + t[0] + ": score '" + t[2 + k] + "' is not an integer");
            if (v < -128 || v > 127) throw bad("row " + t[0] + ": score " + t[2 + k] + " is outside [-128, 127]");
            q.scores.push_back((std::int8_t)v);
        }
        q.scores.push_back((std::int8_t)low);
    }
    if (q.letters.empty()) throw bad("no rows");
    return q;
}

size_t parseMemory(const std::string& s) {
    if (s.empty()) return 0;
    size_t factor = 1;
    std::string num = s;
    switch (s.back()) {
        case 'K': factor = size_t(1) << 10; num.pop_back(); break;
        case 'M': factor = size_t(1) << 20; num.pop_back(); break;
        case 'G': factor = size_t(1) << 30; num.pop_back(); break;
        default: break;
    }
    return factor * std::stoull(num);
}

cudasw4::KernelType parseKernelType(const std::string& s) {
    if (s == "Half2") return cudasw4::KernelType::Half2;
    if (s == "DPXs16") return cudasw4::KernelType::DPXs16;
    if (s == "DPXs32") return cudasw4::KernelType::DPXs32;
    if (s == "Float") return cudasw4::KernelType::Float;
    throw std::runtime_error("unknown kernel type " + s);
}

bool parseArgs(int argc, char** argv, Options& o) {
    bool gotQuery = false, gotDB = false, gotGop = false, gotGex = false, dpx = false, gotIterationOption = false;
    auto need = [&](int& i) -> std::string {
        if (i + 1 >= argc) throw std::runtime_error(std::string("missing value for ") + argv[i]);
        return argv[++i];
    };
    for (int i = 1; i < argc; i++) {
        const std::string a = argv[i];
        if (a == "--help") o.help = true;
        else if (a == "--uploadFull") o.uploadFull = true;
        else if (a == "--verbose") o.verbose = true;
        else if (a == "--interactive") o.interactive = true;
        else if (a == "--batchQueries" && i + 1 < argc) o.batchQueries = std::max(1, std::atoi(argv[++i]));
        else if (a == "--printLengthPartitions") o.printPartitions = true;
        else if (a == "--prefetchDBFile") o.prefetchFile = true;
        else if (a == "--top") o.top = std::atoi(need(i).c_str());
        else if (a == "--gop") { o.gop = std::atoi(need(i).c_str()); gotGop = true; }
        else if (a == "--gex") { o.gex = std::atoi(need(i).c_str()); gotGex = true; }
        else if (a == "--maxBatchBytes") o.mem.maxBatchBytes = parseMemory(need(i));
        else if (a == "--maxBatchSequences") o.mem.maxBatchSequences = (size_t)std::atoll(need(i).c_str());
        else if (a == "--maxTempBytes") o.mem.maxTempBytes = parseMemory(need(i));
        else if (a == "--maxGpuMem") o.mem.maxGpuMem = parseMemory(need(i));
        else if (a == "--query") { o.queries.push_back(need(i)); gotQuery = true; }
        else if (a == "--pssm") o.pssmFiles.push_back(need(i));
        else if (a == "--db") { o.db = need(i); gotDB = true; }
        else if (a == "--mat") {
            const std::string v = need(i);
            if (v == "blosum45" || v == "blosum45_20") o.blosum = cudasw4::BlosumType::BLOSUM45_20;
            if (v == "blosum50" || v == "blosum50_20") o.blosum = cudasw4::BlosumType::BLOSUM50_20;
            if (v == "blosum62" || v == "blosum62_20") o.blosum = cudasw4::BlosumType::BLOSUM62_20;
            if (v == "blosum80" || v == "blosum80_20") o.blosum = cudasw4::BlosumType::BLOSUM80_20;
        }
        else if (a == "--singlePassType") o.kernels.singlePassType = parseKernelType(need(i));
        else if (a == "--manyPassType_small") o.kernels.manyPassType_small = parseKernelType(need(i));
        else if (a == "--manyPassType_large") o.kernels.manyPassType_large = parseKernelType(need(i));
        else if (a == "--overflowType") o.kernels.overflowType = parseKernelType(need(i));
        else if (a == "--pseudodb") { o.pseudo = true; o.pseudoNum = (size_t)std::atoll(need(i).c_str()); o.pseudoLen = std::atoi(need(i).c_str()); gotDB = true; }
        else if (a == "--dpx") dpx = true;
        else if (a == "--tsv") o.output = Options::Output::TSV;
        else if (a == "--coordinates") o.coordinates = true;
        else if (a == "--cigar") o.cigar = true;
        else if (a == "--evalue") o.evalue = true;
        else if (a == "--maxEvalue") {
            const std::string v = need(i);
            char* end = nullptr;
            o.maxEvalue = std::strtod(v.c_str(), &end);
            if (v.empty() || *end != '\0' || !(o.maxEvalue >= 0)) throw std::runtime_error("--maxEvalue needs a number >= 0, got " + v);
            o.evalue = true;
        }
        else if (a == "--iterations") {
            const std::string v = need(i);
            char* end = nullptr;
            const long n = std::strtol(v.c_str(), &end, 10);
            if (v.empty() || *end != '\0' || n < 1 || n > 1000000) throw std::runtime_error("--iterations needs an integer >= 1, got " + v);
            o.iterations = (int)n;
            gotIterationOption = true;
        }
        else if (a == "--inclusionEvalue") {
            const std::string v = need(i);
            char* end = nullptr;
            o.inclusionEvalue = std::strtod(v.c_str(), &end);
            if (v.empty() || *end != '\0' || !(o.inclusionEvalue >= 0)) throw std::runtime_error("--inclusionEvalue needs a number >= 0, got " + v);
            gotIterationOption = true;
        }
        else if (a == "--outPssm") { o.outPssm = need(i); gotIterationOption = true; }
        else if (a == "--of") o.outfile = need(i);
        else std::cout << "Unexpected arg " << a << "\n";
    }
    // matrix-dependent default gap scores (reference src/options.cpp:178-194, Readme.md:83-88)
    const int m = cudasw4::blosumNumber(o.blosum);
    const int dgop = (m == 45 || m == 50) ? -13 : (m == 62 ? -11 : -10);
    const int dgex = (m == 45 || m == 50) ? -2 : -1;
    if (!gotGop) o.gop = dgop;
    if (!gotGex) o.gex = dgex;
    if (dpx) {
        o.kernels.singlePassType = cudasw4::KernelType::DPXs16;
        o.kernels.manyPassType_small = cudasw4::KernelType::DPXs16;
        o.kernels.manyPassType_large = cudasw4::KernelType::DPXs32;
        o.kernels.overflowType = cudasw4::KernelType::DPXs32;
    }
    if (gotQuery && !o.pssmFiles.empty()) throw std::runtime_error("--query and --pssm cannot be combined");
    if (gotIterationOption && !o.pssmFiles.empty())
        throw std::runtime_error("--iterations, --inclusionEvalue and --outPssm start from a --query sequence; they cannot be combined with --pssm");
    if (!gotQuery && o.pssmFiles.empty() && !o.interactive) { std::cout << "Query is missing\n"; return false; }
    if (!gotDB) { std::cout << "DB prefix is missing\n"; return false; }
    return true;
}

void printHelp(const char* prog) {
    std::cout << "Usage: " << prog << " [options]\n"
              << "The GPUs to use are set via CUDA_VISIBLE_DEVICES environment variable.\n"
              << "   --query queryfile : Mandatory. Fasta or Fastq, may be gzip'ed. Repeatable.\n"
              << "   --pssm file : (extension) instead of --query: a PSI-BLAST ASCII PSSM (-out_ascii_pssm) scores the query.\n"
              << "                 Repeatable; the files are numbered as the queries of one query file.\n"
              << "   --db dbPrefix : Mandatory. The same dbPrefix as used for makedb\n"
              << "   --top val : Output the val best scores. Default 10\n"
              << "   --gop val, --gex val : Gap open / extend score. Overwrite the blosum-dependent defaults.\n"
              << "   --mat val : blosum45, blosum50, blosum62 (default), blosum80\n"
              << "   --maxGpuMem val, --maxTempBytes val, --maxBatchBytes val, --maxBatchSequences val : memory limits (K,M,G)\n"
              << "   --dpx : DPX kernel accounting (all kernels of this engine are DPX integer kernels)\n"
              << "   --of file : Result output file. Default /dev/stdout\n"
              << "   --tsv : tab-separated output\n"
              << "   --coordinates : (extension) also print where each hit aligns: 1-based query and reference begin and end\n"
              << "   --cigar : (extension) also print how each hit aligns: length, identities, positives, gaps and CIGAR\n"
              << "   --evalue : (extension) also print each hit's E-value and bit score, fitted to the query's own scores (NA:\n"
              << "              too few subjects to fit)\n"
              << "   --maxEvalue val : (extension) implies --evalue; report only the hits with E-value <= val\n"
              << "   --iterations n : (extension) iterative profile search: up to n rounds of scan, profile of the hits with\n"
              << "                    E-value <= --inclusionEvalue, scan with that profile. Reports the last round. Default 1\n"
              << "   --inclusionEvalue val : (extension) E-value a hit needs to enter the next round's profile. Default 0.002\n"
              << "   --outPssm prefix : (extension) write each query's last profile to prefix.<query number>.pssm, in the\n"
              << "                      ASCII format --pssm reads\n"
              << "   --verbose, --printLengthPartitions, --interactive, --help\n"
              << "   --batchQueries n : (extension) scan n queries of a file with several scans in flight per GPU; same results\n"
              << "   --prefetchDBFile, --uploadFull, --pseudodb num length\n"
              << "   --singlePassType, --manyPassType_small, --manyPassType_large, --overflowType : Half2, DPXs16, DPXs32, Float\n";
}

void printOptions(const Options& o) {
    std::cout << "Selected options:\n"
              << "verbose: " << o.verbose << "\n" << "interactive: " << o.interactive << "\n"
              << "loadFullDBToGpu: " << o.uploadFull << "\n" << "prefetchDBFile: " << o.prefetchFile << "\n"
              << "numTopOutputs: " << o.top << "\n" << "gop: " << o.gop << "\n" << "gex: " << o.gex << "\n"
              << "maxBatchBytes: " << o.mem.maxBatchBytes << "\n" << "maxBatchSequences: " << o.mem.maxBatchSequences << "\n"
              << "maxTempBytes: " << o.mem.maxTempBytes << "\n";
    for (size_t i = 0; i < o.queries.size(); i++) std::cout << "queryFile " << i << " : " << o.queries[i] << "\n";
    for (size_t i = 0; i < o.pssmFiles.size(); i++) std::cout << "pssmFile " << i << " : " << o.pssmFiles[i] << "\n";
    std::cout << "blosum: " << cudasw4::to_string_nodim(o.blosum) << "\n"
              << "singlePassType: " << cudasw4::to_string(o.kernels.singlePassType) << "\n"
              << "manyPassType_small: " << cudasw4::to_string(o.kernels.manyPassType_small) << "\n"
              << "manyPassType_large: " << cudasw4::to_string(o.kernels.manyPassType_large) << "\n"
              << "overflowType: " << cudasw4::to_string(o.kernels.overflowType) << "\n";
    if (o.pseudo) std::cout << "Using built-in pseudo db with " << o.pseudoNum << " sequences of length " << o.pseudoLen << "\n";
    else std::cout << "Using db file: " << o.db << "\n";
    std::cout << "memory limit per gpu: "
              << (o.mem.maxGpuMem == std::numeric_limits<size_t>::max() ? std::string("unlimited") : std::to_string(o.mem.maxGpuMem)) << "\n"
              << "Output mode: " << (o.output == Options::Output::Plain ? "Plain" : "TSV") << "\n"
              << "Output file: " << o.outfile << "\n";
}

// result printers: formats of reference src/main.cu:34-87 and 243-245. With --coordinates (`coords` non-empty, one
// entry per hit) every line also carries where the hit aligns, 1-based inclusive as in BLAST (0 = no alignment); with
// --cigar (`alignments` non-empty) how it aligns: length, identities, positives, gaps and the CIGAR; with --evalue
// (`stats` not null) its E-value and bit score.
std::string formatNumber(double v) {
    char buf[32];
    snprintf(buf, sizeof(buf), "%.6g", v);
    return buf;
}
std::string evalueText(const cudasw4::ScoreStatistics& st, int score) { return st.ok ? formatNumber(st.evalue(score)) : "NA"; }
std::string bitScoreText(const cudasw4::ScoreStatistics& st, int score) { return st.ok ? formatNumber(st.bitScore(score)) : "NA"; }

void printPlain(std::ostream& os, const cudasw4::ScanResult& r, const cudasw4::CudaSW4& sw,
                const std::vector<cudasw4::AlignmentCoordinates>& coords, const std::vector<cudasw4::Alignment>& alignments,
                const cudasw4::ScoreStatistics* stats) {
    for (size_t i = 0; i < r.scores.size(); i++) {
        const auto id = r.referenceIds[i];
        os << "Result " << i << "." << " Score: " << r.scores[i] << "." << " Length: " << sw.getReferenceLength(id) << "."
           << " Header " << sw.getReferenceHeader(id) << "." << " referenceId " << id;
        if (!coords.empty()) {
            const auto& c = coords[i];
            os << " Query " << c.queryBegin + 1 << "-" << c.queryEnd + 1 << ". Reference " << c.referenceBegin + 1 << "-"
               << c.referenceEnd + 1 << ".";
        }
        if (!alignments.empty()) {
            const auto& a = alignments[i];
            os << " Identities " << a.identities << "/" << a.length << ". Positives " << a.positives << "/" << a.length
               << ". Gaps " << a.gaps << "/" << a.length << ". CIGAR " << a.cigar << ".";
        }
        if (stats) os << " E-value " << evalueText(*stats, r.scores[i]) << ". Bit score " << bitScoreText(*stats, r.scores[i]) << ".";
        os << "\n";
    }
}
void printTSVHeader(std::ostream& os, bool coordinates, bool cigar, bool evalue) {
    os << "Query number\tQuery length\tQuery header\tResult number\tResult score\tReference length\tReference header\t"
          "Reference ID in DB";
    if (coordinates) os << "\tQuery begin\tQuery end\tReference begin\tReference end";
    if (cigar) os << "\tAlignment length\tIdentities\tPositives\tGaps\tCIGAR";
    if (evalue) os << "\tE-value\tBit score";
    os << "\n";
}
void printTSV(std::ostream& os, const cudasw4::ScanResult& r, const cudasw4::CudaSW4& sw, int64_t qnum, size_t qlen,
              const std::string& qheader, const std::vector<cudasw4::AlignmentCoordinates>& coords,
              const std::vector<cudasw4::Alignment>& alignments, const cudasw4::ScoreStatistics* stats) {
    for (size_t i = 0; i < r.scores.size(); i++) {
        const auto id = r.referenceIds[i];
        os << qnum << '\t' << qlen << '\t' << qheader << '\t' << i << '\t' << r.scores[i] << '\t' << sw.getReferenceLength(id)
           << '\t' << sw.getReferenceHeader(id) << '\t' << id;
        if (!coords.empty()) {
            const auto& c = coords[i];
            os << '\t' << c.queryBegin + 1 << '\t' << c.queryEnd + 1 << '\t' << c.referenceBegin + 1 << '\t' << c.referenceEnd + 1;
        }
        if (!alignments.empty()) {
            const auto& a = alignments[i];
            os << '\t' << a.length << '\t' << a.identities << '\t' << a.positives << '\t' << a.gaps << '\t' << a.cigar;
        }
        if (stats) os << '\t' << evalueText(*stats, r.scores[i]) << '\t' << bitScoreText(*stats, r.scores[i]);
        os << "\n";
    }
}

// (pssm: the query's [length][21] scores, or nullptr for a sequence query; scanIndex: the query's index in the scan call
// that produced r, for its score statistics)
void reportQuery(const Options& o, cudasw4::CudaSW4& sw, std::ostream& out, int64_t qnum, const std::string& header,
                 const std::string& sequence, const std::int8_t* pssm, const cudasw4::ScanResult& r, int scanIndex);

// --outPssm: the ASCII PSSM that readAsciiPssm reads back unchanged (column 20 is the table's `low` on both sides)
void writeAsciiPssm(const std::string& path, const std::string& letters, const std::vector<std::int8_t>& pssm) {
    std::ofstream f(path);
    if (!f) throw std::runtime_error("cannot write PSSM file " + path);
    f << "Last position-specific scoring matrix computed\n        ";
    for (const char* c = "ARNDCQEGHILKMFPSTWYV"; *c; c++) f << "   " << *c;
    f << "\n";
    for (size_t p = 0; p < letters.size(); p++) {
        char buf[32];
        snprintf(buf, sizeof(buf), "%5zu %c ", p + 1, std::isgraph((unsigned char)letters[p]) ? letters[p] : 'X');
        f << buf;
        for (int a = 0; a < 20; a++) {
            snprintf(buf, sizeof(buf), "%4d", (int)pssm[p * 21 + a]);
            f << buf;
        }
        f << "\n";
    }
    if (!f) throw std::runtime_error("cannot write PSSM file " + path);
}

// --iterations / --outPssm: one query's rounds (one at a time, also under --batchQueries), reported as its last scan
void processQueryIterative(const Options& o, cudasw4::CudaSW4& sw, std::ostream& out, int64_t qnum, const std::string& header,
                           const std::string& sequence) {
    std::cout << "Processing query " << qnum << " ... ";
    std::cout.flush();
    const cudasw4::IterativeSearchResult it = sw.searchIterative(sequence.data(), (int)sequence.size(), o.iterations, o.inclusionEvalue);
    if (!o.outPssm.empty()) writeAsciiPssm(o.outPssm + "." + std::to_string(qnum) + ".pssm", sequence, it.pssm);
    reportQuery(o, sw, out, qnum, header, sequence, it.pssm.data(), it.result, 0);
    std::cout << "Query " << qnum << ": " << it.iterations << (it.iterations == 1 ? " round, " : " rounds, ")
              << (it.converged ? "converged" : "not converged") << "\n";
}

void processQuery(const Options& o, cudasw4::CudaSW4& sw, std::ostream& out, int64_t qnum, const std::string& header,
                  const std::string& sequence, const std::int8_t* pssm = nullptr) {
    if (o.iterative() && !pssm) return processQueryIterative(o, sw, out, qnum, header, sequence);
    std::cout << "Processing query " << qnum << " ... ";
    std::cout.flush();
    cudasw4::ScanResult r = pssm ? sw.scan(sequence.data(), pssm, (int)sequence.size()) : sw.scan(sequence.data(), (int)sequence.size());
    reportQuery(o, sw, out, qnum, header, sequence, pssm, r, 0);
}

// --batchQueries: the queries go through one scanMany call; output is written in query order exactly as above
// (pssms: empty for sequence queries, else one per query)
void processQueryBatch(const Options& o, cudasw4::CudaSW4& sw, std::ostream& out, int64_t firstQnum,
                       const std::vector<std::string>& headers, const std::vector<std::string>& sequences,
                       const std::vector<const std::int8_t*>& pssms = {}) {
    std::vector<std::string_view> views(sequences.begin(), sequences.end());
    const std::vector<cudasw4::ScanResult> results = pssms.empty() ? sw.scanMany(views) : sw.scanMany(views, pssms);
    for (size_t i = 0; i < results.size(); i++) {
        std::cout << "Processing query " << firstQnum + (int64_t)i << " ... ";
        reportQuery(o, sw, out, firstQnum + (int64_t)i, headers[i], sequences[i], pssms.empty() ? nullptr : pssms[i], results[i],
                    (int)i);
    }
}

void reportQuery(const Options& o, cudasw4::CudaSW4& sw, std::ostream& out, int64_t qnum, const std::string& header,
                 const std::string& sequence, const std::int8_t* pssm, const cudasw4::ScanResult& r, int scanIndex) {
    if (o.verbose) std::cout << "Done. Scan time: " << r.stats.seconds << " s, " << r.stats.gcups << " GCUPS\n";
    else std::cout << "Done.\n";
    if (o.top > 0) {
        cudasw4::ScoreStatistics stats{};
        if (o.evalue) stats = sw.lastScoreStatistics(scanIndex);
        std::vector<cudasw4::AlignmentCoordinates> coords;
        std::vector<cudasw4::Alignment> alignments;
        if (o.cigar && !r.referenceIds.empty()) {  // the traceback reports the coordinates too
            alignments = pssm ? sw.computeAlignments(sequence.data(), pssm, (int)sequence.size(), r.referenceIds)
                              : sw.computeAlignments(sequence.data(), (int)sequence.size(), r.referenceIds);
            if (o.coordinates)
                for (const auto& a : alignments) coords.push_back(a.coordinates);
        } else if (o.coordinates && !r.referenceIds.empty()) {
            coords = pssm ? sw.computeAlignmentCoordinates(sequence.data(), pssm, (int)sequence.size(), r.referenceIds)
                          : sw.computeAlignmentCoordinates(sequence.data(), (int)sequence.size(), r.referenceIds);
        }
        if (o.output == Options::Output::Plain) {
            out << "Query " << qnum << ", header" << header << ", length " << sequence.size() << ", num overflows "
                << r.stats.numOverflows << "\n";
            printPlain(out, r, sw, coords, alignments, o.evalue ? &stats : nullptr);
        } else {
            printTSV(out, r, sw, qnum, sequence.size(), header, coords, alignments, o.evalue ? &stats : nullptr);
        }
        out.flush();
    }
}

}  // namespace

int main(int argc, char** argv) {
    Options o;
    try {
        if (!parseArgs(argc, argv, o) || o.help) { printHelp(argv[0]); return 0; }
        // every PSSM file is read before any GPU work, so that a malformed one fails at once
        std::vector<PssmQuery> pssmQueries;
        for (const auto& f : o.pssmFiles) {
            int low = 0;
            for (const auto& t : sw4::kSubstitutionTriangles)
                if (t.id == cudasw4::blosumNumber(o.blosum)) low = t.low;
            pssmQueries.push_back(readAsciiPssm(f, low));
        }
        printOptions(o);
        std::ofstream out(o.outfile);
        if (!out) throw std::runtime_error("Cannot open file " + o.outfile);
        if (o.output == Options::Output::TSV) printTSVHeader(out, o.coordinates, o.cigar, o.evalue);

        cudasw4::CudaSW4 sw({}, o.top, o.blosum, o.kernels, o.mem, o.verbose);  // {} = all visible GPUs
        sw.setGapOpenScore(o.gop);
        sw.setGapExtendScore(o.gex);
        if (o.evalue || o.iterative()) sw.setScoreStatistics(true, o.maxEvalue);  // the rounds need the E-values
        if (!o.pseudo) {
            if (o.verbose) std::cout << "Reading Database: \n";
            sw.setDatabase(std::make_shared<cudasw4::DB>(cudasw4::loadDB(o.db, false, o.prefetchFile)));
        } else {
            if (o.verbose) std::cout << "Generating pseudo db\n";
            sw.setDatabase(std::make_shared<cudasw4::PseudoDB>(cudasw4::loadPseudoDB(o.pseudoNum, o.pseudoLen)));
        }
        if (o.verbose) {
            sw.printDBInfo();
            if (o.printPartitions) sw.printDBLengthPartitions();
        }
        sw.prefetchDBToGpus();

        if (!o.pssmFiles.empty()) {  // the PSSM files are the queries of one query file, header = the path
            std::cout << "Processing PSSM queries\n";
            sw.totalTimerStart();
            for (size_t q0 = 0; q0 < pssmQueries.size(); q0 += (size_t)o.batchQueries) {
                const size_t q1 = std::min(pssmQueries.size(), q0 + (size_t)o.batchQueries);
                if (o.batchQueries <= 1) {
                    const PssmQuery& q = pssmQueries[q0];
                    processQuery(o, sw, out, (int64_t)q0, q.path, q.letters, q.scores.data());
                    continue;
                }
                std::vector<std::string> headers, sequences;
                std::vector<const std::int8_t*> pssms;
                for (size_t i = q0; i < q1; i++) {
                    headers.push_back(pssmQueries[i].path);
                    sequences.push_back(pssmQueries[i].letters);
                    pssms.push_back(pssmQueries[i].scores.data());
                }
                processQueryBatch(o, sw, out, (int64_t)q0, headers, sequences, pssms);
            }
            const auto total = sw.totalTimerStop();
            if (o.verbose) std::cout << "Total time: " << total.seconds << " s, " << total.gcups << " GCUPS\n";
        } else if (!o.interactive) {
            for (const auto& qf : o.queries) {
                std::cout << "Processing query file " << qf << "\n";
                sw4::SequenceFileReader reader(qf);
                int64_t qnum = 0;
                sw.totalTimerStart();
                if (o.batchQueries <= 1 || o.iterative()) {
                    while (reader.next()) {
                        processQuery(o, sw, out, qnum, reader.getCurrentHeader(), reader.getCurrentSequence());
                        qnum++;
                    }
                } else {
                    std::vector<std::string> headers, sequences;
                    bool more = true;
                    while (more) {
                        headers.clear();
                        sequences.clear();
                        while ((int)sequences.size() < o.batchQueries && (more = reader.next())) {
                            headers.push_back(reader.getCurrentHeader());
                            sequences.push_back(reader.getCurrentSequence());
                        }
                        if (!sequences.empty()) processQueryBatch(o, sw, out, qnum, headers, sequences);
                        qnum += (int64_t)sequences.size();
                    }
                }
                const auto total = sw.totalTimerStop();
                if (o.verbose) std::cout << "Total time: " << total.seconds << " s, " << total.gcups << " GCUPS\n";
            }
        } else {  // reference src/main.cu:336-424: read sequences from stdin until "exit"
            std::cout << "Interactive mode ready\nUse 's inputsequence' to query inputsequence against the database. Press ENTER twice to begin.\n"
                         "Use 'f inputfile' to query all sequences in inputfile\nUse 'exit' to terminate\nWaiting for command...\n";
            std::string line;
            int64_t qnum = 0;
            while (std::getline(std::cin, line)) {
                if (line == "exit") break;
                if (line.size() > 2 && line[0] == 's' && line[1] == ' ') {
                    processQuery(o, sw, out, qnum++, "", line.substr(2));
                } else if (line.size() > 2 && line[0] == 'f' && line[1] == ' ') {
                    sw4::SequenceFileReader reader(line.substr(2));
                    while (reader.next()) processQuery(o, sw, out, qnum++, reader.getCurrentHeader(), reader.getCurrentSequence());
                } else if (!line.empty()) {
                    std::cout << "Unrecognized command: " << line << "\n";
                }
                std::cout << "Waiting for command...\n";
            }
        }
    } catch (const std::exception& e) {
        std::cerr << "Error: " << e.what() << "\n";
        return 1;
    }
    return 0;
}
