// decompress <compressed_file> <reference_file> <output_folder>
// Drop-in for the reference's decompression.cpp main (:281-330): `7z e`, reference FASTA read, then the record
// decode (decompress_genome's in-memory part + reconstruct_genome) on a B200 through libsccg_b200.so.
//
// Additive (SURVEY 8f.3): `decompress --batch <list> [--gpus N]` runs many archives in one process -- one line per archive,
// "<compressed_file> <reference_file> <output_folder>" -- over N GPUs with two workers per GPU (host/batch.hpp).
// The reconstructed FASTA is STREAMED: the library hands it over piece by piece from a page-locked double buffer
// (sccg_decompress_fasta_stream) and every piece is written to the output file while the next one crosses PCIe.
//
// Additive: `decompress --regions <regions.bed> <compressed_file> <reference_file> <output_folder>` writes only the BED regions
// (name, 0-based start, exclusive end) to <output_folder>/regions.fa, one record per region labelled ">name:start-end" as
// `bedtools getfasta` does, 50 columns per line; the whole image is never produced (sccg_extract_fasta).
//
// Additive: `decompress --regions <regions.bed> --archives <list> <reference_file> <output_folder>` extracts every BED region from
// every archive of <list> (one .7z per line) in one call: the reference is read once and made resident, each archive is
// unpacked as the 3-argument form does and opened on the device (sccg_archive_open), and sccg_archive_extract gathers all pieces.
// <output_folder>/regions.fa holds, archive by archive in list order and region by region in BED order, records
// ">archive_stem::name:start-end" (with "(-)" appended for the minus strand, `bedtools getfasta -s` style); BED column 6 ("+",
// "-" or "."; absent means "+") sets the strand, and a minus-strand record holds the reverse complement.
//
// Additive: `decompress --search <patterns.fa> --archives <list> [--regions <bed>] [--mismatches K | --edits K] [--strand both|+|-]
// <reference_file> <output_folder>` finds every occurrence of the FASTA patterns (name: the header up to the first whitespace;
// 1 to 64 bytes each) with at most K mismatches (default 0) in every BED region of every archive, or in each archive's whole
// sequence without --regions (sccg_archive_search; archives unpacked and opened as above).  <output_folder>/hits.bed holds one
// line per hit, "archive_stem<TAB>start<TAB>end<TAB>pattern_name<TAB>mismatches<TAB>+|-", archive by archive in list order and
// in the library's (window, position, pattern, strand) order.  With `--edits K` instead of --mismatches (not both) insertions
// and deletions count too: every end of an alignment within K edits (sccg_archive_search_edits), one line per hit with its
// start, end and edit count in the fifth column, in (window, end, pattern, strand) order.
//
// Additive: `decompress --variants --archives <list> [--regions <bed>] <reference_file> <output_folder>` reports how every
// archive of <list> differs from the reference (sccg_archive_variants; archives unpacked and opened as above), in the whole
// reference or in the BED regions (reference coordinates).  <output_folder>/variants.vcf is VCF 4.2:
//   ##fileformat=VCFv4.2, ##contig=<ID=CHROM,length=len(R)>, a GT ##FORMAT line, then the header line
//   #CHROM POS ID REF ALT QUAL FILTER INFO FORMAT <one haploid sample column per archive: its stem, as in hits.bed>.
// CHROM is the first word of the reference FASTA's first header line (the file stem when there is none).  One row per
// distinct (POS, REF, ALT) over all archives, GT 1 for the archives that carry it and 0 for the others, sorted by POS, then
// by the REF and ALT bytes; a record in several regions appears once.  REF is up(R[pos:end]) and ALT the record's ALT bytes
// at POS = pos + 1; an insertion or deletion is padded with the preceding reference base (POS = pos), or at pos = 0 with the
// following one (N if neither exists); substitutions and complex records are not padded.  ID, QUAL, FILTER and INFO are '.'.
// REF and ALT hold ASCII letters only (IUPAC codes included): when a record's REF or ALT would hold any other byte (D and R
// may hold any byte but '\n'), the command names the record's position, exits 1 and writes no variants.vcf.
//
// Additive: `decompress --liftover <bed> --archives <list> [--from reference|archive] <reference_file> <output_folder>` lifts
// BED regions between reference coordinates and the coordinates of each archive's own sequence (sccg_archive_liftover;
// archives unpacked and opened as above) and writes <output_folder>/lifted.bed.  --from reference (the default): every
// region is lifted into every archive, archive by archive in list order and region by region in BED order (as regions.fa).
// --from archive: column 1 of each line must be the stem of a listed archive (hits.bed of --search feeds back directly) and
// lines keep their order; a line that names no listed archive is reported, the command exits 1 and writes no lifted.bed.
// One line per lifted region: "chrom start end name same strand subst records flags source", tab-separated: chrom the
// target system (the archive stem, or CHROM as variants.vcf names it), name BED column 4 and strand BED column 6 ("." when
// absent), same / subst / records / flags as sccg_lift reports them, source "system:start-end" of the input interval.
//
// Additive: `decompress --regions <bed> --archives <list> --reference-coords <reference_file> <output_folder>` extracts every
// BED region, given in reference coordinates, from every archive: one sccg_archive_liftover call, then one
// sccg_archive_extract call of the lifted pieces.  regions.fa holds the records and labels of `--regions --archives`, with
// the BED's reference coordinates in the label (the same gene carries the same label in every archive); a minus-strand
// record holds the reverse complement of the lifted piece.
#include <algorithm>
#include <cstdlib>
#include <filesystem>
#include <iostream>
#include <map>
#include <tuple>

#include "batch.hpp"
#include "fasta_io.hpp"
#include "sccg.h"

namespace fs = std::filesystem;
using sccg_host::Job; using sccg_host::Timing; using sccg_host::Worker;

struct FileSink { int fd; bool failed; double write_s; };
static int file_sink(void* user, int64_t /*offset*/, const char* data, int64_t len) {      // pieces arrive in order: a plain sequential write
    FileSink* s = (FileSink*)user;
    const double t0 = sccg_host::now_s();
    if (!sccg_host::write_all(s->fd, data, (size_t)len)) { s->failed = true; return 1; }
    s->write_s += sccg_host::now_s() - t0;
    return 0;
}

static int decompress_one(Worker& w, const Job& job, Timing& tm, bool verbose) {
    const std::string &arc = job.a, &ref_path = job.b, &out_dir = job.out;
    const double t0 = sccg_host::now_s();
    std::error_code ec;
    if (!fs::exists(out_dir)) fs::create_directory(out_dir, ec);
    const std::string cmd = "7z e \"" + arc + "\" -o\"" + out_dir + "\" -y" + (verbose ? "" : " > /dev/null");   // :34
    if (system(cmd.c_str()) != 0) { std::cerr << "Greska pri dekompresiji: " << arc << "\n"; return 1; }
    const std::string inter_path = out_dir + "/" + fs::path(arc).stem().string();   // :43-44
    const double t1 = sccg_host::now_s();

    // the raw FASTA image goes to the GPU as it is: header lines and whitespace are removed there (decompression.cpp:47-58)
    int64_t nf = 0, ni = 0;
    if (!sccg_host::read_file_pinned(ref_path, w.in0, &nf)) { std::cerr << "Greska pri otvaranju reference: " << ref_path << "\n"; return 1; }
    if (!sccg_host::read_file_pinned(inter_path, w.in1, &ni)) { std::cerr << "Greska pri otvaranju datoteke: " << inter_path << "\n"; return 1; }
    const double t2 = sccg_host::now_s();

    // the reference opens the output only after reconstruct_genome succeeded (:316); here the file is created up front and
    // removed again if the record stream turns out to be malformed (reported before the first piece is delivered)
    const std::string out_path = out_dir + "/reconstructed_genome.fa";
    const std::string tmp_path = out_path + ".part";
    FileSink sink{open(tmp_path.c_str(), O_WRONLY | O_CREAT | O_TRUNC, 0644), false, 0.0};
    if (sink.fd < 0) { std::cerr << "Error opening output file: " << out_dir << "\n"; return 1; }
    int64_t total = 0;
    const int rc = sccg_decompress_fasta_stream(w.ctx, w.in0.p, nf, w.in1.p, ni, file_sink, &sink, &total);
    close(sink.fd);
    if (rc != SCCG_OK) {
        unlink(tmp_path.c_str());
        if (sink.failed) { std::cerr << "Error opening output file: " << out_dir << "\n"; return 1; }
        // SCCG_E_BOUNDS: the reference prints the same ERROR and exit(1)s (:223-229); SCCG_E_FORMAT: it dies in stoi (:309-312)
        std::cerr << (rc == SCCG_E_BOUNDS ? "" : "Error during reconstruction: ") << sccg_last_error() << "\n";
        return 1;
    }
    if (rename(tmp_path.c_str(), out_path.c_str()) != 0) { std::cerr << "Error opening output file: " << out_dir << "\n"; return 1; }
    const double t3 = sccg_host::now_s();
    tm.ext_s = t1 - t0; tm.read_s = t2 - t1; tm.write_s = sink.write_s; tm.gpu_s = (t3 - t2) - sink.write_s;
    if (verbose) {
        if (getenv("SCCG_TIMING")) std::cerr << "timing: 7z " << tm.ext_s << " s, read " << tm.read_s << " s, gpu call " << tm.gpu_s << " s, write (overlapped with PCIe) " << tm.write_s << " s\n";
        std::cout << "Time taken to decompress: " << (t3 - t0) << " s\n";      // :327 (here the write is inside: it overlaps the transfer)
    }
    return 0;
}

// BED lines: "name start end [more columns]", separated by tabs or spaces; blank lines and "#", "track", "browser" lines are
// skipped.  false (with a message) on anything else.
// with_strand: column 6, when present, must be "+", "-" or "." (strand 1 for "-")
// label / strand_text: column 4 and column 6 as written ("." when absent); line: the line number
struct BedRegion { std::string name; int64_t start, end; int strand = 0; std::string label = ".", strand_text = "."; int64_t line = 0; };
static bool parse_bed(const std::string& text, std::vector<BedRegion>* out, std::string* err, bool with_strand = false) {
    std::istringstream in(text);
    std::string line;
    for (int64_t no = 1; std::getline(in, line); ++no) {
        if (!line.empty() && line.back() == '\r') line.pop_back();
        std::vector<std::string> f;
        for (size_t i = 0; i < line.size();) {
            while (i < line.size() && (line[i] == ' ' || line[i] == '\t')) ++i;
            size_t j = i;
            while (j < line.size() && line[j] != ' ' && line[j] != '\t') ++j;
            if (j > i) f.push_back(line.substr(i, j - i));
            i = j;
        }
        if (f.empty() || f[0][0] == '#' || f[0] == "track" || f[0] == "browser") continue;
        auto num = [](const std::string& t, int64_t* v) {
            if (t.empty() || t.size() > 18 || t.find_first_not_of("0123456789") != std::string::npos) return false;
            *v = std::stoll(t);
            return true;
        };
        BedRegion r;
        if (f.size() < 3 || !num(f[1], &r.start) || !num(f[2], &r.end) || r.start > r.end) {
            *err = "malformed BED line " + std::to_string(no) + ": " + line;
            return false;
        }
        if (with_strand && f.size() >= 6) {
            if (f[5] != "+" && f[5] != "-" && f[5] != ".") { *err = "malformed BED line " + std::to_string(no) + " (strand): " + line; return false; }
            r.strand = f[5] == "-";
        }
        r.name = f[0];
        if (f.size() >= 4) r.label = f[3];
        if (f.size() >= 6) r.strand_text = f[5];
        r.line = no;
        out->push_back(r);
    }
    return true;
}

// the records of regions.fa: header line, then the piece in lines of 50; written next to the target and renamed (no partial file)
static bool write_output(const std::string& out_path, const std::string& text);
static bool write_records(const std::string& out_dir, const std::string& text) { return write_output(out_dir + "/regions.fa", text); }

static int extract_regions(const char* bed_path, const Job& job) {
    std::ifstream bf(bed_path, std::ios::binary);
    if (!bf) { std::cerr << "Error opening BED file: " << bed_path << "\n"; return 1; }
    std::stringstream ss; ss << bf.rdbuf();
    std::vector<BedRegion> bed;
    std::string err;
    if (!parse_bed(ss.str(), &bed, &err)) { std::cerr << "Error: " << err << "\n"; return 1; }
    std::error_code ec;
    if (!fs::exists(job.out)) fs::create_directory(job.out, ec);
    const std::string cmd = "7z e \"" + job.a + "\" -o\"" + job.out + "\" -y > /dev/null";                        // as the 3-argument form
    if (system(cmd.c_str()) != 0) { std::cerr << "Greska pri dekompresiji: " << job.a << "\n"; return 1; }
    const std::string inter_path = job.out + "/" + fs::path(job.a).stem().string();
    const char* dev = getenv("SCCG_DEVICE");
    Worker w; w.device = dev ? atoi(dev) : 0;
    w.ctx = sccg_create(w.device);
    if (!w.ctx) { std::cerr << "Error: " << sccg_last_error() << "\n"; return 1; }
    int64_t nf = 0, ni = 0;
    int status = 1;
    std::vector<sccg_region> regs(bed.size());
    int64_t total = 0, out_len = 0, seq_len = -1;
    for (size_t i = 0; i < bed.size(); ++i) { regs[i].start = bed[i].start; regs[i].end = bed[i].end; total += bed[i].end - bed[i].start; }
    std::vector<char> seq((size_t)total + 1);
    if (!sccg_host::read_file_pinned(job.b, w.in0, &nf)) std::cerr << "Greska pri otvaranju reference: " << job.b << "\n";
    else if (!sccg_host::read_file_pinned(inter_path, w.in1, &ni)) std::cerr << "Greska pri otvaranju datoteke: " << inter_path << "\n";
    else {
        const int rc = sccg_extract_fasta(w.ctx, w.in0.p, nf, w.in1.p, ni, regs.data(), (int64_t)regs.size(), seq.data(), total, &out_len, &seq_len);
        if (rc != SCCG_OK && seq_len >= 0 && rc == SCCG_E_ARG) std::cerr << "Error: a region ends past the end of the sequence (" << seq_len << " bp)\n";
        else if (rc != SCCG_OK) std::cerr << (rc == SCCG_E_BOUNDS ? "" : "Error during reconstruction: ") << sccg_last_error() << "\n";
        else status = 0;
    }
    sccg_destroy(w.ctx);
    if (status) return status;
    // ">name:start-end" and the sequence in lines of 50
    std::string text;
    text.reserve((size_t)total + (size_t)total / 50 + bed.size() * 32);
    int64_t at = 0;
    for (const BedRegion& r : bed) {
        text += ">" + r.name + ":" + std::to_string(r.start) + "-" + std::to_string(r.end) + "\n";
        for (int64_t p = r.start; p < r.end; p += 50) {
            const int64_t n = r.end - p < 50 ? r.end - p : 50;
            text.append(seq.data() + at, (size_t)n); text += '\n';
            at += n;
        }
    }
    if (!write_records(job.out, text)) { std::cerr << "Error opening output file: " << job.out << "\n"; return 1; }
    return 0;
}

// the archive list: one path per line, blank lines skipped; false (with a message) when it cannot be read or names none
static bool read_archive_list(const char* list_path, std::vector<std::string>* arcs) {
    std::string list_text;
    if (!sccg_host::read_file(list_path, list_text)) { std::cerr << "Error opening list file: " << list_path << "\n"; return false; }
    std::istringstream in(list_text);
    std::string line;
    while (std::getline(in, line)) {
        const size_t a = line.find_first_not_of(" \t\r"), b = line.find_last_not_of(" \t\r");
        if (a != std::string::npos) arcs->push_back(line.substr(a, b - a + 1));
    }
    if (arcs->empty()) { std::cerr << "Error: the archive list " << list_path << " names no archive\n"; return false; }
    return true;
}

// the reference FASTA read once and made resident on a new context; NULL (with a message) on failure
static sccg_ctx* resident_context(const std::string& ref_path) {
    std::string ref_file, ref;
    if (!sccg_host::read_file(ref_path, ref_file)) { std::cerr << "Greska pri otvaranju reference: " << ref_path << "\n"; return nullptr; }
    sccg_host::parse_fasta(ref_file, false, ref, nullptr);                  // decompression.cpp:47-58
    const char* dev = getenv("SCCG_DEVICE");
    sccg_ctx* ctx = sccg_create(dev ? atoi(dev) : 0);
    if (!ctx) { std::cerr << "Error: " << sccg_last_error() << "\n"; return nullptr; }
    if (sccg_reference_set(ctx, ref.data(), (int64_t)ref.size()) != SCCG_OK) { std::cerr << "Error: " << sccg_last_error() << "\n"; sccg_destroy(ctx); return nullptr; }
    return ctx;
}

// one archive unpacked as the 3-argument form does and opened on the device; NULL (with a message) on failure
static sccg_archive* open_archive_file(sccg_ctx* ctx, const std::string& arc, const std::string& out_dir) {
    const std::string cmd = "7z e \"" + arc + "\" -o\"" + out_dir + "\" -y > /dev/null";
    if (system(cmd.c_str()) != 0) { std::cerr << "Greska pri dekompresiji: " << arc << "\n"; return nullptr; }
    std::string inter;
    const std::string inter_path = out_dir + "/" + fs::path(arc).stem().string();
    if (!sccg_host::read_file(inter_path, inter)) { std::cerr << "Greska pri otvaranju datoteke: " << inter_path << "\n"; return nullptr; }
    sccg_archive* a = nullptr;
    const int rc = sccg_archive_open(ctx, inter.data(), (int64_t)inter.size(), &a);
    if (rc != SCCG_OK) { std::cerr << arc << ": " << (rc == SCCG_E_BOUNDS ? "" : "Error during reconstruction: ") << sccg_last_error() << "\n"; return nullptr; }
    return a;
}

// an output file written next to its target and renamed (no partial file)
static bool write_output(const std::string& out_path, const std::string& text) {
    const std::string tmp_path = out_path + ".part";
    const int fd = open(tmp_path.c_str(), O_WRONLY | O_CREAT | O_TRUNC, 0644);
    const bool ok = fd >= 0 && sccg_host::write_all(fd, text.data(), text.size());
    if (fd >= 0) close(fd);
    if (!ok || rename(tmp_path.c_str(), out_path.c_str()) != 0) { unlink(tmp_path.c_str()); return false; }
    return true;
}

static int extract_archives(const char* bed_path, const char* list_path, const std::string& ref_path, const std::string& out_dir) {
    std::string bed_text;
    std::vector<BedRegion> bed;
    std::string err;
    if (!sccg_host::read_file(bed_path, bed_text)) { std::cerr << "Error opening BED file: " << bed_path << "\n"; return 1; }
    if (!parse_bed(bed_text, &bed, &err, true)) { std::cerr << "Error: " << err << "\n"; return 1; }
    std::vector<std::string> arcs;
    if (!read_archive_list(list_path, &arcs)) return 1;
    sccg_ctx* ctx = resident_context(ref_path);
    if (!ctx) return 1;
    std::error_code ec;
    if (!fs::exists(out_dir)) fs::create_directory(out_dir, ec);
    int status = 1;
    std::vector<sccg_archive*> open;
    std::vector<sccg_query> qs;
    std::string text;
    [&] {
        for (const std::string& arc : arcs) {                               // unpacked one at a time: archives may share a file name
            sccg_archive* a = open_archive_file(ctx, arc, out_dir);
            if (!a) return;
            open.push_back(a);
            int64_t seq_len = 0;
            sccg_archive_info(a, &seq_len, nullptr, nullptr);
            for (const BedRegion& r : bed) {
                if (r.end > seq_len) { std::cerr << "Error: region " << r.name << ":" << r.start << "-" << r.end << " ends past the end of " << arc << " (" << seq_len << " bp)\n"; return; }
                qs.push_back(sccg_query{(int64_t)open.size() - 1, r.start, r.end, r.strand});
            }
        }
        int64_t total = 0, out_len = 0;
        for (const sccg_query& q : qs) total += q.end - q.start;
        std::vector<char> seq((size_t)total + 1);
        if (sccg_archive_extract(ctx, open.data(), (int64_t)open.size(), qs.data(), (int64_t)qs.size(), seq.data(), total, &out_len) != SCCG_OK) {
            std::cerr << "Error: " << sccg_last_error() << "\n";
            return;
        }
        text.reserve((size_t)total + (size_t)total / 50 + qs.size() * 48);
        int64_t at = 0;
        for (size_t i = 0; i < qs.size(); ++i) {
            const BedRegion& r = bed[i % bed.size()];
            text += ">" + fs::path(arcs[i / bed.size()]).stem().string() + "::" + r.name + ":" + std::to_string(r.start) + "-" + std::to_string(r.end) +
                    (r.strand ? "(-)" : "") + "\n";
            for (int64_t p = r.start; p < r.end; p += 50) {
                const int64_t n = r.end - p < 50 ? r.end - p : 50;
                text.append(seq.data() + at, (size_t)n); text += '\n';
                at += n;
            }
        }
        status = 0;
    }();
    sccg_destroy(ctx);                                                      // (releases the archives)
    if (status) return status;
    if (!write_records(out_dir, text)) { std::cerr << "Error opening output file: " << out_dir << "\n"; return 1; }
    return 0;
}

// FASTA patterns: the name is the header up to the first whitespace, the sequence lines are joined (line-end whitespace
// dropped); false (with a message) for text before the first header, a record without sequence, or none at all
struct Pattern { std::string name, seq; };
static bool parse_patterns(const std::string& text, std::vector<Pattern>* out, std::string* err) {
    std::istringstream in(text);
    std::string line;
    for (int64_t no = 1; std::getline(in, line); ++no) {
        while (!line.empty() && isspace((unsigned char)line.back())) line.pop_back();
        if (!line.empty() && line[0] == '>') {
            if (!out->empty() && out->back().seq.empty()) { *err = "pattern " + out->back().name + " has no sequence"; return false; }
            const size_t e = line.find_first_of(" \t", 1);
            out->push_back(Pattern{line.substr(1, e == std::string::npos ? std::string::npos : e - 1), ""});
            continue;
        }
        if (line.empty()) continue;
        if (out->empty()) { *err = "line " + std::to_string(no) + " comes before the first '>' header"; return false; }
        out->back().seq += line;
    }
    if (out->empty()) { *err = "the pattern file holds no pattern"; return false; }
    if (out->back().seq.empty()) { *err = "pattern " + out->back().name + " has no sequence"; return false; }
    for (const Pattern& p : *out)
        if (p.seq.size() > 64) { *err = "pattern " + p.name + " is longer than 64 bytes"; return false; }
    return true;
}

static int search_archives(int argc, char* argv[]) {
    const char *pat_path = argv[2], *list_path = nullptr, *bed_path = nullptr;
    int k = 0, strands = 3;
    bool by_mm = false, by_edits = false;
    int i = 3;
    for (; i + 1 < argc - 2; i += 2) {
        const std::string opt = argv[i], v = argv[i + 1];
        if (opt == "--archives") list_path = argv[i + 1];
        else if (opt == "--regions") bed_path = argv[i + 1];
        else if (opt == "--mismatches" || opt == "--edits") {
            const bool edits = opt == "--edits";
            if (v.empty() || v.size() > 2 || v.find_first_not_of("0123456789") != std::string::npos) { std::cerr << "Error: bad " << (edits ? "edit" : "mismatch") << " count " << v << "\n"; return 1; }
            (edits ? by_edits : by_mm) = true;
            if (by_edits && by_mm) { std::cerr << "Error: --edits and --mismatches exclude each other\n"; return 1; }
            k = std::stoi(v);
        } else if (opt == "--strand") {
            if (v != "both" && v != "+" && v != "-") { std::cerr << "Error: --strand takes both, + or -\n"; return 1; }
            strands = v == "both" ? 3 : v == "+" ? 1 : 2;
        } else { std::cerr << "Error: unknown option " << opt << "\n"; return 1; }
    }
    if (i != argc - 2 || !list_path) { std::cerr << "Error: --search needs --archives <list>, then <reference_file> <output_folder>\n"; return 1; }
    const std::string ref_path = argv[argc - 2], out_dir = argv[argc - 1];
    std::string pat_text, err;
    std::vector<Pattern> pats;
    if (!sccg_host::read_file(pat_path, pat_text)) { std::cerr << "Error opening pattern file: " << pat_path << "\n"; return 1; }
    if (!parse_patterns(pat_text, &pats, &err)) { std::cerr << "Error: " << err << "\n"; return 1; }
    int64_t minlen = 64;
    for (const Pattern& p : pats) minlen = (int64_t)p.seq.size() < minlen ? (int64_t)p.seq.size() : minlen;
    if (k >= minlen) { std::cerr << "Error: the " << (by_edits ? "edit" : "mismatch") << " count must be below the shortest pattern's length (" << minlen << ")\n"; return 1; }
    std::vector<BedRegion> bed;
    if (bed_path) {
        std::string bed_text;
        if (!sccg_host::read_file(bed_path, bed_text)) { std::cerr << "Error opening BED file: " << bed_path << "\n"; return 1; }
        if (!parse_bed(bed_text, &bed, &err)) { std::cerr << "Error: " << err << "\n"; return 1; }
    }
    std::vector<std::string> arcs;
    if (!read_archive_list(list_path, &arcs)) return 1;
    sccg_ctx* ctx = resident_context(ref_path);
    if (!ctx) return 1;
    std::error_code ec;
    if (!fs::exists(out_dir)) fs::create_directory(out_dir, ec);
    int status = 1;
    std::vector<sccg_archive*> open;
    std::vector<sccg_window> wins;
    std::vector<size_t> win_arc;
    std::string text;
    [&] {
        for (const std::string& arc : arcs) {                               // unpacked one at a time: archives may share a file name
            sccg_archive* a = open_archive_file(ctx, arc, out_dir);
            if (!a) return;
            open.push_back(a);
            int64_t seq_len = 0;
            sccg_archive_info(a, &seq_len, nullptr, nullptr);
            const int64_t ai = (int64_t)open.size() - 1;
            if (!bed_path) { wins.push_back(sccg_window{ai, 0, seq_len}); win_arc.push_back((size_t)ai); }
            for (const BedRegion& r : bed) {
                if (r.end > seq_len) { std::cerr << "Error: region " << r.name << ":" << r.start << "-" << r.end << " ends past the end of " << arc << " (" << seq_len << " bp)\n"; return; }
                wins.push_back(sccg_window{ai, r.start, r.end}); win_arc.push_back((size_t)ai);
            }
        }
        std::string blob;
        std::vector<int64_t> off(1, 0);
        for (const Pattern& p : pats) { blob += p.seq; off.push_back((int64_t)blob.size()); }
        std::vector<std::string> stems;
        for (const std::string& arc : arcs) stems.push_back(fs::path(arc).stem().string());
        auto line = [&](int64_t w, int64_t start, int64_t end, int32_t i, int32_t d, int32_t strand) {
            text += stems[win_arc[(size_t)w]] + "\t" + std::to_string(start) + "\t" + std::to_string(end) + "\t" + pats[(size_t)i].name + "\t" +
                    std::to_string(d) + (strand ? "\t-\n" : "\t+\n");
        };
        int64_t n = 0;
        if (by_edits) {
            std::vector<sccg_edit_hit> hits;
            int rc = sccg_archive_search_edits(ctx, open.data(), (int64_t)open.size(), wins.data(), (int64_t)wins.size(), blob.data(), off.data(),
                                               (int64_t)pats.size(), k, strands, nullptr, 0, &n);
            if (rc == SCCG_OK && n > 0) {
                hits.resize((size_t)n);
                rc = sccg_archive_search_edits(ctx, open.data(), (int64_t)open.size(), wins.data(), (int64_t)wins.size(), blob.data(), off.data(),
                                               (int64_t)pats.size(), k, strands, hits.data(), n, &n);
            }
            if (rc != SCCG_OK) { std::cerr << "Error: " << sccg_last_error() << "\n"; return; }
            for (const sccg_edit_hit& h : hits) line(h.window, h.start, h.end, h.pattern, h.edits, h.strand);
            status = 0;
            return;
        }
        std::vector<sccg_hit> hits;
        int rc = sccg_archive_search(ctx, open.data(), (int64_t)open.size(), wins.data(), (int64_t)wins.size(), blob.data(), off.data(), (int64_t)pats.size(),
                                     k, strands, nullptr, 0, &n);
        if (rc == SCCG_OK && n > 0) {
            hits.resize((size_t)n);
            rc = sccg_archive_search(ctx, open.data(), (int64_t)open.size(), wins.data(), (int64_t)wins.size(), blob.data(), off.data(), (int64_t)pats.size(),
                                     k, strands, hits.data(), n, &n);
        }
        if (rc != SCCG_OK) { std::cerr << "Error: " << sccg_last_error() << "\n"; return; }
        for (const sccg_hit& h : hits) line(h.window, h.pos, h.pos + (int64_t)pats[(size_t)h.pattern].seq.size(), h.pattern, h.mismatches, h.strand);
        status = 0;
    }();
    sccg_destroy(ctx);                                                      // (releases the archives)
    if (status) return status;
    if (!write_output(out_dir + "/hits.bed", text)) { std::cerr << "Error opening output file: " << out_dir << "\n"; return 1; }
    return 0;
}

// the reference FASTA's symbols and its CHROM: the first word of its first header line (the file stem when there is none);
// false (with a message) when it cannot be read
static bool reference_symbols(const std::string& ref_path, std::string* ref, std::string* chrom) {
    std::string ref_file;
    if (!sccg_host::read_file(ref_path, ref_file)) { std::cerr << "Greska pri otvaranju reference: " << ref_path << "\n"; return false; }
    sccg_host::parse_fasta(ref_file, false, *ref, nullptr);
    chrom->clear();
    for (size_t p = 0; p < ref_file.size();) {                              // the first header line's first word
        const size_t e = ref_file.find('\n', p);
        const std::string line = ref_file.substr(p, e == std::string::npos ? std::string::npos : e - p);
        if (!line.empty() && line[0] == '>') {
            const size_t w = line.find_first_of(" \t\r", 1);
            *chrom = line.substr(1, w == std::string::npos ? std::string::npos : w - 1);
            break;
        }
        if (e == std::string::npos) break;
        p = e + 1;
    }
    if (chrom->empty()) *chrom = fs::path(ref_path).stem().string();
    return true;
}

// the VCF of `--variants` (format in the header comment)
static int variants_archives(int argc, char* argv[]) {
    const char *list_path = nullptr, *bed_path = nullptr;
    int i = 2;
    for (; i + 1 < argc - 2; i += 2) {
        const std::string opt = argv[i];
        if (opt == "--archives") list_path = argv[i + 1];
        else if (opt == "--regions") bed_path = argv[i + 1];
        else { std::cerr << "Error: unknown option " << opt << "\n"; return 1; }
    }
    if (i != argc - 2 || !list_path) { std::cerr << "Error: --variants needs --archives <list>, then <reference_file> <output_folder>\n"; return 1; }
    const std::string ref_path = argv[argc - 2], out_dir = argv[argc - 1];
    std::string err;
    std::vector<BedRegion> bed;
    if (bed_path) {
        std::string bed_text;
        if (!sccg_host::read_file(bed_path, bed_text)) { std::cerr << "Error opening BED file: " << bed_path << "\n"; return 1; }
        if (!parse_bed(bed_text, &bed, &err)) { std::cerr << "Error: " << err << "\n"; return 1; }
    }
    std::vector<std::string> arcs;
    if (!read_archive_list(list_path, &arcs)) return 1;
    std::string ref, chrom;
    if (!reference_symbols(ref_path, &ref, &chrom)) return 1;
    for (const BedRegion& r : bed)
        if (r.end > (int64_t)ref.size()) { std::cerr << "Error: region " << r.name << ":" << r.start << "-" << r.end << " ends past the end of the reference (" << ref.size() << " bp)\n"; return 1; }
    sccg_ctx* ctx = resident_context(ref_path);
    if (!ctx) return 1;
    std::error_code ec;
    if (!fs::exists(out_dir)) fs::create_directory(out_dir, ec);
    int status = 1;
    std::vector<sccg_archive*> open;
    std::vector<sccg_window> wins;
    std::string text;
    [&] {
        for (const std::string& arc : arcs) {                               // unpacked one at a time: archives may share a file name
            sccg_archive* a = open_archive_file(ctx, arc, out_dir);
            if (!a) return;
            open.push_back(a);
            const int64_t ai = (int64_t)open.size() - 1;
            if (!bed_path) wins.push_back(sccg_window{ai, 0, (int64_t)ref.size()});
            for (const BedRegion& r : bed) wins.push_back(sccg_window{ai, r.start, r.end});
        }
        int64_t n = 0, na = 0;
        int rc = sccg_archive_variants(ctx, open.data(), (int64_t)open.size(), wins.data(), (int64_t)wins.size(), nullptr, 0, &n, nullptr, 0, &na);
        std::vector<sccg_variant> vars((size_t)n);
        std::vector<char> alt((size_t)na + 1);
        if (rc == SCCG_OK && n > 0) rc = sccg_archive_variants(ctx, open.data(), (int64_t)open.size(), wins.data(), (int64_t)wins.size(), vars.data(), n, &n, alt.data(), na, &na);
        if (rc != SCCG_OK) { std::cerr << "Error: " << sccg_last_error() << "\n"; return; }
        auto up = [](char ch) { return (ch >= 'a' && ch <= 'z') ? (char)(ch - 32) : ch; };
        auto letters = [](const std::string& s) {
            for (char ch : s) if (!((ch >= 'A' && ch <= 'Z') || (ch >= 'a' && ch <= 'z'))) return false;
            return true;
        };
        std::map<std::tuple<int64_t, std::string, std::string>, std::vector<char>> rows;
        for (const sccg_variant& v : vars) {
            std::string r, a(alt.data() + v.alt_off, (size_t)(v.d_end - v.d_start));
            for (int64_t q = v.pos; q < v.end; ++q) r += up(ref[(size_t)q]);
            int64_t pos = v.pos + 1;
            if (r.empty() || a.empty()) {
                if (v.pos > 0) { const char b = up(ref[(size_t)v.pos - 1]); r = b + r; a = b + a; pos = v.pos; }
                else { const char b = v.end < (int64_t)ref.size() ? up(ref[(size_t)v.end]) : 'N'; r += b; a += b; }
            }
            if (!letters(r) || !letters(a)) {                                 // a tab, ',' or control byte would corrupt the row
                std::cerr << "Error: the record at reference position " << v.pos + 1 << " of " << fs::path(arcs[(size_t)wins[(size_t)v.window].archive]).stem().string()
                          << " has REF or ALT bytes that are not ASCII letters; VCF cannot hold them\n";
                return;
            }
            std::vector<char>& gt = rows[std::make_tuple(pos, r, a)];
            gt.resize(open.size(), 0);
            gt[(size_t)wins[(size_t)v.window].archive] = 1;
        }
        text = "##fileformat=VCFv4.2\n##contig=<ID=" + chrom + ",length=" + std::to_string(ref.size()) + ">\n"
               "##FORMAT=<ID=GT,Number=1,Type=String,Description=\"Genotype\">\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT";
        for (const std::string& arc : arcs) text += "\t" + fs::path(arc).stem().string();
        text += "\n";
        for (const auto& row : rows) {
            text += chrom + "\t" + std::to_string(std::get<0>(row.first)) + "\t.\t" + std::get<1>(row.first) + "\t" + std::get<2>(row.first) + "\t.\t.\t.\tGT";
            for (char g : row.second) text += g ? "\t1" : "\t0";
            text += "\n";
        }
        status = 0;
    }();
    sccg_destroy(ctx);                                                      // (releases the archives)
    if (status) return status;
    if (!write_output(out_dir + "/variants.vcf", text)) { std::cerr << "Error opening output file: " << out_dir << "\n"; return 1; }
    return 0;
}

// `--liftover` (lifted.bed) and `--regions --reference-coords` (regions.fa): BED regions lifted between the reference and the
// archives of the list (format in the header comment).  from: 0 reference -> archive, 1 archive -> reference.
static int lift_archives(const char* bed_path, const char* list_path, int from, bool extract, const std::string& ref_path, const std::string& out_dir) {
    std::string bed_text, err, ref, chrom;
    std::vector<BedRegion> bed;
    if (!sccg_host::read_file(bed_path, bed_text)) { std::cerr << "Error opening BED file: " << bed_path << "\n"; return 1; }
    if (!parse_bed(bed_text, &bed, &err, true)) { std::cerr << "Error: " << err << "\n"; return 1; }
    std::vector<std::string> arcs, stems;
    if (!read_archive_list(list_path, &arcs)) return 1;
    for (const std::string& arc : arcs) stems.push_back(fs::path(arc).stem().string());
    if (!reference_symbols(ref_path, &ref, &chrom)) return 1;
    std::vector<int64_t> src_arc(bed.size(), 0);                             // --from archive: the archive each line names
    for (size_t i = 0; i < bed.size(); ++i) {
        const BedRegion& r = bed[i];
        if (from == 1) {
            const auto it = std::find(stems.begin(), stems.end(), r.name);
            if (it == stems.end()) { std::cerr << "Error: BED line " << r.line << " names no listed archive: " << r.name << "\n"; return 1; }
            src_arc[i] = it - stems.begin();
        } else if (r.end > (int64_t)ref.size()) {
            std::cerr << "Error: region " << r.name << ":" << r.start << "-" << r.end << " ends past the end of the reference (" << ref.size() << " bp)\n";
            return 1;
        }
    }
    sccg_ctx* ctx = resident_context(ref_path);
    if (!ctx) return 1;
    std::error_code ec;
    if (!fs::exists(out_dir)) fs::create_directory(out_dir, ec);
    int status = 1;
    std::vector<sccg_archive*> open;
    std::vector<sccg_lift_query> qs;
    std::vector<size_t> q_bed;                                              // the BED line of each query
    std::string text;
    [&] {
        for (const std::string& arc : arcs) {                               // unpacked one at a time: archives may share a file name
            sccg_archive* a = open_archive_file(ctx, arc, out_dir);
            if (!a) return;
            open.push_back(a);
        }
        for (size_t i = 0; i < bed.size(); ++i) {
            const BedRegion& r = bed[i];
            if (from == 0) continue;
            int64_t seq_len = 0;
            sccg_archive_info(open[(size_t)src_arc[i]], &seq_len, nullptr, nullptr);
            if (r.end > seq_len) { std::cerr << "Error: region " << r.name << ":" << r.start << "-" << r.end << " ends past the end of " << arcs[(size_t)src_arc[i]] << " (" << seq_len << " bp)\n"; return; }
            qs.push_back(sccg_lift_query{src_arc[i], r.start, r.end, 1, 0});
            q_bed.push_back(i);
        }
        if (from == 0)                                                      // archive by archive, region by region (as regions.fa)
            for (size_t k = 0; k < open.size(); ++k)
                for (size_t i = 0; i < bed.size(); ++i) { qs.push_back(sccg_lift_query{(int64_t)k, bed[i].start, bed[i].end, 0, 0}); q_bed.push_back(i); }
        std::vector<sccg_lift> lifted(qs.size());
        if (sccg_archive_liftover(ctx, open.data(), (int64_t)open.size(), qs.data(), (int64_t)qs.size(), lifted.data()) != SCCG_OK) {
            std::cerr << "Error: " << sccg_last_error() << "\n";
            return;
        }
        if (!extract) {
            for (size_t j = 0; j < qs.size(); ++j) {
                const BedRegion& r = bed[q_bed[j]];
                const sccg_lift& l = lifted[j];
                const std::string target = from ? chrom : stems[(size_t)qs[j].archive], source = from ? r.name : chrom;
                text += target + "\t" + std::to_string(l.start) + "\t" + std::to_string(l.end) + "\t" + r.label + "\t" + std::to_string(l.same) + "\t" +
                        r.strand_text + "\t" + std::to_string(l.subst) + "\t" + std::to_string(l.records) + "\t" + std::to_string(l.flags) + "\t" +
                        source + ":" + std::to_string(r.start) + "-" + std::to_string(r.end) + "\n";
            }
            status = 0;
            return;
        }
        // --reference-coords: the lifted pieces, one sccg_archive_extract call; records and labels as --regions --archives
        std::vector<sccg_query> eq(qs.size());
        int64_t total = 0, out_len = 0;
        for (size_t j = 0; j < qs.size(); ++j) {
            eq[j] = sccg_query{qs[j].archive, lifted[j].start, lifted[j].end, bed[q_bed[j]].strand};
            total += lifted[j].end - lifted[j].start;
        }
        std::vector<char> seq((size_t)total + 1);
        if (sccg_archive_extract(ctx, open.data(), (int64_t)open.size(), eq.data(), (int64_t)eq.size(), seq.data(), total, &out_len) != SCCG_OK) {
            std::cerr << "Error: " << sccg_last_error() << "\n";
            return;
        }
        text.reserve((size_t)total + (size_t)total / 50 + qs.size() * 48);
        int64_t at = 0;
        for (size_t j = 0; j < qs.size(); ++j) {
            const BedRegion& r = bed[q_bed[j]];
            text += ">" + stems[(size_t)qs[j].archive] + "::" + r.name + ":" + std::to_string(r.start) + "-" + std::to_string(r.end) + (r.strand ? "(-)" : "") + "\n";
            for (int64_t p = eq[j].start; p < eq[j].end; p += 50) {
                const int64_t n = eq[j].end - p < 50 ? eq[j].end - p : 50;
                text.append(seq.data() + at, (size_t)n); text += '\n';
                at += n;
            }
        }
        status = 0;
    }();
    sccg_destroy(ctx);                                                      // (releases the archives)
    if (status) return status;
    if (!write_output(out_dir + (extract ? "/regions.fa" : "/lifted.bed"), text)) { std::cerr << "Error opening output file: " << out_dir << "\n"; return 1; }
    return 0;
}

static int liftover_archives(int argc, char* argv[]) {
    const char* list_path = nullptr;
    int from = 0;
    int i = 3;
    for (; i + 1 < argc - 2; i += 2) {
        const std::string opt = argv[i], v = argv[i + 1];
        if (opt == "--archives") list_path = argv[i + 1];
        else if (opt == "--from") {
            if (v != "reference" && v != "archive") { std::cerr << "Error: --from takes reference or archive\n"; return 1; }
            from = v == "archive";
        } else { std::cerr << "Error: unknown option " << opt << "\n"; return 1; }
    }
    if (i != argc - 2 || !list_path) { std::cerr << "Error: --liftover needs --archives <list>, then <reference_file> <output_folder>\n"; return 1; }
    return lift_archives(argv[2], list_path, from, false, argv[argc - 2], argv[argc - 1]);
}

int main(int argc, char* argv[]) {
    const bool batch = argc >= 3 && std::string(argv[1]) == "--batch";
    const bool regions = argc == 6 && std::string(argv[1]) == "--regions";
    const bool archives = argc == 7 && std::string(argv[1]) == "--regions" && std::string(argv[3]) == "--archives";
    const bool ref_coords = argc == 8 && std::string(argv[1]) == "--regions" && std::string(argv[3]) == "--archives" && std::string(argv[5]) == "--reference-coords";
    const bool liftover = argc >= 6 && std::string(argv[1]) == "--liftover";
    const bool search = argc >= 7 && std::string(argv[1]) == "--search";
    const bool variants = argc >= 6 && std::string(argv[1]) == "--variants";
    if (argc != 4 && !batch && !regions && !archives && !ref_coords && !search && !variants && !liftover) {          // decompression.cpp:283-286
        std::cerr << "Usage: " << argv[0] << " <compressed_file> <reference_file> <output_folder>\n"
                  << "       " << argv[0] << " --batch <list of such triples, one per line> [--gpus N]\n"
                  << "       " << argv[0] << " --regions <regions.bed> <compressed_file> <reference_file> <output_folder>\n"
                  << "       " << argv[0] << " --regions <regions.bed> --archives <list of .7z files, one per line> <reference_file> <output_folder>\n"
                  << "       " << argv[0] << " --search <patterns.fa> --archives <list> [--regions <bed>] [--mismatches K | --edits K] [--strand both|+|-] <reference_file> <output_folder>\n"
                  << "       " << argv[0] << " --variants --archives <list> [--regions <bed>] <reference_file> <output_folder>\n"
                  << "       " << argv[0] << " --liftover <bed> --archives <list> [--from reference|archive] <reference_file> <output_folder>\n"
                  << "       " << argv[0] << " --regions <bed> --archives <list> --reference-coords <reference_file> <output_folder>\n";
        return 1;
    }
    try {
        if (archives) return extract_archives(argv[2], argv[4], argv[5], argv[6]);
        if (search) return search_archives(argc, argv);
        if (variants) return variants_archives(argc, argv);
        if (liftover) return liftover_archives(argc, argv);
        if (ref_coords) return lift_archives(argv[2], argv[4], 0, true, argv[6], argv[7]);
        if (regions) {
            Job job; job.a = argv[3]; job.b = argv[4]; job.out = argv[5];
            return extract_regions(argv[2], job);
        }
        if (!batch) {
            const double t0 = sccg_host::now_s();
            const char* dev = getenv("SCCG_DEVICE");
            Worker w; w.device = dev ? atoi(dev) : 0;
            w.ctx = sccg_create(w.device);
            if (!w.ctx) { std::cerr << "Error: " << sccg_last_error() << "\n"; return 1; }
            if (getenv("SCCG_TIMING")) std::cerr << "timing: context " << (sccg_host::now_s() - t0) << " s\n";
            Job job; job.a = argv[1]; job.b = argv[2]; job.out = argv[3];
            Timing tm;
            const int status = decompress_one(w, job, tm, true);
            sccg_destroy(w.ctx);
            return status;
        }
        std::vector<Job> jobs;
        if (!sccg_host::read_job_list(argv[2], &jobs)) { std::cerr << "Error opening list file: " << argv[2] << "\n"; return 1; }
        for (Job& j : jobs) j.weight = sccg_host::file_size(j.b);
        return sccg_host::run_batch(jobs, sccg_host::parse_gpus(argc, argv, 3), [](Worker& w, const Job& j, Timing& tm) { return decompress_one(w, j, tm, false); }, std::cout);
    } catch (const std::exception& ex) {
        std::cerr << "Error: " << ex.what() << "\n";
        return 1;
    }
}
