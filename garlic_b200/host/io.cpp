// io.cpp — text loaders and writers of the GARLIC file formats (SURVEY.md §8b): tped / tfam / map / tgls /
// centromere inputs (plain or gz, read through zlib), .freq.gz / .kde / .roh.bed outputs.
#include <zlib.h>

#include <algorithm>
#include <cctype>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <sstream>

#include "garlic_host.h"

namespace gh {

namespace {

// Line reader over zlib (plain files pass through gzread untouched): 8 MB refills, newlines found with memchr,
// lines handed out as views into the buffer — the tped genotype columns are copied once (into Tped::text) and never
// looked at character by character on the host.
struct GzLines {
    gzFile f = nullptr;
    std::vector<char> buf;
    size_t pos = 0, end = 0;
    bool eof = false;
    bool open(const std::string& p)
    {
        f = gzopen(p.c_str(), "rb");
        if (f) gzbuffer(f, 1 << 20);
        buf.resize((size_t)8 << 20);
        pos = end = 0;
        eof = false;
        return f != nullptr;
    }
    // next line as [p, p+n) without the newline / trailing CR; valid until the following call; false at EOF
    bool next_view(const char*& p, size_t& n)
    {
        for (;;) {
            const char* nl = end > pos ? (const char*)memchr(buf.data() + pos, '\n', end - pos) : nullptr;
            if (nl || (eof && end > pos)) {
                const size_t stop = nl ? (size_t)(nl - buf.data()) : end;
                p = buf.data() + pos;
                n = stop - pos;
                pos = nl ? stop + 1 : end;
                if (n && p[n - 1] == '\r') --n;
                return true;
            }
            if (eof) return false;
            if (pos > 0) { memmove(buf.data(), buf.data() + pos, end - pos); end -= pos; pos = 0; }
            if (end == buf.size()) buf.resize(buf.size() * 2);          // a line longer than the buffer
            const int got = gzread(f, buf.data() + end, (unsigned)std::min<size_t>(buf.size() - end, (size_t)1 << 30));
            if (got <= 0) eof = true; else end += (size_t)got;
        }
    }
    // reads one line (without the newline) of any length; false at EOF
    bool next(std::string& line)
    {
        const char* p; size_t n;
        if (!next_view(p, n)) return false;
        line.assign(p, n);
        return true;
    }
    ~GzLines() { if (f) gzclose(f); }
};

inline const char* skip_ws(const char* p) { while (*p == ' ' || *p == '\t') ++p; return p; }
inline const char* skip_tok(const char* p) { while (*p && *p != ' ' && *p != '\t') ++p; return p; }

int count_fields(const std::string& s)
{
    int n = 0;
    const char* p = s.c_str();
    for (;;) {
        p = skip_ws(p);
        if (!*p) break;
        ++n;
        p = skip_tok(p);
    }
    return n;
}

struct CenRow { const char* build; const char* chr; int start, end; };
const CenRow kCen[] = {
#include "../csrc/centromere_table.inc"
};

}  // namespace

std::string chr_label(const std::string& name) { return (!name.empty() && name[0] == 'c') ? name : "chr" + name; }

// loadTPEDData's parsing (garlic-data.cpp:57-153): <chr> <id> <cM> <bp> then allele characters; the coding
// and counting of those characters is done on the GPU (K1).
bool load_tped(const std::string& path, char missing, Tped& t, bool host_tokenize)
{
    (void)missing;
    GzLines in;
    if (!in.open(path)) { LOG.error("ERROR: Failed to open " + path); return false; }
    std::string line, prev_chr;
    t = Tped();
    t.chr_off.push_back(0);
    t.text_off.push_back(0);
    int64_t cur = 0;
    while (in.next(line)) {
        if (host_tokenize || t.n_loci == 0) {
            // column count: every line on the host path; with K0 only the first line is counted here (it fixes the
            // number of individuals) and the GPU reports each line's allele count (main.cpp checks it)
            const int ncols = count_fields(line) - 4;
            if (ncols < 2) { LOG.error("ERROR: line " + std::to_string(t.n_loci + 1) + " of " + path + " has no genotypes."); return false; }
            const int n_ind = ncols / 2;
            if (t.n_loci == 0) t.n_ind = n_ind;
            else if (n_ind != t.n_ind) {
                LOG.error("ERROR: line " + std::to_string(t.n_loci + 1) + " of " + path + " has a different number of columns.");
                return false;
            }
        }
        const char* p = skip_ws(line.c_str());
        const char* e = skip_tok(p);
        std::string chr(p, e);
        if (t.n_loci == 0) prev_chr = chr;
        if (chr != prev_chr) {
            LOG.line("Chromosome " + chr_label(prev_chr) + ": " + std::to_string(cur) + " sites.");
            t.chr_names.push_back(prev_chr);
            t.chr_off.push_back(t.n_loci);
            prev_chr = chr;
            cur = 0;
        }
        ++cur;
        p = skip_ws(e); e = skip_tok(p);
        t.snp_id.emplace_back(p, e);
        p = skip_ws(e); e = skip_tok(p);          // genetic position column (unused: --map supplies cM)
        p = skip_ws(e); e = skip_tok(p);
        t.pos.push_back((int32_t)strtod(std::string(p, e).c_str(), nullptr));   // read as double, stored as int (:96-99)
        p = e;
        if (host_tokenize) {
            const size_t base = t.alleles.size();
            t.alleles.resize(base + (size_t)2 * t.n_ind);
            uint8_t* dst = t.alleles.data() + base;
            int k = 0;
            for (; *p && k < 2 * t.n_ind; ++p)      // operator>>(char&): successive non-blank characters
                if (*p != ' ' && *p != '\t') dst[k++] = (uint8_t)*p;
            if (k != 2 * t.n_ind) { LOG.error("ERROR: line " + std::to_string(t.n_loci + 1) + " of " + path + " is truncated."); return false; }
        } else {
            if (p == e && *p == 0) { LOG.error("ERROR: line " + std::to_string(t.n_loci + 1) + " of " + path + " has no genotypes."); return false; }
            t.text.insert(t.text.end(), p, line.c_str() + line.size());     // raw tail: tokenised by K0 on the GPU
            t.text_off.push_back((int64_t)t.text.size());
        }
        ++t.n_loci;
    }
    if (t.n_loci == 0) { LOG.error("ERROR: " + path + " is empty."); return false; }
    LOG.line("Chromosome " + chr_label(prev_chr) + ": " + std::to_string(cur) + " sites.");
    t.chr_names.push_back(prev_chr);
    t.chr_off.push_back(t.n_loci);
    return true;
}

// scanIndData3 / readIndData3 (garlic-data.cpp:1893-2014): single population, unique IDs.
bool load_tfam(const std::string& path, Tfam& f)
{
    GzLines in;
    if (!in.open(path)) { LOG.error("ERROR: Failed to open " + path); return false; }
    printf("Reading %s\n", path.c_str());
    std::string line;
    std::map<std::string, int> seen;
    int n = 0;
    while (in.next(line)) {
        ++n;
        const int cols = count_fields(line);
        if (cols < 2) {
            LOG.error("ERROR: Line " + std::to_string(n) + " of " + path + " has " + std::to_string(cols) + ", but expected at least 2");
            return false;
        }
        std::istringstream ss(line);
        std::string pop, id;
        ss >> pop >> id;
        if (seen.count(id)) { LOG.error("ERROR: Found duplicate individual ID (  " + id + " ) in " + path); return false; }
        seen[id] = 1;
        if (n == 1) f.pop = pop;
        else if (pop != f.pop) { LOG.error("ERROR: Found multiple population IDs (  " + pop + ", " + f.pop + " ) in " + path); return false; }
        f.ids.push_back(id);
    }
    if (n < 1) { LOG.error("ERROR: Number of individuals must be positive: 0"); return false; }
    return true;
}

bool load_bim(const std::string& path, Tped& t, std::vector<std::string>& a1, std::vector<std::string>& a2)
{
    GzLines in;
    if (!in.open(path)) { LOG.error("ERROR: Failed to open " + path); return false; }
    std::string line, prev_chr;
    t = Tped();
    t.chr_off.push_back(0);
    a1.clear();
    a2.clear();
    int64_t cur = 0;
    while (in.next(line)) {
        if (count_fields(line) != 6) {
            LOG.error("ERROR: line " + std::to_string(t.n_loci + 1) + " of " + path + " does not have 6 columns.");
            return false;
        }
        std::istringstream ss(line);
        std::string chr, id, cm, bp, x, y;
        ss >> chr >> id >> cm >> bp >> x >> y;
        if (t.n_loci == 0) prev_chr = chr;
        if (chr != prev_chr) {
            LOG.line("Chromosome " + chr_label(prev_chr) + ": " + std::to_string(cur) + " sites.");
            t.chr_names.push_back(prev_chr);
            t.chr_off.push_back(t.n_loci);
            prev_chr = chr;
            cur = 0;
        }
        ++cur;
        t.snp_id.push_back(id);
        t.pos.push_back((int32_t)strtod(bp.c_str(), nullptr));   // as load_tped reads the 4th column
        a1.push_back(x);
        a2.push_back(y);
        ++t.n_loci;
    }
    if (t.n_loci == 0) { LOG.error("ERROR: " + path + " is empty."); return false; }
    LOG.line("Chromosome " + chr_label(prev_chr) + ": " + std::to_string(cur) + " sites.");
    t.chr_names.push_back(prev_chr);
    t.chr_off.push_back(t.n_loci);
    return true;
}

bool open_bed(const std::string& path, int n_ind, int64_t n_loci, FILE*& f)
{
    f = fopen(path.c_str(), "rb");
    if (!f) { LOG.error("ERROR: Failed to open " + path); return false; }
    unsigned char head[3] = {0, 0, 0};
    const size_t got = fread(head, 1, 3, f);
    auto bad = [&](const std::string& why) { LOG.error("ERROR: " + path + ": " + why); fclose(f); f = nullptr; return false; };
    if (got < 3 || head[0] != 0x6c || head[1] != 0x1b) return bad("not a PLINK .bed file (the first bytes are not 6c 1b).");
    if (head[2] == 0) return bad("individual-major .bed (mode byte 00) is not supported; rewrite it SNP-major with plink --make-bed.");
    if (head[2] != 1) return bad("unknown .bed mode byte.");
    fseeko(f, 0, SEEK_END);
    const int64_t size = (int64_t)ftello(f), want = 3 + n_loci * (int64_t)((n_ind + 3) / 4);
    fseeko(f, 3, SEEK_SET);
    if (size != want)
        return bad("has " + std::to_string(size) + " bytes, but " + std::to_string(n_loci) + " SNPs (.bim) x " + std::to_string(n_ind) +
                   " individuals (.fam) need " + std::to_string(want) + ".");
    return true;
}

// loadMapScaffold (garlic-data.cpp:760-839): <chr> <id> <cM> <bp>, exactly four columns.
bool load_map(const std::string& path, std::vector<Scaffold>& out)
{
    GzLines in;
    fprintf(stderr, "Opening %s...\n", path.c_str());
    if (!in.open(path)) { fprintf(stderr, "ERROR: Failed to open %s for reading.\n", path.c_str()); return false; }
    std::string line, cur;
    int n = 0;
    while (in.next(line)) {
        ++n;
        const int cols = count_fields(line);
        if (cols != 4) { fprintf(stderr, "ERROR: line %d of %s has %d, but expected 4.\n", n, path.c_str(), cols); return false; }
        std::istringstream ss(line);
        std::string chr, id;
        double g, p;
        ss >> chr >> id >> g >> p;
        if (out.empty() || chr != cur) { out.emplace_back(); out.back().chr = chr_label(chr); cur = chr; }
        out.back().gen.push_back(g);
        out.back().pos.push_back((int32_t)p);
    }
    fprintf(stderr, "Loading genetic map scaffold for %d loci.\n", n);
    return true;
}

// readTGLSData's parsing (garlic-data.cpp:1516-1554): same SNP order/count as the tped, 4 + N columns; the
// GQ/GL/PL → error transform (:1555-1577) happens on the GPU.
bool load_tgls(const std::string& path, const Tped& t, std::vector<double>& v)
{
    GzLines in;
    fprintf(stderr, "Loading genotype likelihoods from %s\n", path.c_str());
    if (!in.open(path)) { LOG.error("ERROR: Failed to open " + path); return false; }
    v.assign((size_t)t.n_ind * t.n_loci, 0.0);
    std::string line;
    for (int64_t l = 0; l < t.n_loci; ++l) {
        if (!in.next(line)) line.clear();
        const int num = count_fields(line);
        if (num != t.n_ind + 4) {
            LOG.error("ERROR: Incorrect number of columns in tgls file:  " + std::to_string(num) + ". Expected:  " + std::to_string(t.n_ind));
            return false;
        }
        const char* p = line.c_str();
        for (int k = 0; k < 4; ++k) p = skip_tok(skip_ws(p));
        for (int i = 0; i < t.n_ind; ++i) {
            char* e;
            v[(size_t)i * t.n_loci + l] = strtod(p, &e);
            p = e;
        }
    }
    return true;
}

bool TglsBlocks::open(const std::string& path)
{
    GzLines* g = new GzLines;
    fprintf(stderr, "Loading genotype likelihoods from %s\n", path.c_str());
    if (!g->open(path)) { delete g; LOG.error("ERROR: Failed to open " + path); return false; }
    impl = g;
    return true;
}
int TglsBlocks::next(int max_lines, std::vector<char>& text, std::vector<int64_t>& off)
{
    GzLines* g = static_cast<GzLines*>(impl);
    text.clear();
    off.assign(1, 0);
    for (int l = 0; l < max_lines; ++l) {
        const char* p; size_t n;
        if (g->next_view(p, n)) {
            const char* e = p + n;
            const char* q = p;
            for (int k = 0; k < 4; ++k) {                       // <chr> <id> <cM> <bp>
                while (q < e && (*q == ' ' || *q == '\t')) ++q;
                while (q < e && *q != ' ' && *q != '\t') ++q;
            }
            text.insert(text.end(), q, e);
        }
        off.push_back((int64_t)text.size());
    }
    return max_lines;
}
TglsBlocks::~TglsBlocks() { delete static_cast<GzLines*>(impl); }

bool load_freq_file(const std::string& path, const Tped& t, const std::vector<std::string>& one, bool by_name,
                    std::vector<double>& freq)
{
    GzLines in;
    if (!in.open(path)) { LOG.error("ERROR: Failed to open " + path); return false; }
    fprintf(stderr, "Reading %s\n", path.c_str());
    std::string line;
    in.next(line);   // header
    freq.assign(t.n_loci, 0.0);
    int prev_cols = -1;
    for (int64_t l = 0; l < t.n_loci; ++l) {
        const int64_t line_no = l + 2;
        if (!in.next(line)) { LOG.error("ERROR: at line " + std::to_string(line_no) + " in " + path + ". Perhaps too few lines?"); return false; }
        const int cols = count_fields(line);
        if (cols < 5) { LOG.error("ERROR: Found " + std::to_string(cols) + " in " + path + " on line " + std::to_string(line_no) + " but expected at least 5"); return false; }
        if (cols != prev_cols && prev_cols != -1) { LOG.error("ERROR: Differing number of columns across rows found in " + path); return false; }
        prev_cols = cols;
        std::istringstream ss(line);
        std::string chr, id, name;
        double pos, f;
        char allele;
        if (by_name) ss >> chr >> id >> pos >> name >> f;
        else ss >> chr >> id >> pos >> allele >> f;
        if (id != t.snp_id[l]) {
            LOG.error("ERROR: Loci appear mismatched in: " + path);
            LOG.error("ERROR: at line: " + std::to_string(line_no));
            LOG.error("ERROR: freq file locus name: " + id);
            LOG.error("ERROR: tped file locus name: " + t.snp_id[l]);
            return false;
        }
        freq[l] = (by_name ? name != one[l] : allele != one[l][0]) ? 1 - f : f;
    }
    if (in.next(line) && !line.empty()) { LOG.error("ERROR: " + path + " has more rows than the tped file has loci."); return false; }
    return true;
}

// class centromere (garlic-centromeres.cpp:3-101): built-in hg18/hg19/hg38 tables or a custom file.
bool load_centromeres(const std::string& build, const std::string& file, std::map<std::string, std::pair<int, int>>& cen)
{
    cen.clear();
    if (build == "hg18" || build == "hg19" || build == "hg38") {
        for (const CenRow& r : kCen)
            if (build == r.build) cen[r.chr] = {r.start, r.end};
        return true;
    }
    if (file != "none") {
        GzLines in;
        if (!in.open(file)) { LOG.error("ERROR: Could not open " + file); return false; }
        std::string line;
        int n = 0;
        while (in.next(line)) {
            ++n;
            const int cols = count_fields(line);
            if (cols != 3) { LOG.error("ERROR: Custom centromere file requires three columns.  Found " + std::to_string(cols)); continue; }
            std::istringstream ss(line);
            std::string chr;
            int s, e;
            ss >> chr >> s >> e;
            cen[chr_label(chr)] = {s, e};
        }
        fprintf(stderr, "Loaded custom centromere limits for %d chromosomes.\n", n);
    }
    return true;
}

// interpolateGeneticmap → getMapInfo → interpolate (garlic-data.cpp:702-757): exact scaffold hits take the
// scaffold value (map<int,int> lookup, last duplicate wins); other positions use
// ((y1-y0)/(x1-x0))*q + (y0 - ((y1-y0)/(x1-x0))*x0) between the bracketing scaffold sites (forward cursor).
bool interpolate_map(const int32_t* pos, int64_t n, const Scaffold& s, double* gpos, int& n_interp)
{
    const int S = (int)s.pos.size();
    std::map<int, int> hit;
    for (int k = 0; k < S; ++k) hit[s.pos[k]] = k;
    int cur = 0;
    for (int64_t i = 0; i < n; ++i) {
        const int q = pos[i];
        auto it = hit.find(q);
        if (it != hit.end()) { gpos[i] = s.gen[it->second]; continue; }
        if (S < 2 || q < s.pos[0] || q > s.pos[S - 1]) return false;
        int a = -1;
        for (; cur < S - 1; ++cur)
            if (q > s.pos[cur] && q < s.pos[cur + 1]) { a = cur; break; }
        if (a < 0) return false;
        const double x0 = s.pos[a], y0 = s.gen[a], x1 = s.pos[a + 1], y1 = s.gen[a + 1];
        gpos[i] = (((y1 - y0) / (x1 - x0)) * q + (y0 - ((y1 - y0) / (x1 - x0)) * x0));
        ++n_interp;
    }
    return true;
}

// writeFreqData (garlic-data.cpp:1311-1343): all loci before filtering, 6 significant digits.
bool write_freq_gz(const std::string& path, const Tped& t, const std::vector<std::string>& one, const std::vector<double>& freq)
{
    gzFile f = gzopen(path.c_str(), "wb");
    if (!f) { LOG.error("ERROR: Failed to open " + path); return false; }
    gzputs(f, "CHR\tSNP\tPOS\tALLELE\tFREQ\n");
    std::string row;
    for (size_t c = 0; c + 1 < t.chr_off.size(); ++c) {
        const std::string lab = chr_label(t.chr_names[c]);
        for (int64_t l = t.chr_off[c]; l < t.chr_off[c + 1]; ++l) {
            row = lab + "\t" + t.snp_id[l] + "\t" + std::to_string(t.pos[l]) + "\t" + one[l] + "\t" + fmt_g(freq[l]) + "\n";
            gzwrite(f, row.data(), (unsigned)row.size());
        }
    }
    gzclose(f);
    printf("Wrote allele frequency data to %s\n", path.c_str());
    return true;
}

bool write_kde(const Kde& k, const std::string& path)
{
    FILE* f = fopen(path.c_str(), "w");
    if (!f) { LOG.error("ERROR: Failed to open " + path); return false; }
    for (size_t i = 0; i < k.x.size(); ++i) fprintf(f, "%s %s\n", fmt_g(k.x[i]).c_str(), fmt_g(k.y[i]).c_str());
    fclose(f);
    LOG.line("Wrote KDE results to " + path);
    return true;
}

// writeROHData (garlic-roh.cpp:574-644)
bool write_bed(const std::string& path, const std::vector<Roh>& roh, const std::vector<std::string>& ids,
               const std::vector<std::string>& chr_labels, const std::vector<double>& bounds, const std::string& pop, bool cm)
{
    static const char* colors[9] = {"228,26,28", "77,175,74", "55,126,184", "152,78,163", "255,127,0",
                                    "255,255,51", "166,86,40", "247,129,191", "153,153,153"};
    FILE* f = fopen(path.c_str(), "w");
    if (!f) { LOG.error("ERROR: Failed to open " + path); return false; }
    size_t r = 0;
    for (size_t ind = 0; ind < ids.size(); ++ind) {
        fprintf(f, "track name=\"Ind: %s Pop:%s ROH\" description=\"Ind: %s Pop:%s ROH from GARLIC v%s\" visibility=2 itemRgb=\"On\"\n",
                ids[ind].c_str(), pop.c_str(), ids[ind].c_str(), pop.c_str(), kVersion);
        for (; r < roh.size() && roh[r].ind == (int)ind; ++r) {
            const double size = roh[r].length;
            size_t i = 0;
            while (i < bounds.size() && !(size < bounds[i])) ++i;
            const char cls = (char)('A' + i);
            const char* color = colors[i <= 8 ? i : 8];
            std::string chr = chr_labels[roh[r].chr];
            if (chr[0] != 'c' && chr[0] != 'C') chr = "chr" + chr;
            if (cm) fprintf(f, "%s\t%d\t%d\t%c\t%s\t.\t0\t0\t%s\n", chr.c_str(), (int)roh[r].start, (int)roh[r].stop, cls, fmt_g(size).c_str(), color);
            else fprintf(f, "%s\t%d\t%d\t%c\t%d\t.\t0\t0\t%s\n", chr.c_str(), (int)roh[r].start, (int)roh[r].stop, cls, (int)size, color);
        }
    }
    fclose(f);
    LOG.line("ROH calls: " + path);
    return true;
}

}  // namespace gh
