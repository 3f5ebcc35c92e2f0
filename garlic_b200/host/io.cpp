// io.cpp — text loaders and writers of the GARLIC file formats (SURVEY.md §8b): tped / tfam / map / tgls /
// centromere inputs (plain or gz, read through zlib), VCF (plain, gz or BGZF), .freq.gz / .kde / .roh.bed outputs.
#include <zlib.h>

#include <algorithm>
#include <cctype>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <set>
#include <sstream>
#include <thread>

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

// BGZF, the blocked gzip of VCF files: a series of gzip members of at most 64 KiB each, whose total size is in the 'BC'
// extra subfield (BSIZE = size - 1) and whose inflated size is in the ISIZE trailer.  So every block's input and output
// offsets are known before any is inflated: a batch of blocks is read, inflated with raw zlib inflate on
// min(hardware_concurrency, 16) threads, and each block's CRC32 and ISIZE are checked.  Lines are served like
// GzLines::next_view serves them, across block and batch boundaries.
struct BgzfLines {
    FILE* f = nullptr;
    std::string path, err;                     // err: why reading stopped early (truncated block, bad CRC, ...)
    std::vector<unsigned char> in;             // the compressed blocks of the current batch
    std::vector<char> buf;
    size_t pos = 0, end = 0;
    bool eof = false;
    int threads = 1;
    static constexpr size_t kBatch = 1024;     // blocks per batch: at most 64 MiB inflated

    // true if the file starts with a BGZF block header (gzip, FEXTRA, first subfield 'BC' of length 2)
    static bool sniff(const std::string& p)
    {
        FILE* g = fopen(p.c_str(), "rb");
        if (!g) return false;
        unsigned char h[16];
        const bool ok = fread(h, 1, 16, g) == 16 && h[0] == 31 && h[1] == 139 && h[2] == 8 && (h[3] & 4) &&
                        h[12] == 'B' && h[13] == 'C' && h[14] == 2 && h[15] == 0;
        fclose(g);
        return ok;
    }
    bool open(const std::string& p)
    {
        path = p;
        f = fopen(p.c_str(), "rb");
        threads = (int)std::min(16u, std::max(1u, std::thread::hardware_concurrency()));
        return f != nullptr;
    }
    bool fail(const std::string& why) { err = path + ": " + why; return false; }
    // reads and inflates the next batch of blocks behind the unread bytes; false at the end of the file or on an error
    bool refill()
    {
        struct Block { size_t in_off, in_len, out_off; uint32_t crc, isize; };
        std::vector<Block> blocks;
        in.clear();
        size_t out_total = 0;
        while (blocks.size() < kBatch) {
            unsigned char h[12];
            const size_t got = fread(h, 1, 12, f);
            if (got == 0) break;
            if (got < 12) return fail("truncated BGZF block header.");
            if (h[0] != 31 || h[1] != 139 || h[2] != 8 || !(h[3] & 4)) return fail("not a BGZF block header.");
            const size_t xlen = h[10] | (size_t)h[11] << 8;
            std::vector<unsigned char> x(xlen);
            if (fread(x.data(), 1, xlen, f) != xlen) return fail("truncated BGZF block header.");
            long bsize = -1;
            for (size_t q = 0; q + 4 <= xlen;) {
                const size_t slen = x[q + 2] | (size_t)x[q + 3] << 8;
                if (x[q] == 'B' && x[q + 1] == 'C' && slen == 2 && q + 6 <= xlen) bsize = x[q + 4] | (long)x[q + 5] << 8;
                q += 4 + slen;
            }
            if (bsize < 0) return fail("a gzip member without the BGZF block size (BC subfield).");
            const long rest = bsize + 1 - 12 - (long)xlen;
            if (rest < 8) return fail("BGZF block size smaller than its header.");
            const size_t base = in.size();
            in.resize(base + rest);
            if (fread(in.data() + base, 1, rest, f) != (size_t)rest) return fail("truncated BGZF block.");
            const unsigned char* t = in.data() + base + rest - 8;
            const uint32_t crc = t[0] | t[1] << 8 | t[2] << 16 | (uint32_t)t[3] << 24;
            const uint32_t isize = t[4] | t[5] << 8 | t[6] << 16 | (uint32_t)t[7] << 24;
            if (isize > 65536) return fail("BGZF block with ISIZE above 64 KiB.");
            blocks.push_back({base, (size_t)rest - 8, out_total, crc, isize});
            out_total += isize;
        }
        if (blocks.empty()) return false;
        if (pos > 0) { memmove(buf.data(), buf.data() + pos, end - pos); end -= pos; pos = 0; }
        if (buf.size() < end + out_total) buf.resize(end + out_total);
        std::vector<char> bad(blocks.size(), 0);
        auto work = [&](int id) {
            for (size_t k = id; k < blocks.size(); k += threads) {
                const Block& b = blocks[k];
                char dummy;
                Bytef* dst = b.isize ? (Bytef*)buf.data() + end + b.out_off : (Bytef*)&dummy;
                z_stream zs;
                memset(&zs, 0, sizeof(zs));
                if (inflateInit2(&zs, -15) != Z_OK) { bad[k] = 1; continue; }
                zs.next_in = in.data() + b.in_off;
                zs.avail_in = (uInt)b.in_len;
                zs.next_out = dst;
                zs.avail_out = b.isize ? b.isize : 1;
                const int rc = inflate(&zs, Z_FINISH);
                if (rc != Z_STREAM_END || zs.total_out != b.isize) bad[k] = 1;
                else if (crc32(0L, dst, b.isize) != b.crc) bad[k] = 2;
                inflateEnd(&zs);
            }
        };
        const int nt = (int)std::min<size_t>(threads, blocks.size());
        std::vector<std::thread> pool;
        for (int id = 1; id < nt; ++id) pool.emplace_back(work, id);
        work(0);
        for (auto& th : pool) th.join();
        for (size_t k = 0; k < blocks.size(); ++k)
            if (bad[k]) return fail(bad[k] == 2 ? "CRC32 mismatch in a BGZF block." : "corrupt BGZF block (inflate failed or ISIZE mismatch).");
        end += out_total;
        return true;
    }
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
            if (!refill()) eof = true;
            if (!err.empty()) return false;
        }
    }
    ~BgzfLines() { if (f) fclose(f); }
};

std::string read_error(const GzLines&) { return ""; }
std::string read_error(const BgzfLines& b) { return b.err; }

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

// VCF: '##' meta lines, the '#CHROM' header (its columns after FORMAT are the samples), then one record per line with
// 9 tab-separated fixed columns and the sample columns.  CHROM / ID / POS take the places of the tped's columns 1 / 2 / 4;
// the sample text is kept raw, as load_tped keeps its genotype columns, and parsed on the GPU (vcf.cu).
template <class Lines>
bool parse_vcf(Lines& in, const std::string& path, Tped& t, Vcf& v)
{
    t = Tped();
    v = Vcf();
    t.chr_off.push_back(0);
    t.text_off.push_back(0);
    const char* p;
    size_t n;
    int64_t line_no = 0, cur = 0;
    std::string prev_chr;
    bool header = false;
    while (in.next_view(p, n)) {
        ++line_no;
        const char* e = p + n;
        auto bad = [&](const std::string& where, const std::string& why) {
            LOG.error("ERROR: " + path + " line " + std::to_string(line_no) + where + ": " + why);
            return false;
        };
        if (!header) {
            if (n >= 2 && p[0] == '#' && p[1] == '#') continue;
            if (n < 6 || memcmp(p, "#CHROM", 6) != 0) return bad("", "no #CHROM header line before the first record.");
            std::vector<std::string> cols;
            for (const char* q = p;;) {
                const char* tab = (const char*)memchr(q, '\t', e - q);
                cols.emplace_back(q, tab ? tab : e);
                if (!tab) break;
                q = tab + 1;
            }
            if (cols.size() < 9 || cols[8] != "FORMAT") return bad("", "the #CHROM header has no FORMAT column.");
            if (cols.size() == 9) return bad("", "the #CHROM header names no samples.");
            std::set<std::string> seen;
            for (size_t k = 9; k < cols.size(); ++k) {
                if (!seen.insert(cols[k]).second) return bad("", "duplicate sample ID ( " + cols[k] + " ).");
                v.samples.push_back(cols[k]);
            }
            t.n_ind = (int)v.samples.size();
            header = true;
            continue;
        }
        if (n == 0) continue;
        const char* f[9];
        size_t fl[9];
        const char* q = p;
        int k = 0;
        while (k < 9 && q) {
            const char* tab = (const char*)memchr(q, '\t', e - q);
            f[k] = q;
            fl[k] = (size_t)((tab ? tab : e) - q);
            q = tab ? tab + 1 : nullptr;
            ++k;
        }
        const std::string chr(f[0], fl[0]);
        const std::string pos_text = k > 1 ? std::string(f[1], fl[1]) : std::string();
        const std::string where = " (" + chr + ":" + pos_text + ")";
        if (k < 9) return bad(where, "fewer than 9 fixed columns (CHROM POS ID REF ALT QUAL FILTER INFO FORMAT).");
        bool num = !pos_text.empty() && pos_text.size() <= 10;
        for (char c : pos_text) num = num && c >= '0' && c <= '9';
        if (!num || strtoll(pos_text.c_str(), nullptr, 10) > INT32_MAX) return bad(where, "POS is not an integer.");
        if (!(fl[8] == 2 || (fl[8] > 2 && f[8][2] == ':')) || f[8][0] != 'G' || f[8][1] != 'T')
            return bad(where, "FORMAT does not start with GT (" + std::string(f[8], fl[8]) + ").");
        if (t.n_loci == 0) prev_chr = chr;
        if (chr != prev_chr) {
            LOG.line("Chromosome " + chr_label(prev_chr) + ": " + std::to_string(cur) + " sites.");
            t.chr_names.push_back(prev_chr);
            t.chr_off.push_back(t.n_loci);
            prev_chr = chr;
            cur = 0;
        }
        ++cur;
        t.snp_id.emplace_back(f[2], fl[2]);
        t.pos.push_back((int32_t)strtod(pos_text.c_str(), nullptr));
        v.ref.emplace_back(f[3], fl[3]);
        v.alts.emplace_back();
        if (!(fl[4] == 1 && f[4][0] == '.'))
            for (const char *a = f[4], *ae = f[4] + fl[4];;) {
                const char* c = (const char*)memchr(a, ',', ae - a);
                v.alts.back().emplace_back(a, c ? c : ae);
                if (!c) break;
                a = c + 1;
            }
        v.line.push_back(line_no);
        if (q) t.text.insert(t.text.end(), q, e);      // the sample columns: parsed on the GPU
        t.text_off.push_back((int64_t)t.text.size());
        ++t.n_loci;
    }
    const std::string rerr = read_error(in);
    if (!rerr.empty()) { LOG.error("ERROR: " + rerr); return false; }
    if (!header) { LOG.error("ERROR: " + path + " has no #CHROM header line."); return false; }
    if (t.n_loci == 0) { LOG.error("ERROR: " + path + " has no records."); return false; }
    LOG.line("Chromosome " + chr_label(prev_chr) + ": " + std::to_string(cur) + " sites.");
    t.chr_names.push_back(prev_chr);
    t.chr_off.push_back(t.n_loci);
    return true;
}

bool load_vcf(const std::string& path, Tped& t, Vcf& v)
{
    if (BgzfLines::sniff(path)) {
        BgzfLines in;
        if (!in.open(path)) { LOG.error("ERROR: Failed to open " + path); return false; }
        return parse_vcf(in, path, t, v);
    }
    GzLines in;
    if (!in.open(path)) { LOG.error("ERROR: Failed to open " + path); return false; }
    return parse_vcf(in, path, t, v);
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
