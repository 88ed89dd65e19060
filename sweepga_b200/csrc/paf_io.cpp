// paf_io.cpp — host side of the drop-in boundary: PAF text -> compact SoA, tagged writer,
// filter_paf / filter_file, and the multi-GPU shard planner.  Parsing stays on the host
// (north_star); it is chunked over all host threads and emits the u32 SoA the kernels eat.
//
//   swg_paf_parse   <- PafFilter::extract_metadata  (src/paf_filter.rs:292-376)
//                      + paf::parse_cigar_counts    (src/paf.rs:32-64)
//   swg_paf_write   <- write_filtered_output        (src/paf_filter.rs:1689-1726)
//   swg_filter_paf  <- PafFilter::filter_paf        (src/paf_filter.rs:278-289)
//   swg_filter_file <- unified_filter::filter_file  (src/unified_filter.rs:280-347)
#include <algorithm>
#include <cerrno>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <sys/wait.h>
#include <unistd.h>
#include <zlib.h>

#include "sweepga_b200.h"
#include "host_util.h"

extern "C" void swg__set_error(swg_ctx *ctx, const char *msg); // filter_pipeline.cu

using swg::rust_parse_f64;
using swg::rust_parse_u64;

#include "paf_host.h"

namespace {

struct Chunk {
    size_t begin = 0, end = 0;
    uint64_t n_lines = 0;
    std::vector<uint64_t> rank_local, line_off;
    std::vector<uint32_t> line_len, qid, tid, qs, qe, ts, te, blen, matches;
    std::vector<double> identity;
    std::vector<uint8_t> strand;
    std::vector<std::string> names; // local name table (first appearance within the chunk)
    std::string error;
};

struct SvHash {
    size_t operator()(const std::string &s) const { return std::hash<std::string>()(s); }
};

static inline bool parse_u64_field(const char *s, size_t len, uint64_t dflt, uint64_t *out) {
    uint64_t v;
    if (rust_parse_u64(s, len, &v)) { *out = v; return true; }
    *out = dflt; // unwrap_or(default), paf_filter.rs:308-317
    return true;
}

// Σ of '=' run lengths; false when the reference's parse_cigar_counts would return Err
static bool cigar_eq_count(const char *s, size_t len, uint64_t *out) {
    uint64_t m = 0, num = 0;
    bool have = false, overflow = false;
    for (size_t i = 0; i < len; i++) {
        unsigned d = (unsigned)(s[i] - '0');
        if (d <= 9) {
            if (num > (~(uint64_t)0 - d) / 10) overflow = true;
            num = num * 10 + d;
            have = true;
        } else {
            if (!have || overflow) return false; // "".parse::<u64>() / overflow is Err
            if (s[i] == '=') m += num;
            num = 0;
            have = false;
        }
    }
    *out = m;
    return true;
}

// Splits the first 11 tab-separated fields of a line into fs / fl.  Returns the offset of the tags (len + 1 when there
// are none), or 0 when the line has fewer than 11 fields.
static size_t split_fields(const char *line, size_t len, const char *fs[11], size_t fl[11]) {
    size_t a = 0;
    for (int nf = 0; nf < 11; nf++) {
        const char *tab = (const char *)memchr(line + a, '\t', len - a);
        const size_t b = tab ? (size_t)(tab - line) : len;
        fs[nf] = line + a;
        fl[nf] = b - a;
        if (!tab) return nf == 10 ? len + 1 : 0;
        a = b + 1;
    }
    return a;
}

} // namespace

swg::PafLine::Kind swg::paf_parse_line(const char *line, size_t len, PafLine *out) {
    const char *fs[11];
    size_t fl[11];
    size_t a = split_fields(line, len, fs, fl);
    if (a == 0) return PafLine::SKIP; // fewer than 11 fields: skipped, still consumes a rank
    uint64_t qs, qe, ts, te, mt, bl;
    parse_u64_field(fs[2], fl[2], 0, &qs);
    parse_u64_field(fs[3], fl[3], 0, &qe);
    parse_u64_field(fs[7], fl[7], 0, &ts);
    parse_u64_field(fs[8], fl[8], 0, &te);
    parse_u64_field(fs[9], fl[9], 0, &mt);
    parse_u64_field(fs[10], fl[10], 1, &bl);
    double identity = (double)mt / (double)(bl > 1 ? bl : 1);
    uint64_t exact = mt;
    // tags from column 12 on, in order, the later one wins (paf_filter.rs:326-343)
    while (a <= len) {
        const char *tab = a < len ? (const char *)memchr(line + a, '\t', len - a) : nullptr;
        size_t b = tab ? (size_t)(tab - line) : len;
        const char *f = line + a;
        size_t flen = b - a;
        if (flen >= 5 && memcmp(f, "dv:f:", 5) == 0) {
            double dv;
            if (rust_parse_f64(f + 5, flen - 5, &dv)) identity = 1.0 - dv;
        } else if (flen >= 5 && memcmp(f, "cg:Z:", 5) == 0) {
            uint64_t cm;
            if (cigar_eq_count(f + 5, flen - 5, &cm) && cm > 0) {
                exact = cm;
                identity = (double)cm / (double)(bl > 1 ? bl : 1);
            }
        }
        if (!tab) break;
        a = b + 1;
    }
    // A value beyond the u32 SoA, or end < start, does not reject the file here: the reference parses u64 and lets such a
    // record through to its stage-1 retain (paf_filter.rs:384-388), so the record is kept with an impossible interval
    // (query_start = 2^32 - 1 > query_end = 0 when a value had to be saturated; the original values when only the order is
    // wrong) and the filter raises SWG_ERR_RANGE only if it survives that retain (k_prefilter).  identity uses the exact u64s.
    const uint64_t LIM = 0xFFFFFFFFull;
    PafLine::Kind kind = PafLine::OK;
    if (qs > LIM || qe > LIM || ts > LIM || te > LIM || bl > LIM || exact > LIM) {
        kind = PafLine::ERR_RANGE;
        qs = LIM; qe = 0;
        ts = ts > LIM ? LIM : ts; te = te > LIM ? LIM : te; bl = bl > LIM ? LIM : bl; exact = exact > LIM ? LIM : exact;
    } else if (qe < qs || te < ts) kind = PafLine::ERR_ORDER;
    out->qname = fs[0]; out->qname_len = fl[0];
    out->tname = fs[5]; out->tname_len = fl[5];
    out->qs = (uint32_t)qs; out->qe = (uint32_t)qe; out->ts = (uint32_t)ts; out->te = (uint32_t)te;
    out->blen = (uint32_t)bl; out->matches = (uint32_t)exact;
    out->identity = identity;
    out->strand = (fl[4] == 1 && fs[4][0] == '+') ? '+' : '-';
    return kind;
}

bool swg::paf_ani_line(const char *line, size_t len, AniLine *out) {
    if (len == 0 || line[0] == '#') return false; // main.rs:414-416
    const char *fs[11];
    size_t fl[11];
    size_t a = split_fields(line, len, fs, fl);
    if (a == 0) return false;
    out->qname = fs[0]; out->qname_len = fl[0];
    out->tname = fs[5]; out->tname_len = fl[5];
    if (!rust_parse_u64(fs[1], fl[1], &out->qlen)) out->qlen = 0;
    if (!rust_parse_u64(fs[6], fl[6], &out->tlen)) out->tlen = 0;
    double m, b;
    if (!rust_parse_f64(fs[9], fl[9], &m)) m = 0.0;
    if (!rust_parse_f64(fs[10], fl[10], &b)) b = 1.0;
    double fm = m;
    while (a <= len) { // the first dv:f: tag that parses (main.rs:445-453)
        const char *tab = a < len ? (const char *)memchr(line + a, '\t', len - a) : nullptr;
        size_t e = tab ? (size_t)(tab - line) : len;
        if (e - a >= 5 && memcmp(line + a, "dv:f:", 5) == 0) {
            double dv;
            if (rust_parse_f64(line + a + 5, e - a - 5, &dv)) { fm = (1.0 - dv) * b; break; }
        }
        if (!tab) break;
        a = e + 1;
    }
    out->matches = fm;
    out->block = b;
    return true;
}

bool swg::paf_tree_line(const char *line, size_t len, AniLine *out, uint64_t *matches, uint64_t *block) {
    if (len == 0 || line[0] == '#') return false; // tree_filter.rs:221-223
    const char *fs[11];
    size_t fl[11];
    if (split_fields(line, len, fs, fl) == 0) return false;
    out->qname = fs[0]; out->qname_len = fl[0];
    out->tname = fs[5]; out->tname_len = fl[5];
    if (!rust_parse_u64(fs[9], fl[9], matches)) *matches = 0;
    if (!rust_parse_u64(fs[10], fl[10], block)) *block = 1;
    return true;
}

uint64_t swg::siphash13_zero_key(const uint8_t *msg, size_t len) {
    uint64_t v[4] = {0x736f6d6570736575ull, 0x646f72616e646f6dull, 0x6c7967656e657261ull, 0x7465646279746573ull};
    auto rotl = [](uint64_t x, int b) { return (x << b) | (x >> (64 - b)); };
    auto sipround = [&]() {
        v[0] += v[1]; v[1] = rotl(v[1], 13); v[1] ^= v[0]; v[0] = rotl(v[0], 32);
        v[2] += v[3]; v[3] = rotl(v[3], 16); v[3] ^= v[2];
        v[0] += v[3]; v[3] = rotl(v[3], 21); v[3] ^= v[0];
        v[2] += v[1]; v[1] = rotl(v[1], 17); v[1] ^= v[2]; v[2] = rotl(v[2], 32);
    };
    const size_t full = len & ~(size_t)7;
    for (size_t i = 0; i < full; i += 8) {
        uint64_t m;
        memcpy(&m, msg + i, 8); // little endian host
        v[3] ^= m;
        sipround(); // c = 1
        v[0] ^= m;
    }
    uint64_t last = (uint64_t)len << 56;
    for (size_t i = full; i < len; i++) last |= (uint64_t)msg[i] << (8 * (i - full));
    v[3] ^= last;
    sipround();
    v[0] ^= last;
    v[2] ^= 0xff;
    for (int r = 0; r < 3; r++) sipround(); // d = 3
    return v[0] ^ v[1] ^ v[2] ^ v[3];
}

std::vector<uint8_t> swg::tree_select_pairs(const std::vector<std::string> &genomes, const std::vector<uint32_t> &lo,
                                            const std::vector<uint32_t> &hi, const std::vector<double> &identity, uint64_t k_nearest,
                                            uint64_t k_farthest, double random_fraction, bool *has_nan) {
    const size_t np = lo.size();
    std::vector<uint8_t> sel(np, 0);
    *has_nan = false;
    for (double v : identity)
        if (v != v) { *has_nan = true; return sel; }
    // adjacency: for every genome the (pair index, other genome) list
    std::vector<std::vector<uint32_t>> adj(genomes.size());
    for (size_t p = 0; p < np; p++) { adj[lo[p]].push_back((uint32_t)p); adj[hi[p]].push_back((uint32_t)p); }
    for (size_t g = 0; g < genomes.size(); g++) {
        auto &v = adj[g];
        auto other = [&](uint32_t p) { return lo[p] == g ? hi[p] : lo[p]; };
        // identity descending; `genomes` is sorted, so the index order of the other genome is its name order
        std::sort(v.begin(), v.end(), [&](uint32_t x, uint32_t y) { return identity[x] != identity[y] ? identity[x] > identity[y] : other(x) < other(y); });
        for (size_t k = 0; k < v.size() && k < k_nearest; k++) sel[v[k]] = 1;
        for (size_t k = 0; k < v.size() && k < k_farthest; k++) sel[v[v.size() - 1 - k]] = 1;
    }
    if (random_fraction > 0.0) {
        const double t = random_fraction * 18446744073709551616.0; // u64::MAX as f64
        const uint64_t thr = t >= 18446744073709551616.0 ? ~(uint64_t)0 : (uint64_t)t; // `as u64` saturates
        std::string msg;
        for (size_t p = 0; p < np; p++) {
            msg.assign(genomes[lo[p]]);
            msg.push_back((char)0xff); // str::hash: the bytes, then 0xff
            msg.append(genomes[hi[p]]);
            msg.push_back((char)0xff);
            if (siphash13_zero_key((const uint8_t *)msg.data(), msg.size()) <= thr) sel[p] = 1;
        }
    }
    return sel;
}

namespace {

static void parse_chunk(const char *text, Chunk &c) {
    std::unordered_map<std::string, uint32_t, SvHash> ids;
    std::string last_q, last_t;
    uint32_t last_qid = 0, last_tid = 0;
    bool have_q = false, have_t = false;
    auto intern = [&](const char *s, size_t len, std::string &last, uint32_t &last_id, bool &have) -> uint32_t {
        if (have && last.size() == len && memcmp(last.data(), s, len) == 0) return last_id;
        last.assign(s, len);
        auto it = ids.find(last);
        uint32_t id;
        if (it == ids.end()) {
            id = (uint32_t)c.names.size();
            ids.emplace(last, id);
            c.names.push_back(last);
        } else id = it->second;
        last_id = id;
        have = true;
        return id;
    };
    size_t pos = c.begin;
    uint64_t ln = 0;
    swg::PafLine L;
    while (pos < c.end) {
        const char *nl = (const char *)memchr(text + pos, '\n', c.end - pos);
        size_t eol = nl ? (size_t)(nl - text) : c.end;
        size_t len = eol - pos;
        if (len > 0 && text[eol - 1] == '\r') len--; // BufRead::lines strips "\r\n"
        uint64_t this_ln = ln++;
        size_t next = nl ? eol + 1 : c.end;
        const swg::PafLine::Kind kind = swg::paf_parse_line(text + pos, len, &L);
        if (kind != swg::PafLine::SKIP) { // ERR_RANGE / ERR_ORDER lines are records with an impossible interval (see paf_parse_line)
            uint32_t q = intern(L.qname, L.qname_len, last_q, last_qid, have_q);
            uint32_t t = intern(L.tname, L.tname_len, last_t, last_tid, have_t);
            c.rank_local.push_back(this_ln);
            c.line_off.push_back(pos);
            c.line_len.push_back((uint32_t)len);
            c.qid.push_back(q); c.tid.push_back(t);
            c.qs.push_back(L.qs); c.qe.push_back(L.qe); c.ts.push_back(L.ts); c.te.push_back(L.te);
            c.blen.push_back(L.blen); c.matches.push_back(L.matches);
            c.identity.push_back(L.identity);
            c.strand.push_back(L.strand);
        }
        pos = next;
    }
    c.n_lines = ln;
}

template <class T> static void append(std::vector<T> &dst, const std::vector<T> &src) { dst.insert(dst.end(), src.begin(), src.end()); }

} // namespace

std::string swg::paf_prefix_P(const std::string &n) { // src/paf_filter.rs:1022-1030
    size_t p = n.rfind('#');
    return p == std::string::npos ? n : n.substr(0, p + 1);
}
std::string swg::paf_prefix_P2(const std::string &n) { // src/plane_sweep_scaffold.rs:13-22
    size_t p = n.find('#');
    if (p == std::string::npos) return n;
    size_t p2 = n.find('#', p + 1);
    std::string f1 = p2 == std::string::npos ? n.substr(p + 1) : n.substr(p + 1, p2 - p - 1);
    return n.substr(0, p) + "#" + f1 + "#";
}

void swg::paf_prefix_ids(const std::vector<std::string> &names, std::vector<uint32_t> *P, std::vector<uint32_t> *P2) {
    std::unordered_map<std::string, uint32_t> pid, p2id;
    P->clear(); P2->clear();
    P->reserve(names.size()); P2->reserve(names.size());
    for (const auto &n : names) {
        auto ia = pid.emplace(paf_prefix_P(n), (uint32_t)pid.size()).first;
        auto ib = p2id.emplace(paf_prefix_P2(n), (uint32_t)p2id.size()).first;
        P->push_back(ia->second);
        P2->push_back(ib->second);
    }
}

bool swg::paf_open_text(const char *path, swg_paf *p, std::string *err) {
    auto fail = [&](const std::string &m) { *err = m; return false; };
    if (!path) return fail("NULL path");
    // open_paf_input (src/paf.rs:10-28): extension "gz" / "bgz" => bgzf (= multi-member gzip) reader
    const char *dot = strrchr(path, '.');
    const char *slash = strrchr(path, '/');
    const bool compressed = dot && (!slash || dot > slash) && (strcmp(dot, ".gz") == 0 || strcmp(dot, ".bgz") == 0);
    int fd = open(path, O_RDONLY);
    if (fd < 0) return fail(std::string("cannot open ") + path);
    struct stat sb;
    if (fstat(fd, &sb) != 0) { close(fd); return fail("fstat failed"); }
    if (compressed) {
        gzFile gz = gzdopen(fd, "rb");
        if (!gz) { close(fd); return fail("gzdopen failed"); }
        gzbuffer(gz, 1 << 20);
        size_t cap = (size_t)sb.st_size * 4 + (1 << 20), got = 0;
        p->owned.resize(cap);
        while (true) {
            if (got == p->owned.size()) p->owned.resize(p->owned.size() * 2);
            int r = gzread(gz, p->owned.data() + got, (unsigned)std::min<size_t>(p->owned.size() - got, (size_t)1 << 30));
            if (r < 0) { gzclose(gz); return fail("gzip/bgzf stream is corrupt"); }
            if (r == 0) break;
            got += (size_t)r;
        }
        gzclose(gz); // closes fd
        fd = -1;
        p->owned.resize(got);
        p->text = p->owned.data();
        p->text_len = got;
    } else
        p->text_len = (size_t)sb.st_size;
    if (!compressed && p->text_len > 0) {
        void *m = mmap(nullptr, p->text_len, PROT_READ, MAP_PRIVATE, fd, 0);
        if (m != MAP_FAILED) {
            p->text = (const char *)m;
            p->mapped = true;
            madvise(m, p->text_len, MADV_SEQUENTIAL);
            p->fd = fd;
            fd = -1;
        } else { // pipes / special files: read
            p->owned.resize(p->text_len);
            size_t got = 0;
            while (got < p->text_len) {
                ssize_t r = read(fd, p->owned.data() + got, p->text_len - got);
                if (r <= 0) break;
                got += (size_t)r;
            }
            p->text_len = got;
            p->text = p->owned.data();
        }
    }
    if (fd >= 0) close(fd);
    return true;
}

extern "C" {

swg_paf *swg_paf_parse(const char *path, char *err, size_t err_len) {
    auto fail = [&](const std::string &m) -> swg_paf * {
        if (err && err_len) snprintf(err, err_len, "%s", m.c_str());
        return nullptr;
    };
    swg_paf *p = new swg_paf();
    {
        std::string m;
        if (!swg::paf_open_text(path, p, &m)) { delete p; return fail(m); }
    }
    // chunk at line boundaries, one chunk per host thread
    unsigned nt = std::thread::hardware_concurrency();
    if (nt == 0) nt = 1;
    size_t min_chunk = (size_t)1 << 20;
    size_t nchunks = std::max<size_t>(1, std::min<size_t>(nt, p->text_len / min_chunk));
    std::vector<Chunk> chunks(nchunks);
    size_t start = 0;
    for (size_t k = 0; k < nchunks; k++) {
        size_t target = (k + 1 == nchunks) ? p->text_len : p->text_len / nchunks * (k + 1);
        size_t end = target;
        if (k + 1 < nchunks) {
            const char *nl = (const char *)memchr(p->text + target, '\n', p->text_len - target);
            end = nl ? (size_t)(nl - p->text) + 1 : p->text_len;
        }
        if (end < start) end = start;
        chunks[k].begin = start;
        chunks[k].end = end;
        start = end;
    }
    {
        std::vector<std::thread> th;
        for (size_t k = 1; k < nchunks; k++) th.emplace_back(parse_chunk, p->text, std::ref(chunks[k]));
        parse_chunk(p->text, chunks[0]);
        for (auto &t : th) t.join();
    }
    for (auto &c : chunks)
        if (!c.error.empty()) { std::string m = c.error; delete p; return fail(m); }
    // merge: global name ids in first-appearance order (chunk order, then within-chunk order)
    std::unordered_map<std::string, uint32_t> gid;
    size_t total = 0;
    for (auto &c : chunks) total += c.rank_local.size();
    p->rank.reserve(total); p->line_off.reserve(total); p->line_len.reserve(total);
    p->qid.reserve(total); p->tid.reserve(total); p->qs.reserve(total); p->qe.reserve(total);
    p->ts.reserve(total); p->te.reserve(total); p->blen.reserve(total); p->matches.reserve(total);
    p->identity.reserve(total); p->strand.reserve(total);
    uint64_t line_base = 0;
    for (auto &c : chunks) {
        std::vector<uint32_t> remap(c.names.size());
        // first appearance inside the chunk is by record order with query before target — the local table
        // was filled in exactly that order
        for (size_t i = 0; i < c.names.size(); i++) {
            auto it = gid.find(c.names[i]);
            if (it == gid.end()) {
                uint32_t id = (uint32_t)p->names.size();
                gid.emplace(c.names[i], id);
                p->names.push_back(c.names[i]);
                remap[i] = id;
            } else remap[i] = it->second;
        }
        for (size_t i = 0; i < c.rank_local.size(); i++) {
            p->rank.push_back(line_base + c.rank_local[i]);
            p->qid.push_back(remap[c.qid[i]]);
            p->tid.push_back(remap[c.tid[i]]);
        }
        append(p->line_off, c.line_off); append(p->line_len, c.line_len);
        append(p->qs, c.qs); append(p->qe, c.qe); append(p->ts, c.ts); append(p->te, c.te);
        append(p->blen, c.blen); append(p->matches, c.matches); append(p->identity, c.identity); append(p->strand, c.strand);
        line_base += c.n_lines;
        Chunk().names.swap(c.names);
    }
    p->n_lines = line_base;
    swg::paf_prefix_ids(p->names, &p->P, &p->P2);
    return p;
}

void swg_paf_free(swg_paf *p) { delete p; }
uint64_t swg_paf_n_records(const swg_paf *p) { return p ? p->rank.size() : 0; }
uint64_t swg_paf_n_lines(const swg_paf *p) { return p ? p->n_lines : 0; }
uint32_t swg_paf_n_seq(const swg_paf *p) { return p ? (uint32_t)p->names.size() : 0; }
const uint64_t *swg_paf_rank(const swg_paf *p) { return p ? p->rank.data() : nullptr; }
const char *swg_paf_seq_name(const swg_paf *p, uint32_t id) { return (p && id < p->names.size()) ? p->names[id].c_str() : nullptr; }

int swg_paf_view(const swg_paf *p, swg_mappings *out) {
    if (!p || !out) return SWG_ERR_ARG;
    memset(out, 0, sizeof *out);
    out->n = p->rank.size();
    out->query_id = p->qid.data(); out->target_id = p->tid.data();
    out->query_start = p->qs.data(); out->query_end = p->qe.data();
    out->target_start = p->ts.data(); out->target_end = p->te.data();
    out->block_length = p->blen.data(); out->matches = p->matches.data();
    out->identity = p->identity.data(); out->strand = p->strand.data();
    out->score = nullptr;
    out->n_seq = (uint32_t)p->names.size();
    out->seq_genome_id = p->P.data(); out->seq_genome2_id = p->P2.data();
    return SWG_OK;
}

// append "\tch:Z:chain_<k>" / "\tst:Z:<status>\n" without snprintf
static inline char *put_u32(char *o, uint32_t v) {
    char tmp[10];
    int k = 0;
    do { tmp[k++] = (char)('0' + v % 10); v /= 10; } while (v);
    while (k) *o++ = tmp[--k];
    return o;
}
static void format_range(const swg_paf *p, const uint8_t *status, const uint32_t *chain_id, size_t r0, size_t r1, std::vector<char> &out) {
    static const char *st_name[4] = {"", "scaffold", "rescued", "unassigned"};
    static const size_t st_len[4] = {0, 8, 7, 10};
    size_t need = 0;
    for (size_t r = r0; r < r1; r++)
        if (status[r] != SWG_DROPPED && status[r] <= 3) need += (size_t)p->line_len[r] + 48;
    out.resize(need);
    char *o = out.data();
    for (size_t r = r0; r < r1; r++) { // records are in input order
        const uint8_t s = status[r];
        if (s == SWG_DROPPED || s > 3) continue;
        memcpy(o, p->text + p->line_off[r], p->line_len[r]);
        o += p->line_len[r];
        if (chain_id[r]) {
            memcpy(o, "\tch:Z:chain_", 12);
            o = put_u32(o + 12, chain_id[r]);
        }
        memcpy(o, "\tst:Z:", 6);
        o += 6;
        memcpy(o, st_name[s], st_len[s]);
        o += st_len[s];
        *o++ = '\n';
    }
    out.resize((size_t)(o - out.data()));
}

int swg_paf_write(const swg_paf *p, const char *out_path, const uint8_t *status, const uint32_t *chain_id) {
    if (!p || !out_path || (p->rank.size() && (!status || !chain_id))) return SWG_ERR_ARG;
    const int fd = open(out_path, O_WRONLY | O_CREAT | O_TRUNC, 0644);
    if (fd < 0) return SWG_ERR_IO;
    bool ok = true;
    uint64_t file_off = 0;
    auto write_at = [fd](const std::vector<char> *b, uint64_t off, bool *good) {
        size_t done = 0;
        while (done < b->size()) {
            const ssize_t w = pwrite(fd, b->data() + done, b->size() - done, (off_t)(off + done));
            if (w <= 0) { *good = false; return; }
            done += (size_t)w;
        }
    };
    const size_t n = p->rank.size();
    unsigned nt = std::thread::hardware_concurrency();
    if (nt == 0) nt = 1;
    const size_t window = (size_t)4 << 20; // records formatted per round (bounds the extra memory)
    for (size_t w0 = 0; w0 < n && ok; w0 += window) {
        const size_t w1 = std::min(n, w0 + window);
        const size_t parts = std::max<size_t>(1, std::min<size_t>(nt, (w1 - w0) / 65536 + 1));
        std::vector<std::vector<char>> bufs(parts);
        std::vector<std::thread> th;
        for (size_t k = 0; k < parts; k++) {
            const size_t r0 = w0 + (w1 - w0) * k / parts, r1 = w0 + (w1 - w0) * (k + 1) / parts;
            if (k + 1 < parts) th.emplace_back(format_range, p, status, chain_id, r0, r1, std::ref(bufs[k]));
            else format_range(p, status, chain_id, r0, r1, bufs[k]);
        }
        for (auto &t : th) t.join();
        // every part lands at its own file offset: the page-cache copies run on all threads as well
        th.clear();
        std::vector<char> good(parts, 1);
        for (size_t k = 0; k < parts; k++) {
            if (!bufs[k].empty()) {
                if (k + 1 < parts) th.emplace_back(write_at, &bufs[k], file_off, (bool *)&good[k]);
                else write_at(&bufs[k], file_off, (bool *)&good[k]);
            }
            file_off += bufs[k].size();
        }
        for (auto &t : th) t.join();
        for (char g : good) ok = ok && g;
    }
    ok = (close(fd) == 0) && ok;
    return ok ? SWG_OK : SWG_ERR_IO;
}

int swg_filter_paf_host(swg_ctx *ctx, const swg_config *cfg, const char *in_path, const char *out_path, swg_stats *stats) {
    if (!ctx || !cfg || !in_path || !out_path) return SWG_ERR_ARG;
    char err[256];
    err[0] = 0;
    swg_paf *p = swg_paf_parse(in_path, err, sizeof err);
    if (!p) {
        swg__set_error(ctx, err);
        return access(in_path, R_OK) == 0 && !strstr(err, "not supported") ? SWG_ERR_RANGE : SWG_ERR_IO;
    }
    swg_mappings m;
    swg_paf_view(p, &m);
    std::vector<uint8_t> status(m.n);
    std::vector<uint32_t> chain(m.n);
    swg_result res{status.data(), chain.data()};
    int rc = SWG_OK;
    if (m.n) rc = swg_filter(ctx, cfg, &m, &res, stats);
    else if (stats) memset(stats, 0, sizeof *stats);
    if (rc == SWG_OK) rc = swg_paf_write(p, out_path, status.data(), chain.data());
    swg_paf_free(p);
    return rc;
}

// aln_to_paf's fallback, src/main.rs:743-770: `ALNtoPAF -x -T<threads> <file>`, PAF on its standard output
int swg_aln_to_paf(const char *aln_path, const char *paf_path, int threads) {
    if (!aln_path || !paf_path) return SWG_ERR_ARG;
    const char *exe = getenv("SWG_ALNTOPAF");
    if (!exe || !*exe) exe = "ALNtoPAF";
    {   // is there such an executable?  (execvp's own search, done up front so that "absent" and "failed" stay apart)
        bool found = false;
        if (strchr(exe, '/')) found = access(exe, X_OK) == 0;
        else if (const char *path = getenv("PATH")) {
            std::string p(path);
            size_t a = 0;
            while (!found && a <= p.size()) {
                size_t b = p.find(':', a);
                if (b == std::string::npos) b = p.size();
                const std::string cand = (b > a ? p.substr(a, b - a) : std::string(".")) + "/" + exe;
                found = access(cand.c_str(), X_OK) == 0;
                a = b + 1;
            }
        }
        if (!found) return SWG_ERR_UNSUPPORTED;
    }
    const int fd = open(paf_path, O_WRONLY | O_CREAT | O_TRUNC, 0644);
    if (fd < 0) return SWG_ERR_IO;
    const std::string targ = "-T" + std::to_string(threads > 0 ? threads : 1);
    const pid_t pid = fork();
    if (pid < 0) { close(fd); return SWG_ERR_IO; }
    if (pid == 0) {
        dup2(fd, 1);
        close(fd);
        execlp(exe, exe, "-x", targ.c_str(), aln_path, (char *)nullptr);
        _exit(127);
    }
    close(fd);
    int st = 0;
    while (waitpid(pid, &st, 0) < 0)
        if (errno != EINTR) return SWG_ERR_IO;
    if (!WIFEXITED(st) || WEXITSTATUS(st) != 0) { remove(paf_path); return SWG_ERR_IO; }
    return SWG_OK;
}

int swg_filter_file(swg_ctx *ctx, const swg_config *cfg, const char *in_path, const char *out_path, int keep_self,
                    swg_stats *stats) {
    if (!ctx || !cfg || !in_path || !out_path) return SWG_ERR_ARG;
    // sniff: .1aln files start with "1 " (src/unified_filter.rs:291-306)
    FILE *f = fopen(in_path, "rb");
    if (!f) return SWG_ERR_IO;
    char magic[2] = {0, 0};
    size_t got = fread(magic, 1, 2, f);
    fclose(f);
    if (got == 2 && magic[0] == '1' && magic[1] == ' ') {
        // .1aln in, PAF out: through FastGA's ALNtoPAF (the route of the reference's CLI, src/main.rs:737-770); .1aln out needs
        // the container writer of fastga-rs (src/unified_filter.rs:158-277)
        const size_t ol = strlen(out_path);
        if (ol < 4 || strcmp(out_path + ol - 4, ".paf") != 0) return SWG_ERR_UNSUPPORTED;
        std::string tmp = std::string(out_path) + ".swg-aln.paf";
        int rc = swg_aln_to_paf(in_path, tmp.c_str(), 8);
        if (rc == SWG_OK) {
            swg_config c2 = *cfg;
            c2.keep_self = keep_self ? 1 : 0;
            rc = swg_filter_paf(ctx, &c2, tmp.c_str(), out_path, stats);
        }
        remove(tmp.c_str());
        return rc;
    }
    swg_config c2 = *cfg;
    c2.keep_self = keep_self ? 1 : 0; // .with_keep_self(keep_self), src/unified_filter.rs:340-343
    return swg_filter_paf(ctx, &c2, in_path, out_path, stats);
}

// Size-balanced assignment of genome-pair units to shards (LPT greedy).  A unit must be closed under every grouping
// of the filter: (P(q),P(t)) for the primary sweep and (P2(q),P2(t)) for the scaffold sweep / chain numbering, so
// sequences are first merged into classes that share a P id OR a P2 id (for 3-field PanSN names P == P2).
int swg_shard_plan(const swg_mappings *m, int n_shards, uint32_t *shard_of, uint64_t *shard_sizes) {
    if (!m || n_shards < 1 || (m->n && (!shard_of || !m->query_id || !m->target_id))) return SWG_ERR_ARG; // 32-bit id columns only
    const uint32_t ns = m->n_seq;
    std::vector<uint32_t> cls(ns);
    {
        std::vector<uint32_t> parent(ns);
        for (uint32_t i = 0; i < ns; i++) parent[i] = i;
        auto find = [&](uint32_t x) { while (parent[x] != x) { parent[x] = parent[parent[x]]; x = parent[x]; } return x; };
        std::unordered_map<uint32_t, uint32_t> firstP, firstP2;
        for (uint32_t i = 0; i < ns; i++) {
            auto a = firstP.emplace(m->seq_genome_id[i], i);
            if (!a.second) parent[find(i)] = find(a.first->second);
            auto b = firstP2.emplace(m->seq_genome2_id[i], i);
            if (!b.second) parent[find(i)] = find(b.first->second);
        }
        for (uint32_t i = 0; i < ns; i++) cls[i] = find(i);
    }
    std::unordered_map<uint64_t, uint32_t> unit_id;
    std::vector<uint64_t> unit_size;
    std::vector<uint32_t> unit_of(m->n);
    for (uint64_t i = 0; i < m->n; i++) {
        uint32_t q = m->query_id[i], t = m->target_id[i];
        if (q >= ns || t >= ns) return SWG_ERR_RANGE;
        uint64_t key = ((uint64_t)cls[q] << 32) | cls[t];
        auto it = unit_id.find(key);
        uint32_t u;
        if (it == unit_id.end()) { u = (uint32_t)unit_size.size(); unit_id.emplace(key, u); unit_size.push_back(0); }
        else u = it->second;
        unit_size[u]++;
        unit_of[i] = u;
    }
    std::vector<uint32_t> unit_shard(unit_size.size());
    const int rc = swg_shard_plan_units(unit_size.size(), unit_size.data(), n_shards, unit_shard.data(), shard_sizes);
    if (rc != SWG_OK) return rc;
    for (uint64_t i = 0; i < m->n; i++) shard_of[i] = unit_shard[unit_of[i]];
    return SWG_OK;
}

// LPT: largest unit first (ties by unit index), onto the least loaded shard (ties by the lowest shard)
int swg_shard_plan_units(uint64_t n_units, const uint64_t *unit_sizes, int n_shards, uint32_t *shard_of_unit, uint64_t *shard_sizes) {
    if (n_shards < 1 || (n_units && (!unit_sizes || !shard_of_unit))) return SWG_ERR_ARG;
    std::vector<uint32_t> order(n_units);
    for (uint32_t u = 0; u < order.size(); u++) order[u] = u;
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return unit_sizes[a] > unit_sizes[b]; });
    std::vector<uint64_t> load(n_shards, 0);
    for (uint32_t u : order) {
        int best = 0;
        for (int s = 1; s < n_shards; s++) if (load[s] < load[best]) best = s;
        shard_of_unit[u] = (uint32_t)best;
        load[best] += unit_sizes[u];
    }
    if (shard_sizes) for (int s = 0; s < n_shards; s++) shard_sizes[s] = load[s];
    return SWG_OK;
}

} // extern "C"
