// formats.cc — host-side readers/writers for the reference's step-boundary files (no GPU work here).
//
//   .fastb / .qualp : "feudal" files (feudal/FeudalControlBlock.h:156-163, feudal/FeudalFileWriter.cc:24-38,84-95):
//                     24-byte control block {u32 n, u8 flags(nFiles=1), u8 sizeofFixed, u8 sizeofX, u8 sizeofA,
//                     u64 varTableOffset, u64 fixedOffset}; variable data; (n+1) u64 ABSOLUTE file offsets; fixed data.
//   .small_K.hbv    : "BINWRITE" (feudal/BinaryStream.h:34-48) + HyperBasevector::writeBinary
//                     (paths/HyperBasevector.cc:121-125): i32 K, then digraphE::writeBinary (graph/DigraphTemplate.h:2226-2231):
//                     from_, from_edge_obj_, to_edge_obj_ (vec<vec<int>>: u64 n, each u64 m + m x i32), edges_ (u64 n, each
//                     bvec: u32 size + ceil(size/4) bytes, feudal/FieldVec.h:595-597).  to_ is rebuilt on read.
//   .small_K.paths  : paths/long/ReadPath.cc:6-20: u64 n; per read i32 offset, u16 len, len x i32.
//   small_K.freqs   : "i, count" lines for i = 1..100 (paths/long/BuildReadQGraph.cc:1108-1112).
//   .small_K.gfa    : GFA 1.0 of the graph with per-edge k-mer coverage (include/w2rap_coverage.h).
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/w2rap_coverage.h"

namespace {

int fail(int code, char* err, size_t errlen, const char* fmt, const char* a) {
    if (err && errlen) snprintf(err, errlen, fmt, a);
    return code;
}

struct File {
    FILE* f;
    explicit File(const char* path, const char* mode) : f(fopen(path, mode)) {}
    ~File() { if (f) fclose(f); }
    bool put(const void* p, size_t n) { return n == 0 || fwrite(p, 1, n, f) == n; }
    template <class T> bool put(const T& v) { return put(&v, sizeof(T)); }
};

struct FeudalHeader {
    uint32_t n;
    uint8_t flags, sz_fixed, sz_x, sz_a;
    uint64_t var_tab_off, fixed_off;
};
static_assert(sizeof(FeudalHeader) == 24, "feudal control block is 24 bytes");

int write_feudal(const char* path, const uint8_t* var, uint64_t var_len, const uint64_t* off, uint64_t n, const void* fixed, uint64_t fixed_len,
                 uint8_t sz_fixed, uint8_t sz_x, char* err, size_t errlen) {
    File f(path, "wb");
    if (!f.f) return fail(W2RAP_ERR_IO, err, errlen, "cannot create %s", path);
    FeudalHeader h{(uint32_t)n, 1, sz_fixed, sz_x, 1, 24 + var_len, 24 + var_len + 8 * (n + 1)};
    bool ok = f.put(h) && f.put(var, var_len);
    std::vector<uint64_t> abs(n + 1);
    for (uint64_t i = 0; i <= n; ++i) abs[i] = (n ? off[i] : 0) + 24;
    ok = ok && f.put(abs.data(), 8 * (n + 1)) && f.put(fixed, fixed_len);
    if (!ok) return fail(W2RAP_ERR_IO, err, errlen, "short write to %s", path);
    return W2RAP_OK;
}

// Reads a feudal file; returns var data, offsets relative to the var data, fixed data.
int read_feudal(const char* path, std::vector<uint8_t>* var, std::vector<uint64_t>* off, std::vector<uint8_t>* fixed, FeudalHeader* hdr, char* err, size_t errlen) {
    File f(path, "rb");
    if (!f.f) return fail(W2RAP_ERR_IO, err, errlen, "cannot open %s", path);
    fseek(f.f, 0, SEEK_END);
    uint64_t flen = (uint64_t)ftell(f.f);
    fseek(f.f, 0, SEEK_SET);
    FeudalHeader h;
    if (flen < 24 || fread(&h, 1, 24, f.f) != 24) return fail(W2RAP_ERR_IO, err, errlen, "%s is not a feudal file", path);
    if ((h.flags & 3) != 1 || h.var_tab_off < 24 || h.fixed_off < h.var_tab_off + 8 || h.fixed_off > flen || (h.fixed_off - h.var_tab_off) % 8)
        return fail(W2RAP_ERR_IO, err, errlen, "%s: bad feudal control block", path);
    uint64_t n = (h.fixed_off - h.var_tab_off) / 8 - 1;
    var->resize(h.var_tab_off - 24);
    off->resize(n + 1);
    fixed->resize(flen - h.fixed_off);
    if ((var->size() && fread(var->data(), 1, var->size(), f.f) != var->size()) || fread(off->data(), 8, n + 1, f.f) != n + 1 ||
        (fixed->size() && fread(fixed->data(), 1, fixed->size(), f.f) != fixed->size()))
        return fail(W2RAP_ERR_IO, err, errlen, "short read from %s", path);
    for (uint64_t i = 0; i <= n; ++i) {
        if ((*off)[i] < 24 || (*off)[i] > h.var_tab_off || (i && (*off)[i] < (*off)[i - 1])) return fail(W2RAP_ERR_IO, err, errlen, "%s: bad offset table", path);
        (*off)[i] -= 24;
    }
    *hdr = h;
    return W2RAP_OK;
}

}  // namespace

extern "C" {

int w2rap_write_fastb(const char* path, const w2rap_reads* r, char* err, size_t errlen) {
    if (!path || !r) return fail(W2RAP_ERR_BAD_ARG, err, errlen, "%s", "null argument");
    uint64_t n = r->n_reads;
    return write_feudal(path, r->bases, n ? r->base_off[n] : 0, r->base_off, n, r->len, 4 * n, 4, 16, err, errlen);
}
int w2rap_write_qualp(const char* path, const w2rap_reads* r, char* err, size_t errlen) {
    if (!path || !r) return fail(W2RAP_ERR_BAD_ARG, err, errlen, "%s", "null argument");
    uint64_t n = r->n_reads;
    return write_feudal(path, r->quals, n ? r->qual_off[n] : 0, r->qual_off, n, nullptr, 0, 0, 8, err, errlen);
}

int w2rap_read_fastb_qualp(const char* fastb, const char* qualp, w2rap_reads* out, char* err, size_t errlen) {
    if (!fastb || !qualp || !out) return fail(W2RAP_ERR_BAD_ARG, err, errlen, "%s", "null argument");
    std::vector<uint8_t> bv, bf, qv, qf;
    std::vector<uint64_t> bo, qo;
    FeudalHeader bh, qh;
    int rc = read_feudal(fastb, &bv, &bo, &bf, &bh, err, errlen);
    if (rc) return rc;
    rc = read_feudal(qualp, &qv, &qo, &qf, &qh, err, errlen);
    if (rc) return rc;
    uint64_t n = bo.size() - 1;
    if (qo.size() - 1 != n) return fail(W2RAP_ERR_IO, err, errlen, "%s: read count differs from the .fastb", qualp);
    if (bf.size() != 4 * n) return fail(W2RAP_ERR_IO, err, errlen, "%s: fixed section is not one u32 length per read", fastb);
    memset(out, 0, sizeof(*out));
    out->n_reads = n;
    uint8_t* bases = (uint8_t*)malloc(bv.size() + 32);
    uint8_t* quals = (uint8_t*)malloc(qv.size() + 32);
    uint64_t* boff = (uint64_t*)malloc(8 * (n + 1));
    uint64_t* qoff = (uint64_t*)malloc(8 * (n + 1));
    uint32_t* len = (uint32_t*)malloc(4 * (n + 1));
    if (!bases || !quals || !boff || !qoff || !len) { free(bases); free(quals); free(boff); free(qoff); free(len); return fail(W2RAP_ERR_OOM, err, errlen, "%s", "out of host memory"); }
    memcpy(bases, bv.data(), bv.size()); memset(bases + bv.size(), 0, 32);
    memcpy(quals, qv.data(), qv.size()); memset(quals + qv.size(), 0, 32);
    memcpy(boff, bo.data(), 8 * (n + 1)); memcpy(qoff, qo.data(), 8 * (n + 1)); memcpy(len, bf.data(), 4 * n);
    out->bases = bases; out->quals = quals; out->base_off = boff; out->qual_off = qoff; out->len = len;
    return W2RAP_OK;
}

int w2rap_write_freqs(const char* path, const w2rap_graph* g, char* err, size_t errlen) {
    if (!path || !g) return fail(W2RAP_ERR_BAD_ARG, err, errlen, "%s", "null argument");
    File f(path, "w");
    if (!f.f) return fail(W2RAP_ERR_IO, err, errlen, "cannot create %s", path);
    for (int i = 1; i < 101; ++i) fprintf(f.f, "%d, %llu\n", i, (unsigned long long)g->hist[i]);
    return W2RAP_OK;
}

int w2rap_write_paths(const char* path, const w2rap_graph* g, char* err, size_t errlen) {
    if (!path || !g) return fail(W2RAP_ERR_BAD_ARG, err, errlen, "%s", "null argument");
    File f(path, "wb");
    if (!f.f) return fail(W2RAP_ERR_IO, err, errlen, "cannot create %s", path);
    uint64_t n = g->n_paths;
    std::vector<uint8_t> buf;
    buf.reserve(1 << 20);
    bool ok = f.put(n);
    for (uint64_t r = 0; r < n && ok; ++r) {
        int32_t off = g->path_offset[r];
        uint64_t m = g->path_off[r + 1] - g->path_off[r];
        uint16_t ps = (uint16_t)m;                       // the reference truncates the size to u16 (ReadPath.cc:14)
        const uint8_t* p = (const uint8_t*)&off; buf.insert(buf.end(), p, p + 4);
        p = (const uint8_t*)&ps; buf.insert(buf.end(), p, p + 2);
        p = (const uint8_t*)(g->path_edges + g->path_off[r]); buf.insert(buf.end(), p, p + 4 * (size_t)ps);
        if (buf.size() > (1u << 20)) { ok = f.put(buf.data(), buf.size()); buf.clear(); }
    }
    ok = ok && f.put(buf.data(), buf.size());
    if (!ok) return fail(W2RAP_ERR_IO, err, errlen, "short write to %s", path);
    return W2RAP_OK;
}

int w2rap_write_hbv(const char* path, const w2rap_graph* g, char* err, size_t errlen) {
    if (!path || !g) return fail(W2RAP_ERR_BAD_ARG, err, errlen, "%s", "null argument");
    File f(path, "wb");
    if (!f.f) return fail(W2RAP_ERR_IO, err, errlen, "cannot create %s", path);
    const uint64_t E = g->n_edges, nv = g->n_vertices, nh = g->n_hbv_edges;
    // per hbv edge: endpoints and (canonical edge, rc)
    std::vector<int32_t> left(nh), right(nh);
    std::vector<uint64_t> canon(nh);
    std::vector<uint8_t> isrc(nh);
    for (uint64_t e = 0; e < E; ++e) {
        int32_t fw = g->fwd_xlat[e], rv = g->rev_xlat[e];
        left[fw] = g->edge_vertices[4 * e]; right[fw] = g->edge_vertices[4 * e + 1]; canon[fw] = e; isrc[fw] = 0;
        if (rv != fw) { left[rv] = g->edge_vertices[4 * e + 2]; right[rv] = g->edge_vertices[4 * e + 3]; canon[rv] = e; isrc[rv] = 1; }
    }
    // AddEdge in id order with upper_bound insertion (graph/DigraphTemplate.h:1829-1839) == lists sorted by (neighbour, id)
    struct Adj { int32_t own, nb, e; };
    auto build = [&](bool from, std::vector<std::vector<int32_t>>* nbs, std::vector<std::vector<int32_t>>* objs) {
        std::vector<Adj> a(nh);
        for (uint64_t e = 0; e < nh; ++e) a[e] = from ? Adj{left[e], right[e], (int32_t)e} : Adj{right[e], left[e], (int32_t)e};
        std::sort(a.begin(), a.end(), [](const Adj& x, const Adj& y) { return x.own != y.own ? x.own < y.own : (x.nb != y.nb ? x.nb < y.nb : x.e < y.e); });
        nbs->assign(nv, {}); objs->assign(nv, {});
        for (const Adj& x : a) { (*nbs)[x.own].push_back(x.nb); (*objs)[x.own].push_back(x.e); }
    };
    std::vector<std::vector<int32_t>> from_v, from_e, to_v, to_e;
    build(true, &from_v, &from_e);
    build(false, &to_v, &to_e);
    bool ok = f.put("BINWRITE", 8);
    int32_t Kv = W2RAP_K;
    ok = ok && f.put(Kv);
    auto put_vv = [&](const std::vector<std::vector<int32_t>>& vv) {
        uint64_t n = vv.size();
        bool k = f.put(n);
        for (const auto& v : vv) { uint64_t m = v.size(); k = k && f.put(m) && f.put(v.data(), 4 * m); }
        return k;
    };
    ok = ok && put_vv(from_v) && put_vv(from_e) && put_vv(to_e);
    ok = ok && f.put(nh);
    std::vector<uint8_t> rc;
    for (uint64_t he = 0; he < nh && ok; ++he) {
        uint64_t e = canon[he];
        uint32_t len = g->edge_len[e];
        const uint8_t* p = g->edge_bases + g->edge_off[e];
        uint64_t nb = ((uint64_t)len + 3) / 4;
        ok = ok && f.put(len);
        if (!isrc[he]) ok = ok && f.put(p, nb);
        else {
            rc.assign(nb, 0);
            for (uint32_t i = 0; i < len; ++i) {
                uint32_t src = len - 1 - i;
                uint32_t b = 3u - ((p[src >> 2] >> ((src & 3) * 2)) & 3u);
                rc[i >> 2] |= (uint8_t)(b << ((i & 3) * 2));
            }
            ok = ok && f.put(rc.data(), nb);
        }
    }
    if (!ok) return fail(W2RAP_ERR_IO, err, errlen, "short write to %s", path);
    return W2RAP_OK;
}

// include/w2rap_coverage.h: segments are canonical edges named by their fwd hbv id; links are pairs of hbv edges meeting at a vertex,
// each written once for itself and its complement.
int w2rap_write_gfa(const char* path, const w2rap_graph* g, const w2rap_seq_cov* edge_cov, char* err, size_t errlen) {
    if (!path || !g) return fail(W2RAP_ERR_BAD_ARG, err, errlen, "%s", "null argument");
    const uint64_t E = g->n_edges, nv = g->n_vertices, nh = g->n_hbv_edges;
    if (E && (!g->edge_vertices || !g->fwd_xlat || !g->involution))
        return fail(W2RAP_ERR_BAD_ARG, err, errlen, "%s", "graph without edge_vertices, fwd_xlat or involution (a non-root result of a graph_on_root_only run?)");
    if (E && (!g->edge_off || !g->edge_len || !g->edge_bases)) return fail(W2RAP_ERR_BAD_ARG, err, errlen, "%s", "graph without edge sequences");
    // per hbv edge: its segment (fwd id of its canonical edge), orientation and endpoints
    std::vector<int32_t> seg(nh, -1), left(nh), right(nh);
    std::vector<uint8_t> minus(nh, 0);
    for (uint64_t e = 0; e < E; ++e) {
        const int32_t fw = g->fwd_xlat[e];
        if (fw < 0 || (uint64_t)fw >= nh || g->involution[fw] < 0 || (uint64_t)g->involution[fw] >= nh)
            return fail(W2RAP_ERR_BAD_ARG, err, errlen, "%s", "hbv edge id out of range");
        const int32_t rv = g->involution[fw];
        seg[fw] = fw; left[fw] = g->edge_vertices[4 * e]; right[fw] = g->edge_vertices[4 * e + 1];
        if (rv != fw) { seg[rv] = fw; minus[rv] = 1; left[rv] = g->edge_vertices[4 * e + 2]; right[rv] = g->edge_vertices[4 * e + 3]; }
    }
    for (uint64_t x = 0; x < nh; ++x)
        if (seg[x] < 0 || left[x] < 0 || (uint64_t)left[x] >= nv || right[x] < 0 || (uint64_t)right[x] >= nv)
            return fail(W2RAP_ERR_BAD_ARG, err, errlen, "%s", "hbv edges and vertices are inconsistent");
    File f(path, "w");
    if (!f.f) return fail(W2RAP_ERR_IO, err, errlen, "cannot create %s", path);
    bool ok = fputs("H\tVN:Z:1.0\n", f.f) >= 0;
    std::string line;
    for (uint64_t e = 0; e < E && ok; ++e) {
        const uint32_t len = g->edge_len[e];
        const uint8_t* p = g->edge_bases + g->edge_off[e];
        line.assign("S\t");
        line += std::to_string(g->fwd_xlat[e]);
        line += '\t';
        for (uint32_t i = 0; i < len; ++i) line += "ACGT"[(p[i >> 2] >> ((i & 3) * 2)) & 3u];
        line += "\tLN:i:" + std::to_string(len);
        if (edge_cov) {
            char dp[64];
            line += "\tKC:i:" + std::to_string(edge_cov[e].sum);
            if (edge_cov[e].n_kmers) { snprintf(dp, sizeof dp, "\tDP:f:%.3f", (double)edge_cov[e].sum / (double)edge_cov[e].n_kmers); line += dp; }
        }
        line += '\n';
        ok = f.put(line.data(), line.size());
    }
    // in-edges and out-edges of every vertex, in hbv id order
    std::vector<uint64_t> in_off(nv + 1, 0), out_off(nv + 1, 0);
    for (uint64_t x = 0; x < nh; ++x) { ++in_off[right[x] + 1]; ++out_off[left[x] + 1]; }
    for (uint64_t v = 0; v < nv; ++v) { in_off[v + 1] += in_off[v]; out_off[v + 1] += out_off[v]; }
    std::vector<int32_t> ins(nh), outs(nh);
    {
        std::vector<uint64_t> ci(in_off.begin(), in_off.end() - 1), co(out_off.begin(), out_off.end() - 1);
        for (uint64_t x = 0; x < nh; ++x) { ins[ci[right[x]]++] = (int32_t)x; outs[co[left[x]]++] = (int32_t)x; }
    }
    const int32_t* inv = g->involution;
    for (uint64_t v = 0; v < nv && ok; ++v)
        for (uint64_t a = in_off[v]; a < in_off[v + 1] && ok; ++a)
            for (uint64_t b = out_off[v]; b < out_off[v + 1] && ok; ++b) {
                const int32_t x = ins[a], y = outs[b];
                if (std::make_pair(inv[y], inv[x]) < std::make_pair(x, y)) continue;      // its complement is the one written
                ok = fprintf(f.f, "L\t%d\t%c\t%d\t%c\t%dM\n", seg[x], minus[x] ? '-' : '+', seg[y], minus[y] ? '-' : '+', W2RAP_K - 1) > 0;
            }
    if (!ok) return fail(W2RAP_ERR_IO, err, errlen, "short write to %s", path);
    return W2RAP_OK;
}

void w2rap_step2_free_host_reads(w2rap_reads* r);

int w2rap_step2_run_files(const char* dir, const char* prefix, const w2rap_params* p, w2rap_graph* out_or_null, char* err, size_t errlen) {
    if (!dir || !prefix || !p) return fail(W2RAP_ERR_BAD_ARG, err, errlen, "%s", "null argument");
    std::string d(dir);
    w2rap_reads r;
    int rc = w2rap_read_fastb_qualp((d + "/frag_reads_orig.fastb").c_str(), (d + "/frag_reads_orig.qualp").c_str(), &r, err, errlen);
    if (rc) return rc;
    w2rap_params q = *p;
    q.want_paths = 1; q.apply_fixpaths = 1;       // the files hold post-FixPaths paths (w2rap-contigger.cc:340-346)
    if (!q.workdir || !q.workdir[0]) q.workdir = dir;
    w2rap_graph g;
    rc = w2rap_step2_run(&r, &q, &g, err, errlen);
    if (rc == W2RAP_OK) rc = w2rap_write_hbv((d + "/" + prefix + ".small_K.hbv").c_str(), &g, err, errlen);
    if (rc == W2RAP_OK) rc = w2rap_write_paths((d + "/" + prefix + ".small_K.paths").c_str(), &g, err, errlen);
    // w2rap_reads from w2rap_read_fastb_qualp are malloc'ed
    free((void*)r.bases); free((void*)r.quals); free((void*)r.base_off); free((void*)r.qual_off); free((void*)r.len);
    if (rc == W2RAP_OK && out_or_null) *out_or_null = g; else if (rc == W2RAP_OK) w2rap_step2_free(&g);
    return rc;
}

}  // extern "C"
