// tc_pack.h — host-side packing of the map tables (shared by tc_api.cu and the CPU-only test build tc_hosttest.cpp).
#pragma once
#include <algorithm>
#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include "tc_core.cuh"

struct TcPacked {
    TcBlobLayout L{};
    std::vector<unsigned char> blob; // tables of the tracking kernel, sections 16-byte aligned
    std::vector<int32_t> adj;        // per class: [out_off(n+1) | out_edge(m) | in_off(n+1) | in_edge(m)]
    std::vector<size_t> adj_base;    // start of each class inside adj
    int max_nodes = 0;
    std::vector<TcClassBlob> cblob_desc;  // per class
    std::vector<unsigned char> cblob;     // all class blobs, each 16-byte aligned
    int max_cblob_bytes = 0;
};

static inline int32_t tc_align16(int32_t x) { return (x + 15) & ~15; }

// Validates the descriptor and builds the blob + adjacency. Returns "" on success, else the error message.
static inline std::string tc_pack_map(const TcMapDesc *map, TcPacked &pk) {
    const int C = map->n_classes;
    if (C <= 0 || C > TC_MAX_CLASSES) return "n_classes out of range (1..16)";
    const int P = map->lp_n_nodes, Q = map->lp_n_edges;
    if (P <= 0 || Q <= 0) return "empty lanepath";
    const int sumN = map->ll_node_off[C], sumE = map->ll_edge_off[C];
    for (int e = 0; e < Q; e++)
        for (int j = 0; j < 2; j++)
            if (map->lp_edges[2 * e + j] < 0 || map->lp_edges[2 * e + j] >= P) return "lanepath edge out of range";
    for (int c = 0; c < C; c++) {
        int n = map->ll_node_off[c + 1] - map->ll_node_off[c];
        pk.max_nodes = std::max(pk.max_nodes, n);
        for (int e = map->ll_edge_off[c]; e < map->ll_edge_off[c + 1]; e++)
            for (int j = 0; j < 2; j++)
                if (map->ll_edges[2 * e + j] < 0 || map->ll_edges[2 * e + j] >= n) return "laneline edge out of range";
    }
    // lanepath CSR in edge-list order (layer.py:183-185 scan the edge list front to back)
    std::vector<int32_t> next_off(P + 1, 0), prev_off(P + 1, 0), next_edge(Q), prev_edge(Q);
    for (int e = 0; e < Q; e++) { next_off[map->lp_edges[2 * e] + 1]++; prev_off[map->lp_edges[2 * e + 1] + 1]++; }
    for (int i = 0; i < P; i++) { next_off[i + 1] += next_off[i]; prev_off[i + 1] += prev_off[i]; }
    {
        std::vector<int32_t> nc(next_off.begin(), next_off.end() - 1), pc(prev_off.begin(), prev_off.end() - 1);
        for (int e = 0; e < Q; e++) { next_edge[nc[map->lp_edges[2 * e]]++] = e; prev_edge[pc[map->lp_edges[2 * e + 1]]++] = e; }
    }
    TcBlobLayout &L = pk.L;
    L.n_classes = C; L.lp_n_nodes = P; L.lp_n_edges = Q; L.sum_nodes = sumN; L.sum_edges = sumE;
    int32_t off = 0;
    auto place = [&](int32_t bytes) { int32_t o = off; off = tc_align16(off + bytes); return o; };
    L.off_lp_nodes = place(P * 16); L.off_lp_orient = place(Q * 8); L.off_lp_orient_rev = place(Q * 8); L.off_ll_nodes = place(sumN * 16);
    L.off_lp_edges = place(Q * 8); L.off_next_off = place((P + 1) * 4); L.off_next_edge = place(Q * 4); L.off_prev_off = place((P + 1) * 4);
    L.off_prev_edge = place(Q * 4); L.off_ll_edges = place(sumE * 8); L.off_ll_node_off = place((C + 1) * 4); L.off_ll_edge_off = place((C + 1) * 4);
    L.off_ll_nodes32 = place(sumN * 8);
    L.total_bytes = off;
    pk.blob.assign(off, 0);
    unsigned char *b = pk.blob.data();
    memcpy(b + L.off_lp_nodes, map->lp_nodes, (size_t)P * 16);
    memcpy(b + L.off_lp_orient, map->lp_orient, (size_t)Q * 8);
    memcpy(b + L.off_lp_orient_rev, map->lp_orient_rev, (size_t)Q * 8);
    memcpy(b + L.off_ll_nodes, map->ll_nodes, (size_t)sumN * 16);
    memcpy(b + L.off_lp_edges, map->lp_edges, (size_t)Q * 8);
    memcpy(b + L.off_next_off, next_off.data(), (size_t)(P + 1) * 4);
    memcpy(b + L.off_next_edge, next_edge.data(), (size_t)Q * 4);
    memcpy(b + L.off_prev_off, prev_off.data(), (size_t)(P + 1) * 4);
    memcpy(b + L.off_prev_edge, prev_edge.data(), (size_t)Q * 4);
    memcpy(b + L.off_ll_edges, map->ll_edges, (size_t)sumE * 8);
    memcpy(b + L.off_ll_node_off, map->ll_node_off, (size_t)(C + 1) * 4);
    memcpy(b + L.off_ll_edge_off, map->ll_edge_off, (size_t)(C + 1) * 4);
    {
        // float copy of the laneline nodes + the margin of the float pre-filter: float rounding of a coordinate of
        // magnitude X is <= X*2^-24, the whole d0+d1 estimate stays within ~16 ulp(X) ~ X*1e-6; margin = 1e-4*max(1,X)
        float *f32 = (float *)(b + L.off_ll_nodes32);
        double ext = 1.0;
        for (int i = 0; i < 2 * sumN; i++) { f32[i] = (float)map->ll_nodes[i]; ext = std::max(ext, std::fabs(map->ll_nodes[i])); }
        for (int i = 0; i < 2 * P; i++) ext = std::max(ext, std::fabs(map->lp_nodes[i]));
        L.scan_margin = 1e-4 * (4.0 * ext);   // car positions may leave the map: allow 4x the map extent
        L.scan_limit = 4.0 * ext;             // beyond it the tracking kernel scans in plain float64 (tc_get_info)
    }
    // laneline node adjacency per class, in edge order (the clip passes apply a node's edges in list order)
    pk.adj_base.resize(C);
    for (int c = 0; c < C; c++) {
        int n = map->ll_node_off[c + 1] - map->ll_node_off[c], m = map->ll_edge_off[c + 1] - map->ll_edge_off[c];
        const int32_t *ed = map->ll_edges + 2 * (size_t)map->ll_edge_off[c];
        std::vector<int32_t> oo(n + 1, 0), io(n + 1, 0), oe(m), ie(m);
        for (int e = 0; e < m; e++) { oo[ed[2 * e] + 1]++; io[ed[2 * e + 1] + 1]++; }
        for (int i = 0; i < n; i++) { oo[i + 1] += oo[i]; io[i + 1] += io[i]; }
        std::vector<int32_t> oc(oo.begin(), oo.end() - 1), ic(io.begin(), io.end() - 1);
        for (int e = 0; e < m; e++) { oe[oc[ed[2 * e]]++] = e; ie[ic[ed[2 * e + 1]]++] = e; }
        {
            TcClassBlob d;
            d.n_nodes = n; d.n_edges = m;
            int32_t o = 0;
            auto sec = [&](int32_t bytes) { int32_t at = o; o = tc_align16(o + bytes); return at; };
            sec(n * 16);
            d.off_edges = sec(m * 8); d.off_out_off = sec((n + 1) * 4); d.off_out_edge = sec(m * 4);
            d.off_in_off = sec((n + 1) * 4); d.off_in_edge = sec(m * 4);
            d.bytes = o;
            d.offset = (int32_t)pk.cblob.size();
            pk.cblob.resize(pk.cblob.size() + (size_t)o, 0);
            unsigned char *cb = pk.cblob.data() + d.offset;
            memcpy(cb, map->ll_nodes + 2 * (size_t)map->ll_node_off[c], (size_t)n * 16);
            memcpy(cb + d.off_edges, ed, (size_t)m * 8);
            memcpy(cb + d.off_out_off, oo.data(), (size_t)(n + 1) * 4);
            memcpy(cb + d.off_out_edge, oe.data(), (size_t)m * 4);
            memcpy(cb + d.off_in_off, io.data(), (size_t)(n + 1) * 4);
            memcpy(cb + d.off_in_edge, ie.data(), (size_t)m * 4);
            pk.cblob_desc.push_back(d);
            pk.max_cblob_bytes = std::max(pk.max_cblob_bytes, (int)o);
        }
        pk.adj_base[c] = pk.adj.size();
        pk.adj.insert(pk.adj.end(), oo.begin(), oo.end());
        pk.adj.insert(pk.adj.end(), oe.begin(), oe.end());
        pk.adj.insert(pk.adj.end(), io.begin(), io.end());
        pk.adj.insert(pk.adj.end(), ie.begin(), ie.end());
    }
    return "";
}

// Class-table views over a blob copy at `blob_base` and an adjacency copy at `adj_base_ptr` (host or device addresses).
static inline void tc_class_views(const TcMapDesc *map, const TcPacked &pk, const unsigned char *blob_base, const int32_t *adj_ptr,
                                  std::vector<TcClassTables> &cls) {
    const int C = map->n_classes;
    cls.resize(C);
    for (int c = 0; c < C; c++) {
        int n = map->ll_node_off[c + 1] - map->ll_node_off[c], m = map->ll_edge_off[c + 1] - map->ll_edge_off[c];
        cls[c].n_nodes = n; cls[c].n_edges = m;
        cls[c].nodes = (const double *)(blob_base + pk.L.off_ll_nodes) + 2 * (size_t)map->ll_node_off[c];
        cls[c].edges = (const int32_t *)(blob_base + pk.L.off_ll_edges) + 2 * (size_t)map->ll_edge_off[c];
        const int32_t *b = adj_ptr + pk.adj_base[c];
        cls[c].out_off = b; cls[c].out_edge = b + (n + 1); cls[c].in_off = b + (n + 1) + m; cls[c].in_edge = b + 2 * (n + 1) + m;
    }
}
