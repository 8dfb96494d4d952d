// tc_route.h — the route table of the navigation goals (include/tinycarlo_b200.h TcRouteDesc), built on the host by
// tc_set_route and by the CPU-only test build (ht_route_table). Host code only.
#pragma once
#include <functional>
#include <queue>
#include <utility>
#include <vector>

#include "tc_core.cuh"

// the maneuvers a route may use, in the order that breaks ties (the smallest m attaining the minimum)
static const int TC_ROUTE_MANEUVERS[3] = {0, 1, 3};

// T(e, m) for every lanepath edge, slots j = 0, 1, 2 for m = 0, 1, 3: the edge tc_find_local_path_given moves on to (-1: none).
// tc_pick_edge itself decides, quirks included (self-loops filtered from the orientation list, the unfiltered list indexed).
static inline std::vector<int32_t> tc_route_transitions(const TcTrackTables &t) {
    const int Q = t.lp_n_edges;
    std::vector<int32_t> tr((size_t)3 * Q, -1);
    for (int e = 0; e < Q; e++) {
        const int n1 = t.lp_edges[2 * e + 1];
        for (int j = 0; j < 3; j++) {
            const double dir = tc_clip_angle(t.lp_orient[e] + TC_ROUTE_MANEUVERS[j] * TC_PI / 2);
            const int p = tc_pick_edge(t, n1, dir, t.next_edge, t.next_off[n1], t.next_off[n1 + 1], true);
            tr[(size_t)3 * e + j] = p < 0 ? -1 : t.next_edge[p];
        }
    }
    return tr;
}

// D [G][Q] and cmd [G][Q] for goals[0..G-1] (node ids in range): Dijkstra backwards from each goal over the reversed transitions.
// An edge is settled when popped with its final D; relaxing its predecessors with the rounded L(f) + D(f) then gives every edge
// the minimum over its transitions, and cmd is the first m in TC_ROUTE_MANEUVERS whose sum equals it.
static inline void tc_build_route(const TcTrackTables &t, const int32_t *goals, int G, double *D, int8_t *cmd) {
    const int Q = t.lp_n_edges;
    const std::vector<int32_t> tr = tc_route_transitions(t);
    std::vector<double> L(Q);
    for (int e = 0; e < Q; e++) {
        const int a = t.lp_edges[2 * e], b = t.lp_edges[2 * e + 1];
        L[e] = tc_dist(t.lp_nodes[2 * a], t.lp_nodes[2 * a + 1], t.lp_nodes[2 * b], t.lp_nodes[2 * b + 1]);
    }
    std::vector<int32_t> pred_off(Q + 1, 0), pred;   // CSR: the edges e with T(e, m) = f for some m
    for (size_t i = 0; i < tr.size(); i++)
        if (tr[i] >= 0) pred_off[tr[i] + 1]++;
    for (int f = 0; f < Q; f++) pred_off[f + 1] += pred_off[f];
    pred.resize(pred_off[Q]);
    {
        std::vector<int32_t> fill(pred_off.begin(), pred_off.end() - 1);
        for (size_t i = 0; i < tr.size(); i++)
            if (tr[i] >= 0) pred[fill[tr[i]]++] = (int32_t)(i / 3);
    }
    typedef std::pair<double, int> Item;
    for (int k = 0; k < G; k++) {
        double *Dk = D + (size_t)k * Q;
        int8_t *ck = cmd + (size_t)k * Q;
        std::priority_queue<Item, std::vector<Item>, std::greater<Item>> pq;
        for (int e = 0; e < Q; e++) {
            Dk[e] = INFINITY;
            if (t.lp_edges[2 * e + 1] == goals[k]) {
                Dk[e] = 0.0;
                pq.push(Item(0.0, e));
            }
        }
        while (!pq.empty()) {
            const Item it = pq.top();
            pq.pop();
            const int f = it.second;
            if (it.first != Dk[f]) continue;   // a stale entry
            const double via = L[f] + Dk[f];
            for (int p = pred_off[f]; p < pred_off[f + 1]; p++) {
                const int e = pred[p];
                if (via < Dk[e]) {
                    Dk[e] = via;
                    pq.push(Item(via, e));
                }
            }
        }
        for (int e = 0; e < Q; e++) {
            ck[e] = -1;
            if (Dk[e] == 0.0 || !(Dk[e] < INFINITY)) continue;
            for (int j = 0; j < 3; j++) {
                const int f = tr[(size_t)3 * e + j];
                if (f >= 0 && L[f] + Dk[f] == Dk[e]) {
                    ck[e] = (int8_t)TC_ROUTE_MANEUVERS[j];
                    break;
                }
            }
        }
    }
}
