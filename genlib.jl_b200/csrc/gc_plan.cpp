// gc_plan.cpp -- the schedule of gen.gc (gc_plan.hpp, DESIGN.md 2b).  O(N + edges), host only.
#include "gc_plan.hpp"

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <queue>

#include "../../include/genlib_cuda.h"
#include "plan.hpp"

namespace genlib {

int build_gc_plan(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro, const int32_t *proband,
                  int32_t n_anc, const int32_t *ancestor, int direction, GcPlan &P, std::string &err,
                  const int32_t *pro_group, int32_t n_pro_groups, const int32_t *anc_group, int32_t n_anc_groups) {
    P = GcPlan();
    if (n < 0 || n_pro < 0 || n_anc < 0 || n_pro_groups < 0 || n_anc_groups < 0 || (n > 0 && (!father || !mother)) ||
        (n_pro > 0 && !proband) || (n_anc > 0 && !ancestor)) {
        err = "genlib_gc: null pointer or negative size";
        return GENLIB_EINVAL;
    }
    P.n = n; P.n_pro = n_pro; P.n_anc = n_anc;
    if (int rc = check_pedigree(n, father, mother, err)) return rc;   // the pedigree's own errors first
    // list position -> unique index, numbered by first occurrence; rank -> unique index (-1: not listed)
    std::vector<int32_t> pro_of((size_t)n, -1), anc_of((size_t)n, -1);
    auto unique = [&](int32_t len, const int32_t *list, const char *what, std::vector<int32_t> &of,
                      std::vector<int32_t> &uid, int32_t &n_u) {
        uid.resize((size_t)len);
        for (int32_t k = 0; k < len; k++) {
            const int32_t x = list[k];
            if (x < 0 || x >= n) { err = std::string("KeyError: ") + what + " index " + std::to_string(x) + " not in pedigree"; return GENLIB_EKEY; }
            if (of[(size_t)x] < 0) of[(size_t)x] = n_u++;
            uid[(size_t)k] = of[(size_t)x];
        }
        return GENLIB_OK;
    };
    if (int rc = unique(n_pro, proband, "proband", pro_of, P.pro_uid, P.n_pro_u)) return rc;
    if (int rc = unique(n_anc, ancestor, "ancestor", anc_of, P.anc_uid, P.n_anc_u)) return rc;
    // a grouped side: distinct ranks (so its unique index is its list position), every group named
    auto check_groups = [&](int32_t len, const int32_t *list, const int32_t *group, int32_t n_groups, const char *what,
                            const std::vector<int32_t> &uid) {
        std::vector<int32_t> members((size_t)n_groups, 0);
        for (int32_t k = 0; k < len; k++) {
            if (uid[(size_t)k] != k) { err = std::string("genlib_gc_groups: duplicate ") + what + " rank " + std::to_string(list[k]); return GENLIB_EINVAL; }
            if (group[k] < 0 || group[k] >= n_groups) {
                err = "genlib_gc_groups: group index " + std::to_string(group[k]) + " of " + what + " position " +
                      std::to_string(k) + " is not in [0, " + std::to_string(n_groups) + ")";
                return GENLIB_EINVAL;
            }
            members[(size_t)group[k]]++;
        }
        for (int32_t g = 0; g < n_groups; g++)
            if (!members[(size_t)g]) { err = "genlib_gc_groups: " + std::string(what) + " group " + std::to_string(g) + " has no member"; return GENLIB_EINVAL; }
        return GENLIB_OK;
    };
    P.pro_grouped = pro_group != nullptr; P.anc_grouped = anc_group != nullptr;
    if (P.pro_grouped) if (int rc = check_groups(n_pro, proband, pro_group, n_pro_groups, "proband", P.pro_uid)) return rc;
    if (P.anc_grouped) if (int rc = check_groups(n_anc, ancestor, anc_group, n_anc_groups, "ancestor", P.anc_uid)) return rc;
    if (direction < 0) {
        const int32_t w_pro = P.pro_grouped ? n_pro_groups : P.n_pro_u, w_anc = P.anc_grouped ? n_anc_groups : P.n_anc_u;
        direction = w_pro < w_anc ? kGcAscend : kGcDescend;
        if (const char *env = std::getenv("GENLIB_GC_DIRECTION")) {      // test / benchmark knob
            if (!std::strcmp(env, "descend")) direction = kGcDescend;
            else if (!std::strcmp(env, "ascend")) direction = kGcAscend;
        }
    }
    if (direction != kGcDescend && direction != kGcAscend) { err = "genlib_gc: unknown direction"; return GENLIB_EINVAL; }
    P.direction = direction;
    // a grouped side's output positions are its groups: as the column side every member seeds its group's
    // column, as the target side every member keeps its own output-block row and the groups list those rows
    auto regroup = [&](bool is_column, int32_t len, const int32_t *list, const int32_t *group, int32_t n_groups,
                       std::vector<int32_t> &of, std::vector<int32_t> &uid, int32_t &n_u, int32_t &n_out) {
        if (is_column) {
            for (int32_t k = 0; k < len; k++) of[(size_t)list[k]] = group[k];
            n_u = n_groups;
        } else {
            P.grp_ptr.assign((size_t)n_groups + 1, 0);
            for (int32_t k = 0; k < len; k++) P.grp_ptr[(size_t)group[k] + 1]++;
            for (int32_t g = 0; g < n_groups; g++) P.grp_ptr[(size_t)g + 1] += P.grp_ptr[(size_t)g];
            P.grp_row.resize((size_t)len);
            std::vector<int64_t> at(P.grp_ptr.begin(), P.grp_ptr.end() - 1);
            for (int32_t k = 0; k < len; k++) P.grp_row[(size_t)at[(size_t)group[k]]++] = k;
        }
        uid.resize((size_t)n_groups);
        for (int32_t g = 0; g < n_groups; g++) uid[(size_t)g] = g;
        n_out = n_groups;
    };
    if (P.pro_grouped) regroup(direction == kGcAscend, n_pro, proband, pro_group, n_pro_groups, pro_of, P.pro_uid, P.n_pro_u, P.n_pro);
    if (P.anc_grouped) regroup(direction == kGcDescend, n_anc, ancestor, anc_group, n_anc_groups, anc_of, P.anc_uid, P.n_anc_u, P.n_anc);
    P.layer_begin.assign(1, 0);
    if (P.n_pro_u == 0 || P.n_anc_u == 0) return GENLIB_OK;

    // prune: descendants-or-self of a listed ancestor (forward sweep) that are ancestors-or-self of a
    // listed proband (reverse sweep; children have larger ranks, so a rank is final when it is visited)
    std::vector<uint8_t> active((size_t)n, 0);
    for (int32_t i = 0; i < n; i++) {
        const int32_t f = father[i], m = mother[i];
        active[(size_t)i] = anc_of[(size_t)i] >= 0 || (f >= 0 && active[(size_t)f]) || (m >= 0 && active[(size_t)m]);
    }
    {
        std::vector<uint8_t> up((size_t)n, 0);
        for (int32_t i = n - 1; i >= 0; i--) {
            if (pro_of[(size_t)i] >= 0) up[(size_t)i] = 1;
            if (!up[(size_t)i]) { active[(size_t)i] = 0; continue; }
            if (father[i] >= 0) up[(size_t)father[i]] = 1;
            if (mother[i] >= 0) up[(size_t)mother[i]] = 1;
        }
    }
    const bool desc = direction == kGcDescend;
    const std::vector<int32_t> &seed_of = desc ? anc_of : pro_of, &out_of = desc ? pro_of : anc_of;
    // in-edges in topological order (ranks ascending when descending, descending when ascending)
    std::vector<int64_t> child_ptr;
    std::vector<int32_t> child;
    if (!desc) {                                             // active children of every rank, in rank order
        child_ptr.assign((size_t)n + 1, 0);
        for (int32_t c = 0; c < n; c++) {
            if (!active[(size_t)c]) continue;
            if (father[c] >= 0 && active[(size_t)father[c]]) child_ptr[(size_t)father[c] + 1]++;
            if (mother[c] >= 0 && active[(size_t)mother[c]]) child_ptr[(size_t)mother[c] + 1]++;
        }
        for (int32_t i = 0; i < n; i++) child_ptr[(size_t)i + 1] += child_ptr[(size_t)i];
        child.resize((size_t)child_ptr[(size_t)n]);
        std::vector<int64_t> at(child_ptr.begin(), child_ptr.end() - 1);
        for (int32_t c = 0; c < n; c++) {
            if (!active[(size_t)c]) continue;
            if (father[c] >= 0 && active[(size_t)father[c]]) child[(size_t)at[(size_t)father[c]]++] = c;
            if (mother[c] >= 0 && active[(size_t)mother[c]]) child[(size_t)at[(size_t)mother[c]]++] = c;
        }
    }
    auto for_inputs = [&](int32_t i, auto &&fn) {
        if (desc) {
            if (father[i] >= 0 && active[(size_t)father[i]]) fn(father[i]);
            if (mother[i] >= 0 && active[(size_t)mother[i]]) fn(mother[i]);
        } else {
            for (int64_t e = child_ptr[(size_t)i]; e < child_ptr[(size_t)i + 1]; e++) fn(child[(size_t)e]);
        }
    };
    std::vector<int32_t> order;                              // active ranks in topological order
    for (int32_t k = 0; k < n; k++) {
        const int32_t i = desc ? k : n - 1 - k;
        if (active[(size_t)i]) order.push_back(i);
    }
    // layer = longest path from a row without active inputs; last_read = layer of the last reader (-1: none)
    std::vector<int32_t> layer((size_t)n, -1), last_read((size_t)n, -1);
    int32_t n_layers = 0;
    for (int32_t i : order) {
        int32_t t = 0;
        for_inputs(i, [&](int32_t s) { t = std::max(t, layer[(size_t)s] + 1); });
        layer[(size_t)i] = t;
        for_inputs(i, [&](int32_t s) { last_read[(size_t)s] = std::max(last_read[(size_t)s], t); });
        n_layers = std::max(n_layers, t + 1);
    }
    // rows grouped by layer, topological order kept inside a layer
    P.layer_begin.assign((size_t)n_layers + 1, 0);
    for (int32_t i : order) P.layer_begin[(size_t)layer[(size_t)i] + 1]++;
    for (int32_t t = 0; t < n_layers; t++) P.layer_begin[(size_t)t + 1] += P.layer_begin[(size_t)t];
    const size_t R = order.size();
    P.row_ind.resize(R);
    {
        std::vector<int64_t> at(P.layer_begin.begin(), P.layer_begin.end() - 1);
        for (int32_t i : order) P.row_ind[(size_t)at[(size_t)layer[(size_t)i]]++] = i;
    }
    // frontier slots: a row read later takes the lowest free slot; it is free again from the layer after its
    // last reader's (readers of layer t only read rows of earlier layers)
    P.row_slot.resize(R); P.row_seed.resize(R); P.row_out.resize(R); P.in_ptr.assign(R + 1, 0);
    std::vector<int32_t> slot_of((size_t)n, -1);
    std::priority_queue<int32_t, std::vector<int32_t>, std::greater<int32_t>> free_slots;
    std::vector<std::vector<int32_t>> freed_after((size_t)n_layers);
    int64_t cap = 0;
    for (int32_t t = 0; t < n_layers; t++) {
        if (t > 0) for (int32_t s : freed_after[(size_t)t - 1]) free_slots.push(s);
        for (int64_t r = P.layer_begin[(size_t)t]; r < P.layer_begin[(size_t)t + 1]; r++) {
            const int32_t i = P.row_ind[(size_t)r];
            int32_t slot = -1;
            if (last_read[(size_t)i] >= 0) {
                if (free_slots.empty()) slot = (int32_t)cap++;
                else { slot = free_slots.top(); free_slots.pop(); }
                freed_after[(size_t)last_read[(size_t)i]].push_back(slot);
                P.n_slotted++;
            }
            slot_of[(size_t)i] = slot;
            P.row_slot[(size_t)r] = slot;
            P.row_seed[(size_t)r] = seed_of[(size_t)i];
            P.row_out[(size_t)r] = out_of[(size_t)i];
            if (out_of[(size_t)i] >= 0) P.n_out_rows++;
            for_inputs(i, [&](int32_t s) { P.in_slot.push_back(slot_of[(size_t)s]); });
            P.in_ptr[(size_t)r + 1] = (int64_t)P.in_slot.size();
        }
    }
    P.capacity = cap;
    return GENLIB_OK;
}

}  // namespace genlib
