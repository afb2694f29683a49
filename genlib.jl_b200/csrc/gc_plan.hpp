// gc_plan.hpp -- host schedule of gen.gc (genetic contributions, SURVEY.md 2: src/compute.jl:518-595).
//
// G[p, a] = [p == a] + 1/2 G[father(p), a] + 1/2 G[mother(p), a] is propagated over the pruned pedigree
// (descendants-or-self of a listed ancestor AND ancestors-or-self of a listed proband) in one of two
// directions; both are the same computation on a DAG given as in-edges:
//     row = seed + 1/2 * (((0 + in_1) + in_2) + ...)
//   descend: columns = unique ancestors, a row's inputs are its active father, then its active mother
//   ascend:  columns = unique probands,  a row's inputs are its active children in ascending rank
//            (H[i, p] = [i == p] + 1/2 sum_children H[c, p] = G[p, i])
// Rows go in layers (layer = longest path from a row without active inputs); a row that is read later
// lives in a frontier slot from its layer to the layer of its last reader; a target row (a proband when
// descending, an ancestor when ascending) is also written to the output block.  See DESIGN.md 2b.
//
// gen.gcGroups (DESIGN.md 2i): a grouped side lists distinct ranks, each with a group in [0, n_groups).  G is
// linear, so a grouped column side propagates one column per group: every member is seeded in its group's
// column.  A grouped target side keeps one output-block row per member; grp_ptr / grp_row list each group's
// rows in list order, and the device sums them into a block of one row per group before the gather.  The
// grouped side's output positions are its groups: n_pro / n_anc count them and pro_uid / anc_uid are the
// identity (output position -> column, or row of the summed block).
#pragma once
#include <cstdint>
#include <string>
#include <vector>

namespace genlib {

constexpr int kGcDescend = 0, kGcAscend = 1;

struct GcPlan {
    int32_t n = 0, n_pro = 0, n_anc = 0;          // output positions: list lengths (duplicates kept) or groups
    int32_t direction = kGcDescend;
    std::vector<int32_t> pro_uid, anc_uid;         // list position -> unique index (first occurrence order)
    int32_t n_pro_u = 0, n_anc_u = 0;              // columns or output-block rows of each side
    bool pro_grouped = false, anc_grouped = false;
    std::vector<int64_t> grp_ptr;                  // grouped target side: group g's output-block rows are
    std::vector<int32_t> grp_row;                  //   grp_row[grp_ptr[g] .. grp_ptr[g + 1]), in list order
    int64_t capacity = 0;                          // peak live frontier rows
    // rows of every layer, layer after layer (layer t: rows [layer_begin[t], layer_begin[t + 1]))
    std::vector<int64_t> layer_begin;
    std::vector<int32_t> row_ind, row_slot, row_seed, row_out;
    std::vector<int64_t> in_ptr;                   // rows + 1 entries, global offsets into in_slot
    std::vector<int32_t> in_slot;
    int64_t n_slotted = 0, n_out_rows = 0;         // rows written to the frontier / to the output block

    int32_t n_layers() const { return (int32_t)layer_begin.size() - 1; }
    int64_t rows() const { return (int64_t)row_ind.size(); }
    int64_t inputs() const { return (int64_t)in_slot.size(); }
    // columns propagated and targets written (the output block has n_targets() rows)
    int32_t width() const { return direction == kGcDescend ? n_anc_u : n_pro_u; }
    int32_t n_targets() const { return direction == kGcDescend ? n_pro_u : n_anc_u; }
    // the target side's list (rows of the output block) and the column side's list
    const std::vector<int32_t> &target_uid() const { return direction == kGcDescend ? pro_uid : anc_uid; }
    const std::vector<int32_t> &column_uid() const { return direction == kGcDescend ? anc_uid : pro_uid; }
    // the target side is grouped: its output-block rows are summed per group before the gather
    bool target_grouped() const { return direction == kGcDescend ? pro_grouped : anc_grouped; }
    int32_t n_target_groups() const { return (int32_t)grp_ptr.size() - 1; }
    // required traffic over `w` columns: inputs read + frontier rows written + output rows written, binary64
    double alg_bytes(int64_t w) const {
        return (double)(inputs() + n_slotted + n_out_rows) * (double)w * 8.0;
    }
};

// Validates like genlib_plan_create (GENLIB_EKEY / GENLIB_EORDER with the first offending rank; a broken
// pedigree is reported before a bad list entry).  direction: kGcDescend, kGcAscend, or -1 = the narrower
// side, descend on ties (environment GENLIB_GC_DIRECTION=descend|ascend overrides -1).
// pro_group / anc_group (gen.gcGroups): null = that side is a plain list; otherwise the side's ranks must be
// distinct and every group in [0, n_groups) non-empty (GENLIB_EINVAL).  The narrower side counts its groups
// when grouped, its unique entries otherwise.
int build_gc_plan(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro, const int32_t *proband,
                  int32_t n_anc, const int32_t *ancestor, int direction, GcPlan &P, std::string &err,
                  const int32_t *pro_group = nullptr, int32_t n_pro_groups = 0, const int32_t *anc_group = nullptr,
                  int32_t n_anc_groups = 0);

}  // namespace genlib
