// Test-only C shim around eraytracer_b200/csrc/scene_tables.cpp: the checks and the packer of the scene's element
// tables, run the way ert_scene_create (flatten) and ert_scene_update (update_stage) run them, without CUDA.
#include <algorithm>
#include <string>
#include <vector>

#include "../../eraytracer_b200/csrc/scene_tables.h"

using namespace ert;

namespace {
std::string g_msg;
}

extern "C" {

int st_n_tables() { return T_COUNT; }
const char *st_table(int t, int *kind, int *per, unsigned *changed)
{
    *kind = kTables[t].kind;
    *per = kTables[t].per;
    *changed = kTables[t].changed;
    return kTables[t].name;
}

// The create path: check_create, then the packer into tables sized from the list positions.  On success the tables
// (in TableId order) go to tab and the list positions (in ElemKind order) to order.  Returns the message, "" if none.
const char *st_create(const ert_scene_desc *d, double *tab, int *order)
{
    SourceOrder src;
    std::vector<int> ord[K_COUNT];
    g_msg = check_create(d, src, ord);
    if (!g_msg.empty()) return g_msg.c_str();
    std::vector<double> t[T_COUNT];
    double *tp[T_COUNT];
    for (int k = 0; k < T_COUNT; k++) {
        t[k].resize(ord[kTables[k].kind].size() * kTables[k].per);
        tp[k] = t[k].data();
    }
    g_msg = pack_tables(*d, src, tp);
    if (!g_msg.empty()) return g_msg.c_str();
    for (int k = 0; k < T_COUNT; k++) tab = std::copy(t[k].begin(), t[k].end(), tab);
    for (int k = 0; k < K_COUNT; k++) order = std::copy(ord[k].begin(), ord[k].end(), order);
    return g_msg.c_str();
}

// The update path of a scene whose kind k has the n[k] list positions that follow in order: check_update, then the
// packer straight into staging (the tables back to back in TableId order, as in the update's staging buffer).
const char *st_update(const ert_scene_desc *d, const int *order, const long long n[K_COUNT], double *staging)
{
    std::vector<int> ord[K_COUNT];
    for (int k = 0; k < K_COUNT; k++) {
        ord[k].assign(order, order + n[k]);
        order += n[k];
    }
    SourceOrder src;
    g_msg = check_update(d, ord, src);
    if (!g_msg.empty()) return g_msg.c_str();
    double *tp[T_COUNT];
    for (int k = 0; k < T_COUNT; k++) {
        tp[k] = staging;
        staging += n[kTables[k].kind] * kTables[k].per;
    }
    g_msg = pack_tables(*d, src, tp);
    return g_msg.c_str();
}
}
