// Host-side collate for callers whose data set lives in HOST memory (the reference's case): replaces
// `collate_fn` -> `dgl.batch` + `torch.stack` (GCN:292-297) and the DataLoader's pin_memory copy (GCN:567).
// One call gathers a batch of molecules from a packed host table straight into ONE caller-owned (pinned)
// buffer, in the layout eims_batch_build reads after a single H2D copy:
//     [node_ptr i64 | bond_ptr i64 | bond_begin i32 | bond_end i32 | feat f32 | targets f32  or  peak_ptr i64 | mz | intensity f32]
// every section 256-byte aligned.  Pure memcpy work (~2.5 MB for 512 molecules with dense targets): the
// reference does the same job in DGL's C++ `dgl.batch` inside DataLoader worker processes.  No device code here.
#include <cstring>

#include "common.cuh"

namespace {
inline int64_t align256(int64_t v) { return (v + 255) & ~(int64_t)255; }
}  // namespace

#pragma GCC visibility push(default)
// cap_nodes / cap_bonds / cap_peaks > 0: FIXED layout - the sections are sized for those capacities, so their offsets
// are the same for every batch of n molecules (what a captured CUDA graph needs: constant device pointers)
static int pack_impl(const eims_dataset* ds, const int32_t* ids, int32_t n, int32_t node_feat_dim, int32_t max_mz, void* out,
                     int64_t capacity, eims_host_batch* lay, int64_t cap_nodes, int64_t cap_bonds, int64_t cap_peaks) {
  if (!ds || !ds->node_ptr || !ds->bond_ptr || !ds->feat || !lay || n < 0 || node_feat_dim < 1) return EIMS_ERR_ARG;
  const bool dense = ds->targets != nullptr;
  const eims_peaks* pk = dense ? nullptr : ds->peaks;
  if (pk && !(pk->peak_ptr && pk->mz && pk->intensity)) return EIMS_ERR_ARG;
  int64_t atoms = 0, bonds = 0, peaks = 0;
  for (int32_t g = 0; g < n; ++g) {
    const int64_t id = ids ? ids[g] : g;
    if (id < 0 || id >= ds->num_mols) return EIMS_ERR_ARG;
    atoms += ds->node_ptr[id + 1] - ds->node_ptr[id];
    bonds += ds->bond_ptr[id + 1] - ds->bond_ptr[id];
    if (pk) peaks += pk->peak_ptr[id + 1] - pk->peak_ptr[id];
  }
  const int64_t mzsz = pk ? (pk->mz_is_f64 ? 8 : 4) : 0;
  const bool fixed = cap_nodes > 0;
  const int64_t sz_atoms = fixed ? cap_nodes : atoms, sz_peaks = fixed ? cap_peaks : peaks;
  const int64_t sz_bonds = fixed ? (cap_bonds > 0 ? cap_bonds : 1) : bonds;
  eims_host_batch L{};
  int64_t off = 0;
  L.node_ptr = off; off = align256(off + 8 * (int64_t)(n + 1));
  L.bond_ptr = off; off = align256(off + 8 * (int64_t)(n + 1));
  L.bond_begin = off; off = align256(off + 4 * sz_bonds);
  L.bond_end = off; off = align256(off + 4 * sz_bonds);
  L.feat = off; off = align256(off + 4 * sz_atoms * node_feat_dim);
  L.targets = L.peak_ptr = L.peak_mz = L.peak_inten = -1;
  if (dense) { L.targets = off; off = align256(off + 4 * (int64_t)n * max_mz); }
  else if (pk) {
    L.peak_ptr = off; off = align256(off + 8 * (int64_t)(n + 1));
    L.peak_mz = off; off = align256(off + mzsz * (sz_peaks > 0 ? sz_peaks : 1));
    L.peak_inten = off; off = align256(off + 4 * (sz_peaks > 0 ? sz_peaks : 1));
  }
  L.nbytes = off;
  L.num_graphs = n; L.num_nodes = (int32_t)atoms; L.num_edges = (int32_t)(2 * bonds); L.feat_dim = node_feat_dim;
  L.mz_is_f64 = pk ? pk->mz_is_f64 : 0;
  *lay = L;
  // the fixed layout comes back whatever the batch holds: a layout query (out == NULL) may name any molecules
  if (fixed && (atoms > cap_nodes || bonds > cap_bonds || (pk && peaks > cap_peaks))) return EIMS_ERR_CAPACITY;
  if (off > capacity || (n > 0 && !out)) return EIMS_ERR_CAPACITY;  // out == NULL: layout query
  char* base = reinterpret_cast<char*>(out);
  int64_t* np_ = reinterpret_cast<int64_t*>(base + L.node_ptr);
  int64_t* bp_ = reinterpret_cast<int64_t*>(base + L.bond_ptr);
  int64_t* pp_ = pk ? reinterpret_cast<int64_t*>(base + L.peak_ptr) : nullptr;
  int64_t a = 0, b = 0, q = 0;
  for (int32_t g = 0; g < n; ++g) {
    const int64_t id = ids ? ids[g] : g;
    const int64_t a0 = ds->node_ptr[id], na = ds->node_ptr[id + 1] - a0;
    const int64_t b0 = ds->bond_ptr[id], nb = ds->bond_ptr[id + 1] - b0;
    np_[g] = a; bp_[g] = b;
    memcpy(base + L.feat + 4 * a * node_feat_dim, ds->feat + a0 * node_feat_dim, (size_t)(4 * na * node_feat_dim));
    if (nb) {
      memcpy(base + L.bond_begin + 4 * b, ds->bond_begin + b0, (size_t)(4 * nb));
      memcpy(base + L.bond_end + 4 * b, ds->bond_end + b0, (size_t)(4 * nb));
    }
    if (dense) memcpy(base + L.targets + 4 * (int64_t)g * max_mz, ds->targets + id * (int64_t)max_mz, (size_t)(4 * (int64_t)max_mz));
    if (pk) {
      const int64_t k0 = pk->peak_ptr[id], nk = pk->peak_ptr[id + 1] - k0;
      pp_[g] = q;
      if (nk) {
        memcpy(base + L.peak_mz + mzsz * q, reinterpret_cast<const char*>(pk->mz) + mzsz * k0, (size_t)(mzsz * nk));
        memcpy(base + L.peak_inten + 4 * q, pk->intensity + k0, (size_t)(4 * nk));
      }
      q += nk;
    }
    a += na; b += nb;
  }
  np_[n] = a; bp_[n] = b;
  if (pp_) pp_[n] = q;
  return 0;
}

extern "C" int eims_host_pack_batch(const eims_dataset* ds, const int32_t* ids, int32_t n, int32_t node_feat_dim,
                                    int32_t max_mz, void* out, int64_t capacity, eims_host_batch* lay) {
  return pack_impl(ds, ids, n, node_feat_dim, max_mz, out, capacity, lay, 0, 0, 0);
}

extern "C" int eims_host_pack_batch_fixed(const eims_dataset* ds, const int32_t* ids, int32_t n, int32_t node_feat_dim,
                                          int32_t max_mz, int64_t cap_nodes, int64_t cap_bonds, int64_t cap_peaks, void* out,
                                          int64_t capacity, eims_host_batch* lay) {
  if (cap_nodes < 1 || cap_bonds < 0 || cap_peaks < 0) return EIMS_ERR_ARG;
  return pack_impl(ds, ids, n, node_feat_dim, max_mz, out, capacity, lay, cap_nodes, cap_bonds, cap_peaks);
}
#pragma GCC visibility pop
