// Host-side flattening of an rbd_model_desc into the device model (see rbd_types.h).  Plain C++.
#pragma once
#include <stdint.h>

#include <string>
#include <vector>

#include "../../../include/rbd_b200.h"
#include "rbd_types.h"

namespace rbd {

struct HostModel {
  int nb = 0, nq = 0, nv = 0;
  int64_t modcount = 0;
  int nslots = 0;            // pending slots (max nesting of branch nodes)
  bool general = false;      // multi-DoF joint somewhere other than preorder position 0 under the world
  bool other_kinds = false;  // prismatic or fixed joints: the generic kernels need those code paths (else revolute-only)
  std::vector<int> order;    // preorder position -> reference joint index
  std::vector<int> pos;      // reference joint index -> preorder position
  std::vector<int> qstart, vstart;   // reference order
  std::vector<double> alignT;        // preorder position -> A^T (9), canonical body frame <- caller's body frame
  double total_mass = 0;
  ModelDev<double> dev64;    // ABA row layout (row0 / nrows); RNEA and CRBA derive theirs from slot indices
  ModelDev<float> dev32;
};

// The device model in the kernels' scalar type.
template <class T> const ModelDev<T>& dev_model(const HostModel& m);
template <> inline const ModelDev<float>& dev_model<float>(const HostModel& m) { return m.dev32; }
template <> inline const ModelDev<double>& dev_model<double>(const HostModel& m) { return m.dev64; }

// Returns RBD_OK or an rbd_status; `err` gets a human-readable message.
int build_host_model(const rbd_model_desc* desc, HostModel& out, std::string& err);

// Stash rows per sample for the three kernels.
inline int aba_rows(const HostModel& m) { return m.dev64.nrows; }
inline int rnea_rows(const HostModel& m) { return m.nb * 6 + m.nslots * kSlotRowsRnea; }
inline int crba_rows(const HostModel& m) { return m.nb * 2 + m.nslots * kSlotRowsCrba; }
inline int kin_rows(const HostModel& m) { return m.nslots * 24; }

}  // namespace rbd
