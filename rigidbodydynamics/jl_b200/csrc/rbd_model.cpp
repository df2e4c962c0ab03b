// Flatten-once preprocessing: rbd_model_desc (reference joint order, reference frames) -> device model.
//
// Three things happen here, all on the host, all once per Mechanism:
//
//  1. Frame canonicalisation.  Every joint type of the reference has a CONSTANT motion subspace in the frame
//     after the joint (has_fixed_subspaces = true, e.g. src/joint_types/revolute.jl:44, planar.jl:54).  For
//     the 1-DoF types (Revolute, Prismatic, SinCosRevolute) the body frame is re-oriented by a constant
//     rotation A_i with A_i e_z = axis, so that on the device the subspace is the ONE-HOT column e_z
//     (angular z for revolute, linear z for prismatic): U = I^A S is a column read, D a diagonal entry, and
//     the joint rotation is Rz(q).  Scalars q, v, v̇, tau of a 1-DoF joint are invariant under this change of
//     frame, so the q/v/tau layout of the reference is untouched.  Planar joints are re-oriented so that
//     (x_axis, y_axis, rot_axis) = (e_x, e_y, e_z); their velocity coordinates are coefficients of those
//     axes (planar.jl:72-77) and are invariant too.  Floating / spherical joints keep their frame (their
//     velocity IS expressed in it).   X_tree' = A_parent^T X_tree A_i,  I' = A_i^T I A_i.
//
//  2. Depth-first preorder.  The reference's tree order is only topological (mechanism_modification.jl:139);
//     preorder makes every subtree contiguous so the inward pass can hand a child's articulated inertia to
//     its parent in registers, with one "pending slot" per simultaneously-open branch node.
//
//  3. Stash-row allocation for the shared-memory working set of the ABA kernel.
#include "rbd_model.h"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>

namespace rbd {
namespace {

struct Mat3 { double m[9]; };

Mat3 ident() { Mat3 r{}; r.m[0] = r.m[4] = r.m[8] = 1.0; return r; }
Mat3 mul(const Mat3& a, const Mat3& b) {
  Mat3 r{};
  for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) {
    double s = 0;
    for (int k = 0; k < 3; ++k) s += a.m[3 * i + k] * b.m[3 * k + j];
    r.m[3 * i + j] = s;
  }
  return r;
}
Mat3 transp(const Mat3& a) { Mat3 r{}; for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) r.m[3 * i + j] = a.m[3 * j + i]; return r; }
void mulv(const Mat3& a, const double* v, double* o) {
  for (int i = 0; i < 3; ++i) o[i] = a.m[3 * i] * v[0] + a.m[3 * i + 1] * v[1] + a.m[3 * i + 2] * v[2];
}
void cross(const double* a, const double* b, double* o) {
  o[0] = a[1] * b[2] - a[2] * b[1]; o[1] = a[2] * b[0] - a[0] * b[2]; o[2] = a[0] * b[1] - a[1] * b[0];
}
double norm3(const double* a) { return std::sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]); }

// Rotation A with A e_z = axis (unit).  Axis-aligned inputs give signed permutation matrices exactly.
Mat3 align_z_to(const double* axis) {
  double z[3] = {axis[0], axis[1], axis[2]};
  double n = norm3(z);
  for (double& c : z) c /= n;
  // pick the coordinate axis least aligned with z as a helper to build an orthonormal triad
  int k = 0;
  if (std::fabs(z[1]) < std::fabs(z[k])) k = 1;
  if (std::fabs(z[2]) < std::fabs(z[k])) k = 2;
  double e[3] = {0, 0, 0};
  e[k] = 1.0;
  double d = e[0] * z[0] + e[1] * z[1] + e[2] * z[2];
  double x[3] = {e[0] - d * z[0], e[1] - d * z[1], e[2] - d * z[2]};
  double nx = norm3(x);
  for (double& c : x) c /= nx;
  double y[3];
  cross(z, x, y);
  Mat3 A{};
  for (int i = 0; i < 3; ++i) { A.m[3 * i + 0] = x[i]; A.m[3 * i + 1] = y[i]; A.m[3 * i + 2] = z[i]; }
  return A;
}

template <class T> void fill_dev(const HostModel& hm, const ModelDev<double>& src, ModelDev<T>& dst) {
  std::memset(&dst, 0, sizeof(dst));
  dst.nb = src.nb; dst.nq = src.nq; dst.nv = src.nv; dst.nrows = src.nrows;
  dst.slot_base = src.slot_base; dst.nslots = src.nslots;
  for (int k = 0; k < 3; ++k) dst.g[k] = (T)src.g[k];
  for (int i = 0; i < src.nb; ++i) {
    const BodyDev<double>& s = src.body[i];
    BodyDev<T>& d = dst.body[i];
    for (int k = 0; k < 9; ++k) d.Rt[k] = (T)s.Rt[k];
    for (int k = 0; k < 3; ++k) { d.pt[k] = (T)s.pt[k]; d.h[k] = (T)s.h[k]; }
    for (int k = 0; k < 6; ++k) d.J[k] = (T)s.J[k];
    d.m = (T)s.m;
    d.qoff = (T)s.qoff;
    d.kind = s.kind; d.parent = s.parent; d.qrow = s.qrow; d.vrow = s.vrow; d.row0 = s.row0;
    d.oslot = s.oslot; d.pslot = s.pslot; d.flags = s.flags; d.refidx = s.refidx;
  }
  (void)hm;
}

}  // namespace

int build_host_model(const rbd_model_desc* desc, HostModel& out, std::string& err) {
  if (!desc || !desc->parent || !desc->jtype || !desc->X_tree || !desc->jparam || !desc->inertia) {
    err = "rbd_model_create: NULL pointer in model description";
    return RBD_EINVAL;
  }
  if (desc->num_non_tree_joints > 0) {
    err = "This method can currently only handle tree Mechanisms.";   // mechanism_algorithms.jl:549
    return RBD_ELOOP;
  }
  const int nb = desc->nb;
  if (nb < 1) { err = "rbd_model_create: mechanism has no joints"; return RBD_EINVAL; }
  if (nb > kMaxBodies) { err = "rbd_model_create: more than RBD_MAX_BODIES bodies"; return RBD_EUNSUPPORTED; }
  for (int i = 0; i < nb; ++i) {
    if (desc->parent[i] < -1 || desc->parent[i] >= i) { err = "rbd_model_create: parent[] is not a topologically ordered tree"; return RBD_EINVAL; }
    if (desc->jtype[i] < 0 || desc->jtype[i] > 7) { err = "rbd_model_create: unknown joint type"; return RBD_EINVAL; }
  }
  out = HostModel();
  out.nb = nb;
  out.modcount = desc->modcount;
  out.qstart.resize(nb); out.vstart.resize(nb);
  int nq = 0, nv = 0;
  for (int i = 0; i < nb; ++i) {
    out.qstart[i] = nq; out.vstart[i] = nv;
    nq += kind_nq(desc->jtype[i]); nv += kind_nv(desc->jtype[i]);
  }
  out.nq = nq; out.nv = nv;

  // ---- 1. alignment rotations A_i (reference order) -------------------------------------------------------
  std::vector<Mat3> A(nb);
  for (int i = 0; i < nb; ++i) {
    const double* jp = desc->jparam + 9 * i;
    switch (desc->jtype[i]) {
      case K_REV: case K_PRIS: case K_SINCOS: {
        if (norm3(jp) < 1e-12) { err = "rbd_model_create: zero joint axis"; return RBD_EINVAL; }
        A[i] = align_z_to(jp);
        break;
      }
      case K_PLANAR: {
        Mat3 a{};
        for (int r = 0; r < 3; ++r) { a.m[3 * r + 0] = jp[r]; a.m[3 * r + 1] = jp[3 + r]; a.m[3 * r + 2] = jp[6 + r]; }
        A[i] = a;
        break;
      }
      default: A[i] = ident();
    }
  }

  // ---- 2. depth-first preorder ---------------------------------------------------------------------------
  std::vector<std::vector<int>> children(nb);
  std::vector<int> roots;
  for (int i = 0; i < nb; ++i) (desc->parent[i] < 0 ? roots : children[desc->parent[i]]).push_back(i);
  // Ordering heuristic: sibling subtrees that are pure revolute chains of equal length (the legs / arms of a humanoid) are
  // placed first and adjacent (L then R).  (It once fed a lock-step walk of such pairs, measured slower and removed; the order
  // is kept because the slot colouring below and every measurement in DESIGN.md were made with it.)
  struct PairRec { int L, R, len; };
  std::vector<PairRec> pairs;
  {
    std::vector<int> chain_len(nb, 0);
    for (int i = nb - 1; i >= 0; --i) {
      const bool rev = desc->jtype[i] == K_REV || desc->jtype[i] == K_SINCOS;
      if (!rev) continue;
      if (children[i].empty()) chain_len[i] = 1;
      else if (children[i].size() == 1 && chain_len[children[i][0]] > 0) chain_len[i] = 1 + chain_len[children[i][0]];
    }
    for (int x = 0; x < nb; ++x) {
      auto& ch = children[x];
      if (ch.size() < 2) continue;
      std::vector<int> paired, rest;
      std::vector<char> used(ch.size(), 0);
      for (size_t a = 0; a < ch.size(); ++a) {
        if (used[a] || chain_len[ch[a]] == 0) continue;
        for (size_t b = a + 1; b < ch.size(); ++b) {
          if (used[b] || chain_len[ch[b]] != chain_len[ch[a]]) continue;
          used[a] = used[b] = 1;
          paired.push_back(ch[a]); paired.push_back(ch[b]);
          pairs.push_back({ch[a], ch[b], chain_len[ch[a]]});
          break;
        }
      }
      for (size_t a = 0; a < ch.size(); ++a) if (!used[a]) rest.push_back(ch[a]);
      paired.insert(paired.end(), rest.begin(), rest.end());
      ch = paired;
    }
  }
  // Child order is free.  A branch node's pending slot is idle while its LAST child's subtree is processed (inward: that
  // subtree runs first; outward: it runs last), so -- as in Sethi-Ullman numbering -- the child whose subtree needs the
  // most slots goes last:  need(X) = max(need(c_last), 1 + max need(other children)).
  {
    std::vector<int> need(nb, 0);
    for (int i = nb - 1; i >= 0; --i) {
      auto& ch = children[i];
      if (ch.size() == 1) need[i] = need[ch[0]];
      else if (ch.size() >= 2) {
        size_t best = 0;
        for (size_t k = 1; k < ch.size(); ++k) if (need[ch[k]] > need[ch[best]]) best = k;
        int c = ch[best];
        if (need[c] > 0) {               // (paired chains need 0 slots and are never moved)
          ch.erase(ch.begin() + best);
          ch.push_back(c);
        } else {
          c = ch.back();
        }
        int other = 0;
        for (size_t k = 0; k + 1 < ch.size(); ++k) other = std::max(other, need[ch[k]]);
        need[i] = std::max(need[c], 1 + other);
      }
    }
  }
  // A 1-DoF body's canonical frame is only fixed up to a rotation about its own axis.  Spend that freedom on the body's
  // FIRST child (the one that follows it in preorder, i.e. the continuation of the chain): when the child is revolute and
  // its axis is perpendicular to this body's axis, turn this frame so that the child's axis is its +x.  The child's tree
  // rotation then is  P Rz(gamma)  (see F_ZPERP), which the ABA passes exploit.  RBD_ZFAST=0 disables, 1 = perpendicular only.
  const int zfast = getenv("RBD_ZFAST") ? atoi(getenv("RBD_ZFAST")) : 2;
  if (zfast > 0) {
    for (int p = 0; p < nb; ++p) {
      const int kp = desc->jtype[p];
      if (!(kp == K_REV || kp == K_PRIS || kp == K_SINCOS) || children[p].empty()) continue;
      const int c = children[p].front();
      if (desc->jtype[c] != K_REV) continue;
      Mat3 Rt{}; std::memcpy(Rt.m, desc->X_tree + 12 * c, sizeof(Rt.m));
      double ax[3] = {desc->jparam[9 * c], desc->jparam[9 * c + 1], desc->jparam[9 * c + 2]};
      const double na = norm3(ax);
      if (na < 1e-12) continue;
      for (double& v : ax) v /= na;
      double ac[3];
      mulv(Rt, ax, ac);                                   // child's axis in this body's original frame
      const double z[3] = {A[p].m[2], A[p].m[5], A[p].m[8]};
      const double d = ac[0] * z[0] + ac[1] * z[1] + ac[2] * z[2];
      if (std::fabs(d) > 1e-12) continue;                 // not perpendicular
      double x[3] = {ac[0] - d * z[0], ac[1] - d * z[1], ac[2] - d * z[2]};
      const double nx = norm3(x);
      for (double& v : x) v /= nx;
      double y[3];
      cross(z, x, y);
      for (int i = 0; i < 3; ++i) { A[p].m[3 * i + 0] = x[i]; A[p].m[3 * i + 1] = y[i]; }
    }
  }
  out.order.clear();
  out.pos.assign(nb, -1);
  {
    std::vector<int> stack(roots.rbegin(), roots.rend());
    while (!stack.empty()) {
      int j = stack.back(); stack.pop_back();
      out.pos[j] = (int)out.order.size();
      out.order.push_back(j);
      for (auto it = children[j].rbegin(); it != children[j].rend(); ++it) stack.push_back(*it);
    }
  }

  ModelDev<double>& M = out.dev64;
  std::memset(&M, 0, sizeof(M));
  M.nb = nb; M.nq = nq; M.nv = nv;
  for (int k = 0; k < 3; ++k) M.g[k] = desc->gravity[k];

  std::vector<int> subtree_size(nb, 1);   // reference-indexed
  for (int i = nb - 1; i >= 0; --i) if (desc->parent[i] >= 0) subtree_size[desc->parent[i]] += subtree_size[i];
  std::vector<int> slot_free_at;          // slot -> first preorder position at which it may be re-used
  int nslots = 0, row = 0;
  bool general = false, other_kinds = false;
  for (int p = 0; p < nb; ++p) {
    const int j = out.order[p];
    BodyDev<double>& b = M.body[p];
    const int par_ref = desc->parent[j];
    const int par = par_ref < 0 ? -1 : out.pos[par_ref];
    b.kind = desc->jtype[j];
    b.parent = par;
    b.qrow = out.qstart[j];
    b.vrow = out.vstart[j];
    b.refidx = j;
    // canonicalised tree transform and inertia
    Mat3 Rt{}; std::memcpy(Rt.m, desc->X_tree + 12 * j, sizeof(Rt.m));
    const double* pt = desc->X_tree + 12 * j + 9;
    Mat3 Ap = par_ref < 0 ? ident() : A[par_ref];
    Mat3 Rc = mul(mul(transp(Ap), Rt), A[j]);
    double pc[3]; mulv(transp(Ap), pt, pc);
    std::memcpy(b.Rt, Rc.m, sizeof(Rc.m));
    std::memcpy(b.pt, pc, sizeof(pc));
    const double* in = desc->inertia + 13 * j;
    Mat3 Jm{}; std::memcpy(Jm.m, in, sizeof(Jm.m));
    Mat3 Jc = mul(mul(transp(A[j]), Jm), A[j]);
    b.J[0] = Jc.m[0]; b.J[1] = 0.5 * (Jc.m[1] + Jc.m[3]); b.J[2] = 0.5 * (Jc.m[2] + Jc.m[6]);
    b.J[3] = Jc.m[4]; b.J[4] = 0.5 * (Jc.m[5] + Jc.m[7]); b.J[5] = Jc.m[8];
    mulv(transp(A[j]), in + 9, b.h);
    b.m = in[12];
    {
      Mat3 At = transp(A[j]);
      out.alignT.insert(out.alignT.end(), At.m, At.m + 9);
      out.total_mass += in[12];
    }
    // flags
    const int nchild = (int)children[j].size();
    int flags = 0;
    if (nchild == 0) flags |= F_LEAF;
    if (nchild >= 2) flags |= F_HAS_PENDING;
    if (par < 0) flags |= F_ROOT_CHILD;
    else {
      if (par == p - 1) flags |= F_FIRST_CHILD;
      else if (children[par_ref].back() == j) flags |= F_SLOT_INIT;
    }
    // fast classes of revolute joints (F_ZPAR / F_ZPERP): the canonical tree rotation Rc's third column is the child's axis
    b.qoff = 0.0;
    if (b.kind == K_REV && zfast > 0) {
      const double cx = Rc.m[2], cy = Rc.m[5], cz = Rc.m[8];
      const double tol = 1e-12;
      if (std::fabs(cx - 1) < tol && std::fabs(cy) < tol && std::fabs(cz) < tol) {
        flags |= F_ZPERP;                                 // Rc = P Rz(gamma):  P^T Rc = Rz(gamma), (P^T w) = (w_y, w_z, w_x)
        b.qoff = std::atan2(Rc.m[6], Rc.m[3]);
      } else if (zfast > 1 && std::fabs(cz - 1) < tol && std::fabs(cx) < tol && std::fabs(cy) < tol) {
        flags |= F_ZPAR;                                  // Rc = Rz(gamma)
        b.qoff = std::atan2(Rc.m[3], Rc.m[0]);
      }
    }
    if ((flags & (F_ZPAR | F_ZPERP)) && pc[0] == 0.0 && pc[1] == 0.0 && pc[2] == 0.0 &&
        !(getenv("RBD_ZERO_R") && getenv("RBD_ZERO_R")[0] == '0'))
      flags |= F_ZERO_R;
    b.flags = flags;
    // Pending slot of a branch node: live over the preorder interval [p, position of its last child] in BOTH directions
    // (inward: written when the last child's subtree is done, read at p; outward: written at p, last read by the last
    // child).  Greedy interval colouring in order of increasing p.
    b.oslot = -1;
    if (flags & F_HAS_PENDING) {
      int s = 0;
      for (;; ++s) {
        if (s == (int)slot_free_at.size()) slot_free_at.push_back(-1);
        if (slot_free_at[s] <= p) break;
      }
      // children[j] is in evaluation order; the last child's position is not known yet in preorder numbering, but it is
      // p + (size of the subtrees of all earlier children) + 1
      int last_pos = p + 1;
      for (size_t k = 0; k + 1 < children[j].size(); ++k) last_pos += subtree_size[children[j][k]];
      slot_free_at[s] = last_pos;   // reusable by a branch node that starts at or after the last child
      b.oslot = s;
      nslots = std::max(nslots, s + 1);
    }
    b.pslot = (par >= 0 && !(flags & F_FIRST_CHILD)) ? M.body[par].oslot : -1;
    // ABA stash rows
    const int k = kind_nv(b.kind);
    const bool multi = k > 1;
    if (multi && !(p == 0 && par < 0)) general = true;
    if (b.kind == K_PRIS || b.kind == K_FIXED) other_kinds = true;
    b.row0 = row;
    if (k <= 1) row += (b.kind == K_FIXED) ? 6 : kRowsOneDof;
    else if (p == 0 && par < 0) row += 6;                 // root multi-DoF joint: only its velocity is stashed
    else row += 7 * k;                                    // U~ (6k) + u~ (k), also holds v (6) between passes 1 and 2
  }
  // (a non-first child implies >= 2 children, so its parent always owns a slot)
  M.slot_base = row;
  M.nslots = nslots;
  M.nrows = row + nslots * kSlotRowsAba;
  out.nslots = nslots;
  out.general = general;
  out.other_kinds = other_kinds;
  fill_dev(out, M, out.dev32);
  return RBD_OK;
}

}  // namespace rbd
