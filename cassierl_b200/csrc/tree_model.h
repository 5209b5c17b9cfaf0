// Device-constant kinematic tree of a free-base 3-D robot (cassie3d_stiff.xml: BASELINE.json configs[3], SURVEY 8(f) row 2).
//
// What mj_loadXML + mj_setConst produce for the reference's model/cassie3d_stiff.xml:53-192 (free joint :60, abduction /
// yaw / hip / knee / ankle / toe / achilles hinges :67-125, two connects :174-177, ten motors :180-191), flattened on the
// host by mjcf_flatten.cpp into moving LINKS: bodies without a joint (shin, heel spring, knee spring) are welded into their
// parent link (mass, centre of mass and inertia combined; their geoms and connect anchors re-expressed in the link frame).
// Link 0 is the free base (dofs 0..2 world-axis translation, 3..5 rotation about the base's own axes, qpos = position +
// unit quaternion w x y z); link l >= 1 hangs on one hinge, dof 5 + l, qpos 6 + l.  Links are stored in depth order.
#pragma once

namespace cassie {
namespace tree {

constexpr int kMaxLinks = 15;
constexpr int kMaxDof = 20;
constexpr int kMaxGeoms = 12;
constexpr int kMaxPairs = 32;    // collision pairs that pass the contype / conaffinity filter
constexpr int kMaxEq = 2;
constexpr int kMaxAct = 12;
constexpr int kMaxLevels = 12;
constexpr int kMaxCon = 14;      // contacts kept per step (the rest are dropped and counted: mjData nconmax)
constexpr int kMaxRows = 48;     // constraint rows per step (njmax)
// the four foot sites of the env observation, in this order (cassie3d_stiff.xml:43-44, 86-87)
enum FootSite { kSiteLeftFront = 0, kSiteLeftRear = 1, kSiteRightFront = 2, kSiteRightRear = 3, kNumFootSites = 4 };

enum GeomType { kPlane = 0, kSphere = 2, kCapsule = 3 };

template <typename T>
struct TreeModel {
  int nl, nv, nq, ng, npair, neq, nu, iterations, nlevels;
  T timestep, tolerance, impratio, meaninertia;
  T gravity[3];
  // ---- links (depth order; level_off[k]..level_off[k+1] are the links of depth k)
  int parent[kMaxLinks];
  int level_off[kMaxLevels + 1];
  int child_off[kMaxLinks + 1], child[kMaxLinks];     // children of link l: child[child_off[l] .. child_off[l+1])
  unsigned anc[kMaxLinks];                              // bit d set: dof d moves link l
  T lpos[kMaxLinks][3], lmat[kMaxLinks][9];             // link frame in the parent link frame at q = ref (row-major)
  T axis[kMaxLinks][3], jpos[kMaxLinks][3], ref[kMaxLinks];   // hinge axis / anchor in the link frame
  T mass[kMaxLinks], com[kMaxLinks][3], inertia[kMaxLinks][6];  // about the com, link frame: xx yy zz xy xz yz
  // ---- dofs
  T damping[kMaxDof], armature[kMaxDof], dof_invweight[kMaxDof];
  int limited[kMaxDof];
  int user_dof[kMaxDof];   // MuJoCo's dof index (file order) of internal dof d; qpos index = user_dof + 1 for hinges
  int dof_of_user[kMaxDof];   // the inverse map
  T range[kMaxDof][2], lim_solref[kMaxDof][2], lim_solimp[kMaxDof][5];
  // ---- collision geoms on links (sphere: p0 = centre; capsule: p0 = the 'to' end, p1 = the 'from' end -- the order in
  // which mjc_PlaneCapsule emits its two contacts), plus at most one world plane
  int g_link[kMaxGeoms], g_type[kMaxGeoms];
  T g_p0[kMaxGeoms][3], g_p1[kMaxGeoms][3], g_radius[kMaxGeoms];
  int has_plane;
  T plane_pos[3], plane_n[3];
  // ---- collision pairs in MuJoCo's order; a = -1: the world plane.  Contact parameters are mixed per pair on the host
  // (mj_contactParam: condim max, friction max, solref / solimp averaged) and carry the summed body_invweight0
  int pair_a[kMaxPairs], pair_b[kMaxPairs], pair_condim[kMaxPairs];
  T pair_friction[kMaxPairs][3], pair_solref[kMaxPairs][2], pair_solimp[kMaxPairs][5], pair_invweight[kMaxPairs];
  // ---- connects
  int eq_l1[kMaxEq], eq_l2[kMaxEq];
  T eq_a1[kMaxEq][3], eq_a2[kMaxEq][3], eq_solref[kMaxEq][2], eq_solimp[kMaxEq][5], eq_invweight[kMaxEq];
  // ---- motors
  int act_dof[kMaxAct], act_limited[kMaxAct];
  T act_gear[kMaxAct], act_lo[kMaxAct], act_hi[kMaxAct];
  T qpos0[kMaxDof + 1];
  // ---- foot contact sites (kSiteLeftFront, kSiteLeftRear, kSiteRightFront, kSiteRightRear): link and position in the
  // link frame after welding.  Read by the env epilogue only (tree_env.cuh), so they sit behind everything the step reads.
  int site_link[kNumFootSites];
  T site_pos[kNumFootSites][3];
};

template <typename T, typename S>
inline void cast_tree_model(TreeModel<T>* d, const TreeModel<S>& s) {
  // both are standard-layout with identical member order: copy member-wise through the int / real split
  d->nl = s.nl; d->nv = s.nv; d->nq = s.nq; d->ng = s.ng; d->npair = s.npair; d->neq = s.neq; d->nu = s.nu;
  d->iterations = s.iterations; d->nlevels = s.nlevels;
  d->timestep = (T)s.timestep; d->tolerance = (T)s.tolerance; d->impratio = (T)s.impratio; d->meaninertia = (T)s.meaninertia;
  for (int i = 0; i < 3; i++) { d->gravity[i] = (T)s.gravity[i]; d->plane_pos[i] = (T)s.plane_pos[i]; d->plane_n[i] = (T)s.plane_n[i]; }
  d->has_plane = s.has_plane;
  for (int l = 0; l < kMaxLinks; l++) {
    d->parent[l] = s.parent[l]; d->child[l] = s.child[l]; d->anc[l] = s.anc[l];
    for (int i = 0; i < 3; i++) { d->lpos[l][i] = (T)s.lpos[l][i]; d->axis[l][i] = (T)s.axis[l][i]; d->jpos[l][i] = (T)s.jpos[l][i]; d->com[l][i] = (T)s.com[l][i]; }
    for (int i = 0; i < 9; i++) d->lmat[l][i] = (T)s.lmat[l][i];
    for (int i = 0; i < 6; i++) d->inertia[l][i] = (T)s.inertia[l][i];
    d->ref[l] = (T)s.ref[l]; d->mass[l] = (T)s.mass[l];
  }
  for (int l = 0; l <= kMaxLinks; l++) d->child_off[l] = s.child_off[l];
  for (int l = 0; l <= kMaxLevels; l++) d->level_off[l] = s.level_off[l];
  for (int i = 0; i < kMaxDof; i++) {
    d->damping[i] = (T)s.damping[i]; d->armature[i] = (T)s.armature[i]; d->dof_invweight[i] = (T)s.dof_invweight[i];
    d->limited[i] = s.limited[i]; d->user_dof[i] = s.user_dof[i]; d->dof_of_user[i] = s.dof_of_user[i];
    for (int k = 0; k < 2; k++) { d->range[i][k] = (T)s.range[i][k]; d->lim_solref[i][k] = (T)s.lim_solref[i][k]; }
    for (int k = 0; k < 5; k++) d->lim_solimp[i][k] = (T)s.lim_solimp[i][k];
  }
  for (int i = 0; i <= kMaxDof; i++) d->qpos0[i] = (T)s.qpos0[i];
  for (int g = 0; g < kMaxGeoms; g++) {
    d->g_link[g] = s.g_link[g]; d->g_type[g] = s.g_type[g]; d->g_radius[g] = (T)s.g_radius[g];
    for (int i = 0; i < 3; i++) { d->g_p0[g][i] = (T)s.g_p0[g][i]; d->g_p1[g][i] = (T)s.g_p1[g][i]; }
  }
  for (int p = 0; p < kMaxPairs; p++) {
    d->pair_a[p] = s.pair_a[p]; d->pair_b[p] = s.pair_b[p]; d->pair_condim[p] = s.pair_condim[p];
    d->pair_invweight[p] = (T)s.pair_invweight[p];
    for (int k = 0; k < 3; k++) d->pair_friction[p][k] = (T)s.pair_friction[p][k];
    for (int k = 0; k < 2; k++) d->pair_solref[p][k] = (T)s.pair_solref[p][k];
    for (int k = 0; k < 5; k++) d->pair_solimp[p][k] = (T)s.pair_solimp[p][k];
  }
  for (int e = 0; e < kMaxEq; e++) {
    d->eq_l1[e] = s.eq_l1[e]; d->eq_l2[e] = s.eq_l2[e]; d->eq_invweight[e] = (T)s.eq_invweight[e];
    for (int k = 0; k < 3; k++) { d->eq_a1[e][k] = (T)s.eq_a1[e][k]; d->eq_a2[e][k] = (T)s.eq_a2[e][k]; }
    for (int k = 0; k < 2; k++) d->eq_solref[e][k] = (T)s.eq_solref[e][k];
    for (int k = 0; k < 5; k++) d->eq_solimp[e][k] = (T)s.eq_solimp[e][k];
  }
  for (int a = 0; a < kMaxAct; a++) {
    d->act_dof[a] = s.act_dof[a]; d->act_limited[a] = s.act_limited[a];
    d->act_gear[a] = (T)s.act_gear[a]; d->act_lo[a] = (T)s.act_lo[a]; d->act_hi[a] = (T)s.act_hi[a];
  }
  for (int k = 0; k < kNumFootSites; k++) {
    d->site_link[k] = s.site_link[k];
    for (int i = 0; i < 3; i++) d->site_pos[k][i] = (T)s.site_pos[k][i];
  }
}

}  // namespace tree
}  // namespace cassie
