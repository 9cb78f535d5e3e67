// =====================================================================================================================
// Warp-per-env kernel (second mapping).  One warp owns one env; the whole mj_forward working set lives in shared memory
// (~24 KB per env) and every stage is spread over the 32 lanes: bodies / dofs / joints / geoms / collision pairs /
// constraint rows each get a lane, tree recursions run level by level (depth <= 6), the L^T D L factorisation runs its 23
// pivots sequentially with the (i, j) updates of a pivot in parallel, and all M^-1 solves (one per constraint row plus
// the smooth acceleration) run at once, one right-hand side per lane, with the operand vector in registers and
// statically indexed (humanoid_tree.inc).  Every output element is still produced by ONE lane executing the same
// operation order as the thread-per-env code above, so results are bit-identical to it and to oracle/humanoid.c.

// Shared-memory working set of one env (~24 KB: 8 envs resident per SM, which is also what the register file allows).
// Arrays whose lifetimes do not overlap share storage: position-stage temporaries, velocity-stage temporaries and the
// constraint Jacobian (used in that order inside w_forward).  L / M use the packed tree storage of humanoid_tree.inc;
// the symmetric AR matrix is stored as its lower triangle.
constexpr int kTriAR = MAXEFC * (MAXEFC + 1) / 2;
struct WS {
  double qpos[NQ], qvel[NV], warm[NV], ctrl[NU];
  double X0q[NQ], Xv[4][NV], F[4][NV], sv[NV], sa[NV];
  double xipos[NB][3], geom_xpos[NG][3], geom_axis[NG][3], subtree[NB][3];
  double cinert[NB][10], cdof[NV][6], cvel[NB][6], cfrc_ext[NB][6];
  double LDp[B2E_LD_NPACK], dinv[NV], tmp[16], rowk[16];
  double passive[NV], actuator[NV], smooth[NV], qacc_smooth[NV], qacc[NV];
  double ten_length[2], ten_velocity[2];
  int ncon, nefc, overflow, work;  // work: constraint-solver effort of this step (scheduling hint for the next one)
  Contact con[MAXCON];
  union {
    struct { double xpos[NB][3], xquat[NB][4], xmat[NB][9], xanchor[NJ][3], xaxis[NJ][3], crb[NB][10], ql[NJ][4]; } p;  // position stage
    struct { double cdof_dot[NV][6], cacc[NB][6], cfrc[NB][6]; } v;                                          // velocity stage
    double J[MAXEFC][NV];                                                                                    // constraint stage
  } u;
  double AR[kTriAR];
  double R[MAXEFC], D[MAXEFC], aref[MAXEFC], b[MAXEFC], force[MAXEFC], term[MAXEFC];
};
__device__ __forceinline__ int tri(int i, int j) { return i >= j ? i * (i + 1) / 2 + j : j * (j + 1) / 2 + i; }

#define WSYNC() __syncwarp()

// one body of mj_kinematics (same statements as the loop body of kinematics())
__device__ void w_kin_body(const HModel& m, WS& w, int b) {
  const double* q = w.qpos;
  double xpos[3], xquat[4];
  if (m.body_jntnum[b] && m.jnt_type[m.body_jntadr[b]] == 0) {
    cp3(xpos, q);
    for (int k = 0; k < 4; ++k) xquat[k] = q[3 + k];
    const int j = m.body_jntadr[b];
    cp3(w.u.p.xanchor[j], xpos);
    w.u.p.xaxis[j][0] = 0; w.u.p.xaxis[j][1] = 0; w.u.p.xaxis[j][2] = 1;
  } else {
    const int p = m.parent[b];
    double t[3];
    mulmatvec3(t, w.u.p.xmat[p], m.body_pos[b]);
    for (int k = 0; k < 3; ++k) xpos[k] = w.u.p.xpos[p][k] + t[k];
    quat_mul(xquat, w.u.p.xquat[p], m.body_quat[b]);
    for (int jj = 0; jj < m.body_jntnum[b]; ++jj) {
      const int j = m.body_jntadr[b] + jj;
      double v[3];
      quat_rot(v, xquat, m.jnt_pos[j]);
      for (int k = 0; k < 3; ++k) w.u.p.xanchor[j][k] = xpos[k] + v[k];
      quat_rot(w.u.p.xaxis[j], xquat, m.jnt_axis[j]);
      quat_mul(xquat, xquat, w.u.p.ql[j]);  // joint rotation, precomputed for all joints at once
      quat_rot(v, xquat, m.jnt_pos[j]);
      for (int k = 0; k < 3; ++k) xpos[k] = w.u.p.xanchor[j][k] - v[k];
    }
  }
  quat_normalize(xquat);
  cp3(w.u.p.xpos[b], xpos);
  for (int k = 0; k < 4; ++k) w.u.p.xquat[b][k] = xquat[k];
  quat2mat(w.u.p.xmat[b], xquat);
}

// narrow phase of one geom pair; returns the number of contacts (0..2) written to out[]
__device__ int w_collide_pair(const HModel& m, const WS& w, int g1, int g2, Contact* out) {
  int n = 0;
  const int t1 = m.geom_type[g1], t2 = m.geom_type[g2];
  const double *p1 = w.geom_xpos[g1], *p2 = w.geom_xpos[g2];
  if (t1 != G_PLANE) {
    const double df[3] = {p2[0] - p1[0], p2[1] - p1[1], p2[2] - p1[2]};
    const double bound = m.geom_rbound[g1] + m.geom_rbound[g2] + m.margin;
    if (dot3(df, df) > bound * bound) return 0;
  }
  auto emit = [&](double dist, const double* pos, const double* normal, const double* hint) {
    Contact& c = out[n++];
    c.g1 = g1; c.g2 = g2; c.dist = dist;
    cp3(c.pos, pos);
    cp3(c.frame, normal);
    if (hint) cp3(c.frame + 3, hint); else c.frame[3] = c.frame[4] = c.frame[5] = 0;
    make_frame(c.frame);
    c.dim = m.geom_condim[g1] > m.geom_condim[g2] ? m.geom_condim[g1] : m.geom_condim[g2];
    c.mu = m.geom_friction[g1] > m.geom_friction[g2] ? m.geom_friction[g1] : m.geom_friction[g2];
    c.efc_adr = -1;
  };
  auto sph_sph = [&](const double* a, double r1, const double* bq, double r2) {
    double nn[3] = {bq[0] - a[0], bq[1] - a[1], bq[2] - a[2]};
    const double len = norm3(nn);
    const double dist = len - r1 - r2;
    if (dist >= m.margin) return;
    if (len < MINVAL) { nn[0] = 1; nn[1] = 0; nn[2] = 0; } else { nn[0] /= len; nn[1] /= len; nn[2] /= len; }
    double pos[3];
    for (int k = 0; k < 3; ++k) pos[k] = a[k] + nn[k] * (r1 + 0.5 * dist);
    emit(dist, pos, nn, nullptr);
  };
  auto plane_sph = [&](const double* c, double r, const double* hint) {
    const double* ax = w.geom_axis[g1];
    const double nn[3] = {ax[0], ax[1], ax[2]};
    const double df[3] = {c[0] - w.geom_xpos[g1][0], c[1] - w.geom_xpos[g1][1], c[2] - w.geom_xpos[g1][2]};
    const double dist = dot3(df, nn) - r;
    if (dist >= m.margin) return;
    double pos[3];
    for (int k = 0; k < 3; ++k) pos[k] = c[k] - nn[k] * (r + 0.5 * dist);
    emit(dist, pos, nn, hint);
  };
  if (t1 == G_PLANE && t2 == G_SPHERE) {
    plane_sph(p2, m.geom_size[g2][0], nullptr);
  } else if (t1 == G_PLANE && t2 == G_CAPSULE) {
    const double* ax = w.geom_axis[g2];
    const double axis[3] = {ax[0], ax[1], ax[2]}, h = m.geom_size[g2][1];
    double e1[3], e2[3];
    for (int k = 0; k < 3; ++k) { e1[k] = p2[k] + axis[k] * h; e2[k] = p2[k] - axis[k] * h; }
    plane_sph(e1, m.geom_size[g2][0], axis);
    plane_sph(e2, m.geom_size[g2][0], axis);
  } else if (t1 == G_SPHERE && t2 == G_SPHERE) {
    sph_sph(p1, m.geom_size[g1][0], p2, m.geom_size[g2][0]);
  } else if (t1 == G_SPHERE && t2 == G_CAPSULE) {
    const double* ax = w.geom_axis[g2];
    const double axis[3] = {ax[0], ax[1], ax[2]}, h = m.geom_size[g2][1];
    const double df[3] = {p1[0] - p2[0], p1[1] - p2[1], p1[2] - p2[2]};
    double x = dot3(axis, df);
    x = x > h ? h : (x < -h ? -h : x);
    const double cp[3] = {p2[0] + axis[0] * x, p2[1] + axis[1] * x, p2[2] + axis[2] * x};
    sph_sph(p1, m.geom_size[g1][0], cp, m.geom_size[g2][0]);
  } else if (t1 == G_CAPSULE && t2 == G_CAPSULE) {
    const double *x1 = w.geom_axis[g1], *x2 = w.geom_axis[g2];
    const double a1[3] = {x1[0], x1[1], x1[2]}, a2[3] = {x2[0], x2[1], x2[2]}, l1 = m.geom_size[g1][1], l2 = m.geom_size[g2][1];
    const double df[3] = {p1[0] - p2[0], p1[1] - p2[1], p1[2] - p2[2]};
    const double ma = dot3(a1, a1), mb = -dot3(a1, a2), mc = dot3(a2, a2), u = -dot3(a1, df), v = dot3(a2, df);
    const double det = ma * mc - mb * mb;
    if (fabs(det) >= MINVAL) {
      double xa = (mc * u - mb * v) / det, xb = (ma * v - mb * u) / det;
      if (xa > l1) { xa = l1; xb = (v - mb * l1) / mc; }
      else if (xa < -l1) { xa = -l1; xb = (v + mb * l1) / mc; }
      if (xb > l2) { xb = l2; xa = (u - mb * l2) / ma; if (xa > l1) xa = l1; else if (xa < -l1) xa = -l1; }
      else if (xb < -l2) { xb = -l2; xa = (u + mb * l2) / ma; if (xa > l1) xa = l1; else if (xa < -l1) xa = -l1; }
      double c1[3], c2[3];
      for (int k = 0; k < 3; ++k) { c1[k] = p1[k] + a1[k] * xa; c2[k] = p2[k] + a2[k] * xb; }
      sph_sph(c1, m.geom_size[g1][0], c2, m.geom_size[g2][0]);
    } else {
      for (int sgn = -1; sgn <= 1; sgn += 2) {
        double c1[3], c2[3];
        for (int k = 0; k < 3; ++k) c1[k] = p1[k] + a1[k] * (sgn * l1);
        const double dd[3] = {c1[0] - p2[0], c1[1] - p2[1], c1[2] - p2[2]};
        double x = dot3(a2, dd);
        x = x > l2 ? l2 : (x < -l2 ? -l2 : x);
        for (int k = 0; k < 3; ++k) c2[k] = p2[k] + a2[k] * x;
        sph_sph(c1, m.geom_size[g1][0], c2, m.geom_size[g2][0]);
      }
    }
  }
  return n;
}

// children of the parents at one tree level are added into them, K components of every parent at once:
// lane = (parent slot, component).  Same sums as `for b = NB-1..1: arr[parent[b]] += arr[b]`.
template <int K>
__device__ __forceinline__ void w_tree_sum(const HModel& m, double* arr /*[NB][K]*/, int lane, int last_level) {
  const int slot = lane / K, comp = lane - slot * K;
  for (int lvl = 5; lvl >= last_level; --lvl) {
    if (slot < 3) {
      const int p = m.lvl_parents[lvl][slot];
      if (p >= 0) {
        double acc = arr[p * K + comp];
        for (int ci = 0; ci < 3; ++ci) {
          const int c = m.children[p][ci];  // descending body index
          if (c < 0) break;
          acc += arr[c * K + comp];
        }
        arr[p * K + comp] = acc;
      }
    }
    WSYNC();
  }
}

#define LDP(o) w.LDp[o]
#define B2E_SOLVE_FENCE() __syncwarp(solve_mask)  // ptxas keeps shared loads behind it: bounds the loads in flight
#define DINV(i) w.dinv[i]

// mj_forward for the env of this warp; inputs w.qpos, w.qvel, w.warm, w.ctrl; output w.qacc (+ all derived arrays)
__device__ __noinline__ void w_forward(const WModel& wm, WS& w, int lane) {
  const HModel& m = wm.m;
  // ---- position stage ----------------------------------------------------------------------------------------------------
  if (lane == 0) {
    quat_normalize(w.qpos + 3);
    for (int k = 0; k < 3; ++k) { w.u.p.xpos[0][k] = 0; w.xipos[0][k] = 0; }
    w.u.p.xquat[0][0] = 1; w.u.p.xquat[0][1] = w.u.p.xquat[0][2] = w.u.p.xquat[0][3] = 0;
    for (int k = 0; k < 9; ++k) w.u.p.xmat[0][k] = (k % 4 == 0) ? 1.0 : 0.0;
  }
  if (lane >= 1 && lane < NJ)  // everything of mj_kinematics that does not depend on the parent body: the joint rotations
    quat_axisangle(w.u.p.ql[lane], m.jnt_axis[lane], w.qpos[m.jnt_qposadr[lane]] - m.qpos0[m.jnt_qposadr[lane]]);
  WSYNC();
  for (int lvl = 1; lvl <= 6; ++lvl) {
    if (lane > 0 && lane < NB && m.body_depth[lane] == lvl) w_kin_body(m, w, lane);
    WSYNC();
  }
  if (lane > 0 && lane < NB) {
    double t[3];
    mulmatvec3(t, w.u.p.xmat[lane], m.body_ipos[lane]);
    for (int k = 0; k < 3; ++k) w.xipos[lane][k] = w.u.p.xpos[lane][k] + t[k];
  }
  if (lane < NG) {
    const int g = lane, b = m.geom_body[g];
    double t[3];
    mulmatvec3(t, w.u.p.xmat[b], m.geom_pos[g]);
    for (int k = 0; k < 3; ++k) w.geom_xpos[g][k] = w.u.p.xpos[b][k] + t[k];
    double gm[9];
    mulmat3(gm, w.u.p.xmat[b], m.geom_mat[g]);
    w.geom_axis[g][0] = gm[2]; w.geom_axis[g][1] = gm[5]; w.geom_axis[g][2] = gm[8];
  }
  // mj_comPos
  if (lane < NB)
    for (int k = 0; k < 3; ++k) w.subtree[lane][k] = m.body_mass[lane] * w.xipos[lane][k];
  WSYNC();
  w_tree_sum<3>(m, &w.subtree[0][0], lane, 0);
  if (lane < NB) {
    if (m.subtree_mass[lane] < MINVAL) cp3(w.subtree[lane], w.xipos[lane]);
    else for (int k = 0; k < 3; ++k) w.subtree[lane][k] /= m.subtree_mass[lane];
  }
  WSYNC();
  const double root[3] = {w.subtree[1][0], w.subtree[1][1], w.subtree[1][2]};
  if (lane == 0) for (int k = 0; k < 10; ++k) w.cinert[0][k] = 0;
  if (lane > 0 && lane < NB) {
    const int b = lane;
    const double off[3] = {w.xipos[b][0] - root[0], w.xipos[b][1] - root[1], w.xipos[b][2] - root[2]};
    const double* R = w.u.p.xmat[b];
    double RI[9], W[9], Rt[9];
    mulmat3(RI, R, m.body_inertia[b]);
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) Rt[3 * i + j] = R[3 * j + i];
    mulmat3(W, RI, Rt);
    const double mass = m.body_mass[b];
    double* c = w.cinert[b];
    c[0] = W[0] + mass * (off[1] * off[1] + off[2] * off[2]);
    c[1] = W[4] + mass * (off[0] * off[0] + off[2] * off[2]);
    c[2] = W[8] + mass * (off[0] * off[0] + off[1] * off[1]);
    c[3] = W[1] - mass * off[0] * off[1];
    c[4] = W[2] - mass * off[0] * off[2];
    c[5] = W[5] - mass * off[1] * off[2];
    c[6] = mass * off[0]; c[7] = mass * off[1]; c[8] = mass * off[2]; c[9] = mass;
  }
  if (lane < NJ) {
    const int j = lane;
    const double* anchor = w.u.p.xanchor[j];
    const double off[3] = {root[0] - anchor[0], root[1] - anchor[1], root[2] - anchor[2]};
    const int da = m.jnt_dofadr[j];
    if (m.jnt_type[j] == 0) {
      for (int i = 0; i < 3; ++i) {
        for (int k = 0; k < 6; ++k) w.cdof[da + i][k] = 0;
        w.cdof[da + i][3 + i] = 1.0;
      }
      const double* R = w.u.p.xmat[m.jnt_body[j]];
      for (int i = 0; i < 3; ++i) {
        const double ax[3] = {R[i], R[3 + i], R[6 + i]};
        cp3(w.cdof[da + 3 + i], ax);
        cross3(w.cdof[da + 3 + i] + 3, ax, off);
      }
    } else {
      cp3(w.cdof[da], w.u.p.xaxis[j]);
      cross3(w.cdof[da] + 3, w.u.p.xaxis[j], off);
    }
  }
  if (lane < 2) w.ten_length[lane] = -w.qpos[m.ten_q[lane][0]] + w.qpos[m.ten_q[lane][1]];
  WSYNC();
  // mj_crb
  for (int e = lane; e < NB * 10; e += 32) (&w.u.p.crb[0][0])[e] = (&w.cinert[0][0])[e];
  WSYNC();
  w_tree_sum<10>(m, &w.u.p.crb[0][0], lane, 1);
  if (lane < NV) {  // row i of M in the packed tree storage: diagonal, then the ancestors of dof i (nearest first)
    const int i = lane, ro = wm.rowoff[i];
    double buf[6];
    mul_inert_vec(buf, w.u.p.crb[m.dof_body[i]], w.cdof[i]);
    w.LDp[ro] = m.dof_armature[i] + dot6(w.cdof[i], buf);
    const int len = m.dof_chain_len[i];
    for (int a = 0; a < len; ++a) w.LDp[ro + 1 + a] = dot6(w.cdof[m.dof_chain[i][a]], buf);
  }
  WSYNC();
  // mj_factorM: pivots in sequence; the row scaling of a pivot, then all of its (i, j) updates, each in parallel
  for (int k = NV - 1; k >= 0; --k) {
    const int len = m.dof_chain_len[k], ro = wm.rowoff[k];
    const double dkk = w.LDp[ro];
    {  // one division sequence serves the row scaling (lanes < len) and 1 / D[k] (lane 31)
      const double num = lane < len ? w.LDp[ro + 1 + lane] : 1.0;
      const double q = num / dkk;
      if (lane < len) {
        w.rowk[lane] = num;
        w.tmp[lane] = q;
        w.LDp[ro + 1 + lane] = q;
      }
      if (lane == 31) w.dinv[k] = q;
    }
    if (len == 0) continue;
    WSYNC();
    for (int p = wm.fac_start[k] + lane, pe = wm.fac_start[k + 1]; p < pe; p += 32) {
      const unsigned e = wm.fac_pair[p];
      w.LDp[e & 255u] -= w.rowk[(e >> 8) & 15u] * w.tmp[e >> 12];
    }
    WSYNC();
  }
  // mj_collision: pair p = 32 * round + lane, contacts appended in pair order
  {
    int base = 0;
    for (int r0 = 0; r0 < m.npair; r0 += 32) {
      const int p = r0 + lane;
      Contact loc[2];
      int cnt = 0;
      if (p < m.npair) cnt = w_collide_pair(m, w, m.pair_g1[p], m.pair_g2[p], loc);
      const unsigned m1 = __ballot_sync(0xffffffffu, cnt >= 1), m2 = __ballot_sync(0xffffffffu, cnt >= 2);
      const unsigned lt = (1u << lane) - 1u;
      const int off = base + __popc(m1 & lt) + __popc(m2 & lt);
      for (int c = 0; c < cnt; ++c) {
        if (off + c < MAXCON) w.con[off + c] = loc[c];
        else w.overflow = 1;
      }
      base += __popc(m1) + __popc(m2);
    }
    if (lane == 0) w.ncon = base < MAXCON ? base : MAXCON;
  }
  WSYNC();  // the position-stage temporaries (w.u.p) are dead from here on
  // ---- velocity stage (independent of the constraint rows; runs first so that its temporaries can share w.u) -----------
  if (lane == 0) for (int k = 0; k < 6; ++k) w.cvel[0][k] = 0;
  WSYNC();
  for (int lvl = 1; lvl <= 6; ++lvl) {  // mj_comVel, a body per lane, parents first
    if (lane > 0 && lane < NB && m.body_depth[lane] == lvl) {
      const int b = lane;
      double cvel[6];
      for (int k = 0; k < 6; ++k) cvel[k] = w.cvel[m.parent[b]][k];
      for (int jj = 0; jj < m.body_jntnum[b]; ++jj) {
        const int j = m.body_jntadr[b] + jj, da = m.jnt_dofadr[j];
        if (m.jnt_type[j] == 0) {
          for (int i = 0; i < 3; ++i) {
            for (int k = 0; k < 6; ++k) w.u.v.cdof_dot[da + i][k] = 0;
            for (int k = 0; k < 6; ++k) cvel[k] += w.cdof[da + i][k] * w.qvel[da + i];
          }
          for (int i = 3; i < 6; ++i) cross_motion(w.u.v.cdof_dot[da + i], cvel, w.cdof[da + i]);
          for (int i = 3; i < 6; ++i)
            for (int k = 0; k < 6; ++k) cvel[k] += w.cdof[da + i][k] * w.qvel[da + i];
        } else {
          cross_motion(w.u.v.cdof_dot[da], cvel, w.cdof[da]);
          for (int k = 0; k < 6; ++k) cvel[k] += w.cdof[da][k] * w.qvel[da];
        }
      }
      for (int k = 0; k < 6; ++k) w.cvel[b][k] = cvel[k];
    }
    WSYNC();
  }
  if (lane < 2) w.ten_velocity[lane] = -w.qvel[m.ten_v[lane][0]] + w.qvel[m.ten_v[lane][1]];
  if (lane < NV) w.passive[lane] = 0;
  WSYNC();
  if (lane >= 1 && lane < NJ) {
    const int da = m.jnt_dofadr[lane], qa = m.jnt_qposadr[lane];
    w.passive[da] = -m.jnt_stiffness[lane] * (w.qpos[qa] - 0.0) - m.dof_damping[da] * w.qvel[da];
  }
  if (lane == 0) for (int k = 0; k < 3; ++k) { w.u.v.cacc[0][k] = 0; w.u.v.cacc[0][3 + k] = -m.gravity[k]; }
  WSYNC();
  for (int lvl = 1; lvl <= 6; ++lvl) {  // mj_rne forward sweep: only the accelerations depend on the parent body
    if (lane > 0 && lane < NB && m.body_depth[lane] == lvl) {
      const int b = lane;
      double cacc[6];
      for (int k = 0; k < 6; ++k) cacc[k] = w.u.v.cacc[m.parent[b]][k];
      for (int i = 0; i < m.body_dofnum[b]; ++i) {
        const int da = m.body_dofadr[b] + i;
        for (int k = 0; k < 6; ++k) cacc[k] += w.u.v.cdof_dot[da][k] * w.qvel[da];
      }
      for (int k = 0; k < 6; ++k) w.u.v.cacc[b][k] = cacc[k];
    }
    WSYNC();
  }
  if (lane > 0 && lane < NB) {  // cfrc_body = I * cacc + cvel x* (I * cvel), all bodies at once
    const int b = lane;
    double t1[6], t2[6], t3[6];
    mul_inert_vec(t1, w.cinert[b], w.u.v.cacc[b]);
    mul_inert_vec(t2, w.cinert[b], w.cvel[b]);
    cross_force(t3, w.cvel[b], t2);
    for (int k = 0; k < 6; ++k) w.u.v.cfrc[b][k] = t1[k] + t3[k];
  }
  WSYNC();
  w_tree_sum<6>(m, &w.u.v.cfrc[0][0], lane, 1);  // backward sweep (the world body's total is never used)
  if (lane < NV) w.actuator[lane] = 0;
  WSYNC();
  if (lane < NU) {
    double c = w.ctrl[lane];
    c = c < -0.4 ? -0.4 : (c > 0.4 ? 0.4 : c);
    w.actuator[m.act_dof[lane]] += m.act_gear[lane] * c;  // one actuator per dof
  }
  WSYNC();
  if (lane < NV) {
    const double bias = dot6(w.cdof[lane], w.u.v.cfrc[m.dof_body[lane]]);
    w.smooth[lane] = w.passive[lane] - bias + w.actuator[lane];
  }
  WSYNC();  // the velocity-stage temporaries (w.u.v) are dead from here on; w.u.J takes their place
  // ---- mj_makeConstraint: joint-limit rows (joint order, lower side then upper side), then contact rows -----------------
  double* const c_pos = w.b;        // row scratch that is only needed until R / aref are known shares b / force / term
  double* const c_margin = w.force;
  double* const c_diag = w.term;
  int nlim;
  {
    bool lo = false, hi = false;
    double dlo = 0, dhi = 0;
    if (lane >= 1 && lane < NJ) {
      const double value = w.qpos[m.jnt_qposadr[lane]];
      dlo = -1 * (m.jnt_range[lane][0] - value);
      dhi = 1 * (m.jnt_range[lane][1] - value);
      lo = dlo < 0.0;
      hi = dhi < 0.0;
    }
    const unsigned mlo = __ballot_sync(0xffffffffu, lo), mhi = __ballot_sync(0xffffffffu, hi);
    const unsigned lt = (1u << lane) - 1u;
    const int r0 = __popc(mlo & lt) + __popc(mhi & lt);
    nlim = __popc(mlo) + __popc(mhi);
    if (lo) {
      for (int k = 0; k < NV; ++k) w.u.J[r0][k] = 0;
      w.u.J[r0][m.jnt_dofadr[lane]] = 1;
      c_pos[r0] = dlo; c_margin[r0] = 0.0; c_diag[r0] = m.dof_invweight0[m.jnt_dofadr[lane]];
    }
    if (hi) {
      const int r1 = r0 + (lo ? 1 : 0);
      for (int k = 0; k < NV; ++k) w.u.J[r1][k] = 0;
      w.u.J[r1][m.jnt_dofadr[lane]] = -1;
      c_pos[r1] = dhi; c_margin[r1] = 0.0; c_diag[r1] = m.dof_invweight0[m.jnt_dofadr[lane]];
    }
  }
  if (lane == 0) {
    int n = nlim;
    for (int c = 0; c < w.ncon; ++c) {
      const int rows = w.con[c].dim == 1 ? 1 : 4;
      if (n + rows > MAXEFC) { w.con[c].efc_adr = -1; w.overflow = 1; continue; }
      w.con[c].efc_adr = n;
      n += rows;
    }
    w.nefc = n;
  }
  WSYNC();
  const int ncon = w.ncon, n = w.nefc;
  for (int c = 0; c < ncon; ++c) {  // contact Jacobian rows: one dof per lane
    const Contact& con = w.con[c];
    if (con.efc_adr < 0) continue;
    const int b1 = m.geom_body[con.g1], b2 = m.geom_body[con.g2];
    const double tran = m.body_invweight0[b1][0] + m.body_invweight0[b2][0];
    if (lane < NV) {
      const int i = lane;
      const double off[3] = {con.pos[0] - w.subtree[1][0], con.pos[1] - w.subtree[1][1], con.pos[2] - w.subtree[1][2]};
      double j1[3] = {0, 0, 0}, j2[3] = {0, 0, 0}, t[3];
      cross3(t, w.cdof[i], off);
      if ((m.body_dofmask[b1] >> i) & 1u) for (int k = 0; k < 3; ++k) j1[k] = w.cdof[i][3 + k] + t[k];
      if ((m.body_dofmask[b2] >> i) & 1u) for (int k = 0; k < 3; ++k) j2[k] = w.cdof[i][3 + k] + t[k];
      double jc[3];
      for (int r = 0; r < 3; ++r) {
        double sum = 0;
        for (int k = 0; k < 3; ++k) sum += con.frame[3 * r + k] * (j2[k] - j1[k]);
        jc[r] = sum;
      }
      const int a0 = con.efc_adr;
      if (con.dim == 1) {
        w.u.J[a0][i] = jc[0];
      } else {
        int row = a0;
        for (int k = 1; k <= 2; ++k)
          for (int sgn = 1; sgn >= -1; sgn -= 2) w.u.J[row++][i] = jc[0] + sgn * con.mu * jc[k];
      }
    }
    if (lane == 31) {
      const int a0 = con.efc_adr;
      if (con.dim == 1) {
        c_pos[a0] = con.dist; c_margin[a0] = m.margin; c_diag[a0] = tran;
      } else {
        for (int r = 0; r < 4; ++r) {
          c_pos[a0 + r] = con.dist; c_margin[a0 + r] = m.margin;
          c_diag[a0 + r] = tran + con.mu * con.mu * tran;
        }
      }
    }
  }
  WSYNC();
  {
    const double timeconst = m.solref[0] > 2 * m.timestep ? m.solref[0] : 2 * m.timestep, dampratio = m.solref[1];
    const double dmax = m.solimp[1];
    const double K = 1.0 / (dmax * dmax * timeconst * timeconst * dampratio * dampratio), B = 2.0 / (dmax * timeconst);
    if (lane < n) {
      const int i = lane;
      const double imp = impedance(m, c_pos[i], c_margin[i]);
      const double R = (1.0 - imp) / imp * c_diag[i];
      w.R[i] = R < MINVAL ? MINVAL : R;
      double vel = 0;
      for (int k = 0; k < NV; ++k) vel += w.u.J[i][k] * w.qvel[k];
      w.aref[i] = -B * vel - K * imp * (c_pos[i] - c_margin[i]);
    }
  }
  WSYNC();
  if (lane < ncon) {
    const Contact& con = w.con[lane];
    if (con.efc_adr >= 0 && con.dim > 1) {
      const double Rpy = 2.0 * con.mu * con.mu * w.R[con.efc_adr];
      for (int k = 0; k < 4; ++k) w.R[con.efc_adr + k] = Rpy;
    }
  }
  WSYNC();
  if (lane < n) w.D[lane] = 1.0 / w.R[lane];
  // ---- all M^-1 solves at once: lane r < n takes constraint row r, the next lane takes qfrc_smooth ------------------------
  {
    double x[NV];
#pragma unroll 1
    for (int pass = 0; pass < 2; ++pass) {  // pass 1 only when all 32 lanes held a row: lane 0 then solves for qacc_smooth
      const bool row = pass == 0 && lane < n;
      const bool smooth = pass == 0 ? (lane == n) : (n == 32 && lane == 0);
      if (pass == 1 && n < 32) break;
      if (row) {
#pragma unroll
        for (int k = 0; k < NV; ++k) x[k] = w.u.J[lane][k];
      } else {
#pragma unroll
        for (int k = 0; k < NV; ++k) x[k] = w.smooth[k];
      }
      const unsigned solve_mask = __ballot_sync(0xffffffffu, row || smooth);
      if (row || smooth) { B2E_SOLVE_M_UNROLLED(x); }
      if (row) {  // mj_projectConstraint row: AR[r][j] = J_j . (M^-1 J_r), j <= r
        for (int j = 0; j <= lane; ++j) {
          double sum = 0;
#pragma unroll
          for (int k = 0; k < NV; ++k) sum += w.u.J[j][k] * x[k];
          if (j == lane) sum += w.R[lane];
          w.AR[lane * (lane + 1) / 2 + j] = sum;
        }
      }
      if (smooth) {
#pragma unroll
        for (int k = 0; k < NV; ++k) w.qacc_smooth[k] = x[k];
      }
    }
  }
  WSYNC();
  // ---- mj_fwdConstraint (PGS) --------------------------------------------------------------------------------------------------
  if (n == 0) {
    if (lane < NV) w.qacc[lane] = w.qacc_smooth[lane];
    WSYNC();
    return;
  }
  double b_i = 0, f_i = 0;
  if (lane < n) {
    const int i = lane;
    double sum = 0;
    for (int k = 0; k < NV; ++k) sum += w.u.J[i][k] * w.qacc_smooth[k];
    b_i = sum - w.aref[i];
    double jar = 0;
    for (int k = 0; k < NV; ++k) jar += w.u.J[i][k] * w.warm[k];
    jar -= w.aref[i];
    f_i = jar < 0 ? -w.D[i] * jar : 0.0;
    w.force[i] = f_i;  // c_margin (alias of force) is dead: the last reads were two barriers ago
  }
  WSYNC();
  double r_i = 0, aii = 0, ainv = 0;  // this lane's row: running residual (AR f + b)_i, AR[i][i] and its reciprocal
  if (lane < n) {
    const int i = lane;
    double sum = 0;
    for (int j = 0; j < n; ++j) sum += w.AR[tri(i, j)] * w.force[j];
    w.term[i] = f_i * (0.5 * sum + b_i);
    r_i = b_i + sum;
    aii = w.AR[i * (i + 1) / 2 + i];
    ainv = 1.0 / aii;
  }
  WSYNC();
  {
    double cost = 0;  // every lane adds the terms in row order: the decision is warp-uniform without a broadcast
    for (int i = 0; i < n; ++i) cost += w.term[i];
    if (cost > 0) { f_i = 0; r_i = b_i; }
  }
  {
    // Gauss-Seidel sweeps in residual-update form, one row per lane: row j moves by delta_j (computed by lane j from its
    // own residual), every lane then moves its residual by AR[i][j] * delta_j.  Lanes >= n carry zeros.
    const double scale = 1.0 / (m.meaninertia * (NV > 1 ? NV : 1));
    const int iters = m.iterations;
    const double tol = m.tolerance;
    const int tri0 = lane * (lane + 1) / 2;
    for (int it = 0; it < iters; ++it) {
      double d_own = 0, r_own = 0;  // this lane's move and the residual it was computed from (for the cost change)
      int idx = tri0;               // index of AR[lane][j] in the packed lower triangle (in bounds for lanes < MAXEFC)
#pragma unroll 1
      for (int j = 0; j < n; ++j) {
        double f = f_i - r_i * ainv;
        if (f < 0) f = 0;
        const double delta = f - f_i;
        const double dj = __shfl_sync(0xffffffffu, delta, j);
        if (lane == j) { f_i = f; d_own = delta; r_own = r_i; }
        r_i += (lane < MAXEFC ? w.AR[idx] : 0.0) * dj;  // lanes >= n accumulate junk nobody reads; lanes >= MAXEFC have no row
        idx += j < lane ? 1 : j + 1;
      }
      // cost change of the sweep: the per-row gains added in row order by every lane (warp-uniform break, no broadcast)
      double* const gains = (it & 1) ? w.term : w.b;  // b_i is in registers; two buffers: no barrier after the reads
      if (lane < MAXEFC) gains[lane] = 0.5 * d_own * d_own * aii + d_own * r_own;
      WSYNC();
      double improvement = 0;
#pragma unroll 1
      for (int j = 0; j < n; ++j) improvement -= gains[j];
      if (lane == 0) w.work += n + 1;  // one sweep over n rows
      if (improvement * scale < tol) break;
    }
    if (lane == 0) w.work += 8 * n;    // the per-row set-up (solves, AR) that envs without constraints skip
  }
  if (lane < n) w.force[lane] = f_i;
  WSYNC();
  if (lane < NV) {
    double sum = 0;
    for (int i = 0; i < n; ++i) sum += w.u.J[i][lane] * w.force[i];
    w.passive[lane] = sum;  // qfrc_constraint (the passive forces are already folded into w.smooth)
  }
  WSYNC();
  if (lane == 0) {
    double x[NV];
#pragma unroll
    for (int k = 0; k < NV; ++k) x[k] = w.passive[k];
    const unsigned solve_mask = 1u;
    B2E_SOLVE_M_UNROLLED(x);
#pragma unroll
    for (int k = 0; k < NV; ++k) w.qacc[k] = w.qacc_smooth[k] + x[k];
  }
  WSYNC();
}
#undef LDP
#undef B2E_SOLVE_FENCE
#undef DINV


// mj_integratePos on w.qpos with velocity vel[] (shared), one element per lane
__device__ __forceinline__ void w_integrate_pos(WS& w, const double* vel, double h, int lane) {
  if (lane < 3) w.qpos[lane] += h * vel[lane];
  if (lane == 3) {
    const double wv[3] = {vel[3], vel[4], vel[5]};
    const double ang = norm3(wv);
    if (ang >= MINVAL) {
      const double axis[3] = {wv[0] / ang, wv[1] / ang, wv[2] / ang};
      double dq[4];
      quat_axisangle(dq, axis, ang * h);
      quat_mul(w.qpos + 3, w.qpos + 3, dq);
    }
    quat_normalize(w.qpos + 3);
  }
  if (lane >= 6 && lane < NV) w.qpos[lane + 1] += h * vel[lane];
}

// mj_RungeKutta(4) in two pieces so that the caller owns the loop (and the CTA barrier in it): stage i = set the state of
// evaluation i, run mj_forward, keep its acceleration; finish = Butcher combination, one dof per lane
__device__ void w_rk4_stage(const WModel& wm, WS& w, int lane, int i) {
  const HModel& m = wm.m;
  const double h = m.timestep;
  const double A[3][3] = {{0.5, 0, 0}, {0, 0.5, 0}, {0, 0, 1.0}};
  if (i > 0) {
    if (lane < NV) {
      double dv = 0, da = 0;
      for (int j = 0; j < i; ++j) { dv += A[i - 1][j] * w.Xv[j][lane]; da += A[i - 1][j] * w.F[j][lane]; }
      w.sv[lane] = dv;
      w.sa[lane] = da;
    }
    for (int k = lane; k < NQ; k += 32) w.qpos[k] = w.X0q[k];
    WSYNC();
    w_integrate_pos(w, w.sv, h, lane);
    if (lane < NV) {
      w.qvel[lane] = w.Xv[0][lane] + h * w.sa[lane];
      w.Xv[i][lane] = w.qvel[lane];
    }
    WSYNC();
  }
  w_forward(wm, w, lane);
  if (i == 0) {  // X0 is the state after the first evaluation: mj_kinematics normalises the quaternion inside qpos
    for (int k = lane; k < NQ; k += 32) w.X0q[k] = w.qpos[k];
    if (lane < NV) w.Xv[0][lane] = w.qvel[lane];
  }
  if (lane < NV) w.F[i][lane] = w.qacc[lane];
  WSYNC();
}
__device__ void w_rk4_finish(const WModel& wm, WS& w, int lane) {
  const double h = wm.m.timestep;
  const double Bw[4] = {1.0 / 6, 1.0 / 3, 1.0 / 3, 1.0 / 6};
  if (lane < NV) {
    double dv = 0, da = 0;
    for (int j = 0; j < 4; ++j) { dv += Bw[j] * w.Xv[j][lane]; da += Bw[j] * w.F[j][lane]; }
    w.sv[lane] = dv;
    w.sa[lane] = da;
  }
  for (int k = lane; k < NQ; k += 32) w.qpos[k] = w.X0q[k];
  WSYNC();
  if (lane < NV) w.qvel[lane] = w.Xv[0][lane] + h * w.sa[lane];
  w_integrate_pos(w, w.sv, h, lane);
  if (lane < NV) w.warm[lane] = w.qacc[lane];
  WSYNC();
}

__device__ void w_write_obs(const WS& w, double* __restrict__ obs, int lane) {  // humanoid_v5.py:436-470, coalesced
  for (int o = lane; o < 348; o += 32) {
    double v;
    if (o < 22) v = w.qpos[2 + o];
    else if (o < 45) v = w.qvel[o - 22];
    else if (o < 175) v = (&w.cinert[1][0])[o - 45];
    else if (o < 253) v = (&w.cvel[1][0])[o - 175];
    else if (o < 270) v = w.actuator[6 + (o - 253)];
    else v = (&w.cfrc_ext[1][0])[o - 270];
    obs[o] = v;
  }
}
__device__ void w_info_base(const HumanoidArgs& a, int64_t i, const WS& w) {
  const int64_t n = a.n;
  a.info[0 * n + i] = w.qpos[0];
  a.info[1 * n + i] = w.qpos[1];
  a.info[2 * n + i] = w.ten_length[0];
  a.info[3 * n + i] = w.ten_length[1];
  a.info[4 * n + i] = w.ten_velocity[0];
  a.info[5 * n + i] = w.ten_velocity[1];
  a.info[6 * n + i] = sqrt(w.qpos[0] * w.qpos[0] + w.qpos[1] * w.qpos[1]);
}
__device__ void w_mass_center(const HModel& m, const WS& w, double* xy) {
  double nx = 0, ny = 0, den = 0;
  for (int b = 0; b < NB; ++b) { nx += m.body_mass[b] * w.xipos[b][0]; ny += m.body_mass[b] * w.xipos[b][1]; den += m.body_mass[b]; }
  xy[0] = nx / den; xy[1] = ny / den;
}
__device__ void w_store_state(const HModel& m, const HumanoidArgs& a, int64_t i, const WS& w, int lane) {
  const int64_t n = a.n;
  for (int k = lane; k < NQ; k += 32) a.qpos[k * n + i] = w.qpos[k];
  if (lane < NV) { a.qvel[lane * n + i] = w.qvel[lane]; a.warm[lane * n + i] = w.warm[lane]; }
  if (lane == 0) {
    double xy[2];
    w_mass_center(m, w, xy);
    a.com_xy[i] = xy[0];
    a.com_xy[n + i] = xy[1];
    if (w.overflow) *a.overflow = 1;
  }
}
// MujocoEnv.reset + reset_model for this warp's env; the RNG stream is advanced by lane 0 only
__device__ void w_env_reset(const WModel& wm, const HumanoidArgs& a, int64_t i, WS& w, int lane, double* __restrict__ obs) {
  const HModel& m = wm.m;
  if (lane == 0) {
    HDraws D;
    D.numpy = a.rng_mode == B2E_RNG_NUMPY;
    if (D.numpy) D.g = pcg64_load(a.rng, a.n, i);
    D.seed = a.philox_seed; D.env = (uint64_t)(a.env_offset + i); D.counter = a.call_counter; D.k = 0;
    const double c = a.noise;
    for (int k = 0; k < NQ; ++k) w.qpos[k] = m.qpos0[k] + (-c + (c - -c) * D.next());
    for (int k = 0; k < NV; ++k) w.qvel[k] = 0.0 + (-c + (c - -c) * D.next());
    if (D.numpy) pcg64_store_state(a.rng, i, D.g);
  }
  if (lane < NV) w.warm[lane] = 0;
  if (lane < NU) w.ctrl[lane] = 0;
  for (int e = lane; e < NB * 6; e += 32) (&w.cfrc_ext[0][0])[e] = 0;
  WSYNC();
  w_forward(wm, w, lane);
  w_write_obs(w, obs, lane);
  if (lane == 0) {
    for (int k = 7; k < 13; ++k) a.info[k * a.n + i] = 0.0;
    w_info_base(a, i, w);
  }
}

__global__ void __launch_bounds__(32) humanoid_reset_warp_kernel(const HumanoidArgs a) {
  __shared__ WS w;
  const int64_t i = blockIdx.x;
  const int lane = threadIdx.x;
  if (a.mask != nullptr && a.mask[i] == 0) return;
  if (lane == 0) { w.overflow = 0; w.work = 0; }
  WSYNC();
  w_env_reset(g_wmodel, a, i, w, lane, a.obs + 348 * i);
  WSYNC();
  w_store_state(g_wmodel.m, a, i, w, lane);
  if (lane == 0) {
    a.ctrl[i] = 0;
    if (a.work) a.work[i] = 0;
  }
}

// W envs per CTA, one warp each (the warps never exchange data; sharing a CTA only co-schedules them).  The warps also meet
// at a CTA barrier before every mj_forward evaluation, so they walk the ~165 KB of code together and share instruction-cache
// lines (barriers between the stages of mj_forward as well were measured: no further gain; a barrier once per mj_step or
// none at all was slower, DESIGN.md section 4).  The barrier is ONE instruction inside a loop that every warp of the CTA
// runs to the end -- warps without an env and warps whose env only resets in this call skip the work, never the barrier.
template <typename ActT, int W>
__global__ void __launch_bounds__(32 * W) humanoid_step_warp_kernel(const HumanoidArgs a) {
  extern __shared__ __align__(16) unsigned char w_smem[];
  const WModel& wm = *reinterpret_cast<const WModel*>(w_smem);  // per-CTA copy of the model and index tables
  const HModel& m = wm.m;
  for (int e = threadIdx.x; e < (int)(sizeof(WModel) / 16); e += 32 * W)
    reinterpret_cast<uint4*>(w_smem)[e] = reinterpret_cast<const uint4*>(&g_wmodel)[e];
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t slot = (int64_t)blockIdx.x * W + warp, n = a.n;
  const bool live = slot < n;
  const int64_t i = !live ? 0 : a.order ? a.order[slot] : slot;  // envs of similar cost share a CTA (they wait for each other)
  WS& w = reinterpret_cast<WS*>(w_smem + sizeof(WModel))[warp];
  const int32_t c = live ? a.ctrl[i] : 0;
  double* __restrict__ obs = a.obs + 348 * i;
  if (lane == 0) { w.overflow = 0; w.work = 0; }
  WSYNC();
  bool reset = live && a.mode == B2E_AUTORESET_NEXT_STEP && ctrl_pending(c);  // this call is the env's reset step
  const bool stepping = live && !reset;
  int32_t cn = 0;
  if (reset && lane == 0) {
    a.reward[i] = 0.0;
    a.term[i] = 0;
    a.trunc[i] = 0;
  }
  if (stepping) {
    for (int k = lane; k < NQ; k += 32) w.qpos[k] = a.qpos[k * n + i];
    if (lane < NV) { w.qvel[lane] = a.qvel[lane * n + i]; w.warm[lane] = a.warm[lane * n + i]; }
    if (lane < NU) w.ctrl[lane] = (double)reinterpret_cast<const ActT*>(a.actions)[i * NU + lane];
    WSYNC();
  }
#pragma unroll 1
  for (int k = 0; k < a.frame_skip; ++k) {  // mj_step x frame_skip (mujoco_env.py:150)
#pragma unroll 1
    for (int st = 0; st < 4; ++st) {
      __syncthreads();
      if (stepping) w_rk4_stage(wm, w, lane, st);
    }
    if (stepping) w_rk4_finish(wm, w, lane);
  }
  if (stepping) {
    if (lane == 0) {  // mj_rnePostConstraint (cfrc_ext only): a short sequential tail
      for (int b = 0; b < NB; ++b) for (int k = 0; k < 6; ++k) w.cfrc_ext[b][k] = 0;
      for (int cc = 0; cc < w.ncon; ++cc) {
        const Contact& con = w.con[cc];
        if (con.efc_adr < 0) continue;
        double lf[3] = {0, 0, 0};
        const double* f = w.force + con.efc_adr;
        if (con.dim == 1) lf[0] = f[0];
        else { lf[0] = f[0] + f[1] + f[2] + f[3]; lf[1] = (f[0] - f[1]) * con.mu; lf[2] = (f[2] - f[3]) * con.mu; }
        double wf[3];
        for (int k = 0; k < 3; ++k) wf[k] = con.frame[k] * lf[0] + con.frame[3 + k] * lf[1] + con.frame[6 + k] * lf[2];
        const int b1 = m.geom_body[con.g1], b2 = m.geom_body[con.g2];
        for (int side = 0; side < 2; ++side) {
          const int b = side ? b2 : b1;
          const double sgn = side ? 1.0 : -1.0;
          const double* com = w.subtree[b == 0 ? 0 : 1];
          const double r[3] = {con.pos[0] - com[0], con.pos[1] - com[1], con.pos[2] - com[2]};
          double tq[3];
          cross3(tq, r, wf);
          for (int k = 0; k < 3; ++k) { w.cfrc_ext[b][k] += sgn * tq[k]; w.cfrc_ext[b][3 + k] += sgn * wf[k]; }
        }
      }
    }
    WSYNC();
    w_write_obs(w, obs, lane);
    bool term = false, trunc = false;
    if (lane == 0) {  // reward, info, TimeLimit (humanoid_v5.py:472-532)
      double after[2];
      w_mass_center(m, w, after);
      const double dt = m.timestep * a.frame_skip;
      const double xv = (after[0] - a.com_xy[i]) / dt, yv = (after[1] - a.com_xy[n + i]) / dt;
      double ctrl_sq = 0;
      for (int u = 0; u < NU; ++u) ctrl_sq += w.ctrl[u] * w.ctrl[u];
      const bool healthy = a.z_min < w.qpos[2] && w.qpos[2] < a.z_max;
      const double forward_reward = a.w_forward * xv, healthy_reward = healthy ? a.healthy_reward : 0.0;
      double cf = 0;
      for (int b = 0; b < NB; ++b) for (int k = 0; k < 6; ++k) cf += w.cfrc_ext[b][k] * w.cfrc_ext[b][k];
      const double ctrl_cost = a.w_ctrl * ctrl_sq;
      double contact_cost = a.w_contact * cf;
      if (contact_cost > a.contact_max) contact_cost = a.contact_max;
      const double reward = (forward_reward + healthy_reward) - (ctrl_cost + contact_cost);
      term = !healthy && a.terminate_when_unhealthy;
      w_info_base(a, i, w);
      a.info[7 * n + i] = xv;
      a.info[8 * n + i] = yv;
      a.info[9 * n + i] = healthy_reward;
      a.info[10 * n + i] = forward_reward;
      a.info[11 * n + i] = -ctrl_cost;
      a.info[12 * n + i] = -contact_cost;
      const int32_t elapsed = ctrl_elapsed(c) + 1;
      trunc = a.max_steps > 0 && elapsed >= a.max_steps;
      a.reward[i] = reward;
      a.term[i] = term;
      a.trunc[i] = trunc;
      cn = elapsed;
      if ((term || trunc) && a.mode == B2E_AUTORESET_NEXT_STEP) cn |= kPending;
    }
    const bool done = __shfl_sync(0xffffffffu, (int)(term || trunc), 0) != 0;
    if (done && a.mode == B2E_AUTORESET_SAME_STEP) {
      for (int o = lane; o < 348; o += 32) a.final_obs[348 * i + o] = obs[o];
      reset = true;
      cn = 0;
    }
    WSYNC();
  }
  if (!live) return;
  if (reset) {  // one call site for both autoreset flavours
    w_env_reset(wm, a, i, w, lane, obs);
    WSYNC();
  }
  w_store_state(m, a, i, w, lane);
  if (lane == 0) {
    a.ctrl[i] = cn;
    if (a.work) a.work[i] = ctrl_pending(cn) ? -1 : w.work;  // -1: the next call only resets this env
  }
}

// Scheduling helper for the step kernel: order[] = env indices bucketed by the solver work of their last
// step, heaviest first (envs that only reset go last); see group_envs_by_key.
__global__ void __launch_bounds__(1024) humanoid_group_kernel(const int32_t* __restrict__ work, int32_t* __restrict__ order,
                                                              int64_t n) {
  group_envs_by_key<256>([work](int64_t i) { const int32_t wk = work[i]; return wk < 0 ? 255 : 254 - min(wk >> 6, 254); },
                         order, n);
}
