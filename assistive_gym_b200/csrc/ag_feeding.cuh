// ag_feeding.cuh — read-back kernels (K6a-d of SURVEY.md §8(a)) and the fused FeedingEnv logic.
//
// Reference semantics restated here:
//   gather/linkstate    p.getJointStates / p.getLinkState / p.getBasePositionAndOrientation (agents/agent.py:40,49,52,72)
//   contact_query       p.getContactPoints (agents/agent.py:100-116)
//   closest             p.getClosestPoints (agents/agent.py:118-130)
//   feeding_pre         AssistiveEnv.take_step action -> PD targets (envs/env.py:174-222)
//   feeding_food/post   FeedingEnv._get_obs / get_food_rewards / reward assembly (envs/feeding.py:12-112),
//                       AssistiveEnv.human_preferences (envs/env.py:237-274)
#pragma once
#include <string.h>
#include "ag_device.cuh"
#include "../../include/agphys.h"

struct FeedDev {
  AgFeedingParams P;
  int *male, *food_state, *iteration, *task_success, *food_near;
  float* action;
  unsigned long long* rng;
  int* tremor_on; float *tremor_rest, *tremor_amp;     // [N], [4][N], [4][N]
};

// ---- env-major host layout <-> SoA.  thread = (column j, env e), env fastest
AG_HDN inline void gather_body(int tid, const SimDev& S, const KP& p) {
  const int N = S.N;
  int e = tid % N, j = tid / N;
  int comp = p.i0, K = p.i0 * p.i1;
  int item = ((const int*)p.p2)[j / comp], c = j % comp;
  ((float*)p.p1)[(size_t)e * K + j] = ((const float*)p.p0)[((size_t)item * comp + c) * N + e];
}
AG_HDN inline void scatter_body(int tid, const SimDev& S, const KP& p) {
  const int N = S.N;
  int e = tid % N, j = tid / N;
  if (p.p3 && !((const int*)p.p3)[e]) return;
  int comp = p.i0, K = p.i0 * p.i1;
  int item = ((const int*)p.p2)[j / comp], c = j % comp;
  ((float*)p.p1)[((size_t)item * comp + c) * N + e] = ((const float*)p.p0)[(size_t)e * K + j];
}

// spatial velocity of a link's COM (world): linear velocity of the COM, angular velocity
AG_HDN inline void link_velocity(const SimDev& S, int e, int k, f3 com, f3& lin, f3& ang) {
  const int N = S.N;
  int b = AG_LDG(S.link_body + k);
  int kind = AG_LDG(S.body_kind + b);
  lin = f3(); ang = f3();
  if (kind == BK_FREE) { lin = ld3(S.base_lin, b, N, e); ang = ld3(S.base_ang, b, N, e); return; }
  if (kind != BK_ART) return;
  int d = AG_LDG(S.link_dl + k);
  while (d >= 0) {
    int kj = AG_LDG(S.dl_link + d);
    f3 a = qrot(ld4(S.lquat, kj, N, e), tv3(S.link_axis, kj));
    float qd = ld1(S.jqd, kj, N, e);
    if (AG_LDG(S.dl_type + d) == 1) { ang += a * qd; lin += cross(a, com - ld3(S.lpos, kj, N, e)) * qd; }
    else lin += a * qd;
    d = AG_LDG(S.dl_parent + d);
  }
}

AG_HDN inline void linkstate_body(int tid, const SimDev& S, const KP& p) {
  const int N = S.N;
  int e = tid % N, j = tid / N, n = p.i1;
  int k = ((const int*)p.p2)[j];
  float* o = (float*)p.p1 + ((size_t)e * n + j) * 20;
  f3 pos = ld3(S.lpos, k, N, e); q4 q = ld4(S.lquat, k, N, e);
  f3 com = pos + qrot(q, tv3(S.link_com, k));
  q4 cq = qmul(q, tv4(S.link_iquat, k));
  f3 lin, ang; link_velocity(S, e, k, com, lin, ang);
  o[0] = pos.x; o[1] = pos.y; o[2] = pos.z; o[3] = q.x; o[4] = q.y; o[5] = q.z; o[6] = q.w;
  o[7] = com.x; o[8] = com.y; o[9] = com.z; o[10] = cq.x; o[11] = cq.y; o[12] = cq.z; o[13] = cq.w;
  o[14] = lin.x; o[15] = lin.y; o[16] = lin.z; o[17] = ang.x; o[18] = ang.y; o[19] = ang.z;
}

AG_HD float i2f(int v) { float f; memcpy(&f, &v, 4); return f; }

AG_HD void write_contact(float* o, int la, int lb, f3 pa, f3 pb, f3 n, float d, float f) {
  o[0] = i2f(la); o[1] = i2f(lb);
  o[2] = pa.x; o[3] = pa.y; o[4] = pa.z; o[5] = pb.x; o[6] = pb.y; o[7] = pb.z; o[8] = n.x; o[9] = n.y; o[10] = n.z;
  o[11] = d; o[12] = f;
}

// does link k belong to (body, link filter)?  lf = -2 any, else a global link id
AG_HD bool link_matches(const SimDev& S, int k, int body, int lf) {
  if (AG_LDG(S.link_body + k) != body) return false;
  return lf == -2 || lf == k;
}

// one lane per env.  i0 = bodyA, i1 = bodyB (-2 any), i2 / i3 = link filters, f0 = max_pts,
// p1 = out records [N][max_pts][13], p2 = counts, p3 = force sums
AG_HDN inline void contact_query_body(int e, const SimDev& S, const KP& p) {
  const int N = S.N;
  int max_pts = (int)p.f0;
  int cnt = S.c_count[e]; if (cnt > S.maxc) cnt = S.maxc;
  int n = 0; float fsum = 0.f;
  for (int s = 0; s < cnt; s++) {
    unsigned pk = S.s_key[(size_t)s * N + e] >> 2;
    int ca = (int)(pk / (unsigned)S.nc), cb = (int)(pk % (unsigned)S.nc);
    int ka = AG_LDG(S.col_link + ca), kb = AG_LDG(S.col_link + cb);
    bool fwd = link_matches(S, ka, p.i0, p.i2) && (p.i1 < 0 || link_matches(S, kb, p.i1, p.i3));
    bool rev = link_matches(S, kb, p.i0, p.i2) && (p.i1 < 0 || link_matches(S, ka, p.i1, p.i3));
    if (!fwd && !rev) continue;
    float force = cf_ld(S.s_data, s, CF_LAM_N, N, e) / S.dt;
    fsum += force;
    if (n < max_pts) {
      f3 pa(cf_ld(S.s_data, s, CF_PAX, N, e), cf_ld(S.s_data, s, CF_PAY, N, e), cf_ld(S.s_data, s, CF_PAZ, N, e));
      f3 pb(cf_ld(S.s_data, s, CF_PBX, N, e), cf_ld(S.s_data, s, CF_PBY, N, e), cf_ld(S.s_data, s, CF_PBZ, N, e));
      f3 nn(cf_ld(S.s_data, s, CF_NX, N, e), cf_ld(S.s_data, s, CF_NY, N, e), cf_ld(S.s_data, s, CF_NZ, N, e));
      float* o = (float*)p.p1 + ((size_t)e * max_pts + n) * 13;
      if (fwd) write_contact(o, ka, kb, pa, pb, nn, cf_ld(S.s_data, s, CF_DIST, N, e), force);
      else write_contact(o, kb, ka, pb, pa, -nn, cf_ld(S.s_data, s, CF_DIST, N, e), force);
    }
    n++;
  }
  ((int*)p.p2)[e] = n;
  if (p.p3) ((float*)p.p3)[e] = fsum;
}

// one lane per env.  i0 = bodyA, i1 = bodyB, i2 = max_pts, f0 = distance
AG_HDN inline void closest_body(int e, const SimDev& S, const KP& p) {
  const int N = S.N;
  int ba = p.i0, bb = p.i1, max_pts = p.i2; float dist = p.f0;
  int a0 = AG_LDG(S.body_link0 + ba), an = AG_LDG(S.body_nlinks + ba), b0 = AG_LDG(S.body_link0 + bb), bn = AG_LDG(S.body_nlinks + bb);
  int n = 0;
  if (S.body_mode[(size_t)ba * N + e] == 0 || S.body_mode[(size_t)bb * N + e] == 0) { ((int*)p.p2)[e] = 0; return; }
  for (int la = a0; la < a0 + an; la++) {
    int nca = AG_LDG(S.link_ncol + la); if (!nca) continue;
    f3 lamin = ld3(S.lmin, la, N, e), lamax = ld3(S.lmax, la, N, e);
    for (int lb = b0; lb < b0 + bn; lb++) {
      int ncb = AG_LDG(S.link_ncol + lb); if (!ncb) continue;
      if (!aabb_ov(lamin, lamax, ld3(S.lmin, lb, N, e), ld3(S.lmax, lb, N, e), dist)) continue;
      int ca0 = AG_LDG(S.link_col0 + la), cb0 = AG_LDG(S.link_col0 + lb);
      for (int ca = ca0; ca < ca0 + nca; ca++) {
        f3 amin = ld3(S.cmin, ca, N, e), amax = ld3(S.cmax, ca, N, e);
        for (int cb = cb0; cb < cb0 + ncb; cb++) {
          if (!aabb_ov(amin, amax, ld3(S.cmin, cb, N, e), ld3(S.cmax, cb, N, e), dist)) continue;
          NpOut out[4];
          if (!narrow_pair(S, e, ca, cb, dist, false, out)) continue;
          if (n < max_pts) write_contact((float*)p.p1 + ((size_t)e * max_pts + n) * 13, la, lb, out[0].pa, out[0].pb, out[0].n, out[0].d, 0.f);
          n++;
        }
      }
    }
  }
  ((int*)p.p2)[e] = n;
}

// ------------------------------------------------------------------ fused FeedingEnv
// action -> PD targets.  p0 = action [N][7] (env-major), p1 = FeedDev*
AG_HDN inline void feeding_pre_body(int e, const SimDev& S, const KP& p) {
  const FeedDev& F = *(const FeedDev*)p.p1;
  take_step(e, S, (const float*)p.p0, F.iteration, F.action, F.P.arm_links, F.P.arm_lower, F.P.arm_upper, F.P.action_multiplier, F.P.frame_skip);
  // tremor: the head joints
  if (F.tremor_on[e])
    tremor_step(e, S, 4, F.male[e] ? F.P.head_joints_m : F.P.head_joints_f, F.iteration[e], F.tremor_rest, F.tremor_amp);
}

// thread = (food i, env e): is any spoon collider within 0.1 of the food sphere? (feeding.py:71)
AG_HDN inline void feeding_food_body(int tid, const SimDev& S, const KP& p) {
  const int N = S.N;
  const FeedDev& F = *(const FeedDev*)p.p1;
  int e = tid % N, i = tid / N;
  int near = 0;
  if ((F.food_state[e] >> i) & 1) {
    int fb = F.P.food_body0 + i, tb = F.P.tool_body;
    int lf = AG_LDG(S.body_link0 + fb), lt = AG_LDG(S.body_link0 + tb);
    int cf = AG_LDG(S.link_col0 + lf);
    f3 fmin = ld3(S.cmin, cf, N, e), fmax = ld3(S.cmax, cf, N, e);
    const float dist = 0.1f;
    if (aabb_ov(fmin, fmax, ld3(S.lmin, lt, N, e), ld3(S.lmax, lt, N, e), dist)) {
      int c0 = AG_LDG(S.link_col0 + lt), ncl = AG_LDG(S.link_ncol + lt);
      for (int c = c0; c < c0 + ncl && !near; c++) {
        if (!aabb_ov(fmin, fmax, ld3(S.cmin, c, N, e), ld3(S.cmax, c, N, e), dist)) continue;
        NpOut out[4];
        if (narrow_pair(S, e, cf, c, dist, false, out)) near = 1;
      }
    }
  }
  F.food_near[(size_t)i * N + e] = near;
}

AG_HD unsigned long long xorshift64s(unsigned long long& s) {
  s ^= s >> 12; s ^= s << 25; s ^= s >> 27;
  return s * 2685821657736338717ull;
}
AG_HD float rng_uniform(unsigned long long& s) { return (float)(xorshift64s(s) >> 40) * (1.0f / 16777216.0f); }

// obs / reward / done.  p0 = action, p1 = FeedDev*, p2 = obs [N][25], p3 = reward, p4 = done, p5 = info [N][4]
AG_HDN inline void feeding_post_body(int e, const SimDev& S, const KP& p) {
  const int N = S.N;
  const FeedDev& F = *(const FeedDev*)p.p1;
  const AgFeedingParams& P = F.P;
  bool male = F.male[e] != 0;
  int hb = male ? P.human_body_m : P.human_body_f;
  int head = male ? P.head_link_m : P.head_link_f;
  // poses
  int lr = AG_LDG(S.body_link0 + P.robot_body), ltool = AG_LDG(S.body_link0 + P.tool_body);
  // robot base pose = its inertial frame, as p.getBasePositionAndOrientation reports it (agent.py:49,58-63)
  q4 rq = ld4(S.lquat, lr, N, e);
  f3 rp = ld3(S.lpos, lr, N, e) + qrot(rq, tv3(S.link_com, lr));
  rq = qmul(rq, tv4(S.link_iquat, lr));
  q4 rqi = qconj(rq);
  f3 sp = ld3(S.lpos, ltool, N, e) + qrot(ld4(S.lquat, ltool, N, e), tv3(S.link_com, ltool));
  q4 sq = qmul(ld4(S.lquat, ltool, N, e), tv4(S.link_iquat, ltool));
  f3 hp = ld3(S.lpos, head, N, e); q4 hq = ld4(S.lquat, head, N, e);
  f3 mouth = male ? f3(P.mouth_m[0], P.mouth_m[1], P.mouth_m[2]) : f3(P.mouth_f[0], P.mouth_f[1], P.mouth_f[2]);
  f3 target = hp + qrot(hq, mouth);
  f3 sp_r = qrot(rqi, sp - rp); q4 sq_r = qmul(rqi, sq);
  f3 hp_r = qrot(rqi, hp - rp); q4 hq_r = qmul(rqi, hq);
  f3 tg_r = qrot(rqi, target - rp);
  // contact forces on the human from the robot and from the spoon; food-human contacts
  float robot_force = 0.f, spoon_force = 0.f;
  int food_hit_mask = 0;
  int cnt = S.c_count[e]; if (cnt > S.maxc) cnt = S.maxc;
  for (int s = 0; s < cnt; s++) {
    unsigned pk = S.s_key[(size_t)s * N + e] >> 2;
    int ca = (int)(pk / (unsigned)S.nc), cb = (int)(pk % (unsigned)S.nc);
    int ba = AG_LDG(S.link_body + AG_LDG(S.col_link + ca)), bb = AG_LDG(S.link_body + AG_LDG(S.col_link + cb));
    int other = -1;
    if (ba == hb) other = bb; else if (bb == hb) other = ba;
    if (other < 0) continue;
    float force = cf_ld(S.s_data, s, CF_LAM_N, N, e) / S.dt;
    if (other == P.robot_body) robot_force += force;
    else if (other == P.tool_body) spoon_force += force;
    else if (other >= P.food_body0 && other < P.food_body0 + P.n_foods) food_hit_mask |= 1 << (other - P.food_body0);
  }
  float total_force = robot_force + spoon_force;
  float* obs = (float*)p.p2 + (size_t)e * 25;
  obs[0] = sp_r.x; obs[1] = sp_r.y; obs[2] = sp_r.z; obs[3] = sq_r.x; obs[4] = sq_r.y; obs[5] = sq_r.z; obs[6] = sq_r.w;
  obs[7] = sp_r.x - tg_r.x; obs[8] = sp_r.y - tg_r.y; obs[9] = sp_r.z - tg_r.z;
  const float PI = 3.14159265358979323846f;
  for (int j = 0; j < 7; j++) {
    float q = ld1(S.jq, P.arm_links[j], N, e) + PI;
    q = q - 2.f * PI * floorf(q / (2.f * PI)) - PI;
    obs[10 + j] = q;
  }
  obs[17] = hp_r.x; obs[18] = hp_r.y; obs[19] = hp_r.z; obs[20] = hq_r.x; obs[21] = hq_r.y; obs[22] = hq_r.z; obs[23] = hq_r.w;
  obs[24] = spoon_force;
  // food bookkeeping (feeding.py:50-83)
  int st = F.food_state[e];
  int foods = st & 0xffff, active = (st >> 16) & 0xffff;
  float food_reward = 0.f, vel_sum = 0.f, food_hit = 0.f;
  int success = F.task_success[e];
  unsigned long long rs = F.rng[e];
  int active_at_entry = active;
  for (int i = 0; i < P.n_foods; i++) {
    if (!((foods >> i) & 1)) continue;
    int fb = P.food_body0 + i;
    int lf = AG_LDG(S.body_link0 + fb);
    f3 fp = ld3(S.lpos, lf, N, e);
    if (norm(target - fp) < 0.03f) {
      food_reward += 20.f; success += 1;
      vel_sum += norm(ld3(S.base_lin, fb, N, e));
      foods &= ~(1 << i); active &= ~(1 << i);
      f3 far(1000.f + 1000.f * rng_uniform(rs), 1000.f + 1000.f * rng_uniform(rs), 1000.f + 1000.f * rng_uniform(rs));
      st3(S.base_pos, fb, N, e, far); st4(S.base_quat, fb, N, e, q4());
      st3(S.lpos, lf, N, e, far); st4(S.lquat, lf, N, e, q4());
    } else if (!F.food_near[(size_t)i * N + e]) {
      food_reward -= 5.f; foods &= ~(1 << i);
    }
  }
  for (int i = 0; i < P.n_foods; i++) {
    if (!((active_at_entry >> i) & 1)) continue;
    if ((food_hit_mask >> i) & 1) { food_hit -= 1.f; active &= ~(1 << i); }
  }
  F.food_state[e] = foods | (active << 16);
  F.task_success[e] = success;
  F.rng[e] = rs;
  // end-effector velocity (COM of the ee link)
  f3 eecom = ld3(S.lpos, P.ee_link, N, e) + qrot(ld4(S.lquat, P.ee_link, N, e), tv3(S.link_com, P.ee_link));
  f3 lin, ang; link_velocity(S, e, P.ee_link, eecom, lin, ang);
  float ee_vel = norm(lin);
  // human preferences (env.py:237-274), task == 'feeding'
  float r_vel = -ee_vel;
  float r_high = spoon_force < 10.f ? 0.f : -spoon_force;
  float r_nontarget = -total_force;
  float pref = P.c_v * r_vel + P.c_f * r_nontarget + P.c_hf * r_high + P.c_fd * food_hit + P.c_fdv * (-vel_sum);
  float an = 0.f;
  for (int j = 0; j < 7; j++) { float a = F.action[(size_t)j * N + e]; an += a * a; }
  float reward = P.w_distance * (-norm(target - sp)) + P.w_action * (-sqrtf(an)) + P.w_food * food_reward + pref;
  ((float*)p.p3)[e] = reward;
  ((float*)p.p4)[e] = F.iteration[e] >= 200 ? 1.f : 0.f;
  float* info = (float*)p.p5 + (size_t)e * 4;
  info[0] = total_force; info[1] = ((float)success >= P.n_foods * P.task_success_threshold) ? 1.f : 0.f;
  info[2] = robot_force; info[3] = spoon_force;
}
