// ag_bathing.cuh — fused BedBathingEnv step (reference envs/bed_bathing.py:12-111 + envs/env.py:174-274):
// action -> PD targets -> frame_skip substeps -> obs[24] / reward / done, with the wiping-target bookkeeping
// of get_total_force (bed_bathing.py:41-78) as a per-env bit-free mask over the target points.
#pragma once
#include "ag_device.cuh"
#include "ag_feeding.cuh"
#include "../../include/agphys.h"

struct BathDev {
  AgBathingParams P;
  int *male, *iteration, *task_success, *total_targets;
  float* action;                  // [7][N]
  float* targets;                 // [T][3][N] world positions (the person is static after reset)
  int* alive;                     // [T][N] 1 = not wiped yet (0 for padding beyond the env's target count)
  float* dist_part;               // [human collider slot][N] partial minima of the tool-person distance
  int n_slots;                    // max colliders of a person
};

// action -> PD targets (env.py:187-217)
AG_HDN inline void bathing_pre_body(int e, const SimDev& S, const KP& p) {
  const BathDev& B = *(const BathDev*)p.p1;
  take_step(e, S, (const float*)p.p0, B.iteration, B.action, B.P.arm_links, B.P.arm_lower, B.P.arm_upper, B.P.action_multiplier, B.P.frame_skip);
}

// thread = (collider slot of the person, env): distance from that collider to the nearest wiper collider,
// cut off at 5 m (`tool.get_closest_points(human, distance=5.0)`, bed_bathing.py:23)
AG_HDN inline void bathing_dist_body(int tid, const SimDev& S, const KP& p) {
  const int N = S.N;
  const BathDev& B = *(const BathDev*)p.p1;
  int e = tid % N, slot = tid / N;
  bool male = B.male[e] != 0;
  int c0 = male ? B.P.human_col0_m : B.P.human_col0_f, nc = male ? B.P.human_ncol_m : B.P.human_ncol_f;
  float best = 5.0f;
  if (slot < nc) {
    int ch = c0 + slot;
    int lt = AG_LDG(S.body_link0 + B.P.tool_body), nlt = AG_LDG(S.body_nlinks + B.P.tool_body);
    for (int l = lt; l < lt + nlt; l++) {
      int t0 = AG_LDG(S.link_col0 + l), tn = AG_LDG(S.link_ncol + l);
      for (int ct = t0; ct < t0 + tn; ct++) {
        NpOut out[4];
        int ca = ct < ch ? ct : ch, cb = ct < ch ? ch : ct;
        if (narrow_pair(S, e, ca, cb, 5.0f, false, out)) best = fminf(best, out[0].d);
      }
    }
  }
  B.dist_part[(size_t)slot * N + e] = best;
}

// obs / reward / done.  p0 = action, p1 = BathDev*, p2 = obs [N][24], p3 = reward, p4 = done, p5 = info [N][4]
AG_HDN inline void bathing_post_body(int e, const SimDev& S, const KP& p) {
  const int N = S.N;
  const BathDev& B = *(const BathDev*)p.p1;
  const AgBathingParams& P = B.P;
  bool male = B.male[e] != 0;
  int hb = male ? P.human_body_m : P.human_body_f;
  int lr = AG_LDG(S.body_link0 + P.robot_body);
  // robot base pose = its inertial frame, as p.getBasePositionAndOrientation reports it (agent.py:49,58-63)
  q4 rq = ld4(S.lquat, lr, N, e);
  f3 rp = ld3(S.lpos, lr, N, e) + qrot(rq, tv3(S.link_com, lr));
  rq = qmul(rq, tv4(S.link_iquat, lr));
  q4 rqi = qconj(rq);
  // tool link 1 (the cloth) link-frame pose in the robot frame (bed_bathing.py:81-82)
  f3 tp = ld3(S.lpos, P.cloth_link, N, e); q4 tq = ld4(S.lquat, P.cloth_link, N, e);
  f3 tp_r = qrot(rqi, tp - rp); q4 tq_r = qmul(rqi, tq);
  float* obs = (float*)p.p2 + (size_t)e * 24;
  obs[0] = tp_r.x; obs[1] = tp_r.y; obs[2] = tp_r.z; obs[3] = tq_r.x; obs[4] = tq_r.y; obs[5] = tq_r.z; obs[6] = tq_r.w;
  const float PI = 3.14159265358979323846f;
  for (int j = 0; j < 7; j++) {
    float q = ld1(S.jq, P.arm_links[j], N, e) + PI;
    obs[7 + j] = q - 2.f * PI * floorf(q / (2.f * PI)) - PI;
  }
  for (int j = 0; j < 3; j++) {      // shoulder, elbow, wrist link positions in the robot frame
    int k = male ? P.arm_points_m[j] : P.arm_points_f[j];
    f3 q = qrot(rqi, ld3(S.lpos, k, N, e) - rp);
    obs[14 + 3 * j] = q.x; obs[15 + 3 * j] = q.y; obs[16 + 3 * j] = q.z;
  }
  // forces and wiped targets (bed_bathing.py:41-78)
  float tool_force = 0.f, tool_on_human = 0.f, total_on_human = 0.f;
  int new_pts = 0;
  int cnt = S.c_count[e]; if (cnt > S.maxc) cnt = S.maxc;
  const int T = P.n_targets_max;
  for (int s = 0; s < cnt; s++) {
    unsigned pk = S.s_key[(size_t)s * N + e] >> 2;
    int ca = (int)(pk / (unsigned)S.nc), cb = (int)(pk % (unsigned)S.nc);
    int la = AG_LDG(S.col_link + ca), lb = AG_LDG(S.col_link + cb);
    int ba = AG_LDG(S.link_body + la), bb = AG_LDG(S.link_body + lb);
    float force = cf_ld(S.s_data, s, CF_LAM_N, N, e) / S.dt;
    if (ba == P.tool_body || bb == P.tool_body) tool_force += force;
    bool a_h = ba == hb, b_h = bb == hb;
    if (!a_h && !b_h) continue;
    int other = a_h ? bb : ba, lo = a_h ? lb : la;
    if (other == P.robot_body) total_on_human += force;
    else if (other == P.tool_body) {
      total_on_human += force;
      if (lo != P.cloth_link) continue;
      tool_on_human += force;
      f3 ph = a_h ? f3(cf_ld(S.s_data, s, CF_PAX, N, e), cf_ld(S.s_data, s, CF_PAY, N, e), cf_ld(S.s_data, s, CF_PAZ, N, e))
                  : f3(cf_ld(S.s_data, s, CF_PBX, N, e), cf_ld(S.s_data, s, CF_PBY, N, e), cf_ld(S.s_data, s, CF_PBZ, N, e));
      for (int t = 0; t < T; t++) {
        if (!B.alive[(size_t)t * N + e]) continue;
        f3 tw = ld3(B.targets, t, N, e);
        if (norm(ph - tw) < 0.025f) { B.alive[(size_t)t * N + e] = 0; new_pts++; }
      }
    }
  }
  obs[23] = tool_force;
  int success = B.task_success[e] + new_pts;
  B.task_success[e] = success;
  float dmin = 5.0f;
  for (int i = 0; i < B.n_slots; i++) dmin = fminf(dmin, B.dist_part[(size_t)i * N + e]);
  f3 eecom = ld3(S.lpos, P.ee_link, N, e) + qrot(ld4(S.lquat, P.ee_link, N, e), tv3(S.link_com, P.ee_link));
  f3 lin, ang; link_velocity(S, e, P.ee_link, eecom, lin, ang);
  // human preferences (env.py:237-274), task == 'bed_bathing'
  float pref = P.c_v * (-norm(lin)) + P.c_f * (-(total_on_human - tool_on_human)) + P.c_hf * (tool_on_human < 10.f ? 0.f : -tool_on_human);
  float an = 0.f;
  for (int j = 0; j < 7; j++) { float a = B.action[(size_t)j * N + e]; an += a * a; }
  ((float*)p.p3)[e] = P.w_distance * (-dmin) + P.w_action * (-sqrtf(an)) + P.w_wiping * (float)new_pts + pref;
  ((float*)p.p4)[e] = B.iteration[e] >= 200 ? 1.f : 0.f;
  float* info = (float*)p.p5 + (size_t)e * 4;
  info[0] = total_on_human; info[1] = ((float)success >= (float)B.total_targets[e] * P.task_success_threshold) ? 1.f : 0.f;
  info[2] = tool_on_human; info[3] = (float)new_pts;
}
