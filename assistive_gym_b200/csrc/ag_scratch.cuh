// ag_scratch.cuh — fused ScratchItchEnv step (reference envs/scratch_itch.py:10-91 + envs/env.py:174-274): action -> PD targets ->
// frame_skip substeps -> obs[30] / reward / done, with the scratch bookkeeping of get_total_force (scratch_itch.py:46-58) and
// the "moved more than 1 cm along the target" reward (scratch_itch.py:26-30).  SURVEY.md section 8(f)3.
#pragma once
#include "ag_device.cuh"
#include "ag_feeding.cuh"
#include "../../include/agphys.h"

struct ScratchDev {
  AgScratchParams P;
  int *male, *iteration, *task_success;
  int* limb_link;                 // [N] global link id of the limb that carries the target (upper arm or forearm)
  float* target_local;            // [3][N] target point in that link's frame (util.point_on_capsule)
  float* prev_contact;            // [3][N] prev_target_contact_pos
  float* action;                  // [7][N]
};

AG_HDN inline void scratch_pre_body(int e, const SimDev& S, const KP& p) {
  const ScratchDev& D = *(const ScratchDev*)p.p1;
  take_step(e, S, (const float*)p.p0, D.iteration, D.action, D.P.arm_links, D.P.arm_lower, D.P.arm_upper, D.P.action_multiplier, D.P.frame_skip);
}

// p0 = action, p1 = ScratchDev*, p2 = obs [N][30], p3 = reward, p4 = done, p5 = info [N][4] = total force on the person, task
// success, tool force at the target, scratches so far
AG_HDN inline void scratch_post_body(int e, const SimDev& S, const KP& p) {
  const int N = S.N;
  const ScratchDev& D = *(const ScratchDev*)p.p1;
  const AgScratchParams& P = D.P;
  bool male = D.male[e] != 0;
  int hb = male ? P.human_body_m : P.human_body_f;
  int lr = AG_LDG(S.body_link0 + P.robot_body);
  q4 rq = ld4(S.lquat, lr, N, e);
  f3 rp = ld3(S.lpos, lr, N, e) + qrot(rq, tv3(S.link_com, lr));
  rq = qmul(rq, tv4(S.link_iquat, lr));
  q4 rqi = qconj(rq);
  f3 tp = ld3(S.lpos, P.tool_tip_link, N, e); q4 tq = ld4(S.lquat, P.tool_tip_link, N, e);
  int limb = D.limb_link[e];
  f3 target = ld3(S.lpos, limb, N, e) + qrot(ld4(S.lquat, limb, N, e), ld3(D.target_local, 0, N, e));     // update_targets (scratch_itch.py:149-153)
  f3 tp_r = qrot(rqi, tp - rp), tg_r = qrot(rqi, target - rp); q4 tq_r = qmul(rqi, tq);
  float* obs = (float*)p.p2 + (size_t)e * 30;
  obs[0] = tp_r.x; obs[1] = tp_r.y; obs[2] = tp_r.z; obs[3] = tq_r.x; obs[4] = tq_r.y; obs[5] = tq_r.z; obs[6] = tq_r.w;
  obs[7] = tp_r.x - tg_r.x; obs[8] = tp_r.y - tg_r.y; obs[9] = tp_r.z - tg_r.z; obs[10] = tg_r.x; obs[11] = tg_r.y; obs[12] = tg_r.z;
  const float PI = 3.14159265358979323846f;
  for (int j = 0; j < 7; j++) {
    float q = ld1(S.jq, P.arm_links[j], N, e) + PI;
    obs[13 + j] = q - 2.f * PI * floorf(q / (2.f * PI)) - PI;
  }
  for (int j = 0; j < 3; j++) {
    int k = male ? P.arm_points_m[j] : P.arm_points_f[j];
    f3 q = qrot(rqi, ld3(S.lpos, k, N, e) - rp);
    obs[20 + 3 * j] = q.x; obs[21 + 3 * j] = q.y; obs[22 + 3 * j] = q.z;
  }
  // forces (scratch_itch.py:46-58)
  float tool_force = 0.f, at_target = 0.f, total_on_human = 0.f;
  f3 contact_pos(0.f, 0.f, 0.f); bool have_contact = false;
  int cnt = S.c_count[e]; if (cnt > S.maxc) cnt = S.maxc;
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
      f3 ph = a_h ? f3(cf_ld(S.s_data, s, CF_PAX, N, e), cf_ld(S.s_data, s, CF_PAY, N, e), cf_ld(S.s_data, s, CF_PAZ, N, e))
                  : f3(cf_ld(S.s_data, s, CF_PBX, N, e), cf_ld(S.s_data, s, CF_PBY, N, e), cf_ld(S.s_data, s, CF_PBZ, N, e));
      if ((lo == P.tool_link0 || lo == P.tool_tip_link) && norm(ph - target) < 0.025f) { at_target += force; contact_pos = ph; have_contact = true; }
    }
  }
  obs[29] = tool_force;
  float scratch = 0.f;
  int success = D.task_success[e];
  if (have_contact && norm(contact_pos - ld3(D.prev_contact, 0, N, e)) > 0.01f && at_target < 10.f) {
    scratch = 5.f; st3(D.prev_contact, 0, N, e, contact_pos); success += 1;
  }
  D.task_success[e] = success;
  f3 eecom = ld3(S.lpos, P.ee_link, N, e) + qrot(ld4(S.lquat, P.ee_link, N, e), tv3(S.link_com, P.ee_link));
  f3 lin, ang; link_velocity(S, e, P.ee_link, eecom, lin, ang);
  float pref = P.c_v * (-norm(lin)) + P.c_f * (-(total_on_human - at_target)) + P.c_hf * (at_target < 10.f ? 0.f : -at_target);
  float an = 0.f;
  for (int j = 0; j < 7; j++) { float a = D.action[(size_t)j * N + e]; an += a * a; }
  ((float*)p.p3)[e] = P.w_distance * (-norm(target - tp)) + P.w_action * (-sqrtf(an)) + P.w_scratch * scratch + pref;
  ((float*)p.p4)[e] = D.iteration[e] >= 200 ? 1.f : 0.f;
  float* info = (float*)p.p5 + (size_t)e * 4;
  info[0] = total_on_human; info[1] = (float)success >= P.task_success_threshold ? 1.f : 0.f; info[2] = at_target; info[3] = (float)success;
}
