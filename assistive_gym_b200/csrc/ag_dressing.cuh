// ag_dressing.cuh — fused DressingEnv step (reference envs/dressing.py:12-106 + envs/env.py:174-274 + envs/util.py:125-202):
// action -> PD targets -> frame_skip x (numSubSteps rigid substeps + one cloth launch + anchor follows the end effector)
// -> sleeve-on-arm reward, cloth forces on the person, obs[24] / reward / done.
#pragma once
#include "ag_device.cuh"
#include "ag_feeding.cuh"
#include "ag_cloth.cuh"
#include "../../include/agphys.h"

struct DressDev {
  AgDressingParams P;
  int *male, *iteration;
  float* task_success;            // [N] best reward_dressing so far (dressing.py:66-67)
  float* action;                  // [7][N]
  int* tremor_on;                 // [N] the person's impairment is 'tremor' (human.py:80-92)
  float *tremor_rest, *tremor_amp; // [10][N] target_joint_angles of the left arm joints and the tremor amplitudes
};

// action -> PD targets of the robot's 7 arm joints (env.py:187-217)
AG_HDN inline void dressing_pre_body(int e, const SimDev& S, const KP& p) {
  const DressDev& D = *(const DressDev*)p.p1;
  take_step(e, S, (const float*)p.p0, D.iteration, D.action, D.P.arm_links, D.P.arm_lower, D.P.arm_upper, D.P.action_multiplier, D.P.frame_skip);
  // a tremor human is an agent (env.py:130): its arm targets flip sign around the rest pose every env step
  if (D.tremor_on[e])
    tremor_step(e, S, 10, D.male[e] ? D.P.human_arm_m : D.P.human_arm_f, D.iteration[e], D.tremor_rest, D.tremor_amp);
}

AG_HD float dress_sign(float v) { return v > 0.f ? 1.f : (v < 0.f ? -1.f : 0.f); }
AG_HD float dress_signed_volume(f3 a, f3 b, f3 c, f3 d) { return (1.0f / 6.0f) * dot(cross(b - a, c - a), d - a); }
// util.py:125-132
AG_HD bool dress_line_hits_triangle(f3 p0, f3 p1, f3 p2, f3 q0, f3 q1) {
  if (dress_sign(dress_signed_volume(q0, p0, p1, p2)) != dress_sign(dress_signed_volume(q1, p0, p1, p2))) {
    float a = dress_sign(dress_signed_volume(q0, q1, p0, p1)), b = dress_sign(dress_signed_volume(q0, q1, p1, p2)), c = dress_sign(dress_signed_volume(q0, q1, p2, p0));
    if (a == b && b == c) return true;
  }
  return false;
}
// "points above and below both planes through the limb axis" (util.py:147-163, 165-172)
AG_HD bool dress_points_around(const f3* pts, f3 normal, f3 origin) {
  f3 t = cross(f3(1.f, 1.f, 0.f), normal); t = t * (1.f / norm(t));
  f3 b = cross(t, normal); b = b * (1.f / norm(b));
  bool ta = false, tb = false, ba = false, bb = false;
  for (int i = 0; i < 6; i++) {
    float dt = dot(t, pts[i] - origin), db = dot(b, pts[i] - origin);
    ta |= dt > 0.f; tb |= dt < 0.f; ba |= db > 0.f; bb |= db < 0.f;
  }
  return ta && tb && ba && bb;
}

// obs / reward / done.  p0 = action, p1 = DressPost* (the fused step's state + the cloth it reads), p2 = obs [N][24],
// p3 = reward, p4 = done, p5 = info [N][4] = total force on the person, task success, reward_dressing, sleeve state
// (1: forearm in the sleeve, 2: upper arm, 3: both)
struct DressPost { DressDev D; const ClothDev* C; };
AG_HDN inline void dressing_post_body(int e, const SimDev& S, const KP& p) {
  const int N = S.N;
  const DressPost& DP = *(const DressPost*)p.p1;
  const DressDev& D = DP.D;
  const ClothDev& C = *DP.C;
  const AgDressingParams& P = D.P;
  bool male = D.male[e] != 0;
  int hb = male ? P.human_body_m : P.human_body_f;
  int lr = AG_LDG(S.body_link0 + P.robot_body);
  q4 rq = ld4(S.lquat, lr, N, e);
  f3 rp = ld3(S.lpos, lr, N, e) + qrot(rq, tv3(S.link_com, lr));
  rq = qmul(rq, tv4(S.link_iquat, lr));
  q4 rqi = qconj(rq);
  f3 eep = ld3(S.lpos, P.ee_link, N, e); q4 eeq = ld4(S.lquat, P.ee_link, N, e);
  f3 ep_r = qrot(rqi, eep - rp); q4 eq_r = qmul(rqi, eeq);
  float* obs = (float*)p.p2 + (size_t)e * 24;
  obs[0] = ep_r.x; obs[1] = ep_r.y; obs[2] = ep_r.z; obs[3] = eq_r.x; obs[4] = eq_r.y; obs[5] = eq_r.z; obs[6] = eq_r.w;
  const float PI = 3.14159265358979323846f;
  for (int j = 0; j < 7; j++) {
    float q = ld1(S.jq, P.arm_links[j], N, e) + PI;
    obs[7 + j] = q - 2.f * PI * floorf(q / (2.f * PI)) - PI;
  }
  f3 limb[3];                        // shoulder, elbow, wrist link positions (dressing.py:20-22)
  for (int j = 0; j < 3; j++) {
    limb[j] = ld3(S.lpos, male ? P.arm_points_m[j] : P.arm_points_f[j], N, e);
    f3 q = qrot(rqi, limb[j] - rp);
    obs[14 + 3 * j] = q.x; obs[15 + 3 * j] = q.y; obs[16 + 3 * j] = q.z;
  }
  // ---- sleeve_on_arm_reward (util.py:134-202)
  f3 pts[6];
  const size_t xb = (size_t)e * 3 * C.nnp;
  for (int i = 0; i < 6; i++) { int n = i < 3 ? P.tri1[i] : P.tri2[i - 3]; pts[i] = f3(C.x[xb + n], C.x[xb + C.nnp + n], C.x[xb + 2 * (size_t)C.nnp + n]); }
  float hand_r = male ? P.hand_radius_m : P.hand_radius_f, elbow_r = male ? P.elbow_radius_m : P.elbow_radius_f, shoulder_r = male ? P.shoulder_radius_m : P.shoulder_radius_f;
  f3 sh = limb[0], el = limb[1], wr = limb[2];
  float lwe = norm(wr - el);
  f3 hand_end = wr + (wr - el) * (1.f / lwe) * (hand_r * 2.f);
  f3 elbow_end = el + (el - wr) * (1.f / lwe) * elbow_r;
  f3 shoulder_end = sh + (sh - el) * (1.f / norm(sh - el)) * shoulder_r;
  f3 nf = hand_end - elbow_end; nf = nf * (1.f / norm(nf));
  f3 nu = elbow_end - shoulder_end; nu = nu * (1.f / norm(nu));
  bool around_f = dress_points_around(pts, nf, hand_end), around_u = dress_points_around(pts, nu, shoulder_end);
  bool f_hit = dress_line_hits_triangle(pts[0], pts[1], pts[2], hand_end, elbow_end) || dress_line_hits_triangle(pts[3], pts[4], pts[5], hand_end, elbow_end);
  bool u_hit = dress_line_hits_triangle(pts[0], pts[1], pts[2], elbow_end, shoulder_end) || dress_line_hits_triangle(pts[3], pts[4], pts[5], elbow_end, shoulder_end);
  f3 centre(0.f, 0.f, 0.f);
  for (int i = 0; i < 6; i++) centre += pts[i];
  centre = centre * (1.f / 6.f);
  float distance_to_hand = norm(hand_end - centre);
  float distance_along_forearm = norm(centre - hand_end), distance_along_upperarm = norm(centre - el);
  float forearm_length = norm(hand_end - elbow_end), upperarm_length = norm(el - sh);
  bool forearm_in = around_f && f_hit, upperarm_in = around_u && u_hit;
  float reward_dressing;
  if (upperarm_in) { reward_dressing = forearm_length; if (distance_along_upperarm < upperarm_length) reward_dressing += distance_along_upperarm; }
  else if (forearm_in && distance_along_forearm < forearm_length) reward_dressing = distance_along_forearm;
  else reward_dressing = -distance_to_hand;
  // ---- cloth forces on the person (dressing.py:35-45): x10, contacts below the end effector, each below 20 N
  float cloth_sum = 0.f;
  int cnt = C.cc_count[e];
  for (int s = 0; s < cnt; s++) {
    const float* r = C.cc_data + ((size_t)e * C.maxcc + s) * AG_CLOTH_CCF;
    f3 f = f3(r[4], r[5], r[6]) * 10.f;
    float fn = norm(f);
    if (r[3] < eep.z - 0.05f && fn < 20.f) cloth_sum += fn;
  }
  obs[23] = cloth_sum;
  // ---- robot on person (dressing.py:91)
  float robot_on_human = 0.f;
  int rc = S.c_count[e]; if (rc > S.maxc) rc = S.maxc;
  for (int s = 0; s < rc; s++) {
    unsigned pk = S.s_key[(size_t)s * N + e] >> 2;
    int ca = (int)(pk / (unsigned)S.nc), cb = (int)(pk % (unsigned)S.nc);
    int ba = AG_LDG(S.link_body + AG_LDG(S.col_link + ca)), bb = AG_LDG(S.link_body + AG_LDG(S.col_link + cb));
    if ((ba == P.robot_body && bb == hb) || (bb == P.robot_body && ba == hb)) robot_on_human += cf_ld(S.s_data, s, CF_LAM_N, N, e) / S.dt;
  }
  f3 eecom = eep + qrot(eeq, tv3(S.link_com, P.ee_link));
  f3 lin, ang; link_velocity(S, e, P.ee_link, eecom, lin, ang);
  float pref = P.c_v * (-norm(lin)) + P.c_d * (-cloth_sum);          // env.py:237-274 with the dressing arguments
  float an = 0.f;
  for (int j = 0; j < 7; j++) { float a = D.action[(size_t)j * N + e]; an += a * a; }
  ((float*)p.p3)[e] = P.w_dressing * reward_dressing + P.w_action * (-sqrtf(an)) + pref;
  float best = D.task_success[e];
  if (reward_dressing > best) { best = reward_dressing; D.task_success[e] = best; }
  ((float*)p.p4)[e] = D.iteration[e] >= 200 ? 1.f : 0.f;
  float* info = (float*)p.p5 + (size_t)e * 4;
  info[0] = robot_on_human + cloth_sum; info[1] = best >= P.task_success_threshold ? 1.f : 0.f; info[2] = reward_dressing;
  info[3] = (forearm_in ? 1.f : 0.f) + (upperarm_in ? 2.f : 0.f);
}
