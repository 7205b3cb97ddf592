/* agphys.h — C ABI of the B200-native batched physics step for Assistive Gym.
 *
 * Drop-in boundary: the reference drives its physics through ~60 `pybullet` C-extension calls
 * (SURVEY.md §8(b)); every entry point below cites the reference call site(s) it replaces
 * (paths relative to /root/reference/assistive_gym/envs).  The host-side mirror
 * (`assistive_gym_b200/capi.py` + `assistive_gym_b200/sim.py`) binds these with ctypes; INTEGRATION.md shows the stub a
 * maintainer of the reference would add.
 *
 * Conventions
 *   - `extern "C"`, plain pointers and sizes only.  Return 0 on success, <0 on error;
 *     `ag_last_error()` gives the message.  No exceptions cross the ABI.
 *   - A simulation holds N lock-step copies ("envs") of one immutable scene template.
 *   - Batched buffers are env-major: element (env e, item i, component c) of a [N][K][C] buffer is
 *     at ((e*K)+i)*C + c.  `*_host` calls take host pointers and include the H2D/D2H copies;
 *     `*_dev` calls take device pointers valid on the simulation's device and enqueue on the
 *     simulation's stream.
 *   - Quaternions are [x,y,z,w] (reference agents/agent.py:60, env.py:192).
 *   - Link index == joint index == DFS pre-order over the URDF tree, base = -1 (reference
 *     agents/jaco.py:8-18).  In this ABI links are addressed by *global link id* (int) obtained from
 *     the scene description: `body_link0[body] + 1 + pybullet_link_index` (base: +0).
 */
#ifndef AGPHYS_H
#define AGPHYS_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* joint types (per link: the joint that connects it to its parent) */
enum { AG_JOINT_FIXED = 0, AG_JOINT_REVOLUTE = 1, AG_JOINT_PRISMATIC = 2,
       AG_JOINT_FREE_BASE = 3, AG_JOINT_FIXED_BASE = 4 };
/* collider core types: every convex collider is a vertex set ("core") swept by a sphere of
 * `col_radius` (sphere = 1 vertex, capsule = 2, box/hull = n); HALFSPACE is the ground plane. */
enum { AG_COL_SPHERE = 0, AG_COL_CAPSULE = 1, AG_COL_HULL = 2, AG_COL_HALFSPACE = 3 };
/* motor modes (reference agents/agent.py:33 POSITION_CONTROL, agents/human.py:119 VELOCITY_CONTROL) */
enum { AG_MOTOR_OFF = 0, AG_MOTOR_POSITION = 1, AG_MOTOR_VELOCITY = 2 };

/* Solver / world parameters.  Defaults restate PyBullet's (SURVEY.md Appendix A — recalled, not
 * verifiable in this container; every recalled constant is a field).  Replaces
 * p.setTimeStep / p.setGravity / p.setPhysicsEngineParameter (env.py:104-107, dressing.py:184). */
typedef struct AgConfig {
  double dt;                 /* 0.02   env.py:21,104 */
  int    num_substeps;       /* 1      Bullet numSubSteps=0 -> 1 (dressing.py:184 uses 8) */
  int    num_solver_iters;   /* 50     Bullet numSolverIterations */
  double erp;                /* 0.2    non-contact constraint ERP */
  double contact_erp;        /* 0.08   PyBullet erp2 */
  double linear_slop;        /* 1e-5 */
  double residual_threshold; /* 1e-7   leastSquaresResidualThreshold (squared impulses); <=0 disables early exit */
  double contact_threshold;  /* 0.02   contact breaking threshold FACTOR: points with distance <= factor * min(col_thresh_a, col_thresh_b) are contacts */
  double linear_damping;     /* 0.04   btMultiBody default */
  double angular_damping;    /* 0.04 */
  double max_coord_velocity; /* 100 */
  double hull_margin;        /* 0.001  collision margin of mesh/box hull colliders (already baked into col_radius by the builder; informational) */
  int    cone_friction;      /* 1      implicit cone over the 2 friction directions; 0 = pyramid */
  int    gyroscopic;         /* 1      include w x Iw for free bodies */
  int    max_contacts;       /* per-env contact budget for the solver (default 128); overflow is flagged */
  double warmstart_contact;  /* 0      (Bullet m_warmstartingFactor = 0.85, but its multibody solver of the reference's era does not warm start): a contact that persists (same collider pair, same manifold
                                       point index) starts the solve from factor * its last normal impulse; 0 disables */
  double warmstart_joint;    /* 0      the same for joint-limit, motor and fixed-constraint rows (Bullet's multibody solver of
                                       the reference's era starts these from zero) */
} AgConfig;

/* Immutable scene template (host arrays, copied by ag_create).  Built on the host by the
 * `pybullet`-shaped builder calls the reference issues at reset time (loadURDF jaco.py:53,
 * createMultiBody human_creation.py:280 / tool.py:34 / env.py:371-380, createConstraint tool.py:46,
 * setCollisionFilterPair tool.py:44, changeDynamics human.py:110, setGravity(body=) agent.py:197). */
typedef struct AgSceneDesc {
  int n_bodies, n_links, n_colliders, n_verts, n_planes, n_pairs, n_constraints;
  /* bodies [n_bodies] */
  const int32_t* body_link0;    /* global id of the base link; links of a body are contiguous, DFS order */
  const int32_t* body_nlinks;   /* number of links including the base */
  const double*  body_gravity;  /* [n_bodies][3] per-body gravity (fork feature, agent.py:196-197) */
  /* links [n_links] */
  const int32_t* link_body;
  const int32_t* link_parent;   /* global id of parent link, -1 for a base */
  const int32_t* link_jtype;    /* AG_JOINT_* */
  const double*  link_axis;     /* [n_links][3] joint axis in the link frame */
  const double*  link_jpos;     /* [n_links][3] joint frame origin in the parent link frame */
  const double*  link_jquat;    /* [n_links][4] joint frame orientation in the parent link frame */
  const double*  link_com;      /* [n_links][3] centre of mass in the link frame */
  const double*  link_iquat;    /* [n_links][4] inertial (principal) frame orientation in the link frame */
  const double*  link_inertia;  /* [n_links][3] principal moments */
  const double*  link_mass;     /* [n_links]   0 => static/locked ("static joints" trick, human.py:108-112) */
  const double*  link_lower;    /* [n_links] joint limits; limit rows exist iff link_haslimit */
  const double*  link_upper;
  const int32_t* link_haslimit;
  const double*  link_damping;  /* [n_links] joint damping */
  const double*  link_friction; /* [n_links] lateral friction coefficient */
  /* colliders [n_colliders]; vertices/planes are expressed in the owning link's frame */
  const int32_t* col_link;
  const int32_t* col_type;      /* AG_COL_* */
  const double*  col_radius;    /* sphere/capsule radius, hull margin */
  const double*  col_thresh;    /* Bullet's getAngularMotionDisc() of the shape; pair contact threshold =
                                   AgConfig.contact_threshold * min(thresh_a, thresh_b) */
  const int32_t* col_v0;        /* first core vertex */
  const int32_t* col_nv;        /* number of core vertices (<= 64) */
  const int32_t* col_p0;        /* first face plane (hulls), for the penetration fallback */
  const int32_t* col_np;
  const double*  col_center;    /* [n_colliders][3] local AABB centre of the core (link frame) */
  const double*  col_half;      /* [n_colliders][3] local AABB half extents of the core */
  const double*  verts;         /* [n_verts][3] */
  const double*  planes;        /* [n_planes][4] (n, d): n.x <= d inside */
  /* enabled collision pairs between links (global ids), after self-collision flags, parent-child
   * exclusion and setCollisionFilterPair overrides; at least one side movable. */
  const int32_t* pair_link;     /* [n_pairs][2] */
  /* fixed user constraints (p.createConstraint JOINT_FIXED, tool.py:46-47) */
  const int32_t* con_link;      /* [n_constraints][2] global ids (parent link, child link) */
  const double*  con_pivot;     /* [n_constraints][2][3] pivot in each link's frame */
  const double*  con_quat;      /* [n_constraints][2][4] constraint frame in each link's frame */
  const double*  con_maxforce;  /* [n_constraints] */
} AgSceneDesc;

/* One contact point as returned by p.getContactPoints (agent.py:108-115: fields 3,4,5,6,9 used;
 * distance [8] and normal [7] also filled). */
typedef struct AgContact {
  int32_t link_a, link_b;       /* global link ids */
  float   pos_a[3], pos_b[3];   /* world, on the surfaces */
  float   normal[3];            /* on B, pointing towards A */
  float   distance;
  float   normal_force;         /* accumulated normal impulse / dt of the last substep */
} AgContact;

typedef struct AgSim AgSim;     /* opaque */

const char* ag_last_error(void);
void        ag_default_config(AgConfig* cfg);

/* --- lifetime: p.connect / p.resetSimulation / p.disconnect (env.py:34,92-97) ----------------- */
AgSim* ag_create(const AgSceneDesc* scene, const AgConfig* cfg, int n_envs, int device);
void   ag_destroy(AgSim* sim);
int    ag_num_envs(const AgSim* sim);
void*  ag_stream(AgSim* sim);   /* cudaStream_t the sim enqueues on */

/* --- state setters (host buffers, env-major). p.resetBasePositionAndOrientation (agent.py:149),
 * p.resetBaseVelocity (agent.py:152), p.resetJointState (agent.py:156,248,250).
 * `env_mask` (int32[N], may be NULL = all) selects the envs written.  Base pose is the pose of the
 * base LINK frame. */
int ag_set_base_pose(AgSim* sim, int body, const float* pos, const float* quat, const int32_t* env_mask);
int ag_set_base_velocity(AgSim* sim, int body, const float* lin, const float* ang, const int32_t* env_mask);
int ag_set_joint_state(AgSim* sim, int n, const int32_t* links, const float* q, const float* qd, const int32_t* env_mask);
/* per-env lateral friction of one link (env.py:120 randomises the plane's) */
int ag_set_link_friction(AgSim* sim, int link, const float* mu, const int32_t* env_mask);
/* per-env mode of a body: 0 = inactive (neither moves nor collides; the other-gender human,
 * human.py:76-77), 1 = active, 2 = frozen (collides as a static body; a non-tremor human) */
int ag_set_body_active(AgSim* sim, int body, const int32_t* active);
/* Human.enforce_joint_limits (agent.py:240-250, called every substep for a human in `agents`,
 * env.py:229): hard clamp of q to the joint limits with qd := 0, applied after integration. */
int ag_set_hard_limits(AgSim* sim, int n, const int32_t* links, int on);
/* p.setGravity(..., body=) of the fork (agent.py:196-197): gravity felt by one body, the same in every env */
int ag_set_body_gravity(AgSim* sim, int body, const double g[3]);
/* p.getAABB per link (agent.py:132-143 get_heights): world AABB of each link's colliders, [N][n][3] each; links without
 * colliders report an empty box (min > max) */
int ag_get_link_aabb(AgSim* sim, int n, const int32_t* links, float* aabb_min, float* aabb_max);
/* recompute link world poses from the state (after teleports); also done by ag_step */
int ag_forward_kinematics(AgSim* sim);

/* --- motors: p.setJointMotorControlArray(POSITION_CONTROL) (agent.py:33, robot.py:77) and
 * p.setJointMotorControl2(VELOCITY_CONTROL, force=0) (human.py:119).  target is [N][n]
 * (host or device per the suffix); kp/kd/max_force are per joint, shared by all envs. */
int ag_set_motor_host(AgSim* sim, int n, const int32_t* links, int mode, const float* target,
                      const float* kp, const float* kd, const float* max_force);
int ag_set_motor_targets_dev(AgSim* sim, int n, const int32_t* links, const float* target_dev);
int ag_set_motor_targets_host(AgSim* sim, int n, const int32_t* links, const float* target);
/* per-env scale [N][n] of the joints' max_force (Human.strength, human.py:86,126: `forces = reactive_force * strength`) */
int ag_set_motor_force_scale(AgSim* sim, int n, const int32_t* links, const float* scale);

/* --- the hot path: p.stepSimulation (env.py:226; feeding.py:179) ----------------------------- */
int ag_step(AgSim* sim, int n_steps);

/* --- read-back: p.getJointStates (agent.py:40,85), p.getLinkState (agent.py:52,54,72),
 * p.getBasePositionAndOrientation / getBaseVelocity (agent.py:49,71) ------------------------- */
int ag_get_joint_states(AgSim* sim, int n, const int32_t* links, float* q, float* qd, float* applied_torque);
/* world pose of link frames ([N][n][3], [N][n][4]) and, optionally, COM pose and COM linear /
 * angular velocity (NULL to skip). */
int ag_get_link_states(AgSim* sim, int n, const int32_t* links, float* pos, float* quat,
                       float* com_pos, float* com_quat, float* lin_vel, float* ang_vel);
/* p.getContactPoints(bodyA[,bodyB,linkA,linkB]) (agent.py:100-116): body_b/link_a/link_b = -2 for
 * "any" (link -1 is the base).  Writes up to max_pts contacts per env into out[N][max_pts] and the
 * number found into count[N].  A is always the queried body (contacts are flipped as needed). */
int ag_get_contacts(AgSim* sim, int body_a, int body_b, int link_a, int link_b, int max_pts,
                    AgContact* out, int32_t* count);
/* sum of normal forces between two bodies, per env ([N]); feeding.py:45-48 */
int ag_contact_force_sum(AgSim* sim, int body_a, int body_b, int link_a, int link_b, float* out);
/* p.getClosestPoints(bodyA, bodyB, distance) (agent.py:118-130; feeding.py:71): per env the
 * closest pair over all collider pairs of the two bodies within `distance`, independent of
 * collision filters.  count[N] = number of collider pairs within distance. */
int ag_closest_points(AgSim* sim, int body_a, int body_b, float distance, int max_pts,
                      AgContact* out, int32_t* count);

/* --- fused FeedingEnv path (feeding.py:12-112 + env.py:174-235): action -> PD targets ->
 * frame_skip substeps -> obs[25] / reward / done.  All buffers on the device. ------------------- */
typedef struct AgFeedingParams {
  int32_t robot_body, tool_body, human_body_m, human_body_f;
  int32_t arm_links[7];         /* controllable joints (global link ids) */
  int32_t ee_link;              /* right_end_effector */
  int32_t head_link_m, head_link_f;
  int32_t head_joints_m[4], head_joints_f[4]; /* neck, head x/y/z (global link ids): the tremor DoFs (human.py:89-90) */
  int32_t food_body0, n_foods;
  float   arm_lower[7], arm_upper[7];
  float   mouth_m[3], mouth_f[3];
  float   action_multiplier;    /* 0.05 env.py:188 */
  int32_t frame_skip;           /* 5 */
  float   w_distance, w_action, w_food; /* config.ini [feeding] */
  float   c_v, c_f, c_hf, c_fd, c_fdv;  /* config.ini [human_preferences] */
  float   task_success_threshold;
  uint64_t seed;
} AgFeedingParams;
int ag_feeding_init(AgSim* sim, const AgFeedingParams* p, const int32_t* gender_is_male);
int ag_feeding_reset_episode(AgSim* sim, const int32_t* env_mask);
/* tremor impairment (human.py:80-92, env.py:212-215): per env on/off, head-joint rest angles [N][4]
 * and tremor amplitudes [N][4]; targets flip sign every env step.  NULL `on` switches tremor off. */
int ag_feeding_set_tremor(AgSim* sim, const int32_t* on, const float* rest, const float* amplitude);
int ag_feeding_step_dev(AgSim* sim, const float* action_dev, float* obs_dev, float* reward_dev,
                        float* done_dev, float* info_dev);
/* host-buffer variant (pinned or pageable): H2D of action, D2H of obs/reward/done/info inside.  `info` may be NULL, here,
 * in ag_feeding_step_host_end and in the bathing / dressing / scratch *_step_host alike. */
int ag_feeding_step_host(AgSim* sim, const float* action, float* obs, float* reward, float* done, float* info);
/* the same in two halves, so that several sims (sub-batches on their own streams) overlap: `begin` stages the actions and
 * enqueues H2D + step + D2H on the sim's stream and returns, `end` waits for the stream and hands the results out */
int ag_feeding_step_host_begin(AgSim* sim, const float* action);
int ag_feeding_step_host_end(AgSim* sim, float* obs, float* reward, float* done, float* info);

/* --- fused BedBathingEnv path (bed_bathing.py:12-111 + env.py:174-274): action -> PD targets ->
 * frame_skip substeps -> obs[24] / reward / done; wiping targets are points on the person's right arm
 * (bed_bathing.py:173-203), a target within 0.025 m of a wiper-cloth contact point counts once
 * (bed_bathing.py:41-78).  SURVEY.md §8(a) row B1. ------------------------------------------- */
typedef struct AgBathingParams {
  int32_t robot_body, tool_body, human_body_m, human_body_f;
  int32_t arm_links[7];         /* controllable joints (global link ids) */
  int32_t ee_link;              /* left_end_effector */
  int32_t cloth_link;           /* wiper link 1 (global link id): `if linkA in [1]` */
  int32_t arm_points_m[3], arm_points_f[3];   /* right shoulder, elbow, wrist links (global ids) */
  int32_t human_col0_m, human_ncol_m, human_col0_f, human_ncol_f;   /* collider ranges of the two persons */
  int32_t n_targets_max;        /* padded target count T (129 male / 91 female) */
  float   arm_lower[7], arm_upper[7];
  float   action_multiplier;    /* 0.05 env.py:188 */
  int32_t frame_skip;           /* 5 */
  float   w_distance, w_action, w_wiping;   /* config.ini [bed_bathing] */
  float   c_v, c_f, c_hf;                   /* config.ini [human_preferences] */
  float   task_success_threshold;
} AgBathingParams;
/* targets_world [N][T][3], targets_valid [N][T] (host); the person must already be frozen in place */
int ag_bathing_init(AgSim* sim, const AgBathingParams* p, const int32_t* gender_is_male, const float* targets_world,
                    const int32_t* targets_valid);
/* obs [N][24], reward [N], done [N], info [N][4] = total force on person, task success, cloth force on person, new targets */
int ag_bathing_step_dev(AgSim* sim, const float* action_dev, float* obs_dev, float* reward_dev, float* done_dev, float* info_dev);
int ag_bathing_step_host(AgSim* sim, const float* action, float* obs, float* reward, float* done, float* info);

/* --- cloth: p.loadCloth / p.clothParams / p.getSoftBodyData (dressing.py:25,146-154), stepped inside ag_step with the
 * world's numSubSteps (dressing.py:184).  SURVEY.md section 8(a) row D1.  The model restates Bullet's btSoftBody position
 * solver (recalled; DESIGN.md section 9): node masses uniform, links = mesh edges, one-way coupling with the rigid links
 * listed in `col_links` (multibody link colliders are static shapes for btSoftBody). ------------------------------- */
typedef struct AgClothDesc {
  int32_t n_nodes, n_links, n_colours, n_nf, n_anchors, n_col_links;
  const int32_t* links;        /* [n_links][2] node ids, colour-major: links of one colour share no node */
  const double*  link_rest2;   /* [n_links] squared rest length (btSoftBody::Link::m_c1) */
  const int32_t* colour_off;   /* [n_colours + 1] */
  const int32_t* nf_off;       /* [n_nodes + 1] node -> adjacent faces ... */
  const int32_t* nf_pair;      /* [n_nf][2] ... as the two other nodes of the face in winding order */
  const double*  node_area;    /* [n_nodes] a third of the adjacent face areas (btSoftBody::updateArea) */
  double inv_mass;             /* of every node: n_nodes / total mass (loadCloth mass=0.16) */
  double kLST, kDP, kDG, kLF, kDF, kCHR, kKHR, kAHR;   /* p.clothParams (dressing.py:147) */
  double margin;               /* collisionMargin (0.04) */
  double air_density;          /* btSoftBodyWorldInfo::air_density (1.2) */
  int32_t piterations;
  double gravity[3];           /* world gravity acting on the cloth */
  const int32_t* anchor_node;  /* [n_anchors] (loadCloth anchors=[...]) */
  const double*  anchor_local; /* [n_anchors][3] node position relative to the anchor body at attachment time */
  const int32_t* col_links;    /* [n_col_links] global link ids whose colliders the cloth collides with */
  const double*  col_link_bsphere; /* [n_col_links][4] bounding sphere (centre, radius) of each link's colliders, link frame */
  const int32_t* col_link_static;  /* [n_col_links] 1: static shape (contact hardness kKHR), 0: movable (kCHR) */
  int32_t max_contacts;        /* per-env rigid-contact budget of one substep (default 1024); overflow is flagged */
} AgClothDesc;
int ag_cloth_init(AgSim* sim, const AgClothDesc* desc);
/* node positions / velocities, host [N][n_nodes][3]; NULL skips; env_mask [N] or NULL */
int ag_cloth_set_state(AgSim* sim, const float* x, const float* v, const int32_t* env_mask);
int ag_cloth_get_state(AgSim* sim, float* x, float* v);
/* position of the (kinematic, identity-orientation) anchor body, host [N][3] (cloth_attachment.set_base_pos_orient, dressing.py:192) */
int ag_cloth_set_anchor(AgSim* sim, const float* pos, const int32_t* env_mask);
/* the same from the current world position of a link, on the device (update_targets, dressing.py:210) */
int ag_cloth_anchor_follow(AgSim* sim, int link);
int ag_cloth_set_gravity(AgSim* sim, const double g[3]);      /* p.setGravity (dressing.py:178,195) as felt by the cloth */
/* rigid contacts of the last substep, as p.getSoftBodyData reports them: count [N]; per contact (host, [N][max_pts]) the
 * node id, its position [3] and the contact force on the node [3] (accumulated position correction / (inv_mass dt^2)) */
int ag_cloth_get_contacts(AgSim* sim, int max_pts, int32_t* count, int32_t* node, float* pos, float* force, int32_t* link);
/* device pointers for fused consumers: x / v are [N][3][n_nodes_padded] */
int ag_cloth_device_state(AgSim* sim, float** x_dev, float** v_dev, int32_t* n_nodes_padded);

/* --- fused DressingEnv path (dressing.py:12-106 + env.py:174-274 + util.py:125-202): action -> PD targets -> frame_skip x
 * (numSubSteps rigid substeps, one cloth launch, the cloth's anchor body follows the end effector) -> sleeve-on-arm reward,
 * cloth forces on the person, obs [24] / reward / done.  Needs ag_cloth_init.  SURVEY.md section 8(a) row D1. ---------- */
typedef struct AgDressingParams {
  int32_t robot_body, human_body_m, human_body_f;
  int32_t arm_links[7];         /* controllable joints (global link ids): PR2 left arm */
  int32_t ee_link;              /* left_end_effector */
  int32_t arm_points_m[3], arm_points_f[3];   /* left shoulder, elbow, wrist links (global ids) */
  int32_t human_arm_m[10], human_arm_f[10];   /* the person's controllable joints (human.left_arm_joints, dressing_envs.py:13) */
  float   arm_lower[7], arm_upper[7];
  float   hand_radius_m, elbow_radius_m, shoulder_radius_m, hand_radius_f, elbow_radius_f, shoulder_radius_f; /* human_creation.py:89,140 */
  int32_t tri1[3], tri2[3];     /* sleeve-opening nodes (dressing.py:149-150), cloth-internal ids */
  float   action_multiplier;    /* 0.05 env.py:188 */
  int32_t frame_skip;           /* 5 */
  float   w_dressing, w_action; /* config.ini [dressing] */
  float   c_v, c_d;             /* config.ini [human_preferences] velocity_weight, dressing_force_weight */
  float   task_success_threshold;
} AgDressingParams;
int ag_dressing_init(AgSim* sim, const AgDressingParams* p, const int32_t* gender_is_male);
int ag_dressing_reset_episode(AgSim* sim, const int32_t* env_mask);
/* tremor impairment of the person (human.py:80-92, env.py:212-215): per env on/off, rest angles [N][10] and amplitudes [N][10] of
 * the left arm joints; targets flip sign every env step.  NULL `on` switches tremor off. */
int ag_dressing_set_tremor(AgSim* sim, const int32_t* on, const float* rest, const float* amplitude);
/* obs [N][24], reward [N], done [N], info [N][4] = total force on the person, task success, reward_dressing, sleeve state */
int ag_dressing_step_dev(AgSim* sim, const float* action_dev, float* obs_dev, float* reward_dev, float* done_dev, float* info_dev);
int ag_dressing_step_host(AgSim* sim, const float* action, float* obs, float* reward, float* done, float* info);

/* --- fused ScratchItchEnv path (scratch_itch.py:10-91 + env.py:174-274): action -> PD targets -> frame_skip substeps ->
 * obs [30] / reward / done; the target is a point on the person's right upper arm or forearm (scratch_itch.py:134-153), a tool
 * contact within 0.025 m of it that has moved by more than 0.01 m counts as a scratch.  SURVEY.md section 8(f)3. ------------- */
typedef struct AgScratchParams {
  int32_t robot_body, tool_body, human_body_m, human_body_f;
  int32_t arm_links[7];         /* controllable joints (global link ids) */
  int32_t ee_link;              /* left_end_effector */
  int32_t tool_link0, tool_tip_link;          /* tool links 0 and 1 (global ids): `if linkA in [0, 1]`, `tool.get_pos_orient(1)` */
  int32_t arm_points_m[3], arm_points_f[3];   /* right shoulder, elbow, wrist links (global ids) */
  float   arm_lower[7], arm_upper[7];
  float   action_multiplier;    /* 0.05 env.py:188 */
  int32_t frame_skip;           /* 5 */
  float   w_distance, w_action, w_scratch;    /* config.ini [scratch_itch] */
  float   c_v, c_f, c_hf;                     /* config.ini [human_preferences] */
  float   task_success_threshold;             /* 25 scratches */
} AgScratchParams;
/* limb_link [N]: global id of the link that carries each env's target; target_local [N][3]: the point in that link's frame */
int ag_scratch_init(AgSim* sim, const AgScratchParams* p, const int32_t* gender_is_male, const int32_t* limb_link, const float* target_local);
/* obs [N][30], reward [N], done [N], info [N][4] = total force on the person, task success, tool force at the target, scratches */
int ag_scratch_step_dev(AgSim* sim, const float* action_dev, float* obs_dev, float* reward_dev, float* done_dev, float* info_dev);
int ag_scratch_step_host(AgSim* sim, const float* action, float* obs, float* reward, float* done, float* info);

/* --- camera images: p.computeViewMatrix / p.computeProjectionMatrixFOV / p.getCameraImage (env.py:342-359; learn.py:101,125).
 * The collision geometry is ray-cast on the device (the visual meshes are not part of the scene description): RGBA8 image and
 * OpenGL-style depth buffer per requested env.  SURVEY.md section 8(f)4. ----------------------------------------------- */
typedef struct AgCamera {
  float eye[3], target[3], up[3];     /* computeViewMatrix(camera_eye, camera_target, [0,0,1]) */
  float fov_deg, aspect, near_, far_; /* computeProjectionMatrixFOV(fov, w / h, 0.01, 100) */
  int32_t width, height;
  float light_dir[3];                 /* getCameraImage lightDirection (env.py:355: [0,-3,1]) */
  float ambient, diffuse;             /* lightAmbientCoeff 0.8, lightDiffuseCoeff 0.3 (env.py:355) */
} AgCamera;
/* rgba: host uint8 [n][height][width][4], depth: host float [n][height][width] (NULL to skip), env_ids [n] */
int ag_render(AgSim* sim, const AgCamera* cam, int n, const int32_t* env_ids, uint8_t* rgba, float* depth);

/* --- batched inverse kinematics for reset (Robot.ik_random_restarts agents/robot.py:84-121 via
 * AssistiveEnv.init_robot_pose envs/env.py:296; SURVEY.md §8(f)1): damped least squares with random restarts inside
 * the joint limits, one env per thread.  `joint_links` [n_joints <= 8]: the solved joints (global link ids, all on the
 * path from the body's base to `ee_link`); other joints on that path keep their current angles.  target_pos [N][3],
 * target_quat [N][4] (link frame of ee_link), env_mask [N] or NULL, q_out [N][n_joints], err_out [N] =
 * max(position error, quaternion distance) of the best restart.  Host buffers; uses the body's current base pose. */
int ag_ik_solve(AgSim* sim, int n_joints, const int32_t* joint_links, int ee_link, const float* target_pos,
                const float* target_quat, int max_restarts, int iters, float threshold, uint64_t seed,
                const int32_t* env_mask, float* q_out, float* err_out);

/* --- checkpoint / parity: full per-env dynamic state as a flat float blob -------------------- */
/* KINEMATIC state only (base pose / velocity of every body, q / qd of every link): what a parity test needs to put two
 * simulations into the same configuration.  Motor targets and modes, body modes, per-env friction, the hard-limit flags
 * and the fused episodes' bookkeeping (food state, iteration, tremor phase) are NOT part of it. */
size_t ag_state_size(const AgSim* sim);           /* floats per env */
int    ag_state_get(AgSim* sim, float* out);      /* [N][state_size] host */
int    ag_state_set(AgSim* sim, const float* in);

/* --- introspection for measurement --------------------------------------------------------- */
uint64_t ag_kernel_launches(const AgSim* sim);    /* kernels launched since creation */
/* per-kernel device time (CUDA events on the sim's stream around every launch while enabled) */
int      ag_profile_enable(AgSim* sim, int on);
int      ag_profile_get(AgSim* sim, int max_names, char* names, int name_stride, float* total_ms, int32_t* counts);
int      ag_overflow_count(AgSim* sim);            /* envs that exceeded the contact / candidate budget in any substep since the
                                                      last call (sticky flags, cleared by this call); surviving contacts are the
                                                      smallest keys (collider pair, point), independent of arrival order */
/* per-env contact count and PGS iterations used in the last substep (host int32[N] buffers, may be NULL) */
int      ag_get_solver_stats(AgSim* sim, int32_t* contacts, int32_t* iters);
/* SM cycles each env's lane spent inside the PGS kernel of the last substep (load-balance diagnostic) */
int      ag_get_pgs_cycles(AgSim* sim, int32_t* cycles);           /* diagnostic: SM cycles each env spent in the last PGS launch */
int      ag_get_pgs_trips(AgSim* sim, int32_t* trips, int32_t* stream_floats);  /* diagnostic: records its warp consumed / floats of its row stream */

#ifdef __cplusplus
}
#endif
#endif /* AGPHYS_H */
