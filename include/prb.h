/* prb.h — C ABI of the B200-native batched playroom simulator (libprb_b200.so).
 *
 * The reference has no FFI/plugin API of its own: its boundary is the Python gym.GoalEnv
 * surface of `playEnv` (roboticsPlayroomPybullet/envs/environments.py:58-314), which talks to
 * PyBullet through ~60 C-API calls per step.  Every entry point below replaces one piece of
 * that surface for a whole batch of environments; the reference lines it stands in for are
 * cited per function.  The Python mirror (roboticsplayroompybullet_b200/envs.py) binds these
 * with ctypes; INTEGRATION.md shows the stub.
 *
 * Conventions: return 0 on success, a negative prb_status on failure (never throws across the
 * ABI); prb_last_error() gives the message.  All `*_dev` pointers are device pointers on the
 * handle's GPU; calls are asynchronous on the given CUDA stream (a cudaStream_t passed as
 * void*; NULL = legacy default stream) and serialised per handle; one handle per GPU/process.
 * No host synchronisation happens inside prb_step / prb_observe / prb_substeps / prb_set_goal; prb_reset
 * synchronises the stream (once per reset round, see below), like the reference's reset() it replaces.
 */
#ifndef PRB_H
#define PRB_H
#include <stdint.h>
#include "prb_model.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct prb_handle prb_handle;

typedef enum prb_status {
  PRB_OK = 0,
  PRB_ERR_INVALID = -1,   /* bad argument / model not representable */
  PRB_ERR_CUDA = -2,      /* CUDA runtime failure (message has the cudaError string) */
  PRB_ERR_NO_DEVICE = -3  /* no CUDA device: there is no CPU fallback */
} prb_status;

typedef struct prb_config {
  int32_t num_envs;     /* environments owned by this handle (this rank's shard) */
  int32_t env_offset;   /* global index of local env 0: RNG streams are keyed by global env id */
  int32_t device;       /* CUDA device ordinal */
  int32_t reserved;
  uint64_t seed;        /* base seed of the counter-based per-env RNG (reset sampling) */
} prb_config;

/* Device buffers owned by the handle.  Each observation key of the reference's calc_state dict
 * (environments.py:849-861) is its own dense [num_envs, dim] fp32 array inside one contiguous
 * allocation `out_base` of `out_floats` floats (so one copy moves a whole step's results).
 * `state` is [num_envs, state_stride] fp32, see DESIGN.md "state layout". */
typedef struct prb_buffers {
  float* state;
  float* out_base;
  float* obs_quat;
  float* achieved_goal;
  float* desired_goal;
  float* controllable_achieved_goal;
  float* full_positional_state;
  float* joints;                   /* [N,8]  environments.py:758 */
  float* velocity;                 /* [N,6]  environments.py:857 */
  float* observation;              /* [N,6|12|18] environments.py:859 (dimension quirk kept) */
  float* gripper_proprioception;   /* [N]    environments.py:720-743 */
  float* reward;                   /* [N]    environments.py:211 */
  float* is_success;               /* [N]    environments.py:213 */
  float* target_poses;             /* [N,n_ik] environments.py:214,1034 */
  int64_t out_floats;
  int32_t num_envs, state_dim, state_stride;
  int32_t obs_dim, goal_dim, fps_dim, observation_dim, n_ik;
} prb_buffers;

/* playEnv.__init__ + activate_physics_client + instance.__init__ (environments.py:64-170,
 * 218-249, 321-454): builds the world for `num_envs` independent environments from a compiled
 * model.  All environments start in the load state (arm at q=0, default joint motors). */
int prb_create(const prb_model* model, const prb_config* cfg, prb_handle** out);
int prb_destroy(prb_handle* h);

/* playEnv.reset() (environments.py:173-187 -> instance.reset :599-603): for every env whose
 * mask byte is non-zero (NULL = all) re-seat objects, settle 100 substeps, reset the arm through
 * one IK call, sample a goal, and repeat while the sampled state already satisfies the goal.
 * Refreshes all output buffers of the reset envs.  Runs as rounds of {seat objects, settle on the masked step
 * pipeline, finish} over the envs still pending and reads one device counter per round (synchronous on `stream`);
 * prb_reset_rounds returns the number of rounds the most recent call needed. */
int prb_reset(prb_handle* h, const uint8_t* mask_dev, void* stream);
int prb_reset_rounds(prb_handle* h);

/* playEnv.reset(o) (environments.py:173-187, 541-556, 582-596): re-seat the masked envs FROM AN OBSERVATION — trajectory
 * replay.  obs_dev is [N, obs_dim] in the obs_quat layout: the object pose is taken from it (no settle steps), the arm
 * goes from its rest pose through one IK call to the observed end-effector pose, a new goal is drawn (again while already
 * satisfied).  Two documented differences from the reference: the object is read at its real offset in the layout (the
 * reference's hard-coded 11 / 10 indexing is wrong for the 19-D play layout), and with restore_env != 0 the drawer, door,
 * button and dial are restored from the observation too (the reference leaves them at their defaults).  Asynchronous. */
int prb_reset_to(prb_handle* h, const float* obs_dev, const uint8_t* mask_dev, int32_t restore_env, void* stream);

/* playEnv.reset_goal_pos(goal) (environments.py:190-191, 492-501): goal_dev is [N, goal_dim]. */
int prb_set_goal(prb_handle* h, const float* goal_dev, const uint8_t* mask_dev, void* stream);

/* playEnv.step(action) (environments.py:206-214): action_dev is [N,A]; A = 7 (8 for the quaternion decoders), the
 * decoder is the model's action_type parameter (environments.py:915-981).  Default [N,7] absolute xyz + rpy +
 * gripper; clip -> IK -> motor targets -> 12 substeps -> calc_state -> reward / is_success. */
int prb_step(prb_handle* h, const float* action_dev, void* stream);

/* instance.calc_state() (environments.py:799-864) without stepping: refresh the output buffers
 * from the current state (used after prb_set_state / prb_set_goal). */
int prb_observe(prb_handle* h, void* stream);

/* Run `n` raw stepSimulation() substeps without touching motors or outputs
 * (environments.py:490,535); used by the parity tests. */
int prb_substeps(prb_handle* h, int32_t n, void* stream);

int prb_get_buffers(prb_handle* h, prb_buffers* out);

/* playEnv.compute_reward / compute_reward_sparse (environments.py:278-304,
 * playRewardFunc.py:66-77), stateless and batched for goal relabelling: ag, dg are [B, goal_dim]. */
int prb_compute_reward(prb_handle* h, const float* ag_dev, const float* dg_dev, int64_t B, float* out_dev, void* stream);

/* Raw simulation state (host copies, synchronous): [N, state_dim] fp32.  The reference has no
 * save/restore (SURVEY.md §5); these exist so tests can start oracle and device from identical
 * states, and double as checkpoint/restore. */
int prb_get_state(prb_handle* h, float* host_out);
int prb_set_state(prb_handle* h, const float* host_in);

/* Same as prb_step, but through HOST buffers: copies action_host [N,A] to the device, steps,
 * copies the whole output block (out_floats floats) back into out_host and synchronises the
 * stream.  This is the call the Python gym mirror makes for numpy in / numpy out stepping.
 * out_host may be pinned (one asynchronous copy) or ordinary pageable memory, e.g. the fresh array a
 * gym step returns: then the block comes back through the handle's pinned staging in chunks that
 * PRB_HOST_THREADS worker threads (default: 8 on hosts with >= 16 cores) copy out while the next chunk
 * is still in flight. */
int prb_step_host(prb_handle* h, const float* action_host, float* out_host, void* stream);

/* Per-kernel device timing for reports: when enabled, prb_step brackets its two kernels with
 * CUDA events on the launching stream; prb_last_kernel_ms synchronises on them and returns the
 * durations of the most recent step's IK kernel and fused substep kernel. */
int prb_enable_kernel_timing(prb_handle* h, int32_t enable);
int prb_last_kernel_ms(prb_handle* h, float* ik_ms, float* step_ms);
/* split of step_ms into the summed durations of the warp-per-env setup launches and the
 * thread-per-env solver launches of the most recent step */
int prb_last_tier_ms(prb_handle* h, float* setup_ms, float* pgs_ms);

/* Camera images of every env (the reference's calc_state 'img', environments.py:841-845, and its gripper camera,
 * :33-49).  Every collider is drawn as the box it is in the compiled model, coloured from col_rgb_host ([n_col,3] in
 * [0,1]: colours are not part of prb_model) and shaded rgb = clamp(colour (ambient + diffuse max(0, n.l)), 0, 1)
 * with n the world normal of the face hit; no shadows.  view / proj are column-major 4x4 matrices in the layout
 * PyBullet's computeViewMatrix* / computeProjectionMatrixFOV return; proj must be a perspective projection
 * (clip w = -z_eye) and view a rigid transform.  Pixel (i, j), row 0 at the top, is the ray through NDC
 * (2(j+0.5)/W-1, 1-2(i+0.5)/H). */
typedef struct prb_camera {
  int32_t width, height;   /* 1..1024 */
  int32_t attach;          /* 0: view maps world to eye; 1: view maps the end-effector site frame to eye (gripper camera) */
  float view[16];
  float proj[16];
  float light_dir[3];      /* towards the light, world frame; normalised by the library */
  float ambient, diffuse;
  float background[3];     /* colour of pixels that hit nothing */
} prb_camera;

/* Renders the current state of all envs: rgb_dev uint8 [N,H,W,3]; depth_dev float [N,H,W] eye-space depth in metres
 * (far plane where nothing is hit) and seg_dev int32 [N,H,W] collider index (-1 where nothing is hit) are optional
 * (NULL).  Reads the state only: no simulation state or step output changes.  Asynchronous on `stream`. */
int prb_render(prb_handle* h, const prb_camera* cam, const float* col_rgb_host, uint8_t* rgb_dev, float* depth_dev,
               int32_t* seg_dev, void* stream);
/* Pixel-box slab tests prb_render has run since creation (after tile culling; for reports).  Synchronises the device. */
int64_t prb_render_box_tests(prb_handle* h);

/* Ray casts against the collision boxes of every env, like PyBullet's rayTestBatch() on each client: the nearest hit of
 * each segment from -> to.  Reads the current state (the state prb_render reads) and writes only the given arrays;
 * asynchronous on `stream`, no host synchronisation, no allocation, exactly one kernel launch.  Works with either
 * PRB_PIPELINE.
 *
 * Endpoints are given in `frame`: the world (-1) or site s of the arm (the model's site_link[s] / site_pos / site_rot;
 * 0 is the end effector, the frame of an attached prb_camera, 1 the wrist, 2 and 3 the finger pads), where a point x
 * is p_s + R_s x in the world.  Results are in the world.  In the box coordinates of collider c the ray is o + t dl,
 * dl = R_box^T (to - from) (not normalised), t in [0, 1]: an axis with |dl_k| < 1e-12 is parallel and keeps the ray
 * only if o_k is in [-h_k, h_k]; otherwise t is clipped to the slab.  The box is hit when the clipped t0 <= t1 and
 * t0 < 1; the nearest hit wins, the lower collider index on equal t0.  (The rule of the step's gripper_proprioception
 * ray.)  So a ray that starts inside a box hits it at fraction 0, a hit exactly at `to` is a miss, and a zero-length ray
 * hits only when it starts inside a box.  A ray with a non-finite endpoint is a miss.
 *
 * The normal is the world axis of the box slab whose entry set t0, pointing against the ray (the lowest axis on equal
 * entries); when the ray starts inside the box (no entry > 0) it is -(to - from) / |to - from|, and 0 for a zero-length
 * ray. */
typedef struct prb_rays {
  int32_t num_rays;        /* R per env, 1..16384 */
  int32_t per_env;         /* 0: from / to are [R,3], shared by every env; 1: [N,R,3] */
  int32_t frame;           /* -1: world; 0..3: site s of the arm */
  int32_t reserved;        /* must be 0 */
  uint64_t collider_mask;  /* bit c set: collider c can be hit (~0: all; bits >= n_col ignored) */
} prb_rays;
/* from_dev, to_dev: float device arrays in the layout of r->per_env.  Outputs (device, indexed in 64 bits):
 * hit_collider_dev int32 [N,R] (required; -1 for a miss), hit_fraction_dev float [N,R] (required; in [0,1), 1 for a
 * miss), hit_position_dev float [N,R,3] (optional, NULL; world, 0 for a miss), hit_normal_dev float [N,R,3] (optional,
 * NULL; world unit vector, 0 for a miss).  Fails (PRB_ERR_INVALID, with a message, before any launch) for num_rays
 * outside 1..16384, frame outside -1..3, per_env not 0 or 1, reserved not 0, or a NULL required pointer. */
int prb_ray_test(prb_handle* h, const prb_rays* r, const float* from_dev, const float* to_dev, int32_t* hit_collider_dev,
                 float* hit_fraction_dev, float* hit_position_dev, float* hit_normal_dev, void* stream);

/* Closest points between collision boxes in every env, like PyBullet's getClosestPoints(bodyA, bodyB, distance[,
 * linkIndexA, linkIndexB]) on each client.  Reads the current state (the state prb_render reads) and writes only the
 * given arrays; asynchronous on `stream`, no host synchronisation, no allocation, exactly one kernel launch (the queries
 * travel in its parameters).  Works with either PRB_PIPELINE.
 *
 * For env e and query k the candidates are every collider pair (a, b), a in mask_a, b in mask_b, a != b (two colliders of
 * one body are a pair too).  The pair with the smallest signed distance d is reported when d <= max_distance (inclusive);
 * ties go to the lower a, then the lower b.  Conventions of the contact report: the normal points from B towards A and
 * position_on_a = position_on_b + distance * normal_on_b, all in the world.
 *   * separated boxes (d > 0): d is the Euclidean distance of the two boxes, the positions a closest pair of points and
 *     the normal (position_on_a - position_on_b) / d;
 *   * touching or overlapping boxes (d <= 0): d = -(penetration depth), the minimum overlap over 15 separating-axis
 *     candidates: A's 3 face axes, B's 3, the 9 edge crosses a_i x b_j (in that order; a cross with |a_i x b_j|^2 < 1e-10
 *     is skipped).  The normal is that axis, turned towards A; on equal overlaps the lowest axis wins.  The witness is ONE
 *     deepest point, not a manifold (prb_get_contacts gives the solver's manifolds).  Its candidates, in this order: for
 *     an edge cross the point of A's supporting edge nearest B's supporting edge as position_on_a; A's deepest vertex
 *     (its support along -normal) as position_on_a; B's deepest vertex (its support along the normal) as position_on_b;
 *     two points found by projecting alternately onto A's and B's supporting features (vertex, edge or face; a box axis
 *     with |normal . axis| < 1e-4 spans the feature), from B's or from A's feature centre.  The other point always
 *     follows from position_on_a = position_on_b + distance * normal, and the first candidate whose two points lie
 *     nearest their boxes and supporting planes (L1) wins; supports take sign(0) = +.
 * Recalled from PyBullet, not verified against a PyBullet run: `distance` is an inclusive bound, the sign and direction
 * conventions above.  PyBullet returns one point per pair of shapes within reach; this call returns only the nearest
 * pair of each query. */
typedef struct prb_closest_query {
  uint64_t mask_a, mask_b;   /* colliders of side A and side B (bit c: collider c; bits >= n_col ignored) */
} prb_closest_query;
typedef struct prb_closest {
  int32_t num_queries;       /* Q, 1..64 */
  int32_t reserved;          /* must be 0 */
  float max_distance;        /* PyBullet's `distance`: finite, >= 0 (m) */
  int32_t reserved2;         /* must be 0 */
} prb_closest;
/* queries_host: Q host structs.  Outputs (device, indexed in 64 bits): collider_a_dev, collider_b_dev int32 [N,Q] and
 * distance_dev float [N,Q] (required), position_on_a_dev, position_on_b_dev, normal_on_b_dev float [N,Q,3] (optional,
 * NULL).  No pair within reach: colliders -1, distance +inf, positions and normal 0.  Fails (PRB_ERR_INVALID, with a
 * message, before any launch) for num_queries outside 1..64, a reserved field not 0, a non-finite or negative
 * max_distance, or a NULL required pointer. */
int prb_closest_points(prb_handle* h, const prb_closest* q, const prb_closest_query* queries_host, int32_t* collider_a_dev,
                       int32_t* collider_b_dev, float* distance_dev, float* position_on_a_dev, float* position_on_b_dev,
                       float* normal_on_b_dev, void* stream);

/* The arm's Jacobians, joint-space mass matrix and inverse dynamics in every env, like PyBullet's calculateJacobian,
 * calculateMassMatrix and calculateInverseDynamics on each client.  Reads the current state and the caller's arrays and
 * writes only the given outputs; asynchronous on `stream`, no host synchronisation, no allocation, exactly one kernel
 * launch (the points travel in its parameters).  Works with either PRB_PIPELINE.
 *
 * The arm (body 0) only: its nd DoF (12 UR5, 9 Panda) in the compiled model's link order, with the model's fixed base.
 * Free and slide bodies are not covered.  Each env is evaluated at q and qd from q_dev / qd_dev (float [N,nd], device)
 * when given, each from the env's state row when NULL; qdd from qdd_dev when given, 0 when NULL.  The state is never
 * written.
 *
 * Points (num_points P in 0..16): site = -1: local_position in the frame of model arm link `link` (0..nd-1), the link
 * (joint) frame after the joint's motion; site = 0..3: local_position in site s's frame (as prb_ray_test's frames: 0 the
 * end effector, 1 the wrist, 2 and 3 the finger pads), and link must be -1.
 * Outputs (device, float, indexed in 64 bits; each optional, at least one given):
 *   * jacobian_dev [N,P,6,nd]: rows 0-2 linear, 3-5 angular, world frame.  Column j for a point x on link l is 0 unless
 *     j is an ancestor-or-self of l; revolute j: (a_j x (x - p_j), a_j); prismatic j: (a_j, 0), with a_j the joint's
 *     world axis and p_j its link frame origin;
 *   * point_position_dev [N,P,3]: the world position of each point;
 *   * point_velocity_dev [N,P,6]: J qd (linear, angular), the point's world velocity;
 *   * mass_matrix_dev [N,nd,nd]: M(q), symmetric bit for bit; the step's own arithmetic (composite rigid bodies);
 *   * tau_dev [N,nd]: tau = M(q) qdd + h(q, qd), h the Coriolis, centrifugal and gravity term (the step's recursive
 *     Newton-Euler bias, before joint damping).  Joint damping, motors, limits, gears, contacts and link damping are
 *     not included.  qdd = 0 gives the bias h; qd = qdd = 0 the gravity-holding torques.  Without qdd_dev tau is h.
 * Fails (PRB_ERR_INVALID, with a message, before any launch) for num_points outside 0..16, points without a point
 * output or a point output without points, a NULL points_host with points, a link outside 0..nd-1 for site -1, a site
 * outside -1..3 or a site with link != -1, a reserved field not 0, or no output at all.
 * Recalled from PyBullet, not verified against a PyBullet run: PyBullet's localPosition is relative to the link's centre
 * of mass (its inertial frame), here to the link frame or a site frame; PyBullet's inverse dynamics is believed to
 * leave out joint damping, as here.  The columns here are in the model's link order; the Python layer
 * (arm_dof_joints) maps them to PyBullet joint indices. */
typedef struct prb_arm_point {
  int32_t link;              /* model arm link 0..nd-1 (site -1), or -1 (a site point) */
  int32_t site;              /* -1: the link frame; 0..3: a site frame */
  float local_position[3];   /* m, in that frame */
  int32_t reserved;          /* must be 0 */
} prb_arm_point;
typedef struct prb_arm_query {
  int32_t num_points;        /* P, 0..16 */
  int32_t reserved;          /* must be 0 */
} prb_arm_query;
int prb_arm_dynamics(prb_handle* h, const prb_arm_query* q, const prb_arm_point* points_host, const float* q_dev,
                     const float* qd_dev, const float* qdd_dev, float* jacobian_dev, float* point_position_dev,
                     float* point_velocity_dev, float* mass_matrix_dev, float* tau_dev, void* stream);

/* Link and joint states of every env, like PyBullet's getLinkStates(computeLinkVelocity=1, computeForwardKinematics=1),
 * getBasePositionAndOrientation, getBaseVelocity and getJointStates on each client.  Reads the current state only and
 * writes only the given outputs; asynchronous on `stream`, no host synchronisation, no allocation, exactly one kernel
 * launch.  Works with either PRB_PIPELINE.
 *
 * body_dev float [N,K,13], K = nd + n_free + n_slide: one row per body frame, pos[3] | quat[4] (x, y, z, w) | linear
 * velocity[3] | angular velocity[3], all in the world frame (the layout of a free body in the state row).  Rows, in order:
 *   * the arm's nd links in the compiled model's link order (the columns of prb_arm_dynamics);
 *   * the n_free free bodies (block, drawer): their 13 state floats, bit for bit, in either frame;
 *   * the n_slide slide bodies (door, button, dial): the body frame after its joint's motion; the linear velocity of a
 *     prismatic body, or the angular velocity of a revolute one, is sqd times its world joint axis, the other part 0.
 *     The compiled model keeps no centre-of-mass offset for them, so both frames are the same.
 * q->frame 0 reports each arm link's link (joint) frame, PyBullet's worldLinkFramePosition / Orientation; 1 its inertial
 * frame, PyBullet's linkWorldPosition / Orientation: the link frame moved to the link's centre of mass (the compiled
 * model keeps the inertia in the link frame, so the orientation is the link frame's).  Velocities are those of the
 * chosen frame's origin: the COM frame's linear velocity is v + w x (c - p).  Orientations come from the link's
 * rotation matrix (Shepperd's method, mat_to_quat), so their sign is not tied to any earlier reading.
 * joint_q_dev, joint_qd_dev float [N, nd + n_slide]: the arm's DoF (model link order), then the slide joints (door,
 * button, dial), straight from the state row.  Each output is optional (NULL); at least one is required.
 * Fails (PRB_ERR_INVALID, with a message, before any launch) for frame not 0 or 1, reserved not 0, or no output.
 * Recalled from PyBullet, not verified against a PyBullet run: which of PyBullet's two frames carries the "link frame"
 * name, and that computeLinkVelocity reports the COM frame's velocity.  Applied joint torques and reaction forces are
 * not reported. */
typedef struct prb_body_query {
  int32_t frame;             /* 0: link (joint) frames; 1: centre-of-mass (inertial) frames */
  int32_t reserved;          /* must be 0 */
} prb_body_query;
int prb_body_states(prb_handle* h, const prb_body_query* q, float* body_dev, float* joint_q_dev, float* joint_qd_dev,
                    void* stream);

/* Masked writes of joint positions and velocities and free-body poses and velocities, like PyBullet's resetJointState,
 * resetBasePositionAndOrientation and resetBaseVelocity on each client.  Asynchronous on `stream`, no host
 * synchronisation, no allocation.
 *
 * Selection: bit j of joint_positions / joint_velocities is column j of [0, nd + n_slide) (the columns of
 * prb_body_states' joint arrays: arm DoF, then slide joints); bit b of free_poses / free_velocities is free body b of
 * [0, n_free).  Inputs use the read layouts: joint_q_dev, joint_qd_dev float [N, nd + n_slide], body_dev float [N,K,13]
 * of which only the selected words of the free-body rows (pos | quat, or linear | angular velocity) are read, so a
 * prb_body_states read, an edit and this call round-trip.  Only envs with mask_dev[e] != 0 (uint8 [N]; NULL: all) are
 * written.
 *
 * Positions and velocities are written exactly; a written quaternion is divided by its norm in fp32 (unfused, correctly
 * rounded: n = sqrt(((x x + y y) + z z) + w w), q / n).  Motor targets, gains and impulse limits, the goal, the reset
 * counter and the per-env dynamics table are left alone, as PyBullet's resetJointState leaves motors alone.  A masked env
 * whose selected inputs hold a non-finite value, or a quaternion of norm < 1e-6 (or beyond fp32), is left completely
 * unchanged.  status_dev (uint8 [N], optional) gets 0 for an env not masked, 1 written, 2 rejected.
 *
 * In the same call, for the written envs only: the contact report (when enabled) is emptied, and the output buffers are
 * refreshed as prb_observe does (the masked setup launch), so that for them the call gives the same bits as editing
 * the rows, prb_set_state, then prb_observe.  Other envs keep their state and outputs bit for bit.  Launches: the write
 * kernel, the report clear when the report is enabled, one setup launch.
 *
 * No constraint is enforced at the write: a write that breaks one (the UR5 gripper's gear and mimic rows, joint limits,
 * the drawer's rail) is allowed, and the next physics substep's joint rows pull it back, as in PyBullet.
 * Fails (PRB_ERR_INVALID, with a message, before any launch) for bits at or beyond nd + n_slide or n_free, no bit set,
 * a selected input that is NULL, or reserved not 0. */
typedef struct prb_state_write {
  uint32_t joint_positions;   /* bit j: write q of column j */
  uint32_t joint_velocities;  /* bit j: write qd of column j */
  uint32_t free_poses;        /* bit b: write position and orientation of free body b */
  uint32_t free_velocities;   /* bit b: write linear and angular velocity of free body b */
  int32_t reserved;           /* must be 0 */
} prb_state_write;
int prb_write_state(prb_handle* h, const prb_state_write* w, const float* joint_q_dev, const float* joint_qd_dev,
                    const float* body_dev, const uint8_t* mask_dev, uint8_t* status_dev, void* stream);

/* Device-side snapshots, like PyBullet's saveState / restoreState for every env.  prb_save_state copies the state
 * [N, state_stride] (prb_buffers.state_stride) into dst_dev with one cudaMemcpyAsync.  prb_restore_state copies the
 * rows of the envs of mask_dev (uint8 [N]; NULL: all) back from src_dev (one launch), empties their contact report when
 * it is enabled and refreshes their output buffers as prb_observe does.  Restored rows equal the saved rows bit for bit;
 * the other rows are not touched.  The per-env dynamics table is not part of a snapshot (as with prb_set_state).
 * Asynchronous on `stream`.  Fails (PRB_ERR_INVALID) for a NULL dst_dev / src_dev. */
int prb_save_state(prb_handle* h, float* dst_dev, void* stream);
int prb_restore_state(prb_handle* h, const float* src_dev, const uint8_t* mask_dev, void* stream);

/* Contact report: the contact points and forces of every env after a step, like PyBullet's getContactPoints() after
 * stepSimulation().  Off by default; prb_enable_contacts(h, 1) allocates the report (the first time) and empties it.
 * While enabled, prb_step, prb_step_host and prb_substeps (n >= 1) fill it with the contacts the LAST physics substep of
 * the call solved; prb_reset, prb_reset_to, prb_set_state, prb_write_state and prb_restore_state empty it (count 0)
 * for every env whose state they change;
 * prb_observe, prb_set_goal and prb_render leave it unchanged.  With PRB_PIPELINE=fused enabling fails (PRB_ERR_INVALID).
 *
 * Env e has count[e] (0..max_contacts = 64) contacts: those after manifold reduction (<= 4 per pair of collision
 * objects), in the order the setup kernel generated them, which is the order the solver visits them (Bullet's).  For
 * contact i < count[e], at [e, i] of each [N, 64] array and [e, i, :] of each [N, 64, 3] array:
 *   collider_a, collider_b   collider indices of the model (the ids prb_render's segmentation uses); A is the pair's first
 *                            collider (prb_model pair_a: the movable side of lowest body index)
 *   position_on_a, _on_b     world, m; position_on_a = position_on_b + distance * normal_on_b
 *   normal_on_b              unit, world, pointing from B towards A
 *   distance                 m; negative: penetration
 *   normal_force             normal impulse of the contact's row / dt, N, >= 0
 *   lateral_friction_1, _2   friction impulses of its two rows / dt, N: signed force on A along lateral_friction_dir_1, _2
 *   lateral_friction_dir_1, _2   the friction rows' directions (Bullet's btPlaneSpace1 of the normal)
 * Entries i >= count[e] hold -1 (collider ids) and 0 (floats).  The torsional-friction impulse is not reported (PyBullet
 * does not report it either).  That PyBullet reports applied impulse / time step as its forces, and the direction of
 * its normal, are recalled from Bullet's sources, not verified against a PyBullet run. */
typedef struct prb_contacts {
  int32_t* count;                   /* [N] */
  int32_t* collider_a;              /* [N,64] */
  int32_t* collider_b;              /* [N,64] */
  float* position_on_a;             /* [N,64,3] */
  float* position_on_b;             /* [N,64,3] */
  float* normal_on_b;               /* [N,64,3] */
  float* distance;                  /* [N,64] */
  float* normal_force;              /* [N,64] */
  float* lateral_friction_1;        /* [N,64] */
  float* lateral_friction_2;        /* [N,64] */
  float* lateral_friction_dir_1;    /* [N,64,3] */
  float* lateral_friction_dir_2;    /* [N,64,3] */
  int32_t num_envs, max_contacts;
} prb_contacts;
int prb_enable_contacts(prb_handle* h, int32_t enable);
/* Device pointers of the report (handle-owned; valid until prb_destroy).  Fails if the report was never enabled. */
int prb_get_contacts(prb_handle* h, prb_contacts* out);

/* Per-env dynamics, like PyBullet's changeDynamics() on each client: every env gets its own collider friction and
 * free-body mass, inertia and damping.  Off by default: every env runs with the model's values and nothing is allocated.
 * prb_enable_dynamics(h, 1) allocates the table (the first time) and, on every off -> on, fills every env's row with the
 * model's values; prb_enable_dynamics(h, 0) returns to the model's values and keeps the table.  With PRB_PIPELINE=fused
 * enabling fails (PRB_ERR_INVALID).  The table is not part of the state row (prb_get_state / prb_set_state).
 *
 * The arrays are handle-owned device memory (valid until prb_destroy); callers may write them directly.  A write takes
 * effect from the next physics substep issued on the same stream.  Values must be finite, mass and inertia > 0, friction
 * and damping >= 0.  The friction of a contact is the product of its colliders' lateral frictions, clamped to +-10; its
 * torsional coefficient is spinning_friction * lateral_friction summed over its two colliders. */
typedef struct prb_dynamics {
  float* lateral_friction;        /* [N, n_col]      per collider (the model's col_friction) */
  float* spinning_friction;       /* [N, n_col]      per collider (the model's col_spin) */
  float* mass;                    /* [N, n_free]     kg, free bodies */
  float* local_inertia_diagonal;  /* [N, n_free, 3]  kg m^2, principal moments about the COM */
  float* linear_damping;          /* [N, n_free] */
  float* angular_damping;         /* [N, n_free] */
  int32_t num_envs, n_col, n_free;
} prb_dynamics;
int prb_enable_dynamics(prb_handle* h, int32_t enable);
/* Device pointers of the table.  Fails if the table was never enabled. */
int prb_get_dynamics(prb_handle* h, prb_dynamics* out);

/* [lo, hi] scale of the model's value; lo = hi = 1 keeps the model's value exactly. */
typedef struct prb_dynamics_ranges {
  float lateral_friction[2], spinning_friction[2];        /* one draw per body (static scene, arm, each free / slide body) */
  float mass[2], linear_damping[2], angular_damping[2];   /* one draw per free body; the inertia diagonal follows mass */
} prb_dynamics_ranges;
/* Draws new dynamics for the envs of mask_dev (uint8 [N] on the device; NULL: every env): value = model value * s,
 * s ~ U[lo, hi], in fp32, never compounding earlier draws.  The draws depend only on the seed, the global env id
 * (env_offset + e) and the env's reset counter, so calling this before prb_reset gives each episode its own dynamics
 * (prb_reset does not draw on its own; the objects then settle with their new mass).  Fails (PRB_ERR_INVALID, before any
 * launch) unless the table is enabled and every bound is finite with 0 <= lo <= hi, and 0 < lo for mass. */
int prb_randomize_dynamics(prb_handle* h, const prb_dynamics_ranges* r, const uint8_t* mask_dev, void* stream);

/* Number of kernels launched by this handle since creation (bench.py reports it). */
int64_t prb_launch_count(prb_handle* h);
/* Env steps (since creation; a reset counts as one) in which a contact had to be dropped because the per-env
 * capacity (overlapping pairs, contacts, joint rows) was exceeded: an env is counted once per step however many of
 * its 12 substeps dropped one.  Synchronises the device. */
int64_t prb_overflow_count(prb_handle* h);
/* Per-env facts of the last substep built, for sizing reports and for tests that must sample every solver path:
 * [N,4] int32 = {arm-island solver class (0: joint-row kernel, 1..4: size class of the arm-island kernel) | q count of
 * the arm island's region << 8, contacts, q count of the env's whole record stream, joint rows | capacity flags << 8
 * (1: more than 32 overlapping collider pairs, 2: more than 32 contacts, 4: contact between two slide bodies)}; synchronous. */
int prb_debug_usage(prb_handle* h, int32_t* host_out);
/* Static facts of the step kernel for reports: dynamic shared memory per block, warps per block. */
int prb_kernel_info(prb_handle* h, int32_t* smem_bytes_per_block, int32_t* envs_per_block, int32_t* regs_per_thread);

const char* prb_last_error(prb_handle* h);
const char* prb_version(void);

#ifdef __cplusplus
}
#endif
#endif
