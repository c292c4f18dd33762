/*
 * sg_b200.h -- C ABI of the B200-native batched rollout engine for Scenario Gym.
 *
 * The reference (driskai/scenario_gym v0.3.1) is pure Python and has no FFI; the
 * "plugin API" is Python subclassing.  This header is the boundary a maintainer
 * would bind (ctypes stub in INTEGRATION.md) to replace the reference's per-tick
 * path.  Each entry point cites the reference code it replaces (paths relative
 * to the reference root).
 *
 * Conventions
 *   - plain C: pointers + sizes, no C++/torch types.
 *   - every array pointer inside SgScene / SgState / SgInputs given to the sg_*
 *     entry points is CALLER-OWNED DEVICE memory (e.g. torch allocations); the
 *     library never frees it.  The *_host entry points take HOST pointers.
 *   - layout is structure-of-arrays: a "plane" is [N*M] (N scenarios x M entity
 *     slots, scenario-major), multi-component fields are [C][N*M].
 *   - all floating point is IEEE fp64 and follows the reference's operation order
 *     (no FMA contraction where the reference has none).
 *   - return code: 0 ok, negative = error; text via sg_last_error().
 *   - stream-ordered and non-blocking unless stated; `stream` is a cudaStream_t
 *     passed as void* (NULL = legacy default stream).
 *   - no global mutable state except the last-error string (thread-local).
 *   - which kernel runs is the library's choice (vehicle-only scenes, replay-only scenes, crowds and
 *     everything else have their own kernels).  Discrete results -- presence, tick counts and times,
 *     collision flags / pairs / events, RSS records and flags, goal indices -- are decided by exact
 *     predicates and do not depend on that choice.  Continuous results agree with the reference
 *     within 1e-9, but not bit for bit ACROSS kernel families: the vehicle-only kernels use
 *     Newton-refined reciprocals / square roots and their own sincos (< 1 ulp), the general kernel
 *     libm and IEEE division, so adding one replayed entity to a vehicle scene changes the vehicles'
 *     poses in the last place.  RSS branches that compare such values with zero (`vr == 0.0`,
 *     sign(pos) == sign(v), callback.py:243-268) are only reached with exact zeros produced by
 *     clamping, which every kernel produces identically.  Within one family (table / in-kernel
 *     action source, fused / chunked / host-buffer rollouts, trace on / off) results are bit-equal.
 *
 * The CPU oracle (oracle/sg_oracle.c, test infrastructure) exports the same
 * signatures with the prefix sgo_ and host pointers, so tests drive both through
 * identical code.
 */
#ifndef SG_B200_H
#define SG_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SG_ABI_VERSION 16

/* entity slot kinds (who produces the slot's next pose each tick) */
enum SgKind {
  SG_KIND_EMPTY = 0,        /* padding slot                                               */
  SG_KIND_REPLAY = 1,       /* no agent: BatchReplayEntity, entity/batch.py:34-53,55-128   */
  SG_KIND_AGENT_REPLAY = 2, /* ReplayTrajectoryAgent (default ego), agent.py:118-128       */
  SG_KIND_VEHICLE = 3,      /* agent with VehicleController, controller.py:57-140          */
  SG_KIND_PEDESTRIAN = 4,   /* PedestrianAgent + SocialForce, pedestrian/                  */
  SG_KIND_HOST = 5,         /* pose supplied by a host-side (Python) agent every tick      */
  SG_KIND_PID = 6           /* PIDAgent + PIDController, agent.py:131-148, controller.py:143-258 */
};

/* catalog type of the entity (collision.py:85, pedestrian/sensor.py:61) */
enum SgEntityType { SG_ETYPE_VEHICLE = 0, SG_ETYPE_PEDESTRIAN = 1, SG_ETYPE_MISC = 2 };

/* terminal conditions, state/state.py:397-408 (bit flags) */
enum SgTerminal {
  SG_TERM_MAX_LENGTH = 1,
  SG_TERM_COLLISION = 2,
  SG_TERM_EGO_COLLISION = 4,
  SG_TERM_EGO_OFF_ROAD = 8  /* entities[0] absent or not strictly inside the driveable surface */
};

/* feature switches (bit flags in SgParams.features) */
enum SgFeature {
  SG_FEAT_COLLISIONS = 1,   /* state.collisions() + CollisionMetric, a8-a10 */
  SG_FEAT_EGO_METRICS = 2,  /* EgoAvgSpeed/EgoMaxSpeed/EgoDistanceTravelled, a11 */
  SG_FEAT_RSS = 4,          /* RSSDistances callback + RSS metric, a13-a14 */
  SG_FEAT_COLL_MATRIX = 8,  /* also write the per-tick pair matrix SgState.coll_mask */
  SG_FEAT_NO_GRID = 16,     /* crowd scenarios: exhaustive O(M^2) sensor / broad-phase sweeps instead of
                               the shared-memory cell grid (same results; kept for cross-checks) */
  SG_FEAT_SEQUENTIAL = 32   /* replay-only scenes: walk the ticks one after another instead of the
                               tick-parallel kernel (same results up to the summation order of the
                               distances; kept for cross-checks) */
};

/* facts about a scene the packer knows (SgScene.scene_flags) */
enum SgSceneFlag {
  SG_SCENE_FLAT_BOXES = 1 /* some live slot has a box without area (width * length == 0): such scenes
                             take the general kernel, whose narrow phase knows the degenerate rules */
};

/* record codes appended to RSSDistances.intersect[e] (rss/callback.py:168-228,304-338) */
enum SgRssRecord {
  SG_RSS_SAFE = 0,
  SG_RSS_LATERAL = 1,
  SG_RSS_LONGITUDINAL = 2,
  SG_RSS_BOTH = 3,
  SG_RSS_UNSAFE_LATERAL = 4,
  SG_RSS_UNSAFE_LONGITUDINAL = 5,
  SG_RSS_FOUND = 6,
  SG_RSS_NONE = 255 /* entity absent this tick: nothing appended */
};

/* scalar parameters (gym / controller / behaviour constructor arguments) */
typedef struct SgParams {
  double timestep;         /* ScenarioGym(timestep), scenario_gym.py:31                   */
  int32_t persist;         /* ScenarioGym(persist), scenario_gym.py:32                    */
  int32_t terminal;        /* SgTerminal bits, scenario_gym.py:34-36                      */
  int32_t features;        /* SgFeature bits                                              */
  int32_t max_ticks;       /* safety bound for sg_rollout loops                           */
  /* VehicleController(max_steer, max_accel, max_speed, allow_reverse) controller.py:64-98 */
  double veh_max_steer;
  double veh_max_accel;
  double veh_max_speed;    /* NaN = None                                                  */
  int32_t veh_allow_reverse;
  int32_t _pad0;
  /* PedestrianAgent / SocialForceParameters, pedestrian/agent.py:18-44, social_force.py:16-30 */
  double ped_max_speed;          /* PedestrianController(max_speed=5.0)                   */
  double ped_head_rot_angle;     /* PedestrianSensor(head_rot_angle=0.0)                  */
  double ped_distance_threshold; /* PedestrianSensor(distance_threshold=1.0)              */
  double sf_max_speed_factor;    /* BehaviourParameters.max_speed_factor = 1.3            */
  double sf_bias_lon, sf_bias_lat; /* noise means (std must be 0 for parity)              */
  double sf_sight_weight;        /* 0.5                                                   */
  int32_t sf_sight_weight_use;   /* True                                                  */
  int32_t _pad1;
  double sf_sight_angle;         /* 200 (degrees)                                         */
  double sf_relaxation_time;     /* 1.5                                                   */
  double sf_ped_repulse_V;       /* 1.0                                                   */
  double sf_ped_repulse_sigma;   /* 1.0                                                   */
  double sf_ped_attract_C;       /* 0.0                                                   */
  /* RSSParameters, metrics/rss/callback.py:21-31 */
  double rss_response_time;      /* 0.6                                                   */
  double rss_min_long_accel;     /* 1.2*9.81                                              */
  double rss_max_long_accel;     /* 1.2*9.81                                              */
  double rss_min_safe_clearance; /* 0.1                                                   */
  /* PIDController gains, controller.py:154-161 (vehicle limits above apply to it too) */
  double pid_steer_Kp, pid_steer_Kd, pid_accel_Kp, pid_accel_Kd, pid_accel_Ki;
  /* SocialForce boundary forces, pedestrian/social_force.py:24-29, 86-104, 190-211 */
  double sf_boundary_repulse_U, sf_boundary_repulse_R;         /* walkable surface: 10.0, 0.2 */
  double sf_imp_boundary_repulse_U, sf_imp_boundary_repulse_R; /* impenetrable surface: 2.0, 0.1 */
  /* SocialForce random fluctuations (RandomWalkParameters.std_lon / std_lat, random_walk.py:13-19,
     drawn at social_force.py:106-108).  The reference draws them from the global numpy generator, so
     no engine can reproduce its values: with a non-zero std the engine adds N(0, std) noise from its
     own counter-based stream (a function of sf_noise_seed, scenario, slot and tick; the CPU oracle
     evaluates the same function).  std = 0 (the parity configurations) adds the bias exactly. */
  double sf_std_lon, sf_std_lat;
  uint64_t sf_noise_seed;
} SgParams;

/* immutable description of N scenarios x M slots */
typedef struct SgScene {
  int32_t n_scenarios; /* N */
  int32_t n_slots;     /* M, 1..1024 */
  int64_t n_traj_rows; /* total control points in traj_rows */
  int64_t n_union_rows;/* total rows in union_t            */
  int64_t n_route_pts; /* total points in route_xy         */
  /* OR of (1u << SgKind) over all slots, or 0 = unspecified (always valid).  A non-zero mask
     lets the library pick a specialised kernel; {VEHICLE[,EMPTY]} additionally promises that
     every vehicle slot is present at reset (its trajectory covers t0). */
  uint32_t kind_mask;
  uint32_t scene_flags; /* SgSceneFlag bits */
  const uint8_t* kind;   /* [N*M] SgKind */
  const uint8_t* etype;  /* [N*M] SgEntityType */
  const double* box;     /* [4][N*M]: width, length, center_x, center_y (catalog_entry.py:83-90) */
  /* every slot's own trajectory (trajectory.py:34-96), CSR over slots; rows are
     [t,x,y,z,h,p,r]; a slot with 1 row is "static" (entity/base.py:154-156) */
  const int64_t* traj_off; /* [N*M+1] */
  const double* traj_rows; /* [n_traj_rows][7] */
  /* BatchReplayEntity union-knot table of scenario n (entity/batch.py:80-128):
     knots union_t[union_off[n] .. union_off[n+1]) ; values union_x[row][6][M] */
  const int64_t* union_off; /* [N+1] */
  const double* union_t;    /* [n_union_rows] */
  const double* union_x;    /* [n_union_rows][6][M] */
  const double* t0;         /* [N] start time, scenario_gym.py:213-215 */
  const double* length;     /* [N] scenario.length, scenario/scenario.py:88-91 */
  const int32_t* ego_slot;  /* [N] slot of scenario.ego */
  const int32_t* first_slot;/* [N] slot of scenario.entities[0] (ego_collision) */
  /* pedestrians (pedestrian/agent.py:18-47) */
  const double* ped_speed_desired; /* [N*M] */
  const int64_t* route_off;        /* [N*M+1] */
  const double* route_xy;          /* [n_route_pts][2] */
  /* Road-network surfaces (road_network/road_network.py:306-328: the unions of the driveable /
     walkable / impenetrable geometries' boundaries), kept as polygon soups and shared between
     scenarios.  Scenario n uses network rn_of[n] (-1 or rn_of == NULL: an empty network).
     Surface k (0 driveable, 1 walkable, 2 impenetrable) of network r = polygons
     rn_poly_off[3r+k] .. rn_poly_off[3r+k+1]; polygon q = edges rn_edge_off[q] .. rn_edge_off[q+1]
     (every ring of the polygon, holes included: membership is the crossing parity over them);
     edge e = rn_edges[4e .. 4e+3] = x0, y0, x1, y1.  rn_has_area[3r+k]: surface.area > 0.
     Used by the ego_off_road terminal condition (state/state.py:401-407) and the social-force
     boundary forces. */
  int32_t n_networks;
  int32_t _pad1;
  int64_t n_rn_polys;
  int64_t n_rn_edges;
  const int32_t* rn_of;       /* [N] */
  const int64_t* rn_poly_off; /* [3*n_networks+1] */
  const int64_t* rn_edge_off; /* [n_rn_polys+1] */
  const double* rn_edges;     /* [n_rn_edges][4] */
  const uint8_t* rn_has_area; /* [3*n_networks] */
  /* Per-agent VehicleController limits (controller.py:64-98 are constructor arguments of each
     instance): [4][N*M] max_steer, max_accel, max_speed (NaN = None), allow_reverse (0 / 1); NULL: every
     vehicle / PID slot uses the SgParams values. */
  const double* veh_limits;
  /* A window onto scenarios [scenario_base, scenario_base + n_scenarios) of a larger batch whose arrays
     were laid out for plane_stride / n_slots scenarios: every pointer above (and in the SgState passed
     with it) addresses the window's first element, planes of [k][N*M] arrays stay plane_stride elements
     apart, and slot / scenario numbers that mean something outside the arrays (the action stream's
     draw index, the noise stream, SgEvent.scenario) are counted from the start of the batch.
     plane_stride = 0: the whole batch (plane_stride = N*M, scenario_base = 0).  sg_rollout_host uses
     windows to overlap the upload of one part of a batch with the rollout of another; traces
     (trace_cap > 0) are not supported on a window. */
  int64_t plane_stride;
  int32_t scenario_base;
  int32_t _pad2;
} SgScene;

/* one recorded ego-collision rising edge (metrics/collision.py:70-75) */
typedef struct SgEvent {
  int32_t scenario;
  int32_t tick;   /* 1-based tick index at which it was recorded */
  int32_t slot;   /* hazard slot */
  int32_t _pad;
  double t;       /* state.t */
} SgEvent;

/* mutable state + outputs; all arrays caller-owned */
typedef struct SgState {
  /* State buffers, state/state.py:90-96 */
  double* pose;      /* [6][N*M] x,y,z,h,p,r */
  double* vel;       /* [6][N*M] */
  double* dist;      /* [N*M] */
  uint8_t* present;  /* [N*M] entity in state.poses */
  double* t;         /* [N] */
  double* prev_t;    /* [N] */
  int32_t* tick;     /* [N] ticks taken since reset */
  uint8_t* done;     /* [N] state.is_done */
  /* controller state */
  double* speed;     /* [N*M] VehicleController.speed / PedestrianController.speed */
  int32_t* goal_idx; /* [N*M] PedestrianAgent.goal_idx */
  double* force;     /* [2][N*M] PedestrianAgent.force */
  /* search cursors (implementation state; reset by sg_reset) */
  int32_t* cur_own;   /* [N*M] */
  int32_t* cur_union; /* [N] */
  /* ego metrics, metrics/trajectory.py */
  double* ego_avg_speed; /* [N] */
  double* ego_avg_t;     /* [N] EgoAvgSpeed.t */
  double* ego_max_speed; /* [N] */
  double* ego_dist;      /* [N] */
  /* collisions */
  uint32_t* ego_hits;       /* [N][W] CollisionMetric.last_timestep as a bit set, W=ceil(M/32) */
  uint32_t* coll_mask;      /* [N][M][W] pair matrix of the current tick (SG_FEAT_COLL_MATRIX) */
  uint8_t* collided;        /* [N*M] slot was in any collision so far */
  int32_t* first_coll_tick; /* [N] first tick with any collision, -1 = none */
  int32_t* first_coll_pair; /* [N][2] smallest (i,j), i<j, colliding at that tick */
  int64_t* n_pair_ticks;    /* [N] sum over ticks of #colliding unordered pairs */
  SgEvent* events;          /* [event_cap] ego rising-edge events (unordered) */
  int32_t* event_count;     /* [1] total events produced (may exceed event_cap) */
  int32_t event_cap;
  int32_t trace_cap;        /* ticks of trace storage, 0 = no trace */
  /* RSS, metrics/rss/callback.py */
  uint8_t* rss_state;   /* [N*M] bits0-1 last marker (0 none,1 lateral,2 longitudinal); bits2-3 found (0,1 unsafe_lateral,2 unsafe_longitudinal) */
  uint8_t* rss_last;    /* [N*M] SgRssRecord appended this tick */
  double* safe_dist;    /* [2][N*M] RSSDistances.safe_distances[e] = [lat, long] */
  double* safe_ratio;   /* [2][N*M] RSSDistances.entity_safe_ratios[e] */
  uint8_t* rss_flags;   /* [N] bit0: safe_longitudinal violated, bit1: safe_lateral violated */
  /* optional trace (State._recorded_poses, state/state.py:227-228); index 0 = reset */
  double* trace_pose;      /* [trace_cap][6][N*M] */
  uint8_t* trace_present;  /* [trace_cap][N*M] */
  double* trace_t;         /* [trace_cap][N] */
  /* PIDController state: e_lon_prev, e_lon_int, e_lat_prev (controller.py:198-203) */
  double* pid_err;         /* [3][N*M] */
} SgState;

/* Device-side VehicleAction source for agents that draw uniform random actions (the "random
   accel/steer" configurations): the value consumed by slot i (= n*M + s) at the k-th tick after
   reset is
       low[c] + scale[c] * u_j ,   j = offset[c] + k * tick_stride + i ,   c = 0 accel, 1 steer,
   where u_j is the j-th double (0-based) of numpy.random.Generator(PCG64).random() started from the
   given bit-generator state -- PCG64 XSL-RR 128/64, u = (next_uint64 >> 11) * 2^-53, the stream
   numpy.random.default_rng(seed) produces -- so a host policy drawing
   rng.uniform(low, high, (T, N*M)) and the device consume bit-identical actions without the table
   ever crossing PCIe.  The kernels jump ahead per slot (O(log j) at launch, one 128-bit
   multiply-add per draw afterwards). */
typedef struct SgActionRng {
  uint64_t state_hi, state_lo; /* bit_generator.state["state"]["state"] (128 bit) */
  uint64_t inc_hi, inc_lo;     /* bit_generator.state["state"]["inc"]                */
  int64_t offset[2];
  int64_t tick_stride;
  double low[2], scale[2];
} SgActionRng;

/* per-call inputs */
typedef struct SgInputs {
  /* VehicleAction(accel, steer) tables, action.py:66-83: actions[k][c][N*M] is consumed
     by the k-th tick executed in this call (k = 0 .. n_action_ticks-1) */
  const double* actions;
  int32_t n_action_ticks;
  /* non-zero: tick scenarios whose is_done flag is already set too -- ScenarioGym.step() has no
     is_done guard (scenario_gym.py:227-254); rollout() loops `while not is_done` (:262) */
  int32_t step_done;
  /* SG_KIND_HOST slots: pose returned by the host agent for the next tick */
  const double* host_pose;      /* [6][N*M] or NULL */
  const uint8_t* host_present;  /* [N*M] 0 = agent returned None */
  /* fp32 action table (policy networks emit fp32; widening is exact): same layout as `actions`,
     used when `actions` is NULL */
  const float* actions_f32;
  /* use_rng != 0 (and no table): actions come from `rng`; the k-th tick executed in this call
     consumes row rng_tick0 + k, and n_action_ticks bounds the rows as for a table */
  int32_t use_rng;
  int32_t rng_tick0;
  SgActionRng rng;
} SgInputs;

/* Closed-loop environment (sg_env_observe / sg_env_reward): which slots a policy drives, what it
   observes and how it is rewarded.  Agent a of scenario n is slot agent_slot[n*A + a] (-1: padding).
   An observation row has F floats (below), all in the agent's frame
   (x, y, h its pose, (c, s) = (cos h, sin h), rot(dx, dy) = (c*dx + s*dy, -s*dx + c*dy)):
     self       speed (controller state), rot(vx, vy), vel[3] (heading rate)
     target     per lookahead tau: q = position_at_t(own trajectory, t + tau, clamped):
                rot(qx - x, qy - y), remainder(qh - h, 2 pi)
     neighbours the K present other slots j with the smallest (d2, j), d2 = dx*dx + dy*dy < radius^2
                (radius <= 0: no cut-off), ascending: rot(dx, dy), cos(hj - h), sin(hj - h),
                rot(vxj - vx, vyj - vy), width_j, length_j, [etype_j == pedestrian], 1; missing: zeros
     road       driveable surface strictly contains (x, y); distance from (x, y) to the surface's rings
                (zeros when the network has no driveable area)
     lidar      (n_rays = R > 0) R readings, ray k along (ex, ey) = ray_dir[k] in the agent's frame, which must
                be (cos, sin)(2 pi k / R) to within 1e-12 (the caller passes the values, so every
                implementation uses the same bits).  World direction u = (c*ex - s*ey, s*ex + c*ey), ray
                (x, y) + t*u, t >= 0.  Every present slot j != the agent's, of any type, is the oriented box
                the collision test uses: (cj, sj) = (cos hj, sin hj), centre X = xj + (bcx*cj - bcy*sj),
                Y = yj + (bcx*sj + bcy*cj), half extents hl = length / 2 along hj, hw = width / 2 across.
                Hit test (closed set, slab form, this operation order, no FMA):
                  p = (x - X, y - Y); ox = cj*px + sj*py, oy = -sj*px + cj*py;
                  dx = cj*ux + sj*uy, dy = -sj*ux + cj*uy;
                  per axis (o, d, e) in {(ox, dx, hl), (oy, dy, hw)}: d != 0: lo, hi = min, max of
                  (-e - o) / d and (e - o) / d; d == 0: a miss if |o| > e, else (-inf, +inf);
                  enter = max(lo_x, lo_y), exit = min(hi_x, hi_y); a hit iff exit >= enter and exit >= 0,
                  at distance (enter > 0 ? enter : 0).
                So a touching corner or a ray along an edge hits, an origin inside another box reads 0 and
                boxes without width / size act as segments / points.  Reading = min(ray_range, smallest hit
                distance over j) in fp64, rounded once to fp32 (ray_range when nothing is hit).
   The row is F = 4 + 3*L + 10*K + (road ? 2 : 0) + R floats; with R = 0 it is the row without the lidar
   block, bit for bit.  Absent / padding agents get zero rows.  Reward terms (after a tick, against the snapshot the last
   observe took): progress = dist - dist_snap; collision = collided rose 0 -> 1; off_road = network has
   driveable area and the present slot is not strictly inside it; tracking = -|(x, y) - position_at_t(own
   trajectory, t, clamped)[:2]|; rss = the slot is the ego and rss_flags gained a bit.  Absent / padding
   agents get zero terms.  reward = sum_k w[k] * term_k. */
typedef struct SgEnvSpec {
  int32_t n_agents;          /* A >= 1 */
  int32_t k_neighbours;      /* K, 0..32 */
  const int32_t* agent_slot; /* [N*A] device */
  double radius;
  int32_t n_lookahead;       /* L, 0..8 */
  int32_t road;              /* non-zero: append the road block */
  double lookahead[8];       /* seconds */
  double weights[5];         /* progress, collision, off_road, tracking, rss */
  /* snapshot written by sg_env_observe for the scenarios it observes, read by sg_env_reward (device) */
  double* snap_dist;         /* [N*A] */
  uint8_t* snap_collided;    /* [N*A] */
  int64_t* snap_pair_ticks;  /* [N] */
  uint8_t* snap_rss;         /* [N] */
  /* lidar block (appended after the road block; read by sg_env_observe only) */
  int32_t n_rays;            /* R, 0..256 (0: no lidar block) */
  int32_t _pad0;
  double ray_range;          /* metres, finite and > 0 when R > 0 */
  const double* ray_dir;     /* [R][2] device: unit directions in the agent frame (see above) */
} SgEnvSpec;

int sg_abi_version(void);
/* sizeof() of the ABI structs so bindings can verify their mirror: which = 0 SgParams,
   1 SgScene, 2 SgState, 3 SgInputs, 4 SgEvent, 5 SgActionRng, 6 SgHostResults, 7 SgEnvSpec */
int64_t sg_sizeof(int which);
const char* sg_last_error(void);
void sg_default_params(SgParams* p);

/* State.reset(t0) + Metric.reset + Agent.reset: state/state.py:106-143,
   scenario_gym.py:217-225, controller.py:100-103, metrics/trajectory.py:13-18 */
int sg_reset(const SgScene* scene, const SgParams* params, SgState* state, int device, void* stream);

/* sg_reset of the scenarios with mask[n] != 0 only (mask [N], device memory; NULL: all of them).  Every
   field of every other scenario is left as it was, and event_count is not touched. */
int sg_reset_scenarios(const SgScene* scene, const SgParams* params, SgState* state, const uint8_t* mask,
                       int device, void* stream);

/* Observations of the agents of SgEnvSpec (see there) for the scenarios with mask[n] != 0 (NULL: all):
   obs [N][A][F] fp32 (computed in fp64, rounded once), agent_mask [N][A] (the slot exists and is present),
   and the snapshot the next sg_env_reward compares against.  Rows of other scenarios are not written. */
int sg_env_observe(const SgScene* scene, const SgParams* params, const SgState* state, const SgEnvSpec* spec,
                   const uint8_t* mask, float* obs, uint8_t* agent_mask, int device, void* stream);

/* Rewards of one environment step, after the tick and before any reset: reward [N][A], terms [N][A][5]
   (fp32).  For the scenarios whose done flag is set (an environment steps only scenarios that are not
   done, so: the ones this tick finished) terminated [N] = a collision / ego_collision / ego_off_road
   condition of params->terminal holds at this tick, truncated [N] = otherwise (max_length); both are 0
   for the other scenarios.  The conditions are recomputed from the state as the tick decided them:
   collision = n_pair_ticks grew since the snapshot, ego_collision = collided[first_slot],
   ego_off_road = first_slot absent or not strictly inside the driveable surface.
   After several ticks (a branch forked with sg_fork_state and rolled out H ticks) the same evaluation, done
   once, scores the horizon against the state at the fork: progress = dist_H - dist_0, collision = collided
   rose at some tick of the horizon (it is sticky), off_road / tracking at the end state (frozen once the
   scenario is done), rss = flags gained over the horizon, terminated / truncated = how a scenario that
   finished within the horizon finished.  That is not the sum of the per-tick rewards; with H = 1 it is the
   reward of one environment step. */
int sg_env_reward(const SgScene* scene, const SgParams* params, const SgState* state, const SgEnvSpec* spec,
                  float* reward, float* terms, uint8_t* terminated, uint8_t* truncated, int device,
                  void* stream);

/* Fork: copy the state of every scenario of `src` into each of the n_dst states dst[0..n_dst), which must be
   allocated for the same scene (same N, M: the states do not carry their sizes, so this cannot be checked here)
   and must not overlap `src` or each other.  Copied: every per-slot plane and per-scenario field of SgState
   (pose, vel, dist, present, t, prev_t, tick, done, speed, goal_idx, force, cur_own, cur_union, ego_avg_speed,
   ego_avg_t, ego_max_speed, ego_dist, ego_hits, collided, first_coll_tick, first_coll_pair, n_pair_ticks,
   rss_state, rss_last, safe_dist, safe_ratio, rss_flags, pid_err; coll_mask for each destination where both
   sides have one, i.e. non-NULL).  Every destination's event_count is set to 0; events are not copied.  Every
   destination's trace_cap must be 0 (traces are not copied); the source's trace is ignored.
   src_spec / dst_spec (both NULL or both given, same n_agents): the snapshot arrays of SgEnvSpec (snap_dist,
   snap_collided, snap_pair_ticks, snap_rss) are copied the same way, so sg_env_reward of a destination compares
   against the source's snapshot.  A scenario window (SgScene.plane_stride) applies to the source and every
   destination alike.  One launch per 64 destinations: each element of the source is read once per launch and
   stored to every destination.  A rollout of a destination then continues exactly as the source would have:
   the state is all the tick kernels read. */
int sg_fork_state(const SgScene* scene, const SgState* src, SgState* const* dst, int n_dst,
                  const SgEnvSpec* src_spec, SgEnvSpec* const* dst_spec, int device, void* stream);

/* MPPI planning over the branch action tables (model-predictive path integral: sample perturbed action sequences,
   weight each by exp(reward / lambda), move the mean to the weighted average).  With A = spec->n_agents, agent a
   of scenario n is slot s = spec->agent_slot[n*A + a] (s = -1: padding, never read or written here).  The mean
   mu [N][H][A][2] is fp64, component c = 0 accel, 1 steer.  `table` is the flat branch action table
   [B][H][2][N*M] that sg_rollout consumes per branch (table_b = table + b*H*2*N*M): fp32, or fp64 with
   table_is_f64 != 0.  All arrays are device memory but `sigma` (host, [2]).

   sg_plan_sample: for every real agent, branch b and tick h, with i = ((n*A + a)*B + b)*H + h (int64) and
   (z0, z1) = the engine's counter-based N(0, 1) pair of (seed, i, k) (splitmix64 + Box-Muller, the SocialForce
   noise of SgParams.sf_std_*), eps_c = sigma_c * z_c for b >= 1 and 0 for b = 0 (branch 0 is the mean):
     table_b[h][c][n*M + s] = mu[n][h][a][c] + eps_c, rounded once to the table's type.
   No other table entry is written and nothing is clipped (the VehicleController clips actions).  Scenarios with
   reset[n] != 0 (reset NULL: none) have their mean zeroed first.  sigma finite and >= 0, k >= 0.

   sg_plan_update: reward [B][N][A] fp32 (sg_env_reward of each branch after its H ticks).  In fp64, summing in
   ascending b: Rmax = max_b R_b, w_b = exp((R_b - Rmax) / lambda), eps_hat_b = (double)table_b[h][c][n*M + s]
   - mu_in[n][h][a][c] (the noise is read back from the table, not stored), mu' = mu_in + (sum_b w_b eps_hat_b) /
   (sum_b w_b).  best_branch [N][A] int32 = the smallest b with R_b = Rmax, best_reward [N][A] = Rmax.
   finish = 0: mu_out = mu'.  finish != 0 (the last iteration of a planning step): action [N][A][2] fp32 =
   mu'[n][0][a], and mu_out holds the mean of the next step, shifted one tick: mu_out[h] = mu'[h + 1],
   mu_out[H-1] = 0.  mu_in and mu_out must not overlap; lambda finite and > 0. */
int sg_plan_sample(const SgEnvSpec* spec, int n_scenarios, int n_slots, int n_branches, int horizon, uint64_t seed,
                   int k, const double* sigma, double* mu, const uint8_t* reset, void* table, int table_is_f64,
                   int device, void* stream);
int sg_plan_update(const SgEnvSpec* spec, int n_scenarios, int n_slots, int n_branches, int horizon, double lambda,
                   const float* reward, const void* table, int table_is_f64, const double* mu_in, double* mu_out,
                   int finish, float* action, int32_t* best_branch, float* best_reward, int device, void* stream);

/* n_ticks x ScenarioGym.step() fused on device (scenario_gym.py:227-254): agents /
   batch replay -> State.step -> RSSDistances -> terminal check -> metrics.  Scenarios
   that are done are skipped.  n_ticks < 0: run every scenario to is_done
   (ScenarioGym.rollout, scenario_gym.py:256-267), bounded by params->max_ticks. */
int sg_rollout(const SgScene* scene, const SgParams* params, SgState* state,
               const SgInputs* inputs, int n_ticks, int device, void* stream);

/* FutureCollisionDetector._step (sensor/common.py:88-105) for a whole batch: does the box of
   slot `slot[n]` (NULL: the scenario's ego) meet the box of any other entity of scenario n at
   one of the times numpy.linspace(t[n], t[n] + horizon, n_samples), every entity placed at
   trajectory.position_at_t(time) (clamped at the trajectory ends, present or not)?
   t [N], slot [N] or NULL, out [N] (0 / 1): device memory. */
int sg_future_collisions(const SgScene* scene, const double* t, const int32_t* slot, double horizon,
                         int n_samples, uint8_t* out, int device, void* stream);

/* Materialise rows [tick0, tick0 + n_ticks) of the action table an SgActionRng describes:
   out [n_ticks][2][nm], device memory.  (Used for scenes the fused vehicle kernel does not take,
   and by the tests that pin the device stream against numpy.) */
int sg_fill_random_actions(const SgActionRng* rng, int tick0, int n_ticks, int64_t nm, double* out,
                           int device, void* stream);

/* State.get_entities_in_radius (state/state.py:352-372) for a whole batch: out[n*M + s] = 1 iff slot s
   of scenario n is present and its position lies strictly inside Point(x[n], y[n]).buffer(r[n]) --
   GEOS' 64-gon, the predicate of the pedestrians' sensor.  Scenarios with r[n] <= 0 are skipped
   (their rows are zeroed).  x, y, r [N], out [N*M]: device memory. */
int sg_entities_in_radius(const SgState* state, int n_scenarios, int n_slots, const double* x, const double* y,
                          const double* r, uint8_t* out, int device, void* stream);

/* BatchReplayEntity.add_entities (entity/batch.py:80-112) on the device: fill scene->union_x
   [n_union_rows][6][M] from the replayed slots' own control points (traj_off / traj_rows) resampled,
   clamped, at the union knot times union_t -- the rows packing.build_union_table computes on the host,
   bit for bit (trajectories with finite values; the reference passes the data through
   numpy.nan_to_num first).  All pointers device memory.  sg_rollout_host calls it when the host scene
   carries union_t but no union_x: the table is 6 M times the size of its knot times and need not cross
   PCIe. */
int sg_build_union_x(const SgScene* scene, int device, void* stream);

/* Measurement aid for the secondary roofline (bench.py): DFMA thread-instructions per second this
   GPU sustains at its current clocks (8 independent chains per thread, all SMs, best of 3 timed
   launches with CUDA events on `stream`).  Blocking. */
int sg_measure_fp64_peak(double* inst_per_s, int device, void* stream);

/* exact closed-set intersection test of oriented boxes (entity/base.py:100-138 +
   utils.py:28-62), for unit tests: poses [n][3] = x,y,h ; boxes [n][4] ; out[n] */
int sg_test_box_pairs(const double* pose_a, const double* box_a, const double* pose_b,
                      const double* box_b, uint8_t* out, int64_t n, int device, void* stream);

/* Trajectory.position_at_t / velocity_at_t on the device, for unit tests (trajectory.py:142-205,
   243-273): rows [K][7] = t, x, y, z, h, p, r; t [n]; mode 0 extrapolate=False (None outside the time
   range), 1 extrapolate=(False, False) (clamped), 2 extrapolate=True; pos [n][6], ok [n] (0: None),
   vel [n][6] or NULL.  All device memory. */
int sg_test_trajectory(const double* rows, int64_t K, const double* t, int64_t n, int mode, double* pos,
                       uint8_t* ok, double* vel, int device, void* stream);

/* Host-buffer entry point (the end-to-end number): copy the scene / initial inputs H2D (pinned host
   memory recommended), reset, roll every scenario out to completion and copy the per-scenario results
   back, all enqueued on `stream`.  `dev_*` are device mirrors with the same shapes.
   - copy_static = 0: the device scene is already up to date, nothing but the action table is copied.
   - An action table (host_inputs->actions / actions_f32) is streamed in chunks of 16 ticks, each chunk's
     copy overlapping the previous chunk's rollout; with host_inputs->use_rng the actions are drawn on the
     device and nothing but the scene crosses PCIe.
   - Without a table the batch is uploaded in windows of scenarios (SgScene.plane_stride) on an internal
     copy stream and every window is reset and rolled out as soon as it has arrived (scenes of 8 MiB or
     more: four windows ending at 1/32, 1/8, 1/2, 1 of the batch (under 4096 scenarios three, from 1/8 on), or -- replay-only scenes, whose rollout costs
     less than their upload -- five ending at 1/8, 3/8, 5/8, 7/8, 1, so that only a small last window's
     rollout is left when the upload ends; the environment variable SG_HOST_WINDOWS = 1 .. 6 overrides the
     number): the results equal the one-piece rollout's bit for bit, the upload hides behind the rollout.
   - host_scene->union_x = NULL with union_t present: the union table is built on the device
     (sg_build_union_x) instead of being uploaded. */
typedef struct SgHostResults {
  double* ego_avg_speed;    /* [N] */
  double* ego_max_speed;    /* [N] */
  double* ego_dist;         /* [N] */
  int32_t* first_coll_tick; /* [N] */
  int32_t* first_coll_pair; /* [N][2] */
  int64_t* n_pair_ticks;    /* [N] */
  uint8_t* rss_flags;       /* [N] */
  int32_t* tick;            /* [N] */
  double* t;                /* [N] */
  int32_t* event_count;     /* [1] */
} SgHostResults;

int sg_rollout_host(const SgScene* host_scene, const SgScene* dev_scene, const SgParams* params,
                    SgState* dev_state, const SgInputs* host_inputs, const SgInputs* dev_inputs,
                    SgHostResults* host_results, int copy_static, int device, void* stream);

/* bytes moved by sg_rollout_host per call (for the e2e report) */
int64_t sg_host_h2d_bytes(const SgScene* host_scene, const SgInputs* host_inputs, int copy_static);
int64_t sg_host_d2h_bytes(const SgScene* host_scene);

#ifdef __cplusplus
}
#endif
#endif /* SG_B200_H */
