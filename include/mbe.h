/*
 * mbe.h -- C ABI of libmbe.so: batched, GPU-resident replacement for the per-step hot path
 * of mobile-env (reference fork yang-peilin/mobile-env-gan), i.e. MComCore.step over N
 * independent environments (reference mobile_env/core/base.py:230-296).
 *
 * The reference is pure Python and has no FFI; the entry points below are what a binding
 * for this path would need (INTEGRATION.md shows the ctypes stub a maintainer would add to
 * mobile_env/core/base.py).  Each entry cites the reference code it replaces.
 *
 * Conventions
 *   - plain C types only; every pointer inside mbe_buffers is a DEVICE pointer owned by the
 *     caller (e.g. torch tensors) and must stay alive while bound;
 *   - all calls are stream-ordered on the given cudaStream_t (passed as void*), enqueue
 *     only, never synchronise (except the *_host convenience entry, which says so);
 *   - return 0 on success, non-zero on error; mbe_last_error() gives a thread-local text;
 *   - a handle belongs to the device named in mbe_config.device; every call makes that device current
 *     for its duration and restores the caller's current device before returning;
 *   - a handle is not thread-safe, different handles are.
 *
 * Shapes: U <= 32 and B <= 32 run on the warp-segment kernels (an env is a slice of a warp; the
 * scenario shapes have fused compile-time variants: several UEs per thread for 15 x 4, a thread per
 * env for the fork's 7 UEs x 10 per-env BS slots -- mbe_step_kernel_name() tells which);
 * 32 < U <= 1024 or 32 < B <= 64, and the ProportionalFair / RateFair schedulers, run on the
 * block-per-env kernel (every entry point; needs width^2 + height^2 < 2^24).
 *
 * Data layout (structure of arrays, env-major; E = envs on this rank, U = UEs, B = BS slots,
 * MW = ceil(B/32), F = 2B+1 (central) or 4B+1 (multi-agent)):
 *   pos      int16 [E,U,2]   UE position (integers after the first move, movement.py:60)
 *   wp       int16 [E,U,2]   current waypoint; x < 0 = none (movement.py:44-47,54-56)
 *   t        int32 [E]       step clock of the episode (base.py:280, "time")
 *   episode  int32 [E]       episode counter (-1 before the first reset)
 *   bs_xy    int16 [B,2] or [E,B,2]  int-truncated BS coordinates (entities.py:24-26); a shared
 *                            [B,2] layout is read once by mbe_bind (re-bind after editing it)
 *   nbs      int32 [E]       live BS slots per env (random layouts, custom.py:68-77) or NULL
 *   conn     uint32 [E,U,MW] GYM: connection bitmask (bs2ue_connections, base.py:76)
 *   assoc    int32 [E,U]     FORK: BS index the UE is attached to, -1 = none (base.py:236-241)
 *   actions  int32 [E,U]     GYM: 0 = NOOP (base.py:29), a>0 toggles BS a-1
 *   rate     f64  [E,U]      per-UE total of the 2-decimal-rounded pair rates (base.py:413-435)
 *   utility  f32  [E,U]      scaled utility in [-1,1] (utilities.py:44-55; base.py:253-258)
 *   obs      f32  [E,U,F]    GYM observation written straight into the policy input
 *   reward   f32  [E] (central) or [E,U] (multi-agent)
 *   done     uint8 [E]       time_is_up (base.py:407-409)
 *   metrics  f32  [E,4]      number connections, number connected, mean utility, mean
 *                            datarate (metrics.py:5-28)
 */
#ifndef MBE_H_
#define MBE_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MBE_ABI_VERSION 2

enum { MBE_MODE_FORK = 0, MBE_MODE_GYM = 1 };
enum { MBE_HANDLER_CENTRAL = 0, MBE_HANDLER_MA = 1 };
enum { MBE_SCHED_RESOURCE_FAIR = 0, MBE_SCHED_PROPORTIONAL_FAIR = 1, MBE_SCHED_RATE_FAIR = 2 };
enum { MBE_BS_SHARED = 0, MBE_BS_PER_ENV = 1 };
enum { MBE_MAX_CLASSES = 16 };   /* link classes = BS classes x UE classes */
enum { MBE_MAX_UE_CLASSES = 8 };
/* mbe_config.flags */
enum {
  MBE_FLAG_GENERIC_KERNEL = 1,    /* never use the shape-specialised fused kernels */
  MBE_FLAG_SHARED_TRAJECTORY = 2, /* all envs draw the SAME UE initial positions and waypoints (the fork: movement
                                     reset_rng_episode=True makes every epoch replay one UE trajectory, base.py:130-134;
                                     with env index = epoch number only the BS layouts differ) */
};

/* phases of one step (bit mask for mbe_stage); the fused step runs all of them in one launch.
 * FORK order: MOVE, PRE, CLOCK.  GYM order: PRE, MOVE, CLOCK, POST. */
enum {
  MBE_PHASE_MOVE = 1,  /* RandomWaypointMovement.move         movement.py:42-62            */
  MBE_PHASE_PRE = 2,   /* connectivity / association / action, scheduler split, utility,
                          reward, metrics                     base.py:212-258, 421-435     */
  MBE_PHASE_CLOCK = 4, /* time += 1, departures, done          base.py:280-291, 407-409     */
  MBE_PHASE_POST = 8,  /* observation writer (GYM)                                          */
  MBE_PHASE_ALL = 15
};

/* One LINK class: all (BS, UE) pairs whose BS shares bw/freq/tx/height (entities.py:6-29) and whose UE
 * shares snr_threshold/noise/height (entities.py:32-57).  Link class of the pair (b, u) =
 * bs_class[b] * num_ue_classes + ue_class[u].  The tables are folded on the host in FP64 from the
 * channel's power_loss (channels.py:18-21, 132-146) through Channel.calculateSNR (channels.py:24-27),
 * evaluated at the integer offsets that realise each squared distance d2 (entities.py:24-26,52-54):
 *    d2max        largest d2 with snr > snr_threshold (base.py:212-214), -1: never connectable;
 *    rate_lut     HOST pointer, d2max+1 doubles, copied by mbe_create: Channel.datarate =
 *                 bw*log2(1+snr) (channels.py:78-83);
 *    log2(snr(d2)) for the FP32 observation path: l0 - k*log2(d2) for d2 >= 1 and l_zero for
 *                 d2 == 0 (EPSILON, channels.py:8) when log2snr_lut is NULL, else the table
 *                 log2snr_lut[d2] (HOST pointer, log2snr_len floats covering every d2 of the map,
 *                 copied by mbe_create) for losses that are not affine in log-distance. */
typedef struct mbe_link_class {
  double l0;
  double k;
  double l_zero;
  int32_t d2max; /* -1: never connectable */
  int32_t log2snr_len;
  const double* rate_lut;
  const float* log2snr_lut;
} mbe_link_class;
typedef mbe_link_class mbe_bs_class; /* ABI 1 name */

/* One UE class: the movement parameters of the UEs that share a parameter set (entities.py:32-57) */
typedef struct mbe_ue_class {
  double velocity;    /* ue.velocity (base.py:119) */
  int32_t move_d2max; /* largest integer d2 with sqrt(d2) <= velocity (movement.py:54) */
  int32_t reserved;
} mbe_ue_class;

typedef struct mbe_config {
  int32_t abi_version; /* MBE_ABI_VERSION */
  int32_t device;      /* CUDA device ordinal */
  int32_t num_envs;    /* E on this rank */
  int32_t num_ues;     /* U */
  int32_t num_bs;      /* B (slots) */
  int32_t mode;        /* MBE_MODE_* */
  int32_t handler;     /* MBE_HANDLER_* (GYM) */
  int32_t scheduler;   /* MBE_SCHED_* */
  int32_t bs_layout;   /* MBE_BS_* */
  int32_t bs_random_min, bs_random_max; /* >0: reset draws nbs in [min,max] and their
                                           coordinates per env and episode (custom.py:68-77) */
  int32_t autoreset;   /* GYM/FORK: re-initialise an env in the step that ends its episode */
  int32_t reset_rng_episode; /* movement_params.reset_rng_episode (base.py:130-134) */
  int32_t ep_time;     /* min(EP_MAX_TIME, max departure) (base.py:407-409) */
  int32_t move_d2max;  /* largest integer d2 with sqrt(d2) <= velocity (movement.py:54) */
  int64_t env_offset;  /* global id of local env 0 (multi-GPU sharding; Philox counters use it). Global env ids are
                          one 32-bit counter word: 0 <= env_offset and env_offset + num_envs <= 2^32 - 1, else
                          mbe_create fails (4.29e9 envs across the job) */
  uint64_t seed;       /* movement seed = config seed + 4 (base.py:155-170) */
  double width, height;/* map (base.py:103) */
  double velocity;     /* ue.velocity (base.py:119) of UE class 0 */
  double util_lower, util_upper, util_w1, util_w2, util_w3; /* utilities.py:30-55 */
  int32_t num_classes; /* number of BS classes, >= 1; num_classes * max(1, num_ue_classes) <= MBE_MAX_CLASSES */
  int32_t flags;       /* MBE_FLAG_* */
  mbe_link_class classes[MBE_MAX_CLASSES]; /* [bs class][ue class], ue class fastest */
  const uint8_t* bs_class; /* HOST [B] class id per BS slot, or NULL = all class 0 */
  int32_t num_ue_classes;  /* 0 or 1: all UEs alike (velocity / move_d2max above); else 2..MBE_MAX_UE_CLASSES */
  /* M: UE trajectories per BS layout.  0 or 1: the flags alone decide (MBE_FLAG_SHARED_TRAJECTORY: one
     trajectory for all envs).  M >= 2 needs MBE_FLAG_SHARED_TRAJECTORY, M a power of two, M <= num_envs,
     num_envs % M == 0 and env_offset % M == 0; env of global id g then follows trajectory g mod M (its BS
     layout draws still use g).  Convention: layout l occupies env rows l*M .. l*M + M-1 and replica m
     follows trajectory m, on every rank and in every env window.  mbe_evolve_layouts breeds L =
     num_envs / M layouts on such a handle. */
  int32_t num_trajectories;
  const uint8_t* ue_class; /* HOST [U] class id per UE (required when num_ue_classes > 1) */
  mbe_ue_class ue_classes[MBE_MAX_UE_CLASSES]; /* used when num_ue_classes > 1 */
} mbe_config;

typedef struct mbe_buffers {
  int16_t* pos;
  int16_t* wp;
  int32_t* t;
  int32_t* episode;
  int16_t* bs_xy;
  int32_t* nbs;          /* optional */
  uint32_t* conn;        /* GYM */
  int32_t* assoc;        /* FORK */
  const int32_t* actions;/* GYM */
  double* rate;          /* optional in GYM */
  float* utility;        /* required (carried between phases) */
  float* obs;            /* GYM */
  float* reward;         /* GYM */
  uint8_t* done;
  float* metrics;        /* optional */
  float* dbg_snr;        /* optional f32 [E,U,B]: SNR at the positions the PRE phase sees */
  /* replay of reference trajectories: waypoints injected instead of Philox draws */
  const int16_t* inj_wp; /* optional int16 [E,U,K,2] */
  int32_t* wp_cnt;       /* int32 [E,U] draws consumed so far (required with inj_wp) */
  int32_t inj_k;         /* K */
  int32_t reserved;
} mbe_buffers;

typedef struct mbe_env mbe_env;

/* library / build information */
int mbe_abi_version(void);
const char* mbe_build_info(void);
const char* mbe_last_error(void);
/* sizeof of the ABI structs as the library was compiled (0 mbe_config, 1 mbe_buffers, 2 mbe_link_class,
 * 3 mbe_ue_class, 4 mbe_rollout_out, 5 mbe_render_style, 6 mbe_evolve_params, 7 mbe_map_params; -1
 * otherwise): lets a
 * binding in another language check its layout */
int mbe_struct_size(int which);

/* replaces MComCore.__init__ (base.py:32-100): validates, copies the constant tables */
int mbe_create(const mbe_config* cfg, mbe_env** out);
void mbe_destroy(mbe_env* env);

/* binds caller-owned device buffers (the SoA state of entities.py:6-57 / base.py:69-79) */
int mbe_bind(mbe_env* env, const mbe_buffers* bufs);

/* replaces MComCore.reset + MComCustom.reset (base.py:172-209, custom.py:40-62) for the envs
 * whose mask byte is non-zero (DEVICE pointer, NULL = all): clock, initial positions
 * (movement.py:64-72), optional BS layout, cleared connections, reset observation. */
int mbe_reset(mbe_env* env, const uint8_t* env_mask, void* stream);

/* replaces MComCore.step (base.py:230-296): one fused launch over all bound envs */
int mbe_step(mbe_env* env, void* stream);

/* the same fused step for the envs [first_env, first_env + num_envs) only (first_env a multiple of
 * 32; envs are independent, base.py:69-79): lets one handle keep several env groups in flight on
 * different streams (step group A while a policy reads group B's observations) */
int mbe_step_window(mbe_env* env, int first_env, int num_envs, void* stream);

/* the same step split into phases (MBE_PHASE_* mask), for per-stage parity and profiling */
int mbe_stage(mbe_env* env, int phase_mask, void* stream);

/* Channel.calculateSNR for every UE x BS pair (channels.py:24-27): f32 [E,U,B] into out_snr,
 * connectable bitmask uint32 [E,U,MW] into out_elig (either may be NULL) */
int mbe_channel(mbe_env* env, float* out_snr, uint32_t* out_elig, void* stream);

/* recompute the observation of the current state (after the caller edited pos / conn) */
int mbe_observe(mbe_env* env, void* stream);

/* adds this step's two-decimal QoE values (base.py:269) to acc f32 [E,4] = (sum q, sum q^2,
 * #q < threshold, #values): the statistics of chooseBaseStation.ipynb cell 5 `qoeValue`.
 * The cent k of a value is the exact half-even rounding of its FP32 utility times 100, q is
 * float32(k / 100), and q counts as low when float32(k / 100) < float32(threshold).  That is Python's
 * round(u, 2) < t for every cent-valued t; a threshold that rounds to the same float32 as a cent acts as
 * that cent.  The counts are exact, the sums are FP32 in a fixed order (DESIGN.md section 2). */
int mbe_accumulate_qoe(mbe_env* env, float* acc, float threshold, void* stream);

/* per-step series of a fused episode: DEVICE pointers, any may be NULL; 16-byte aligned */
typedef struct mbe_rollout_out {
  int16_t* pos;   /* [T,E,U,2] positions after each step's move (what base.py:298-404 dumps per step) */
  int16_t* wp;    /* [T,E,U,2] waypoints after the move; (-1,-1) = arrived this step (movement.py:54-56) */
  int32_t* assoc; /* [T,E,U] serving BS or -1 (base.py:236-241) */
  double* rate;   /* [T,E,U] rounded data rates (base.py:435) */
  float* utility; /* [T,E,U] scaled utility = QoE (base.py:253-258) */
} mbe_rollout_out;

/* FORK mode: `steps` consecutive MComCore.step calls (base.py:230-296; the fork's collect loop
 * `for s in range(20): env.step(e, s)`) in ONE launch -- state stays on chip between the steps.
 * qoe_acc (f32 [E,4], may be NULL) accumulates the statistics of mbe_accumulate_qoe over all steps,
 * with the same cents and low-QoE test, bit for bit;
 * `out` (may be NULL) receives the per-step series.  After the call the bound buffers hold exactly
 * what `steps` calls of mbe_step would have left.  Shapes without the fused kernel run the same
 * episode as a sequence of step launches (same results). */
int mbe_rollout(mbe_env* env, int steps, float* qoe_acc, float threshold, const mbe_rollout_out* out, void* stream);

/* Map-panel frames (DESIGN.md section 9).  palette rows: 0 background, 1..3 coverage by 1 / 2 / >= 3
 * BSs, 4 BS square, 5 unconnected UE, 6..261 utility ramp (index clamp(floor((u + 1) * 128), 0, 255)). */
enum { MBE_RENDER_PALETTE = 262, MBE_RENDER_MAX_STYLE_PX = 64 };
typedef struct mbe_render_style {
  int32_t height, width;                  /* 8..4096, width % 4 == 0 */
  int32_t ue_radius, bs_half, line_width; /* pixels, 0..MBE_RENDER_MAX_STYLE_PX */
  uint8_t palette[MBE_RENDER_PALETTE][3]; /* RGB */
} mbe_render_style;

/* Frames of envs env_ids[0..n) (DEVICE int32, NULL = envs 0..n-1) into out uint8 [steps, n, H, W, 3]
 * (DEVICE, 4-byte aligned), one launch.  series == NULL: the bound state (steps must be 1).
 * series != NULL (FORK): the pos / assoc / utility series [steps, E, U(,2)] that mbe_rollout wrote,
 * one frame per step.  BS layouts, nbs and link classes are the handle's bound ones, so a series
 * should not cross an episode boundary.  An env id outside 0..E-1 gives a background-only frame. */
int mbe_render(mbe_env* env, const int32_t* env_ids, int n, const mbe_rollout_out* series, int steps,
               const mbe_render_style* style, uint8_t* out, void* stream);

/* One generation of a genetic search over per-env BS layouts (DESIGN.md section 10).  Philox key = seed,
 * counter (env_offset + child, generation, block, 3).  Probabilities are compared as r * 2^-32 < p. */
typedef struct mbe_evolve_params {
  uint64_t seed;
  uint32_t generation;
  int32_t tournament; /* candidates per tournament, 1..4 */
  int32_t step;       /* largest per-axis move, 0..32767 */
  int32_t reserved;
  double p_cross, p_move, p_add, p_del; /* each in [0, 1] */
} mbe_evolve_params;

/* Breeds child_xy int16 [E,B,2] / child_nbs int32 [E] from parent_xy / parent_nbs and fitness f32 [E]
 * (all DEVICE, 4-byte aligned; E, B and the layout ranges are the handle's, which needs random per-env
 * layouts).  Child c < n_elite copies parent elite_ids[c] verbatim when that id is in 0..E-1.  The
 * child buffers must not overlap any input.  One launch.  On a handle with num_trajectories = M >= 2 the
 * population is the L = num_envs / M layouts, not the env rows: every array above is [L, ...], n_elite
 * lies in 0..L, and the Philox child id is env_offset / M + child. */
int mbe_evolve_layouts(mbe_env* env, const float* fitness, const int16_t* parent_xy, const int32_t* parent_nbs,
                       const int32_t* elite_ids, int n_elite, const mbe_evolve_params* p, int16_t* child_xy,
                       int32_t* child_nbs, void* stream);

/* Layout maps (DESIGN.md section 10.2) of envs env_ids[0..n) (DEVICE int32, NULL = envs 0..n-1), with the
 * layout the step kernels see: the coordinates a shared layout had at mbe_bind, or the bound bs_xy[e] with
 * the live slots b < clamp(nbs[e], 0, B).  The grid points are (x, y) = (i*stride, j*stride) with
 * 0 <= x <= XM = ceil(width) - 1 and 0 <= y <= YM = ceil(height) - 1 (the range UE positions are drawn
 * from): GX = XM / stride + 1 columns, GY = YM / stride + 1 rows, row j is y = j*stride (y ascends with the
 * row, unlike a render frame), point index j*GX + i.  Per point, with d2 the exact integer squared
 * distance to a live BS and a BS connectable iff d2 <= d2max of link class (bs_class[b], ue_class):
 *   coverage  uint8 [n, GY, GX]  connectable BSs, saturated at 255;
 *   serving   int8  [n, GY, GX]  the connectable BS of smallest d2, ties to the lower slot (the FORK
 *                                association), -1 = none;
 *   qoe       int8  [n, GY, GX]  the cent k in [-100, 100] of a UE served there that shares its BS with
 *                                load - 1 others: the exact half-even rounding of 100 * scaled utility
 *                                (FP32, as the step kernels compute it) of the rate
 *                                nearbyint(rate_lut[d2] / load * 100) / 100 (FP64); -100 without a server.
 * stats int64 [n, 6] = (points, covered (>= 1 BS), overlap (>= 2 BSs), sum k, sum k^2, low), where a point is
 * low iff float32(k / 100) < float32(threshold), the test of mbe_accumulate_qoe; area int32 [n, B] = points
 * each slot serves.  An env id outside 0..E-1 gives zero stats and area, coverage 0, serving -1, qoe -128.
 * Every output may be NULL; stats 8-byte and area 4-byte aligned (DEVICE).  Two launches; leaves every bound
 * buffer untouched. */
typedef struct mbe_map_params {
  int32_t stride;   /* grid step in map units, >= 1 */
  int32_t ue_class; /* UE class of the map's UE, 0..num_ue_classes-1 */
  int32_t load;     /* UEs sharing the serving BS, >= 1 */
  int32_t reserved;
  float threshold;  /* low-QoE threshold, finite */
} mbe_map_params;

int mbe_layout_map(mbe_env* env, const int32_t* env_ids, int n, const mbe_map_params* p, int64_t* stats,
                   int32_t* area, uint8_t* coverage, int8_t* serving, int8_t* qoe, void* stream);

/* number of kernel launches this handle has enqueued so far */
int64_t mbe_launch_count(const mbe_env* env);

/* which kernel family mbe_step dispatches to for this handle's shape and bound buffers, e.g.
 * "step_upt_kernel" (several UEs per thread), "step_spec_kernel" (warp segment, compile-time shape),
 * "step_tpe_fork_kernel" (thread per env), "step_big_kernel" (block per env), "step_kernel" (generic) */
const char* mbe_step_kernel_name(const mbe_env* env);

/* Host-buffer convenience: H2D actions, step, D2H obs/reward/done, then synchronises the
 * stream.  Host pointers should be pinned.  NULL pointers are skipped.  Large batches with
 * observations are processed as env windows on two streams so uploads and the step overlap the
 * download. */
int mbe_step_host(mbe_env* env, const int32_t* actions_host, float* obs_host,
                  float* reward_host, uint8_t* done_host, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MBE_H_ */
