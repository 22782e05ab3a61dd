// car_common.cuh -- device-side layout of the batched cCarRacing simulator (sm_100a).
//
// Reference path being replaced (paths relative to /root/reference/competitive_rl/):
//   car_racing/car_dynamics.py              Car (hull + 4 wheels + 4 revolute joints), wheel model
//   car_racing/car_racing_multi_players.py  CarRacing.step/reset, FrictionDetector, _create_track, renderer
//   box2d-py ~=2.3.5 (un-vendored)          b2World.Step(1/50, 180, 60) for 5 bodies + 4 joints per car
//
// One thread per CAR runs the whole per-step pipeline (controls, wheel model, sensor contacts,
// 180+60-iteration joint solver) with its island in registers; one CTA per (env, player) rasterises
// the 96x96 observation.  Everything below is per shard (one crl_car handle, one GPU).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "pong_common.cuh"   // philox4x32_10

namespace crl {

constexpr int CAR_W = 96, CAR_H = 96, CAR_PIX = CAR_W * CAR_H;
constexpr int CAR_MAX_TRACK = 512;          // tiles per track (standard tracks: 230-330)
constexpr int CAR_MAX_PLAYERS = 2;
constexpr int CAR_CHECKPOINTS = 12;
constexpr int CAR_DRAWS = 2 * CAR_CHECKPOINTS;   // np_random.uniform draws per _create_track attempt
constexpr int CAR_SAMPLE_STRIDE = 8;        // every 8th track point feeds the contact prefilter
constexpr int CAR_MAX_SAMPLES = CAR_MAX_TRACK / CAR_SAMPLE_STRIDE;
constexpr int CAR_MAX_STACK = 8;
constexpr int CAR_MAX_ROTATION = 16;       // registered observation buffers of the ahead-write stack mode
constexpr int CAR_GLYPH_BYTES = 11 * 8 * 4 + 11;
// the painted road map of a track, kept as a sparse raster (car_spans.cuh): 16 x 16 px blocks of the 2048 x 2048 px window
// of the reference's 10 000 x 10 000 px surface that starts at road-map pixel CAR_MAP_ORIGIN on both axes
constexpr int CAR_MAP_BLOCK = 16, CAR_MAP_GRID = 128, CAR_MAP_ORIGIN = 5000 - 1032;
constexpr int CAR_MAP_MAX_BLOCKS = 768;     // blocks a track may paint (standard tracks: 260-450); 192 KB per track slot
constexpr int CAR_MAX_CONTACTS = 8;         // touching car-car fixture pairs kept per env (of 48 possible)
constexpr int CAR_RAW_RING = 1024;          // raw points of the curve follower kept while it walks (last lap + tail)
// Tiles of a track that the wheel-tile prefilter's constant radii do not cover (sensor_wheel_overlaps): a vertex farther
// than CAR_WIDE_REACH from the tile's track point, or a track point farther than CAR_WIDE_GROUP from its group's sample
// point.  Generated tracks have one, the seam tile 0 (its gap along the track is up to ~14.5 units against 3.5 elsewhere);
// recorded tracks with more than CAR_MAX_WIDE are refused by crl_car_load_tracks.
constexpr int CAR_MAX_WIDE = 4;
constexpr float CAR_WIDE_REACH = 8.3f;      // 9 (wheel radius of the prefilter) - 0.6083 (wheel circumradius) - 2 skins, less slack
constexpr float CAR_WIDE_GROUP = 24.9f;     // 36 (sample radius) - 11 (track point to hull of a touching wheel), less slack

// A road tile, 124 bytes: for the physics the convex hull (CCW, fp32) of the reference's 5 listed
// vertices, with the edge normals the sensor-overlap test needs; for the renderer the listed vertices and the kerb quad in ROAD-MAP PIXELS, i.e.
// (int)(obs_scale * -v + 5000) of the fp64 vertex as pygame truncates it (render_road_for_observation_map).
struct CarTile {
    float px[5], py[5];       // hull vertices (n of them)
    float nx[5], ny[5];       // outward unit normals of the hull edges i -> i + 1 (nx = 3e38: degenerate edge)
    uint8_t n, flags;         // flags: 1 = exists, 2 = has kerb, 4 = white kerb (block_id even)
    uint16_t pad;
    float cx, cy;             // track point (x, y): centre used for culling
    int16_t mx[5], my[5];     // listed vertices l1, m, r1, r2, l2 in road-map pixels
    int16_t kmx[4], kmy[4];   // kerb quad in road-map pixels
};

// One touching fixture pair between the two cars of an env (b2Contact + its solver constraints), 160 bytes.
// The manifold part and the accumulated impulses persist between steps (warm start); the rest is per-step scratch.
struct __align__(16) CarContact {
    uint8_t pair, count, type, vcount;   // canonical pair index (0..47), manifold points, 0 = e_faceA / 1 = e_faceB, solver points
    uint8_t ia, ib, pad0, pad1;          // bodies: 0..4 = car 0 (hull, wheels 0..3), 5..9 = car 1
    uint32_t id[2];                      // b2ContactFeature keys
    float lnx, lny, lpx, lpy;            // manifold.localNormal, manifold.localPoint
    float px[2], py[2];                  // manifold.points[].localPoint
    float ni[2], ti[2];                  // normal / tangent impulses
    float nx, ny;                        // world normal
    float rAx[2], rAy[2], rBx[2], rBy[2];
    float nmass[2], tmass[2];
    float k11, k12, k22, nm00, nm01, nm10, nm11;
};

struct CarHullConst {         // mass data of the car bodies (b2Body::ResetMassData), computed on the host
    float hull_inv_mass, hull_inv_I, hull_lcx, hull_lcy;
    float wheel_inv_mass, wheel_inv_I;
    // body-local fixture polygons as b2PolygonShape::Set leaves them (hull order, edge normals, centroid):
    // 0..3 = the hull's four polygons, 4 = the wheel box; radius = farthest vertex from the body origin
    int fix_n[5];
    float fix_vx[5][8], fix_vy[5][8], fix_nx[5][8], fix_ny[5][8];
    float fix_cx[5], fix_cy[5], fix_radius[5], fix_cradius[5];   // cradius = farthest vertex from the centroid
    uint8_t gray[16];         // palette: see CarGray
    int checker[80];          // [axis][20][lo, hi]: road-map pixel bounds of the checker squares (car_checker_table)
};
enum CarGray { G_GRASS = 0, G_CHECK, G_ROAD0, G_ROAD1, G_ROAD2, G_KERB_W, G_KERB_R, G_WHEEL, G_OWN, G_OTHER, G_HUD,
               G_BLUE, G_BLUE2, G_GREEN, G_RED, G_TEXT };

struct FrameMap;              // per-frame camera / screen -> road-map mapping (car_raster.cu)

struct CarDev {
    int n;                    // envs in this shard
    int players;              // 1 = cCarRacing-v0, 2 = cCarRacingDouble-v0
    int c;                    // frames per player in the observation (frame_stack or 1)
    int action_repeat;
    int max_episode_steps;    // gym TimeLimit of the registry entry (1000); 0 = none
    // stack_mode 1: the observation buffer is a double-write ring [n][players][2c][96][96]: the new frame goes to slots
    // ring_phase and ring_phase + c, the observation is the strided view of slots ring_phase + 1 .. ring_phase + c
    int ring_mode;
    int ring_phase;           // host-tracked, advanced per step
    int fill_all;             // 1 after reset(): every frame written goes to all slots
    // stack mode over a rotation of B >= C + 1 registered observation buffers (crl_car_set_obs_rotation): the k-th call
    // after a reset returns buffer (k mod B), and every new frame is written straight into the C buffers it will appear
    // in -- channel C-1 of the current one, C-2 of the next, ... -- so no frame is ever moved and no ring is kept
    uint8_t* rot[CAR_MAX_ROTATION];
    int rot_n;                // 0 = not registered
    int rot_pos;              // host-tracked: index of the buffer the current call returns
    int done_mode;            // 0 = any car done (FlattenMultiAgentObservation), 1 = car 0 only (make_competitive_car_racing)
    int64_t first_env;
    uint64_t seed;
    // ---- per track SLOT: every env owns two, slot = env + n * sel[env] is the track it drives on, the other one
    //      receives the NEXT track ahead of time (car_pregen_kernel on a side stream), so that an auto-reset is a
    //      slot swap + car spawn instead of a serial 2500-step curve walk on the step's critical path ----
    int32_t* n_track;         // [2n]
    CarTile* tiles;           // [2n][CAR_MAX_TRACK]
    float2* samples;          // [CAR_MAX_SAMPLES][2n] every 8th track point (transposed: coalesced per-thread scans)
    double* start_pose;       // [2n][3] beta, x, y of track[0]
    double* track_pts;        // [2n][CAR_MAX_TRACK][3] beta, x, y of the track (fp64, as generated)
    // ---- per env ----
    int32_t* sel;             // [n] which of its two slots env e currently drives on
    int32_t* next_state;      // [n] the other slot: 0 = empty, 1 = being generated, 2 = holds the next track
    int32_t* next_att0;       // [n] attempt_count before the next track was generated (restored when it is discarded)
    double* raw_ring;         // [n][CAR_RAW_RING][3] scratch of the generator: the last raw points of the walk
    int32_t* step_count;      // [n] CarRacing.step_count
    int32_t* elapsed;         // [n] TimeLimit._elapsed_steps
    int32_t* reset_count;     // [n] resets so far (RNG / injection cursor)
    int32_t* attempt_count;   // [n] track attempts so far (injection cursor)
    float* inv_dt0;           // [n] b2World::m_inv_dt0
    uint8_t* env_done;        // [n] done flag of the LAST step (what the vec-env saw)
    int32_t* ring_pos;        // [n] newest slot of the frame ring
    // ---- per car (index = env * players + player), all [n*players] unless noted ----
    float* body;              // [n*players][5][8]: cx, cy, a, vx, vy, w, sleep_time, awake   (0 = hull, 1..4 = wheels)
    float* joint;             // [n*players][4][6]: impulse x, y, z, motor impulse, limit state, motor speed
    double* wheel;            // [n*players][8]: omega[4], gas[2] (rear), brake, steer
    double* reward;           // [n*players][2]: reward, prev_reward
    int32_t* counters;        // [n*players][4]: tile_visited_count, last_block, has_block, done
    uint32_t* touching;       // [n*players][4][16] wheel.tiles bitmasks
    uint32_t* visited;        // [n*players][16] tile.road_visited[car]
    uint32_t* sensor_now;     // [n*players][4][16] tiles each wheel overlaps at the start of the step (car_sensor_kernel)
    // ---- car-car contacts (players == 2): [n][CAR_MAX_CONTACTS] records, [n] counts, one overflow counter ----
    CarContact* contacts;
    int32_t* n_contacts;
    int32_t* n_contacts_step;    // [n] contacts the last executed (sub-)step worked with: the diagnostic of crl_car_get_contacts
    int32_t* contact_overflow;
    // two-pass stepping of two-car envs (car_step_kernel modes 1 / 2): envs whose cars are near each other
    int32_t* slow_list;       // [n] envs with a touching pair of fixtures this step (car_collide_kernel): merged islands
    int32_t* slow_count;      // [1]
    int32_t* near_list;       // [n] envs whose cars are near each other (oriented-box gate of the sensor kernel)
    int32_t* near_count;      // [1] = slow_count + 1: both cleared by one memset
    uint8_t* deferred;        // [n] 1 = on the slow list this step
    // envs that finished in this step, listed by the post-step render passes (collect_done = 1) so that the auto-reset
    // kernels run over the list instead of launching a thread block per env
    int32_t* done_list;       // [n]
    int32_t* done_count;      // [1] cleared at the start of every step
    int collect_done;
    // ---- per slot: the painted road map (it depends on the track only, so it is painted once per track by the generator
    //      instead of once per frame): block index [2n][CAR_MAP_GRID][CAR_MAP_GRID], block pool [2n][CAR_MAP_MAX_BLOCKS][256] ----
    uint16_t* map_index;
    uint8_t* map_blocks;
    const uint8_t* chk;       // [2][2048] 0xFF where map column (axis 0) / row (axis 1) CAR_MAP_ORIGIN + i lies in a checker square (:733-746)
    float2* tile_centres;     // [2n][CAR_MAX_TRACK] tile centres (= CarTile::cx, cy), contiguous for the step kernel's candidate search
    float4* wide_tiles;       // [2n][CAR_MAX_WIDE] tiles the prefilter radii miss: track point x, y, reach, tile id (reach < 0: unused)
    // ---- per frame (env * players + player): written by car_frame_setup_kernel, read by car_render_kernel ----
    FrameMap* frame_map;      // [n*players]
    uint8_t* frame_aux;       // [n*players] FrameAux records (car polygon span tables, road-map block list)
    // ---- observation ring: [n][players][c][CAR_PIX] ----
    uint8_t* ring;
    // ---- validation mode ----
    const double* track_draws;   // [n][k_draws][CAR_DRAWS] or nullptr
    int k_draws;
    const int32_t* birth;        // [n][k_birth][players] or nullptr
    int k_birth;
    // fixed tracks (CarRacing.reset(use_local_track=...), car_racing_multi_players.py:376-381): env e replays track
    // e % n_fixed at every reset instead of generating one
    const double* fixed_tracks;  // [n_fixed][CAR_MAX_TRACK][3] beta, x, y or nullptr
    const int32_t* fixed_counts; // [n_fixed]
    int n_fixed;
    int32_t* overrun;            // [0] device flag: an injection table ran out; [1] road-map pixels / blocks dropped while painting a track
                                 // (outside the 2048 px window, block pool full); [2] frames with a car polygon scanned per pixel (> 16 rows)
                                 // [3] auto-resets that had to generate (or wait for) their track on the step's critical path
    // ---- constants ----
    const CarHullConst* consts;
    const uint8_t* glyphs;       // [CAR_GLYPH_BYTES]
    unsigned long long* stats;   // [0] episodes, [1] sum length, [2] sum tiles visited (player 0)
};

__device__ __forceinline__ int car_slot(const CarDev& p, int e) { return e + p.n * p.sel[e]; }

cudaError_t launch_car_reset(const CarDev& p, int only_done, cudaStream_t s);
cudaError_t launch_car_pregen(const CarDev& p, cudaStream_t s);        // next tracks of the envs that have none (side stream)
cudaError_t launch_car_discard_next(const CarDev& p, cudaStream_t s);  // forget pre-generated tracks (seed / injection changed)
// wheel-tile overlaps, before launch_car_step; classify = 1: also the slow list of the two-pass schedule (slow_count cleared before)
cudaError_t launch_car_sensors(const CarDev& p, int classify, cudaStream_t s);
// two-car envs: manifolds of the near envs, one thread per fixture pair; fills the slow list (after launch_car_sensors(classify = 1))
cudaError_t launch_car_collide(const CarDev& p, cudaStream_t s);
cudaError_t launch_car_step(const CarDev& p, int mode, const float* actions, float* rew, uint8_t* done, int32_t* num_steps,
                            uint8_t* truncated, cudaStream_t s);
// which: 0 = every frame, 1 = envs not deferred to the slow stepping pass, 2 = deferred envs only; advance: move the frame ring on
cudaError_t launch_car_render(const CarDev& p, int only_done, int which, int advance, uint8_t* obs, uint8_t* term_obs, cudaStream_t s);
// stack mode: the C - 1 frames that stay in the observation, ring -> obs; before the render passes of a step (not after a reset)
cudaError_t launch_car_stack_shift(const CarDev& p, uint8_t* obs, cudaStream_t s);
cudaError_t launch_car_ring_advance(const CarDev& p, cudaStream_t s);
cudaError_t car_raster_init();
size_t car_frame_map_bytes();
size_t car_frame_aux_bytes();
void car_checker_table(int* out);
cudaError_t launch_car_get_state(const CarDev& p, double* state, cudaStream_t s);
cudaError_t launch_car_set_state(const CarDev& p, const double* state, cudaStream_t s);
cudaError_t launch_car_random_actions(float* actions, int n_values, uint64_t seed, uint64_t step, cudaStream_t s);

}  // namespace crl
