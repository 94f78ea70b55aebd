/* ssd_b200 -- C ABI of the B200-native batched SSD grid-world simulator
 * (Cleanup / Harvest) that replaces the env step + observation path of
 * drdh/Homophily-MARL.
 *
 * The reference has no FFI: its seam is the duck-typed PyMARL MultiAgentEnv
 * surface (src/envs/multiagentenv.py:6-75) implemented by MapEnv
 * (src/envs/ssd/map_env.py:874-1022) and reached through
 * src/envs/__init__.py:6-11 REGISTRY.  Every entry point below names the
 * reference method(s) it replaces; homophily_marl_b200/pymarl_env.py is the
 * Python binding a maintainer registers in that REGISTRY (INTEGRATION.md).
 *
 * Conventions: plain C types only; all buffers are caller-owned DEVICE
 * pointers unless the name starts with h_ (host, pinned); `stream` is a
 * cudaStream_t passed as void*; every call returns 0 or a negative SSD_ERR_*
 * code and never throws; no internal threads; calls on one handle must be
 * serialised by the caller (except ssd_step_range / ssd_step_autoreset on disjoint ranges).  There is no CPU fallback: without a CUDA device
 * ssd_create fails with SSD_ERR_CUDA.
 * Launches of at most 2048 envs are chained to the preceding kernel of `stream` by programmatic dependent launch: their
 * CTAs may become resident early, but they read nothing before all earlier work of the stream has completed, so stream
 * order holds exactly as for a plain launch (environment variable SSD_B200_PDL=0 disables it).
 */
#ifndef SSD_B200_H
#define SSD_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SSD_B200_ABI_VERSION 2

#define SSD_OK             0
#define SSD_ERR_INVALID   -1   /* bad argument / unsupported geometry            */
#define SSD_ERR_CUDA      -2   /* CUDA runtime error (see ssd_last_cuda_error)   */
#define SSD_ERR_SPAWN     -3   /* fewer spawn points than agents (map_env.py:783) */
#define SSD_ERR_MAP       -4   /* map is not wall-enclosed / unknown character   */

#define SSD_KIND_CLEANUP 0
#define SSD_KIND_HARVEST 1

#define SSD_MAX_AGENTS 16
#define SSD_MAX_CELLS  2048
#define SSD_MAX_SPAWN  32
#define SSD_MAX_VARIANTS 256   /* variant ids are u8 (ssd_set_env_variants) */

/* per-agent episode counters (ssd_set_stats): field indices of stats[B][SSD_N_STATS][agent_stride] */
#define SSD_N_STATS          7
#define SSD_STAT_APPLES      0   /* apples the agent consumed (the lowest index on a cell eats)                              */
#define SSD_STAT_APPLE_T     1   /* sum of t over those consumptions, t = the step's 1-based index in the episode (its `t`)  */
#define SSD_STAT_FIRES       2   /* FIRE actions taken in play (the ones fire_cost charges)                                  */
#define SSD_STAT_HITS_DEALT  3   /* rays of the agent's FIRE beams that hit an agent                                         */
#define SSD_STAT_HITS_TAKEN  4   /* FIRE rays that hit the agent (the one hit_penalty charges); CLEAN never hits             */
#define SSD_STAT_OUT_STEPS   5   /* steps the agent started out of play (tagging-out timer > 0); 0 without tagging           */
#define SSD_STAT_CLEANED     6   /* sum of clean_num: waste cells the agent cleaned                                          */

/* cell codes stored in the device grid (one byte per cell) */
#define SSD_CELL_EMPTY  0
#define SSD_CELL_WALL   1
#define SSD_CELL_APPLE  2
#define SSD_CELL_WASTE  3
#define SSD_CELL_RIVER  4
#define SSD_CELL_STREAM 5

/* observation formats (ssd_set_obs_format) */
#define SSD_OBS_RGB    0   /* u8 RGB planes [n][3][N][N], rows padded (ssd_layout strides): the default            */
#define SSD_OBS_INDEX4 1   /* packed colour indices [n][N][N], 4 bits per pixel (ssd_obs_layout strides; DESIGN.md §3) */

typedef struct ssd_handle ssd_handle;

/* Constructor arguments == the reference's env_args (config/envs/*.yaml:3-15,
 * cleanup.py:29-54, harvest.py:18-22) after the host resolved `map=` into an
 * ASCII map and probabilities. */
typedef struct ssd_config {
    int32_t kind;                 /* SSD_KIND_*                                        */
    int32_t n_envs;               /* B: env instances resident on this device          */
    int32_t n_agents;             /* num_agents (<= SSD_MAX_AGENTS)                    */
    int32_t height, width;        /* ASCII map shape                                    */
    int32_t view;                 /* view_size V; observations are (2V+1)^2            */
    int32_t episode_limit;
    int32_t fire_cost;            /* agent.py:188-190,239-241 -> 1                      */
    int32_t hit_penalty;          /* agent.py:184-186,246-248 -> 0                      */
    int32_t beam_len;             /* cleanup.py:10-11, harvest.py:11 -> 5               */
    int32_t random_spawn_point;   /* extra_args.random_spawn_point                      */
    int32_t spawn_rotation;       /* extra_args.random_spawn_rotation: 0..3, -1 = random */
    int32_t device;               /* CUDA device ordinal                                */
    int32_t tag_timeout;          /* 0..255: steps an agent hit by a FIRE ray stays off the map (tagged out); 0 = never, as
                                   * in the reference.  An agent out of play is not on the map, its action is ignored, its
                                   * reward, clean count and observation are 0; it then respawns like at reset (DESIGN.md §3) */
    uint64_t seed;                /* Philox key                                         */
    uint32_t env_gid_base;        /* global id of env 0 (multi-GPU shards keep trajectories) */
    uint32_t n_waste_lut;         /* entries in thr_apple / thr_waste (= #waste points + 1)   */
    const char* ascii_map;        /* [height*width] row-major, reference alphabet       */
    const uint32_t* thr_apple;    /* cleanup: ceil(pA(h) * 2^32) per waste count h (cleanup.py:189-204) */
    const uint32_t* thr_waste;    /* cleanup: ceil(pW(h) * 2^32), 0 when isclose(pW, 0)  */
    uint32_t thr_harvest[4];      /* harvest: ceil(SPAWN_PROB[k] * 2^32) (harvest.py:118) */
    uint8_t color_lut[16][4];     /* RGB0 per colour index: 0-5 cell codes, 6 outside, 6+c agent char c */
} ssd_config;

/* One env variant (ssd_set_variants): the fields of ssd_config that may differ between the envs of one handle.  Everything else
 * (kind, size, view, n_agents, episode_limit, beam_len, colours, formats, spawn options, seed, env_gid_base) is the handle's. */
typedef struct ssd_variant {
    const char* ascii_map;        /* [height*width] row-major, the handle's size and kind alphabet                      */
    uint32_t n_waste_lut;         /* entries in thr_apple / thr_waste (= #waste points of this map + 1); cleanup only    */
    const uint32_t* thr_apple;    /* cleanup: as ssd_config.thr_apple                                                    */
    const uint32_t* thr_waste;    /* cleanup: as ssd_config.thr_waste                                                    */
    uint32_t thr_harvest[4];      /* harvest: as ssd_config.thr_harvest                                                  */
    int32_t fire_cost;            /* as ssd_config.fire_cost                                                             */
    int32_t hit_penalty;          /* as ssd_config.hit_penalty                                                           */
    int32_t tag_timeout;          /* 0..255, as ssd_config.tag_timeout                                                   */
} ssd_variant;

/* Strides the caller must allocate with (all in elements of the buffer type). */
typedef struct ssd_layout {
    int32_t n_actions;        /* 9 cleanup / 8 harvest                          */
    int32_t n_cells;          /* G = H*W                                        */
    int32_t obs_n;            /* N = 2V+1                                       */
    int32_t grid_stride;      /* bytes per env in `grid` (G rounded up to 16)   */
    int32_t agent_stride;     /* entries per env in `agent` / `ep_ret`          */
    int32_t obs_plane_stride; /* bytes between colour planes (= N * obs_row_stride)   */
    int32_t obs_agent_stride; /* bytes between agents (3 planes rounded to 16)  */
    int32_t obs_env_stride;   /* bytes between envs = n_agents * obs_agent_stride */
    int32_t n_apple_pts, n_waste_pts, n_spawn_pts;
    int32_t obs_row_stride;   /* bytes between pixel rows (N rounded up to 4); pad bytes are 0 */
} ssd_layout;

/* Observation strides of one format, in bytes.
 * SSD_OBS_RGB: the obs_* members of ssd_layout.
 * SSD_OBS_INDEX4: pixel (y, x) of agent a's view is the colour index the RGB renderer looks up for it, so
 *   color_lut[index] is the RGB pixel byte for byte: 0-5 cell codes, 6 outside the map, agents 7 in the simplified
 *   scheme (every agent has one colour) and 6 + agent char of the highest index on the cell in the full scheme.  It
 *   carries more than RGB: empty and outside (both black), or agents and walls (both blue when simplified), differ.
 *   Two pixels per byte: pixel x of a row is byte x >> 1, low nibble when x is even.  An agent out of play (tagging-out)
 *   sees all zero bytes and is absent from every view, as in RGB.  Every pad nibble and pad byte is 0.
 *   row_stride = ceil(N/2) rounded up to 4, plane_stride = 0, agent_stride = N * row_stride rounded up to 16,
 *   env_stride = n_agents * agent_stride. */
typedef struct ssd_obs_layout {
    int32_t format;           /* SSD_OBS_*                                       */
    int32_t row_stride;       /* bytes between pixel rows                        */
    int32_t plane_stride;     /* bytes between colour planes (0 for index4)      */
    int32_t agent_stride;     /* bytes between agents                            */
    int32_t env_stride;       /* bytes between envs                              */
} ssd_obs_layout;

/* State image strides of one format, in bytes (ssd_set_state_format).
 * SSD_OBS_RGB: u8 [3][H][W] per env (get_state * 256): row_stride = W, plane_stride = H*W, env_stride = 3*H*W.
 * SSD_OBS_INDEX4: cell (r, c) is the colour index the RGB state renderer looks up for it, so color_lut[index] is the RGB
 *   state pixel byte for byte: 0-5 the cell code; where an agent in play stands, the colour index of the highest agent
 *   index on the cell (7 in the simplified scheme, 6 + agent char in the full scheme).  An agent out of play (tagging-out)
 *   is absent, as in RGB, and index 6 (outside) never occurs.  Two cells per byte: cell c of row r is byte c >> 1 of the
 *   row, low nibble when c is even.  Every pad nibble and pad byte is 0.
 *   row_stride = ceil(W/2) rounded up to 4, plane_stride = 0, env_stride = H * row_stride rounded up to 16. */
typedef struct ssd_state_layout {
    int32_t format;           /* SSD_OBS_*                                       */
    int32_t row_stride;       /* bytes between map rows                          */
    int32_t plane_stride;     /* bytes between colour planes (0 for index4)      */
    int32_t env_stride;       /* bytes between envs                              */
} ssd_state_layout;

/* Persistent per-env state (MapEnv.world_map, Agent.pos/orientation, _episode_steps, rewards). */
typedef struct ssd_state {
    uint8_t*  grid;      /* [B][grid_stride]   cell codes, padding bytes stay 0           */
    uint32_t* agent;     /* [B][agent_stride]  row | col<<8 | orientation<<16 | tag_out<<24: tag_out = steps the agent is
                          *                     still out of play (tagging-out), 0 = on the map; an agent out keeps the
                          *                     row, col and orientation it had when it was tagged                          */
    int32_t*  ep_ret;    /* [B][agent_stride]  episode return per agent (map_env.py:885-888) */
    int32_t*  t;         /* [B]                _episode_steps                             */
    uint32_t* tick;      /* [B]                Philox step counter (never reset)          */
    uint32_t* counts;    /* [B]                #'A' cells | #'H' cells << 16 of `grid` (the reference recounts the map every
                          *                     step: map_env.py:291-292, cleanup.py:206-212).  Whoever writes `grid` directly
                          *                     must refresh this word; ssd_reset / ssd_step keep it up to date              */
} ssd_state;

/* Outputs of one step == (reward, terminated, info) of MapEnv.step + get_obs/get_state. */
typedef struct ssd_step_out {
    int8_t*   reward;     /* [B][n]                                                     */
    uint8_t*  clean;      /* [B][n]   info["clean_num"]                                 */
    uint16_t* apple_cnt;  /* [B]      info["apple_den"] * H*W                           */
    uint8_t*  done;       /* [B]      terminated                                        */
    uint8_t*  obs;        /* [B][env_stride] observations in the handle's format (ssd_set_obs_format): u8 RGB planes, rows
                           * padded to obs_row_stride (get_obs * 256), or packed colour indices; or NULL              */
    uint8_t*  state_rgb;  /* [B][env_stride] state image in the handle's state format (ssd_set_state_format): u8 RGB
                           * [B][3][H][W] (get_state * 256, the default), or packed colour indices; or NULL             */
} ssd_step_out;

/* Injected, position-indexed random draws (parity harness).  NULL members fall
 * back to Philox4x32-10 keyed (seed; env_gid, tick, stream, index). */
typedef struct ssd_draws {
    const uint32_t* prio;       /* [B][n]     np.random.shuffle of movers (map_env.py:541): ascending (key, index) */
    const uint32_t* u_apple;    /* [B][G]     np.random.rand per apple cell (cleanup.py:172, harvest.py:119)     */
    const uint32_t* u_waste;    /* [B][G]     np.random.rand per waste cell (cleanup.py:183)                      */
    const uint32_t* wkey;       /* [B][G]     random.shuffle(waste_points) (cleanup.py:178): ascending (key, cell) */
    const uint32_t* spawn_key;  /* [B][n][G]  random.shuffle(spawn_points) (map_env.py:777): max (key, cell) wins;
                                 *            read by reset, and by a step for the agents whose tagging-out ends   */
    const uint8_t*  rot;        /* [B][n]     np.random.randint(4) (map_env.py:789); reset, and respawn in a step  */
} ssd_draws;

int ssd_abi_version(void);
const char* ssd_error_string(int code);
/* CUDA error of the most recent failing call on this thread (cudaError_t as int). */
int ssd_last_cuda_error(void);

/* u32 threshold T with (k / 2^32 < p) <=> (k < T); helper for non-Python hosts. */
uint32_t ssd_prob_to_threshold(double p);

/* CleanupEnv/HarvestEnv.__init__ (cleanup.py:29-105, harvest.py:18-48, map_env.py:116-175). */
int ssd_create(const ssd_config* cfg, ssd_handle** out);
int ssd_destroy(ssd_handle* h);
int ssd_get_layout(const ssd_handle* h, ssd_layout* out);

/* Strides of observation format `format` (SSD_OBS_*), whichever format the handle is in, so that a caller can allocate
 * before switching.  ssd_get_layout always reports the RGB strides.  SSD_ERR_INVALID for a NULL handle or an unknown format. */
int ssd_get_obs_layout(const ssd_handle* h, int32_t format, ssd_obs_layout* out);

/* Selects the format of every later `obs` buffer of ssd_reset, ssd_step, ssd_step_range, ssd_render and ssd_step_host
 * (which then copies B * env_stride bytes).  A handle starts in SSD_OBS_RGB.  It is a host-side property of the handle,
 * serialised like every other call on it; a CUDA graph keeps the format it was captured with.  SSD_ERR_INVALID, before
 * any CUDA call, for a NULL handle or an unknown format. */
int ssd_set_obs_format(ssd_handle* h, int32_t format);

/* Strides of state image format `format` (SSD_OBS_*), whichever format the handle is in.  SSD_ERR_INVALID for a NULL
 * handle or an unknown format. */
int ssd_get_state_layout(const ssd_handle* h, int32_t format, ssd_state_layout* out);

/* Selects the format of every later state image (the state_rgb buffer of ssd_step, ssd_step_range, ssd_render and
 * ssd_step_host, which then copies B * env_stride bytes), independently of the observation format.  A handle starts in
 * SSD_OBS_RGB.  Host-side and serialised like ssd_set_obs_format; a CUDA graph keeps the format it was captured with.
 * SSD_ERR_INVALID, before any CUDA call, for a NULL handle or an unknown format. */
int ssd_set_state_format(ssd_handle* h, int32_t format);

/* Forward-offset observation windows (DESIGN.md §3 item 18).  Every later observation of ssd_reset, ssd_step, ssd_step_range,
 * ssd_step_autoreset (obs and the episode-end obs), ssd_render and ssd_step_host is the view an agent at (r, c) facing o would
 * have with offset 0, the default and the reference's view, but with the N x N window centred on (r + f*dr, c + f*dc), where
 * (dr, dc) is the agent's firing direction (LEFT (-1, 0), RIGHT (+1, 0), UP (0, -1), DOWN (0, +1), as ssd_step's FIRE travels):
 * the agent sees V + f cells ahead, V - f behind and V to either side, and its own cell is pixel (V, V + f) of its view.  Cells
 * outside the map, the agent overlay, both colour schemes, tagging-out and the rotation by orientation are as with offset 0, and
 * so are the observation strides: no buffer is reallocated, and every buffer but the observations is bit-identical to that of a
 * handle with offset 0.  A handle with f > 0 runs kernels of its own, whatever SSD_B200_GENERIC says.
 * SSD_ERR_INVALID, before any CUDA call, for a NULL handle or an offset outside 0..view; and SSD_ERR_INVALID when the wider
 * staging tile does not fit the device's opt-in shared memory (the check ssd_create makes).  On an error nothing changes.
 * Host-side and serialised like ssd_set_obs_format; a CUDA graph keeps the offset it was captured with. */
int ssd_set_view_offset(ssd_handle* h, int32_t offset);

/* Row masks of tracked observation buffers (DESIGN.md §3 item 19): the render does not store a pixel row that is all zero now
 * and was all zero when the buffer was last written, so a mostly-black view costs fewer stored bytes; every buffer still holds
 * exactly the bytes it would hold with full stores.  A mask is a caller-owned DEVICE u32 [B][ssd_obs_mask_words(h)] array with
 * one bit per (agent, colour plane, pixel row) of each env's views: row u = agent * N + y of plane pl is bit u % 32 of word
 * 3 * (u / 32) + pl.  A clear bit promises that the row is all zero in the buffer; a set bit promises nothing.  So a mask of
 * zeros goes with a zeroed buffer, a mask of ones with any buffer; whoever writes into a tracked buffer other than through the
 * launches below sets its mask to all ones.
 * ssd_obs_mask_words: words per env of a mask in the handle's current observation format, or 0 where the stores stay full:
 * index4, a row stride other than 32 bytes (only N = 29 and 31 qualify), or more than 32 words per env (n * N > 320).  Negative
 * for a NULL handle.
 * ssd_set_obs_mask: every later ssd_reset, ssd_step, ssd_step_range, ssd_render and ssd_step_host whose observation buffer IS
 * `obs` (the same pointer) reads and updates `obs_mask`.  ssd_step_autoreset stores every row, and sets the words of the envs of
 * its range to all ones in `obs_mask` (buffer `obs`) and `end_obs_mask` (episode-end buffer `end_obs`), one memset each on the
 * launch stream.  A launch with any other buffer stores every row and touches no mask.  NULL masks (the default) turn
 * tracking off.  SSD_ERR_INVALID, before any CUDA call, for a NULL handle, a mask without its buffer, or a mask while
 * ssd_obs_mask_words is 0.  ssd_set_obs_format clears both pairings.  Host-side and serialised like ssd_set_obs_format; a CUDA
 * graph keeps the pairing it was captured with.  The masks of the checked build's skipped rows are verified: a skipped row that
 * is not zero in memory is counted by ssd_debug_oob_count. */
int ssd_obs_mask_words(const ssd_handle* h);
int ssd_set_obs_mask(ssd_handle* h, const uint8_t* obs, uint32_t* obs_mask, const uint8_t* end_obs, uint32_t* end_obs_mask);

/* Sets the handle's variant table to variants[0 .. n_variants) (DESIGN.md §3 item 15), entry 0 included; n_variants = 0 restores
 * the creation config as the only variant.  Env b running variant v is bit-identical, in every buffer and pad byte, to env b of a
 * handle created with v's config alone (same seed and env_gid_base), in every call.  Each entry is validated as ssd_create
 * validates its config, before any CUDA call: SSD_ERR_MAP (not wall-enclosed, or a character outside the kind's alphabet),
 * SSD_ERR_SPAWN (fewer spawn points than agents), SSD_ERR_INVALID (NULL map, n_waste_lut != #waste points + 1 or NULL LUTs for
 * Cleanup, more than SSD_MAX_SPAWN spawn points, too many apple points, |fire_cost| + n|hit_penalty| + 1 > 127, tag_timeout
 * outside 0..255, n_variants outside 0..SSD_MAX_VARIANTS).  On an error nothing changes.  A configuration call, serialised like
 * ssd_set_obs_format: it synchronises the device before it overwrites the table, which is allocated once at its full size, so no
 * launch ever reads a freed table.  A CUDA graph captured before it reads the new table with the launch parameters it was captured
 * with (capture again).  A launch uses the tagging-out kernels when any variant has tag_timeout > 0; an env whose variant has
 * tag_timeout 0 is then never tagged. */
int ssd_set_variants(ssd_handle* h, int32_t n_variants, const ssd_variant* variants);

/* variant_of: caller-owned DEVICE array [B] of variant ids indexed by env index, read by every later launch (a step, auto-reset or
 * render uses the env's current id; a reset builds the env from its current variant's layout, so an env moves to a variant with
 * another layout by writing its id and resetting it).  An id >= n_variants runs the last variant (the checked build counts it).
 * NULL (the default) runs every env as variant 0, with no per-env load.  Host-side and serialised like ssd_set_obs_format; a CUDA
 * graph keeps the pointer it was captured with. */
int ssd_set_env_variants(ssd_handle* h, const uint8_t* variant_of);

/* Per-agent episode counters (DESIGN.md §3 item 16).  stats: caller-owned DEVICE u32 [B][SSD_N_STATS][agent_stride], field-major
 * (SSD_STAT_*); every counter counts since its env's last reset.  Every later ssd_step, ssd_step_range and ssd_step_autoreset adds
 * the step's events; every ssd_reset zeroes the counters of the envs it resets (one more kernel launch on the same stream), and so
 * does the reset half of ssd_step_autoreset, which first copies the finished episode's counters to end_stats (same shape) when
 * that is set; the end_stats slots of other envs are not written.  ssd_render and ssd_step_host leave the counters alone.  Setting
 * counters changes no other byte of any buffer.  Hits are counted whatever hit_penalty and tag_timeout are.
 * Bounds: SSD_STAT_APPLE_T of an episode is at most T(T+1)/2 < 2^31 for T = episode_limit <= 65 535; a caller that steps past
 * `done` without resetting owns any wrap-around (t above 65 535 enters APPLE_T modulo 2^16).
 * NULL, NULL (the default) turns counting off.  SSD_ERR_INVALID, before any CUDA call, for a NULL handle, end_stats without
 * stats, or counters on a handle with episode_limit > 65 535.  Host-side and serialised like ssd_set_obs_format; a CUDA graph
 * keeps the pointers it was captured with. */
int ssd_set_stats(ssd_handle* h, uint32_t* stats, uint32_t* end_stats);

/* One parameter set of the shaped reward (ssd_set_reward_shaping): inequity aversion (Hughes et al., 2018) with disadvantageous
 * weight alpha >= 0, advantageous weight beta >= 0 and trace decay gamma*lambda in [0, 1], mixed with the mean reward of the env
 * at weight prosocial in [0, 1] (Peysakhovich & Lerer, 2018).  Every value finite. */
typedef struct ssd_shaping {
    float alpha, beta, decay, prosocial;
} ssd_shaping;

/* Shaped rewards (DESIGN.md §3 item 17).  trace, shaped: caller-owned DEVICE f32 [B][agent_stride].  Every later ssd_step,
 * ssd_step_range, ssd_step_autoreset and ssd_step_host launches one more kernel on the same stream, over the same envs, that
 * computes, in fp32 with every operation rounded once in this order (a = alpha/(n-1), b = beta/(n-1), both 0 for n = 1, and
 * w1 = 1 - prosocial, all precomputed on the host in fp32), for each agent i of the env, r_i = the step's int8 reward:
 *   e_i <- e_i*decay + r_i;  c = (sum_j r_j)/n;  m_i = w1*r_i + prosocial*c;
 *   D_i = sum_{j != i} max(e_j - e_i, 0), A_i = sum_{j != i} max(e_i - e_j, 0) (ascending j, updated traces);
 *   shaped_i = (m_i - a*D_i) - b*A_i.
 * e is `trace`; every agent's trace is updated, tagged-out agents (reward 0) included.  With alpha = beta = prosocial = 0,
 * shaped_i == r_i exactly.  Every ssd_reset zeroes the traces of the envs it resets (one more kernel launch on the same stream);
 * an ssd_step_autoreset step writes the finished step's shaped reward and then zeroes the trace of every env whose episode it
 * ended.  ssd_render leaves both buffers alone.  Setting shaping changes no other byte of any buffer.
 * params: n_params = 1 applies params[0] to every env; with per-env variant ids (ssd_set_env_variants) env b uses
 * params[min(variant_of[b], n_params - 1)], without them params[0].  n_params = 0 with NULL, NULL (the default) turns shaping off.
 * SSD_ERR_INVALID, before any CUDA call, for a NULL handle, n_params outside 0..SSD_MAX_VARIANTS, NULL params with n_params > 0,
 * trace without shaped or shaped without trace, buffers without parameters or parameters without buffers, or a parameter that is
 * not finite or outside its range.  On an error nothing changes.  A configuration call, serialised like ssd_set_obs_format: the
 * parameter table is allocated once at its full size and overwritten after a device synchronise, so no launch ever reads a freed
 * table; a CUDA graph keeps the buffer pointers it was captured with.
 * Equivalent to ssd_set_reward_preferences(h, n_params, sets, 0, NULL, trace, shaped) with svo_angle = svo_weight = 0. */
int ssd_set_reward_shaping(ssd_handle* h, int32_t n_params, const ssd_shaping* params, float* trace, float* shaped);

/* One preference set (ssd_set_reward_preferences): the four values of ssd_shaping plus a social value orientation (McKee et
 * al., 2020) -- the target reward angle svo_angle in fp32 radians, in [-pi, pi] (pi rounded to fp32; 0 individualistic, pi/4
 * prosocial, pi/2 altruistic), and its weight svo_weight >= 0.  Every value finite. */
typedef struct ssd_preference {
    float alpha, beta, decay, prosocial, svo_angle, svo_weight;
} ssd_preference;

/* Shaped rewards with a preference set per agent (DESIGN.md §3 item 20; extends ssd_set_reward_shaping, whose buffers, resets,
 * launches and graph behaviour it keeps).  Agent i of env b uses set s = set_of[row][i] with row = min(variant_of[b], n_rows-1)
 * (row 0 without per-env variant ids) when a roster is given (n_rows > 0; set_of: HOST u8 [n_rows][n_agents], copied), else
 * s = min(variant_of[b], n_sets-1) (0 without ids), as ssd_set_reward_shaping.  With a, b, w1 precomputed per set as there, and
 * th* = svo_angle, ws = svo_weight, each agent computes, in fp32 with every operation rounded once in this order:
 *   e_i <- e_i*decay_i + r_i;  c = (sum_j r_j)/n;  m_i = w1_i*r_i + prosocial_i*c;
 *   D_i, A_i as ssd_set_reward_shaping;  o_i = (sum_{j != i} e_j)/(n-1) (ascending j, updated traces);
 *   v_i = ws_i*|th*_i - atan2f_ssd(o_i, e_i)|  (v_i = +0 when n = 1 or ws_i = 0: the angle is not computed);
 *   shaped_i = ((m_i - a_i*D_i) - b_i*A_i) - v_i.
 * atan2f_ssd(y, x) is a fixed fp32 sequence, within 2e-6 rad of the exact angle for finite inputs (DESIGN.md §3 item 20):
 *   ax = |x|, ay = |y|, mx = max(ax, ay), mn = min(ax, ay); mx == 0 gives 0;  q = mn/mx, s = q*q;
 *   t = q*(((((( C6*s + C5)*s + C4)*s + C3)*s + C2)*s + C1)*s + C0)  with
 *   C0 = 0.9999961256980896, C1 = -0.3331736922264099, C2 = 0.19807815551757812, C3 = -0.1323334127664566,
 *   C4 = 0.07962366193532944, C5 = -0.0336042121052742, C6 = 0.006811790633946657 (each exactly an fp32 value);
 *   ay > ax: t = pi/2 - t;  x < 0: t = pi - t;  y < 0: t = -t  (pi/2 and pi rounded to fp32).
 * With every svo_weight 0 and no roster the result is that of ssd_set_reward_shaping bit for bit.
 * SSD_ERR_INVALID, before any CUDA call and changing nothing, for a NULL handle, n_sets or n_rows outside 0..SSD_MAX_VARIANTS,
 * NULL sets with n_sets > 0, NULL set_of with n_rows > 0, a roster entry >= n_sets, a field that is not finite or outside its
 * range, or the buffer mismatches ssd_set_reward_shaping refuses.  The set table and the roster table (SSD_MAX_VARIANTS x
 * SSD_MAX_AGENTS bytes) are allocated once at full size and overwritten after a device synchronise. */
int ssd_set_reward_preferences(ssd_handle* h, int32_t n_sets, const ssd_preference* sets, int32_t n_rows, const uint8_t* set_of,
                               float* trace, float* shaped);

/* MapEnv.reset (map_env.py:986-993 -> _reset 297-326).  mask: [B] bytes, non-zero = reset this
 * env, NULL = all.  When obs != NULL the first observations are rendered too. */
int ssd_reset(ssd_handle* h, const ssd_state* st, const uint8_t* mask, const ssd_draws* draws,
              uint8_t* obs, void* stream);

/* MapEnv.step (map_env.py:874-915 -> _step 227-295) fused with get_obs (923-945) and,
 * optionally, get_state (950-957).  actions: [B][n] u8, values < n_actions; a larger value makes that agent do
 * nothing this step (the reference raises KeyError, which the Python facade reproduces before calling). */
int ssd_step(ssd_handle* h, const ssd_state* st, const uint8_t* actions, const ssd_draws* draws,
             const ssd_step_out* out, void* stream);

/* ssd_step restricted to the env instances [env_begin, env_begin + env_count).  Every pointer is still the base of the
 * whole-batch buffer.  Independent ranges may be stepped concurrently on different streams (an asynchronous sampler
 * that overlaps the policy of one group with the env step of another); a range's trajectory does not depend on how the
 * batch is split, because draws are keyed by the global env id. */
int ssd_step_range(ssd_handle* h, const ssd_state* st, const uint8_t* actions, const ssd_draws* draws,
                   const ssd_step_out* out, int32_t env_begin, int32_t env_count, void* stream);

/* Episode-end outputs of ssd_step_autoreset: what an env whose episode ended in the step saw before its reset.  Written
 * only for those envs; the slots of every other env are left as they are.  Every member may be NULL. */
typedef struct ssd_episode_end {
    uint8_t* obs;         /* [B][obs env_stride]   the finished step's observations, in the handle's observation format */
    uint8_t* state_rgb;   /* [B][state env_stride] its state image, in the handle's state format                          */
    int32_t* ep_ret;      /* [B][agent_stride]     the finished episode's return, this step's reward included            */
} ssd_episode_end;

/* ssd_step_range with auto-reset in the same launch (DESIGN.md §3 item 14).  In every buffer, pads included, the result is
 * bit-identical to ssd_step_range(h, st, actions, draws, out, env_begin, env_count), then ssd_reset(h, st, mask = done,
 * draws) of the envs of the range whose `done` the step raised, with the same `draws`, then ssd_render of their
 * observations (out->obs) and state images (out->state_rgb).  So for a reset env: done, reward, clean and apple_cnt are
 * those of the finished step; out->obs / out->state_rgb hold the first observation / state image of the new episode;
 * t = 0, ep_ret = 0, every agent is in play, and tick advances by 2 (the reset draws are keyed by the post-step tick).
 * `end` (or NULL) receives the episode-end outputs.  Validated like ssd_step_range before any CUDA call; disjoint ranges may
 * run concurrently on different streams.  One kernel launch. */
int ssd_step_autoreset(ssd_handle* h, const ssd_state* st, const uint8_t* actions, const ssd_draws* draws,
                       const ssd_step_out* out, const ssd_episode_end* end, int32_t env_begin, int32_t env_count,
                       void* stream);

/* get_obs / get_state without stepping (map_env.py:923-957).  Either pointer may be NULL; state_rgb is written in the
 * handle's state format. */
int ssd_render(ssd_handle* h, const ssd_state* st, uint8_t* obs, uint8_t* state_rgb, void* stream);

/* Host-buffer variant of ssd_step: copies h_actions -> d_actions, steps, copies every non-NULL
 * member of d_out to the same member of h_out, then synchronises the stream. */
int ssd_step_host(ssd_handle* h, const ssd_state* st, const uint8_t* h_actions, uint8_t* d_actions,
                  const ssd_step_out* d_out, const ssd_step_out* h_out, void* stream);

/* Incentive bookkeeping of the homophily learner (homophily_learner.py:98-115):
 * actions_inc [R][n][n] int64 (0 none, 1 reward, 2 punish; diagonal ignored), reward [R][n] f32
 * -> rewards_for_env, rewards_for_inc [R][n] f32, recv_sign [R][n] f32. */
int ssd_incentive(const int64_t* actions_inc, const float* reward, int64_t rows, int32_t n_agents,
                  float incentive, float cost, float ratio, int32_t max_seq_length,
                  float* rewards_for_env, float* rewards_for_inc, float* recv_sign, void* stream);

/* ---- policy side of the rollout loop (SURVEY 8f rows f2 / f3) ------------------------------------------------- */

/* EpsilonGreedyActionSelector.select_action (src/components/action_selectors.py:44-68) on the device.
 * q [rows][n_actions] f32; avail [rows][n_actions] i32 0/1 or NULL (everything available); picked [rows] i64.
 *   greedy      = first index of max over q with unavailable actions at -inf          (lines 57-58, 67)
 *   pick_random = u_pick[row] < epsilon                                                (lines 62-64)
 *   random      = the floor(u_act[row] * #available)-th available action               (line 66: multinomial over the mask)
 * u_pick / u_act: injected uniforms in [0,1) (both or neither); NULL -> Philox4x32-10 keyed (seed; row, counter).
 * The caller evaluates the epsilon schedule (epsilon_schedules.py) and passes 0 in test mode. */
int ssd_select_actions(const float* q, const int32_t* avail, int64_t rows, int32_t n_actions, float epsilon,
                       const float* u_pick, const float* u_act, uint64_t seed, uint64_t counter,
                       int64_t* picked, void* stream);
/* CUDA error of the most recent failing policy-side call on this thread. */
int ssd_policy_last_cuda_error(void);

/* Fused observation front end of the agent network: HomophilyAgent.rgb_preprocess == conv_to_fc
 * (src/modules/agents/homophily_agent.py:19-27; call site src/controllers/homophily_controller.py:132-136) for rollouts:
 *   u8 obs planes (the env's layout) -> /256 -> Conv2d(3,6,k3,s1)+LeakyReLU -> Flatten -> Linear(6(N-2)^2, 32)+LeakyReLU.
 * conv on the CUDA cores, the Linear contraction on tcgen05 tensor cores (tf32 hi/lo split, fp32 accumulate in TMEM).
 * conv_w [6][3][3][3], conv_b [6], fc_w [32][6(N-2)^2] (nn.Linear.weight, Flatten order), fc_b [32]: HOST pointers, copied.
 * Shapes are the reference's defaults (config/default.yaml: conv_out 6, conv_kernel 3, conv_stride 1, obs_dim_net 32). */
typedef struct ssd_frontend ssd_frontend;
int ssd_frontend_create(int32_t view, const float* conv_w, const float* conv_b, const float* fc_w, const float* fc_b,
                        float negative_slope, int32_t device, ssd_frontend** out);
/* obs: DEVICE u8, `rows` agent views `obs_agent_stride` bytes apart (ssd_layout strides); out: DEVICE f32 [rows][32].
 * One kernel launch on `stream`.  The handle owns scratch and counters for tiles shared between CTAs: one forward at a time
 * per handle (stream order is enough), so a handle must not be shared across streams that run concurrently -- the batched
 * runner holds one per env range.  The result does not depend on timing. */
int ssd_frontend_forward(ssd_frontend* f, const uint8_t* obs, int64_t rows, int32_t obs_agent_stride, int32_t obs_plane_stride,
                         int32_t obs_row_stride, float* out, void* stream);
/* ssd_frontend_forward on SSD_OBS_INDEX4 agent views: pixel (y, x) of a view is nibble x of row y (byte x >> 1, low nibble
 * when x is even), and stands for the RGB bytes color_lut[nibble][0..2] (RGB0 rows, the layout of ssd_config.color_lut;
 * HOST pointer, copied into the launch).  The result is bit-identical to ssd_frontend_forward on the RGB planes
 * color_lut[index] with any valid RGB strides.  Same handle rules: one forward at a time per handle, whatever the format.
 * obs_row_stride >= ceil(N / 2) and obs_agent_stride >= N * obs_row_stride, both multiples of 4 (ssd_obs_layout strides). */
int ssd_frontend_forward_index4(ssd_frontend* f, const uint8_t* obs, int64_t rows, int32_t obs_agent_stride,
                                int32_t obs_row_stride, const uint8_t (*color_lut)[4], float* out, void* stream);
int ssd_frontend_destroy(ssd_frontend* f);
int ssd_frontend_last_cuda_error(void);

/* SSD_OBS_INDEX4 observations of envs [env_begin, env_begin + env_count) -> f32 out [env_count][n][3][N][N] contiguous,
 * each value color_lut[index][c] / 256: bit-identical to the RGB observation / 256, zero views of agents out of play
 * included.  obs_index4 is the base of the whole-batch buffer, `out` holds the range only.  One kernel launch on `stream`. */
int ssd_expand_obs(const ssd_handle* h, const uint8_t* obs_index4, int32_t env_begin, int32_t env_count, float* out,
                   void* stream);

/* SSD_OBS_INDEX4 state images of envs [env_begin, env_begin + env_count) -> f32 out [env_count][3][H][W] contiguous, each
 * value color_lut[index][c] / 256: bit-identical to the RGB state image / 256.  state_index4 is the base of the
 * whole-batch buffer, `out` holds the range only.  One kernel launch on `stream` (the kernel of ssd_expand_obs). */
int ssd_expand_state(const ssd_handle* h, const uint8_t* state_index4, int32_t env_begin, int32_t env_count, float* out,
                     void* stream);

/* Kernels launched through this handle since creation (bench.py's gpu_launches), ssd_expand_obs / _state included. */
int64_t ssd_launch_count(const ssd_handle* h);

/* Checked build only (-DSSD_BOUNDS_CHECK, libssd_b200_check.so): number of shared-memory index violations seen so
 * far on the current device; -1 in the normal build. */
int64_t ssd_debug_oob_count(void);

#ifdef __cplusplus
}
#endif
#endif /* SSD_B200_H */
