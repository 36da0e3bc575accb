/* procgen_b200 — C ABI of the B200 vectorised Procgen backend (libprocgen_b200.so).
 *
 * Part 1 is the libenv interface that the reference's libenv.so exports and that gym3's
 * `CEnv` binds through cffi (reference: procgen/src/vecgame.cpp:42-99 for the seven libenv_*
 * entry points, :437-457 for get_state/set_state, declared to cffi at procgen/env.py:132-135).
 * The struct layouts restate gym3==0.3.3 `gym3/libenv.h` (pinned by environment.yml:12), which is
 * not vendored in the reference tree; they are reconstructed from their uses in vecgame.cpp:212-282
 * (libenv_tensortype), vecoptions.cpp:4-54 (libenv_option[s]) and vecgame.cpp:30-40,74-83
 * (libenv_buffers: bufs[space_idx * num_envs + env_idx]).
 *
 * Part 2 is the device-resident extension: the same environment, but observations, rewards,
 * firsts, infos and actions stay in HBM and are exposed as raw device pointers (plain pointers
 * and sizes, no framework types) so a caller can wrap them as tensors without a host round trip.
 */
#ifndef PROCGEN_B200_H
#define PROCGEN_B200_H

#include <stdbool.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define LIBENV_API __declspec(dllexport)
#else
#define LIBENV_API __attribute__((visibility("default")))
#endif

/* ------------------------------------------------------------------ Part 1: libenv */

#define LIBENV_VERSION 1
#define LIBENV_MAX_NAME_LEN 128
#define LIBENV_MAX_NDIM 16

enum libenv_dtype {
    LIBENV_DTYPE_UNUSED = 0,
    LIBENV_DTYPE_UINT8 = 1,
    LIBENV_DTYPE_INT32 = 2,
    LIBENV_DTYPE_FLOAT32 = 3,
};

enum libenv_scalar_type {
    LIBENV_SCALAR_TYPE_UNUSED = 0,
    LIBENV_SCALAR_TYPE_REAL = 1,
    LIBENV_SCALAR_TYPE_DISCRETE = 2,
};

enum libenv_space_name {
    LIBENV_SPACE_UNUSED = 0,
    LIBENV_SPACE_OBSERVATION = 1,
    LIBENV_SPACE_ACTION = 2,
    LIBENV_SPACE_INFO = 3,
};

union libenv_value {
    uint8_t uint8;
    int32_t int32;
    float float32;
};

struct libenv_tensortype {
    char name[LIBENV_MAX_NAME_LEN];
    enum libenv_scalar_type scalar_type;
    enum libenv_dtype dtype;
    int shape[LIBENV_MAX_NDIM];
    int ndim;
    union libenv_value low;
    union libenv_value high;
};

struct libenv_option {
    char name[LIBENV_MAX_NAME_LEN];
    enum libenv_dtype dtype;
    int count;
    void *data;
};

struct libenv_options {
    struct libenv_option *items;
    int count;
};

struct libenv_buffers {
    void **ob;      /* [n_ob_spaces * num_envs], index space_idx * num_envs + env_idx */
    float *rew;     /* [num_envs] */
    uint8_t *first; /* [num_envs] */
    void **info;    /* [n_info_spaces * num_envs] */
    void **ac;      /* [n_ac_spaces * num_envs] */
};

typedef void libenv_env;

/* vecgame.cpp:43-45 */
LIBENV_API int libenv_version(void);

/* vecgame.cpp:47-50. Options consumed: every option of VecGame::VecGame (vecgame.cpp:183-190:
 * env_name, num_levels, start_level, num_actions, rand_seed, num_threads, resource_root,
 * render_human) and of Game::parse_options (game.cpp:42-75).  Unknown options are fatal
 * (vecoptions.cpp:34-38).  num_threads is accepted and ignored: stepping is one asynchronous
 * kernel launch per act().  resource_root names the directory holding assets.pack (or the pack
 * file itself).  Extra, optional int32 options understood by this backend only:
 *   cuda_device        device ordinal (default: current device)
 *   env_index_offset   global index of env 0 when one logical VecGame of `env_index_total` envs
 *   env_index_total    is sharded over several handles/GPUs; the per-env seed chain
 *                      (vecgame.cpp:301-314) and game_n are replayed for the global indices
 *   snap_target_rect   uint8 bool, default 1: Qt>=6 integer snapping of un-rotated image targets */
LIBENV_API libenv_env *libenv_make(int num_envs, const struct libenv_options options);

/* vecgame.cpp:52-72; `types` may be NULL to query the count. */
LIBENV_API int libenv_get_tensortypes(libenv_env *handle, enum libenv_space_name name, struct libenv_tensortype *types);

/* vecgame.cpp:74-83 -> VecGame::set_buffers (:333-361): stores the caller-owned HOST pointers and
 * performs the initial reset + observe of every env. */
LIBENV_API void libenv_set_buffers(libenv_env *handle, struct libenv_buffers *bufs);

/* vecgame.cpp:85-88 -> VecGame::observe (:363-376): waits for the step in flight and fills the
 * host buffers given to libenv_set_buffers. */
LIBENV_API void libenv_observe(libenv_env *handle);

/* vecgame.cpp:90-93 -> VecGame::act (:378-401): copies the actions out of the host buffers
 * (they are only valid during this call) and starts the step asynchronously. */
LIBENV_API void libenv_act(libenv_env *handle);

/* vecgame.cpp:95-98 */
LIBENV_API void libenv_close(libenv_env *handle);

/* State snapshots — replaces get_state / set_state, src/vecgame.cpp:437-457 (declared to cffi at
 * procgen/env.py:132-135). The blob is the reference's own wire format, byte for byte
 * (Game::serialize game.cpp:170-229, BasicAbstractGame::serialize basic-abstract-game.cpp:1169-1223,
 * Entity::serialize entity.cpp:90-131, RandGen::serialize randgen.cpp:100-107, per-game tails): a
 * state saved by the reference loads here and vice versa. get_state returns the number of bytes
 * written (a too small buffer is fatal, like the reference's fassert); set_state also re-renders
 * the env's observation and rewrites its rew / first / info slots from the restored state (Game::observe).
 * Both wait for the step in flight. */
LIBENV_API int get_state(libenv_env *handle, int env_idx, char *data, int length);
LIBENV_API void set_state(libenv_env *handle, int env_idx, char *data, int length);

/* ------------------------------------------------------------------ Part 2: device-resident */

struct pgb200_device_buffers {
    uint8_t *rgb;                  /* [num_envs][64][64][3] uint8, device */
    float *rew;                    /* [num_envs] */
    uint8_t *first;                /* [num_envs] */
    int32_t *prev_level_seed;      /* [num_envs] info */
    uint8_t *prev_level_complete;  /* [num_envs] info */
    int32_t *level_seed;           /* [num_envs] info */
    int32_t *action;               /* [num_envs], written by the caller before pgb200_act_device */
    int32_t num_envs;
    int32_t device;                /* CUDA device ordinal, -1 for the CPU debug build */
    void *stream;                  /* cudaStream_t all work of this handle is ordered on */
};

/* Returns 0 on success. The first call performs the initial reset + render (the work
 * libenv_set_buffers does in host mode). Pointers stay valid until libenv_close. */
LIBENV_API int pgb200_get_device_buffers(libenv_env *handle, struct pgb200_device_buffers *out);

/* Re-home all subsequent work of this handle onto the caller's stream (a cudaStream_t, e.g. the
 * framework's current stream) so launches are ordered with the caller's own kernels and copies
 * without events. The handle's previous work is drained first. The value is used literally: NULL is
 * CUDA's legacy default stream. A new handle starts on a private non-blocking stream;
 * PGB200_PRIVATE_STREAM goes back to it. */
#define PGB200_PRIVATE_STREAM ((void *)(intptr_t)-1)
LIBENV_API void pgb200_set_stream(libenv_env *handle, void *stream);

/* Steps every env with the actions currently in the device action buffer. Asynchronous: enqueues
 * on the handle's stream and returns. */
LIBENV_API void pgb200_act_device(libenv_env *handle);

/* Blocks until all enqueued work of this handle is complete (VecGame::wait_for_stepping_threads). */
LIBENV_API void pgb200_sync(libenv_env *handle);

/* Per-env sticky error bits (0 = healthy): where the reference would fassert/exit, the device code
 * latches a bit instead. Copies num_envs words to `host_out`; returns the OR of all of them. */
LIBENV_API uint32_t pgb200_get_errors(libenv_env *handle, uint32_t *host_out);

/* Profiling aid: when the environment variable PGB200_DEBUG_TIMING is set at libenv_make time, the
 * logic kernel records each env's duration of the last step in SM cycles; copies num_envs words.
 * Returns -1 when timing was not enabled. */
LIBENV_API int pgb200_debug_cycles(libenv_env *handle, uint32_t *host_out);

/* Debug/inspection aid: copies env `env`'s header (512 B, layout csrc/pg_state.cuh EnvHdr) and up to
 * max_ents entity records (128 B each, csrc/pg_state.cuh Entity) to host memory; returns n_ents. */
LIBENV_API int pgb200_debug_read_env(libenv_env *handle, int env, void *hdr_out, void *ents_out, int max_ents);

/* Peer mirror for the single gather of a sharded run (SURVEY §8e, BASELINE configs[4]): mirror0 / mirror1
 * are device-accessible addresses (typically another GPU's memory mapped over NVLink: CUDA IPC or
 * torch symmetric memory) of this shard's [num_envs][64][64][3] slot in the gathered array. Every
 * step then copies each launch's frames there right behind its render kernel, alternating between
 * the two buffers step by step (pgb200_mirror_parity = the buffer the latest step wrote). Passing
 * NULL switches it off. The caller owns the synchronisation between ranks. Returns 0, or -1 in the
 * host debug build. */
LIBENV_API int pgb200_set_rgb_mirror(libenv_env *handle, void *mirror0, void *mirror1);
LIBENV_API int pgb200_mirror_parity(libenv_env *handle);

/* Consumer epilogue (SURVEY §8(f)4: the uint8 -> float normalise + frame-stack step that train-procgen style
 * learners run on every observation, README.md:13): a second output written by the render kernel.
 * `buffer` = device memory of [num_envs][slots][3][64][64] 16-bit floats, dtype 1 = fp16, 2 = bf16,
 * value = rgb / 255 (fp32 division, rounded to nearest even), planar CHW, slots = 1 for k_frames == 1
 * else 2*k_frames: the frame of step t goes to ring slots s = t mod k and s + k, so the ordered stack
 * (oldest first) is always the contiguous slot range [s + 1, s + k] (pgb200_consumer_slot = s). When
 * an env starts an episode the older frames of its window are zeroed (baselines' VecFrameStack). At
 * the call the current frames are written as step 0. buffer == NULL or dtype == 0 switches it off.
 * Returns 0, -1 on bad arguments or in the host debug build. */
LIBENV_API int pgb200_set_consumer_output(libenv_env *handle, void *buffer, int dtype, int k_frames);
LIBENV_API int pgb200_consumer_slot(libenv_env *handle);

/* Profiling variant only (-DPG_PHASE_TIMING): byte offset of the 12 phase-cycle counters inside the
 * header pgb200_debug_read_env returns; -1 in the product build. */
LIBENV_API int pgb200_debug_phase_offset(void);

/* Host debug build only: which path of the render kernel's gather each of the 64 x 64 pixels of env's
 * last frame takes (0 tile cell, opaque texel | 1 tile cell, texel not opaque or empty cell | 2 overlap
 * strip of two cell columns / rows | 3 solid-colour cell | 4 other general cell | 5 no cell), bit 7 set
 * where the box of an entity or overlay blit covers the pixel; out = 4096 bytes, row-major. Returns 0,
 * -1 in the product build. */
LIBENV_API int pgb200_debug_pixel_classes(libenv_env *handle, int env, uint8_t *out);

/* Introspection: shared memory of one render CTA (the per-game frame) and the number of render CTAs
 * per SM the render kernel of `game` is compiled for. Returns -1 for an unknown game. */
LIBENV_API int pgb200_frame_info(const char *game, int *frame_bytes, int *ctas_per_sm);

/* Number of CUDA kernels this handle has launched so far (bench accounting). */
LIBENV_API int64_t pgb200_kernel_launches(libenv_env *handle);

/* Per-kernel device timing for measurement (bench.py roofline): between begin and end every
 * (logic_kernel, setup_kernel, render_kernel) launch triple is bracketed by CUDA events on the stream it
 * runs on. end() synchronises and writes out[0] = sum of logic-kernel ms, out[1] = sum of render-kernel
 * ms, out[2] = number of launch triples timed, out[3] = env-steps those launches processed, out[4] =
 * sum of setup-kernel ms (out must hold 5 doubles); returns the number of triples. At most
 * max_launch_pairs triples are timed (further launches run untimed). */
LIBENV_API int pgb200_kernel_timing_begin(libenv_env *handle, int max_launch_pairs);
/* Measurement knob: chunks > 0 forces that many env chunks per game and step (0 = the default
 * policy); serialize != 0 keeps every launch on the handle's stream, back to back, so a kernel's
 * event-timed duration is its own and not shared with kernels of other chunks. */
LIBENV_API void pgb200_set_launch_shape(libenv_env *handle, int chunks, int serialize);
LIBENV_API int pgb200_kernel_timing_end(libenv_env *handle, double *out);

/* 1 if this library was built for the GPU (the product), 0 for the CPU debug harness in tests/. */
LIBENV_API int pgb200_is_device_build(void);

#ifdef __cplusplus
}
#endif

#endif /* PROCGEN_B200_H */
