// libprocgen_b200.so — host runtime + CUDA kernels + the C ABI of include/procgen_b200.h.
//
// Replaces the reference's vector runtime (vecgame.cpp: N Game objects + worker-thread pool behind
// one mutex and two condvars) with: all env state resident in HBM, one CTA per env, one
// asynchronous kernel launch per act() on a private stream, and observe() = stream wait.
//
// Build modes: nvcc (product, sm_100a).  With -DPG_HOSTSIM the same file builds with g++ into the
// CPU debug harness used ONLY by tests/ (every kernel becomes a plain loop); that build reports
// pgb200_is_device_build() == 0 and the Python package refuses to load it.
#include <dlfcn.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <random>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/procgen_b200.h"
#include "pg_asset_tables.h"
#include "pg_launch.cuh"
#include "games/bigfish.cuh"
#include "games/bossfight.cuh"
#include "games/dodgeball.cuh"
#include "games/caveflyer.cuh"
#include "games/chaser.cuh"
#include "games/climber.cuh"
#include "games/coinrun.cuh"
#include "games/fruitbot.cuh"
#include "games/heist.cuh"
#include "games/jumper.cuh"
#include "games/leaper.cuh"
#include "games/maze.cuh"
#include "games/miner.cuh"
#include "games/ninja.cuh"
#include "games/plunder.cuh"
#include "games/starpilot.cuh"
#include "pg_state_io.h"

#ifndef PG_HOSTSIM
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#endif

namespace pg {
const GameVTable *pg_vtable_bigfish();
const GameVTable *pg_vtable_bossfight();
const GameVTable *pg_vtable_dodgeball();
const GameVTable *pg_vtable_caveflyer();
const GameVTable *pg_vtable_chaser();
const GameVTable *pg_vtable_climber();
const GameVTable *pg_vtable_coinrun();
const GameVTable *pg_vtable_fruitbot();
const GameVTable *pg_vtable_heist();
const GameVTable *pg_vtable_jumper();
const GameVTable *pg_vtable_leaper();
const GameVTable *pg_vtable_maze();
const GameVTable *pg_vtable_miner();
const GameVTable *pg_vtable_ninja();
const GameVTable *pg_vtable_plunder();
const GameVTable *pg_vtable_starpilot();
}  // namespace pg

using namespace pg;

// ================================================================= option parsing (vecoptions.cpp)
namespace {

struct OptParser {
    std::vector<libenv_option> opts;
    explicit OptParser(const libenv_options &o) : opts(o.items, o.items + o.count) {}
    bool find(const std::string &name, libenv_dtype dtype, libenv_option *out) {
        for (size_t i = 0; i < opts.size(); i++) {
            if (name == std::string(opts[i].name)) {
                if (opts[i].dtype != dtype)
                    pg_fatal("invalid dtype for option %s\n", name.c_str());
                *out = opts[i];
                opts.erase(opts.begin() + i);
                return true;
            }
        }
        return false;
    }
    void consume_string(const std::string &name, std::string *v) {
        libenv_option o;
        if (find(name, LIBENV_DTYPE_UINT8, &o))
            *v = std::string((char *)o.data, o.count);
    }
    void consume_int(const std::string &name, int32_t *v) {
        libenv_option o;
        if (find(name, LIBENV_DTYPE_INT32, &o))
            *v = *(int32_t *)o.data;
    }
    void consume_bool(const std::string &name, bool *v) {
        libenv_option o;
        if (find(name, LIBENV_DTYPE_UINT8, &o)) {
            uint8_t b = *(uint8_t *)o.data;
            pg_fassert(b == 0 || b == 1);
            *v = (bool)b;
        }
    }
    void ensure_empty() {
        if (!opts.empty())
            pg_fatal("unused options found, first unused option: %s\n", opts[0].name);
    }
};

std::vector<std::string> split(std::string s, const std::string &delim) {
    std::vector<std::string> out;
    size_t pos;
    while ((pos = s.find(delim)) != std::string::npos) {
        out.push_back(s.substr(0, pos));
        s.erase(0, pos + delim.length());
    }
    out.push_back(s);
    return out;
}

const GameVTable *find_game(const std::string &name) {
    // one entry per games_tu/tu_<game>.cu
    static const GameVTable *const table[] = {
        pg_vtable_bigfish(),
        pg_vtable_bossfight(),
        pg_vtable_dodgeball(),
        pg_vtable_caveflyer(),
        pg_vtable_chaser(),
        pg_vtable_climber(),
        pg_vtable_coinrun(),
        pg_vtable_fruitbot(),
        pg_vtable_heist(),
        pg_vtable_jumper(),
        pg_vtable_leaper(),
        pg_vtable_maze(),
        pg_vtable_miner(),
        pg_vtable_ninja(),
        pg_vtable_plunder(),
        pg_vtable_starpilot(),
    };
    for (const GameVTable *g : table)
        if (name == g->name)
            return g;
    return nullptr;
}

// ================================================================= memory helpers
template <class T>
T *dev_alloc(size_t n) {
    T *ptr = nullptr;
    if (n == 0)
        n = 1;
#ifndef PG_HOSTSIM
    CUDA_CHECK(cudaMalloc((void **)&ptr, n * sizeof(T)));
    CUDA_CHECK(cudaMemset(ptr, 0, n * sizeof(T)));
#else
    ptr = (T *)calloc(n, sizeof(T));
#endif
    return ptr;
}
void dev_free(void *ptr) {
#ifndef PG_HOSTSIM
    if (ptr)
        cudaFree(ptr);
#else
    free(ptr);
#endif
}
void copy_to_dev(void *dst, const void *src, size_t bytes) {
#ifndef PG_HOSTSIM
    CUDA_CHECK(cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice));
#else
    memcpy(dst, src, bytes);
#endif
}

// vecgame.cpp:156-167: system-independent hash of the game name
static int32_t fnv1a(const char *str) {
    uint32_t hash = 0x811c9dc5u;
    for (const char *c = str; *c; c++) {
        hash ^= (uint8_t)*c;
        hash *= 0x1000193u;
    }
    return (int32_t)hash;
}

// ================================================================= pre-scaled tile table
#ifndef PG_HOSTSIM
// one CTA per (sprite slot, tw, th)
__global__ void tile_table_kernel(const SpriteDesc *sprites, const uint32_t *index, uint32_t *texels, const uint32_t *atlas) {
    const int slot = (int)blockIdx.x / TILE_VARIANTS, v = (int)blockIdx.x % TILE_VARIANTS;
    tile_table_fill(sprites, index, texels, atlas, slot, v / MAX_TILE_DIM + 1, v % MAX_TILE_DIM + 1, (int)threadIdx.x, (int)blockDim.x);
}
#endif

#ifndef PG_HOSTSIM
// (16-bit float)(v / 255.f) for v = 0..255: IEEE fp32 division, then round-to-nearest-even
__global__ void consumer_lut_kernel(uint16_t *lut, int bf16) {
    const int v = (int)threadIdx.x;
    const float x = __fdiv_rn((float)v, 255.0f);
    if (bf16) {
        const uint32_t u = __float_as_uint(x);
        lut[v] = (uint16_t)((u + 0x7fffu + ((u >> 16) & 1u)) >> 16);
    } else {
        lut[v] = __half_as_ushort(__float2half_rn(x));
    }
}
#endif

// ================================================================= VecEnv (VecGame, vecgame.h)
struct VecEnv {
    int num_envs = 0;
    int device = -1;
    std::vector<const GameVTable *> games;  // joint games, env n <-> games[n % size] (vecgame.cpp:310)
    std::vector<int> view;                  // per game: 0 = its usual view, 1 = the whole-world view (center_agent = false)
    std::vector<libenv_tensortype> observation_types, action_types, info_types;
    int num_actions = -1;

    KParams base{};                  // common launch parameters
    std::vector<GameAssets *> d_assets;  // per joint game
    uint32_t *d_atlas = nullptr;
    uint32_t *d_tile_texels = nullptr, *d_tile_index = nullptr;
    SpriteDesc *d_tile_sprites = nullptr;
    uint32_t *d_lvl_seeds = nullptr;
    int32_t *d_action = nullptr;
    bool initial_reset_done = false;
    int64_t launches = 0;
    host::ConstGameFields const_fields;  // options Game::serialize writes but no kernel reads

#ifndef PG_HOSTSIM
    cudaStream_t stream = nullptr;
    cudaStream_t own_stream = nullptr;
    static constexpr int kAuxStreams = PG_AUX_STREAMS;
    cudaStream_t aux[kAuxStreams] = {};
    // PGB200_PRIORITY_SPLIT=1: logic kernels go to high-priority twins of the auxiliary streams so
    // their (small) blocks are dispatched ahead of the render CTAs queued by other chunks
    bool priority_split = false;
    cudaStream_t aux_hi[kAuxStreams] = {};
    cudaEvent_t ev_link[kAuxStreams] = {};
    cudaEvent_t ev_fork = nullptr;
    cudaEvent_t ev_join[kAuxStreams] = {};
    // optional per-launch kernel timing (pgb200_kernel_timing_begin/end): a pool of event triples
    std::vector<cudaEvent_t> tev_pool;
    std::vector<int> tev_envs;   // env count of each timed launch pair
    size_t tev_used = 0;
    bool timing = false;
#endif
    static constexpr int kChunks = PG_STEP_CHUNKS;
    int force_chunks = 0;            // measurement knobs (pgb200_set_launch_shape)
    bool serialize_launches = false;
    static constexpr int kMaxTickets = 64;   // launch slots in flight (one ticket counter each)
    unsigned int *d_tickets = nullptr;
    int max_logic_blocks = 1 << 30;
    int render_smem_floor = 0;
    // host-buffer (libenv) mode
    // peer mirror (config 5, SURVEY §8e): when set, every launch's frames are also copied into
    // these buffers (another GPU's memory, mapped through NVLink) right behind its render kernel
    uint8_t *mirror[2] = {nullptr, nullptr};
    int mirror_parity = 0;
    uint16_t *d_consumer_lut = nullptr;
    int64_t consumer_steps = 0;
    bool have_host_bufs = false;
    bool rgb_copy_enqueued = false;  // this step's observation DMA already follows the render kernels
    bool ob_direct = false;      // caller's obs block is contiguous and page-locked: DMA straight into it
    bool ob_registered = false;
    std::vector<void *> h_ob, h_ac;
    std::vector<std::vector<void *>> h_info;  // [space][env]
    float *h_rew = nullptr;
    uint8_t *h_first = nullptr;
    // pinned staging
    uint8_t *st_rgb = nullptr;
    int32_t *st_action = nullptr;
    float *st_rew = nullptr;
    uint8_t *st_first = nullptr;
    int32_t *st_prev_seed = nullptr;
    uint8_t *st_prev_complete = nullptr;
    int32_t *st_seed = nullptr;

    LaunchCtx lctx() {
        LaunchCtx lc;
#ifndef PG_HOSTSIM
        lc.stream = stream;
        lc.logic_stream = nullptr;
        lc.link = nullptr;
        lc.ticket = d_tickets;
        lc.max_logic_blocks = max_logic_blocks;
        lc.render_smem_floor = render_smem_floor;
        lc.tev = nullptr;
#endif
        lc.launch_counter = &launches;
        return lc;
    }

    // One step = for every (game, env chunk): logic kernel then render kernel. Chunks go round-robin
    // onto a few auxiliary streams forked from / joined to the handle's stream with events, so the
    // latency-bound logic kernel of one chunk overlaps the issue-bound render kernel of another on
    // the same SMs (the two kernels stress different limits; back to back they leave both idle).
    void launch(bool init) {
        const int G = (int)games.size();
        const int per_game = num_envs / G;
        int chunks = force_chunks > 0 ? force_chunks : kChunks;
        if (force_chunks <= 0 && per_game < 4096 * chunks)
            chunks = 1;
#ifndef PG_HOSTSIM
        // more than one (logic, render) pair in the step — env chunks of one game, or the games of a
        // joint list — are spread over the auxiliary streams so they overlap on the SMs
        const int nstreams = (chunks * G > 1 && !serialize_launches) ? kAuxStreams : 0;
        if (nstreams) {
            CUDA_CHECK(cudaEventRecord(ev_fork, stream));
            for (int s = 0; s < nstreams; s++) {
                CUDA_CHECK(cudaStreamWaitEvent(aux[s], ev_fork, 0));
                if (priority_split)
                    CUDA_CHECK(cudaStreamWaitEvent(aux_hi[s], ev_fork, 0));
            }
        }
#endif
        if (!init && mirror[0])
            mirror_parity ^= 1;
        if (!init && base.consumer) {
            consumer_steps++;
            base.consumer_slot = (int32_t)(consumer_steps % base.consumer_k);
        }
        int k = 0;
        for (int g = 0; g < G; g++) {
            for (int cidx = 0; cidx < chunks; cidx++, k++) {
                const int lo = (int)((int64_t)per_game * cidx / chunks);
                const int hi = (int)((int64_t)per_game * (cidx + 1) / chunks);
                KParams p = base;
                p.assets = d_assets[g];
                p.game_id = games[g]->id;
                p.fixed_asset_seed = fnv1a(games[g]->name);
                p.env_first = g + lo * G;
                p.env_step = G;
                p.env_count = hi - lo;
                LaunchCtx lc = lctx();
#ifndef PG_HOSTSIM
                if (nstreams) {
                    lc.stream = aux[k % nstreams];
                    if (priority_split) {
                        lc.logic_stream = aux_hi[k % nstreams];
                        lc.link = ev_link[k % nstreams];
                    }
                }
                lc.ticket = d_tickets + (k % kMaxTickets);
                if (timing && tev_used + 4 <= tev_pool.size()) {
                    lc.tev = &tev_pool[tev_used];
                    tev_used += 4;
                    tev_envs.push_back(p.env_count);
                }
#endif
                if (init)
                    games[g]->init[view[g]](p, lc);
                else
                    games[g]->step[view[g]](p, lc);
#ifndef PG_HOSTSIM
                // libenv (host buffer) mode: start this chunk's observation DMA right behind its
                // render kernel, on the same stream, so the copy of one chunk overlaps the kernels
                // of the next instead of waiting for the whole step (PCIe is the e2e bottleneck:
                // 12 KiB per env and step)
                if (!init && mirror[0] && hi > lo) {
                    // the gather of SURVEY §8e without a collective: this launch's frames go straight
                    // to their place in the destination rank's buffer, overlapping the other launches
                    const size_t frame = RES_W * RES_H * 3;
                    const size_t first = (size_t)(g + lo * G) * frame;
                    if (G == 1)
                        CUDA_CHECK(cudaMemcpyAsync(mirror[mirror_parity] + first, base.rgb + first, (size_t)(hi - lo) * frame,
                                                   cudaMemcpyDeviceToDevice, lc.stream));
                    else
                        CUDA_CHECK(cudaMemcpy2DAsync(mirror[mirror_parity] + first, (size_t)G * frame, base.rgb + first, (size_t)G * frame, frame,
                                                     (size_t)(hi - lo), cudaMemcpyDeviceToDevice, lc.stream));
                }
                if (have_host_bufs && G == 1 && hi > lo) {
                    const size_t frame = RES_W * RES_H * 3;
                    uint8_t *rgb_dst = ob_direct ? (uint8_t *)h_ob[0] : st_rgb;
                    CUDA_CHECK(cudaMemcpyAsync(rgb_dst + (size_t)lo * frame, base.rgb + (size_t)lo * frame, (size_t)(hi - lo) * frame,
                                               cudaMemcpyDeviceToHost, lc.stream));
                    rgb_copy_enqueued = true;
                }
#endif
            }
        }
#ifndef PG_HOSTSIM
        if (nstreams) {
            for (int s = 0; s < nstreams; s++) {
                CUDA_CHECK(cudaEventRecord(ev_join[s], aux[s]));
                CUDA_CHECK(cudaStreamWaitEvent(stream, ev_join[s], 0));
            }
        }
#endif
    }

    void ensure_initial_reset() {
        if (initial_reset_done)
            return;
        launch(true);
        initial_reset_done = true;
    }

    void sync() {
#ifndef PG_HOSTSIM
        CUDA_CHECK(cudaStreamSynchronize(stream));
#endif
    }

    void set_device() {
#ifndef PG_HOSTSIM
        CUDA_CHECK(cudaSetDevice(device));
#endif
    }
};

std::string default_pack_path() {
    // <dir of this .so>/data/assets.pack, overridable with PROCGEN_B200_ASSET_PACK
    const char *e = getenv("PROCGEN_B200_ASSET_PACK");
    if (e && e[0])
        return e;
    Dl_info info;
    if (dladdr((void *)&libenv_version, &info) && info.dli_fname) {
        std::string so(info.dli_fname);
        size_t slash = so.rfind('/');
        std::string dir = slash == std::string::npos ? "." : so.substr(0, slash);
        return dir + "/data/assets.pack";
    }
    return "assets.pack";
}

void fill_tensortypes(VecEnv *v) {
    // vecgame.cpp:212-268
    libenv_tensortype s;
    memset(&s, 0, sizeof(s));
    strcpy(s.name, "rgb");
    s.scalar_type = LIBENV_SCALAR_TYPE_DISCRETE;
    s.dtype = LIBENV_DTYPE_UINT8;
    s.shape[0] = RES_W;
    s.shape[1] = RES_H;
    s.shape[2] = 3;
    s.ndim = 3;
    s.low.uint8 = 0;
    s.high.uint8 = 255;
    v->observation_types.push_back(s);

    memset(&s, 0, sizeof(s));
    strcpy(s.name, "action");
    s.scalar_type = LIBENV_SCALAR_TYPE_DISCRETE;
    s.dtype = LIBENV_DTYPE_INT32;
    s.ndim = 0;
    s.low.int32 = 0;
    s.high.int32 = v->num_actions - 1;
    v->action_types.push_back(s);

    const char *info_names[3] = {"prev_level_seed", "prev_level_complete", "level_seed"};
    for (int i = 0; i < 3; i++) {
        memset(&s, 0, sizeof(s));
        strcpy(s.name, info_names[i]);
        s.scalar_type = LIBENV_SCALAR_TYPE_DISCRETE;
        s.ndim = 0;
        if (i == 1) {
            s.dtype = LIBENV_DTYPE_UINT8;
            s.low.uint8 = 0;
            s.high.uint8 = 1;
        } else {
            s.dtype = LIBENV_DTYPE_INT32;
            s.low.int32 = 0;
            s.high.int32 = INT32_MAX;
        }
        v->info_types.push_back(s);
    }
}

}  // namespace

// ================================================================= C ABI
extern "C" {

int libenv_version(void) { return LIBENV_VERSION; }

int pgb200_is_device_build(void) {
#ifndef PG_HOSTSIM
    return 1;
#else
    return 0;
#endif
}

libenv_env *libenv_make(int num_envs, const struct libenv_options options) {
    OptParser opts(options);
    VecEnv *v = new VecEnv;
    v->num_envs = num_envs;

    // ---- VecGame::VecGame options (vecgame.cpp:169-190)
    std::string env_name, resource_root;
    int32_t num_levels = 0, start_level = -1, rand_seed = 0, num_threads = 4;
    bool render_human = false;
    opts.consume_string("env_name", &env_name);
    opts.consume_int("num_levels", &num_levels);
    opts.consume_int("start_level", &start_level);
    opts.consume_int("num_actions", &v->num_actions);
    opts.consume_int("rand_seed", &rand_seed);
    opts.consume_int("num_threads", &num_threads);
    opts.consume_string("resource_root", &resource_root);
    opts.consume_bool("render_human", &render_human);
    // ---- backend extensions
    int32_t cuda_device = -1, env_index_offset = 0, env_index_total = -1;
    bool snap = true;
    opts.consume_int("cuda_device", &cuda_device);
    opts.consume_int("env_index_offset", &env_index_offset);
    opts.consume_int("env_index_total", &env_index_total);
    opts.consume_bool("snap_target_rect", &snap);
    if (env_index_total < 0)
        env_index_total = env_index_offset + num_envs;

    pg_fassert(num_threads >= 0);
    pg_fassert(env_name != "");
    pg_fassert(v->num_actions > 0);
    pg_fassert(num_levels >= 0);
    pg_fassert(start_level >= 0);
    if (render_human)
        pg_fatal("render_human (512x512 antialiased info['rgb']) is not supported by procgen_b200\n");

    // ---- Game::parse_options (game.cpp:42-75)
    bool use_easy_jump = false, paint_vel_info = false, use_generated_assets = false, use_monochrome_assets = false;
    bool restrict_themes = false, use_backgrounds = true, center_agent = false, use_sequential_levels = false;
    opts.consume_bool("use_easy_jump", &use_easy_jump);
    opts.consume_bool("paint_vel_info", &paint_vel_info);
    opts.consume_bool("use_generated_assets", &use_generated_assets);
    opts.consume_bool("use_monochrome_assets", &use_monochrome_assets);
    opts.consume_bool("restrict_themes", &restrict_themes);
    opts.consume_bool("use_backgrounds", &use_backgrounds);
    opts.consume_bool("center_agent", &center_agent);
    opts.consume_bool("use_sequential_levels", &use_sequential_levels);
    int32_t dist_mode = EasyMode, plain_assets = 0, physics_mode = 0, debug_mode = 0, game_type = 0;
    opts.consume_int("distribution_mode", &dist_mode);
    opts.consume_int("plain_assets", &plain_assets);
    opts.consume_int("physics_mode", &physics_mode);
    opts.consume_int("debug_mode", &debug_mode);
    opts.consume_int("game_type", &game_type);
    opts.ensure_empty();
    if (use_generated_assets)
        pg_fatal("use_generated_assets is not supported by procgen_b200\n");

    std::vector<std::string> env_names = split(env_name, ",");
    const int G = (int)env_names.size();
    pg_fassert(num_envs % G == 0);
    pg_fassert(env_index_offset % G == 0);
    for (const auto &name : env_names) {
        const GameVTable *g = find_game(name);
        if (!g)
            pg_fatal("unknown or not yet supported env_name '%s'\n", name.c_str());
        // Five games honour center_agent=false by drawing their whole (up to 64x64-cell) world
        // (basic-abstract-game.cpp:819-838) through the render path sized for that view.
        int view = 0;
        if (!center_agent && (name == "coinrun" || name == "climber" || name == "caveflyer" || name == "jumper" || name == "ninja")) {
            if (g->step[1] == nullptr)
                pg_fatal("center_agent=false is not supported for '%s' by procgen_b200 yet\n", name.c_str());
            view = 1;
        }
        v->view.push_back(view);
        // mode validity, game.cpp:56-66
        if (dist_mode == EasyMode || dist_mode == HardMode) {
        } else if (dist_mode == ExtremeMode) {
            pg_fassert(name == "chaser" || name == "dodgeball" || name == "leaper" || name == "starpilot");
        } else if (dist_mode == MemoryMode) {
            pg_fassert(name == "caveflyer" || name == "dodgeball" || name == "heist" || name == "jumper" || name == "maze" || name == "miner");
        } else {
            pg_fatal("invalid distribution_mode %d\n", dist_mode);
        }
        v->games.push_back(g);
    }

    // ---- device
#ifndef PG_HOSTSIM
    if (cuda_device < 0)
        CUDA_CHECK(cudaGetDevice(&cuda_device));
    v->device = cuda_device;
    v->set_device();
    CUDA_CHECK(cudaStreamCreateWithFlags(&v->own_stream, cudaStreamNonBlocking));
    v->stream = v->own_stream;
    {
        const char *e = getenv("PGB200_PRIORITY_SPLIT");
        v->priority_split = e && atoi(e) != 0;
    }
    int prio_lo = 0, prio_hi = 0;
    CUDA_CHECK(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));  // numerically lower = higher priority
    for (int s = 0; s < VecEnv::kAuxStreams; s++) {
        CUDA_CHECK(cudaStreamCreateWithFlags(&v->aux[s], cudaStreamNonBlocking));
        CUDA_CHECK(cudaEventCreateWithFlags(&v->ev_join[s], cudaEventDisableTiming));
        if (v->priority_split) {
            CUDA_CHECK(cudaStreamCreateWithPriority(&v->aux_hi[s], cudaStreamNonBlocking, prio_hi));
            CUDA_CHECK(cudaEventCreateWithFlags(&v->ev_link[s], cudaEventDisableTiming));
        }
    }
    CUDA_CHECK(cudaEventCreateWithFlags(&v->ev_fork, cudaEventDisableTiming));
    {
        cudaDeviceProp prop;
        CUDA_CHECK(cudaGetDeviceProperties(&prop, v->device));
        v->max_logic_blocks = prop.multiProcessorCount * PG_LOGIC_MIN_BLOCKS;
        // tuning knobs (defaults chosen from the sweeps in profiles/): resident logic blocks and
        // render CTAs per SM
        if (const char *e = getenv("PGB200_LOGIC_BLOCKS_PER_SM"))
            if (atoi(e) > 0)
                v->max_logic_blocks = prop.multiProcessorCount * atoi(e);
        int render_ctas = PG_RENDER_CTAS_PER_SM;
        if (const char *e = getenv("PGB200_RENDER_CTAS_PER_SM"))
            render_ctas = atoi(e);
        if (render_ctas > 0 && render_ctas < 16) {
            // usable shared memory per SM is 227 KiB, each CTA also pays 1 KiB of system reserve
            v->render_smem_floor = (227 * 1024) / render_ctas - 1024 - 16;
            v->render_smem_floor &= ~15;
        }
        CUDA_CHECK(cudaMalloc((void **)&v->d_tickets, VecEnv::kMaxTickets * sizeof(unsigned int)));
    }
    // sub_step <-> push_obj recurse to depth 5 on the logic thread
    {
        size_t cur = 0;
        CUDA_CHECK(cudaDeviceGetLimit(&cur, cudaLimitStackSize));
        if (cur < 4096)  // only ever raise it: the host application may have asked for more
            CUDA_CHECK(cudaDeviceSetLimit(cudaLimitStackSize, 4096));
    }
#else
    v->device = -1;
#endif

    // ---- assets
    std::string pack_path = resource_root;
    if (pack_path.size() >= 5 && pack_path.compare(pack_path.size() - 5, 5, ".pack") == 0) {
    } else if (!pack_path.empty()) {
        if (pack_path.back() != '/')
            pack_path += "/";
        pack_path += "assets.pack";
    } else {
        pack_path = default_pack_path();
    }
    try {
        host::AssetPackReader pack(pack_path);
        host::AtlasBuilder atlas(pack);
        std::vector<GameAssets> tables(G);
        for (int g = 0; g < G; g++) atlas.build_game(v->games[g]->id, tables[g]);
        v->d_atlas = dev_alloc<uint32_t>(atlas.texels.size());
        copy_to_dev(v->d_atlas, atlas.texels.data(), atlas.texels.size() * sizeof(uint32_t));
        for (int g = 0; g < G; g++) {
            GameAssets *d = dev_alloc<GameAssets>(1);
            copy_to_dev(d, &tables[g], sizeof(GameAssets));
            v->d_assets.push_back(d);
        }
        // pre-scaled cell tiles of every sprite (pg_raster.cuh TileTable), filled on the device by
        // the general blit path's own arithmetic
        const bool want_tiles = !(getenv("PGB200_NO_TILES") && atoi(getenv("PGB200_NO_TILES")) != 0);
        const int S = (int)atlas.tile_sprites.size();
        if (want_tiles && S > 0) {
            std::vector<uint32_t> index((size_t)S * TILE_VARIANTS);
            size_t top = 0;
            for (int sl = 0; sl < S; sl++)
                for (int tw = 1; tw <= MAX_TILE_DIM; tw++)
                    for (int th = 1; th <= MAX_TILE_DIM; th++) {
                        index[((size_t)sl * MAX_TILE_DIM + (tw - 1)) * MAX_TILE_DIM + (th - 1)] = (uint32_t)top;
                        top += (size_t)tile_words(tw, th);
                    }
            if (top >= (size_t)1 << 32)
                throw std::runtime_error("tile table too large");
            v->d_tile_index = dev_alloc<uint32_t>(index.size());
            copy_to_dev(v->d_tile_index, index.data(), index.size() * sizeof(uint32_t));
            v->d_tile_sprites = dev_alloc<SpriteDesc>((size_t)S);
            copy_to_dev(v->d_tile_sprites, atlas.tile_sprites.data(), (size_t)S * sizeof(SpriteDesc));
            v->d_tile_texels = dev_alloc<uint32_t>(top);
#ifndef PG_HOSTSIM
            tile_table_kernel<<<S * TILE_VARIANTS, 64>>>(v->d_tile_sprites, v->d_tile_index, v->d_tile_texels, v->d_atlas);
            CUDA_CHECK(cudaGetLastError());
#else
            for (int sl = 0; sl < S; sl++)
                for (int vv = 0; vv < TILE_VARIANTS; vv++)
                    tile_table_fill(v->d_tile_sprites, v->d_tile_index, v->d_tile_texels, v->d_atlas, sl, vv / MAX_TILE_DIM + 1, vv % MAX_TILE_DIM + 1, 0, 1);
#endif
            v->base.tiles.texels = v->d_tile_texels;
            v->base.tiles.index = v->d_tile_index;
            v->base.tiles.sprites = v->d_tile_sprites;
            v->base.tiles.n_slots = S;
        }
    } catch (const std::exception &e) {
        pg_fatal("failed to load images %s\n", e.what());
    }

    fill_tensortypes(v);

    // ---- state arrays
    int ent_cap = 0, grid_cap = 0, scratch_words = 0, rot_records = 0, blit_records = 0, setup_bytes = 0, cell_records = 0;
    for (const auto &g : v->games) {
        rot_records = std::max(rot_records, g->rot_records);
        blit_records = std::max(blit_records, g->blit_records);
        const int vw = v->view[&g - &v->games[0]];
        setup_bytes = std::max(setup_bytes, g->setup_bytes[vw]);
        cell_records = std::max(cell_records, g->cell_records[vw]);
        ent_cap = std::max(ent_cap, g->ent_cap);
        grid_cap = std::max(grid_cap, g->grid_cap);
        scratch_words = std::max(scratch_words, g->scratch_words);
    }
    KParams &p = v->base;
    const size_t N = (size_t)num_envs;
    p.ent_stride = ent_cap + 1;
    p.grid_stride = grid_cap;
    p.scratch_stride = scratch_words;
    p.hdr = dev_alloc<EnvHdr>(N);
    p.ents = dev_alloc<Entity>(N * p.ent_stride);
    p.grid = dev_alloc<int16_t>(N * p.grid_stride);
    p.rng = dev_alloc<MT19937>(N);
    p.lvl_rng = dev_alloc<MT19937>(N);
    p.scratch = dev_alloc<int32_t>(N * (size_t)scratch_words);
    p.rot_stride = rot_records;
    p.rot_scratch = rot_records > 0 ? dev_alloc<RotBlit>(N * (size_t)rot_records) : nullptr;
    p.blit_stride = blit_records;
    p.blit_list = dev_alloc<Blit>(N * (size_t)blit_records);
    p.cell_spill_stride = cell_records;
    p.cell_spill = dev_alloc<Blit>(N * (size_t)cell_records);
    p.frame_setup_stride = (setup_bytes + 15) & ~15;
    p.frame_setup = dev_alloc<unsigned char>(N * (size_t)p.frame_setup_stride);
    p.atlas = v->d_atlas;
    v->d_action = dev_alloc<int32_t>(N);
    p.action = v->d_action;
    p.rgb = dev_alloc<uint8_t>(N * RES_W * RES_H * 3);
    p.rew = dev_alloc<float>(N);
    p.first = dev_alloc<uint8_t>(N);
    p.info_prev_level_seed = dev_alloc<int32_t>(N);
    p.info_prev_level_complete = dev_alloc<uint8_t>(N);
    p.info_level_seed = dev_alloc<int32_t>(N);
    p.dbg_cycles = getenv("PGB200_DEBUG_TIMING") ? dev_alloc<uint32_t>(N) : nullptr;


    // ---- per-env seed chain (vecgame.cpp:301-314), replayed for the global env indices
    {
        std::mt19937 game_level_seed_gen;
        game_level_seed_gen.seed((uint32_t)rand_seed);
        for (int i = 0; i < env_index_offset; i++) (void)game_level_seed_gen();
        std::vector<uint32_t> seeds(N);
        for (size_t i = 0; i < N; i++) seeds[i] = (uint32_t)game_level_seed_gen();
        v->d_lvl_seeds = dev_alloc<uint32_t>(N);
        copy_to_dev(v->d_lvl_seeds, seeds.data(), N * sizeof(uint32_t));
        p.lvl_seeds = v->d_lvl_seeds;
    }

    // vecgame.cpp:284-293
    if (num_levels == 0) {
        p.level_seed_low = 0;
        p.level_seed_high = INT32_MAX;
    } else {
        p.level_seed_low = start_level;
        p.level_seed_high = start_level + num_levels;
    }
    memset(&p.options, 0, sizeof(p.options));
    p.options.paint_vel_info = paint_vel_info;
    p.options.use_generated_assets = use_generated_assets;
    p.options.use_monochrome_assets = use_monochrome_assets;
    p.options.restrict_themes = restrict_themes;
    p.options.use_backgrounds = use_backgrounds;
    p.options.center_agent = center_agent;
    p.options.use_sequential_levels = use_sequential_levels;
    p.options.debug_mode = debug_mode;
    v->const_fields.use_easy_jump = use_easy_jump;
    v->const_fields.plain_assets = plain_assets;
    v->const_fields.physics_mode = physics_mode;
    v->const_fields.game_type = game_type;
    p.options.distribution_mode = dist_mode;
    p.snap = snap ? 1 : 0;
    p.env_global_offset = env_index_offset;
#ifndef PG_HOSTSIM
    // every upload and memset above ran on the legacy default stream; the step kernels run on
    // non-blocking streams that do not order against it
    CUDA_CHECK(cudaDeviceSynchronize());
#endif
    return (libenv_env *)v;
}

int libenv_get_tensortypes(libenv_env *handle, enum libenv_space_name name, struct libenv_tensortype *out_types) {
    VecEnv *v = (VecEnv *)handle;
    const std::vector<libenv_tensortype> *types = nullptr;
    if (name == LIBENV_SPACE_OBSERVATION)
        types = &v->observation_types;
    else if (name == LIBENV_SPACE_ACTION)
        types = &v->action_types;
    else if (name == LIBENV_SPACE_INFO)
        types = &v->info_types;
    else
        return 0;
    if (out_types)
        for (size_t i = 0; i < types->size(); i++) out_types[i] = (*types)[i];
    return (int)types->size();
}

static void *host_alloc(size_t bytes) {
#ifndef PG_HOSTSIM
    void *ptr = nullptr;
    CUDA_CHECK(cudaHostAlloc(&ptr, bytes ? bytes : 1, cudaHostAllocDefault));
    return ptr;
#else
    return malloc(bytes ? bytes : 1);
#endif
}
static void host_free(void *ptr) {
#ifndef PG_HOSTSIM
    if (ptr)
        cudaFreeHost(ptr);
#else
    free(ptr);
#endif
}

static void fetch_to_host(VecEnv *v) {
    const size_t N = (size_t)v->num_envs;
    const KParams &p = v->base;
    const size_t frame = RES_W * RES_H * 3;
    uint8_t *rgb_dst = v->ob_direct ? (uint8_t *)v->h_ob[0] : v->st_rgb;
#ifndef PG_HOSTSIM
    if (!v->rgb_copy_enqueued)
        CUDA_CHECK(cudaMemcpyAsync(rgb_dst, p.rgb, N * frame, cudaMemcpyDeviceToHost, v->stream));
    v->rgb_copy_enqueued = false;
    CUDA_CHECK(cudaMemcpyAsync(v->st_rew, p.rew, N * sizeof(float), cudaMemcpyDeviceToHost, v->stream));
    CUDA_CHECK(cudaMemcpyAsync(v->st_first, p.first, N, cudaMemcpyDeviceToHost, v->stream));
    CUDA_CHECK(cudaMemcpyAsync(v->st_prev_seed, p.info_prev_level_seed, N * 4, cudaMemcpyDeviceToHost, v->stream));
    CUDA_CHECK(cudaMemcpyAsync(v->st_prev_complete, p.info_prev_level_complete, N, cudaMemcpyDeviceToHost, v->stream));
    CUDA_CHECK(cudaMemcpyAsync(v->st_seed, p.info_level_seed, N * 4, cudaMemcpyDeviceToHost, v->stream));
    CUDA_CHECK(cudaStreamSynchronize(v->stream));
#else
    memcpy(rgb_dst, p.rgb, N * frame);
    memcpy(v->st_rew, p.rew, N * sizeof(float));
    memcpy(v->st_first, p.first, N);
    memcpy(v->st_prev_seed, p.info_prev_level_seed, N * 4);
    memcpy(v->st_prev_complete, p.info_prev_level_complete, N);
    memcpy(v->st_seed, p.info_level_seed, N * 4);
#endif
    if (!v->ob_direct)
        for (size_t e = 0; e < N; e++) memcpy(v->h_ob[e], v->st_rgb + e * frame, frame);
    memcpy(v->h_rew, v->st_rew, N * sizeof(float));
    memcpy(v->h_first, v->st_first, N);
    for (size_t e = 0; e < N; e++) {
        *(int32_t *)v->h_info[0][e] = v->st_prev_seed[e];
        *(uint8_t *)v->h_info[1][e] = v->st_prev_complete[e];
        *(int32_t *)v->h_info[2][e] = v->st_seed[e];
    }
}

void libenv_set_buffers(libenv_env *handle, struct libenv_buffers *bufs) {
    VecEnv *v = (VecEnv *)handle;
    v->set_device();
    const size_t N = (size_t)v->num_envs;
    pg_fassert(!v->initial_reset_done);
    v->h_ob.assign(bufs->ob, bufs->ob + N);  // one observation space
    v->h_ac.assign(bufs->ac, bufs->ac + N);  // one action space
    v->h_info.resize(v->info_types.size());
    for (size_t s = 0; s < v->info_types.size(); s++) v->h_info[s].assign(bufs->info + s * N, bufs->info + (s + 1) * N);
    v->h_rew = bufs->rew;
    v->h_first = bufs->first;
    v->have_host_bufs = true;
    {
        // gym3 hands out one contiguous [N][64][64][3] array: page-lock it once and DMA into it
        // directly instead of bouncing 12 KiB/env through a staging buffer every step
        const size_t frame = RES_W * RES_H * 3;
        bool contiguous = true;
        for (size_t e = 1; e < N && contiguous; e++)
            contiguous = ((uint8_t *)v->h_ob[e] == (uint8_t *)v->h_ob[0] + e * frame);
        v->ob_direct = false;
#ifndef PG_HOSTSIM
        if (contiguous) {
            cudaPointerAttributes attr;
            if (cudaPointerGetAttributes(&attr, v->h_ob[0]) == cudaSuccess && attr.type == cudaMemoryTypeHost) {
                v->ob_direct = true;
            } else {
                cudaGetLastError();
                if (cudaHostRegister(v->h_ob[0], N * frame, cudaHostRegisterDefault) == cudaSuccess) {
                    v->ob_direct = true;
                    v->ob_registered = true;
                } else {
                    cudaGetLastError();
                }
            }
        }
#else
        v->ob_direct = contiguous;
#endif
    }
    v->st_rgb = v->ob_direct ? nullptr : (uint8_t *)host_alloc(N * RES_W * RES_H * 3);
    v->st_action = (int32_t *)host_alloc(N * 4);
    v->st_rew = (float *)host_alloc(N * 4);
    v->st_first = (uint8_t *)host_alloc(N);
    v->st_prev_seed = (int32_t *)host_alloc(N * 4);
    v->st_prev_complete = (uint8_t *)host_alloc(N);
    v->st_seed = (int32_t *)host_alloc(N * 4);
    v->ensure_initial_reset();  // vecgame.cpp:349-353
}

void libenv_observe(libenv_env *handle) {
    VecEnv *v = (VecEnv *)handle;
    v->set_device();
    pg_fassert(v->have_host_bufs);
    fetch_to_host(v);
}

void libenv_act(libenv_env *handle) {
    VecEnv *v = (VecEnv *)handle;
    v->set_device();
    pg_fassert(v->have_host_bufs);
    const size_t N = (size_t)v->num_envs;
    v->sync();  // staging buffer reuse (wait_for_stepping_threads, vecgame.cpp:379)
    for (size_t e = 0; e < N; e++) v->st_action[e] = *(int32_t *)v->h_ac[e];
#ifndef PG_HOSTSIM
    CUDA_CHECK(cudaMemcpyAsync(v->d_action, v->st_action, N * 4, cudaMemcpyHostToDevice, v->stream));
#else
    memcpy(v->d_action, v->st_action, N * 4);
#endif
    v->launch(false);
}

void libenv_close(libenv_env *handle) {
    VecEnv *v = (VecEnv *)handle;
    if (!v)
        return;
    v->set_device();
    v->sync();
    KParams &p = v->base;
    dev_free(p.hdr);
    dev_free(p.ents);
    dev_free(p.grid);
    dev_free(p.rng);
    dev_free(p.lvl_rng);
    dev_free(p.scratch);
    if (p.rot_scratch)
        dev_free(p.rot_scratch);
    dev_free(p.blit_list);
    dev_free(p.frame_setup);
    dev_free(p.cell_spill);
    dev_free(v->d_atlas);
    dev_free(v->d_tile_texels);
    dev_free(v->d_tile_index);
    dev_free(v->d_tile_sprites);
    dev_free(v->d_action);
    dev_free(p.rgb);
    dev_free(p.rew);
    dev_free(p.first);
    dev_free(p.info_prev_level_seed);
    dev_free(p.info_prev_level_complete);
    dev_free(p.info_level_seed);
    dev_free(v->d_lvl_seeds);
    dev_free(v->d_consumer_lut);
    if (p.dbg_cycles)
        dev_free(p.dbg_cycles);
#ifndef PG_HOSTSIM
    for (cudaEvent_t e : v->tev_pool) cudaEventDestroy(e);
#endif
#ifndef PG_HOSTSIM
    if (v->d_tickets)
        cudaFree(v->d_tickets);

#endif
    for (auto a : v->d_assets) dev_free(a);
    host_free(v->st_rgb);
#ifndef PG_HOSTSIM
    if (v->ob_registered)
        cudaHostUnregister(v->h_ob[0]);
#endif
    host_free(v->st_action);
    host_free(v->st_rew);
    host_free(v->st_first);
    host_free(v->st_prev_seed);
    host_free(v->st_prev_complete);
    host_free(v->st_seed);
#ifndef PG_HOSTSIM
    for (int s = 0; s < VecEnv::kAuxStreams; s++) {
        if (v->aux[s])
            cudaStreamDestroy(v->aux[s]);
        if (v->aux_hi[s])
            cudaStreamDestroy(v->aux_hi[s]);
        if (v->ev_link[s])
            cudaEventDestroy(v->ev_link[s]);
        if (v->ev_join[s])
            cudaEventDestroy(v->ev_join[s]);
    }
    if (v->ev_fork)
        cudaEventDestroy(v->ev_fork);
    if (v->own_stream)
        cudaStreamDestroy(v->own_stream);
#endif
    delete v;
}

int pgb200_get_device_buffers(libenv_env *handle, struct pgb200_device_buffers *out) {
    VecEnv *v = (VecEnv *)handle;
    v->set_device();
    v->ensure_initial_reset();
    const KParams &p = v->base;
    out->rgb = p.rgb;
    out->rew = p.rew;
    out->first = p.first;
    out->prev_level_seed = p.info_prev_level_seed;
    out->prev_level_complete = p.info_prev_level_complete;
    out->level_seed = p.info_level_seed;
    out->action = v->d_action;
    out->num_envs = v->num_envs;
    out->device = v->device;
#ifndef PG_HOSTSIM
    out->stream = (void *)v->stream;
#else
    out->stream = nullptr;
#endif
    return 0;
}

void pgb200_set_stream(libenv_env *handle, void *stream) {
    VecEnv *v = (VecEnv *)handle;
    v->set_device();
    v->sync();
#ifndef PG_HOSTSIM
    v->stream = (stream == PGB200_PRIVATE_STREAM) ? v->own_stream : (cudaStream_t)stream;
#else
    (void)stream;
#endif
}

int pgb200_set_rgb_mirror(libenv_env *handle, void *mirror0, void *mirror1) {
#ifndef PG_HOSTSIM
    VecEnv *v = (VecEnv *)handle;
    v->set_device();
    v->sync();
    v->mirror[0] = (uint8_t *)mirror0;
    v->mirror[1] = (uint8_t *)(mirror1 ? mirror1 : mirror0);
    v->mirror_parity = 0;
    return 0;
#else
    (void)handle; (void)mirror0; (void)mirror1;
    return -1;
#endif
}

int pgb200_set_consumer_output(libenv_env *handle, void *buffer, int dtype, int k_frames) {
#ifndef PG_HOSTSIM
    VecEnv *v = (VecEnv *)handle;
    v->set_device();
    v->ensure_initial_reset();
    v->sync();
    if (buffer == nullptr || dtype == 0) {
        v->base.consumer = nullptr;
        return 0;
    }
    if ((dtype != 1 && dtype != 2) || k_frames < 1 || k_frames > 16)
        return -1;
    if (!v->d_consumer_lut)
        v->d_consumer_lut = dev_alloc<uint16_t>(256);
    consumer_lut_kernel<<<1, 256, 0, v->stream>>>(v->d_consumer_lut, dtype == 2);
    CUDA_CHECK(cudaGetLastError());
    v->base.consumer = buffer;
    v->base.consumer_lut = v->d_consumer_lut;
    v->base.consumer_k = k_frames;
    v->base.consumer_slot = 0;
    v->consumer_steps = 0;
    // the current frame of every env becomes the newest frame of an otherwise empty stack
    for (size_t g = 0; g < v->games.size(); g++) {
        KParams p = v->base;
        p.assets = v->d_assets[g];
        p.game_id = v->games[g]->id;
        p.env_first = (int)g;
        p.env_step = (int)v->games.size();
        p.env_count = v->num_envs / (int)v->games.size();
        LaunchCtx lc = v->lctx();
        v->games[g]->observe_only[v->view[g]](p, lc);
    }
    v->sync();
    return 0;
#else
    (void)handle; (void)buffer; (void)dtype; (void)k_frames;
    return -1;
#endif
}

int pgb200_debug_phase_offset(void) {
#ifdef PG_PHASE_TIMING
    return (int)offsetof(EnvHdr, dbg_phase);
#else
    return -1;
#endif
}

int pgb200_debug_pixel_classes(libenv_env *handle, int env, uint8_t *out) {
    VecEnv *v = (VecEnv *)handle;
    if (env < 0 || env >= v->num_envs)
        return -1;
    v->set_device();
    v->sync();
    const size_t gi = (size_t)env % v->games.size();
    return v->games[gi]->pixel_classes[v->view[gi]](v->base, env, out);
}

int pgb200_consumer_slot(libenv_env *handle) { return ((VecEnv *)handle)->base.consumer_slot; }

int pgb200_mirror_parity(libenv_env *handle) { return ((VecEnv *)handle)->mirror_parity; }

void pgb200_act_device(libenv_env *handle) {
    VecEnv *v = (VecEnv *)handle;
    v->set_device();
    v->ensure_initial_reset();
    v->launch(false);
}

void pgb200_sync(libenv_env *handle) {
    VecEnv *v = (VecEnv *)handle;
    v->set_device();
    v->sync();
}

uint32_t pgb200_get_errors(libenv_env *handle, uint32_t *host_out) {
    VecEnv *v = (VecEnv *)handle;
    v->set_device();
    v->sync();
    const size_t N = (size_t)v->num_envs;
    std::vector<EnvHdr> hdr(N);
#ifndef PG_HOSTSIM
    CUDA_CHECK(cudaMemcpy(hdr.data(), v->base.hdr, N * sizeof(EnvHdr), cudaMemcpyDeviceToHost));
#else
    memcpy(hdr.data(), v->base.hdr, N * sizeof(EnvHdr));
#endif
    uint32_t any = 0;
    for (size_t e = 0; e < N; e++) {
        if (host_out)
            host_out[e] = hdr[e].err;
        any |= hdr[e].err;
    }
    return any;
}

int pgb200_debug_cycles(libenv_env *handle, uint32_t *host_out) {
    VecEnv *v = (VecEnv *)handle;
    if (!v->base.dbg_cycles)
        return -1;
    v->set_device();
    v->sync();
#ifndef PG_HOSTSIM
    CUDA_CHECK(cudaMemcpy(host_out, v->base.dbg_cycles, (size_t)v->num_envs * 4, cudaMemcpyDeviceToHost));
#endif
    return 0;
}

int pgb200_debug_read_env(libenv_env *handle, int env, void *hdr_out, void *ents_out, int max_ents) {
    VecEnv *v = (VecEnv *)handle;
    v->set_device();
    v->sync();
    EnvHdr hdr;
    const KParams &p = v->base;
#ifndef PG_HOSTSIM
    CUDA_CHECK(cudaMemcpy(&hdr, p.hdr + env, sizeof(EnvHdr), cudaMemcpyDeviceToHost));
#else
    memcpy(&hdr, p.hdr + env, sizeof(EnvHdr));
#endif
    if (hdr_out)
        memcpy(hdr_out, &hdr, sizeof(EnvHdr));
    int n = hdr.n_ents < max_ents ? hdr.n_ents : max_ents;
    if (ents_out && n > 0) {
#ifndef PG_HOSTSIM
        CUDA_CHECK(cudaMemcpy(ents_out, p.ents + (size_t)env * p.ent_stride, (size_t)n * sizeof(Entity), cudaMemcpyDeviceToHost));
#else
        memcpy(ents_out, p.ents + (size_t)env * p.ent_stride, (size_t)n * sizeof(Entity));
#endif
    }
    return hdr.n_ents;
}

// ---- get_state / set_state (vecgame.cpp:437-457)
static void copy_from_dev(void *dst, const void *src, size_t bytes) {
#ifndef PG_HOSTSIM
    CUDA_CHECK(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
#else
    memcpy(dst, src, bytes);
#endif
}

static void fetch_env(VecEnv *v, int env, host::HostEnv &e) {
    const KParams &p = v->base;
    e.ent_cap = p.ent_stride - 1;
    e.ents.resize((size_t)p.ent_stride);
    e.grid.resize((size_t)p.grid_stride);
    e.scratch.resize((size_t)p.scratch_stride);
    copy_from_dev(&e.h, p.hdr + env, sizeof(EnvHdr));
    copy_from_dev(e.ents.data(), p.ents + (size_t)env * p.ent_stride, e.ents.size() * sizeof(Entity));
    copy_from_dev(e.grid.data(), p.grid + (size_t)env * p.grid_stride, e.grid.size() * sizeof(int16_t));
    copy_from_dev(&e.rng, p.rng + env, sizeof(MT19937));
    copy_from_dev(&e.lvl_rng, p.lvl_rng + env, sizeof(MT19937));
    if (!e.scratch.empty())
        copy_from_dev(e.scratch.data(), p.scratch + (size_t)env * p.scratch_stride, e.scratch.size() * sizeof(int32_t));
}

static void store_env(VecEnv *v, int env, const host::HostEnv &e) {
    const KParams &p = v->base;
    copy_to_dev(p.hdr + env, &e.h, sizeof(EnvHdr));
    copy_to_dev(p.ents + (size_t)env * p.ent_stride, e.ents.data(), e.ents.size() * sizeof(Entity));
    copy_to_dev(p.grid + (size_t)env * p.grid_stride, e.grid.data(), e.grid.size() * sizeof(int16_t));
    copy_to_dev(p.rng + env, &e.rng, sizeof(MT19937));
    copy_to_dev(p.lvl_rng + env, &e.lvl_rng, sizeof(MT19937));
    if (!e.scratch.empty())
        copy_to_dev(p.scratch + (size_t)env * p.scratch_stride, e.scratch.data(), e.scratch.size() * sizeof(int32_t));
}

int get_state(libenv_env *handle, int env_idx, char *data, int length) {
    VecEnv *v = (VecEnv *)handle;
    v->set_device();
    pg_fassert(env_idx >= 0 && env_idx < v->num_envs);
    v->ensure_initial_reset();
    v->sync();  // wait_for_stepping_threads
    host::HostEnv e;
    fetch_env(v, env_idx, e);
    const GameVTable *g = v->games[(size_t)env_idx % v->games.size()];
    try {
        host::WriteBuf b(data, (size_t)(length < 0 ? 0 : length));
        host::serialize_env(g->name, g->id, e, v->const_fields, b);
        return (int)b.offset;
    } catch (const std::exception &ex) {
        pg_fatal("get_state: %s\n", ex.what());
    }
    return 0;
}

void set_state(libenv_env *handle, int env_idx, char *data, int length) {
    VecEnv *v = (VecEnv *)handle;
    v->set_device();
    pg_fassert(env_idx >= 0 && env_idx < v->num_envs);
    v->ensure_initial_reset();
    v->sync();
    host::HostEnv e;
    fetch_env(v, env_idx, e);  // capacities, game id and the fields the blob does not carry
    const size_t gi = (size_t)env_idx % v->games.size();
    const GameVTable *g = v->games[gi];
    try {
        host::ReadBuf b(data, (size_t)(length < 0 ? 0 : length));
        host::deserialize_env(g->name, g->id, e, b);
    } catch (const std::exception &ex) {
        pg_fatal("set_state: %s\n", ex.what());
    }
    store_env(v, env_idx, e);
#ifndef PG_HOSTSIM
    CUDA_CHECK(cudaDeviceSynchronize());  // the uploads ran on the legacy stream; the kernels below do not order against it
#endif
    // Game::observe(): re-render this env and rewrite its rew / first / info slots from the restored step_data
    KParams p = v->base;
    p.assets = v->d_assets[gi];
    p.game_id = g->id;
    p.env_first = env_idx;
    p.env_step = 1;
    p.env_count = 1;
    LaunchCtx lc = v->lctx();
    g->observe_only[v->view[gi]](p, lc);
    v->sync();
    v->rgb_copy_enqueued = false;  // a DMA started behind the last step predates this frame: observe copies again
}

int pgb200_frame_info(const char *game, int *frame_bytes, int *ctas_per_sm) {
    const GameVTable *g = find_game(game);
    if (!g)
        return -1;
    *frame_bytes = g->frame_bytes[0];
    *ctas_per_sm = g->render_ctas_per_sm[0];
    return 0;
}

int64_t pgb200_kernel_launches(libenv_env *handle) { return ((VecEnv *)handle)->launches; }

void pgb200_set_launch_shape(libenv_env *handle, int chunks, int serialize) {
    VecEnv *v = (VecEnv *)handle;
    v->set_device();
    v->sync();
    v->force_chunks = chunks;
    v->serialize_launches = serialize != 0;
}

int pgb200_kernel_timing_begin(libenv_env *handle, int max_launch_pairs) {
#ifndef PG_HOSTSIM
    VecEnv *v = (VecEnv *)handle;
    v->set_device();
    v->sync();
    while ((int)v->tev_pool.size() < 4 * max_launch_pairs) {
        cudaEvent_t e;
        CUDA_CHECK(cudaEventCreate(&e));
        v->tev_pool.push_back(e);
    }
    v->tev_used = 0;
    v->tev_envs.clear();
    v->timing = true;
    return 0;
#else
    return -1;
#endif
}

int pgb200_kernel_timing_end(libenv_env *handle, double *out) {
#ifndef PG_HOSTSIM
    VecEnv *v = (VecEnv *)handle;
    v->set_device();
    v->sync();
    v->timing = false;
    double logic_ms = 0, setup_ms = 0, render_ms = 0, envs = 0;
    const int pairs = (int)(v->tev_used / 4);
    for (int i = 0; i < pairs; i++) {
        float a = 0, b = 0, c2 = 0;
        CUDA_CHECK(cudaEventElapsedTime(&a, v->tev_pool[4 * i], v->tev_pool[4 * i + 1]));
        CUDA_CHECK(cudaEventElapsedTime(&b, v->tev_pool[4 * i + 1], v->tev_pool[4 * i + 2]));
        CUDA_CHECK(cudaEventElapsedTime(&c2, v->tev_pool[4 * i + 2], v->tev_pool[4 * i + 3]));
        logic_ms += a;
        setup_ms += b;
        render_ms += c2;
        envs += v->tev_envs[i];
    }
    out[0] = logic_ms;
    out[1] = render_ms;
    out[2] = pairs;
    out[3] = envs;
    out[4] = setup_ms;
    v->tev_used = 0;
    v->tev_envs.clear();
    return pairs;
#else
    return -1;
#endif
}

}  // extern "C"
