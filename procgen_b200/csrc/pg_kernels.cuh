// Per-env work items (logic phase, render phases) and the launch parameter block. The CUDA
// kernels in pg_runtime.cu are thin wrappers that map one CTA to one env and put barriers between
// the phases; the CPU debug harness runs the very same phase functions in plain loops.
#pragma once
#include "pg_raster.cuh"

namespace pg {

struct KParams {
    // state (HBM)
    EnvHdr *hdr;
    Entity *ents;
    int16_t *grid;
    MT19937 *rng;
    MT19937 *lvl_rng;
    int32_t *scratch;
    RotBlit *rot_scratch;       // [N][rot_stride] rotated-sprite / span records
    Blit *blit_list;            // [N][blit_stride] background-less blit lists (entities in draw order, then overlays)
    unsigned char *frame_setup; // [N][frame_setup_stride bytes] FrameSetupT of the env's game
    Blit *cell_spill;           // [N][cell_spill_stride] general cell blits that do not fit the render CTA's shared memory
    const GameAssets *assets;   // table of the game this launch handles
    const uint32_t *atlas;
    TileTable tiles;            // pre-scaled cell tiles of every sprite (texels == nullptr: disabled)
    // libenv-visible buffers (vecgame.cpp:212-268), one slot per env
    const int32_t *action;
    uint8_t *rgb;               // [N][64][64][3]
    float *rew;
    uint8_t *first;
    int32_t *info_prev_level_seed;
    uint8_t *info_prev_level_complete;
    int32_t *info_level_seed;
    const uint32_t *lvl_seeds;  // per-env seed for level_seed_rand_gen (vecgame.cpp:301-314)
    // strides (elements)
    int32_t ent_stride;         // ent_cap + 1 (ghost slot)
    int32_t grid_stride;
    int32_t scratch_stride;
    int32_t rot_stride;
    int32_t blit_stride;
    int32_t frame_setup_stride;
    int32_t cell_spill_stride;
    // which envs this launch covers: env = env_first + i * env_step, i in [0, env_count)
    int32_t env_first, env_step, env_count;
    // construction-time options (game.cpp:42-75, vecgame.cpp:284-293)
    Options options;
    int32_t level_seed_low, level_seed_high;
    int32_t game_id;
    int32_t fixed_asset_seed;   // FNV-1a of the game name (vecgame.cpp:156-167, 324-327)
    int32_t snap;
    int32_t env_global_offset;  // game_n = env_global_offset + env
    // optional second output for on-device learners (SURVEY §8(f)4): normalised fp16 / bf16, planar
    // CHW, k-frame stack kept as a 2k-slot ring so that the ordered stack is always one contiguous view
    void *consumer;             // [N][slots][3][64][64] 16-bit elements; null = off
    const uint16_t *consumer_lut;  // [256] = (16-bit float)(v / 255.f)
    int32_t consumer_k;         // frames per stack; slots = k == 1 ? 1 : 2k
    int32_t consumer_slot;      // ring position this step writes: t mod k
    uint32_t *dbg_cycles;       // optional [N] per-env logic duration in SM cycles (profiling aid)
};

PG_HD Ctx make_ctx(const KParams &p, int env) {
    Ctx c;
    c.h = p.hdr + env;
    c.ents = p.ents + (size_t)env * p.ent_stride;
    c.grid = p.grid + (size_t)env * p.grid_stride;
    c.rng = p.rng + env;
    c.lvl_rng = p.lvl_rng + env;
    c.assets = p.assets;
    c.scratch = p.scratch + (size_t)env * p.scratch_stride;
    c.ent_cap = p.ent_stride - 1;
    c.grid_cap = p.grid_stride;
    c.scratch_cap = p.scratch_stride;
    c.obst_hi = -1;
    c.rot_scratch_raw = (p.rot_scratch && p.rot_stride > 0) ? (void *)(p.rot_scratch + (size_t)env * p.rot_stride) : nullptr;
    c.blit_list = p.blit_list ? p.blit_list + (size_t)env * p.blit_stride : nullptr;
    c.cell_spill = p.cell_spill ? p.cell_spill + (size_t)env * p.cell_spill_stride : nullptr;
    ctx_refresh(c);
    return c;
}

// Game::observe's scalar stores (game.cpp:160-164)
PG_HD void write_step_outputs(const KParams &p, int env, const EnvHdr &h) {
    p.rew[env] = h.reward;
    p.first[env] = (uint8_t)(h.done != 0);
    p.info_prev_level_seed[env] = h.prev_level_seed;
    p.info_prev_level_complete[env] = (uint8_t)(h.level_complete != 0);
    p.info_level_seed[env] = h.current_level_seed;
}

// Construction + first reset (VecGame ctor per-env part vecgame.cpp:309-330, then
// set_buffers -> reset(); observe(), vecgame.cpp:349-353). One thread.
template <class G, class Frame>
PG_HD void env_init_logic(const KParams &p, int env) {
    Ctx c = make_ctx(p, env);
    G::init_constants(c);
    ctx_refresh(c);
    EnvHdr &h = *c.h;
    h.options = p.options;
    h.game_id = p.game_id;
    h.fixed_asset_seed = p.fixed_asset_seed;
    h.game_n = p.env_global_offset + env;
    h.level_seed_low = p.level_seed_low;
    h.level_seed_high = p.level_seed_high;
    mt_seed(*c.lvl_rng, p.lvl_seeds[env]);
    c.rng->seeded = 0;
    Engine<G>::reset(c);
    h.initial_reset_complete = 1;
    Raster<G, Frame>::prepare_camera(c);
    write_step_outputs(p, env, h);
}

#if defined(__CUDACC__)
// Warm the env's working set. A step's logic is one long dependent chain; touched cold, every
// entity record / header line / grid row costs a serial DRAM round trip. Here the 32 lanes issue
// all those line fetches at once (prefetch.global.L2 + L1), so the chain later runs on cache hits.
__device__ __forceinline__ void pg_prefetch_line(const void *ptr) {
    asm volatile("prefetch.global.L1 [%0];" ::"l"(ptr));
}
__device__ __forceinline__ void env_prefetch(const KParams &p, int env) {
    const int lane = (int)(threadIdx.x & 31u);
    const char *hdr = reinterpret_cast<const char *>(p.hdr + env);
    if (lane < (int)((sizeof(EnvHdr) + 127) / 128))
        pg_prefetch_line(hdr + lane * 128);
    const MT19937 *rng = p.rng + env;
    if (lane == 8)
        pg_prefetch_line(&rng->p);
    const Entity *ents = p.ents + (size_t)env * p.ent_stride;
    const int n = p.hdr[env].n_ents;   // first demand load (same line as the prefetch above)
    for (int i = lane; i < n; i += 32) pg_prefetch_line(ents + i);
    // RNG words of the next draw and the grid rows around the agent
    if (lane == 9) {
        int k = rng->p >= 624 ? 0 : rng->p;
        pg_prefetch_line(&rng->mt[k]);
        pg_prefetch_line(&rng->mt[(k + 397) % 624]);
    }
    if (lane >= 16 && lane < 24 && n > 0) {
        const EnvHdr &h = p.hdr[env];
        const Entity &a = ents[h.agent_idx];
        int row = (int)a.y + (lane - 16) - 3;
        if (row >= 0 && row < h.main_height) {
            int col = (int)a.x - 4;
            if (col < 0) col = 0;
            pg_prefetch_line(p.grid + (size_t)env * p.grid_stride + row * h.main_width + col);
        }
    }
    __syncwarp();
}
#endif

// Game::step (game.cpp:120-155) up to, not including, the pixel work. One thread.
template <class G, class Frame>
PG_HD void env_step_logic(const KParams &p, int env) {
#if defined(__CUDA_ARCH__)
    env_prefetch(p, env);
#endif
    Ctx c = make_ctx(p, env);
    c.h->action = p.action[env];  // vecgame.cpp:388
    Engine<G>::step(c);
    Raster<G, Frame>::prepare_camera(c);
    write_step_outputs(p, env, *c.h);
}

// ---- setup kernel body: one warp (lanes `lane` of `nlanes`) prepares everything about env's frame that
// does not depend on pixels or cells: camera, spans, background / overlay / entity blits
template <class G, class Setup>
PG_HD void env_setup_frame(const KParams &p, int env, Setup &f, int lane, int nlanes) {
    Ctx c = make_ctx(p, env);
    using R = Raster<G, Setup>;
    R::setup_frame(c, f, p.snap != 0, lane, nlanes);
#if defined(__CUDA_ARCH__)
    __syncwarp();
#endif
    R::build_entity_blits(c, f, lane, nlanes);
#if defined(__CUDA_ARCH__)
    __syncwarp();
#endif
    if (f.n_jobs > 0) {
        R::frame_tiles(c, f, lane, nlanes);
#if defined(__CUDA_ARCH__)
        __syncwarp();
#endif
    }
    if (G::DEFER_ROTATED) {
        R::frame_rots(c, f, lane, nlanes);
#if defined(__CUDA_ARCH__)
        __syncwarp();
#endif
    }
    if (lane == 0)
        R::frame_append_overlays(f);
    // cells: pixel -> cell lookups, classification, the tiles they need and where those will sit in the
    // render CTA's arena
    if (G::DRAWS_GRID) {
#if defined(__CUDA_ARCH__)
        __syncwarp();
#endif
        R::frame_build(c, f, lane, nlanes, 0);
#if defined(__CUDA_ARCH__)
        __syncwarp();
#endif
        R::frame_tile_alloc(c, f, p.tiles, lane, nlanes);
#if defined(__CUDA_ARCH__)
        __syncwarp();
#endif
        R::frame_cells_finish(c, f, lane, nlanes);
    } else {
        R::frame_build(c, f, lane, nlanes, 0);  // background row offsets only
    }
}

// Host debug harness twin of the bulk copies that stage the frame's tiles
template <class Frame>
PG_HD void env_stage_tiles_serial(const KParams &p, Frame &f) {
    const int nj = f.n_tjobs < MAX_TILE_JOBS ? f.n_tjobs : MAX_TILE_JOBS;
    for (int j = 0; j < nj; j++)
        for (int w = 0; w < (int)f.tjob[j].words; w++) f.arena[f.tjob[j].dst + w] = p.tiles.texels[f.tjob[j].src + w];
}

// Compose the rows row_first, row_first + row_step, ... of the frame (`lane` of `nlanes` threads own them)
template <class G, class Frame>
PG_HD void env_render_compose(const KParams &p, Frame &f, int row_first, int row_step, int lane, int nlanes, uint32_t *dbg = nullptr) {
    Raster<G, Frame>::compose_rows(f, f.fb, row_first, row_step, lane, nlanes, p.atlas, dbg);
}

// Fill one tile of the global table (TileTable): tile (slot, tw, th) = the texels an un-clipped
// drawImage of the sprite at snapped size tw x th samples, by the general path's own arithmetic.
PG_HD void tile_table_fill(const SpriteDesc *sprites, const uint32_t *index, uint32_t *texels, const uint32_t *atlas, int slot, int tw, int th, int tid,
                           int nthreads) {
    Blit b;
    make_image_blit(b, 0.0, 0.0, (double)tw, (double)th, sprites[slot], false, 256, true);
    uint32_t *dst = texels + index[(slot * MAX_TILE_DIM + (tw - 1)) * MAX_TILE_DIM + (th - 1)];
    const int words = tile_words(tw, th);
    for (int i = tid; i < words; i += nthreads) {
        const int dy = i / tw, dx = i - dy * tw;
        dst[i] = dy < th ? tile_texel(b, atlas, dx, dy) : 0u;
    }
}

// Frame sizing per game: visible window (cells per side) and entity capacity.
// VIEW = cells per side of the largest visible grid window: G::MAX_VIEW_CELLS for the game's usual view,
// G::FULL_VIEW_CELLS for the whole-world view the scrolling games draw with center_agent = false
template <class G, int VIEW = G::MAX_VIEW_CELLS>
struct FrameFor {
    using type = FrameT<(G::DRAWS_GRID ? VIEW : 1), G::MAX_VISIBLE_ENTS, G::MAX_ROT_BLITS>;
    using setup = FrameSetupT<(G::DRAWS_GRID ? VIEW : 1), G::MAX_VISIBLE_ENTS, G::MAX_ROT_BLITS>;
    using shared = typename type::Shared;
};

}  // namespace pg
