// Kernels, launch wrappers and the per-game dispatch table. Included by pg_runtime.cu (host runtime +
// C ABI) and by one translation unit per game (games_tu/tu_<game>.cu), so the 16 games compile in
// parallel; a game's kernels are instantiated only in its own unit.
#pragma once
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "pg_kernels.cuh"

#ifndef PG_HOSTSIM
#include <cuda_runtime.h>
#endif

namespace pg {

// ================================================================= errors (cpp-utils.cpp:8-20)
static inline void pg_fatal(const char *fmt, ...) {
    fprintf(stderr, "fatal: ");
    va_list args;
    va_start(args, fmt);
    vfprintf(stderr, fmt, args);
    va_end(args);
    exit(EXIT_FAILURE);
}
#define pg_fassert(cond)                                                                  \
    do {                                                                                  \
        if (!(cond)) {                                                                    \
            fprintf(stderr, "fassert failed '%s' at %s:%d\n", #cond, __FILE__, __LINE__); \
            exit(EXIT_FAILURE);                                                           \
        }                                                                                 \
    } while (0)

#ifndef PG_HOSTSIM
#define CUDA_CHECK(expr)                                                                          \
    do {                                                                                          \
        cudaError_t _e = (expr);                                                                  \
        if (_e != cudaSuccess)                                                                    \
            pg_fatal("CUDA error %s at %s:%d: %s\n", cudaGetErrorName(_e), __FILE__, __LINE__, cudaGetErrorString(_e)); \
    } while (0)
#endif

// ================================================================= kernels
// Two launches per step:
//   logic_kernel   one WARP per env. All 32 lanes execute the serial game logic redundantly and in
//                  lockstep (every load/store is warp-uniform), and fan out only inside
//                  pg_scan_down, which turns the reference's O(E) entity-collision loops into E/32
//                  ballots. A warp, not a thread, is the unit so unrelated envs never diverge
//                  against each other and dozens of envs per SM hide each other's load latency.
//   render_kernel  one CTA per env: blit-list build + per-pixel gather + packed RGB store
#ifndef PG_LOGIC_WARPS
#define PG_LOGIC_WARPS 2
#endif
#ifndef PG_LOGIC_MIN_BLOCKS
#define PG_LOGIC_MIN_BLOCKS 24
#endif
#ifndef PG_STEP_CHUNKS
#define PG_STEP_CHUNKS 8
#endif
#ifndef PG_AUX_STREAMS
#define PG_AUX_STREAMS 16   // one per game of the 16-game list: the slow games (level generation) must not queue behind each other
#endif
constexpr int kLogicThreads = 32 * PG_LOGIC_WARPS;  // one warp = one env; few warps per CTA so a finished
constexpr int kLogicEnvsPerBlock = PG_LOGIC_WARPS;  // env frees its slot without waiting on many siblings
constexpr int kRenderThreads = 128;

#ifndef PG_HOSTSIM
// Persistent: the grid is sized to fill the machine once and every warp pulls env indices from a
// global ticket counter until the launch's range is exhausted, so a long env (level reset) only
// delays its own warp and no SM slot idles waiting for a block launch.
template <class G, bool INIT>
__global__ void __launch_bounds__(kLogicThreads, PG_LOGIC_MIN_BLOCKS) logic_kernel(KParams p, unsigned int *ticket) {
    using Frame = typename FrameFor<G>::type;
    const unsigned lane = threadIdx.x & 31u;
    while (true) {
        unsigned t = 0;
        if (lane == 0)
            t = atomicAdd(ticket, 1u);
        t = __shfl_sync(0xffffffffu, t, 0);
        if (t >= (unsigned)p.env_count)
            break;
        const int env = p.env_first + (int)t * p.env_step;
        const long long t0 = p.dbg_cycles ? clock64() : 0;
        if (INIT)
            env_init_logic<G, Frame>(p, env);
        else
            env_step_logic<G, Frame>(p, env);
        __syncwarp();
        if (p.dbg_cycles && lane == 0)
            p.dbg_cycles[env] = (uint32_t)(clock64() - t0);
    }
}

// Frame setup: one warp per env (4 envs per block). Everything about a frame that is O(entities +
// cell columns): camera, visible window, per-column / per-row pixel spans, background, overlay and
// entity blits (incl. the scan conversion of rotated sprites). Every warp of the grid runs this
// same code, which is what the instruction cache wants; the render kernel that follows — one CTA
// per env — is left with the O(pixels + cells) work and picks the result up with one bulk copy.
constexpr int kSetupThreads = 128;
#ifndef PG_SETUP_MIN_BLOCKS
#define PG_SETUP_MIN_BLOCKS 8   // measured (profiles/r02_ab_setup_kernel_occupancy.txt): 64 registers x 32 warps/SM beats 96 x 20
#endif
template <class G, int VIEW>
__global__ void __launch_bounds__(kSetupThreads, PG_SETUP_MIN_BLOCKS) setup_kernel(KParams p) {
    using Setup = typename FrameFor<G, VIEW>::setup;
    const int i = (int)blockIdx.x * (kSetupThreads / 32) + (int)(threadIdx.x >> 5);
    if (i >= p.env_count)
        return;
    const int env = p.env_first + i * p.env_step;
    Setup &f = *reinterpret_cast<Setup *>(p.frame_setup + (size_t)env * p.frame_setup_stride);
    env_setup_frame<G, Setup>(p, env, f, (int)(threadIdx.x & 31u), 32);
}

#ifndef PG_RENDER_CTAS_PER_SM
#define PG_RENDER_CTAS_PER_SM 0  // 0 = as many as registers / the frame allow
#endif
// Resident CTAs per SM the render kernel is compiled for: as many as the frame (shared memory)
// allows; the register cap follows (65536 / (128 * CTAs)).
template <class G, int VIEW>
struct RenderTune {
    static constexpr size_t kFrameBytes = sizeof(typename FrameFor<G, VIEW>::type);
#ifdef PG_RENDER_MIN_BLOCKS
    static constexpr int kMinBlocks = PG_RENDER_MIN_BLOCKS;
#else
    // 227 KiB usable per SM, 1 KiB reserved per resident CTA
    static constexpr int kFit = (int)((227 * 1024) / (kFrameBytes + 1024 + 16));
    // 8 CTAs = 64 registers, which the gather fits without spilling (profiles/r03_ab_render_ctas.txt)
    static constexpr int kWant = 8;
    static constexpr int kMinBlocks = kFit >= kWant ? kWant : (kFit >= 1 ? kFit : 1);
#endif
};

// ---- async-proxy plumbing (PTX): mbarrier + bulk copies (the TMA engine's 1-D mode; SASS UBLKCP)
__device__ __forceinline__ uint32_t pg_smem_addr(const void *ptr) { return (uint32_t)__cvta_generic_to_shared(ptr); }
__device__ __forceinline__ void pg_mbar_init(unsigned long long *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(pg_smem_addr(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void pg_mbar_arrive_expect_tx(unsigned long long *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(pg_smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void pg_mbar_expect_tx(unsigned long long *bar, unsigned bytes) {
    asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(pg_smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void pg_mbar_wait(unsigned long long *bar, unsigned parity) {
    unsigned done = 0;
    while (!done) {  // try_wait suspends the thread in hardware for a while before it returns false
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(pg_smem_addr(bar)), "r"(parity)
            : "memory");
    }
}
// global -> shared, completion counted on the mbarrier; 16-byte aligned, size a multiple of 16
__device__ __forceinline__ void pg_bulk_load(void *dst_smem, const void *src_gmem, unsigned bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(pg_smem_addr(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(pg_smem_addr(bar))
                 : "memory");
}
// shared -> global; returns once the engine has read the source (the CTA may then exit / reuse it)
__device__ __forceinline__ void pg_bulk_store_and_wait(void *dst_gmem, const void *src_smem, unsigned bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(pg_smem_addr(src_smem)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

// One CTA renders one env's frame:
//   stage                  warp 0 arms the mbarrier and queues the bulk copies: what the setup kernel prepared
//                          (spans, background, counts, cell map, lookups) and one per pre-scaled tile (global
//                          table -> shared arena)
//   compose                warp w owns rows y = w (mod 4): gather (cells over background; a lane = 4 pixel
//                          columns x 8 rows), then paint the entity blits in draw order, lanes sharing each blit
//   pack + store           RGB32 -> RGB888 in place, one bulk copy of the 12 KiB frame to the observation buffer
template <class G, int VIEW>
__global__ void __launch_bounds__(kRenderThreads, RenderTune<G, VIEW>::kMinBlocks) render_kernel(KParams p) {
    using Frame = typename FrameFor<G, VIEW>::type;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Frame &f = *reinterpret_cast<Frame *>(smem_raw);
    const int env = p.env_first + (int)blockIdx.x * p.env_step;
    const int tid = (int)threadIdx.x;
#ifdef PG_PHASE_TIMING
    long long t0 = clock64(), t1;
#define PG_RENDER_PHASE(id)                                       \
    do {                                                          \
        t1 = clock64();                                           \
        if (tid == 0)                                             \
            p.hdr[env].dbg_phase[id] = (uint32_t)(t1 - t0);       \
        t0 = t1;                                                  \
    } while (0)
#else
#define PG_RENDER_PHASE(id) do { } while (0)
#endif
    using Shared = typename FrameFor<G, VIEW>::shared;
    using Setup = typename FrameFor<G, VIEW>::setup;
    const Setup *gs = reinterpret_cast<const Setup *>(p.frame_setup + (size_t)env * p.frame_setup_stride);
    if (tid == 0)
        pg_mbar_init(&f.mbar, 1);
    __syncthreads();
    if (tid < 32) {
        // Everything the setup kernel prepared for this env — one bulk copy into the head of the frame —
        // and the pre-scaled tiles its cells need, one bulk copy each, all counted on one mbarrier phase.
        // The record's copy goes first: its bytes are expected without arriving, so the phase cannot
        // complete before the tile bytes are expected too (by the arrival, after the job records are read).
        if (tid == 0) {
            pg_mbar_expect_tx(&f.mbar, (unsigned)sizeof(Shared));
            pg_bulk_load(static_cast<Shared *>(&f), static_cast<const Shared *>(gs), (unsigned)sizeof(Shared), &f.mbar);
        }
        const int nj = G::DRAWS_GRID ? (gs->n_tjobs < MAX_TILE_JOBS ? gs->n_tjobs : MAX_TILE_JOBS) : 0;
        TileJob job = {0u, 0, 0};
        if (tid < nj)
            job = gs->tjob[tid];
        unsigned words = job.words;
        for (int j = tid + 32; j < nj; j += 32) words += gs->tjob[j].words;
        for (int d = 16; d > 0; d >>= 1) words += __shfl_xor_sync(0xffffffffu, words, d);
        if (tid == 0)
            pg_mbar_arrive_expect_tx(&f.mbar, 4u * words);
        __syncwarp();
        if (tid < nj)
            pg_bulk_load(f.arena + job.dst, p.tiles.texels + job.src, 4u * job.words, &f.mbar);
        for (int j = tid + 32; j < nj; j += 32)
            pg_bulk_load(f.arena + gs->tjob[j].dst, p.tiles.texels + gs->tjob[j].src, 4u * gs->tjob[j].words, &f.mbar);
    }
    pg_mbar_wait(&f.mbar, 0);
    PG_RENDER_PHASE(0);
    // warp w owns rows y = w (mod warps): gather and paint need no block barrier in between
#ifdef PG_PHASE_TIMING
    env_render_compose<G, Frame>(p, f, tid >> 5, kRenderThreads >> 5, tid & 31, 32, p.hdr[env].dbg_phase + 8);  // 8 gather, 9 paint
#else
    env_render_compose<G, Frame>(p, f, tid >> 5, kRenderThreads >> 5, tid & 31, 32);
#endif
    __syncthreads();
    PG_RENDER_PHASE(5);
    if (p.consumer != nullptr) {
        // Consumer epilogue: the frame as normalised 16-bit floats, planar, into ring slot s (and its
        // twin s + k); an env that starts an episode this step gets the older frames of its window
        // zeroed (the frame-stack convention of baselines' VecFrameStack). Thread = pixel pairs.
        const int kf = p.consumer_k, s = p.consumer_slot;
        const int slots = kf == 1 ? 1 : 2 * kf;
        uint32_t *base = reinterpret_cast<uint32_t *>(p.consumer) + (size_t)env * slots * (3 * RES_W * RES_H / 2);
        const uint16_t *lut = p.consumer_lut;
        for (int pair = tid; pair < RES_W * RES_H / 2; pair += kRenderThreads) {
            const uint32_t c0 = f.fb[2 * pair], c1 = f.fb[2 * pair + 1];
#pragma unroll
            for (int ch = 0; ch < 3; ch++) {
                const int sh = 16 - 8 * ch;  // R, G, B planes
                const uint32_t v = (uint32_t)lut[(c0 >> sh) & 0xffu] | ((uint32_t)lut[(c1 >> sh) & 0xffu] << 16);
                base[(size_t)(s * 3 + ch) * (RES_W * RES_H / 2) + pair] = v;
                if (kf > 1)
                    base[(size_t)((s + kf) * 3 + ch) * (RES_W * RES_H / 2) + pair] = v;
            }
        }
        if (kf > 1 && p.first[env]) {
            // window of this step = ring slots s+1 .. s+k (the newest is s+k); zero the k-1 older ones
            // wherever they live: slot j and its twin j +- k
            for (int j = 1; j < kf; j++) {
                const int a = (s + j) % kf;
                for (int w = tid; w < 3 * RES_W * RES_H / 2; w += kRenderThreads) {
                    base[(size_t)a * (3 * RES_W * RES_H / 2) + w] = 0u;
                    base[(size_t)(a + kf) * (3 * RES_W * RES_H / 2) + w] = 0u;
                }
            }
        }
    }
    {
        // RGB32 -> RGB888 in place: every thread reads its 8 pixel quads, then (barrier) writes them packed
        constexpr int kQuadsPerThread = RES_W * RES_H / 4 / kRenderThreads;
        uint32_t c[kQuadsPerThread][4];
#pragma unroll
        for (int j = 0; j < kQuadsPerThread; j++) {
            const uint4 v = reinterpret_cast<const uint4 *>(f.fb)[tid + j * kRenderThreads];
            c[j][0] = v.x; c[j][1] = v.y; c[j][2] = v.z; c[j][3] = v.w;
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < kQuadsPerThread; j++) Raster<G, Frame>::pack_quad(c[j], f.fb + 3 * (tid + j * kRenderThreads));
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes of f.fb -> visible to the bulk copy
    __syncthreads();
    PG_RENDER_PHASE(6);
    if (tid == 0)
        pg_bulk_store_and_wait(p.rgb + (size_t)env * (RES_W * RES_H * 3), f.fb, RES_W * RES_H * 3);
    PG_RENDER_PHASE(7);
#undef PG_RENDER_PHASE
}

#endif

#ifndef PG_HOSTSIM
// Game::observe without a step (set_state, vecgame.cpp:454-456): camera, then the render kernel
template <class G>
__global__ void camera_kernel(KParams p) {
    using Frame = typename FrameFor<G>::type;
    if (threadIdx.x == 0 && blockIdx.x < (unsigned)p.env_count) {
        const int env = p.env_first + (int)blockIdx.x * p.env_step;
        Ctx c = make_ctx(p, env);
        Raster<G, Frame>::prepare_camera(c);
        write_step_outputs(p, env, *c.h);  // Game::observe's scalar stores, game.cpp:160-164
    }
}
#endif

// the setup + render kernels' phases as plain loops (host debug harness; also documents the phase order)
template <class G, int VIEW, class Frame>
void render_env_serial(const KParams &p, int env, Frame &f) {
    using Setup = typename FrameFor<G, VIEW>::setup;
    using Shared = typename FrameFor<G, VIEW>::shared;
    Setup &s = *reinterpret_cast<Setup *>(p.frame_setup + (size_t)env * p.frame_setup_stride);
    env_setup_frame<G, Setup>(p, env, s, 0, 1);
    static_cast<Shared &>(f) = static_cast<const Shared &>(s);
    env_stage_tiles_serial<Frame>(p, f);
    for (int w = 0; w < 4; w++) env_render_compose<G, Frame>(p, f, w, 4, 0, 1);  // the device's row ownership, one lane per owner
    uint32_t *out = reinterpret_cast<uint32_t *>(p.rgb + (size_t)env * (RES_W * RES_H * 3));
    for (int g = 0; g < RES_W * RES_H / 4; g++) Raster<G, Frame>::pack_quad(f.fb + 4 * g, out + 3 * g);
}

// Which path of the gather each pixel of env's last frame takes (PixelClass), bit 7 set where an entity or
// overlay blit's box covers it. Host debug build only, where the frame record is host memory; the
// census of tools/render_pixel_classes.py.
enum PixelClass : uint8_t { PC_TILE_OPAQUE = 0, PC_TILE_UNDER = 1, PC_STRIP = 2, PC_GEN_SOLID = 3, PC_GEN_OTHER = 4, PC_NO_CELL = 5, PC_PAINTED = 0x80 };
template <class G, int VIEW>
int frame_pixel_classes(const KParams &p, int env, uint8_t *out) {
#ifdef PG_HOSTSIM
    using Setup = typename FrameFor<G, VIEW>::setup;
    const Setup &f = *reinterpret_cast<const Setup *>(p.frame_setup + (size_t)env * p.frame_setup_stride);
    const int nj = f.n_tjobs < MAX_TILE_JOBS ? f.n_tjobs : MAX_TILE_JOBS;
    for (int py = 0; py < RES_H; py++)
        for (int px = 0; px < RES_W; px++) {
            uint8_t cls = PC_NO_CELL;
            const uint32_t ci = G::DRAWS_GRID ? f.colinfo[px] : 0u, ri = G::DRAWS_GRID ? f.rowinfo[py] : 0u;
            if ((ci & ri & CI_VALID) && !(ci & ri & CI_FAST)) {
                cls = PC_STRIP;
            } else if (ci & ri & CI_FAST) {
                const uint32_t code = f.cellmap[(ci & CI_BASE_MASK) + (ri & CI_BASE_MASK)];
                if (code & CELL_GENERAL) {
                    cls = f.gen_blit((int)(code & 0x7fffu))->kind == BLIT_SOLID ? PC_GEN_SOLID : PC_GEN_OTHER;
                } else {
                    uint32_t texel = 0;
                    if (code) {  // arena word -> the table word its staging job copies there
                        const uint32_t a = code - 1 + ((ri >> CI_D_SHIFT) & 31u) * ((ci >> CI_TW_SHIFT) & 31u) + ((ci >> CI_D_SHIFT) & 31u);
                        for (int j = 0; j < nj; j++)
                            if (a >= f.tjob[j].dst && a < (uint32_t)f.tjob[j].dst + f.tjob[j].words)
                                texel = p.tiles.texels[f.tjob[j].src + a - f.tjob[j].dst];
                    }
                    cls = texel >= 0xff000000u ? PC_TILE_OPAQUE : PC_TILE_UNDER;
                }
            }
            for (int i = 0; i < f.n_ent + f.n_overlay; i++) {
                const Blit &b = f.ents[i];
                if ((uint32_t)(px - b.x1) < b.w && (uint32_t)(py - b.y1) < b.h)
                    cls |= PC_PAINTED;
            }
            out[py * RES_W + px] = cls;
        }
    return 0;
#else
    (void)p; (void)env; (void)out;
    return -1;
#endif
}

struct LaunchCtx {
#ifndef PG_HOSTSIM
    cudaStream_t stream;
    cudaStream_t logic_stream;  // null, or a higher-priority stream the logic kernel goes to (then `link` orders render behind it)
    cudaEvent_t link;
    unsigned int *ticket;     // work counter of this launch slot (one per in-flight logic kernel)
    int max_logic_blocks;     // SM count x resident CTAs per SM
    int render_smem_floor;    // dynamic shared memory requested per render CTA is at least this (co-residency knob)
    cudaEvent_t *tev;         // optional: 4 events (before logic, after it, after setup, after render) for kernel timing
#endif
    int64_t *launch_counter;
};

#ifndef PG_HOSTSIM
// Dynamic shared memory of one render CTA (frame, or the co-residency floor) with the kernel's
// opt-in limit raised to it once.
template <class G, int VIEW>
int prepare_render_smem(const LaunchCtx &lc) {
    using Frame = typename FrameFor<G, VIEW>::type;
    const int bytes = (int)sizeof(Frame) > lc.render_smem_floor ? (int)sizeof(Frame) : lc.render_smem_floor;
    // the attribute is per device: remember what each device of this process was given
    static int attr_set[64] = {};
    int dev = 0;
    CUDA_CHECK(cudaGetDevice(&dev));
    int &have = attr_set[dev & 63];
    if (have < bytes) {
        CUDA_CHECK(cudaFuncSetAttribute(render_kernel<G, VIEW>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
        have = bytes;
    }
    return bytes;
}
#endif

template <class G, bool INIT, int VIEW>
void launch_env_kernel(const KParams &p, const LaunchCtx &lc) {
    using Frame = typename FrameFor<G, VIEW>::type;
    if (p.env_count <= 0)
        return;
#ifndef PG_HOSTSIM
    // Shared memory per render CTA: the frame, or more when the handle asks for fewer resident
    // render CTAs per SM. At 8 CTAs x 128 threads x 64 registers the render kernel owns the whole
    // register file of an SM and no logic-kernel block of another env chunk can run beside it;
    // capping its residency trades a little render speed for real overlap of the two kernels.
    const int render_smem = prepare_render_smem<G, VIEW>(lc);
    int logic_blocks = (p.env_count + kLogicEnvsPerBlock - 1) / kLogicEnvsPerBlock;
    if (logic_blocks > lc.max_logic_blocks)
        logic_blocks = lc.max_logic_blocks;
    cudaStream_t ls = lc.logic_stream ? lc.logic_stream : lc.stream;
    CUDA_CHECK(cudaMemsetAsync(lc.ticket, 0, sizeof(unsigned int), ls));
    if (lc.tev)
        CUDA_CHECK(cudaEventRecord(lc.tev[0], ls));
    logic_kernel<G, INIT><<<logic_blocks, kLogicThreads, 0, ls>>>(p, lc.ticket);
    if (lc.logic_stream) {
        CUDA_CHECK(cudaEventRecord(lc.link, ls));
        CUDA_CHECK(cudaStreamWaitEvent(lc.stream, lc.link, 0));
    }
    if (lc.tev)
        CUDA_CHECK(cudaEventRecord(lc.tev[1], lc.stream));
    setup_kernel<G, VIEW><<<(p.env_count + kSetupThreads / 32 - 1) / (kSetupThreads / 32), kSetupThreads, 0, lc.stream>>>(p);
    if (lc.tev)
        CUDA_CHECK(cudaEventRecord(lc.tev[2], lc.stream));
    render_kernel<G, VIEW><<<p.env_count, kRenderThreads, render_smem, lc.stream>>>(p);
    if (lc.tev)
        CUDA_CHECK(cudaEventRecord(lc.tev[3], lc.stream));
    CUDA_CHECK(cudaGetLastError());
    (*lc.launch_counter) += 3;
#else
    static thread_local Frame *f = new Frame;
    for (int b = 0; b < p.env_count; b++) {
        int env = p.env_first + b * p.env_step;
        if (INIT)
            env_init_logic<G, Frame>(p, env);
        else
            env_step_logic<G, Frame>(p, env);
        render_env_serial<G, VIEW, Frame>(p, env, *f);
    }
    (*lc.launch_counter) += 3;
#endif
}

template <class G, int VIEW>
void launch_observe_only(const KParams &p, const LaunchCtx &lc) {
    using Frame = typename FrameFor<G, VIEW>::type;
    if (p.env_count <= 0)
        return;
#ifndef PG_HOSTSIM
    const int render_smem = prepare_render_smem<G, VIEW>(lc);
    camera_kernel<G><<<p.env_count, 32, 0, lc.stream>>>(p);
    setup_kernel<G, VIEW><<<(p.env_count + kSetupThreads / 32 - 1) / (kSetupThreads / 32), kSetupThreads, 0, lc.stream>>>(p);
    render_kernel<G, VIEW><<<p.env_count, kRenderThreads, render_smem, lc.stream>>>(p);
    CUDA_CHECK(cudaGetLastError());
#else
    static thread_local Frame *f = new Frame;
    for (int b = 0; b < p.env_count; b++) {
        int env = p.env_first + b * p.env_step;
        Ctx c = make_ctx(p, env);
        Raster<G, Frame>::prepare_camera(c);
        write_step_outputs(p, env, *c.h);
        render_env_serial<G, VIEW, Frame>(p, env, *f);
    }
#endif
    (*lc.launch_counter) += 2;
}

struct GameVTable {
    const char *name;
    int id;
    int ent_cap, grid_cap, scratch_words;
    int rot_records;  // rotated-sprite / span records per env (global)
    int blit_records; // blit list capacity per env (global)
    // [0] = the game's usual view, [1] = the whole-world view of center_agent = false (step[1] null: the game has none)
    int setup_bytes[2];   // sizeof(FrameSetupT)
    int cell_records[2];  // cells of the largest visible window (capacity for general cell blits)
    int frame_bytes[2];   // shared memory of one render CTA
    int render_ctas_per_sm[2];  // residency the render kernel is compiled for
    void (*init[2])(const KParams &, const LaunchCtx &);
    void (*step[2])(const KParams &, const LaunchCtx &);
    void (*observe_only[2])(const KParams &, const LaunchCtx &);
    int (*pixel_classes[2])(const KParams &, int, uint8_t *);
};

template <class G, int VIEW>
void fill_view(GameVTable &vt, int slot) {
    using F = FrameFor<G, VIEW>;
    vt.setup_bytes[slot] = (int)sizeof(typename F::setup);
    vt.cell_records[slot] = F::type::kMaxCells1D * F::type::kMaxCells1D;
    vt.frame_bytes[slot] = (int)sizeof(typename F::type);
#ifndef PG_HOSTSIM
    vt.render_ctas_per_sm[slot] = RenderTune<G, VIEW>::kMinBlocks;
#else
    vt.render_ctas_per_sm[slot] = 0;
#endif
    vt.init[slot] = &launch_env_kernel<G, true, VIEW>;
    vt.step[slot] = &launch_env_kernel<G, false, VIEW>;
    vt.observe_only[slot] = &launch_observe_only<G, VIEW>;
    vt.pixel_classes[slot] = &frame_pixel_classes<G, VIEW>;
}

template <class G>
GameVTable make_vtable(int id) {
    GameVTable vt{};
    vt.name = G::NAME;
    vt.id = id;
    vt.ent_cap = G::ENT_CAP;
    vt.grid_cap = G::GRID_CAP;
    vt.scratch_words = G::SCRATCH_WORDS;
    vt.rot_records = FrameFor<G>::type::kMaxRot;
    vt.blit_records = FrameFor<G>::type::kMaxList;
    fill_view<G, G::MAX_VIEW_CELLS>(vt, 0);
    if constexpr (G::FULL_VIEW_CELLS > G::MAX_VIEW_CELLS)
        fill_view<G, G::FULL_VIEW_CELLS>(vt, 1);
    return vt;
}

}  // namespace pg
