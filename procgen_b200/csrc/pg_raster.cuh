// Software rasteriser: 64x64 RGB observation of one env, composited per pixel (gather) from an
// ordered list of "blits" that restate what the reference asks Qt's raster engine to draw
// (game.cpp:77-91 -> basic-abstract-game.cpp:799-1066).  No framebuffer read-modify-write: every
// output pixel walks the (short, culled) list of blits that can touch it, in draw order, blends in
// registers and is written once as packed RGB.
//
// Raster rules (Qt raster engine, non-antialiased, restated; see oracle/shim/qt_raster.cpp for
// the CPU twin and DESIGN.md for how they are pinned against real Qt 6.6.3):
//   F fillRect -> [qRound(x), qRound(x+w)) x [qRound(y), qRound(y+h)), qRound = half away from zero
//   S scaled drawImage -> nearest neighbour, 16.16 fixed point, target snapped to ints (switch)
//   B src-over with BYTE_MUL; O opacity int(o*256) -> (io*255)>>8
//   R rotated drawImage -> per-row spans from Qt's scan converter + 16.16 texel stepping (two paths)
//   E / L drawEllipse (integer midpoint) and cosmetic drawLine, as per-row spans (jumper compass)
//
// Phases (render kernel: one CTA per env; `tid`/`nthreads` are explicit so the same code runs in
// the host debug harness with nthreads = 1; a barrier separates consecutive phases):
//   prepare_camera   logic thread  prepare_for_drawing -> env header (runs in the logic kernel)
//   frame_begin      all threads   thread 0: window + background/overlay blits; threads i<nx / j<ny:
//                                  geometry + pixel span of grid column i / row j
//   frame_build      all threads   entities -> blits, one entity per thread and round, culled and
//                                  compacted in draw order with a block-wide prefix sum (few
//                                  entities: warp 0 alone while the other warps build one blit per
//                                  visible grid cell and the pixel-column/row -> cell lookups; fp64
//                                  math happens here, once per sprite instead of once per pixel)
//   frame_tiles      all threads   tiles of tiled entities whose slots frame_build reserved
//   frame_rots       all threads   (games with DEFER_ROTATED) rotated sprites whose slots were reserved
//   frame_tile_alloc / frame_cells_finish   pre-scaled tiles the cells need -> arena + staging jobs
//   compose_rows     row owners    gather (cells over background) then paint (entity blits in order)
#pragma once
#include "pg_engine.cuh"

namespace pg {

enum BlitKind : uint8_t { BLIT_NONE = 0, BLIT_IMAGE = 1, BLIT_SOLID = 2, BLIT_ROTATED = 3, BLIT_SPANS = 4,
                          BLIT_ROT_PENDING = 5 /* slot reserved while the list is built; resolved by frame_rots */ };

struct Blit {
    uint8_t x1, y1, w, h;    // device pixels [x1,x1+w) x [y1,y1+h) after clip + Qt's edge guards;
                             // w == 0 <=> nothing to draw (first word = one 32-bit load in the shader)
    uint8_t kind;
    uint8_t mirror;
    uint16_t opacity;        // Qt intOpacity, 256 = opaque path
    int32_t ix, iy;          // 16.16 source step per device pixel
    uint32_t basex, srcy;    // 16.16 source coordinate at (x1, y1)
    uint32_t src;            // IMAGE: texel offset of the sprite in the atlas; SOLID: 0xFFRRGGBB
    uint16_t sw, sh;
};
static_assert(sizeof(Blit) == 32, "Blit is 32 B");

// Extra record of a rotated sprite (Blit.kind == BLIT_ROTATED, Blit.ix = index): per device row the
// covered span, plus the texel map of whichever of Qt's two transformed-image paths applies.
struct RotBlit {
    uint8_t x1[RES_H], x2[RES_H];  // row y covers [x1[y], x2[y]); x2 <= x1: nothing
    int32_t absolute;               // 1: qt_transform_image (u = px*dudx + py*dudy + u0); 0: fetchTransformed
    int32_t dudx, dvdx, dudy, dvdy, u0, v0;  // absolute map; span-relative uses dudx,dvdx as fdx,fdy
    int32_t pad;
    double m11, m12, m21, m22, dx, dy;       // inverse matrix for the span-start texel (fetchTransformed)
};

constexpr int MAX_BG_BLITS = 8;
constexpr int MAX_OVERLAY_BLITS = 8;

// camera of one frame = what prepare_for_drawing leaves in the env header
struct Camera {
    float unit, view_dim, x_off, y_off;
};

// ---- pre-scaled cell tiles (global table, built once per VecEnv by tile_table_fill)
// With Qt's integer snapping an un-clipped, un-rotated, un-mirrored drawImage of integer target
// size (tw, th) samples the same tw x th texels of its sprite wherever it lands (make_image_blit:
// the 16.16 start `ceil(0.5 * sx * 65536) - 1` and the step do not depend on the position). Grid
// cells are exactly that, hundreds per frame, in one or two sizes: so every sprite is resampled
// once for every target size up to MAX_TILE_DIM^2 — by make_image_blit itself, so the texels are
// the ones the general path would fetch — and a frame stages the few tiles it needs in shared
// memory with bulk async copies (cp.async.bulk + mbarrier) while its entity blits are built.
constexpr int MAX_TILE_DIM = 12;
constexpr int TILE_VARIANTS = MAX_TILE_DIM * MAX_TILE_DIM;
struct TileTable {
    const uint32_t *texels;   // tile (slot, tw, th): tw*th texels, row stride tw, padded to a multiple of 4 texels
    const uint32_t *index;    // [slot][tw-1][th-1] -> texel offset of the tile (multiple of 4)
    const SpriteDesc *sprites;  // [slot]
    int32_t n_slots;
};
PG_HD int tile_words(int tw, int th) { return (tw * th + 3) & ~3; }

constexpr int CELL_KEY_TYPES = 64;               // grid object ids that can use a tile (others take the general path)
constexpr int CELL_KEYS = CELL_KEY_TYPES * 4;    // x (tw - W0, th - H0) in {0,1}^2
constexpr uint16_t CELL_GENERAL = 0x8000u;       // cellmap code: 0 none | 1 + texel offset of its tile in the arena | CELL_GENERAL | blit index
constexpr int MAX_TILE_JOBS = 64;
constexpr uint32_t BG_NONE = 0xffffffffu;

// colinfo / rowinfo word of a pixel column / row (cells of the visible grid window)
constexpr uint32_t CI_BASE_MASK = 0xfffu;        // column: ci * ny (< 64 * 64); row: cj
constexpr uint32_t CI_VALID = 1u << 12;          // some cell column / row covers the pixel
constexpr int CI_D_SHIFT = 13;                   // 5 bits: px - col_p1 (py - row_p1)
constexpr int CI_TW_SHIFT = 18;                  // 5 bits, column only: row stride of its tiles (0: not tile-eligible)
constexpr uint32_t CI_MULTI = 1u << 23;          // more than one cell column / row covers the pixel
constexpr uint32_t CI_FAST = 1u << 24;           // exactly one does
constexpr uint32_t CI_WIDE = 1u << 25;           // more than two do (colinfo_lo / rowinfo_lo do not describe them all)

// one pre-scaled tile to stage: texel offset in the table, arena word offset, words (one 8-byte load)
struct alignas(8) TileJob {
    uint32_t src;
    uint16_t dst, words;
};

// One frame's working set, in three parts:
//   FrameSharedT  what the setup kernel (one warp per env) hands to the render kernel: camera, cell
//                 spans, background, blit counts, the classified cell map with its pixel -> cell
//                 lookups, and the list of pre-scaled tiles to stage — everything that is O(entities
//                 + cells) and heavy on fp64 or control flow. Lives in global memory; the render
//                 CTA stages it into its shared memory with one bulk copy.
//   FrameSetupT   + the setup kernel's own scratch (global, per env)
//   FrameT        + the render kernel's scratch (shared memory): frame buffer, tile arena
template <int MAX_CELLS_1D, int MAX_ENT_BLITS, int MAX_ROT_BLITS>
struct alignas(16) FrameSharedT {
    static constexpr int kMaxCells1D = MAX_CELLS_1D;
    static constexpr int kMaxRot = MAX_ROT_BLITS > 0 ? MAX_ROT_BLITS : 1;
    // `ents` = VISIBLE entity blits (after culling) in draw order, then the overlay blits (drawn last)
    static constexpr int kMaxEntBlits = MAX_ENT_BLITS;
    static constexpr int kMaxList = MAX_ENT_BLITS + MAX_OVERLAY_BLITS;
    // shared-memory words the render CTA keeps for staged tiles; tiles that do not fit turn their cells into general blits
    static constexpr int kArenaWords = MAX_CELLS_1D > 1 ? (MAX_CELLS_1D * MAX_CELLS_1D * 8 < 1280 ? MAX_CELLS_1D * MAX_CELLS_1D * 8 : 1280) : 4;
    Camera cam;
    int32_t low_x, low_y, nx, ny;   // visible grid window: cells [low_x, low_x+nx) x [low_y, low_y+ny)
    int32_t n_bg, n_ent, n_ent_below, n_overlay;  // n_ent_below = entities with render_z == -1
    int32_t snap;
    int32_t pad;                    // 1: the background is one opaque un-mirrored image (it may cover only part of the device)
    int32_t tile_w0, tile_h0;       // smaller of the two snapped cell sizes of this frame
    int32_t n_rot;
    int32_t n_gen;                  // general cell blits in use (gen_spill)
    int32_t tile_top;               // arena words used by tiles
    int32_t n_tjobs;
    RotBlit *rot;                   // this env's rotated-sprite / span records (global)
    Blit *ents;                     // this env's blit list (global): the painter reads it sequentially
    Blit *gen_spill;                // this env's general cell blits (global): solid-colour cells, clipped walks that differ, un-snapped targets
    int32_t spare[2];
    // geometry shared by all cells of a column / row (the cell rect is separable)
    double cell_w;                  // QRectF.width == height
    double spare_d;
    double col_x[MAX_CELLS_1D];     // QRectF.x of column i
    double row_y[MAX_CELLS_1D];     // QRectF.y of row j
    // device pixel span [p1,p2) of column i; padded to whole words with 255 (cell_lookup compares 4 at a time)
    static constexpr int kSpanBytes = (MAX_CELLS_1D + 3) & ~3;
    alignas(4) uint8_t col_p1[kSpanBytes];
    alignas(4) uint8_t col_p2[kSpanBytes];
    alignas(4) uint8_t row_p1[kSpanBytes];
    alignas(4) uint8_t row_p2[kSpanBytes];
    uint8_t col_tw[MAX_CELLS_1D], row_th[MAX_CELLS_1D];  // snapped size if the column / row can use tiles, else 0
    uint8_t col_k0[MAX_CELLS_1D], row_k0[MAX_CELLS_1D];  // pixels the device edge cuts off the near side (tile offset of the first visible one)
    uint8_t col_lo[RES_W], col_hi[RES_W];   // window-relative cell columns covering pixel column
    uint8_t row_lo[RES_H], row_hi[RES_H];
    alignas(16) uint32_t colinfo[RES_W];      // CI_* words of the cell column (row) covering the pixel; the later one in
    alignas(16) uint32_t rowinfo[RES_H];      // draw order where two overlap (CI_MULTI)
    alignas(16) uint32_t colinfo_lo[RES_W];   // CI_MULTI: the same for the earlier of the two (else = colinfo / rowinfo)
    alignas(16) uint32_t rowinfo_lo[RES_H];
    alignas(16) uint32_t bgcol[RES_W];        // pad == 1: source column of the background image sampled by pixel column px, BG_NONE outside it
    uint32_t bgrow[RES_H];                    // pad == 1: atlas offset of the background row sampled by pixel row py, BG_NONE outside the image
    TileJob tjob[MAX_TILE_JOBS];              // tile copies to stage
    uint16_t cellmap[MAX_CELLS_1D * MAX_CELLS_1D];  // [ci * ny + cj], x outer / y inner = draw order
    alignas(16) Blit bg[MAX_BG_BLITS];

    PG_HD Blit *gen_blit(int k) { return gen_spill + k; }
    PG_HD const Blit *gen_blit(int k) const { return gen_spill + k; }
};

template <int MAX_CELLS_1D, int MAX_ENT_BLITS, int MAX_ROT_BLITS>
struct alignas(16) FrameSetupT : FrameSharedT<MAX_CELLS_1D, MAX_ENT_BLITS, MAX_ROT_BLITS> {
    using Shared = FrameSharedT<MAX_CELLS_1D, MAX_ENT_BLITS, MAX_ROT_BLITS>;
    // tiled entities only reserve their blit slots while the list is built; the tiles themselves
    // are filled in by all lanes afterwards (frame_tiles)
    static constexpr int kMaxTileJobs = 64;
    int32_t n_jobs;
    int32_t job_ei[kMaxTileJobs], job_pos[kMaxTileJobs], job_n[kMaxTileJobs], job_j0[kMaxTileJobs];
    Blit overlay[MAX_OVERLAY_BLITS];
    alignas(4) uint16_t tilekey[MAX_CELLS_1D > 1 ? CELL_KEYS : 4];  // per (type, size variant): 0 unused | 1 wanted | 2 + arena texel offset | 0xffff unavailable
};

template <int MAX_CELLS_1D, int MAX_ENT_BLITS, int MAX_ROT_BLITS>
struct alignas(16) FrameT : FrameSharedT<MAX_CELLS_1D, MAX_ENT_BLITS, MAX_ROT_BLITS> {
    using Shared = FrameSharedT<MAX_CELLS_1D, MAX_ENT_BLITS, MAX_ROT_BLITS>;
    // the frame as 0xFFRRGGBB pixels while it is composed; packed to RGB888 in place (its first
    // 12 KiB) and written out with one bulk store
    alignas(16) uint32_t fb[RES_W * RES_H];
    alignas(16) uint32_t arena[Shared::kArenaWords];   // staged tiles (texels)
    alignas(8) unsigned long long mbar;                // staging barrier (shared part + tiles)
};

// ---- rule S: un-rotated scaled image (qt_scale_image_32bit)
PG_HD void blit_clear(Blit &b) {
    b.x1 = b.y1 = b.w = b.h = 0;
    b.kind = BLIT_NONE;
}

#ifndef PG_SETUP_INLINE_BLIT
#define PG_SETUP_INLINE_BLIT 1   // the setup kernel's per-entity blit: inlined (1) or through the out-of-line builders (0)
#endif
PG_HD void make_image_blit_inl(Blit &b, double tx, double ty, double tw, double th, SpriteDesc sd, bool mirror, int int_opacity, bool snap);
PG_HD_FREE_NOINLINE void make_image_blit(Blit &b, double tx, double ty, double tw, double th, SpriteDesc sd, bool mirror, int int_opacity, bool snap) {
    make_image_blit_inl(b, tx, ty, tw, th, sd, mirror, int_opacity, snap);
}
PG_HD void make_image_blit_inl(Blit &b, double tx, double ty, double tw, double th, SpriteDesc sd, bool mirror, int int_opacity, bool snap) {
    blit_clear(b);
    const int sw = sd.w, sh = sd.h;
    if (sw <= 0 || sh <= 0)
        return;
    if (snap) {
        double x = pg_qround(tx);
        double y = pg_qround(ty);
        double w = pg_qround(tx + tw - x);
        double h = pg_qround(ty + th - y);
        tx = x;
        ty = y;
        tw = w;
        th = h;
    }
    if (tw == 0 || th == 0 || tw != tw || th != th)
        return;
    // Qt 6.6.3 qt_scale_image_32bit: step and start both come from the source/target ratio in double.
    // Negative sizes (a mirroring scale, e.g. rotate(180)) step backwards from the far source edge.
    const double sx = (double)sw / tw;
    const double sy = (double)sh / th;
    const int ix = (int)(65536.0 * sx);
    const int iy = (int)(65536.0 * sy);
    double nx = tx, ny = ty, nw = tw, nh = th;  // targetRect.normalized()
    if (nw < 0) { nx += nw; nw = -nw; }
    if (nh < 0) { ny += nh; nh = -nh; }
    int tx1 = pg_qround(nx), ty1 = pg_qround(ny);
    int tx2 = pg_qround(nx + nw), ty2 = pg_qround(ny + nh);
    if (tx1 < 0) tx1 = 0;
    if (ty1 < 0) ty1 = 0;
    if (tx2 > RES_W) tx2 = RES_W;
    if (ty2 > RES_H) ty2 = RES_H;
    if (tx2 <= tx1 || ty2 <= ty1)
        return;
    int h = ty2 - ty1;
    int w = tx2 - tx1;
    int dstx, dsty;
    if (sx < 0)
        dstx = (int)pg_dfloor((tx1 + 0.5 - (tx + tw)) * sx * 65536) + 1 + sw * 65536;
    else
        dstx = (int)pg_dceil((tx1 + 0.5 - tx) * sx * 65536) - 1;
    if (sy < 0)
        dsty = (int)pg_dfloor((ty1 + 0.5 - (ty + th)) * sy * 65536) + 1 + sh * 65536;
    else
        dsty = (int)pg_dceil((ty1 + 0.5 - ty) * sy * 65536) - 1;
    uint32_t basex = (uint32_t)dstx;
    uint32_t srcy = (uint32_t)dsty;
    if ((int)(srcy >> 16) >= sh && iy < 0) {
        srcy += (uint32_t)iy;
        --h;
    }
    if ((int)(basex >> 16) >= sw && ix < 0) {
        basex += (uint32_t)ix;
        --w;
    }
    if (w <= 0 || h <= 0)
        return;
    int yend = ((int)(srcy + (uint32_t)iy * (uint32_t)(h - 1))) >> 16;
    if (yend < 0 || yend >= sh)
        --h;
    int xend = ((int)(basex + (uint32_t)ix * (uint32_t)(w - 1))) >> 16;
    if (xend < 0 || xend >= sw)
        --w;
    if (w <= 0 || h <= 0)
        return;
    b.x1 = (uint8_t)tx1;
    b.y1 = (uint8_t)ty1;
    b.w = (uint8_t)w;
    b.h = (uint8_t)h;
    b.kind = BLIT_IMAGE;
    b.mirror = mirror ? 1 : 0;
    b.opacity = (uint16_t)int_opacity;
    b.ix = ix;
    b.iy = iy;
    b.basex = basex;
    b.srcy = srcy;
    b.src = sd.off;
    b.sw = (uint16_t)sw;
    b.sh = (uint16_t)sh;
}


// ================================================================= rotated sprites
// Device twin of oracle/shim/qt_raster.cpp's transformed-image restatement (see there for the Qt
// provenance of every rule): per-row spans + a texel map, built once per rotated sprite.
struct RotXform {
    double m11, m12, m21, m22, dx, dy;  // Qt convention: x' = m11*x + m21*y + dx ; y' = m12*x + m22*y + dy
};

PG_HD void rot_span(RotBlit &rb, int x, int len, int y) {
    if (y < (rb.pad & 0xff) || y >= ((rb.pad >> 8) & 0xff))  // outside the cleared row window (and the device)
        return;
    if (x < 0) {
        len += x;
        x = 0;
    }
    if (x + len > RES_W)
        len = RES_W - x;
    if (len <= 0)
        return;
    if (rb.x2[y] <= rb.x1[y]) {
        rb.x1[y] = (uint8_t)x;
        rb.x2[y] = (uint8_t)(x + len);
    } else {  // a second span on a row of a convex quad: keep the union
        if (x < rb.x1[y]) rb.x1[y] = (uint8_t)x;
        if (x + len > rb.x2[y]) rb.x2[y] = (uint8_t)(x + len);
    }
}

// QScanConverter on a quad: vertices shifted by -0.5, truncated to 26.6, edges stepped in 16.16
PG_HD void rot_scan_convert_quad(RotBlit &rb, const double *vx, const double *vy) {
    long long X[4], Y[4];
    for (int i = 0; i < 4; i++) {
        X[i] = (long long)((vx[i] - 0.5) * 64);
        Y[i] = (long long)((vy[i] - 0.5) * 64);
    }
    int lx[4], ldelta[4], ltop[4], lbottom[4], lwind[4];
    int n = 0;
    for (int i = 0; i < 4; i++) {
        long long ax = X[i], ay = Y[i], bx = X[(i + 1) & 3], by = Y[(i + 1) & 3];
        if (ax == bx && ay == by)
            continue;
        int winding = 1;
        if (ay > by) {
            long long t = ax; ax = bx; bx = t;
            t = ay; ay = by; by = t;
            winding = -1;
        }
        ax += 32; ay += 32; bx += 32; by += 32;
        int iTop = (int)((ay + 32 - 1) >> 6);
        if (iTop < 0) iTop = 0;
        int iBottom = (int)((by - 32 - 1) >> 6);
        if (iBottom > RES_H - 1) iBottom = RES_H - 1;
        if (iTop <= iBottom) {
            int aFP = 0x8000 + (int)(ax * 1024) - 1;
            if (bx == ax) {
                lx[n] = aFP; ldelta[n] = 0;
            } else {
                const double slope = (double)(bx - ax) / (double)(by - ay);
                const int slopeFP = (int)(slope * 65536.);
                const long long dy = (long long)(iTop << 16) + 0x8000 - ay * 1024;
                lx[n] = aFP + (int)(((long long)slopeFP * dy) >> 16);
                ldelta[n] = slopeFP;
            }
            ltop[n] = iTop; lbottom[n] = iBottom; lwind[n] = winding;
            n++;
        }
    }
    if (n == 0)
        return;
    // stable sort by top (n <= 4)
    int order[4];
    for (int i = 0; i < n; i++) order[i] = i;
    for (int i = 1; i < n; i++) {
        int t = order[i], j = i;
        while (j > 0 && ltop[order[j - 1]] > ltop[t]) {
            order[j] = order[j - 1];
            --j;
        }
        order[j] = t;
    }
    int active[4];
    int na = 0, li = 0;
    for (int y = ltop[order[0]]; y < RES_H; ++y) {
        for (; li < n && ltop[order[li]] == y; ++li) active[na++] = order[li];
        if (na == 0 && li >= n)
            break;
        for (int i = 1; i < na; ++i) {
            int t = active[i], j = i;
            while (j > 0 && lx[active[j - 1]] > lx[t]) {
                active[j] = active[j - 1];
                --j;
            }
            active[j] = t;
        }
        int x = 0, winding = 0, keep = 0;
        int nexta[4];
        for (int i = 0; i < na; ++i) {
            const int node = active[i];
            const int current = lx[node] >> 16;
            if (winding & 1) {
                int x0 = x < 0 ? 0 : x, x1 = current > RES_W ? RES_W : current;
                if (x1 > x0)
                    rot_span(rb, x0, x1 - x0, y);
            }
            x = current;
            winding += lwind[node];
            if (lbottom[node] != y) {
                lx[node] += ldelta[node];
                nexta[keep++] = node;
            }
        }
        for (int i = 0; i < keep; i++) active[i] = nexta[i];
        na = keep;
    }
}

PG_HD bool rot_q26Dot6Compare(double p1, double p2) { return (int)((p2 - p1) * 64.) == 0; }
PG_HD double rot_bound(double lo, double v, double hi) { return v < lo ? lo : (v > hi ? hi : v); }

// QRasterizer::rasterizeLine(a, b, width), non-antialiased, clip = the 64x64 device
PG_HD void rot_rasterize_line(RotBlit &rb, double ax, double ay, double bx, double by, double width) {
    const int clipL = 0, clipT = 0, clipR = RES_W - 1, clipB = RES_H - 1;
    if ((ax == bx && ay == by) || width == 0)
        return;
    double pax = ax, pay = ay, pbx = bx, pby = by;
    {
        const double offx = pg_dfabs(by - ay) * width * 0.5, offy = pg_dfabs(bx - ax) * width * 0.5;
        const double cl = clipL - offx, ct = clipT - offy, cr = (clipR + 1) + offx, cb = (clipB + 1) + offy;
        const bool a_in = !(pax < cl || pax > cr || pay < ct || pay > cb);
        const bool b_in = !(pbx < cl || pbx > cr || pby < ct || pby > cb);
        if (!a_in || !b_in) {
            double t1 = 0, t2 = 1;
            const double o[2] = {pax, pay};
            const double dd[2] = {pbx - pax, pby - pay};
            const double low[2] = {cl, ct};
            const double high[2] = {cr, cb};
            for (int i = 0; i < 2; ++i) {
                if (dd[i] == 0) {
                    if (o[i] <= low[i] || o[i] >= high[i])
                        return;
                    continue;
                }
                const double d_inv = 1 / dd[i];
                double t_low = (low[i] - o[i]) * d_inv;
                double t_high = (high[i] - o[i]) * d_inv;
                if (t_low > t_high) {
                    double t = t_low; t_low = t_high; t_high = t;
                }
                if (t1 < t_low) t1 = t_low;
                if (t2 > t_high) t2 = t_high;
                if (t1 >= t2)
                    return;
            }
            const double npax = pax + (pbx - pax) * t1, npay = pay + (pby - pay) * t1;
            const double npbx = pax + (pbx - pax) * t2, npby = pay + (pby - pay) * t2;
            pax = npax; pay = npay; pbx = npbx; pby = npby;
        }
        const double d0x = ax - bx, d0y = ay - by;
        const double w0 = d0x * d0x + d0y * d0y;
        const double d1x = pax - pbx, d1y = pay - pby;
        const double w = d1x * d1x + d1y * d1y;
        if (w == 0)
            return;
        width *= pg_dsqrt(w0 / w);
    }
    if (rot_q26Dot6Compare(pay, pby)) {
        const double x = (pax + pbx) * 0.5f;
        const double dx = pg_dfabs(pbx - pax) * 0.5f;
        const double y = pay;
        const double dy = width * dx;
        pax = x; pay = y - dy;
        pbx = x; pby = y + dy;
        width = 1 / width;
    }
    if (rot_q26Dot6Compare(pax, pbx)) {
        if (pay > pby) {
            double t = pax; pax = pbx; pbx = t;
            t = pay; pay = pby; pby = t;
        }
        const double dy = pby - pay;
        const double halfWidth = 0.5f * width * dy;
        double left = pax - halfWidth;
        double right = pax + halfWidth;
        left = rot_bound((double)clipL, left, (double)(clipR + 1));
        right = rot_bound((double)clipL, right, (double)(clipR + 1));
        pay = rot_bound((double)clipT, pay, (double)(clipB + 1));
        pby = rot_bound((double)clipT, pby, (double)(clipB + 1));
        if (rot_q26Dot6Compare(left, right) || rot_q26Dot6Compare(pay, pby))
            return;
        int iTop = (int)(pay + 0.5f);
        int iBottom = pby < 0.5f ? -1 : (int)(pby - 0.5f);
        int iLeft = (int)(left + 0.5f);
        int iRight = right < 0.5f ? -1 : (int)(right - 0.5f);
        int iWidth = iRight - iLeft + 1;
        for (int y = iTop; y <= iBottom; ++y) rot_span(rb, iLeft, iWidth, y);
        return;
    }
    if (pay > pby) {
        double t = pax; pax = pbx; pbx = t;
        t = pay; pay = pby; pby = t;
    }
    const double deltax = (pbx - pax) * (0.5f * width), deltay = (pby - pay) * (0.5f * width);
    const double perpx = deltay, perpy = -deltax;
    double vx[4], vy[4];  // top, right, bottom, left
    if (pax < pbx) {
        vx[0] = pax + perpx; vy[0] = pay + perpy;
        vx[3] = pax - perpx; vy[3] = pay - perpy;
        vx[1] = pbx + perpx; vy[1] = pby + perpy;
        vx[2] = pbx - perpx; vy[2] = pby - perpy;
    } else {
        vx[0] = pax - perpx; vy[0] = pay - perpy;
        vx[3] = pbx - perpx; vy[3] = pby - perpy;
        vx[1] = pax + perpx; vy[1] = pay + perpy;
        vx[2] = pbx + perpx; vy[2] = pby + perpy;
    }
    rot_scan_convert_quad(rb, vx, vy);
}

struct RotVertex {
    double x, y, u, v;
};

PG_HD void rot_transform_trapezoid(RotBlit &rb, const RotVertex &topLeft, const RotVertex &bottomLeft, const RotVertex &topRight,
                                   const RotVertex &bottomRight, double topY, double bottomY) {
    long long fromY = pg_qround(topY);
    if (fromY < 0) fromY = 0;
    long long toY = pg_qround(bottomY);
    if (toY > RES_H) toY = RES_H;
    if (fromY >= toY)
        return;
    const double leftSlope = (bottomLeft.x - topLeft.x) / (bottomLeft.y - topLeft.y);
    const double rightSlope = (bottomRight.x - topRight.x) / (bottomRight.y - topRight.y);
    const long long dx_l = (long long)(leftSlope * 0x10000);
    const long long dx_r = (long long)(rightSlope * 0x10000);
    long long x_l = (long long)((topLeft.x + (0.5 + fromY - topLeft.y) * leftSlope + 0.5) * 0x10000);
    long long x_r = (long long)((topRight.x + (0.5 + fromY - topRight.y) * rightSlope + 0.5) * 0x10000);
    for (long long y = fromY; y < toY; ++y) {
        long long fromX = x_l >> 16;
        if (fromX < 0) fromX = 0;
        long long toX = x_r >> 16;
        if (toX > RES_W) toX = RES_W;
        if (fromX < toX)
            rot_span(rb, (int)fromX, (int)(toX - fromX), (int)y);
        x_l += dx_l;
        x_r += dx_r;
    }
}

// qt_transform_image: three trapezoids + absolute 16.16 texel map
PG_HD void rot_transform_image(RotBlit &rb, int sw, int sh, const double *r, const RotXform &m) {
    RotVertex v[4];
    v[0].u = v[3].u = 0;
    v[0].v = v[1].v = 0;
    v[1].u = v[2].u = sw;
    v[3].v = v[2].v = sh;
    v[0].x = v[3].x = r[0];
    v[0].y = v[1].y = r[1];
    v[1].x = v[2].x = r[0] + r[2];
    v[3].y = v[2].y = r[1] + r[3];
    for (int i = 0; i < 4; i++) {
        double fx = v[i].x, fy = v[i].y;
        v[i].x = m.m11 * fx + m.m21 * fy + m.dx;
        v[i].y = m.m12 * fx + m.m22 * fy + m.dy;
    }
    int topmost = 0;
    for (int i = 1; i < 4; ++i)
        if (v[i].y < v[topmost].y)
            topmost = i;
    if (topmost == 1) {
        RotVertex t = v[0];
        v[0] = v[1]; v[1] = v[2]; v[2] = v[3]; v[3] = t;
    } else if (topmost == 2) {
        RotVertex t = v[0]; v[0] = v[2]; v[2] = t;
        t = v[1]; v[1] = v[3]; v[3] = t;
    } else if (topmost == 3) {
        RotVertex t = v[3];
        v[3] = v[2]; v[2] = v[1]; v[1] = v[0]; v[0] = t;
    }
    const double dx1 = v[1].x - v[0].x, dy1 = v[1].y - v[0].y;
    const double dx2 = v[3].x - v[0].x, dy2 = v[3].y - v[0].y;
    if (dx1 * dy2 - dx2 * dy1 > 0) {
        RotVertex t = v[1]; v[1] = v[3]; v[3] = t;
    }
    const RotVertex u = {v[1].x - v[0].x, v[1].y - v[0].y, v[1].u - v[0].u, v[1].v - v[0].v};
    const RotVertex w = {v[2].x - v[0].x, v[2].y - v[0].y, v[2].u - v[0].u, v[2].v - v[0].v};
    const double det = u.x * w.y - u.y * w.x;
    if (det == 0)
        return;
    const double invDet = 1.0 / det;
    const double m11 = (u.u * w.y - u.y * w.u) * invDet;
    const double m12 = (u.x * w.u - u.u * w.x) * invDet;
    const double m21 = (u.v * w.y - u.y * w.v) * invDet;
    const double m22 = (u.x * w.v - u.v * w.x) * invDet;
    const double mdx = v[0].u - m11 * v[0].x - m12 * v[0].y;
    const double mdy = v[0].v - m21 * v[0].x - m22 * v[0].y;
    rb.absolute = 1;
    rb.dudx = (int)(m11 * 0x10000);
    rb.dvdx = (int)(m21 * 0x10000);
    rb.dudy = (int)(m12 * 0x10000);
    rb.dvdy = (int)(m22 * 0x10000);
    rb.u0 = (int)pg_dceil((0.5 * m11 + 0.5 * m12 + mdx) * 0x10000) - 1;
    rb.v0 = (int)pg_dceil((0.5 * m21 + 0.5 * m22 + mdy) * 0x10000) - 1;
    if (v[1].y < v[3].y) {
        rot_transform_trapezoid(rb, v[0], v[1], v[0], v[3], v[0].y, v[1].y);
        rot_transform_trapezoid(rb, v[1], v[2], v[0], v[3], v[1].y, v[3].y);
        rot_transform_trapezoid(rb, v[1], v[2], v[3], v[2], v[3].y, v[2].y);
    } else {
        rot_transform_trapezoid(rb, v[0], v[1], v[0], v[3], v[0].y, v[3].y);
        rot_transform_trapezoid(rb, v[0], v[1], v[3], v[2], v[3].y, v[1].y);
        rot_transform_trapezoid(rb, v[1], v[2], v[3], v[2], v[1].y, v[2].y);
    }
}

// QRasterPaintEngine::drawImage under a rotating matrix: fills rb, returns false if nothing drawn
PG_HD_FREE_NOINLINE void rot_draw(RotBlit &rb, int sw, int sh, const double *r, const RotXform &m) {
    rb.pad = 0;  // row window [lo, hi) the spans can fall in: lo | hi << 8 (set below)
    rb.absolute = 0;
    rb.dudx = rb.dvdx = rb.dudy = rb.dvdy = rb.u0 = rb.v0 = 0;
    rb.m11 = rb.m12 = rb.m21 = rb.m22 = rb.dx = rb.dy = 0;
    if (sw <= 0 || sh <= 0 || !(r[2] > 0) || !(r[3] > 0))
        return;
    double minx = 1e300, miny = 1e300, maxx = -1e300, maxy = -1e300;
    for (int cidx = 0; cidx < 4; cidx++) {
        const double fx = (cidx & 1) ? r[0] + r[2] : r[0], fy = (cidx & 2) ? r[1] + r[3] : r[1];
        const double X = m.m11 * fx + m.m21 * fy + m.dx, Y = m.m12 * fx + m.m22 * fy + m.dy;
        if (X < minx) minx = X;
        if (X > maxx) maxx = X;
        if (Y < miny) miny = Y;
        if (Y > maxy) maxy = Y;
    }
    {
        // only the rows the quad can touch are cleared here and scanned by the caller afterwards
        // (every rasteriser below emits spans inside the quad's bounding box, +-1 row of rounding)
        int lo = (int)pg_dfloor(miny) - 2, hi = (int)pg_dceil(maxy) + 3;
        if (lo < 0) lo = 0;
        if (hi > RES_H) hi = RES_H;
        if (!(maxy >= -2) || !(miny <= RES_H + 2) || hi <= lo) {
            rb.pad = 0;
            return;
        }
        for (int y = lo; y < hi; y++) rb.x1[y] = rb.x2[y] = 0;
        rb.pad = lo | (hi << 8);
    }
    if (maxx - minx >= 16 && maxy - miny >= 16) {
        rot_transform_image(rb, sw, sh, r, m);
        return;
    }
    double c11 = m.m11, c12 = m.m12, c21 = m.m21, c22 = m.m22;
    const double cdx = m.dx + r[0] * m.m11 + r[1] * m.m21;
    const double cdy = m.dy + r[1] * m.m22 + r[0] * m.m12;
    const double sx = r[2] / (double)sw, sy = r[3] / (double)sh;
    c11 *= sx; c12 *= sx; c21 *= sy; c22 *= sy;
    const double t = 1.0 / 65536;
    const double pdx = t * c11 + t * c21 + cdx;
    const double pdy = t * c12 + t * c22 + cdy;
    const double det = c11 * c22 - c12 * c21;
    if (det == 0)
        return;
    const double dinv = 1.0 / det;
    rb.m11 = c22 * dinv;
    rb.m12 = -c12 * dinv;
    rb.m21 = -c21 * dinv;
    rb.m22 = c11 * dinv;
    rb.dx = (c21 * pdy - c22 * pdx) * dinv;
    rb.dy = (c12 * pdx - c11 * pdy) * dinv;
    rb.dudx = (int)(rb.m11 * 65536.0);  // fdx
    rb.dvdx = (int)(rb.m12 * 65536.0);  // fdy
    const double ly = (r[1] + (r[1] + r[3])) * 0.5f;
    const double lx = (r[0] + r[0]) * 0.5f;
    const double rx = ((r[0] + r[2]) + (r[0] + r[2])) * 0.5f;
    const double ax = m.m11 * lx + m.m21 * ly + m.dx, ay = m.m12 * lx + m.m22 * ly + m.dy;
    const double bx = m.m11 * rx + m.m21 * ly + m.dx, by = m.m12 * rx + m.m22 * ly + m.dy;
    rot_rasterize_line(rb, ax, ay, bx, by, r[3] / r[2]);
}

// ---- rule F: opaque fillRect
PG_HD_FREE_NOINLINE void make_solid_blit(Blit &b, double x, double y, double w, double h, uint32_t rgb) {
    int x1 = pg_qround(x), y1 = pg_qround(y);
    int x2 = pg_qround(x + w), y2 = pg_qround(y + h);
    if (x2 < x1) { int t = x1; x1 = x2; x2 = t; }
    if (y2 < y1) { int t = y1; y1 = y2; y2 = t; }
    if (x1 < 0) x1 = 0;
    if (y1 < 0) y1 = 0;
    if (x2 > RES_W) x2 = RES_W;
    if (y2 > RES_H) y2 = RES_H;
    blit_clear(b);
    if (x2 <= x1 || y2 <= y1)
        return;
    b.x1 = (uint8_t)x1;
    b.y1 = (uint8_t)y1;
    b.w = (uint8_t)(x2 - x1);
    b.h = (uint8_t)(y2 - y1);
    b.kind = BLIT_SOLID;
    b.mirror = 0;
    b.opacity = 256;
    b.src = 0xff000000u | rgb;
    b.ix = b.iy = 0;
    b.basex = b.srcy = 0;
    b.sw = b.sh = 0;
}

// ---- rules B + O
// One layer of the composition = the premultiplied source value a blit contributes at a pixel
// (0: nothing), with the painter opacity already applied; layer_over is Qt's src-over.
//   opaque (alpha 255): replaces what is below — the shader's top-down walk stops there
//   opacity != 256:     s = BYTE_MUL(src, (io*255)>>8) has alpha <= 254, so it never looks opaque
PG_HD uint32_t layer_over(uint32_t dst, uint32_t s) {
    if (s >= 0xff000000u)
        return s;
    if (s != 0)
        return s + pg_byte_mul(dst, (~s) >> 24);
    return dst;
}
PG_HD uint32_t layer_of(uint32_t src, int int_opacity) {
    if (int_opacity == 256 || src == 0)
        return src;
    return pg_byte_mul(src, (uint32_t)((int_opacity * 255) >> 8));
}

// Out of line on the device: it is the rare path of the shader, and inlined at its dozen call sites
// it made the render kernel ten times the size of the instruction cache.
PG_HD_FREE_NOINLINE uint32_t blit_texel(const Blit &b, int px, int py, const uint32_t *atlas, const RotBlit *rots) {
    const uint32_t box = *reinterpret_cast<const uint32_t *>(&b);  // x1 | y1<<8 | w<<16 | h<<24
    const uint32_t dx = (uint32_t)px - (box & 0xffu);
    const uint32_t dy = (uint32_t)py - ((box >> 8) & 0xffu);
    if (dx >= ((box >> 16) & 0xffu) || dy >= (box >> 24))
        return 0;
    if (b.kind == BLIT_SOLID)
        return b.src;
    if (b.kind == BLIT_SPANS) {  // one solid-colour span per row (ellipse / cosmetic line), src-over
        const RotBlit &rb = rots[b.ix];
        if (px < (int)rb.x1[py] || px >= (int)rb.x2[py])
            return 0;
        return b.src;
    }
    if (b.kind == BLIT_ROTATED) {
        const RotBlit &rb = rots[b.ix];
        const int xs = rb.x1[py];
        if (px < xs || px >= (int)rb.x2[py])
            return 0;
        long long tu, tv;
        if (rb.absolute) {
            tu = ((long long)px * rb.dudx + (long long)py * rb.dudy + rb.u0) >> 16;
            tv = ((long long)px * rb.dvdx + (long long)py * rb.dvdy + rb.v0) >> 16;
        } else {
            const double cx = xs + 0.5, cy = py + 0.5;
            int fx = (int)((rb.m21 * cy + rb.m11 * cx + rb.dx) * 65536.0);
            int fy = (int)((rb.m22 * cy + rb.m12 * cx + rb.dy) * 65536.0);
            fx = (int)((uint32_t)fx + (uint32_t)rb.dudx * (uint32_t)(px - xs));
            fy = (int)((uint32_t)fy + (uint32_t)rb.dvdx * (uint32_t)(px - xs));
            tu = fx >> 16;
            tv = fy >> 16;
        }
        if (tu < 0) tu = 0;
        if (tu > (long long)b.sw - 1) tu = (long long)b.sw - 1;
        if (tv < 0) tv = 0;
        if (tv > (long long)b.sh - 1) tv = (long long)b.sh - 1;
        if (b.mirror)
            tu = b.sw - 1 - tu;
        return layer_of(atlas[b.src + (uint32_t)tv * b.sw + (uint32_t)tu], b.opacity);
    }
    if (b.kind != BLIT_IMAGE)
        return 0;
    uint32_t sx = (b.basex + (uint32_t)b.ix * dx) >> 16;
    uint32_t sy = (b.srcy + (uint32_t)b.iy * dy) >> 16;
    if (b.mirror)
        sx = b.sw - 1 - sx;
    return layer_of(atlas[b.src + sy * b.sw + sx], b.opacity);
}

// Tile (sprite, tw, th) of the global table: what an un-clipped, un-mirrored, opaque-painter
// drawImage of snapped size tw x th fetches, pixel by pixel. Texels the edge guards of
// make_image_blit drop are 0 (= nothing drawn).
PG_HD uint32_t tile_texel(const Blit &b, const uint32_t *atlas, int dx, int dy) {
    if (b.kind != BLIT_IMAGE || dx >= (int)b.w || dy >= (int)b.h)
        return 0;
    const uint32_t sx = (b.basex + (uint32_t)b.ix * (uint32_t)dx) >> 16;
    const uint32_t sy = (b.srcy + (uint32_t)b.iy * (uint32_t)dy) >> 16;
    return atlas[b.src + sy * b.sw + sx];
}

// ---- rules E / L: QPainter::drawEllipse and drawLine as the raster engine runs them for the
// jumper compass (jumper.cpp:137-169); oracle/shim/qt_raster.cpp has the provenance and the sweep
// against Qt 6.6.3. Both produce one span per pixel row, kept in a RotBlit slot taken from the END
// of the frame's rot array (entity rotations allocate from the front).
template <class Frame>
PG_HD RotBlit *span_blit_begin(Frame &f, Blit &b, int k, uint32_t argb_premultiplied) {
    blit_clear(b);
    const int slot = Frame::kMaxRot - 1 - k;
    if (slot < 0)
        return nullptr;
    RotBlit &rb = f.rot[slot];
    for (int y = 0; y < RES_H; y++) rb.x1[y] = rb.x2[y] = 0;
    rb.pad = RES_H << 8;  // row window = the whole device
    b.ix = slot;
    b.src = argb_premultiplied;
    b.opacity = 256;
    return &rb;
}
PG_HD void span_blit_finish(Blit &b, const RotBlit &rb) {
    int y0 = RES_H, y1 = -1, x0 = RES_W, x1 = 0;
    for (int y = 0; y < RES_H; y++) {
        if (rb.x2[y] > rb.x1[y]) {
            if (y < y0) y0 = y;
            y1 = y;
            if (rb.x1[y] < x0) x0 = rb.x1[y];
            if (rb.x2[y] > x1) x1 = rb.x2[y];
        }
    }
    if (y1 < y0)
        return;
    b.x1 = (uint8_t)x0;
    b.y1 = (uint8_t)y0;
    b.w = (uint8_t)(x1 - x0);
    b.h = (uint8_t)(y1 - y0 + 1);
    b.kind = BLIT_SPANS;
}

// drawEllipsePoints (qpaintengine_raster.cpp): mirrored outline spans of one step + the fill between
PG_HD void ellipse_points(RotBlit &rb, int rx, int ry, int rw, int rh, bool pen, bool brush, int x, int y, int length) {
    if (length == 0)
        return;
    const int midx = rx + (rw + 1) / 2;
    const int midy = ry + (rh + 1) / 2;
    x = x + midx;
    y = midy - y;
    const int ox0 = midx + (midx - x) - (length - 1) - (rw & 0x1);
    const int ol0 = length < x - ox0 ? length : x - ox0;
    const int oy_top = y;
    const int oy_bot = midy + (midy - y) - (rh & 0x1);
    if (brush && ox0 + ol0 < x) {
        const int fx = ox0 + ol0 - 1;
        const int fl = x - fx > 0 ? x - fx : 0;
        rot_span(rb, fx, fl, oy_top);
        if (!(oy_top >= oy_bot))
            rot_span(rb, fx, fl, oy_bot);
    }
    if (pen) {
        rot_span(rb, ox0, ol0, oy_top);
        rot_span(rb, x, length, oy_top);
        if (!(oy_top >= oy_bot)) {
            rot_span(rb, ox0, ol0, oy_bot);
            rot_span(rb, x, length, oy_bot);
        }
    }
}

// QRasterPaintEngine::drawEllipse on a device rect (pen at most one pixel wide, same colour as the
// brush, or no pen). Integer-aligned rects run drawEllipse_midpoint_i; the three non-aligned rects in
// scope — jumper's compass disc in easy mode and in the whole-world views of center_agent = false,
// constants of the 64x64 contract — replay the rows captured from Qt 6.6.3
// (tests/tools/qt6_compass_mask.py). Returns false for anything else.
template <class Frame>
PG_HD bool make_ellipse_blit(Frame &f, Blit &b, int k, double x, double y, double w, double h, uint32_t argb_premultiplied, bool pen) {
    RotBlit *rbp = span_blit_begin(f, b, k, argb_premultiplied);
    if (!rbp)
        return false;
    RotBlit &rb = *rbp;
    const bool integral = x == pg_dfloor(x) && y == pg_dfloor(y) && w == pg_dfloor(w) && h == pg_dfloor(h);
    if (!integral) {
        // {x, y, w} of the three non-integer discs of the 64x64 contract, then first row, row count
        const double rects[3][3] = {{46.66666793823242, 1.3333333730697632, 16.0},            // easy, agent-centred
                                    {53.60000228881836, 0.800000011920929, 9.600000381469727},   // easy, whole world (center_agent = false)
                                    {60.400001525878906, 0.4000000059604645, 3.200000047683716}};  // hard, whole world
        const uint8_t first_row[3] = {1, 0, 0}, n_rows[3] = {17, 11, 4}, row0[3] = {0, 17, 28};
        const uint8_t rows[32][2] = {{52, 58}, {50, 59}, {49, 60}, {48, 61}, {48, 62}, {47, 63}, {47, 63}, {46, 63}, {46, 63}, {46, 63}, {47, 63},
                                     {47, 63}, {47, 62}, {48, 61}, {49, 60}, {51, 59}, {53, 57},
                                     {58, 59}, {56, 61}, {55, 62}, {54, 63}, {53, 63}, {53, 64}, {53, 64}, {54, 64}, {54, 63}, {55, 62}, {57, 61},
                                     {61, 63}, {60, 64}, {60, 64}, {61, 63}};
        int which = -1;
        for (int i = 0; i < 3; i++)
            if (x == rects[i][0] && y == rects[i][1] && w == rects[i][2] && h == rects[i][2])
                which = i;
        if (which < 0 || !pen || (argb_premultiplied >> 24) != 255u)
            return false;
        for (int i = 0; i < n_rows[which]; i++) {
            const uint8_t *r = rows[row0[which] + i];
            rot_span(rb, r[0], r[1] - r[0], first_row[which] + i);
        }
        span_blit_finish(b, rb);
        return true;
    }
    const int rx = (int)x, ry = (int)y;
    const int rw = (int)(x + w) - (int)x, rh = (int)(y + h) - (int)y;
    if (rw <= 0 || rh <= 0)
        return true;
    const double a = (double)rw / 2;
    const double bb = (double)rh / 2;
    double d = bb * bb - (a * a * bb) + 0.25 * a * a;
    int ex = 0;
    int ey = (rh + 1) / 2;
    int startx = ex;
    while (a * a * (2 * ey - 1) > 2 * bb * bb * (ex + 1)) {  // region 1
        if (d < 0) {
            d += bb * bb * (2 * ex + 3);
            ++ex;
        } else {
            d += bb * bb * (2 * ex + 3) + a * a * (-2 * ey + 2);
            ellipse_points(rb, rx, ry, rw, rh, pen, true, startx, ey, ex - startx + 1);
            startx = ++ex;
            --ey;
        }
    }
    ellipse_points(rb, rx, ry, rw, rh, pen, true, startx, ey, ex - startx + 1);
    d = bb * bb * (ex + 0.5) * (ex + 0.5) + a * a * ((ey - 1) * (ey - 1) - bb * bb);  // region 2
    const int miny = rh & 0x1;
    while (ey > miny) {
        if (d < 0) {
            d += bb * bb * (2 * ex + 2) + a * a * (-2 * ey + 3);
            ++ex;
        } else {
            d += a * a * (-2 * ey + 3);
        }
        --ey;
        ellipse_points(rb, rx, ry, rw, rh, pen, true, ex, ey, 1);
    }
    span_blit_finish(b, rb);
    return true;
}

// QCosmeticStroker::drawLine for one isolated line: integer end points (QPainter::drawLine(int...)),
// square caps, not clipped by the device edge (the caller guarantees it: the compass needle).
PG_HD int pg_fdot16_div(int x, int y) {
    int ax = x < 0 ? -x : x;
    if (ax > 0x7fff)
        return (int)((long long)x * (1 << 16) / y);
    return x * (1 << 16) / y;
}
template <class Frame>
PG_HD bool make_line_blit(Frame &f, Blit &b, int k, int ix1, int iy1, int ix2, int iy2, uint32_t argb_premultiplied) {
    RotBlit *rbp = span_blit_begin(f, b, k, argb_premultiplied);
    if (!rbp)
        return false;
    RotBlit &rb = *rbp;
    // clipLine's guard band: outside it Qt moves the end points and the stepping changes
    if (ix1 < 0 || ix1 >= RES_W || ix2 < 0 || ix2 >= RES_W || iy1 < 0 || iy1 >= RES_H || iy2 < 0 || iy2 >= RES_H)
        return false;
    if (ix1 == ix2 && iy1 == iy2) {
        rot_span(rb, ix1, 1, iy1);
        span_blit_finish(b, rb);
        return true;
    }
    int x1 = ix1 * 64, x2 = ix2 * 64, y1 = iy1 * 64, y2 = iy2 * 64;
    const int dx = x2 > x1 ? x2 - x1 : x1 - x2, dy = y2 > y1 ? y2 - y1 : y1 - y2;
    if (dx < dy) {
        if (y1 > y2) {
            int t = y1; y1 = y2; y2 = t;
            t = x1; x1 = x2; x2 = t;
        }
        const int xinc = pg_fdot16_div(x2 - x1, y2 - y1);
        int x = x1 * (1 << 10);
        y1 -= 32;  // CapBegin
        x -= xinc >> 1;
        y2 += 32;  // CapEnd
        int y = (y1 + 32) >> 6;
        const int ys = (y2 + 32) >> 6;
        const int round = (xinc > 0) ? 32 : 0;
        if (y != ys) {
            x += ((y * (1 << 6)) + round - y1) * xinc >> 6;
            do {
                rot_span(rb, x >> 16, 1, y);
                x += xinc;
            } while (++y < ys);
        }
    } else {
        if (x1 > x2) {
            int t = x1; x1 = x2; x2 = t;
            t = y1; y1 = y2; y2 = t;
        }
        const int yinc = pg_fdot16_div(y2 - y1, x2 - x1);
        int y = y1 * (1 << 10);
        x1 -= 32;
        y -= yinc >> 1;
        x2 += 32;
        int x = (x1 + 32) >> 6;
        const int xs = (x2 + 32) >> 6;
        const int round = (yinc > 0) ? 32 : 0;
        if (x != xs) {
            y += ((x * (1 << 6)) + round - x1) * yinc >> 6;
            do {
                rot_span(rb, x, 1, y >> 16);
                y += yinc;
            } while (++x < xs);
        }
    }
    span_blit_finish(b, rb);
    return true;
}

template <class G, class Frame>
struct Raster {
    using E = Engine<G>;

    static PG_HD Camera camera_of(const EnvHdr &h) {
        Camera cam;
        cam.unit = h.unit;
        cam.view_dim = h.view_dim;
        cam.x_off = h.x_off;
        cam.y_off = h.y_off;
        return cam;
    }
    // basic-abstract-game.cpp:799-801 — float math, then widened to QRectF doubles
    static PG_HD void screen_rect(const Camera &f, float x, float y, float dx, float dy, float render_eps, double *r) {
        r[0] = (double)((x - render_eps) * f.unit - f.x_off);
        r[1] = (double)((f.view_dim - y - render_eps) * f.unit + f.y_off);
        r[2] = (double)((dx + 2 * render_eps) * f.unit);
        r[3] = (double)((dy + 2 * render_eps) * f.unit);
    }
    // basic-abstract-game.cpp:803-805
    static PG_HD void abs_rect(const Camera &f, float x, float y, float dx, float dy, double *r) {
        r[0] = (double)(x * f.unit);
        r[1] = (double)(y * f.unit);
        r[2] = (double)(dx * f.unit);
        r[3] = (double)(dy * f.unit);
    }
    // qt-utils.h:12-19
    static PG_HD void adjust_rect(double *r, const double *adj) {
        double x = r[0] + r[2] * adj[0];
        double y = r[1] + r[3] * adj[1];
        double w = r[2] * adj[2];
        double h = r[3] * adj[3];
        r[0] = x; r[1] = y; r[2] = w; r[3] = h;
    }
    // basic-abstract-game.cpp:811-817
    static PG_HD void object_rect(const Camera &f, const Entity &o, double *r) {
        if (o.use_abs_coords) {
            abs_rect(f, f.view_dim * (o.x - o.rx), f.view_dim * (o.y + o.ry), 2 * f.view_dim * o.rx, 2 * f.view_dim * o.ry, r);
            return;
        }
        screen_rect(f, o.x - o.rx, o.y + o.ry, 2 * o.rx, 2 * o.ry, 0, r);
    }

    // draw_image (basic-abstract-game.cpp:877-913) for the un-rotated, un-tiled case
    static PG_HD_NOINLINE void make_sprite_blit(Ctx &cref, Frame &f, Blit &b, double *rect, float rotation, bool is_reflected, int base_type, int theme, float alpha,
                                                int defer_ei = -1) {
        Ctx c = cref;  // private copy: see Engine::sub_step
        make_sprite_blit_body<false>(c, f, b, rect, rotation, is_reflected, base_type, theme, alpha, defer_ei);
    }
    // the same, inlined into its caller (the per-entity site of the setup kernel: ~20 calls per frame, each
    // of which otherwise saves and restores its registers twice, here and in make_image_blit)
    static PG_HD void make_sprite_blit_inl(Ctx &c, Frame &f, Blit &b, double *rect, float rotation, bool is_reflected, int base_type, int theme, float alpha,
                                           int defer_ei = -1) {
        make_sprite_blit_body<true>(c, f, b, rect, rotation, is_reflected, base_type, theme, alpha, defer_ei);
    }
    template <bool INL>
    static PG_HD void make_sprite_blit_body(Ctx &c, Frame &f, Blit &b, double *rect, float rotation, bool is_reflected, int base_type, int theme, float alpha,
                                            int defer_ei) {
        blit_clear(b);
        int img_type = G::image_for_type(c, base_type);
        if (img_type < 0)
            return;
        if (c.h->options.use_monochrome_assets || img_type >= USE_ASSET_THRESHOLD) {
            if (img_type == SPACE)
                return;
            if (!G::make_grid_obj_blit(c, f, b, rect, img_type, theme))
                c.h->err |= ERR_UNSUPPORTED;
            return;
        }
        if (theme < 0 || theme >= MAX_IMAGE_THEMES) {
            c.h->err |= ERR_FASSERT;
            return;
        }
        int masked_theme = (c.h->options.restrict_themes && !G::should_preserve_type_themes(c, img_type)) ? 0 : theme;
        double adj[4];
        if (G::get_adjusted_image_rect(c, img_type, adj))
            adjust_rect(rect, adj);
        SpriteDesc sd = c.assets->sprites[img_type + masked_theme * MAX_ASSETS];
        if (sd.w == 0) {
            c.h->err |= ERR_UNSUPPORTED;  // reference would synthesise an asset (assetgen.cpp)
            return;
        }
        int io = 256;
        if (alpha != 1)
            io = (int)((double)alpha * 256);
        if (rotation == 0) {
            if (INL)
                make_image_blit_inl(b, rect[0], rect[1], rect[2], rect[3], sd, is_reflected, io, f.snap != 0);
            else
                make_image_blit(b, rect[0], rect[1], rect[2], rect[3], sd, is_reflected, io, f.snap != 0);
            return;
        }
        // basic-abstract-game.cpp:901-906: translate to the rect centre, rotate, draw the centred rect
        RotXform m;
        m.dx = rect[0] + rect[2] / 2;
        m.dy = rect[1] + rect[3] / 2;
        const double a = (double)(rotation * 180 / PI_F);
        double sina = 0, cosa = 0;  // QTransform::rotate: exact at right angles
        if (a == 90. || a == -270.)
            sina = 1.;
        else if (a == 270. || a == -90.)
            sina = -1.;
        else if (a == 180.)
            cosa = -1.;
        else {
            const double rad = 0.017453292519943295769 * a;
            sina = sin(rad);
            cosa = cos(rad);
        }
        m.m11 = cosa; m.m12 = sina; m.m21 = -sina; m.m22 = cosa;
        double r[4] = {-rect[2] / 2, -rect[3] / 2, rect[2], rect[3]};
        if (pg_dfabs(m.m12) <= 1e-12 && pg_dfabs(m.m21) <= 1e-12) {
            // QTransform::type() is fuzzy: +-180 degrees is a (mirroring) scale
            make_image_blit(b, m.m11 * r[0] + m.dx, m.m22 * r[1] + m.dy, m.m11 * r[2], m.m22 * r[3], sd, is_reflected, io, f.snap != 0);
            return;
        }
        if (defer_ei >= 0) {
            // The scan conversion below is long and branchy; done here, by the thread that happens
            // to own the entity, it would serialise against the (different) code paths its warp
            // neighbours take for their entities. Reserve the slot and let frame_rots run all
            // rotated sprites of the frame side by side.
            b.kind = BLIT_ROT_PENDING;
            b.src = (uint32_t)defer_ei;
            return;
        }
        int slot;
#if defined(__CUDA_ARCH__)
        slot = atomicAdd(&f.n_rot, 1);
#else
        slot = f.n_rot++;
#endif
        if (slot >= Frame::kMaxRot) {
            c.h->err |= ERR_ROT_BLITS;
            return;
        }
        RotBlit &rb = f.rot[slot];
        rot_draw(rb, sd.w, sd.h, r, m);
        int y0 = RES_H, y1 = -1, x0 = RES_W, x1 = 0;
        const int row_lo = rb.pad & 0xff, row_hi = (rb.pad >> 8) & 0xff;
        for (int y = row_lo; y < row_hi; y++) {
            if (rb.x2[y] > rb.x1[y]) {
                if (y < y0) y0 = y;
                y1 = y;
                if (rb.x1[y] < x0) x0 = rb.x1[y];
                if (rb.x2[y] > x1) x1 = rb.x2[y];
            }
        }
        if (y1 < y0)
            return;
#if defined(__CUDA_ARCH__)
        f.rot[slot] = rb;  // rows outside [y0, y1] are never read: the blit's box excludes them
#endif
        b.x1 = (uint8_t)x0;
        b.y1 = (uint8_t)y0;
        b.w = (uint8_t)(x1 - x0);
        b.h = (uint8_t)(y1 - y0 + 1);
        b.kind = BLIT_ROTATED;
        b.mirror = is_reflected ? 1 : 0;
        b.opacity = (uint16_t)io;
        b.ix = slot;
        b.iy = 0;
        b.basex = b.srcy = 0;
        b.src = sd.off;
        b.sw = sd.w;
        b.sh = sd.h;
    }

    // draw_image's inner part for an already-resolved image type and already-adjusted rect
    static PG_HD_NOINLINE void make_sprite_blit_noadjust(Ctx &cref, Frame &f, Blit &b, double *rect, bool is_reflected, int img_type, int theme, float alpha) {
        Ctx c = cref;
        blit_clear(b);
        if (theme < 0 || theme >= MAX_IMAGE_THEMES) {
            c.h->err |= ERR_FASSERT;
            return;
        }
        int masked_theme = (c.h->options.restrict_themes && !G::should_preserve_type_themes(c, img_type)) ? 0 : theme;
        SpriteDesc sd = c.assets->sprites[img_type + masked_theme * MAX_ASSETS];
        if (sd.w == 0) {
            c.h->err |= ERR_UNSUPPORTED;
            return;
        }
        int io = 256;
        if (alpha != 1)
            io = (int)((double)alpha * 256);
        make_image_blit(b, rect[0], rect[1], rect[2], rect[3], sd, is_reflected, io, f.snap != 0);
    }

    // prepare_for_drawing (basic-abstract-game.cpp:819-838). Writes the camera into the env
    // header (those fields are part of the serialized state, :1202-1220). Logic thread.
    static PG_HD void prepare_camera(Ctx &c) {
        EnvHdr &h = *c.h;
        h.center_x = (float)(h.main_width * .5);
        h.center_y = (float)(h.main_height * .5);
        if (h.options.center_agent) {
            G::choose_center(c, h.center_x, h.center_y);
        } else {
            h.visibility = (float)(h.main_width > h.main_height ? h.main_width : h.main_height);
            if (h.visibility < h.min_visibility)
                h.visibility = h.min_visibility;
        }
        float raw_unit = 64 / h.visibility;
        h.unit = (float)((double)raw_unit * ((double)64.0f / 64.0));
        h.view_dim = (float)(64.0 / (double)raw_unit);
        h.x_off = h.unit * (h.center_x - h.view_dim / 2);
        h.y_off = h.unit * (h.center_y - h.view_dim / 2);
    }

    // visible grid window (basic-abstract-game.cpp:926-938); pure function of the header
    static PG_HD void grid_window(const EnvHdr &h, int &low_x, int &low_y, int &nx, int &ny) {
        int high_x, high_y;
        if (h.options.center_agent) {
            float margin = (float)((double)h.visibility / 2.0 + 1);
            low_x = (int)(h.center_x - margin);
            high_x = (int)(h.center_x + margin);
            low_y = (int)(h.center_y - margin);
            high_y = (int)(h.center_y + margin);
        } else {
            low_x = 0;
            high_x = h.main_width - 1;
            low_y = 0;
            high_y = h.main_height - 1;
        }
        nx = high_x - low_x + 1;
        ny = high_y - low_y + 1;
    }

    // device pixel span [p1, p2) of a cell column / row, and (tile_size) its snapped size when the
    // column's cells are un-clipped on the near side so that pre-scaled tiles apply (else 0)
    static PG_HD void span_of(double t, double tw, bool snap, int limit, uint8_t &p1, uint8_t &p2, uint8_t &tile_size, uint8_t &clip) {
        tile_size = 0;
        clip = 0;
        if (snap) {
            double x = pg_qround(t);
            tw = pg_qround(t + tw - x);
            t = x;
            if (tw >= 1 && tw <= MAX_TILE_DIM && x > -tw) {
                tile_size = (uint8_t)(int)tw;
                clip = x < 0 ? (uint8_t)(int)(-x) : 0;
            }
        }
        int a = pg_qround(t), b2 = pg_qround(t + tw);
        if (a < 0) a = 0;
        if (b2 > limit) b2 = limit;
        if (b2 < a) b2 = a;
        p1 = (uint8_t)a;
        p2 = (uint8_t)b2;
    }

    // ---- setup kernel, step 1: camera, visible window, background + overlay blits, cell spans
    // (prepare_for_drawing's results are in the header already; this is draw_background's and
    // draw_foreground's geometry, basic-abstract-game.cpp:921-1007). `tid` of `nthreads` lanes of one warp.
    static PG_HD void setup_frame(Ctx &c, Frame &f, bool snap, int tid, int nthreads) {
        EnvHdr &h = *c.h;
        const Camera cam = camera_of(h);
        int low_x, low_y, nx, ny;
        grid_window(h, low_x, low_y, nx, ny);
        if (!G::DRAWS_GRID) {
            // the game never puts anything into its grid and never looks outside it: no cell blits
            if (h.options.center_agent)
                h.err |= ERR_UNSUPPORTED;  // a centred view would show out-of-bounds cells
            nx = 0;
            ny = 0;
        }
        bool overflow = false;
        if (nx > Frame::kMaxCells1D) { nx = Frame::kMaxCells1D; overflow = true; }
        if (ny > Frame::kMaxCells1D) { ny = Frame::kMaxCells1D; overflow = true; }
        // the two snapped sizes a cell can have: floor(w) and floor(w) + 1 (w = QRectF width of a cell)
        double cw[4];
        screen_rect(cam, 0.f, 1.f, 1, 1, RENDER_EPS, cw);
        const int w0 = (int)pg_dfloor(cw[2]);
        if (tid == 0) {
            f.cam = cam;
            f.snap = snap ? 1 : 0;
            f.low_x = low_x;
            f.low_y = low_y;
            f.nx = nx;
            f.ny = ny;
            f.n_overlay = 0;
            f.n_bg = 0;
            f.n_ent = 0;
            f.n_ent_below = 0;
            f.n_rot = 0;
            f.n_jobs = 0;
            f.n_gen = 0;
            f.tile_top = 0;
            f.n_tjobs = 0;
            f.tile_w0 = f.tile_h0 = w0;
            f.cell_w = cw[2];
            f.rot = reinterpret_cast<RotBlit *>(c.rot_scratch_raw);
            f.ents = c.blit_list;
            f.gen_spill = c.cell_spill;
            if (overflow)
                h.err |= ERR_BLIT_OVERFLOW;
            if (h.options.use_backgrounds)
                G::make_background_blits(c, f);
            // the usual case — one opaque background image (RGB32: alpha 255) — gets per-row / per-column
            // source offsets instead of a blit walk (Frame::pad = 1); where the view leaves the
            // world the image covers only part of the device and the rest stays black
            f.pad = 0;
            if (f.n_bg == 1) {
                const Blit &b0 = f.bg[0];
                if (b0.kind == BLIT_IMAGE && b0.opacity == 256 && !b0.mirror)
                    f.pad = 1;
            }
            if (h.has_useful_vel_info && h.options.paint_vel_info) {
                // draw_foreground's last step (basic-abstract-game.cpp:960-969): two grey squares
                // whose shade encodes the agent's velocity; to_shade is qt-utils.h:21-28
                const Entity &a = agent_of(c);
                const float infodim = (float)(RES_H * .2);
                float f1 = (float)(.5 * (double)a.vx / (double)h.maxspeed + .5);
                float f2 = (float)(.5 * (double)a.vy / (double)h.max_jump + .5);
                int s1 = (int)(f1 * 255), s2 = (int)(f2 * 255);
                s1 = s1 < 0 ? 0 : (s1 > 255 ? 255 : s1);
                s2 = s2 < 0 ? 0 : (s2 > 255 ? 255 : s2);
                make_solid_blit(f.overlay[0], 0, 0, (double)infodim, (double)infodim, ((uint32_t)s1 << 16) | ((uint32_t)s1 << 8) | (uint32_t)s1);
                make_solid_blit(f.overlay[1], (double)infodim, 0, (double)infodim, (double)infodim,
                                ((uint32_t)s2 << 16) | ((uint32_t)s2 << 8) | (uint32_t)s2);
                f.n_overlay = 2;
            }
            G::make_overlay_blits(c, f);  // game overlays are appended after the velocity squares
        }
        if (G::DRAWS_GRID) {
            uint32_t *keys = reinterpret_cast<uint32_t *>(f.tilekey);
            for (int i = tid; i < CELL_KEYS / 2; i += nthreads) keys[i] = 0;
        }
        // columns by lanes 0.., rows by lanes from the top end
        for (int i = tid; i < nx; i += nthreads) {
            double r[4];
            screen_rect(cam, (float)(low_x + i), (float)(low_y + 1), 1, 1, RENDER_EPS, r);
            f.col_x[i] = r[0];
            uint8_t ts;
            span_of(r[0], r[2], snap, RES_W, f.col_p1[i], f.col_p2[i], ts, f.col_k0[i]);
            f.col_tw[i] = (ts == w0 || ts == w0 + 1) ? ts : 0;
        }
        for (int jj = tid; jj < ny; jj += nthreads) {
            int j = ny - 1 - jj;
            double r[4];
            screen_rect(cam, (float)low_x, (float)(low_y + j + 1), 1, 1, RENDER_EPS, r);
            f.row_y[j] = r[1];
            uint8_t ts;
            span_of(r[1], r[3], snap, RES_H, f.row_p1[j], f.row_p2[j], ts, f.row_k0[j]);
            f.row_th[j] = (ts == w0 || ts == w0 + 1) ? ts : 0;
        }
        for (int i = nx + tid; i < Frame::kSpanBytes; i += nthreads) f.col_p1[i] = f.col_p2[i] = 255;
        for (int j = ny + tid; j < Frame::kSpanBytes; j += nthreads) f.row_p1[j] = f.row_p2[j] = 255;
    }

    // cell columns (rows) covering pixel column (row) p -> lo / hi and the packed CI_* words of hi and of lo
    // Spans are monotonic in the cell index (columns left to right; rows bottom-up, i.e. decreasing), so the
    // cells covering pixel p are a contiguous index range that two counts give: how many spans start at or
    // before p, how many end at or before p. Four spans per compare (byte-wise SIMD on the device).
    static PG_HD uint32_t ci_word(const uint8_t *p1, const uint8_t *tsize, const uint8_t *k0, int base_mul, int px, int i) {
        return (uint32_t)(i * base_mul) | CI_VALID | ((uint32_t)((px - p1[i] + k0[i]) & 31) << CI_D_SHIFT) | ((uint32_t)tsize[i] << CI_TW_SHIFT);
    }
    static PG_HD uint32_t cell_lookup(const uint8_t *p1, const uint8_t *p2, const uint8_t *tsize, const uint8_t *k0, int n, int base_mul, int px, uint8_t &lo,
                                      uint8_t &hi, uint32_t &lo_word) {
        int started = 0, ended = 0;
#if defined(__CUDA_ARCH__)
        const uint32_t pv = (uint32_t)px * 0x01010101u;
        const uint32_t *w1 = reinterpret_cast<const uint32_t *>(p1), *w2 = reinterpret_cast<const uint32_t *>(p2);
        for (int w = 0; w < Frame::kSpanBytes / 4; w++) {
            started += __popc(__vcmpleu4(w1[w], pv));   // padding bytes are 255: never counted
            ended += __popc(__vcmpleu4(w2[w], pv));
        }
        started >>= 3;
        ended >>= 3;
#else
        for (int i = 0; i < n; i++) {
            started += p1[i] <= px;
            ended += p2[i] <= px;
        }
#endif
        const bool reversed = n > 1 && p1[n - 1] < p1[0];
        int l, hgh;
        if (!reversed) {
            l = ended;
            hgh = started - 1;
        } else {
            l = n - started;
            hgh = n - ended - 1;
        }
        if (l > hgh) {
            lo = 255;
            hi = 0;
            lo_word = 0;
            return 0;
        }
        lo = (uint8_t)l;
        hi = (uint8_t)hgh;
        uint32_t w = ci_word(p1, tsize, k0, base_mul, px, hgh);
        w |= l != hgh ? CI_MULTI : CI_FAST;
        if (hgh - l > 1)
            w |= CI_WIDE;
        lo_word = l == hgh ? w : ci_word(p1, tsize, k0, base_mul, px, l);
        return w;
    }

    // tile_image (basic-abstract-game.cpp:840-869): number of tiles an entity's sprite is repeated
    // over (0 = plain single draw) and the rect of tile i. Float/double mix as in the reference.
    static PG_HD int tile_count(const double *rect, float tile_ratio) {
        if (tile_ratio == 0)
            return 0;
        int num_tiles;
        if (tile_ratio < 0) {
            tile_ratio = -1 * tile_ratio;
            num_tiles = (int)(rect[3] / (rect[2] * (double)tile_ratio));
        } else {
            num_tiles = (int)(rect[2] / (rect[3] * (double)tile_ratio));
        }
        if (num_tiles < 1)
            num_tiles = 1;
        return num_tiles;
    }
    static PG_HD void tile_rect(const double *rect, float tile_ratio, int num_tiles, int i, double *out) {
        if (tile_ratio < 0) {
            float tile_height = (float)(rect[3] / num_tiles);
            float tile_width = (float)rect[2];
            out[0] = rect[0];
            out[1] = rect[1] + (double)(tile_height * i);
            out[2] = (double)tile_width;
            out[3] = (double)tile_height;
        } else {
            float tile_width = (float)(rect[2] / num_tiles);
            float tile_height = (float)rect[3];
            out[0] = rect[0] + (double)(tile_width * i);
            out[1] = rect[1];
            out[2] = (double)tile_width;
            out[3] = (double)tile_height;
        }
    }

    // Tiles are laid along one axis, so the ones that can touch the device form one contiguous run
    // [j0, j0 + count): everything else would only produce empty blits. One pixel of guard band
    // covers the rounding rules.
    static PG_HD int visible_tiles(const double *r, float tile_ratio, int nt, int &j0) {
        // same arithmetic as tile_rect, with the per-tile size computed once
        const bool vertical = tile_ratio < 0;
        const float step = vertical ? (float)(r[3] / nt) : (float)(r[2] / nt);
        const double origin = vertical ? r[1] : r[0];
        const double limit = vertical ? RES_H + 1 : RES_W + 1;
        // the other axis is the same for every tile
        const bool cross_visible = vertical ? !(r[0] + (double)(float)r[2] < -1 || r[0] > RES_W + 1) : !(r[1] + (double)(float)r[3] < -1 || r[1] > RES_H + 1);
        int first = -1, last = -2;
        if (cross_visible) {
            for (int i = 0; i < nt; i++) {
                const double lo = origin + (double)(step * i);
                const bool vis = !(lo + (double)step < -1 || lo > limit);
                if (vis) {
                    if (first < 0)
                        first = i;
                    last = i;
                }
            }
        }
        j0 = first < 0 ? 0 : first;
        return first < 0 ? 0 : last - first + 1;
    }

    // Blits of entity `ei`: 0 (not drawn / off screen), 1 (normal) or one per tile. `emit(j, blit)`
    // is called for j in [0, count) when `store` is set; returns count.
    template <class Emit>
    static PG_HD int entity_blits(Ctx &c, Frame &f, int ei, bool store, Blit &single, Emit emit) {
        blit_clear(single);
        if (!G::should_draw_entity(c, ei))
            return 0;
        const Entity &o = c.ents[ei];
        double r[4];
        object_rect(f.cam, o, r);
        float tile_ratio = G::get_tile_aspect_ratio(c, ei);
        if (tile_ratio != 0 && o.rotation == 0) {
            // draw_image: the adjusted rect is tiled (adjustment first, basic-abstract-game.cpp:890-900)
            int img_type = G::image_for_type(c, o.image_type);
            if (img_type < 0 || img_type >= USE_ASSET_THRESHOLD || c.h->options.use_monochrome_assets) {
                if (store)
                    make_sprite_blit(c, f, single, r, 0, o.is_reflected != 0, o.image_type, o.image_theme, o.alpha);
                else
                    make_sprite_blit(c, f, single, r, 0, o.is_reflected != 0, o.image_type, o.image_theme, o.alpha);
                if (single.kind == BLIT_NONE)
                    return 0;
                if (store)
                    emit(0, single);
                return 1;
            }
            double adj[4];
            if (G::get_adjusted_image_rect(c, img_type, adj))
                adjust_rect(r, adj);
            // entirely off screen (with a one pixel guard band for the rounding rules): no tiles
            if (r[0] + r[2] < -1 || r[1] + r[3] < -1 || r[0] > RES_W + 1 || r[1] > RES_H + 1)
                return 0;
            const int nt = tile_count(r, tile_ratio);
            int j0;
            const int nvis = visible_tiles(r, tile_ratio, nt, j0);
            if (store) {
                for (int i = 0; i < nvis; i++) {
                    double tr[4];
                    tile_rect(r, tile_ratio, nt, j0 + i, tr);
                    Blit b;
                    make_sprite_blit_noadjust(c, f, b, tr, o.is_reflected != 0, img_type, o.image_theme, o.alpha);
                    emit(i, b);
                }
            }
            return nvis;
        }
#if defined(__CUDA_ARCH__)
#if PG_SETUP_INLINE_BLIT
        make_sprite_blit_inl(c, f, single, r, o.rotation, o.is_reflected != 0, o.image_type, o.image_theme, o.alpha, G::DEFER_ROTATED ? ei : -1);
#else
        make_sprite_blit(c, f, single, r, o.rotation, o.is_reflected != 0, o.image_type, o.image_theme, o.alpha, G::DEFER_ROTATED ? ei : -1);
#endif
#else
        make_sprite_blit(c, f, single, r, o.rotation, o.is_reflected != 0, o.image_type, o.image_theme, o.alpha);
#endif
        if (single.kind == BLIT_NONE)
            return 0;
        if (store)
            emit(0, single);
        return 1;
    }

    // Tile j of tiled entity ei (same geometry as the tiled branch of entity_blits)
    static PG_HD void entity_tile_blit(Ctx &c, Frame &f, int ei, int j, Blit &b) {
        const Entity &o = c.ents[ei];
        double r[4];
        object_rect(f.cam, o, r);
        const float tile_ratio = G::get_tile_aspect_ratio(c, ei);
        const int img_type = G::image_for_type(c, o.image_type);
        double adj[4];
        if (G::get_adjusted_image_rect(c, img_type, adj))
            adjust_rect(r, adj);
        const int nt = tile_count(r, tile_ratio);
        double tr[4];
        tile_rect(r, tile_ratio, nt, j, tr);
        make_sprite_blit_noadjust(c, f, b, tr, o.is_reflected != 0, img_type, o.image_theme, o.alpha);
    }
    // first visible tile of tiled entity ei (see visible_tiles)
    static PG_HD int entity_first_visible_tile(Ctx &c, Frame &f, int ei) {
        const Entity &o = c.ents[ei];
        double r[4];
        object_rect(f.cam, o, r);
        const float tile_ratio = G::get_tile_aspect_ratio(c, ei);
        const int img_type = G::image_for_type(c, o.image_type);
        double adj[4];
        if (G::get_adjusted_image_rect(c, img_type, adj))
            adjust_rect(r, adj);
        int j0;
        visible_tiles(r, tile_ratio, tile_count(r, tile_ratio), j0);
        return j0;
    }

    // Entities -> blits in draw order (draw_entities z=-1 / 0 / 1, basic-abstract-game.cpp:1059-1066),
    // culled. The whole CTA cooperates (the host harness runs it with one thread): each thread owns
    // one entity per round and builds its blit(s) — for a rotated sprite that is a scan conversion
    // in fp64, the expensive part — and a block-wide prefix sum of the per-entity blit counts keeps
    // the list in draw order.
    static PG_HD void build_entity_blits(Ctx &c, Frame &f, int tid, int nthreads) {
        const int n = c.h->n_ents;
        int count = 0;
        int below = 0;
#if defined(__CUDA_ARCH__)
        __shared__ int warp_tot[32];
        const int lane = tid & 31, warp = tid >> 5, nwarps = (nthreads + 31) >> 5;
        const bool multi_warp = nthreads > 32;
#endif
        for (int z = -1; z <= 1; z++) {
            for (int base = 0; base < n; base += nthreads) {
                const int ei = base + tid;
                Blit single;
                blit_clear(single);
                int mine = 0;
                const bool active = ei < n && c.ents[ei].render_z == z;
                bool tiled = false;
                if (active) {
                    tiled = G::get_tile_aspect_ratio(c, ei) != 0 && c.ents[ei].rotation == 0;
                    mine = entity_blits(c, f, ei, false, single, [](int, const Blit &) {});
                }
                int pos = count;
                int total = mine;
#if defined(__CUDA_ARCH__)
                int incl = mine;
                for (int d = 1; d < 32; d <<= 1) {
                    int t = __shfl_up_sync(0xffffffffu, incl, d);
                    if (lane >= d)
                        incl += t;
                }
                if (multi_warp) {
                    if (lane == 31)
                        warp_tot[warp] = incl;
                    __syncthreads();
                    int woff = 0;
                    total = 0;
                    for (int w = 0; w < nwarps; w++) {
                        const int t = warp_tot[w];
                        if (w < warp)
                            woff += t;
                        total += t;
                    }
                    pos = count + woff + incl - mine;
                } else {
                    pos = count + incl - mine;
                    total = __shfl_sync(0xffffffffu, incl, 31);
                }
#endif
                if (mine > 0) {
                    if (pos + mine <= Frame::kMaxEntBlits) {
                        if (!tiled) {
                            f.ents[pos] = single;
                        } else {
#if defined(__CUDA_ARCH__)
                            const int job = mine > 1 ? atomicAdd(&f.n_jobs, 1) : Frame::kMaxTileJobs;
                            if (job < Frame::kMaxTileJobs) {
                                f.job_ei[job] = ei;
                                f.job_pos[job] = pos;
                                f.job_n[job] = mine;
                                f.job_j0[job] = entity_first_visible_tile(c, f, ei);
                            } else
#endif
                            {
                                Blit *dst = f.ents + pos;
                                entity_blits(c, f, ei, true, single, [=](int j, const Blit &b) { dst[j] = b; });
                            }
                        }
                    } else {
                        c.h->err |= ERR_ENT_BLITS;
                    }
                }
                count += total;
#if defined(__CUDA_ARCH__)
                if (multi_warp)
                    __syncthreads();  // warp_tot is reused by the next round
#endif
            }
            if (z == -1)
                below = count;
        }
        if (count > Frame::kMaxEntBlits)
            count = Frame::kMaxEntBlits;
        if (below > count)
            below = count;
        if (tid == 0) {
            if (!G::ENTS_BELOW_GRID && below > 0)
                c.h->err |= ERR_UNSUPPORTED;  // the game would have to declare ENTS_BELOW_GRID
            f.n_ent = count;
            f.n_ent_below = below;
            if (count > c.h->max_blits_seen)
                c.h->max_blits_seen = count;
            if (f.n_rot > c.h->max_rots_seen)
                c.h->max_rots_seen = f.n_rot;
        }
    }

    // qt_scale_image_32bit's source walk along one axis for a target of snapped size `t` whose first `k0`
    // pixels are cut off by the device edge (make_image_blit with tx = -k0, tx1 = 0) against the walk
    // of the un-clipped target (the pre-scaled tile): same texel for every visible pixel?
    static PG_HD bool clipped_walk_matches(int s, int t, int k0) {
        if (k0 == 0)
            return true;
        const double sx = (double)s / (double)t;
        const int ix = (int)(65536.0 * sx);
        const uint32_t bu = (uint32_t)((int)pg_dceil((0 + 0.5 - 0.0) * sx * 65536) - 1);
        const uint32_t bc = (uint32_t)((int)pg_dceil((0 + 0.5 - (double)(-k0)) * sx * 65536) - 1);
        for (int j = 0; j + k0 < t; j++)
            if (((bc + (uint32_t)ix * (uint32_t)j) >> 16) != ((bu + (uint32_t)ix * (uint32_t)(j + k0)) >> 16))
                return false;
        return true;
    }

    // ---- setup kernel, step 3: pixel -> cell lookups and the first pass over the visible cells
    static PG_HD void frame_build(Ctx &c, Frame &f, int tid, int nthreads, int /*unused*/) {
        const int wtid = tid, wn = nthreads;
        {
            const Blit &b = f.bg[0];
            const bool one = f.pad == 1;
            for (int p = wtid; p < RES_W + RES_H; p += wn) {
                if (p < RES_W) {
                    const uint32_t dx = (uint32_t)p - b.x1;
                    f.bgcol[p] = one && dx < b.w ? (b.basex + (uint32_t)b.ix * dx) >> 16 : BG_NONE;
                } else {
                    const uint32_t dy = (uint32_t)(p - RES_W) - b.y1;
                    f.bgrow[p - RES_W] = one && dy < b.h ? b.src + ((b.srcy + (uint32_t)b.iy * dy) >> 16) * b.sw : BG_NONE;
                }
            }
        }
        if (!G::DRAWS_GRID)
            return;
        for (int px = wtid; px < RES_W + RES_H; px += wn) {
            if (px < RES_W)
                f.colinfo[px] = cell_lookup(f.col_p1, f.col_p2, f.col_tw, f.col_k0, f.nx, f.ny, px, f.col_lo[px], f.col_hi[px], f.colinfo_lo[px]);
            else
                f.rowinfo[px - RES_W] = cell_lookup(f.row_p1, f.row_p2, f.row_th, f.row_k0, f.ny, 1, px - RES_W, f.row_lo[px - RES_W], f.row_hi[px - RES_W],
                                                    f.rowinfo_lo[px - RES_W]);
        }
        // Cells, pass A (draw_grid_obj / draw_image for a grid cell, basic-abstract-game.cpp:877-919,
        // 940-950): a cell whose sprite can come from the pre-scaled tile table only registers the
        // tile it needs; everything else (near-side clipped columns and rows, solid-colour cells,
        // adjusted rects, no snapping) becomes a general blit right away.
        const int ncells = f.nx * f.ny;
        const bool mono = c.h->options.use_monochrome_assets != 0;
#if defined(__CUDA_ARCH__)
        // the window's grid rows are ny short segments in ny different cache lines: touch them all at
        // once so the classification loop below runs on cache hits
        for (int j = wtid; j < f.ny; j += wn) {
            const int gy = f.low_y + j, gx = f.low_x < 0 ? 0 : f.low_x;
            if (gy >= 0 && gy < c.mh && gx < c.mw) {
                const int16_t *row = c.grid + gy * c.mw + gx;
                asm volatile("prefetch.global.L1 [%0];" ::"l"(row));
                if (f.nx > 32 || ((reinterpret_cast<uintptr_t>(row) & 127) + 2 * f.nx > 128))
                    asm volatile("prefetch.global.L1 [%0];" ::"l"(row + f.nx - 1 < c.grid + c.mh * c.mw ? row + f.nx - 1 : row));
            }
        }
#endif
        int ci = f.ny > 0 ? wtid / f.ny : 0, cj = wtid - ci * f.ny;  // (ci, cj) of cell k, advanced without dividing
        for (int k = wtid; k < ncells; k += wn) {
            if (k != wtid) {
                cj += wn;
                while (cj >= f.ny) {
                    cj -= f.ny;
                    ci++;
                }
            }
            f.cellmap[k] = 0;
            if (f.col_p1[ci] >= f.col_p2[ci] || f.row_p1[cj] >= f.row_p2[cj])
                continue;  // entirely off screen
            int type = E::get_obj(c, f.low_x + ci, f.low_y + cj);
            if (type == INVALID_OBJ)
                continue;
            // most of a level is empty: draw_image returns before drawing anything when the image type is
            // negative, and draw_grid_obj when it is SPACE (basic-abstract-game.cpp:880-882, 916)
            const int img_type = G::image_for_type(c, type);
            if (img_type < 0 || img_type == SPACE)
                continue;
            const int theme = G::theme_for_grid_obj(c, type);
            const int tw = f.col_tw[ci], th = f.row_th[cj];
            if (tw && th && !mono && type >= 0 && type < CELL_KEY_TYPES && theme >= 0 && theme < MAX_IMAGE_THEMES) {
                double adj[4];
                bool ok = img_type >= 0 && img_type < USE_ASSET_THRESHOLD && !G::get_adjusted_image_rect(c, img_type, adj);
                if (ok && (f.col_k0[ci] | f.row_k0[cj])) {
                    // a cell the near device edge cuts: its blit starts its 16.16 walk from the first visible
                    // pixel, the tile from the un-clipped origin — usable only if both visit the same texels
                    const int masked_theme = (c.h->options.restrict_themes && !G::should_preserve_type_themes(c, img_type)) ? 0 : theme;
                    const SpriteDesc sd = c.assets->sprites[img_type + masked_theme * MAX_ASSETS];
                    ok = sd.w != 0 && clipped_walk_matches(sd.w, tw, f.col_k0[ci]) && clipped_walk_matches(sd.h, th, f.row_k0[cj]);
                }
                if (ok) {
                    const int key = type * 4 + (tw - f.tile_w0) + 2 * (th - f.tile_h0);
                    f.tilekey[key] = 1;  // benign race: every writer stores 1
                    f.cellmap[k] = (uint16_t)(0x4000 | key);
                    continue;
                }
            }
            int slot;
#if defined(__CUDA_ARCH__)
            slot = atomicAdd(&f.n_gen, 1);
#else
            slot = f.n_gen++;
#endif
            Blit b;
            double r[4] = {f.col_x[ci], f.row_y[cj], f.cell_w, f.cell_w};
            make_sprite_blit(c, f, b, r, 0, false, type, theme, 1.0f);
            if (b.kind == BLIT_NONE)
                continue;
            *f.gen_blit(slot) = b;
            f.cellmap[k] = (uint16_t)(CELL_GENERAL | slot);
        }
    }

    // ---- phase C1a: arena space and a staging job for every tile the frame registered
    static PG_HD void frame_tile_alloc(Ctx &c, Frame &f, const TileTable &tt, int tid, int nthreads) {
        if (!G::DRAWS_GRID)
            return;
        for (int key = tid; key < CELL_KEYS; key += nthreads) {
            if (f.tilekey[key] != 1)
                continue;
            const int type = key >> 2;
            const int tw = f.tile_w0 + (key & 1), th = f.tile_h0 + ((key >> 1) & 1);
            const int img_type = G::image_for_type(c, type);
            const int theme = G::theme_for_grid_obj(c, type);
            const int masked_theme = (c.h->options.restrict_themes && !G::should_preserve_type_themes(c, img_type)) ? 0 : theme;
            const int slot = tt.texels ? c.assets->sprite_slot[img_type + masked_theme * MAX_ASSETS] : -1;
            uint16_t code = 0xffffu;
            if (slot >= 0) {
                const int words = tile_words(tw, th);
                int off, job;
#if defined(__CUDA_ARCH__)
                off = atomicAdd(&f.tile_top, words);
#else
                off = f.tile_top;
                f.tile_top += words;
#endif
                if (off + words <= Frame::kArenaWords) {
#if defined(__CUDA_ARCH__)
                    job = atomicAdd(&f.n_tjobs, 1);
#else
                    job = f.n_tjobs++;
#endif
                    if (job < MAX_TILE_JOBS) {
                        f.tjob[job].src = tt.index[(slot * MAX_TILE_DIM + (tw - 1)) * MAX_TILE_DIM + (th - 1)];
                        f.tjob[job].dst = (uint16_t)off;
                        f.tjob[job].words = (uint16_t)words;
                        code = (uint16_t)(2 + off);
                    }
                }
            }
            f.tilekey[key] = code;
        }
    }

    // ---- phase C1d: cells, pass B — tile cells learn where their tile was put; tiles that found
    // no room (or have no table entry) fall back to a general blit
    static PG_HD void frame_cells_finish(Ctx &c, Frame &f, int tid, int nthreads) {
        if (!G::DRAWS_GRID)
            return;
        const int ncells = f.nx * f.ny;
        for (int k = tid; k < ncells; k += nthreads) {
            const uint16_t code = f.cellmap[k];
            if ((code & 0xC000u) != 0x4000u)
                continue;
            const int key = code & 0x3fff;
            const uint16_t tk = f.tilekey[key];
            if (tk != 0xffffu) {
                f.cellmap[k] = (uint16_t)(tk - 1);  // 1 + arena texel offset
                continue;
            }
            f.cellmap[k] = 0;
            int slot;
#if defined(__CUDA_ARCH__)
            slot = atomicAdd(&f.n_gen, 1);
#else
            slot = f.n_gen++;
#endif
            const int ci = k / f.ny, cj = k - ci * f.ny;
            const int type = key >> 2;
            Blit b;
            double r[4] = {f.col_x[ci], f.row_y[cj], f.cell_w, f.cell_w};
            make_sprite_blit(c, f, b, r, 0, false, type, G::theme_for_grid_obj(c, type), 1.0f);
            if (b.kind == BLIT_NONE)
                continue;
            *f.gen_blit(slot) = b;
            f.cellmap[k] = (uint16_t)(CELL_GENERAL | slot);
        }
    }

    // ---- phase C1b (device): the tiles reserved by build_entity_blits, one tile per thread
    static PG_HD void frame_tiles(Ctx &c, Frame &f, int tid, int nthreads) {
        const int nj = f.n_jobs < Frame::kMaxTileJobs ? f.n_jobs : Frame::kMaxTileJobs;
        for (int job = 0; job < nj; job++) {
            const int ei = f.job_ei[job], pos = f.job_pos[job], nt = f.job_n[job], j0 = f.job_j0[job];
            for (int j = tid; j < nt; j += nthreads) entity_tile_blit(c, f, ei, j0 + j, f.ents[pos + j]);
        }
    }

    // ---- phase C1c (device): rotated sprites whose slots build_entity_blits reserved
    static PG_HD void frame_rots(Ctx &c, Frame &f, int tid, int nthreads) {
        const int n = f.n_ent;
        for (int i = tid; i < n; i += nthreads) {
            if (f.ents[i].kind != BLIT_ROT_PENDING)
                continue;
            const int ei = (int)f.ents[i].src;
            const Entity &o = c.ents[ei];
            double r[4];
            object_rect(f.cam, o, r);
            Blit nb;
            make_sprite_blit(c, f, nb, r, o.rotation, o.is_reflected != 0, o.image_type, o.image_theme, o.alpha);
            f.ents[i] = nb;
        }
    }

    // the overlay blits (drawn after everything else) join the end of the entity list; one thread
    static PG_HD void frame_append_overlays(Frame &f) {
        for (int i = 0; i < f.n_overlay; i++) f.ents[f.n_ent + i] = f.overlay[i];
    }

    static PG_HD int ctz64(uint64_t m) {
#if defined(__CUDA_ARCH__)
        return __ffsll((long long)m) - 1;
#else
        return __builtin_ctzll(m);
#endif
    }
    static PG_HD int top_bit64(uint64_t m) {  // m != 0
#if defined(__CUDA_ARCH__)
        return 63 - __clzll((long long)m);
#else
        return 63 - __builtin_clzll(m);
#endif
    }

    static PG_HD int ctz32(uint32_t m) {  // m != 0
#if defined(__CUDA_ARCH__)
        return __ffs((int)m) - 1;
#else
        return __builtin_ctz(m);
#endif
    }

    // ---- phase D: composition. Colours are 0xFFRRGGBB (Format_RGB32).
    //   gather   per pixel: the grid cells over the background (draw_background + the cell loop of
    //            draw_foreground, basic-abstract-game.cpp:921-1007) — the cell under a pixel is a table
    //            lookup, and an opaque tile texel makes the background fetch unnecessary
    //   paint    entity blits and overlays in draw order onto the frame (draw_entities z = 0, 1 and
    //            game_draw overrides): every blit's pixels are spread over the lanes that own its rows
    // Rows are owned by warps (row y belongs to warp y % 4) in both phases, so a warp-level barrier
    // is all that separates them; the host debug harness runs the same functions with one "lane".

    // source value of cell (ci, cj) at a pixel; `code` = cellmap entry (non-zero)
    static PG_HD uint32_t cell_layer(const Frame &f, uint32_t code, int ci, int cj, int px, int py, const uint32_t *atlas) {
        if (code & CELL_GENERAL)
            return blit_texel(*f.gen_blit((int)(code & 0x7fffu)), px, py, atlas, f.rot);
        const int dx = px - f.col_p1[ci] + f.col_k0[ci], dy = py - f.row_p1[cj] + f.row_k0[cj];
        return f.arena[(int)code - 1 + dy * f.col_tw[ci] + dx];
    }

    static PG_HD uint32_t bg_single(uint32_t bgrow, uint32_t bgcol, const uint32_t *atlas) {
        return (bgrow != BG_NONE && bgcol != BG_NONE) ? atlas[bgrow + bgcol] : 0xff000000u;  // fillRect(rect, black), basic-abstract-game.cpp:980
    }
    // draw_background at one pixel, any number of background blits (tiled backgrounds), bottom-up
    static PG_HD_NOINLINE uint32_t bg_generic(const Frame &f, int px, int py, const uint32_t *atlas) {
        uint32_t dst = 0xff000000u;
        if (f.pad == 1)
            return bg_single(f.bgrow[py], f.bgcol[px], atlas);
        for (int i = 0; i < f.n_bg; i++) dst = layer_over(dst, blit_texel(f.bg[i], px, py, atlas, f.rot));
        return dst;
    }

    // all cells over `under` at one pixel, in draw order (x outer / y inner), found by their spans: the
    // fallback for pixels more than two cell columns (rows) cover
    static PG_HD uint32_t cells_over(const Frame &f, int px, int py, const uint32_t *atlas, uint32_t under) {
        uint32_t dst = under;
        const int clo = f.col_lo[px], chi = f.col_hi[px], rlo = f.row_lo[py], rhi = f.row_hi[py];
        if (clo != 255 && rlo != 255) {
            for (int ci = clo; ci <= chi; ci++)
                for (int cj = rlo; cj <= rhi; cj++) {
                    const uint32_t code = f.cellmap[ci * f.ny + cj];
                    if (code && px >= f.col_p1[ci] && px < f.col_p2[ci] && py >= f.row_p1[cj] && py < f.row_p2[cj])
                        dst = layer_over(dst, cell_layer(f, code, ci, cj, px, py, atlas));
                }
        }
        return dst;
    }
    static PG_HD_NOINLINE uint32_t cells_generic(const Frame &f, int px, int py, const uint32_t *atlas, uint32_t under) {
        return cells_over(f, px, py, atlas, under);
    }

    // source value at a pixel of the cell that column word `cw` and row word `rw` (CI_* words) point at
    static PG_HD uint32_t cell_texel(const Frame &f, uint32_t cw, uint32_t rw, int px, int py, const uint32_t *atlas) {
        const uint32_t code = f.cellmap[(cw & CI_BASE_MASK) + (rw & CI_BASE_MASK)];
        if (code == 0)
            return 0;
        if (code & CELL_GENERAL) {
            const Blit &gb = *f.gen_blit((int)(code & 0x7fffu));
            if (gb.kind == BLIT_SOLID) {  // solid-colour cells (chaser's orbs, monochrome mode) are a box test
                const uint32_t box = *reinterpret_cast<const uint32_t *>(&gb);
                const uint32_t ddx = (uint32_t)px - (box & 0xffu), ddy = (uint32_t)py - ((box >> 8) & 0xffu);
                return (ddx < ((box >> 16) & 0xffu) && ddy < (box >> 24)) ? gb.src : 0u;
            }
            return blit_texel(gb, px, py, atlas, f.rot);  // other kinds take the long way
        }
        return f.arena[code - 1 + ((rw >> CI_D_SHIFT) & 31u) * ((cw >> CI_TW_SHIFT) & 31u) + ((cw >> CI_D_SHIFT) & 31u)];
    }

    // The pixels off the one-tile-cell path: a one-pixel overlap strip of two cell columns and / or rows
    // (up to 2 x 2 cells, blended in draw order: column lo, hi outer, row lo, hi inner) or a cell that is
    // a general blit. `ci` / `ri` are the pixel's column / row words.
    static PG_HD uint32_t cells_odd(const Frame &f, uint32_t ci, uint32_t ri, int px, int py, const uint32_t *atlas, uint32_t under) {
        if ((ci | ri) & CI_WIDE)
            return cells_generic(f, px, py, atlas, under);
        const uint32_t cl = (ci & CI_MULTI) ? f.colinfo_lo[px] : ci;
        const uint32_t rl = (ri & CI_MULTI) ? f.rowinfo_lo[py] : ri;
        uint32_t dst = under;
        if (ci & CI_MULTI) {
            if (ri & CI_MULTI)
                dst = layer_over(dst, cell_texel(f, cl, rl, px, py, atlas));
            dst = layer_over(dst, cell_texel(f, cl, ri, px, py, atlas));
        }
        if (ri & CI_MULTI)
            dst = layer_over(dst, cell_texel(f, ci, rl, px, py, atlas));
        return layer_over(dst, cell_texel(f, ci, ri, px, py, atlas));
    }

    enum GatherMode { GATHER_ALL = 0, GATHER_BG = 1, GATHER_CELLS = 2 };  // background + cells | background only | cells over what fb holds

    // Four horizontally adjacent pixels of row py -> fb. The common pixel — at most one cell and that one
    // from a pre-scaled tile — is one cellmap and one arena load; the four pixels then fetch what lies
    // under them (the background, or what fb holds) in one pass, only where the texel is not opaque.
    // Strip pixels and general-blit cells (`odd`) get cells_odd over that afterwards. `bgc` = the
    // background source columns of the four pixels (pad == 1).
    template <int MODE>
    static PG_HD void gather_quad(const Frame &f, const uint32_t *bgc, bool bg_one, int px0, int py, const uint32_t *atlas, uint32_t *fb) {
        constexpr bool kCells = G::DRAWS_GRID && MODE != GATHER_BG;
        uint32_t *dst = fb + py * RES_W + px0;
        uint32_t ci[4] = {0u, 0u, 0u, 0u}, s[4] = {0u, 0u, 0u, 0u};
        uint32_t odd = 0;
        const uint32_t rowinfo = kCells ? f.rowinfo[py] : 0u;
        if (kCells && (rowinfo & CI_VALID)) {  // a cell row covers the pixel row
#if defined(__CUDA_ARCH__)
            const uint4 cv = *reinterpret_cast<const uint4 *>(f.colinfo + px0);
            ci[0] = cv.x; ci[1] = cv.y; ci[2] = cv.z; ci[3] = cv.w;
#else
            for (int k = 0; k < 4; k++) ci[k] = f.colinfo[px0 + k];
#endif
            const uint32_t rbase = rowinfo & CI_BASE_MASK, dy = (rowinfo >> CI_D_SHIFT) & 31u;
            for (int k = 0; k < 4; k++) {
                const uint32_t both = ci[k] & rowinfo;
                if (both & CI_FAST) {  // one cell column and one cell row cover the pixel
                    const uint32_t code = f.cellmap[(ci[k] & CI_BASE_MASK) + rbase];
                    if (code & CELL_GENERAL) {
                        // solid-colour cells (half of chaser's pixels) are a box test; other kinds are odd
                        const Blit &gb = *f.gen_blit((int)(code & 0x7fffu));
                        if (gb.kind == BLIT_SOLID) {
                            const uint32_t box = *reinterpret_cast<const uint32_t *>(&gb);
                            const uint32_t ddx = (uint32_t)(px0 + k) - (box & 0xffu), ddy = (uint32_t)py - ((box >> 8) & 0xffu);
                            s[k] = (ddx < ((box >> 16) & 0xffu) && ddy < (box >> 24)) ? gb.src : 0u;
                        } else {
                            odd |= 1u << k;
                        }
                    } else if (code)
                        s[k] = f.arena[code - 1 + dy * ((ci[k] >> CI_TW_SHIFT) & 31u) + ((ci[k] >> CI_D_SHIFT) & 31u)];
                } else if (both & CI_VALID) {
                    odd |= 1u << k;
                }
            }
        }
        const uint32_t bgrow = bg_one ? f.bgrow[py] : BG_NONE;
        uint32_t c[4];
        for (int k = 0; k < 4; k++) {
            c[k] = s[k];
            if (s[k] >= 0xff000000u)
                continue;  // opaque tile texel (odd pixels have s = 0)
            uint32_t under;
            if (MODE == GATHER_CELLS)
                under = dst[k];
            else if (bg_one)
                under = bg_single(bgrow, bgc[k], atlas);
            else
                under = bg_generic(f, px0 + k, py, atlas);
            c[k] = s[k] != 0 ? s[k] + pg_byte_mul(under, (~s[k]) >> 24) : under;  // odd pixels: under
        }
#if defined(__CUDA_ARCH__)
        *reinterpret_cast<uint4 *>(dst) = make_uint4(c[0], c[1], c[2], c[3]);
#else
        for (int k = 0; k < 4; k++) dst[k] = c[k];
#endif
        // the odd pixels' cells over what was just stored there (one copy of that code, not four)
        while (kCells && odd != 0) {
            const int k = ctz32(odd);
            odd &= odd - 1;
            dst[k] = cells_odd(f, f.colinfo[px0 + k], rowinfo, px0 + k, py, atlas, dst[k]);
        }
    }

    // Paint blits [lo, hi) of the entity list, in list order, onto the rows row_first, row_first +
    // row_step, ... of fb. The `nlanes` threads that share those rows split every blit's pixels.
    static PG_HD void paint_blits(const Frame &f, uint32_t *fb, int lo, int hi, int row_first, int row_step, int lane, int nlanes, const uint32_t *atlas) {
        for (int i = lo; i < hi; i++) {
            const Blit &b = f.ents[i];
            const uint32_t box = *reinterpret_cast<const uint32_t *>(&b);  // x1 | y1<<8 | w<<16 | h<<24
            const int x1 = (int)(box & 0xffu), y1 = (int)((box >> 8) & 0xffu), w = (int)((box >> 16) & 0xffu), h = (int)(box >> 24);
            if (w == 0)
                continue;
            int r0 = (row_first - y1) % row_step;  // first row of the box that is ours
            if (r0 < 0)
                r0 += row_step;
            const int nrows = r0 < h ? (h - 1 - r0) / row_step + 1 : 0;
            const int n = nrows * w;
            const bool plain = b.kind == BLIT_IMAGE;
            for (int idx = lane; idx < n; idx += nlanes) {
                const int r = idx / w, dx = idx - r * w, dy = r0 + r * row_step;
                uint32_t s;
                if (plain) {
                    uint32_t sx = (b.basex + (uint32_t)b.ix * (uint32_t)dx) >> 16;
                    const uint32_t sy = (b.srcy + (uint32_t)b.iy * (uint32_t)dy) >> 16;
                    if (b.mirror)
                        sx = b.sw - 1 - sx;
                    s = layer_of(atlas[b.src + sy * b.sw + sx], b.opacity);
                } else {
                    s = blit_texel(b, x1 + dx, y1 + dy, atlas, f.rot);
                }
                if (s != 0) {
                    uint32_t *px = fb + (y1 + dy) * RES_W + x1 + dx;
                    *px = layer_over(*px, s);
                }
            }
#if defined(__CUDA_ARCH__)
            __syncwarp();  // the next blit may overlap this one
#endif
        }
    }

    // 0xFFRRGGBB x 4 -> 12 packed RGB bytes (3 words): bgr32_to_rgb888 (game.cpp:8-23)
    static PG_HD void pack_quad(const uint32_t *c, uint32_t *out) {
#if defined(__CUDA_ARCH__)
        out[0] = __byte_perm(c[0], c[1], 0x6012);
        out[1] = __byte_perm(c[1], c[2], 0x5601);
        out[2] = __byte_perm(c[2], c[3], 0x4560);
#else
        const uint32_t r0 = (c[0] >> 16) & 0xff, g0 = (c[0] >> 8) & 0xff, b0 = c[0] & 0xff;
        const uint32_t r1 = (c[1] >> 16) & 0xff, g1 = (c[1] >> 8) & 0xff, b1 = c[1] & 0xff;
        const uint32_t r2 = (c[2] >> 16) & 0xff, g2 = (c[2] >> 8) & 0xff, b2 = c[2] & 0xff;
        const uint32_t r3 = (c[3] >> 16) & 0xff, g3 = (c[3] >> 8) & 0xff, b3 = c[3] & 0xff;
        out[0] = r0 | (g0 << 8) | (b0 << 16) | (r1 << 24);
        out[1] = g1 | (b1 << 8) | (r2 << 16) | (g2 << 24);
        out[2] = b2 | (r3 << 8) | (g3 << 16) | (b3 << 24);
#endif
    }

    // Everything the owner of rows row_first, row_first + row_step, ... does to them: `lane` of
    // `nlanes` threads (a warp on the device; 16 quad columns x 2 interleaved row sets per lane pair)
    template <int MODE>
    static PG_HD void gather_rows(const Frame &f, uint32_t *fb, int row_first, int row_step, int lane, int nlanes, const uint32_t *atlas) {
        // lanes tile the rows: quad column = lane % 16, and lane / 16 picks every (nlanes / 16)-th of our rows
        const int per_row = RES_W / 4;
        const int sub = nlanes >= per_row ? nlanes / per_row : 1;
        const bool bg_one = f.pad == 1;
        for (int qx = lane % per_row; qx < per_row; qx += (nlanes < per_row ? nlanes : per_row)) {
            uint32_t bgc[4];
            for (int k = 0; k < 4; k++) bgc[k] = f.bgcol[qx * 4 + k];
            const int first = row_first + row_step * (nlanes >= per_row ? lane / per_row : 0);
            for (int py = first; py < RES_H; py += row_step * sub) gather_quad<MODE>(f, bgc, bg_one, qx * 4, py, atlas, fb);
        }
    }
    // `dbg` (profiling variant, PG_PHASE_TIMING): the first row owner's SM cycles in gather ([0]) and paint ([1])
    static PG_HD void compose_rows(const Frame &f, uint32_t *fb, int row_first, int row_step, int lane, int nlanes, const uint32_t *atlas,
                                   uint32_t *dbg = nullptr) {
        const int nb = f.n_ent_below, n_all = f.n_ent + f.n_overlay;
#if defined(PG_PHASE_TIMING) && defined(__CUDA_ARCH__)
        const long long t0 = clock64();
#endif
        if (G::ENTS_BELOW_GRID && nb > 0) {
            gather_rows<GATHER_BG>(f, fb, row_first, row_step, lane, nlanes, atlas);
#if defined(__CUDA_ARCH__)
            __syncwarp();
#endif
            paint_blits(f, fb, 0, nb, row_first, row_step, lane, nlanes, atlas);
#if defined(__CUDA_ARCH__)
            __syncwarp();
#endif
            gather_rows<GATHER_CELLS>(f, fb, row_first, row_step, lane, nlanes, atlas);
        } else {
            gather_rows<GATHER_ALL>(f, fb, row_first, row_step, lane, nlanes, atlas);
        }
#if defined(__CUDA_ARCH__)
        __syncwarp();
#endif
#if defined(PG_PHASE_TIMING) && defined(__CUDA_ARCH__)
        const long long t1 = clock64();
#endif
        paint_blits(f, fb, (G::ENTS_BELOW_GRID ? nb : 0), n_all, row_first, row_step, lane, nlanes, atlas);
#if defined(PG_PHASE_TIMING) && defined(__CUDA_ARCH__)
        __syncwarp();
        if (dbg && row_first == 0 && lane == 0) {
            dbg[0] = (uint32_t)(t1 - t0);
            dbg[1] = (uint32_t)(clock64() - t1);
        }
#else
        (void)dbg;
#endif
    }
};

// ---- default draw hooks that need Frame (kept out of Defaults<G> to avoid a circular include)
template <class G>
struct DrawDefaults {
    // draw_background's single scaled bg image (basic-abstract-game.cpp:986-1006)
    template <class Frame>
    static PG_HD void make_background_blits(Ctx &c, Frame &f) {
        EnvHdr &h = *c.h;
        double main_rect[4];
        Raster<G, Frame>::screen_rect(f.cam, 0, (float)h.main_height, (float)h.main_width, (float)h.main_height, 0, main_rect);
        SpriteDesc bg = c.assets->backgrounds[h.background_index];
        if (h.bg_tile_ratio < 0) {
            // tile_image(p, background, main_rect, bg_tile_ratio), basic-abstract-game.cpp:990-991
            const int nt = Raster<G, Frame>::tile_count(main_rect, h.bg_tile_ratio);
            int n = 0;
            for (int i = 0; i < nt; i++) {
                double tr[4];
                Raster<G, Frame>::tile_rect(main_rect, h.bg_tile_ratio, nt, i, tr);
                Blit b;
                make_image_blit(b, tr[0], tr[1], tr[2], tr[3], bg, false, 256, f.snap != 0);
                if (b.kind == BLIT_NONE)
                    continue;  // tile entirely off screen
                if (n < MAX_BG_BLITS)
                    f.bg[n++] = b;
                else
                    h.err |= ERR_BLIT_OVERFLOW;
            }
            f.n_bg = n;
            return;
        }
        float bgw = bg.w;
        float bgh = bg.h;
        float bg_ar = bgw / bgh;
        float world_ar = (float)(h.main_width * 1.0 / h.main_height);
        float extra_w = bg_ar - world_ar;
        float offset_x = h.bg_pct_x * extra_w;
        double adj[4] = {(double)(-offset_x), 0, (double)(bg_ar / world_ar), 1};
        Raster<G, Frame>::adjust_rect(main_rect, adj);
        make_image_blit(f.bg[0], main_rect[0], main_rect[1], main_rect[2], main_rect[3], bg, false, 256, f.snap != 0);
        f.n_bg = 1;
    }
    // game_draw overrides that paint after draw_foreground: append at f.overlay[f.n_overlay...]
    template <class Frame>
    static PG_HD void make_overlay_blits(Ctx &c, Frame &f) {}
    // draw_grid_obj (basic-abstract-game.cpp:915-919): a fillRect in color_for_type's colour
    // (:455-481) — defined only in monochrome mode; false = the reference would fassert
    template <class Frame>
    static PG_HD bool make_grid_obj_blit(Ctx &c, const Frame &f, Blit &b, double *rect, int type, int theme) {
        if (!c.h->options.use_monochrome_assets)
            return false;
        if (c.h->options.restrict_themes && !G::should_preserve_type_themes(c, type))
            theme = 0;
        const int k = 4;
        const int kcubed = k * k * k;
        const int chunk = 256 / k;
        if (type >= kcubed)
            return false;
        int new_type = (29 * (type + 1)) % kcubed;
        new_type = (new_type + 19 * theme) % kcubed;
        const uint32_t r = (uint32_t)(chunk * (new_type / (k * k) + 1) - 1);
        const uint32_t g = (uint32_t)(chunk * ((new_type / k) % k + 1) - 1);
        const uint32_t bl = (uint32_t)(chunk * (new_type % k + 1) - 1);
        make_solid_blit(b, rect[0], rect[1], rect[2], rect[3], (r << 16) | (g << 8) | bl);
        return true;
    }
};

}  // namespace pg
