/*
 * ORACLE -- test infrastructure, NOT product code.
 *
 * Scalar CPU rasteriser that *defines* the correct palette-index framebuffer for a compiled
 * scene ("B2DS" blob, see oracle/scene.py) and a camera pose.  Only tests/, __graft_entry__.smoke()
 * and bench.py's cpu_baseline / --impl reference legs may build, load or call this file.
 *
 * Parity status: UNPINNED.  The reference (cristicbz/rust-doom) has no CPU implementation of
 * this path -- visibility and raster happen inside the OpenGL driver (engine/src/renderer.rs:
 * 49-57,99-157) -- and no golden frames or fixtures (SURVEY.md 4, 8c).  What this file restates
 * from the reference is the *data semantics* that decide each pixel:
 *   - BSP side rule, near child first           wad/src/visitor.rs:1051-1057, math/src/line.rs:41-43
 *   - which wall pieces exist + pegging          wad/src/visitor.rs:711-937 (pre-resolved by the scene
 *                                                compiler into texA/tA/hA, texB/tB/hB, otop/obot)
 *   - wall texel  tex[(s mod w) + (t mod h)*w]   assets/shaders/static.frag:19-22 (floor-mod)
 *   - flat texel  flat[(wad_y mod 64) + 64*(wad_x mod 64)]   game/src/level.rs:537-549
 *                 at the map position eye + z(row) * dir(column)
 *   - colormap row = clamp(floor((1-light)*32),0,31), light = 2*b/255 - (1 - 0.9/(w+0.9)),
 *     w = view depth / 100                       assets/shaders/static.vert:41-43, static.frag:15-27,
 *                                                wad/src/tex.rs:137-166
 *   - sky: u = ndc.x - 4*yaw/pi, v = 1 - ndc.y, mirrored below the horizon, colormap row 0
 *                                                assets/shaders/sky.vert:9-16, sky.frag:12-26
 *   - projection fovy 65deg, aspect*1.2, near .01 (= 1 map unit)
 *                                                game/src/player.rs:84-89, engine/src/projections.rs:93-101
 *   - masked two-sided middles, decoration sprites (billboards), level time (animated flats / walls, scrolling
 *     walls, sector light effects): DESIGN.md C12-C15 with their reference citations
 * The visibility algorithm itself (front-to-back BSP walk with per-column clip windows, Doom
 * style) is new; it is written here column by column, the way a CPU Doom renderer draws (per-column
 * set-up once, a tight row loop per wall piece; the plane constants of a screen row memoised per plane).
 * All arithmetic is integer (DESIGN.md "pixel contract"); the CUDA path must reproduce every bit.
 * It doubles as bench.py's CPU baseline, so it is compiled for the host it runs on.
 *
 * Build: gcc -O3 -march=native -fopenmp -shared -fPIC (see oracle/build.py).
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

typedef struct { int32_t x, y, z; uint32_t angle; } b2o_pose;       /* 16.16 map units, BAM */
typedef struct { int32_t W, H, F, FY2; } b2o_view;                  /* F = round(2*focal_x) px */

enum { H_MAGIC, H_VERSION, H_TOTAL, H_NVERTS, H_NNODES, H_NSSECTORS, H_NSEGS, H_NSECTORS, H_NTEX,
       H_NFLATS, H_OFF_VERTS, H_OFF_NODES, H_OFF_SSECTORS, H_OFF_SEGS, H_OFF_SECTORS, H_OFF_TEX,
       H_OFF_TEXELS, H_TEXEL_BYTES, H_OFF_FLATS, H_OFF_COLORMAP, H_OFF_PALETTE, H_ROOT, H_SKY_TEX,
       H_NMIDS = 30, H_OFF_MIDS = 31, H_NSPRITES = 32, H_OFF_SPRITES = 33, H_NANIM = 34, H_OFF_ANIM = 35,
       H_OFF_FLAT_ANIM = 36 };

#define LEAF 0x80000000u
#define SEG_TWO_SIDED 1
#define SEG_SCROLL 2
#define SEG_INVALID 0x80
#define FLAT_SKY (-1)

typedef struct {
    const uint32_t *hdr;
    const int32_t *verts, *nodes, *ssectors, *segs, *sectors, *mids, *sprites, *anim, *flat_anim;
    const uint32_t *tex;
    const uint8_t *texels, *flats, *colormap;
    const uint32_t *palette;
    int nverts, nnodes, nss, nsegs, nsectors, ntex, nflats, sky_tex, nmids, nsprites, nanim;
} Scene;

static int scene_bind(Scene *s, const uint8_t *blob) {
    const uint32_t *h = (const uint32_t *)blob;
    if (h[H_MAGIC] != 0x53443242u || h[H_VERSION] != 6) return -1;
    s->hdr = h;
    s->verts = (const int32_t *)(blob + h[H_OFF_VERTS]);
    s->nodes = (const int32_t *)(blob + h[H_OFF_NODES]);
    s->ssectors = (const int32_t *)(blob + h[H_OFF_SSECTORS]);
    s->segs = (const int32_t *)(blob + h[H_OFF_SEGS]);
    s->sectors = (const int32_t *)(blob + h[H_OFF_SECTORS]);
    s->tex = (const uint32_t *)(blob + h[H_OFF_TEX]);
    s->mids = (const int32_t *)(blob + h[H_OFF_MIDS]);
    s->nmids = (int)h[H_NMIDS];
    s->sprites = (const int32_t *)(blob + h[H_OFF_SPRITES]);
    s->nsprites = (int)h[H_NSPRITES];
    s->anim = (const int32_t *)(blob + h[H_OFF_ANIM]);
    s->nanim = (int)h[H_NANIM];
    s->flat_anim = (const int32_t *)(blob + h[H_OFF_FLAT_ANIM]);
    s->texels = blob + h[H_OFF_TEXELS];
    s->flats = blob + h[H_OFF_FLATS];
    s->colormap = blob + h[H_OFF_COLORMAP];
    s->palette = (const uint32_t *)(blob + h[H_OFF_PALETTE]);
    s->nverts = (int)h[H_NVERTS]; s->nnodes = (int)h[H_NNODES]; s->nss = (int)h[H_NSSECTORS];
    s->nsegs = (int)h[H_NSEGS]; s->nsectors = (int)h[H_NSECTORS]; s->ntex = (int)h[H_NTEX];
    s->nflats = (int)h[H_NFLATS]; s->sky_tex = (int32_t)h[H_SKY_TEX];
    return 0;
}

/* ---------------------------------------------------------------- integer helpers ------------ */
static inline int64_t asr64(int64_t v, int s) {            /* arithmetic shift = floor(v / 2^s) */
    return v >= 0 ? (v >> s) : -(((-v) + (((int64_t)1 << s) - 1)) >> s);
}
static inline int64_t floordiv64(int64_t a, int64_t b) {   /* b > 0 */
    int64_t q = a / b;
    if ((a % b) != 0 && (a < 0)) q -= 1;
    return q;
}
static inline int32_t floormod32(int32_t a, int32_t b) {   /* b > 0 */
    int32_t r = a % b;
    return r < 0 ? r + b : r;
}
static inline int bitlen64(uint64_t v) { int n = 0; while (v) { n++; v >>= 1; } return n; }
static inline int64_t clamp64(int64_t v, int64_t lo, int64_t hi) { return v < lo ? lo : (v > hi ? hi : v); }
static inline int32_t clamp32(int32_t v, int32_t lo, int32_t hi) { return v < lo ? lo : (v > hi ? hi : v); }

/* sin/cos of a BAM angle in Q30.  Pure integer Taylor series on [0, pi/4] (DESIGN.md C1). */
#define Q30 ((int64_t)1 << 30)
void b2o_sincos_q30(uint32_t angle, int32_t *cos_out, int32_t *sin_out) {
    uint32_t quad = angle >> 30;
    uint32_t r = angle & 0x3FFFFFFFu;          /* fraction of a quarter turn, /2^30 */
    int swap = 0;
    if (r > 0x20000000u) { r = 0x40000000u - r; swap = 1; }
    int64_t x = ((int64_t)r * 1686629713LL) >> 30;   /* round(pi/2 * 2^30) */
    int64_t x2 = (x * x) >> 30;
    int64_t t;
    /* sin x = x (1 - x2/6 (1 - x2/20 (1 - x2/42 (1 - x2/72)))) */
    t = Q30 - x2 / 72;
    t = Q30 - ((x2 * t) >> 30) / 42;
    t = Q30 - ((x2 * t) >> 30) / 20;
    t = Q30 - ((x2 * t) >> 30) / 6;
    int64_t s = (x * t) >> 30;
    /* cos x = 1 - x2/2 (1 - x2/12 (1 - x2/30 (1 - x2/56 (1 - x2/90)))) */
    t = Q30 - x2 / 90;
    t = Q30 - ((x2 * t) >> 30) / 56;
    t = Q30 - ((x2 * t) >> 30) / 30;
    t = Q30 - ((x2 * t) >> 30) / 12;
    int64_t c = Q30 - ((x2 * t) >> 30) / 2;
    if (swap) { int64_t tmp = s; s = c; c = tmp; }
    int64_t cc, ss;
    switch (quad) {
        case 0: cc = c; ss = s; break;
        case 1: cc = -s; ss = c; break;
        case 2: cc = -c; ss = -s; break;
        default: cc = s; ss = -c; break;
    }
    *cos_out = (int32_t)cc; *sin_out = (int32_t)ss;
}

/* colormap row from the light byte b and view depth z8 (1/8 map units, <= 65535):
 * row = clamp(floor(64(255-b)/255 - 2880/(z+90)), 0, 31)   (static.frag:15-27 with w = z/100) */
static inline int light_row(int b, int32_t z8) {
    int64_t Z = (int64_t)z8 + 720;
    int64_t num = (int64_t)64 * (255 - b) * Z - 5875200;
    if (num <= 0) return 0;
    int64_t r = num / (255 * Z);
    return r > 31 ? 31 : (int)r;
}

/* ---------------------------------------------------------------- per-frame state ------------ */
/* one screen column of a masked two-sided middle texture, with the clip window that was open behind the
 * seg when the front-to-back pass reached it (Doom's drawseg silhouette, per column) */
struct Masked { int owner, x, ya, yb, row; int32_t tex, tA, hA, iscale, ucol; };

typedef struct {
    const Scene *sc;
    b2o_view vw;
    b2o_pose pose;
    uint32_t tics;            /* level time in 1/35 s (DESIGN.md C14) */
    const int16_t *light_ov;  /* per sector: light byte at `tics` of a sector with a light effect, -1 = static (C15) */
    int32_t cosq, sinq;       /* Q30 */
    int32_t *tx, *tz;         /* view-space vertices, Q8 */
    int32_t *ctop, *cbot;     /* open window per column: rows [ctop, cbot) */
    uint32_t *yslope;         /* floor(FY2*65536 / |2y+1-H|) */
    int open_cols;
    uint32_t invF;            /* floor(2^32 / F) */
    uint8_t *fb;
    int32_t *seg_hits;        /* optional: pixels drawn per seg (may be NULL) */
    int cur_seg;
    struct Masked *masked;    /* masked middle-texture columns met during the solid pass, front to back */
    int n_masked, cap_masked;
    /* per screen row: the plane constants of the last (height, light) drawn on that row.  Columns of one seg are drawn
     * one after the other and share their floor / ceiling plane, so the 64-bit set-up runs once per row per plane, not
     * once per pixel (same values: this is a memo, not a different formula). */
    int64_t *prow_key;        /* (h << 9 | lightb) + 1, 0 = empty */
    uint32_t *prow;           /* 2 words per row: view depth Q8, 256 * light row */
} Frame;

static inline void put(Frame *f, int x, int y, uint8_t v) {
    f->fb[(size_t)y * f->vw.W + x] = v;
    if (f->seg_hits && f->cur_seg >= 0) f->seg_hits[f->cur_seg]++;       /* sprites have no seg */
}

/* Animated textures and flats (static.vert:23-39, ANIM_FPS = 8/35 s per frame): every frame name of an n-frame group
 * is bound to the atlas position of the group's FIRST frame (wad/src/tex.rs:260 `positions[i - entry.frame_offset]`,
 * tex.rs:302-306 `anim_start_pos`), so whichever frame name a wall or flat uses, it shows group frame
 * floor(tics/8) mod n -- frame 0 at tic 0.  anim_nk = n | k << 16 (k is informational); 0 = not animated. */
static inline int32_t anim_now(const Scene *sc, int32_t first, uint32_t nk, uint32_t tics, int32_t self) {
    uint32_t n = nk & 0xFFFF;
    if (n < 2 || first < 0 || (int64_t)first + n > sc->nanim) return self;
    return sc->anim[first + (int32_t)((tics >> 3) % n)];
}
static inline int32_t tex_now(const Frame *f, int32_t tex) {
    const Scene *sc = f->sc;
    if (tex < 0 || tex >= sc->ntex) return tex;
    const uint32_t *T = sc->tex + 8 * tex;
    return anim_now(sc, (int32_t)T[6], T[7], f->tics, tex);
}
static inline int32_t flat_now(const Frame *f, int32_t flat) {
    const Scene *sc = f->sc;
    if (flat < 0 || flat >= sc->nflats) return flat;
    return anim_now(sc, sc->flat_anim[2 * flat], (uint32_t)sc->flat_anim[2 * flat + 1], f->tics, flat);
}

/* light byte of something lit by `sector`: the effect's value at the frame's time, else the static byte */
static inline int lit(const Frame *f, int32_t sector, int32_t static_byte) {
    if (f->light_ov && sector >= 0 && sector < f->sc->nsectors && f->light_ov[sector] >= 0) return f->light_ov[sector];
    return static_byte;
}

static void draw_sky(Frame *f, int x, int ya, int yb) {
    const Scene *sc = f->sc;
    if (ya >= yb || sc->sky_tex < 0) return;
    const uint32_t *T = sc->tex + 8 * sc->sky_tex;
    int32_t w = (int32_t)T[1], h = (int32_t)T[2];
    const uint8_t *px = sc->texels + T[0];
    int W = f->vw.W, H = f->vw.H;
    int64_t c2 = 2 * (int64_t)x + 1 - W;
    uint32_t u32 = (uint32_t)(uint64_t)floordiv64(c2 * 4294967296LL, W) - (f->pose.angle << 3);
    int32_t col = (int32_t)(((uint64_t)u32 * (uint32_t)w) >> 32);
    for (int y = ya; y < yb; y++) {
        int32_t r = 2 * y + 1, v;
        if (r < H) v = (r * h) / H;
        else v = floormod32(((2 * H - r) * h) / H, h);
        put(f, x, y, sc->colormap[px[v * w + col]]);          /* colormap row 0 */
    }
}

/* floor(n * invF / 2^40), exact: n * invF itself exceeds 64 bits on low, wide views (W/F > ~31), so the product is
 * taken in two halves, n = hi * 2^20 + lo with 0 <= lo < 2^20 */
static inline int32_t mul_invF_q40(int64_t n, uint32_t invF) {
    const int64_t hi = asr64(n, 20), lo = n - hi * ((int64_t)1 << 20);
    return (int32_t)asr64(hi * (int64_t)invF + asr64(lo * (int64_t)invF, 20), 20);
}

/* direction of column x's ray, Q18 (DESIGN.md C8): (cos*F + sin*c2)/F, (sin*F - cos*c2)/F with c2 = 2x+1-W */
static inline void plane_dir(int32_t cosq, int32_t sinq, const b2o_view *vw, uint32_t invF, int x, int32_t *ax, int32_t *ay) {
    const int64_t c2 = 2 * (int64_t)x + 1 - vw->W;
    const int64_t nx = asr64((int64_t)cosq * vw->F + (int64_t)sinq * c2, 4);
    const int64_t ny = asr64((int64_t)sinq * vw->F - (int64_t)cosq * c2, 4);
    *ax = mul_invF_q40(nx, invF);
    *ay = mul_invF_q40(ny, invF);
}

static void draw_plane(Frame *f, int x, int ya, int yb, int32_t h, int32_t flat, int lightb) {
    const Scene *sc = f->sc;
    if (ya >= yb) return;
    if (flat == FLAT_SKY) { draw_sky(f, x, ya, yb); return; }
    flat = flat_now(f, flat);
    if (flat < 0 || flat >= sc->nflats) return;               /* missing flat: pixels stay void */
    const uint8_t *px = sc->flats + 4096 * (size_t)flat;
    int64_t hrel = clamp64(((int64_t)h << 16) - f->pose.z, -((int64_t)1 << 27), (int64_t)1 << 27);
    uint64_t a = (uint64_t)(hrel < 0 ? -hrel : hrel);
    const int64_t key = (((int64_t)h << 9) | (int64_t)(lightb & 0x1FF)) + 1;
    int32_t dx, dy;
    plane_dir(f->cosq, f->sinq, &f->vw, f->invF, x, &dx, &dy);
    const uint32_t ax = (uint32_t)dx, ay = (uint32_t)dy;
    const uint32_t bu = (uint32_t)f->pose.x << 10, bv = (uint32_t)f->pose.y << 10;
    for (int y = ya; y < yb; y++) {
        uint32_t *pr = f->prow + 2 * (size_t)y;
        if (f->prow_key[y] != key) {
            uint64_t zz = (a * f->yslope[y]) >> 16;
            int32_t z16 = zz > 0x7FFFFFFFull ? 0x7FFFFFFF : (int32_t)zz;
            pr[0] = (uint32_t)(z16 >> 8);                         /* view depth of the row on this plane, Q8 */
            int32_t z8 = z16 >> 13; if (z8 > 65535) z8 = 65535;
            pr[1] = 256u * (uint32_t)light_row(lightb, z8);
            f->prow_key[y] = key;
        }
        uint32_t U = bu + pr[0] * ax;                             /* wad x, Q26 mod 64 */
        uint32_t V = bv + pr[0] * ay;                             /* wad y */
        uint8_t texel = px[((U >> 26) << 6) | (V >> 26)];
        put(f, x, y, sc->colormap[pr[1] + texel]);
    }
}

static void draw_wall(Frame *f, int x, int ya, int yb, int32_t tex, int32_t tA, int32_t hA,
                      int32_t ucol, int32_t iscale, int row) {
    const Scene *sc = f->sc;
    tex = tex_now(f, tex);
    if (ya >= yb || tex < 0 || tex >= sc->ntex) return;       /* untextured: pixels stay void */
    const uint32_t *T = sc->tex + 8 * tex;
    int32_t w = (int32_t)T[1], h = (int32_t)T[2];
    const uint8_t *px = sc->texels + T[0];
    int32_t col = floormod32(ucol, w);
    int64_t hrel = clamp64(((int64_t)hA << 16) - f->pose.z, -((int64_t)1 << 27), (int64_t)1 << 27);
    int64_t tbase = ((int64_t)tA << 16) + hrel + asr64((int64_t)(1 - f->vw.H) * iscale, 5);
    int32_t tstep = iscale >> 4;
    const uint8_t *cm = sc->colormap + 256 * row;
    px += col;
    if ((h & (h - 1)) == 0) {                                 /* power-of-two height: floor-mod is a mask */
        const int32_t hm = h - 1;
        for (int y = ya; y < yb; y++) {
            int32_t t = (int32_t)(tbase + (int64_t)y * tstep);
            put(f, x, y, cm[px[((t >> 16) & hm) * w]]);
        }
    } else {
        for (int y = ya; y < yb; y++) {
            int32_t t = (int32_t)(tbase + (int64_t)y * tstep);
            int32_t v = floormod32((int32_t)asr64(t, 16), h);
            put(f, x, y, cm[px[v * w]]);
        }
    }
}

/* first row whose centre lies at or below the projected height h: ceil(Y - 0.5), Y in Q26 */
static inline int yrow(const Frame *f, int32_t h, int32_t scale) {
    int64_t hrel8 = ((int64_t)h << 8) - asr64(f->pose.z, 8);
    int64_t Y = ((int64_t)f->vw.H << 25) - hrel8 * scale;
    int64_t r = asr64(Y + ((int64_t)1 << 25) - 1, 26);
    return (int)clamp64(r, 0, f->vw.H);
}

static void constrain(int64_t *lo, int64_t *hi, int64_t a, int64_t b, int64_t c) {
    /* a + b*x >= c */
    if (b > 0) { int64_t v = -floordiv64(-(c - a), b); if (v > *lo) *lo = v; }       /* ceil */
    else if (b < 0) { int64_t v = floordiv64(a - c, -b); if (v < *hi) *hi = v; }
    else if (a < c) { *hi = *lo - 1; }
}

static void draw_seg(Frame *f, int si) {
    const Scene *sc = f->sc;
    const int32_t *S = sc->segs + 16 * si;
    if (S[3] & SEG_INVALID) return;
    f->cur_seg = si;
    const int W = f->vw.W, H = f->vw.H;
    const int64_t F = f->vw.F, FY2 = f->vw.FY2;
    int64_t ax = f->tx[S[0]], az = f->tz[S[0]], bx = f->tx[S[1]], bz = f->tz[S[1]];
    int64_t dxs = bx - ax, dzs = bz - az;
    int64_t C = az * dxs - ax * dzs;
    if (C <= 0) return;                                       /* back-facing or degenerate */
    int64_t Nx = 2 * az, Nc = az * (1 - W) - ax * F;          /* N(x) = az*c2 - ax*F */
    int64_t Dx = -2 * dzs, Dc = dxs * F - dzs * (1 - W);      /* D(x) = dxs*F - dzs*c2 */
    int64_t lo = 0, hi = W - 1;
    constrain(&lo, &hi, Dc, Dx, 1);                           /* D > 0 */
    constrain(&lo, &hi, Nc, Nx, 0);                           /* N >= 0 */
    constrain(&lo, &hi, Dc - Nc, Dx - Nx, 0);                 /* N <= D */
    if (lo > hi) return;
    int64_t Dbound = (dxs < 0 ? -dxs : dxs) * F + (dzs < 0 ? -dzs : dzs) * W;
    int sh = bitlen64((uint64_t)Dbound) - 31; if (sh < 0) sh = 0;
    int64_t M = F * C;
    int shm = bitlen64((uint64_t)M) - 31;
    uint64_t Mn = shm >= 0 ? ((uint64_t)M >> shm) : ((uint64_t)M << (-shm));
    uint64_t Rm = ((uint64_t)1 << 62) / Mn; if (Rm > 0xFFFFFFFFull) Rm = 0xFFFFFFFFull;
    int e = 5 - sh + shm;
    int64_t Dmax = M >> 8;                                    /* z >= 1 map unit */
    int64_t scale_cap = FY2 << 17;

    const int32_t *SF = sc->sectors + 8 * S[2];
    int32_t fc = SF[1], ff = SF[0];
    int two = S[3] & SEG_TWO_SIDED;
    int32_t otop = S[13], obot = S[14];
    int ceil_vis = ((int64_t)fc << 16) > f->pose.z || SF[3] == FLAT_SKY;
    int floor_vis = ((int64_t)ff << 16) < f->pose.z || SF[2] == FLAT_SKY;

    for (int x = (int)lo; x <= (int)hi; x++) {
        int ct = f->ctop[x], cb = f->cbot[x];
        if (ct >= cb) continue;
        int64_t N = Nc + Nx * x, D = Dc + Dx * x;
        int64_t Dt = D >> sh;
        if (Dt < 1) continue;
        int64_t Nn = N >> sh;
        uint32_t s24 = (uint32_t)(((uint64_t)Nn << 24) / (uint64_t)Dt);
        int64_t Dcl = D < Dmax ? D : Dmax;
        uint64_t Dn = (uint64_t)(Dcl >> sh);
        if (Dn < 1) continue;
        uint64_t P = (Dn * Rm) >> 32;
        uint64_t prod = (uint64_t)FY2 * P;
        int64_t scale;
        if (e >= 0) scale = e > 63 ? 0 : (int64_t)(prod >> e);
        else scale = (-e) >= 20 ? scale_cap : (int64_t)(prod << (-e));
        if (scale > scale_cap) scale = scale_cap;
        if (scale < 1) continue;
        int64_t isc = ((int64_t)1 << 38) / scale;
        int32_t iscale = (int32_t)clamp64(isc, 1, 1 << 23);
        int64_t z8l = ((int64_t)iscale * FY2) >> 18;
        int32_t z8 = z8l > 65535 ? 65535 : (int32_t)z8l;
        int row = light_row(lit(f, S[2], S[12]), z8);
        /* scrolling walls (visitor.rs:922, 35 px/s = 1 px per tic): the texture column advances with time */
        int32_t ucol = S[4] + (int32_t)(((uint64_t)s24 * (uint32_t)S[5]) >> 36)
                     + ((S[3] & SEG_SCROLL) ? (int32_t)(f->tics & 0xFFFFFF) : 0);

        int yfc = yrow(f, fc, (int32_t)scale), yff = yrow(f, ff, (int32_t)scale);
        if (!two) {
            int y1 = clamp32(yfc, ct, cb);
            int y2 = clamp32(yff, y1, cb);
            if (ceil_vis) draw_plane(f, x, ct, y1, fc, SF[3], lit(f, S[2], SF[4]));
            draw_wall(f, x, y1, y2, S[6], S[7], S[8], ucol, iscale, row);
            if (floor_vis) draw_plane(f, x, y2, cb, ff, SF[2], lit(f, S[2], SF[4]));
            f->ctop[x] = H; f->cbot[x] = 0; f->open_cols--;
        } else {
            int yot = yrow(f, otop, (int32_t)scale), yob = yrow(f, obot, (int32_t)scale);
            int y1 = clamp32(yfc, ct, cb);
            int y2 = clamp32(yot, y1, cb);
            int y3 = clamp32(yob, y2, cb);
            int y4 = clamp32(yff, y3, cb);
            if (ceil_vis) draw_plane(f, x, ct, y1, fc, SF[3], lit(f, S[2], SF[4]));
            if (otop < fc) draw_wall(f, x, y1, y2, S[6], S[7], S[8], ucol, iscale, row);
            if (obot > ff) draw_wall(f, x, y3, y4, S[9], S[10], S[11], ucol, iscale, row);
            if (floor_vis) draw_plane(f, x, y4, cb, ff, SF[2], lit(f, S[2], SF[4]));
            if (y2 >= y3) { f->ctop[x] = H; f->cbot[x] = 0; f->open_cols--; }
            else {
                f->ctop[x] = y2; f->cbot[x] = y3;
                if (S[15] >= 0 && S[15] < sc->nmids) {       /* masked middle: drawn after the solid pass */
                    if (f->n_masked == f->cap_masked) {
                        f->cap_masked = f->cap_masked ? 2 * f->cap_masked : 1024;
                        f->masked = (struct Masked *)realloc(f->masked, (size_t)f->cap_masked * sizeof *f->masked);
                    }
                    const int32_t *M = sc->mids + 8 * S[15];
                    int mya = yrow(f, M[3], (int32_t)scale), myb = yrow(f, M[2], (int32_t)scale);
                    struct Masked *m = &f->masked[f->n_masked++];
                    m->owner = si; m->x = x; m->row = row;
                    m->ya = mya > y2 ? mya : y2; m->yb = myb < y3 ? myb : y3;
                    m->tex = M[0]; m->tA = M[1]; m->hA = M[3]; m->iscale = iscale; m->ucol = ucol;
                }
            }
        }
    }
}

/* back-to-front pass over the recorded masked columns: texture rows [yrow(high), yrow(low)) clipped to the
 * recorded window; transparent texels (opacity plane 0) leave the pixel untouched (static.frag:21-22) */
static void draw_masked(Frame *f) {
    const Scene *sc = f->sc;
    for (int i = f->n_masked - 1; i >= 0; i--) {
        const struct Masked *m = &f->masked[i];
        const int32_t mtex = m->owner >= 0 ? tex_now(f, m->tex) : m->tex;
        if (mtex < 0 || mtex >= sc->ntex || m->ya >= m->yb) continue;
        const uint32_t *T = sc->tex + 8 * mtex;
        int32_t w = (int32_t)T[1], h = (int32_t)T[2];
        const uint8_t *px = sc->texels + T[0];
        const uint8_t *opaque = T[5] != 0xFFFFFFFFu ? sc->texels + T[5] : NULL;
        f->cur_seg = m->owner;
        int32_t col = floormod32(m->ucol, w);
        int64_t hrel = clamp64(((int64_t)m->hA << 16) - f->pose.z, -((int64_t)1 << 27), (int64_t)1 << 27);
        int64_t tbase = ((int64_t)m->tA << 16) + hrel + asr64((int64_t)(1 - f->vw.H) * m->iscale, 5);
        int32_t tstep = m->iscale >> 4;
        const uint8_t *cm = sc->colormap + 256 * m->row;
        for (int y = m->ya; y < m->yb; y++) {
            int32_t t = (int32_t)(tbase + (int64_t)y * tstep);
            int32_t v = floormod32((int32_t)asr64(t, 16), h);
            if (opaque && !opaque[v * w + col]) continue;
            put(f, m->x, y, cm[px[v * w + col]]);
        }
    }
}

/* sprite light (assets/shaders/sprite.frag:15-27): light = min(v, 2v - dist), dist = 1 - 1/(w+1), w = z/100:
 * row = clamp(max(floor(32(255-b)/255), floor(64(255-b)/255 - 3200/(z+100))), 0, 31) */
static inline int light_row_sprite(int b, int32_t z8) {
    int64_t r1 = (32 * (int64_t)(255 - b)) / 255;
    int64_t Z = (int64_t)z8 + 800;
    int64_t num = (int64_t)64 * (255 - b) * Z - 6528000;
    int64_t r2 = num <= 0 ? 0 : num / (255 * Z);
    int64_t r = r1 > r2 ? r1 : r2;
    return r > 31 ? 31 : (int)r;
}

/* A decoration thing (visitor.rs:1062-1137, sprite.vert:40-42): camera-facing billboard of its sprite image's
 * size, at constant view depth.  Recorded when the front-to-back walk enters the thing's subsector, with the
 * clip windows open at that moment; drawn with the masked pass. */
static void record_sprite(Frame *f, int idx) {
    const Scene *sc = f->sc;
    const int32_t *SP = sc->sprites + 8 * idx;
    if (SP[3] < 0 || SP[3] >= sc->ntex) return;
    const uint32_t *T = sc->tex + 8 * SP[3];
    const int32_t w = (int32_t)T[1], h = (int32_t)T[2];
    const int W = f->vw.W;
    const int64_t F = f->vw.F, FY2 = f->vw.FY2;
    int64_t px8 = asr64(f->pose.x, 8), py8 = asr64(f->pose.y, 8);
    int64_t dx = ((int64_t)SP[0] << 8) - px8, dy = ((int64_t)SP[1] << 8) - py8;
    int64_t cx = asr64(dx * f->sinq - dy * f->cosq, 30), cz = asr64(dx * f->cosq + dy * f->sinq, 30);
    if (cz < 256) return;                                         /* nearer than 1 map unit / behind */
    int64_t L = (cx - (int64_t)w * 128) * F, R = (cx + (int64_t)w * 128) * F;
    int64_t lo = 0, hi = W - 1;
    constrain(&lo, &hi, cz * (1 - W) - L, 2 * cz, 0);            /* cz*c2 >= L */
    constrain(&lo, &hi, R - 1 - cz * (1 - W), -2 * cz, 0);       /* cz*c2 <= R-1 */
    if (lo > hi) return;
    int64_t scale = (FY2 << 25) / cz;
    if (scale > (FY2 << 17)) scale = FY2 << 17;
    if (scale < 1) return;
    int32_t iscale = (int32_t)clamp64(((int64_t)1 << 38) / scale, 1, 1 << 23);
    int64_t z8l = ((int64_t)iscale * FY2) >> 18;
    int32_t z8 = z8l > 65535 ? 65535 : (int32_t)z8l;
    int row = light_row_sprite(lit(f, SP[5], SP[4]), z8);
    int ys_a = yrow(f, SP[2] + h, (int32_t)scale), ys_b = yrow(f, SP[2], (int32_t)scale);
    for (int x = (int)lo; x <= (int)hi; x++) {
        int ct = f->ctop[x], cb = f->cbot[x];
        if (ct >= cb) continue;
        int ya = ys_a > ct ? ys_a : ct, yb = ys_b < cb ? ys_b : cb;
        if (ya >= yb) continue;
        int64_t c2 = 2 * (int64_t)x + 1 - W;
        int64_t u = floordiv64(cz * c2 - L, 256 * F);
        if (f->n_masked == f->cap_masked) {
            f->cap_masked = f->cap_masked ? 2 * f->cap_masked : 1024;
            f->masked = (struct Masked *)realloc(f->masked, (size_t)f->cap_masked * sizeof *f->masked);
        }
        struct Masked *m = &f->masked[f->n_masked++];
        m->owner = -1; m->x = x; m->ya = ya; m->yb = yb; m->row = row;
        m->tex = SP[3]; m->tA = 0; m->hA = SP[2] + h; m->iscale = iscale;
        m->ucol = (int32_t)clamp64(u, 0, w - 1);
    }
}

static void walk(Frame *f, uint32_t child, int depth) {
    const Scene *sc = f->sc;
    if (f->open_cols <= 0 || depth > 4096) return;
    if (child & LEAF) {
        uint32_t id = child & 0x7FFFFFFFu;
        if ((int)id >= sc->nss) return;
        const int32_t *ss = sc->ssectors + 4 * id;
        if (ss[2] < 0) return;
        {   /* decoration things of this subsector: in front of its far segs, behind everything drawn so far; among
             * themselves nearest first (they are drawn back to front, so the nearer billboard ends up on top, as a depth
             * test would have it: sprite.vert:40-42 puts a billboard at one view depth); ties keep the stored order */
            int first = ss[3] & 0xFFFFFF, cnt = (ss[3] >> 24) & 0xFF;
            if (first + cnt > sc->nsprites) cnt = sc->nsprites > first ? sc->nsprites - first : 0;
            int64_t cz[256];
            int order[256];
            for (int i = 0; i < cnt; i++) {
                const int32_t *SP = sc->sprites + 8 * (first + i);
                int64_t dx = ((int64_t)SP[0] << 8) - asr64(f->pose.x, 8), dy = ((int64_t)SP[1] << 8) - asr64(f->pose.y, 8);
                cz[i] = asr64(dx * f->cosq + dy * f->sinq, 30);
                int k = i;
                while (k > 0 && cz[order[k - 1]] > cz[i]) { order[k] = order[k - 1]; k--; }     /* stable insertion sort */
                order[k] = i;
            }
            for (int i = 0; i < cnt; i++) record_sprite(f, first + order[i]);
        }
        for (int i = 0; i < ss[1]; i++) draw_seg(f, ss[0] + i);
        return;
    }
    if ((int)child >= sc->nnodes) return;
    const int32_t *n = sc->nodes + 16 * child;
    /* (py-oy)*dx - (px-ox)*dy > 0  =>  left child is the near side */
    int64_t sd = ((int64_t)f->pose.y - ((int64_t)n[1] << 16)) * n[2]
               - ((int64_t)f->pose.x - ((int64_t)n[0] << 16)) * n[3];
    int side = sd > 0 ? 1 : 0;
    walk(f, (uint32_t)n[12 + side], depth + 1);
    walk(f, (uint32_t)n[12 + (side ^ 1)], depth + 1);
}

static void render_frame(const Scene *sc, const b2o_view *vw, const b2o_pose *pose, uint32_t tics,
                         const int16_t *light_ov, uint8_t *fb, int32_t *scratch, int32_t *seg_hits) {
    Frame f;
    f.tics = tics; f.light_ov = light_ov;
    f.sc = sc; f.vw = *vw; f.pose = *pose; f.fb = fb; f.seg_hits = seg_hits; f.cur_seg = 0;
    const int W = vw->W, H = vw->H;
    f.tx = scratch; f.tz = f.tx + sc->nverts;
    f.ctop = f.tz + sc->nverts; f.cbot = f.ctop + W;
    f.yslope = (uint32_t *)(f.cbot + W);
    f.prow = f.yslope + H;
    f.prow_key = (int64_t *)(((uintptr_t)(f.prow + 2 * (size_t)H) + 7) & ~(uintptr_t)7);
    memset(f.prow_key, 0, sizeof(int64_t) * (size_t)H);
    b2o_sincos_q30(pose->angle, &f.cosq, &f.sinq);
    f.invF = (uint32_t)(4294967296ULL / (uint64_t)vw->F);
    memset(fb, 0, (size_t)W * H);                              /* void index = 0 */
    int64_t px8 = asr64(pose->x, 8), py8 = asr64(pose->y, 8);
    for (int i = 0; i < sc->nverts; i++) {
        int64_t dx = ((int64_t)sc->verts[2 * i] << 8) - px8;
        int64_t dy = ((int64_t)sc->verts[2 * i + 1] << 8) - py8;
        f.tx[i] = (int32_t)asr64(dx * f.sinq - dy * f.cosq, 30);
        f.tz[i] = (int32_t)asr64(dx * f.cosq + dy * f.sinq, 30);
    }
    for (int x = 0; x < W; x++) { f.ctop[x] = 0; f.cbot[x] = H; }
    for (int y = 0; y < H; y++) {
        int32_t r2 = 2 * y + 1 - H; if (r2 < 0) r2 = -r2; if (r2 == 0) r2 = 1;
        f.yslope[y] = (uint32_t)(((uint64_t)vw->FY2 << 16) / (uint32_t)r2);
    }
    f.open_cols = W;
    f.masked = NULL; f.n_masked = 0; f.cap_masked = 0;
    walk(&f, sc->hdr[H_ROOT], 0);
    draw_masked(&f);
    free(f.masked);
}

/* ---------------------------------------------------------------- public entry points -------- */
void b2o_view_init(b2o_view *v, int W, int H, double tan_half_fovy) {
    /* perspective(fovy, aspect = (W/H)*1.2): focal_y = (H/2)/tan, focal_x = (H/2)/(1.2*tan) */
    double fy2 = (double)H / tan_half_fovy;
    double fx2 = (double)H / (1.2 * tan_half_fovy);
    v->W = W; v->H = H;
    v->FY2 = (int32_t)(fy2 + 0.5);
    v->F = (int32_t)(fx2 + 0.5);
}

/* direction of every column's ray at yaw `angle`, Q18, as draw_plane uses it (DESIGN.md C8): out[2x] = ax, out[2x+1] = ay */
void b2o_plane_dirs(const b2o_view *vw, uint32_t angle, int32_t *out) {
    int32_t c, s;
    b2o_sincos_q30(angle, &c, &s);
    for (int x = 0; x < vw->W; x++) plane_dir(c, s, vw, (uint32_t)(4294967296ULL / (uint64_t)vw->F), x, &out[2 * x], &out[2 * x + 1]);
}

/* light_ov: NULL, or one int16 per sector (oracle/scene.py sector_lights_at(blob, tics)) */
int b2o_render_t(const uint8_t *scene_blob, const b2o_view *vw, const b2o_pose *poses, int n, uint32_t tics,
                 const int16_t *light_ov, uint8_t *index_fb, uint32_t *rgba_fb, int32_t *seg_hits, int nthreads) {
    Scene sc;
    if (scene_bind(&sc, scene_blob) != 0) return -1;
    if (vw->W < 1 || vw->H < 1 || vw->W > 4096 || vw->H > 2160 || vw->F < 2 || vw->FY2 < 2) return -2;
    const size_t npix = (size_t)vw->W * vw->H;
    const size_t scratch_ints = 2 * (size_t)sc.nverts + 2 * (size_t)vw->W + (size_t)vw->H + 16
                              + 5 * (size_t)vw->H + 2 * (size_t)vw->H + 4;      /* + plane-row memo (5 words + one int64 per row) */
    int err = 0;
    if (nthreads < 1) nthreads = 1;
#pragma omp parallel num_threads(nthreads)
    {
        int32_t *scratch = (int32_t *)malloc(scratch_ints * sizeof(int32_t));
        if (!scratch) {
#pragma omp atomic write
            err = -3;
        } else {
#pragma omp for schedule(dynamic, 1)
            for (int i = 0; i < n; i++) {
                uint8_t *fb = index_fb + npix * (size_t)i;
                render_frame(&sc, vw, &poses[i], tics, light_ov, fb, scratch,
                             seg_hits ? seg_hits + (size_t)sc.nsegs * i : NULL);
                if (rgba_fb) {
                    uint32_t *out = rgba_fb + npix * (size_t)i;
                    for (size_t p = 0; p < npix; p++) out[p] = sc.palette[fb[p]];
                }
            }
            free(scratch);
        }
    }
    return err;
}

int b2o_render(const uint8_t *scene_blob, const b2o_view *vw, const b2o_pose *poses, int n,
               uint8_t *index_fb, uint32_t *rgba_fb, int32_t *seg_hits, int nthreads) {
    return b2o_render_t(scene_blob, vw, poses, n, 0, NULL, index_fb, rgba_fb, seg_hits, nthreads);
}

/* CRC-32 (IEEE, reflected) of a byte range: golden-vector digest for frames */
uint32_t b2o_crc32(const uint8_t *p, size_t n) {
    static uint32_t table[256]; static int init = 0;
    if (!init) {
        for (uint32_t i = 0; i < 256; i++) {
            uint32_t c = i;
            for (int k = 0; k < 8; k++) c = (c & 1) ? 0xEDB88320u ^ (c >> 1) : (c >> 1);
            table[i] = c;
        }
        init = 1;
    }
    uint32_t c = 0xFFFFFFFFu;
    for (size_t i = 0; i < n; i++) c = table[(c ^ p[i]) & 0xFF] ^ (c >> 8);
    return c ^ 0xFFFFFFFFu;
}
