// Integer pixel-contract arithmetic shared by the CUDA kernels (DESIGN.md "Pixel contract").
//
// Every function is exact integer math so that the palette-index framebuffer is reproducible bit
// for bit.  The functions are __host__ __device__ so that tests/hostcheck can run the very same
// code on the CPU (one lane at a time) and compare it with the oracle before any GPU time is spent;
// the shipped library contains no CPU rendering path.
//
// Reference semantics restated here (cristicbz/rust-doom):
//   BSP side rule                      math/src/line.rs:41-43, wad/src/visitor.rs:1051-1057
//   wall texel floor-mod sampling      assets/shaders/static.frag:19-22
//   flat texel rule                    game/src/level.rs:537-549
//   light -> colormap row              assets/shaders/static.vert:41-43, static.frag:15-27
//   sky lookup                         assets/shaders/sky.vert:9-16, sky.frag:12-26
//   projection constants               game/src/player.rs:84-89, engine/src/projections.rs:93-101
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define B2D_HD __host__ __device__ __forceinline__
#else
#define B2D_HD inline
#endif

namespace b2d {

struct Pose { int32_t x, y, z; uint32_t angle; };     // == b2d_pose
struct View { int32_t W, H, F, FY2; };                // == b2d_view

// Per-frame constants produced by the BSP-walk kernel and consumed by the raster kernel.
struct FrameConst {
    Pose pose;
    int32_t cosq, sinq;        // Q30
    int32_t px8, py8;          // camera position, Q8
    int32_t count;             // worklist length
    int32_t status;            // 0 ok, 1 = traversal stack overflow
    int32_t pad[6];
};
static_assert(sizeof(FrameConst) == 64, "FrameConst");

// One worklist entry: a front-facing seg that may be visible, with its per-frame projection
// coefficients.  N(x) = Nc + Nx*x and D(x) = Dc + Dx*x are the numerator / denominator of the
// seg parameter s = N/D at screen column x; 1/depth is proportional to D.
struct SegFrame {
    int64_t Nc, Nx, Dc, Dx;
    int64_t Dmax;              // D clamp: depth >= 1 map unit
    uint32_t Rm;               // floor(2^62 / normalised(F*C))
    int16_t sh, e;             // normalisation shift of N,D; scale exponent
    int32_t seg;
    int16_t xlo, xhi;          // exact visible column interval
    int32_t flags;             // bit0: every column in [xlo,xhi] passes column_eval
    int32_t pad;
};
static_assert(sizeof(SegFrame) == 64, "SegFrame");

constexpr int32_t kSegFrameNoSkip = 1;

// ------------------------------------------------------------------------------------------------
B2D_HD int bitlen64(uint64_t v) {
#if defined(__CUDA_ARCH__)
    return 64 - __clzll((long long)v);
#else
    return v ? 64 - __builtin_clzll(v) : 0;
#endif
}
B2D_HD int64_t floordiv64(int64_t a, int64_t b) {      // b > 0
    int64_t q = a / b;
    return (a % b != 0 && a < 0) ? q - 1 : q;
}
B2D_HD int32_t floormod32(int32_t a, int32_t b) {      // b > 0
    int32_t r = a % b;
    return r < 0 ? r + b : r;
}
template <typename T> B2D_HD T clampv(T v, T lo, T hi) { return v < lo ? lo : (v > hi ? hi : v); }
B2D_HD uint32_t umulhi32(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
    return __umulhi(a, b);
#else
    return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}

// sin/cos of a BAM angle, Q30, integer Taylor series on [0, pi/4] with octant folding.
B2D_HD void sincos_q30(uint32_t angle, int32_t &cosq, int32_t &sinq) {
    const int64_t one = (int64_t)1 << 30;
    uint32_t quad = angle >> 30;
    uint32_t r = angle & 0x3FFFFFFFu;
    bool swap = false;
    if (r > 0x20000000u) { r = 0x40000000u - r; swap = true; }
    int64_t x = ((int64_t)r * 1686629713LL) >> 30;
    int64_t x2 = (x * x) >> 30;
    int64_t t = one - x2 / 72;
    t = one - ((x2 * t) >> 30) / 42;
    t = one - ((x2 * t) >> 30) / 20;
    t = one - ((x2 * t) >> 30) / 6;
    int64_t s = (x * t) >> 30;
    t = one - x2 / 90;
    t = one - ((x2 * t) >> 30) / 56;
    t = one - ((x2 * t) >> 30) / 30;
    t = one - ((x2 * t) >> 30) / 12;
    int64_t c = one - ((x2 * t) >> 30) / 2;
    if (swap) { int64_t tmp = s; s = c; c = tmp; }
    int64_t cc, ss;
    if (quad == 0) { cc = c; ss = s; }
    else if (quad == 1) { cc = -s; ss = c; }
    else if (quad == 2) { cc = -c; ss = -s; }
    else { cc = s; ss = -c; }
    cosq = (int32_t)cc; sinq = (int32_t)ss;
}

B2D_HD void frame_setup(const Pose &p, FrameConst &f) {
    f.pose = p;
    sincos_q30(p.angle, f.cosq, f.sinq);
    f.px8 = p.x >> 8;
    f.py8 = p.y >> 8;
    f.count = 0;
    f.status = 0;
}

// world (map units) -> view space Q8: tx to the right, tz forward.
B2D_HD void to_view(const FrameConst &f, int32_t wx, int32_t wy, int32_t &tx, int32_t &tz) {
    int64_t dx = ((int64_t)wx << 8) - f.px8;
    int64_t dy = ((int64_t)wy << 8) - f.py8;
    tx = (int32_t)((dx * f.sinq - dy * f.cosq) >> 30);
    tz = (int32_t)((dx * f.cosq + dy * f.sinq) >> 30);
}

// BSP side: 1 = left child is on the camera's side (sd > 0), 0 = right child.
B2D_HD int node_side(const Pose &p, int32_t nx, int32_t ny, int32_t ndx, int32_t ndy) {
    int64_t sd = ((int64_t)p.y - ((int64_t)ny << 16)) * ndx - ((int64_t)p.x - ((int64_t)nx << 16)) * ndy;
    return sd > 0 ? 1 : 0;
}

// a + b*x >= c over integer x, intersected into [lo, hi]
B2D_HD void constrain(int64_t &lo, int64_t &hi, int64_t a, int64_t b, int64_t c) {
    if (b > 0) { int64_t v = -floordiv64(-(c - a), b); if (v > lo) lo = v; }
    else if (b < 0) { int64_t v = floordiv64(a - c, -b); if (v < hi) hi = v; }
    else if (a < c) { hi = lo - 1; }
}

struct ColumnEval {
    uint32_t s24;      // seg parameter s in Q24
    int32_t scale;     // pixels per map unit, Q18
    int32_t iscale;    // map units per pixel, Q20, clamped to [1, 2^23]
    int32_t z8;        // view depth in 1/8 map units, <= 65535
};

// Per-frame projection setup of one seg from its view-space endpoints.  Returns false if the seg is
// back-facing / degenerate or covers no screen column.
B2D_HD bool seg_frame_setup(const View &vw, int32_t ax_, int32_t az_, int32_t bx_, int32_t bz_, SegFrame &sf,
                            bool want_noskip = true);

// Column predicate + per-column projection values.  Exact: does not rely on xlo/xhi.
B2D_HD bool column_eval(const SegFrame &sf, const View &vw, int x, ColumnEval &out) {
    int64_t N = sf.Nc + sf.Nx * x, D = sf.Dc + sf.Dx * x;
    if (D <= 0 || N < 0 || N > D) return false;
    int64_t Dt = D >> sf.sh;
    if (Dt < 1) return false;
    uint64_t Nn = (uint64_t)(N >> sf.sh);
    out.s24 = (uint32_t)((Nn << 24) / (uint64_t)Dt);
    int64_t Dcl = D < sf.Dmax ? D : sf.Dmax;
    uint64_t Dn = (uint64_t)(Dcl >> sf.sh);
    if (Dn < 1) return false;
    uint64_t P = (Dn * (uint64_t)sf.Rm) >> 32;
    uint64_t prod = (uint64_t)vw.FY2 * P;
    const int64_t cap = (int64_t)vw.FY2 << 17;
    int e = sf.e;
    int64_t scale;
    if (e >= 0) scale = e > 63 ? 0 : (int64_t)(prod >> e);
    else scale = (-e) >= 20 ? cap : (int64_t)(prod << (-e));
    if (scale > cap) scale = cap;
    if (scale < 1) return false;
    out.scale = (int32_t)scale;
    int64_t isc = ((int64_t)1 << 38) / scale;
    out.iscale = (int32_t)clampv<int64_t>(isc, 1, 1 << 23);
    int64_t z8 = ((int64_t)out.iscale * vw.FY2) >> 18;
    out.z8 = z8 > 65535 ? 65535 : (int32_t)z8;
    return true;
}

B2D_HD bool seg_frame_setup(const View &vw, int32_t ax_, int32_t az_, int32_t bx_, int32_t bz_, SegFrame &sf,
                            bool want_noskip) {
    const int64_t ax = ax_, az = az_, bx = bx_, bz = bz_;
    const int64_t F = vw.F, W = vw.W;
    if (az_ <= 0 && bz_ <= 0) return false;       // wholly behind the camera plane: no column can see it
    int64_t dxs = bx - ax, dzs = bz - az;
    int64_t C = az * dxs - ax * dzs;
    if (C <= 0) return false;
    sf.Nx = 2 * az; sf.Nc = az * (1 - W) - ax * F;
    sf.Dx = -2 * dzs; sf.Dc = dxs * F - dzs * (1 - W);
    {   // division-free rejects: a linear function that is negative at both screen edges is negative on
        // the whole screen (exact; the interval solve below would come out empty)
        const int64_t xr = W - 1;
        const int64_t n0 = sf.Nc, n1 = sf.Nc + sf.Nx * xr, d0 = sf.Dc, d1 = sf.Dc + sf.Dx * xr;
        if ((n0 < 0 && n1 < 0) || (d0 < 1 && d1 < 1) || (d0 - n0 < 0 && d1 - n1 < 0)) return false;
    }
    int64_t lo = 0, hi = W - 1;
    constrain(lo, hi, sf.Dc, sf.Dx, 1);
    constrain(lo, hi, sf.Nc, sf.Nx, 0);
    constrain(lo, hi, sf.Dc - sf.Nc, sf.Dx - sf.Nx, 0);
    if (lo > hi) return false;
    sf.xlo = (int16_t)lo; sf.xhi = (int16_t)hi;
    int64_t Dbound = (dxs < 0 ? -dxs : dxs) * F + (dzs < 0 ? -dzs : dzs) * W;
    int sh = bitlen64((uint64_t)Dbound) - 31;
    if (sh < 0) sh = 0;
    int64_t M = F * C;
    int shm = bitlen64((uint64_t)M) - 31;
    uint64_t Mn = shm >= 0 ? ((uint64_t)M >> shm) : ((uint64_t)M << (-shm));
    uint64_t Rm = ((uint64_t)1 << 62) / Mn;
    if (Rm > 0xFFFFFFFFull) Rm = 0xFFFFFFFFull;
    sf.Rm = (uint32_t)Rm;
    sf.sh = (int16_t)sh;
    sf.e = (int16_t)(5 - sh + shm);
    sf.Dmax = M >> 8;
    // no-skip guarantee (only solid segs need it): column_eval's early-outs are monotone in D, so the
    // two endpoints decide for the whole interval
    sf.flags = 0;
    if (want_noskip) {
        ColumnEval ce;
        bool ok = column_eval(sf, vw, (int)lo, ce) && column_eval(sf, vw, (int)hi, ce);
        sf.flags = ok ? kSegFrameNoSkip : 0;
    }
    sf.pad = 0;
    return true;
}

// colormap row from light byte b and depth z8: clamp(floor(64(255-b)/255 - 2880/(z+90)), 0, 31)
B2D_HD int light_row(int b, int32_t z8) {
    uint32_t Z = (uint32_t)z8 + 720u;
    int32_t num = (int32_t)(64u * (uint32_t)(255 - b) * Z) - 5875200;    // < 2^31
    if (num <= 0) return 0;
    uint32_t r = (uint32_t)num / (255u * Z);
    return r > 31u ? 31 : (int)r;
}

// first row whose centre lies at or below the projection of height h (map units): ceil(Y - 1/2)
B2D_HD int yrow(int32_t h, int32_t scale, int32_t pose_z, int32_t H) {
    int64_t hrel8 = ((int64_t)h << 8) - (int64_t)(pose_z >> 8);
    int64_t Y = ((int64_t)H << 25) - hrel8 * scale;
    int64_t r = (Y + ((int64_t)1 << 25) - 1) >> 26;
    return (int)clampv<int64_t>(r, 0, H);
}

B2D_HD uint32_t yslope_entry(int y, const View &vw) {
    int32_t r2 = 2 * y + 1 - vw.H;
    if (r2 < 0) r2 = -r2;
    if (r2 == 0) r2 = 1;
    return (uint32_t)(((uint64_t)vw.FY2 << 16) / (uint32_t)r2);
}

// |h*2^16 - eye_z| clamped to 2048 map units
B2D_HD uint32_t plane_habs(int32_t h, int32_t pose_z) {
    int64_t hrel = clampv<int64_t>(((int64_t)h << 16) - pose_z, -((int64_t)1 << 27), (int64_t)1 << 27);
    return (uint32_t)(hrel < 0 ? -hrel : hrel);
}
B2D_HD int32_t wall_hrel(int32_t h, int32_t pose_z) {
    return (int32_t)clampv<int64_t>(((int64_t)h << 16) - pose_z, -((int64_t)1 << 27), (int64_t)1 << 27);
}

// Texture mapping of a horizontal plane (DESIGN.md C8): the map position under pixel (x, y) is eye + z(y) * dir(x) with
// z the view depth of screen row y on the plane and dir(x) = forward + right * (2x+1-W)/F the direction of column x's ray
// (unit forward component).  Per column (once per frame): dir in Q18.  Per row and plane: z in Q8 and the light row.
// Per pixel: U = (pose.x << 10) + z * dirx, V likewise -- two 32-bit multiply-adds, Q26 modulo 64 texels by wrap-around.
struct PlaneDir { int32_t ax, ay; };                     // Q18
// floor(n * invF / 2^40) without a 128-bit product: n * invF reaches 2^58 * (1 + |c2|/F) and overflows 64 bits once
// W/F > ~31 (low, wide views), so n is split as hi * 2^20 + lo, 0 <= lo < 2^20, and
// floor((hi*invF*2^20 + lo*invF) / 2^40) = (hi*invF + ((lo*invF) >> 20)) >> 20.  |hi*invF| < 2^38 * (1 + W/F) < 2^50
// for every F >= 2; the result is at most 2^18 * (1 + W/F) < 2^30 in magnitude.
B2D_HD int32_t mul_invF_q40(int64_t n, uint32_t invF) {
    const int64_t hi = n >> 20, lo = n & 0xFFFFF;
    return (int32_t)((hi * (int64_t)invF + ((lo * (int64_t)invF) >> 20)) >> 20);
}
B2D_HD PlaneDir plane_dir(const FrameConst &f, const View &vw, int x, uint32_t invF) {
    const int64_t c2 = 2 * (int64_t)x + 1 - vw.W;
    // (cos*F + sin*c2) / F and (sin*F - cos*c2) / F, Q30 -> Q18 through invF = floor(2^32 / F)
    const int64_t nx = ((int64_t)f.cosq * vw.F + (int64_t)f.sinq * c2) >> 4;
    const int64_t ny = ((int64_t)f.sinq * vw.F - (int64_t)f.cosq * c2) >> 4;
    PlaneDir d;
    d.ax = mul_invF_q40(nx, invF);
    d.ay = mul_invF_q40(ny, invF);
    return d;
}
struct PlaneRow { uint32_t z8q; int32_t z8; };           // depth Q8 (for the texel), depth in 1/8 units (for the light row)
B2D_HD PlaneRow plane_row(uint32_t habs, uint32_t yslope) {
    PlaneRow pr;
    uint64_t zz = ((uint64_t)habs * yslope) >> 16;
    int32_t z16 = zz > 0x7FFFFFFFull ? 0x7FFFFFFF : (int32_t)zz;
    pr.z8q = (uint32_t)(z16 >> 8);
    int32_t z8 = z16 >> 13;
    pr.z8 = z8 > 65535 ? 65535 : z8;
    return pr;
}
B2D_HD uint32_t plane_u(int32_t pose_xy, uint32_t z8q, int32_t a) { return ((uint32_t)pose_xy << 10) + z8q * (uint32_t)a; }
B2D_HD uint32_t flat_index(uint32_t U, uint32_t V) { return ((U >> 26) << 6) | (V >> 26); }
// the same index on top of a plane/flat offset given in units of 64 bytes: ((cm6 + (U >> 26)) << 6) | (V >> 26)
B2D_HD uint32_t flat_offset(uint32_t cm6, uint32_t U, uint32_t V) {
#if defined(__CUDA_ARCH__)
    return __funnelshift_l(V, cm6 + (U >> 26), 6);
#else
    return ((cm6 + (U >> 26)) << 6) | (V >> 26);
#endif
}

// wall texture row: t(y) = tbase + y*tstep (Q16); row index = floor-mod of t>>16 by the height,
// evaluated with the per-texture magic reciprocal (exact for |t>>16| < 2^14, h <= 4096).
B2D_HD int32_t wall_tbase(int32_t tA, int32_t hA, int32_t pose_z, int32_t H, int32_t iscale) {
    int64_t t = ((int64_t)tA << 16) + wall_hrel(hA, pose_z) + (((int64_t)(1 - H) * iscale) >> 5);
    return (int32_t)t;
}
B2D_HD uint32_t wall_row(int32_t t, uint32_t h, uint32_t hmagic, uint32_t hbias) {
    uint32_t n = ((uint32_t)t + (hbias << 16)) >> 16;
    uint32_t q = umulhi32(n, hmagic);
    return n - q * h;
}

// ---- pre-lit texel planes (product-side data layout; results are the same bytes as colormap[row][texel]) -------
// Layout of a texture inside a pre-lit plane.  Heights that are a multiple of 4 (every stock wall texture) are
// stored **4 rows interleaved**: texel (row, col) lives at ((row >> 2) * w + col) * 4 + (row & 3), so one aligned
// 32-bit word holds four vertically adjacent texels of a column and the 32 lanes of a warp (adjacent columns) read
// one 128-byte line.  A wall column that is magnified on screen -- the common case at 1080p -- then needs two word
// loads for eight rows instead of eight byte loads.  Other heights keep the blob's row-major layout.
B2D_HD bool tex_interleaved(uint32_t h, uint32_t texel_off) { return (h & 3u) == 0u && (texel_off & 3u) == 0u && h <= 4096u; }
B2D_HD uint32_t lit_index(bool inter, uint32_t w, uint32_t row, uint32_t col) {
    return inter ? ((row >> 2) * w + col) * 4u + (row & 3u) : row * w + col;
}
// Word path of a batch of rows t, t + tstep, ...: `acc` is t with its integer part replaced by (first row & 3);
// pixel k of the batch reads byte (acc + k * tstep) >> 16 of the 8 bytes {row quad r0 >> 2, next row quad}.
B2D_HD uint32_t wall_acc(uint32_t t, uint32_t r0) { return (t & 0xFFFFu) | ((r0 & 3u) << 16); }
B2D_HD uint32_t next_quad(uint32_t q0, uint32_t h) { return q0 + 1u == (h >> 2) ? 0u : q0 + 1u; }
// the byte PRMT selects for a selector below 8 (bytes 0-3 from lo, 4-7 from hi)
B2D_HD uint32_t pick_byte(uint32_t lo, uint32_t hi, uint32_t sel) {
#if defined(__CUDA_ARCH__)
    uint32_t d;                      // raw PRMT: sel < 8, so no sign-replicate bit and no need for __byte_perm's mask
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(lo), "r"(hi), "r"(sel));
    return d;
#else
    return ((sel & 4u) ? hi : lo) >> (8u * (sel & 3u)) & 0xFFu;
#endif
}

// ---- magnified wall columns: incremental row tracking -----------------------------------------------------------
// A column whose texture step is small enough that R consecutive screen rows (and the step to the next batch),
// starting anywhere inside a row quad, stay inside that quad and the next one (R * tstep <= 4 texture rows) needs no
// per-batch floor-mod: the state is the row quad q (0 .. h/4-1) and a Q29 accumulator whose top three bits are the
// byte index inside the 8-byte window {quad q, quad q+1} and whose low 29 bits are the fraction of the texture row.
// Row k of a batch reads byte (acc + k * (tstep << 13)) >> 29 of that window: one IMAD, one shift.  Same rows as
// wall_row(t0 + k*tstep) by construction: (t0 + k*tstep) >> 16 == (t0 >> 16) + (((t0 & 0xFFFF) + k*tstep) >> 16)
// while nothing wraps, and the byte index never exceeds 3 + 4 = 7.
constexpr uint32_t kWallFast8 = 32768u;    // 8 * tstep <= 4 * 65536
constexpr uint32_t kWallFast16 = 16384u;   // 16 * tstep <= 4 * 65536
B2D_HD uint32_t wall_acc29(uint32_t t, uint32_t r0) { return ((r0 & 3u) << 29) | ((t & 0xFFFFu) << 13); }
B2D_HD uint32_t wall_sel(uint32_t acc, uint32_t ts29, uint32_t k) { return (acc + k * ts29) >> 29; }
// after R rows: move the window by whole quads (at most one: the index is <= 7; nq >= 2), keep (row & 3 | fraction)
B2D_HD void wall_advance(uint32_t &acc, uint32_t &q, uint32_t ts29, uint32_t R, uint32_t nq) {
    acc += R * ts29;
    q += acc >> 31;
    if (q >= nq) q -= nq;
    acc &= 0x7FFFFFFFu;
}
// bit k set <=> row y + k lies in [ya, yb), k < R <= 16
B2D_HD uint32_t row_mask(int y, int ya, int yb, int R) {
    int lo = ya - y, hi = yb - y;
    if (lo < 0) lo = 0;
    if (hi > R) hi = R;
    if (hi <= lo) return 0u;
    return ((1u << hi) - 1u) & ~((1u << lo) - 1u);
}

// sky: column from yaw + screen x (one texture width per NDC unit, 8 widths per turn); row mirrored
// below the horizon.
B2D_HD uint32_t sky_u32(int x, const View &vw, uint32_t angle) {
    uint64_t num = ((uint64_t)(2 * x + 1)) << 32;
    return (uint32_t)(num / (uint32_t)vw.W) - (angle << 3);
}
B2D_HD int32_t sky_row(int y, int32_t H, int32_t skyh) {
    int32_t r = 2 * y + 1;
    if (r < H) return (r * skyh) / H;
    return floormod32(((2 * H - r) * skyh) / H, skyh);
}

// Conservative screen-column range of an axis-aligned map box (top, bottom, left, right).
// false => nothing inside the box can be visible.  Boxes that come within 32 map units of the
// camera plane are treated as covering the whole screen.
constexpr int32_t kBoxNearQ8 = 32 * 256;
B2D_HD bool box_range(const FrameConst &f, const View &vw, const int32_t box[4], int &lo, int &hi) {
    bool all_behind = true, any_near = false;
    int64_t mn = 0x7FFFFFFFFFFFFFFFLL, mx = -0x7FFFFFFFFFFFFFFFLL;
    for (int i = 0; i < 4; i++) {
        int32_t tx, tz;
        to_view(f, box[2 + (i & 1)], box[i >> 1], tx, tz);
        if (tz >= -256) all_behind = false;
        if (tz < kBoxNearQ8) { any_near = true; continue; }
        int64_t c = floordiv64((int64_t)tx * vw.F, tz);
        int64_t xc = floordiv64(c - 1 + vw.W, 2);
        if (xc < mn) mn = xc;
        if (xc > mx) mx = xc;
    }
    if (all_behind) return false;
    if (any_near) { lo = 0; hi = vw.W - 1; return true; }
    mn -= 2; mx += 2;
    if (mx < 0 || mn > vw.W - 1) return false;
    lo = (int)(mn < 0 ? 0 : mn);
    hi = (int)(mx > vw.W - 1 ? vw.W - 1 : mx);
    return true;
}

// ---- decoration sprites (billboards at constant view depth; visitor.rs:1062-1137, sprite.vert:40-42) ----
// light (sprite.frag:15-27): light = min(v, 2v - dist), dist = 1 - 1/(w+1), w = z/100
B2D_HD int light_row_sprite(int b, int32_t z8) {
    int32_t r1 = (32 * (255 - b)) / 255;
    uint32_t Z = (uint32_t)z8 + 800u;
    int32_t num = (int32_t)(64u * (uint32_t)(255 - b) * Z) - 6528000;
    int32_t r2 = num <= 0 ? 0 : (int32_t)((uint32_t)num / (255u * Z));
    int32_t r = r1 > r2 ? r1 : r2;
    return r > 31 ? 31 : r;
}

struct SpriteFrame {
    int64_t cx, cz;          // view-space centre, Q8
    int32_t lo, hi;          // exact covered column interval
    int32_t scale, iscale, z8;
};

// Per-frame projection of a sprite of width w (map units) centred at world (x, y).  false = not on screen.
B2D_HD bool sprite_setup(const FrameConst &f, const View &vw, int32_t x, int32_t y, int32_t w, SpriteFrame &sp) {
    int32_t tx, tz;
    to_view(f, x, y, tx, tz);
    sp.cx = tx; sp.cz = tz;
    if (tz < 256) return false;                              // nearer than one map unit, or behind
    const int64_t F = vw.F, W = vw.W;
    const int64_t L = (sp.cx - (int64_t)w * 128) * F, R = (sp.cx + (int64_t)w * 128) * F;
    int64_t lo = 0, hi = W - 1;
    constrain(lo, hi, sp.cz * (1 - W) - L, 2 * sp.cz, 0);            // cz*c2 >= L
    constrain(lo, hi, R - 1 - sp.cz * (1 - W), -2 * sp.cz, 0);       // cz*c2 <= R-1
    if (lo > hi) return false;
    sp.lo = (int32_t)lo; sp.hi = (int32_t)hi;
    int64_t scale = ((int64_t)vw.FY2 << 25) / sp.cz;
    const int64_t cap = (int64_t)vw.FY2 << 17;
    if (scale > cap) scale = cap;
    if (scale < 1) return false;
    sp.scale = (int32_t)scale;
    sp.iscale = (int32_t)clampv<int64_t>(((int64_t)1 << 38) / scale, 1, 1 << 23);
    int64_t z8 = ((int64_t)sp.iscale * vw.FY2) >> 18;
    sp.z8 = z8 > 65535 ? 65535 : (int32_t)z8;
    return true;
}

// texture column of screen column x (0..w-1)
B2D_HD int32_t sprite_column(const SpriteFrame &sp, const View &vw, int x, int32_t w) {
    const int64_t c2 = 2 * (int64_t)x + 1 - vw.W;
    const int64_t L = (sp.cx - (int64_t)w * 128) * vw.F;
    return (int32_t)clampv<int64_t>(floordiv64(sp.cz * c2 - L, 256 * (int64_t)vw.F), 0, w - 1);
}

}  // namespace b2d
