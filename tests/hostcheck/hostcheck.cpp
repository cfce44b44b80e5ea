// TEST-ONLY: runs the product's pixel-contract arithmetic (rust-doom_b200/csrc/b2d_math.cuh) and the
// exact algorithms of the CUDA kernels on the CPU, one lane at a time, so that the maths can be
// checked against the oracle without a GPU.  This file is compiled into tests/hostcheck/
// libb2d_hostcheck.so by tests/conftest.py; it is NOT part of libb2d.so and no product code calls it.
#include <cstdint>
#include <algorithm>
#include <cstring>
#include <vector>

#include "../../rust-doom_b200/csrc/b2d_math.cuh"
#include "../../rust-doom_b200/csrc/b2d_scene.hpp"

using namespace b2d;

namespace {

struct HostScene {
    const uint32_t *hdr;
    const int32_t *verts;
    const NodeRec *nodes;
    const SSectorRec *ssectors;
    const SegRec *segs;
    const SectorRec *sectors;
    const TexRec *tex;
    const MidRec *mids;
    const SpriteRec *sprites;
    const uint8_t *texels, *flats, *colormap;
    const uint8_t *lit_texels, *lit_flats;      // host restatement of the b2d_prelight kernels (see build_lit)
    uint32_t lit_texel_stride, lit_flat_stride;
    int nverts, nnodes, nss, nsegs, ntex, nflats, sky_tex, nmids, nsprites;
    uint32_t root;
};

HostScene bind(const uint8_t *blob) {
    HostScene s;
    const uint32_t *h = reinterpret_cast<const uint32_t *>(blob);
    s.hdr = h;
    s.verts = reinterpret_cast<const int32_t *>(blob + h[H_OFF_VERTS]);
    s.nodes = reinterpret_cast<const NodeRec *>(blob + h[H_OFF_NODES]);
    s.ssectors = reinterpret_cast<const SSectorRec *>(blob + h[H_OFF_SSECTORS]);
    s.segs = reinterpret_cast<const SegRec *>(blob + h[H_OFF_SEGS]);
    s.sectors = reinterpret_cast<const SectorRec *>(blob + h[H_OFF_SECTORS]);
    s.tex = reinterpret_cast<const TexRec *>(blob + h[H_OFF_TEX]);
    s.mids = reinterpret_cast<const MidRec *>(blob + h[H_OFF_MIDS]);
    s.nmids = (int)h[H_NMIDS];
    s.sprites = reinterpret_cast<const SpriteRec *>(blob + h[H_OFF_SPRITES]);
    s.nsprites = (int)h[H_NSPRITES];
    s.texels = blob + h[H_OFF_TEXELS];
    s.flats = blob + h[H_OFF_FLATS];
    s.colormap = blob + h[H_OFF_COLORMAP];
    s.nverts = (int)h[H_NVERTS]; s.nnodes = (int)h[H_NNODES]; s.nss = (int)h[H_NSSECTORS];
    s.nsegs = (int)h[H_NSEGS]; s.ntex = (int)h[H_NTEX]; s.nflats = (int)h[H_NFLATS];
    s.sky_tex = (int32_t)h[H_SKY_TEX];
    s.root = h[H_ROOT];
    return s;
}

// The pre-lit planes the raster kernel reads (b2d_prelight_tex_kernel / b2d_prelight_kernel), built on the host with
// the same layout helpers (b2d_math.cuh): lit[r * stride + off + lit_index(...)] = colormap[r][texel].
struct LitPlanes { std::vector<uint8_t> texels, flats; };
void build_lit(HostScene &sc, LitPlanes &lp) {
    const uint32_t *h = sc.hdr;
    const size_t tstride = (h[H_TEXEL_BYTES] + 255u) & ~(size_t)255, fstride = (size_t)sc.nflats * 4096u;
    lp.texels.assign(33 * tstride + 256, 0);          // plane 32: opacity of textures with holes
    lp.flats.assign(32 * fstride + 256, 0);
    for (int ti = 0; ti < sc.ntex; ti++) {
        const TexRec &T = sc.tex[ti];
        const bool inter = tex_interleaved(T.h, T.texel_off);
        for (uint32_t row = 0; row < T.h; row++)
            for (uint32_t col = 0; col < T.w; col++) {
                const uint32_t t = sc.texels[T.texel_off + row * T.w + col];
                for (int r = 0; r < 32; r++)
                    lp.texels[(size_t)r * tstride + T.texel_off + lit_index(inter, T.w, row, col)] = sc.colormap[256 * r + t];
                if (T.mask_off != 0xFFFFFFFFu)
                    lp.texels[(size_t)32 * tstride + T.texel_off + lit_index(inter, T.w, row, col)] = sc.texels[T.mask_off + row * T.w + col];
            }
    }
    for (size_t i = 0; i < fstride; i++)
        for (int r = 0; r < 32; r++) lp.flats[(size_t)r * fstride + i] = sc.colormap[256 * r + sc.flats[i]];
    sc.lit_texels = lp.texels.data(); sc.lit_flats = lp.flats.data();
    sc.lit_texel_stride = (uint32_t)tstride; sc.lit_flat_stride = (uint32_t)fstride;
}

struct Range { int lo = 0, hi = -1; bool vis = false, solid = false; };

// mirrors b2d_walk_kernel
void walk(const HostScene &sc, const View &vw, const Pose &pose, FrameConst &fc, std::vector<SegFrame> &out) {
    frame_setup(pose, fc);
    std::vector<int32_t> tx((size_t)sc.nverts), tz((size_t)sc.nverts);
    for (int i = 0; i < sc.nverts; i++) to_view(fc, sc.verts[2 * i], sc.verts[2 * i + 1], tx[(size_t)i], tz[(size_t)i]);
    std::vector<Range> segr((size_t)sc.nsegs), boxr((size_t)sc.nnodes * 2);
    for (int i = 0; i < sc.nsegs; i++) {
        const SegRec &S = sc.segs[i];
        if (S.flags & kSegInvalid) continue;
        SegFrame sf;
        const bool closes = !(S.flags & kSegTwoSided) || S.otop <= S.obot;
        if (seg_frame_setup(vw, tx[(size_t)S.v1], tz[(size_t)S.v1], tx[(size_t)S.v2], tz[(size_t)S.v2], sf, closes)) {
            Range &r = segr[(size_t)i];
            r.vis = true; r.lo = sf.xlo; r.hi = sf.xhi;
            r.solid = closes && (sf.flags & kSegFrameNoSkip);
        }
    }
    for (int i = 0; i < 2 * sc.nnodes; i++) {
        const NodeRec &N = sc.nodes[i >> 1];
        const int32_t *box = (i & 1) ? N.lbox : N.rbox;
        int lo, hi;
        Range &r = boxr[(size_t)i];
        r.vis = box_range(fc, vw, box, lo, hi);
        if (r.vis) { r.lo = lo; r.hi = hi; }
    }
    std::vector<Range> sprr((size_t)sc.nsprites);
    std::vector<int32_t> sprz((size_t)sc.nsprites, 0);
    for (int i = 0; i < sc.nsprites; i++) {
        const SpriteRec &P = sc.sprites[i];
        SpriteFrame sp;
        sp.cz = 0;
        if (P.tex >= 0 && P.tex < sc.ntex && sprite_setup(fc, vw, P.x, P.y, (int32_t)sc.tex[P.tex].w, sp)) {
            sprr[(size_t)i].vis = true; sprr[(size_t)i].lo = sp.lo; sprr[(size_t)i].hi = sp.hi;
        }
        sprz[(size_t)i] = (int32_t)sp.cz;
    }
    std::vector<char> solid((size_t)vw.W, 0);
    auto range_open = [&](int lo, int hi) {
        for (int x = lo; x <= hi; x++) if (!solid[(size_t)x]) return true;
        return false;
    };
    std::vector<uint32_t> stack;
    stack.push_back(sc.root);
    std::vector<int> list;
    int status = 0;
    int budget = 2 * (sc.nnodes + sc.nss) + 64;
    while (!stack.empty()) {
        if (--budget < 0) { status |= 4; break; }
        uint32_t child = stack.back();
        stack.pop_back();
        if (child & kLeaf) {
            uint32_t id = child & 0x7FFFFFFFu;
            if (id >= (uint32_t)sc.nss) continue;
            const SSectorRec &ss = sc.ssectors[id];
            if (ss.sector < 0) continue;
            {
                const int sfirst = ss.sprites & 0xFFFFFF, scnt = (ss.sprites >> 24) & 0xFF;
                std::vector<int> vis;                 // nearest first, ties in stored order (as the walk kernel ranks them)
                for (int k = 0; k < scnt && sfirst + k < sc.nsprites; k++) {
                    const Range &r = sprr[(size_t)(sfirst + k)];
                    if (r.vis && range_open(r.lo, r.hi)) vis.push_back(sfirst + k);
                }
                std::stable_sort(vis.begin(), vis.end(), [&](int a, int b) { return sprz[(size_t)a] < sprz[(size_t)b]; });
                for (int pi : vis) list.push_back(sc.nsegs + pi);
            }
            for (int k0 = 0; k0 < ss.num_segs; k0 += 32) {
                std::vector<int> emitted;
                for (int lane = 0; lane < 32 && k0 + lane < ss.num_segs; lane++) {
                    int si = ss.first_seg + k0 + lane;
                    const Range &r = segr[(size_t)si];
                    if (r.vis && range_open(r.lo, r.hi)) { list.push_back(si); emitted.push_back(si); }
                }
                for (int si : emitted) {
                    const Range &r = segr[(size_t)si];
                    if (r.solid) for (int x = r.lo; x <= r.hi; x++) solid[(size_t)x] = 1;
                }
            }
            if (!range_open(0, vw.W - 1)) break;
        } else {
            if (child >= (uint32_t)sc.nnodes) continue;
            const NodeRec &N = sc.nodes[child];
            int side = node_side(fc.pose, N.x, N.y, N.dx, N.dy);
            const Range &rn = boxr[2 * (size_t)child + (size_t)side], &rf = boxr[2 * (size_t)child + (size_t)(side ^ 1)];
            bool far_vis = rf.vis && range_open(rf.lo, rf.hi);
            bool near_vis = rn.vis && range_open(rn.lo, rn.hi);
            if (stack.size() + (far_vis ? 1 : 0) + (near_vis ? 1 : 0) > 128) { status = 1; break; }
            if (far_vis) stack.push_back(N.child[side ^ 1]);
            if (near_vis) stack.push_back(N.child[side]);
        }
    }
    out.clear();
    for (int si : list) {
        SegFrame sf;
        if (si >= sc.nsegs) {
            const int pi = si - sc.nsegs;
            const SpriteRec &P = sc.sprites[pi];
            SpriteFrame sp;
            sprite_setup(fc, vw, P.x, P.y, (int32_t)sc.tex[P.tex].w, sp);
            std::memset(&sf, 0, sizeof sf);
            sf.Nc = sp.cx; sf.Nx = sp.cz; sf.seg = -1 - pi; sf.xlo = (int16_t)sp.lo; sf.xhi = (int16_t)sp.hi;
            out.push_back(sf);
            continue;
        }
        const SegRec &S = sc.segs[si];
        seg_frame_setup(vw, tx[(size_t)S.v1], tz[(size_t)S.v1], tx[(size_t)S.v2], tz[(size_t)S.v2], sf, false);
        sf.seg = si;
        out.push_back(sf);
    }
    fc.count = (int)out.size();
    fc.status = status;
}

struct Lane { int ct, cb; uint32_t skycol; };

// mirrors b2d_raster_kernel, lanes executed one after the other
struct RasterStats { long long iters = 0, pixels = 0, entries = 0, evals = 0; };

void raster(const HostScene &sc, const View &vw, const FrameConst &fc, const std::vector<SegFrame> &wl,
            const std::vector<uint32_t> &yslope, uint32_t invF, uint8_t *fb, int SW = 32, RasterStats *st = nullptr) {
    const int W = vw.W, H = vw.H;
    auto put = [&](int x, int y, uint8_t v) { fb[(size_t)y * W + x] = v; };
    auto fill_void = [&](int x, int ya, int yb) { for (int y = ya; y < yb; y++) put(x, y, 0); };
    auto draw_sky = [&](int x, const Lane &ln, int ya, int yb) {
        if (sc.sky_tex < 0) { fill_void(x, ya, yb); return; }
        const TexRec &T = sc.tex[sc.sky_tex];
        const bool inter = tex_interleaved(T.h, T.texel_off);
        const uint8_t *px = sc.lit_texels + T.texel_off;                       // light row 0
        for (int y = ya; y < yb; y++) {
            int v = sky_row(y, H, (int32_t)T.h);
            put(x, y, px[lit_index(inter, T.w, (uint32_t)v, ln.skycol)]);
        }
    };
    auto draw_plane = [&](int x, const Lane &ln, int ya, int yb, int32_t h, int32_t flat, int lightb, bool visible) {
        if (ya >= yb) return;
        if (!visible) { fill_void(x, ya, yb); return; }
        if (flat == kFlatSky) { draw_sky(x, ln, ya, yb); return; }
        if (flat < 0 || flat >= sc.nflats) { fill_void(x, ya, yb); return; }
        const uint8_t *px = sc.lit_flats;
        uint32_t habs = plane_habs(h, fc.pose.z);
        const PlaneDir dir = plane_dir(fc, vw, x, invF);
        for (int y = ya; y < yb; y++) {
            PlaneRow pr = plane_row(habs, yslope[(size_t)y]);
            const uint32_t cm6 = (sc.lit_flat_stride >> 6) * (uint32_t)light_row(lightb, pr.z8) + 64u * (uint32_t)flat;
            put(x, y, px[flat_offset(cm6, plane_u(fc.pose.x, pr.z8q, dir.ax), plane_u(fc.pose.y, pr.z8q, dir.ay))]);
        }
    };
    auto draw_wall = [&](int x, int ya, int yb, int32_t tex, int32_t tA, int32_t hA, int32_t ucol, int32_t iscale, int row) {
        if (ya >= yb) return;
        if (tex < 0 || tex >= sc.ntex) { fill_void(x, ya, yb); return; }
        const TexRec &T = sc.tex[tex];
        const uint32_t col = (uint32_t)floormod32(ucol, (int32_t)T.w);
        const uint8_t *pl = sc.lit_texels + (size_t)row * sc.lit_texel_stride + T.texel_off;
        const uint32_t tstep = (uint32_t)(iscale >> 4);
        uint32_t t = (uint32_t)wall_tbase(tA, hA, fc.pose.z, H, iscale) + (uint32_t)ya * tstep;
        if (!tex_interleaved(T.h, T.texel_off)) {
            for (int y = ya; y < yb; y++, t += tstep) put(x, y, pl[wall_row((int32_t)t, T.h, T.hmagic, T.hbias) * T.w + col]);
            return;
        }
        if (T.h >= 8u && tstep <= kWallFast8) {
            // the incremental path of wall_fast_loop (the kernel takes it when every lane of the warp qualifies; here per
            // lane, alternating between the 16- and the 8-row form, and starting a few rows above ya the way a lane whose
            // neighbours start higher does)
            const int R = (tstep <= kWallFast16 && (x & 1) == 0) ? 16 : 8;
            const int y0 = std::max(0, ya - (x % 5) * 3);
            const uint32_t t0 = (uint32_t)wall_tbase(tA, hA, fc.pose.z, H, iscale) + (uint32_t)y0 * tstep;
            const uint32_t r0 = wall_row((int32_t)t0, T.h, T.hmagic, T.hbias);
            uint32_t q = r0 >> 2, acc = wall_acc29(t0, r0);
            const uint32_t ts29 = tstep << 13, nq = T.h >> 2, w4f = 4u * T.w;
            for (int y = y0; y < yb; y += R) {
                const uint32_t q1 = q + 1u == nq ? 0u : q + 1u;
                uint32_t w0, w1;
                std::memcpy(&w0, pl + 4u * col + (size_t)q * w4f, 4);
                std::memcpy(&w1, pl + 4u * col + (size_t)q1 * w4f, 4);
                const uint32_t m = row_mask(y, ya, yb, R);
                for (int k = 0; k < R; k++)
                    if ((m >> k) & 1u) put(x, y + k, (uint8_t)(pick_byte(w0, w1, wall_sel(acc, ts29, (uint32_t)k)) & 0xFFu));
                wall_advance(acc, q, ts29, (uint32_t)R, nq);
            }
            return;
        }
        // batches of 8 rows as in draw_wall_warp: two aligned words + byte pick when the 8 rows stay inside two
        // consecutive row quads, eight byte fetches otherwise (the kernel decides per warp, here per lane: both
        // forms must give the same bytes, which is what the comparison with the oracle checks)
        const uint32_t colb = 4u * col, w4 = 4u * T.w;
        for (int y = ya; y < yb; y += 8, t += 8u * tstep) {
            const uint32_t r0 = wall_row((int32_t)t, T.h, T.hmagic, T.hbias);
            const uint32_t acc = wall_acc(t, r0);
            uint32_t v[8];
            if (((acc + 7u * tstep) >> 16) < 8u) {
                const uint32_t q0 = r0 >> 2, q1 = next_quad(q0, T.h);
                uint32_t w0, w1;
                std::memcpy(&w0, pl + (q0 * w4 + colb), 4);
                std::memcpy(&w1, pl + (q1 * w4 + colb), 4);
                for (uint32_t k = 0; k < 8; k++) v[k] = pick_byte(w0, w1, (acc + k * tstep) >> 16) & 0xFFu;
            } else {
                const uint32_t t4 = t + 4u * tstep;
                const uint32_t r4 = wall_row((int32_t)t4, T.h, T.hmagic, T.hbias);
                const uint32_t acc4 = wall_acc(t4, r4);
                if (((acc + 3u * tstep) >> 16) < 8u && ((acc4 + 3u * tstep) >> 16) < 8u) {   // two 4-row halves
                    const uint32_t q0 = r0 >> 2, q4 = r4 >> 2;
                    uint32_t a0, a1, b0, b1;
                    std::memcpy(&a0, pl + (q0 * w4 + colb), 4);
                    std::memcpy(&a1, pl + (next_quad(q0, T.h) * w4 + colb), 4);
                    std::memcpy(&b0, pl + (q4 * w4 + colb), 4);
                    std::memcpy(&b1, pl + (next_quad(q4, T.h) * w4 + colb), 4);
                    for (uint32_t k = 0; k < 4; k++) {
                        v[k] = pick_byte(a0, a1, (acc + k * tstep) >> 16) & 0xFFu;
                        v[k + 4] = pick_byte(b0, b1, (acc4 + k * tstep) >> 16) & 0xFFu;
                    }
                } else {
                    for (uint32_t k = 0; k < 8; k++) {
                        const uint32_t rk = wall_row((int32_t)(t + k * tstep), T.h, T.hmagic, T.hbias);
                        v[k] = pl[(rk >> 2) * w4 + colb + (rk & 3u)];
                    }
                }
            }
            for (int k = 0; k < 8 && y + k < yb; k++) put(x, y + k, (uint8_t)v[k]);
        }
    };

    const int strips = (W + SW - 1) / SW;
    for (int strip = 0; strip < strips; strip++) {
        const int x0 = strip * SW;
        std::vector<Lane> lanes((size_t)SW);
        for (int l = 0; l < SW; l++) {
            int x = x0 + l;
            lanes[l].ct = 0; lanes[l].cb = x < W ? H : 0; lanes[l].skycol = 0;
            if (sc.sky_tex >= 0 && x < W) lanes[l].skycol = umulhi32(sky_u32(x, vw, fc.pose.angle), sc.tex[sc.sky_tex].w);
        }
        struct Deferred { size_t k; std::vector<uint32_t> win; };
        int masked_cap = sc.nmids + sc.nsprites;          // as b2d_renderer_create sizes the deferred lists
        masked_cap = masked_cap < 8 ? 8 : (masked_cap > 128 ? 128 : masked_cap);
        std::vector<Deferred> deferred;
        for (size_t k = 0; k < wl.size(); k++) {
            const SegFrame &sf = wl[k];
            if (!(sf.xhi >= x0 && sf.xlo <= x0 + SW - 1)) continue;
            bool any_open = false;
            for (int l = 0; l < SW; l++) any_open |= lanes[l].ct < lanes[l].cb;
            if (!any_open) break;
            if (sf.seg < 0) {        // decoration sprite: defer with the windows open right now
                Deferred d{k, std::vector<uint32_t>((size_t)SW, 0u)};
                bool any = false;
                for (int l = 0; l < SW; l++) {
                    int x = x0 + l;
                    const Lane &ln = lanes[(size_t)l];
                    if (x < W && ln.ct < ln.cb && x >= sf.xlo && x <= sf.xhi) {
                        d.win[(size_t)l] = (uint32_t)ln.ct | ((uint32_t)ln.cb << 16);
                        any = true;
                    }
                }
                if (any && deferred.size() < (size_t)masked_cap) deferred.push_back(d);
                continue;
            }
            const SegRec &S = sc.segs[sf.seg];
            const SectorRec &SF = sc.sectors[S.front];
            const int32_t fcl = SF.ceil, ffl = SF.floor;
            const bool two = S.flags & kSegTwoSided;
            const bool ceil_vis = ((int64_t)fcl << 16) > fc.pose.z || SF.ceil_flat == kFlatSky;
            const bool floor_vis = ((int64_t)ffl << 16) < fc.pose.z || SF.floor_flat == kFlatSky;
            Deferred dfr{k, std::vector<uint32_t>((size_t)SW, 0u)};
            bool any_deferred = false;
            // lock-step extents of the five draws (ceiling, A, B, floor) over the strip, for statistics
            int lo[4] = {1 << 30, 1 << 30, 1 << 30, 1 << 30}, hi[4] = {0, 0, 0, 0};
            if (st) st->entries++;
            for (int l = 0; l < SW; l++) {
                int x = x0 + l;
                Lane &ln = lanes[l];
                if (!(x < W && ln.ct < ln.cb && x >= sf.xlo && x <= sf.xhi)) continue;
                ColumnEval ce;
                if (!column_eval(sf, vw, x, ce)) continue;
                if (st) st->evals++;
                int ct = ln.ct, cb = ln.cb;
                int row = light_row(S.light, ce.z8);
                int32_t ucol = S.uoff + (int32_t)(((uint64_t)ce.s24 * (uint32_t)S.len_q12) >> 36);
                int yfc = yrow(fcl, ce.scale, fc.pose.z, H), yff = yrow(ffl, ce.scale, fc.pose.z, H);
                int y1 = clampv(yfc, ct, cb), y2, y3, y4;
                if (!two) { y2 = clampv(yff, y1, cb); y3 = y2; y4 = y2; }
                else {
                    int yot = yrow(S.otop, ce.scale, fc.pose.z, H), yob = yrow(S.obot, ce.scale, fc.pose.z, H);
                    y2 = clampv(yot, y1, cb); y3 = clampv(yob, y2, cb); y4 = clampv(yff, y3, cb);
                }
                if (st) {
                    auto acc = [&](int d, int a, int b) { if (a < b) { if (a < lo[d]) lo[d] = a; if (b > hi[d]) hi[d] = b; st->pixels += b - a; } };
                    acc(0, ct, y1);
                    if (!two || S.otop < fcl) acc(1, y1, y2);
                    if (two && S.obot > ffl) acc(2, y3, y4);
                    acc(3, y4, cb);
                }
                draw_plane(x, ln, ct, y1, fcl, SF.ceil_flat, SF.light, ceil_vis);
                if (!two) draw_wall(x, y1, y2, S.texA, S.tA, S.hA, ucol, ce.iscale, row);
                else {
                    if (S.otop < fcl) draw_wall(x, y1, y2, S.texA, S.tA, S.hA, ucol, ce.iscale, row);
                    if (S.obot > ffl) draw_wall(x, y3, y4, S.texB, S.tB, S.hB, ucol, ce.iscale, row);
                }
                draw_plane(x, ln, y4, cb, ffl, SF.floor_flat, SF.light, floor_vis);
                if (!two || y2 >= y3) { ln.ct = H; ln.cb = 0; }
                else { ln.ct = y2; ln.cb = y3; }
                if (two && S.mid >= 0 && y2 < y3) { dfr.win[(size_t)l] = (uint32_t)y2 | ((uint32_t)y3 << 16); any_deferred = true; }
            }
            if (any_deferred && deferred.size() < (size_t)masked_cap) deferred.push_back(dfr);
            if (st) for (int d = 0; d < 4; d++) if (hi[d] > lo[d]) st->iters += hi[d] - lo[d];
        }
        for (int l = 0; l < SW; l++)
            if (x0 + l < W) fill_void(x0 + l, lanes[l].ct, lanes[l].cb);
        // masked middle textures, back to front (mirrors masked_pass in b2d_kernels.cu)
        for (size_t e = deferred.size(); e-- > 0;) {
            const SegFrame &sf = wl[deferred[e].k];
            for (int l = 0; l < SW; l++) {
                uint32_t packed = deferred[e].win[(size_t)l];
                int ya = (int)(packed & 0xFFFFu), yb = (int)(packed >> 16), x = x0 + l;
                if (!(ya < yb)) continue;
                int32_t tex, tA, hA, ucol, iscale, row;
                if (sf.seg < 0) {
                    const SpriteRec &P = sc.sprites[-1 - sf.seg];
                    if (P.tex < 0 || P.tex >= sc.ntex) continue;
                    const int32_t sw = (int32_t)sc.tex[P.tex].w, sh = (int32_t)sc.tex[P.tex].h;
                    SpriteFrame sp;
                    sp.cx = sf.Nc; sp.cz = sf.Nx;
                    int64_t scale = ((int64_t)vw.FY2 << 25) / sp.cz;
                    const int64_t cap = (int64_t)vw.FY2 << 17;
                    if (scale > cap) scale = cap;
                    iscale = (int32_t)clampv<int64_t>(((int64_t)1 << 38) / scale, 1, 1 << 23);
                    int64_t z8 = ((int64_t)iscale * vw.FY2) >> 18;
                    row = light_row_sprite(P.light, z8 > 65535 ? 65535 : (int32_t)z8);
                    tex = P.tex; tA = 0; hA = P.low + sh;
                    ya = std::max(ya, yrow(P.low + sh, (int32_t)scale, fc.pose.z, H));
                    yb = std::min(yb, yrow(P.low, (int32_t)scale, fc.pose.z, H));
                    ucol = sprite_column(sp, vw, x, sw);
                } else {
                    const SegRec &S = sc.segs[sf.seg];
                    if (S.mid < 0 || S.mid >= sc.nmids) continue;
                    const MidRec &M = sc.mids[S.mid];
                    ColumnEval ce;
                    if (!column_eval(sf, vw, x, ce)) continue;
                    tex = M.tex; tA = M.t_high; hA = M.high;
                    ya = std::max(ya, yrow(M.high, ce.scale, fc.pose.z, H));
                    yb = std::min(yb, yrow(M.low, ce.scale, fc.pose.z, H));
                    ucol = S.uoff + (int32_t)(((uint64_t)ce.s24 * (uint32_t)S.len_q12) >> 36);
                    iscale = ce.iscale;
                    row = light_row(S.light, ce.z8);
                }
                if (tex < 0 || tex >= sc.ntex) continue;
                const TexRec &T = sc.tex[tex];
                uint32_t col = (uint32_t)floormod32(ucol, (int32_t)T.w);
                const bool inter = tex_interleaved(T.h, T.texel_off);
                const uint8_t *px = sc.lit_texels + (size_t)row * sc.lit_texel_stride + T.texel_off;
                const bool has_mask = T.mask_off != 0xFFFFFFFFu;
                const uint8_t *pm = sc.lit_texels + (size_t)32 * sc.lit_texel_stride + T.texel_off;   // opacity plane
                int32_t tbase = wall_tbase(tA, hA, fc.pose.z, H, iscale), tstep = iscale >> 4;
                for (int y = ya; y < yb; y++) {
                    const uint32_t r = wall_row(tbase + y * tstep, T.h, T.hmagic, T.hbias);
                    if (has_mask && !pm[lit_index(inter, T.w, r, col)]) continue;
                    put(x, y, px[lit_index(inter, T.w, r, col)]);
                }
            }
        }
    }
}

}  // namespace

static int render_impl(const uint8_t *blob, const View *vw, const Pose *poses, int n, uint8_t *fb,
                       int32_t *counts, int32_t *seg_ids, int stride, uint32_t tics, const SectorMove *moves = nullptr,
                       int n_moves = 0) {
    HostScene sc = bind(blob);
    LitPlanes lit;
    build_lit(sc, lit);                // from the blob's own table: set_time only re-points records
    // the product's time handling: the three time-dependent tables are rebuilt by scene_at_time (b2d_scene.hpp)
    // exactly as b2d_renderer_set_time does before it uploads them
    std::vector<TexRec> tex_t((size_t)sc.ntex);
    std::vector<SectorRec> sectors_t((size_t)sc.hdr[H_NSECTORS]);
    std::vector<SegRec> segs_t((size_t)sc.nsegs);
    std::vector<SpriteRec> sprites_t((size_t)sc.nsprites);
    std::vector<MidRec> mids_t((size_t)sc.hdr[H_NMIDS]);
    std::vector<int32_t> floor_off, ceil_off;             // the moving sectors' state (b2d_renderer_set_sector_moves)
    if (n_moves > 0 && expand_moves(blob, moves, (size_t)n_moves, floor_off, ceil_off)) return -1;
    if (scene_is_timed(blob)) {          // tic 0 included: a frame name with k > 0 shows the group's frame 0
        scene_at_time(blob, tics, tex_t.data(), sectors_t.data(), segs_t.data(), sprites_t.data(), mids_t.data(),
                      n_moves > 0 ? floor_off.data() : nullptr, n_moves > 0 ? ceil_off.data() : nullptr);
        sc.tex = tex_t.data(); sc.sectors = sectors_t.data(); sc.segs = segs_t.data(); sc.sprites = sprites_t.data();
        sc.mids = mids_t.data();
    }
    std::vector<uint32_t> yslope((size_t)vw->H);
    for (int y = 0; y < vw->H; y++) yslope[(size_t)y] = yslope_entry(y, *vw);
    uint32_t invF = (uint32_t)(4294967296ULL / (uint64_t)vw->F);
    const size_t npix = (size_t)vw->W * vw->H;
    for (int i = 0; i < n; i++) {
        FrameConst fc;
        std::vector<SegFrame> wl;
        walk(sc, *vw, poses[i], fc, wl);
        // poison the frame first: the raster must overwrite every pixel exactly like the GPU does
        std::memset(fb + npix * (size_t)i, 0xAB, npix);
        raster(sc, *vw, fc, wl, yslope, invF, fb + npix * (size_t)i);
        if (counts) counts[i] = fc.status ? -fc.status : fc.count;
        if (seg_ids) for (int k = 0; k < fc.count && k < stride; k++) seg_ids[(size_t)i * stride + k] = wl[(size_t)k].seg;
    }
    return 0;
}

extern "C" int hostcheck_render(const uint8_t *blob, const View *vw, const Pose *poses, int n, uint8_t *fb,
                                int32_t *counts, int32_t *seg_ids, int stride) {
    return render_impl(blob, vw, poses, n, fb, counts, seg_ids, stride, 0);
}

extern "C" int hostcheck_render_t(const uint8_t *blob, const View *vw, const Pose *poses, int n, uint8_t *fb,
                                  int32_t *counts, int32_t *seg_ids, int stride, uint32_t tics) {
    return render_impl(blob, vw, poses, n, fb, counts, seg_ids, stride, tics);
}

extern "C" int hostcheck_render_m(const uint8_t *blob, const View *vw, const Pose *poses, int n, uint8_t *fb,
                                  int32_t *counts, int32_t *seg_ids, int stride, uint32_t tics, const SectorMove *moves, int n_moves) {
    return render_impl(blob, vw, poses, n, fb, counts, seg_ids, stride, tics, moves, n_moves);
}

// the product's light-effect evaluation (scene_at_time): light byte per sector at `tics`, -1 without effect
extern "C" void hostcheck_lights(const uint8_t *blob, uint32_t tics, int16_t *out) {
    const uint32_t *h = reinterpret_cast<const uint32_t *>(blob);
    std::vector<TexRec> tex(h[H_NTEX]);
    std::vector<SectorRec> sectors(h[H_NSECTORS]);
    std::vector<SegRec> segs(h[H_NSEGS]);
    std::vector<SpriteRec> sprites(h[H_NSPRITES]);
    scene_at_time(blob, tics, tex.data(), sectors.data(), segs.data(), sprites.data());
    const LightRec *lights = reinterpret_cast<const LightRec *>(blob + h[H_OFF_LIGHTS]);
    for (uint32_t i = 0; i < h[H_NSECTORS]; i++) out[i] = lights[i].kind != kLightNone ? (int16_t)sectors[i].light : (int16_t)-1;
}

extern "C" void hostcheck_sincos(uint32_t angle, int32_t *c, int32_t *s) { sincos_q30(angle, *c, *s); }

// the product's flat-texel ray direction (plane_dir, Q18) of every column, as the raster kernel computes it per column:
// out[2x] = ax, out[2x+1] = ay
extern "C" void hostcheck_plane_dirs(const View *vw, const Pose *pose, int32_t *out) {
    FrameConst fc;
    frame_setup(*pose, fc);
    const uint32_t invF = (uint32_t)(4294967296ULL / (uint64_t)vw->F);
    for (int x = 0; x < vw->W; x++) {
        const PlaneDir d = plane_dir(fc, *vw, x, invF);
        out[2 * x] = d.ax; out[2 * x + 1] = d.ay;
    }
}

// lock-step iteration statistics for a strip width (design exploration; test-only)
extern "C" int hostcheck_stats(const uint8_t *blob, const View *vw, const Pose *poses, int n, int strip_width,
                               long long *out4) {
    HostScene sc = bind(blob);
    LitPlanes lit;
    build_lit(sc, lit);
    std::vector<uint32_t> yslope((size_t)vw->H);
    for (int y = 0; y < vw->H; y++) yslope[(size_t)y] = yslope_entry(y, *vw);
    uint32_t invF = (uint32_t)(4294967296ULL / (uint64_t)vw->F);
    std::vector<uint8_t> fb((size_t)vw->W * vw->H);
    RasterStats st;
    for (int i = 0; i < n; i++) {
        FrameConst fc;
        std::vector<SegFrame> wl;
        walk(sc, *vw, poses[i], fc, wl);
        raster(sc, *vw, fc, wl, yslope, invF, fb.data(), strip_width, &st);
    }
    out4[0] = st.iters; out4[1] = st.pixels; out4[2] = st.entries; out4[3] = st.evals;
    return 0;
}
