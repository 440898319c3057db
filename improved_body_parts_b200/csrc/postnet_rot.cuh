// postnet_rot.cuh -- K0 with rotation search: one (scale, angle) item of predict()'s loop with angle != 0, fused.
//
// With rotation_search != [0] the reference warps the up-sampled maps back before the crop, evaluate.py:143-158:
//   flip ensemble -> cv2.resize(x stride, INTER_CUBIC) -> cv2.warpAffine(map, rotate_matrix_reverse, (0, 0))
//   -> crop the padding -> cv2.resize(image size, INTER_CUBIC) -> heatmap_avg += map / n
// on the FULL padded up-sampled map (Hp x Wp = h * stride x w * stride), so bilinear taps may land in the padding.
//
// Arithmetic of the warp: OpenCV's generic fixed-point path (imgproc/src/imgwarp.cpp, warpAffine + remapBilinear on
// float32) as restated -- and pinned to cv2 bit for bit -- by tests/rotation_port.py; warp_affine.cuh holds the
// fixed-point coordinates and weights.  The host inverts the matrix in float64 exactly as warpAffine does and passes
// the destination -> source map m[6]; taps outside [0,Hp) x [0,Wp) read 0.
// The resizes and the epilogue are postnet_generic_kernel's operations in the same order; the translation unit is built
// with -fmad=false and spells out every *_rn operation, so the maps are BIT-IDENTICAL to the port's
// (tests/test_gpu_postnet_rotation.py).
//
// One CTA computes one output tile of one image over a chunk of channels.  Everything that depends on the tile position
// only is built once per CTA: the second resize's tables give the tile's footprint on the crop grid; the warp's
// per-column adelta / bdelta and per-row X0 / Y0 give that footprint's source box in the up-sampled map -- exact, from
// the four corners, because the fixed-point coordinates are monotone in x and in y -- clamped to the map; the x stride
// resize's tables cover that box.  Per channel: source tile (flip-averaged on load) -> horizontal x stride -> vertical
// x stride (the box of the up-sampled map) -> warp into the footprint -> horizontal / vertical pass of the second
// resize -> epilogue.  Neither the up-sampled nor the warped map exists in HBM.  The float64 sums over the items of the
// loop continue through memory between launches (one launch per rotated item).
#pragma once

#include <cassert>
#include <climits>

#include "postnet.cuh"
#include "warp_affine.cuh"

namespace spg {

struct PostRotArgs {
    PostArgs a;      // the item (net, strides, h, w, crop, sx2 / sy2 of the generic kernel), outputs, epilogue, tiling
    double m[6];     // destination -> source map of the warp: cv2.warpAffine's inverse of rotate_matrix_reverse
    int Hp, Wp;      // up-sampled (padded) map: h * stride x w * stride
    int cap_fw, cap_fh, cap_bw, cap_bh, cap_cs, cap_rs;  // shared-memory capacities sized by the host for the tile
};

__host__ __device__ constexpr size_t postrot_smem_bytes(int tw, int th, int fw, int fh, int bw, int bh, int cs, int rs) {
    return sizeof(AxisTab) * (size_t)(tw + th + bw + bh) + sizeof(int) * (size_t)(2 * fw + 2 * fh + 8) +
           sizeof(float) * ((size_t)rs * cs + (size_t)rs * bw + (size_t)bh * bw + (size_t)fh * fw + (size_t)fh * tw);
}

__global__ void __launch_bounds__(kPostThreads) postnet_rot_kernel(PostRotArgs r) {
    const PostArgs &a = r.a;
    extern __shared__ __align__(16) unsigned char rot_smem[];
    const int TW = a.tile_w;
    AxisTab *t2x = reinterpret_cast<AxisTab *>(rot_smem), *t2y = t2x + TW, *t1x = t2y + a.tile_h, *t1y = t1x + r.cap_bw;
    int *adx = reinterpret_cast<int *>(t1y + r.cap_bh), *bdx = adx + r.cap_fw;  // per footprint column
    int *x0y = bdx + r.cap_fw, *y0y = x0y + r.cap_fh;                           // per footprint row
    int *rng = y0y + r.cap_fh;
    float *s0 = reinterpret_cast<float *>(rng + 8);  // source tile, flip-averaged            [RS][cap_cs]
    float *s1 = s0 + r.cap_rs * r.cap_cs;            // after the horizontal x stride pass    [RS][cap_bw]
    float *s2 = s1 + r.cap_rs * r.cap_bw;            // the box of the up-sampled map         [BH][cap_bw]
    float *sw = s2 + r.cap_bh * r.cap_bw;            // warped, on the crop grid (footprint)  [FH][cap_fw]
    float *s3 = sw + r.cap_fh * r.cap_fw;            // after the second resize's h. pass     [FH][TW]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = kPostThreads / 32;
    const int tile = blockIdx.x, n = blockIdx.z;
    const int c_begin = blockIdx.y * a.chan_chunk, c_end = min(c_begin + a.chan_chunk, a.n_out);
    const int ty = tile / a.tiles_x, tx = tile - ty * a.tiles_x;
    const int ox0 = tx * a.tile_w, oy0 = ty * a.tile_h;
    const int tw = min(a.tile_w, a.W - ox0), th = min(a.tile_h, a.H - oy0);
    const bool identity = a.crop_h == a.H && a.crop_w == a.W;  // second resize with scale 1: weights (0, 1, 0, 0)

    // ---- once per CTA: the tile's footprint on the crop grid (taps clamped to the cropped array, :148-149)
    for (int i = tid; i < tw; i += kPostThreads) t2x[i].s = axis_entry(ox0 + i, a.sx2, t2x[i].c);
    for (int i = tid; i < th; i += kPostThreads) t2y[i].s = axis_entry(oy0 + i, a.sy2, t2y[i].c);
    __syncthreads();
    if (tid == 0) {
        const int c_lo = identity ? ox0 : clampi(t2x[0].s, 0, a.crop_w - 1), c_hi = identity ? ox0 + tw - 1 : clampi(t2x[tw - 1].s + 3, 0, a.crop_w - 1);
        const int y_lo = identity ? oy0 : clampi(t2y[0].s, 0, a.crop_h - 1), y_hi = identity ? oy0 + th - 1 : clampi(t2y[th - 1].s + 3, 0, a.crop_h - 1);
        rng[0] = c_lo; rng[1] = c_hi - c_lo + 1; rng[2] = y_lo; rng[3] = y_hi - y_lo + 1;
    }
    __syncthreads();
    const int c_lo = rng[0], FW = rng[1], y_lo = rng[2], FH = rng[3];
    // ---- the warp's fixed-point coordinate tables (warpAffine: AB_BITS = 10, round_delta = 16); the crop starts at
    // the padded map's origin (pad[0] = pad[1] = 0), so crop-grid coordinates are destination coordinates of the warp
    for (int i = tid; i < FW; i += kPostThreads) warp_col(r.m, c_lo + i, adx[i], bdx[i]);
    for (int i = tid; i < FH; i += kPostThreads) warp_row(r.m, y_lo + i, x0y[i], y0y[i]);
    __syncthreads();
    if (tid == 0) {
        // source box: X0 + adelta and Y0 + bdelta are sums of a monotone function of x and one of y, so their extremes
        // over the footprint are at its corners; the second tap of each axis adds one
        int bx_lo = INT_MAX, bx_hi = INT_MIN, by_lo = INT_MAX, by_hi = INT_MIN;
        for (int k = 0; k < 4; k++) {
            const int i = (k & 1) ? FW - 1 : 0, j = (k & 2) ? FH - 1 : 0;
            const int sx = (x0y[j] + adx[i]) >> 10, sy = (y0y[j] + bdx[i]) >> 10;
            bx_lo = min(bx_lo, sx); bx_hi = max(bx_hi, sx + 1);
            by_lo = min(by_lo, sy); by_hi = max(by_hi, sy + 1);
        }
        bx_lo = max(bx_lo, 0); bx_hi = min(bx_hi, r.Wp - 1);
        by_lo = max(by_lo, 0); by_hi = min(by_hi, r.Hp - 1);
        const bool empty = bx_lo > bx_hi || by_lo > by_hi;  // the whole footprint maps outside: every value is 0
        rng[4] = bx_lo; rng[5] = empty ? 0 : bx_hi - bx_lo + 1;
        rng[6] = by_lo; rng[7] = empty ? 0 : by_hi - by_lo + 1;
        assert(FW <= r.cap_fw && FH <= r.cap_fh && rng[5] <= r.cap_bw && rng[7] <= r.cap_bh);
    }
    __syncthreads();
    const int bx_lo = rng[4], BW = rng[5], by_lo = rng[6], BH = rng[7];
    // ---- tables of the first resize (x stride) for the box's columns / rows
    for (int i = tid; i < BW; i += kPostThreads) t1x[i].s = axis_entry(bx_lo + i, a.sx1, t1x[i].c);
    for (int i = tid; i < BH; i += kPostThreads) t1y[i].s = axis_entry(by_lo + i, a.sy1, t1y[i].c);
    __syncthreads();
    const int sc_lo = BW ? clampi(t1x[0].s, 0, a.w - 1) : 0, sc_hi = BW ? clampi(t1x[BW - 1].s + 3, 0, a.w - 1) : -1;
    const int sr_lo = BH ? clampi(t1y[0].s, 0, a.h - 1) : 0, sr_hi = BH ? clampi(t1y[BH - 1].s + 3, 0, a.h - 1) : -1;
    const int CS = sc_hi - sc_lo + 1, RS = sr_hi - sr_lo + 1;
    assert(CS <= r.cap_cs && RS <= r.cap_rs);

    const float nf = (float)a.n_scales;
    const size_t plane = (size_t)a.H * a.W;
    const bool first = a.scale_index == 0, last = a.scale_index == a.n_scales - 1;
    for (int c = c_begin; c < c_end; c++) {
        // ---- source tile: (out[c] + mirrored_out[flip(c)][:, ::-1]) / 2  (:139-140), float32
        {
            const long long base0 = (long long)n * a.img_stride + (long long)a.src_chan[c] * a.chan_stride;
            const long long base1 = (long long)n * a.img_stride + a.pair_stride + (long long)a.flip_chan[c] * a.chan_stride;
            for (int i = warp; i < RS; i += NW) {
                const int y = sr_lo + i;
                for (int j = lane; j < CS; j += 32) {
                    const int x = sc_lo + j;
                    float v0, v1;
                    if (a.net_is_f16) {
                        const __half *p = static_cast<const __half *>(a.net);
                        v0 = __half2float(p[base0 + (long long)y * a.w + x]);
                        v1 = __half2float(p[base1 + (long long)y * a.w + (a.w - 1 - x)]);
                    } else {
                        const float *p = static_cast<const float *>(a.net);
                        v0 = p[base0 + (long long)y * a.w + x];
                        v1 = p[base1 + (long long)y * a.w + (a.w - 1 - x)];
                    }
                    s0[i * r.cap_cs + j] = __fdiv_rn(__fadd_rn(v0, v1), 2.0f);
                }
            }
        }
        __syncthreads();
        // ---- pass 1: horizontal x stride on every source row of the tile, over the box's columns
        for (int i = warp; i < RS; i += NW) {
            const float *row = s0 + i * r.cap_cs - sc_lo;
            for (int X = lane; X < BW; X += 32) {
                const AxisTab &t = t1x[X];
                s1[i * r.cap_bw + X] = tap4(row[clampi(t.s, 0, a.w - 1)], row[clampi(t.s + 1, 0, a.w - 1)],
                                            row[clampi(t.s + 2, 0, a.w - 1)], row[clampi(t.s + 3, 0, a.w - 1)], t.c);
            }
        }
        __syncthreads();
        // ---- pass 2: vertical x stride -> the box of the up-sampled map (:143 / :152)
        for (int Y = warp; Y < BH; Y += NW) {
            const AxisTab &t = t1y[Y];
            const int o0 = (clampi(t.s, 0, a.h - 1) - sr_lo) * r.cap_bw, o1 = (clampi(t.s + 1, 0, a.h - 1) - sr_lo) * r.cap_bw;
            const int o2 = (clampi(t.s + 2, 0, a.h - 1) - sr_lo) * r.cap_bw, o3 = (clampi(t.s + 3, 0, a.h - 1) - sr_lo) * r.cap_bw;
            for (int X = lane; X < BW; X += 32) s2[Y * r.cap_bw + X] = tap4(s1[o0 + X], s1[o1 + X], s1[o2 + X], s1[o3 + X], t.c);
        }
        __syncthreads();
        // ---- warp with rotate_matrix_reverse (:144-146 / :153-155) into the footprint; taps outside the map read 0
        for (int yy = warp; yy < FH; yy += NW) {
            const int X0 = x0y[yy], Y0 = y0y[yy];
            for (int xx = lane; xx < FW; xx += 32) {
                int sx, sy;
                float wt[4];
                warp_tap(X0, Y0, adx[xx], bdx[xx], sx, sy, wt);
                const bool x0in = sx >= 0 && sx < r.Wp, x1in = sx + 1 >= 0 && sx + 1 < r.Wp;
                const bool y0in = sy >= 0 && sy < r.Hp, y1in = sy + 1 >= 0 && sy + 1 < r.Hp;
                const float *p = s2 + (sy - by_lo) * r.cap_bw + (sx - bx_lo);
                const float p00 = (y0in && x0in) ? p[0] : 0.0f, p01 = (y0in && x1in) ? p[1] : 0.0f;
                const float p10 = (y1in && x0in) ? p[r.cap_bw] : 0.0f, p11 = (y1in && x1in) ? p[r.cap_bw + 1] : 0.0f;
                sw[yy * r.cap_fw + xx] = tap4(p00, p01, p10, p11, wt);
            }
        }
        __syncthreads();
        // ---- pass 3: horizontal pass of the second resize (clamped to the cropped array)
        if (!identity) {
            for (int Y = warp; Y < FH; Y += NW) {
                const float *row = sw + Y * r.cap_fw - c_lo;
                for (int x = lane; x < tw; x += 32) {
                    const AxisTab &t = t2x[x];
                    s3[Y * TW + x] = tap4(row[clampi(t.s, 0, a.crop_w - 1)], row[clampi(t.s + 1, 0, a.crop_w - 1)],
                                          row[clampi(t.s + 2, 0, a.crop_w - 1)], row[clampi(t.s + 3, 0, a.crop_w - 1)], t.c);
                }
            }
            __syncthreads();
        }
        // ---- pass 4 + epilogue: vertical pass, / n in float32, float64 accumulation over the loop (:160-161)
        const bool is_heat = c < a.K;
        const size_t pbase = is_heat ? ((size_t)n * a.K + c) * plane : ((size_t)n * (a.n_out - a.K) + (c - a.K)) * plane;
        for (int y = warp; y < th; y += NW) {
            for (int x = lane; x < tw; x += 32) {
                float v;
                if (identity) {
                    v = sw[y * r.cap_fw + x];
                } else {
                    const AxisTab &t = t2y[y];
                    const float *col = s3 + x - y_lo * TW;
                    v = tap4(col[clampi(t.s, 0, a.crop_h - 1) * TW], col[clampi(t.s + 1, 0, a.crop_h - 1) * TW],
                             col[clampi(t.s + 2, 0, a.crop_h - 1) * TW], col[clampi(t.s + 3, 0, a.crop_h - 1) * TW], t.c);
                }
                const size_t o = pbase + (size_t)(oy0 + y) * a.W + (ox0 + x);
                const float part = __fdiv_rn(v, nf);  // float32 array / Python int -> float32
                if (a.n_scales == 1) {  // avg = 0.0 + part: exact, the float64 value is the float32 one
                    const float rv = (a.nan_scrub && part != part) ? 0.0f : part;
                    if (is_heat) a.heat[o] = rv;
                    else if (a.paf_is_f64) static_cast<double *>(a.paf)[o] = (double)rv;
                    else static_cast<float *>(a.paf)[o] = rv;
                } else {
                    double *acc = is_heat ? a.heat_acc : static_cast<double *>(a.paf);
                    double s = __dadd_rn(first ? 0.0 : acc[o], (double)part);
                    if (a.nan_scrub && s != s) s = 0.0;  // demo_image.py:179-180 scrubs after every item
                    acc[o] = s;
                    if (is_heat && last) a.heat[o] = (float)s;  // find_peaks: heatmap_avg.astype(np.float32)
                }
            }
        }
        __syncthreads();  // s0..s3 are reused by the next channel
    }
}

}  // namespace spg
