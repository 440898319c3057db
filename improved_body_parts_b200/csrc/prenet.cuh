// prenet.cuh -- the pre-network stage: one scale of predict()'s loop before the forward pass (evaluate.py:98-116).
//
//   imageToTest        = cv2.resize(image, (0, 0), fx=scale, fy=scale, interpolation=cv2.INTER_CUBIC)   uint8 BGR
//   imageToTest_padded = padRightDownCorner(imageToTest, max_downsample, padValue)
//   input_img          = np.float32(imageToTest_padded / 255)
//   input_img          = cv2.warpAffine(input_img, getRotationMatrix2D((Hp / 2, Wp / 2), angle, 1), (0, 0))  angle != 0
//   pair               = [input_img, input_img[:, ::-1]]                                          [2][Hp][Wp][3]
//
// prenet_resize_kernel writes imageToTest_padded (uint8, handle workspace) once per scale; prenet_emit_kernel<ROT> turns
// it into one item's pair per angle.  The arithmetic is OpenCV's 8-bit generic INTER_CUBIC path without IPP, as
// restated -- and pinned to cv2 bit for bit -- by tests/prenet_port.py:
//   axis tables: f = (float)((d + 0.5) / fx - 0.5) (axis_entry), weights interpolateCubic(f - floor f) converted to
//     saturate_cast<short>(c 2048); taps floor(f) - 1 .. floor(f) + 2 clamped to the axis;
//   horizontal pass: exact int32 sums of u8 x short;
//   vertical pass: float32, b_k = (float)beta_k / 2048^2, S0 b0 + (S1 b1 + (S2 b2 + S3 b3)), rint, saturated -- except
//     the last (W 3) mod 8 values of each row, which OpenCV's vector loop does not reach: its scalar integer form
//     (sum S_k beta_k + 2^21) >> 22, saturated;
//   dsize == ssize: a plain copy.
// /255 is the 256-entry table (float)((double)u / 255); the warp is warp_affine.cuh's fixed-point bilinear path with
// border 0.  The translation unit is built with -fmad=false and spells out every *_rn operation.
#pragma once

#include <cassert>

#include "postnet.cuh"
#include "warp_affine.cuh"

namespace spg {

constexpr int kPreThreads = 256;
constexpr int kPreTW = 32;     // output columns of a resize tile
constexpr int kPreMaxTH = 32;  // output rows of a resize tile (the host lowers it for strong down-scales)
constexpr int kPreRows = 64;   // source rows of a tile's horizontal pass held in shared memory
constexpr int kPreVecLanes = 8;  // values per iteration of OpenCV's vertical vector loop (int16 lanes of 128 bits)

struct PrenetResizeArgs {
    const unsigned char *src;  // [h][row bytes] HWC, 3 channels, pixel stride 3
    long long src_row;         // bytes between source rows
    int h, w;                  // source size
    int H, W;                  // resized size (imageToTest)
    int Hp, Wp;                // padded size
    double sx, sy;             // 1 / fx, 1 / fy: cv2.resize's scale_x / scale_y
    int pad_value;
    int tile_h;                // output rows per CTA: the source rows of a tile fit kPreRows
    bool copy;                 // dsize == ssize
    unsigned char *dst;        // [Hp][Wp][3]
};

__device__ __forceinline__ int u8_axis_entry(int d, double scale, int beta[4]) {
    float c[4];
    const int s = axis_entry(d, scale, c);
    for (int k = 0; k < 4; k++) beta[k] = __float2int_rn(__fmul_rn(c[k], 2048.0f));  // saturate_cast<short>(c * 2048)
    return s;
}

__global__ void __launch_bounds__(kPreThreads) prenet_resize_kernel(PrenetResizeArgs a) {
    __shared__ int tx_s[kPreTW], tx_b[kPreTW][4], ty_s[kPreMaxTH], ty_b[kPreMaxTH][4];
    __shared__ int S[kPreRows * kPreTW * 3];  // horizontal pass of the tile's source rows, [row][x * 3 + c]
    const int tid = threadIdx.x;
    const int x0 = blockIdx.x * kPreTW, y0 = blockIdx.y * a.tile_h;
    const int tw = min(kPreTW, a.Wp - x0), th = min(a.tile_h, a.Hp - y0);
    const int rw = max(0, min(tw, a.W - x0)), rh = max(0, min(th, a.H - y0));  // the part of the tile inside imageToTest
    const int TW3 = kPreTW * 3, tw3 = tw * 3, rw3 = rw * 3;
    int r_lo = 0;
    if (!a.copy && rw > 0 && rh > 0) {
        if (tid < rw) tx_s[tid] = u8_axis_entry(x0 + tid, a.sx, tx_b[tid]);
        if (tid >= 64 && tid < 64 + rh) ty_s[tid - 64] = u8_axis_entry(y0 + tid - 64, a.sy, ty_b[tid - 64]);
        __syncthreads();
        r_lo = clampi(ty_s[0], 0, a.h - 1);
        const int RS = clampi(ty_s[rh - 1] + 3, 0, a.h - 1) - r_lo + 1;
        assert(RS <= kPreRows);
        // horizontal pass: exact integer sums, taps clamped per channel
        for (int e = tid; e < RS * rw3; e += kPreThreads) {
            const int i = e / rw3, j = e - i * rw3, x = j / 3, c = j - x * 3;
            const unsigned char *row = a.src + (long long)(r_lo + i) * a.src_row + c;
            int v = 0;
            for (int k = 0; k < 4; k++) v += (int)row[clampi(tx_s[x] + k, 0, a.w - 1) * 3] * tx_b[x][k];
            S[i * TW3 + j] = v;
        }
        __syncthreads();
    }
    const int vec_end = (a.W * 3) / kPreVecLanes * kPreVecLanes;  // flat row index where OpenCV's scalar tail starts
    const float scale = 1.0f / (2048.0f * 2048.0f);
    for (int e = tid; e < th * tw3; e += kPreThreads) {
        const int y = e / tw3, j = e - y * tw3;
        int v = a.pad_value;
        if (y < rh && j < rw3) {
            if (a.copy) {
                v = a.src[(long long)(y0 + y) * a.src_row + x0 * 3 + j];
            } else {
                int s[4];
                for (int k = 0; k < 4; k++) s[k] = S[(clampi(ty_s[y] + k, 0, a.h - 1) - r_lo) * TW3 + j];
                const int *beta = ty_b[y];
                if (x0 * 3 + j < vec_end) {  // VResizeCubicVec_32s8u: float32, no FMA, rint
                    float p[4];
                    for (int k = 0; k < 4; k++) p[k] = __fmul_rn(__int2float_rn(s[k]), __fmul_rn((float)beta[k], scale));
                    v = __float2int_rn(__fadd_rn(p[0], __fadd_rn(p[1], __fadd_rn(p[2], p[3]))));
                } else {                     // VResizeCubic + FixedPtCast<int, uchar, 22>
                    v = (s[0] * beta[0] + s[1] * beta[1] + s[2] * beta[2] + s[3] * beta[3] + (1 << 21)) >> 22;
                }
                v = clampi(v, 0, 255);
            }
        }
        a.dst[(long long)(y0 + y) * a.Wp * 3 + x0 * 3 + j] = (unsigned char)v;
    }
}

struct PrenetEmitArgs {
    const unsigned char *img;  // imageToTest_padded [Hp][Wp][3]
    int Hp, Wp;
    double m[6];               // ROT: destination -> source map of the warp (warpAffine's inverse of rotate_matrix)
    float *out;                // [2][Hp][Wp][3]: the item, then its mirror
};

// One row segment of kPreThreads pixels per CTA, one pixel per thread; the thread writes the pixel and its mirror.
template <bool ROT>
__global__ void __launch_bounds__(kPreThreads) prenet_emit_kernel(PrenetEmitArgs a) {
    __shared__ float lut[256];  // np.float32(u8 / 255)
    static_assert(kPreThreads == 256, "one table entry per thread");
    lut[threadIdx.x] = __double2float_rn(__ddiv_rn((double)threadIdx.x, 255.0));
    __syncthreads();
    const int y = blockIdx.y, x = blockIdx.x * kPreThreads + threadIdx.x;
    if (x >= a.Wp) return;
    float v[3];
    if (!ROT) {
        const unsigned char *p = a.img + ((long long)y * a.Wp + x) * 3;
        for (int c = 0; c < 3; c++) v[c] = lut[p[c]];
    } else {
        int adelta, bdelta, X0, Y0, sx, sy;
        float wt[4];
        warp_col(a.m, x, adelta, bdelta);
        warp_row(a.m, y, X0, Y0);
        warp_tap(X0, Y0, adelta, bdelta, sx, sy, wt);
        const bool x0in = sx >= 0 && sx < a.Wp, x1in = sx + 1 >= 0 && sx + 1 < a.Wp;
        const bool y0in = sy >= 0 && sy < a.Hp, y1in = sy + 1 >= 0 && sy + 1 < a.Hp;
        const unsigned char *p = a.img + ((long long)sy * a.Wp + sx) * 3;
        const long long row = (long long)a.Wp * 3;
        for (int c = 0; c < 3; c++) {
            const float p00 = (y0in && x0in) ? lut[p[c]] : 0.0f, p01 = (y0in && x1in) ? lut[p[3 + c]] : 0.0f;
            const float p10 = (y1in && x0in) ? lut[p[row + c]] : 0.0f, p11 = (y1in && x1in) ? lut[p[row + 3 + c]] : 0.0f;
            v[c] = tap4(p00, p01, p10, p11, wt);
        }
    }
    float *o0 = a.out + ((long long)y * a.Wp + x) * 3;
    float *o1 = a.out + (long long)a.Hp * a.Wp * 3 + ((long long)y * a.Wp + (a.Wp - 1 - x)) * 3;
    for (int c = 0; c < 3; c++) { o0[c] = v[c]; o1[c] = v[c]; }
}

}  // namespace spg
