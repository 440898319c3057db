// warp_affine.cuh -- the fixed-point coordinates and bilinear weights of OpenCV's warpAffine (INTER_LINEAR), shared by
// the warp of the network input (prenet.cuh) and the warp of the maps back (postnet_rot.cuh).
//
// imgproc/src/imgwarp.cpp, as restated -- and pinned to cv2 bit for bit -- by tests/rotation_port.py: with the
// destination -> source map m[6] (the host inverts the matrix in float64 as warpAffine does),
//   adelta[x] = rint(m0 x 1024), bdelta[x] = rint(m3 x 1024), X0(y) = rint((m1 y + m2) 1024) + 16,
//   Y0(y) = rint((m4 y + m5) 1024) + 16 (AB_BITS = 10, round_delta = 16, round half to even);
//   X = (X0 + adelta) >> 5, Y = (Y0 + bdelta) >> 5 (INTER_BITS = 5); integer tap (Y >> 5, X >> 5);
//   weights the float32 products of 1 - t and t with t = (Y & 31) / 32, (X & 31) / 32.
// The caller sums p00 w00 + p01 w01 + p10 w10 + p11 w11 left to right (tap4), taps outside the source reading 0.
#pragma once

namespace spg {

// the per-column half of the fixed-point source coordinate
__device__ __forceinline__ void warp_col(const double m[6], int x, int &adelta, int &bdelta) {
    adelta = __double2int_rn(__dmul_rn(__dmul_rn(m[0], (double)x), 1024.0));
    bdelta = __double2int_rn(__dmul_rn(__dmul_rn(m[3], (double)x), 1024.0));
}

// the per-row half, round_delta included
__device__ __forceinline__ void warp_row(const double m[6], int y, int &X0, int &Y0) {
    X0 = __double2int_rn(__dmul_rn(__dadd_rn(__dmul_rn(m[1], (double)y), m[2]), 1024.0)) + 16;
    Y0 = __double2int_rn(__dmul_rn(__dadd_rn(__dmul_rn(m[4], (double)y), m[5]), 1024.0)) + 16;
}

// integer tap (sy, sx) of the pixel and its four weights (w00, w01, w10, w11)
__device__ __forceinline__ void warp_tap(int X0, int Y0, int adelta, int bdelta, int &sx, int &sy, float wt[4]) {
    const int X = (X0 + adelta) >> 5, Y = (Y0 + bdelta) >> 5;
    sx = X >> 5; sy = Y >> 5;
    const float fx = __fmul_rn((float)(X & 31), 0.03125f), fy = __fmul_rn((float)(Y & 31), 0.03125f);
    const float gx = __fsub_rn(1.0f, fx), gy = __fsub_rn(1.0f, fy);
    wt[0] = __fmul_rn(gy, gx); wt[1] = __fmul_rn(gy, fx); wt[2] = __fmul_rn(fy, gx); wt[3] = __fmul_rn(fy, fx);
}

}  // namespace spg
