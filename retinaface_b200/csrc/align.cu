// align.cu -- see align.cuh.  Compiled with -fmad=false: the FP64 inversion and the fixed-point coordinates restate OpenCV's
// double arithmetic operation by operation, and a contracted multiply-add would round differently.
#include <mutex>

#include "align.cuh"

namespace rf {

namespace {

constexpr int INTER_BITS = 5, INTER_TAB = 1 << INTER_BITS;   // 5-bit fractions, 32 x 32 weight table
constexpr int AB_BITS = 10, AB_SCALE = 1 << AB_BITS;         // source coordinates in 1/1024 pixels
constexpr int COEF_BITS = 15;                                // weights in 1/32768
constexpr int ALIGN_THREADS = 384;   // one CTA per crop: 3,136 four-pixel groups of a 112^2 crop, ~8 per thread (512 spills)

__constant__ short4 c_wtab[INTER_TAB * INTER_TAB];           // (y0x0, y0x1, y1x0, y1x1) per fy * 32 + fx

// initInterTab2D(INTER_LINEAR, fixpt = true): float weights (1 - f, f) per axis, products rounded to 1/32768 and saturated to
// short; where the four do not sum to 32768 (only fx = fy = 0: 32768 saturates to 32767) OpenCV fixes the sum on the tap its
// search settles on -- for a 2 x 2 kernel the search starts at tap (1, 1) and only compares entries past this cell, which are
// still zero, so the correction lands on tap (1, 1).
void build_weight_table(short4 *tab) {
    float lin[INTER_TAB][2];
    for (int i = 0; i < INTER_TAB; i++) {
        const float x = i * (1.f / INTER_TAB);
        lin[i][0] = 1.f - x;
        lin[i][1] = x;
    }
    for (int i = 0; i < INTER_TAB; i++)
        for (int j = 0; j < INTER_TAB; j++) {
            int w[4], sum = 0;
            for (int k1 = 0; k1 < 2; k1++)
                for (int k2 = 0; k2 < 2; k2++) {
                    const float v = lin[i][k1] * lin[j][k2];
                    int r = (int)lrintf(v * (1 << COEF_BITS));
                    r = r < -32768 ? -32768 : (r > 32767 ? 32767 : r);
                    sum += w[2 * k1 + k2] = r;
                }
            w[3] -= sum - (1 << COEF_BITS);
            tab[i * INTER_TAB + j] = make_short4((short)w[0], (short)w[1], (short)w[2], (short)w[3]);
        }
}

// Forward similarity from the 5 image-pixel landmarks to the template: closed-form least squares of [a -b; b a] p + t = q
// (Umeyama without reflection), FP64.
__device__ void similarity_fit(const double px[5], const double py[5], const double qx[5], const double qy[5], double M[6]) {
    double pmx = 0, pmy = 0, qmx = 0, qmy = 0;
    for (int k = 0; k < 5; k++) { pmx += px[k]; pmy += py[k]; qmx += qx[k]; qmy += qy[k]; }
    pmx /= 5; pmy /= 5; qmx /= 5; qmy /= 5;
    double den = 0, sa = 0, sb = 0;
    for (int k = 0; k < 5; k++) {
        const double ux = px[k] - pmx, uy = py[k] - pmy, vx = qx[k] - qmx, vy = qy[k] - qmy;
        den += ux * ux + uy * uy;
        sa += ux * vx + uy * vy;
        sb += ux * vy - uy * vx;
    }
    const double a = den != 0 ? sa / den : 0.0, b = den != 0 ? sb / den : 0.0;
    M[0] = a; M[1] = -b; M[2] = qmx - (a * pmx - b * pmy);
    M[3] = b; M[4] = a;  M[5] = qmy - (b * pmx + a * pmy);
}

// cv::warpAffine's inversion of the forward map, in its operation order (imgwarp.cpp)
__device__ void invert_affine(double M[6]) {
    double D = M[0] * M[4] - M[1] * M[3];
    D = D != 0 ? 1. / D : 0;
    const double A11 = M[4] * D, A22 = M[0] * D;
    M[0] = A11; M[1] *= -D;
    M[3] *= -D; M[4] = A22;
    const double b1 = -M[0] * M[2] - M[1] * M[5];
    const double b2 = -M[3] * M[2] - M[4] * M[5];
    M[2] = b1; M[5] = b2;
}

// One destination pixel from its fixed-point source coordinate (X, Y in 1/32 pixels): remapBilinear with BORDER_CONSTANT 0.
__device__ __forceinline__ void sample(const AlignSrc &s, int X, int Y, const short4 *tab, int v[3]) {
    const int sx = min(max(X >> INTER_BITS, -32768), 32767), sy = min(max(Y >> INTER_BITS, -32768), 32767);   // saturate_cast<short>
    const short4 w = tab[((Y & (INTER_TAB - 1)) << INTER_BITS) | (X & (INTER_TAB - 1))];
    const int wt[4] = {w.x, w.y, w.z, w.w};
    int acc[3] = {0, 0, 0};
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int tx = sx + (k & 1), ty = sy + (k >> 1);
        if ((unsigned)tx < (unsigned)s.w && (unsigned)ty < (unsigned)s.h) {
            const uint8_t *p = s.ptr + (size_t)ty * s.row_bytes + tx * 3;
            acc[0] += p[0] * wt[k]; acc[1] += p[1] * wt[k]; acc[2] += p[2] * wt[k];
        }
    }
#pragma unroll
    for (int c = 0; c < 3; c++) v[c] = min(max((acc[c] + (1 << (COEF_BITS - 1))) >> COEF_BITS, 0), 255);
}

// grid (max_crops, n): one CTA per crop slot; slots past the image's face count exit at once.
__global__ void __launch_bounds__(ALIGN_THREADS) k_align(const __grid_constant__ AlignArgs a) {
    const int img = blockIdx.y, slot = blockIdx.x;
    if (slot >= min(a.counts[img], a.max_crops)) return;
    __shared__ short4 s_tab[INTER_TAB * INTER_TAB];
    __shared__ int s_adelta[ALIGN_MAX_CROP], s_bdelta[ALIGN_MAX_CROP], s_x0[ALIGN_MAX_CROP], s_y0[ALIGN_MAX_CROP];
    __shared__ double s_m[6];
    AlignSrc src;
    if (a.table) src = a.table[img];
    else { src = a.uniform; src.ptr += (size_t)img * a.uniform_stride; }
    const size_t crop_px = (size_t)a.crop_w * a.crop_h, crop_id = (size_t)img * a.max_crops + slot;

    if (threadIdx.x == 0) {
        const rf_face &f = a.dets[(size_t)img * a.max_faces + slot].face;
        double px[5], py[5], qx[5], qy[5], M[6];
        for (int k = 0; k < 5; k++) {
            px[k] = __fmul_rn(f.lx[k], src.scale);
            py[k] = __fmul_rn(f.ly[k], src.scale);
            qx[k] = a.dst_x[k];
            qy[k] = a.dst_y[k];
        }
        similarity_fit(px, py, qx, qy, M);
        if (a.affine)
            for (int k = 0; k < 6; k++) a.affine[crop_id * 6 + k] = M[k];
        invert_affine(M);
        for (int k = 0; k < 6; k++) s_m[k] = M[k];
    }
    for (int i = threadIdx.x; i < INTER_TAB * INTER_TAB; i += ALIGN_THREADS) s_tab[i] = c_wtab[i];
    __syncthreads();
    // per column / per row parts of the source coordinate (WarpAffineInvoker): the pixel loop below is integer only
    const int round_delta = AB_SCALE / INTER_TAB / 2;
    for (int x = threadIdx.x; x < a.crop_w; x += ALIGN_THREADS) {
        s_adelta[x] = __double2int_rn(s_m[0] * x * AB_SCALE);
        s_bdelta[x] = __double2int_rn(s_m[3] * x * AB_SCALE);
    }
    for (int y = threadIdx.x; y < a.crop_h; y += ALIGN_THREADS) {
        s_x0[y] = __double2int_rn((s_m[1] * y + s_m[2]) * AB_SCALE) + round_delta;
        s_y0[y] = __double2int_rn((s_m[4] * y + s_m[5]) * AB_SCALE) + round_delta;
    }
    __syncthreads();

    constexpr int SH = AB_BITS - INTER_BITS;
    if (a.layout == RF_CROP_U8_BGR) {
        uint8_t *out = reinterpret_cast<uint8_t *>(a.crops) + crop_id * crop_px * 3;
        if ((a.crop_w & 3) == 0 && (reinterpret_cast<uintptr_t>(a.crops) & 3) == 0) {
            // 4 consecutive pixels = 12 bytes = three aligned 32-bit stores (crop rows and crops are multiples of 12 bytes)
            const int qw = a.crop_w >> 2;
            for (int q = threadIdx.x; q < qw * a.crop_h; q += ALIGN_THREADS) {
                const int y = q / qw, x4 = (q - y * qw) << 2;
                unsigned char px[12];
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    int v[3];
                    sample(src, (s_x0[y] + s_adelta[x4 + k]) >> SH, (s_y0[y] + s_bdelta[x4 + k]) >> SH, s_tab, v);
                    px[3 * k] = (unsigned char)v[0]; px[3 * k + 1] = (unsigned char)v[1]; px[3 * k + 2] = (unsigned char)v[2];
                }
                uint32_t *o = reinterpret_cast<uint32_t *>(out + ((size_t)y * a.crop_w + x4) * 3);
                o[0] = px[0] | (px[1] << 8) | (px[2] << 16) | ((uint32_t)px[3] << 24);
                o[1] = px[4] | (px[5] << 8) | (px[6] << 16) | ((uint32_t)px[7] << 24);
                o[2] = px[8] | (px[9] << 8) | (px[10] << 16) | ((uint32_t)px[11] << 24);
            }
        } else {
            for (int i = threadIdx.x; i < (int)crop_px; i += ALIGN_THREADS) {
                const int y = i / a.crop_w, x = i - y * a.crop_w;
                int v[3];
                sample(src, (s_x0[y] + s_adelta[x]) >> SH, (s_y0[y] + s_bdelta[x]) >> SH, s_tab, v);
                out[(size_t)i * 3] = (uint8_t)v[0]; out[(size_t)i * 3 + 1] = (uint8_t)v[1]; out[(size_t)i * 3 + 2] = (uint8_t)v[2];
            }
        }
    } else {
        // RGB planes of (v - mean) * scale, one rounding to FP16
        __half *out = reinterpret_cast<__half *>(a.crops) + crop_id * crop_px * 3;
        for (int i = threadIdx.x; i < (int)crop_px; i += ALIGN_THREADS) {
            const int y = i / a.crop_w, x = i - y * a.crop_w;
            int v[3];
            sample(src, (s_x0[y] + s_adelta[x]) >> SH, (s_y0[y] + s_bdelta[x]) >> SH, s_tab, v);
#pragma unroll
            for (int c = 0; c < 3; c++) out[(size_t)c * crop_px + i] = __float2half_rn(__fmul_rn(__fsub_rn((float)v[2 - c], a.mean), a.scale));
        }
    }
}

// the weight table goes to each device's __constant__ once (synchronously, so no launch on any stream can overtake it)
cudaError_t align_init() {
    static std::mutex mu;
    static bool done[64] = {false};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lock(mu);
    if (dev < 64 && done[dev]) return cudaSuccess;
    static short4 tab[INTER_TAB * INTER_TAB];
    static bool built = false;
    if (!built) { build_weight_table(tab); built = true; }
    if ((e = cudaMemcpyToSymbol(c_wtab, tab, sizeof tab)) != cudaSuccess) return e;
    if (dev < 64) done[dev] = true;
    return cudaSuccess;
}

}  // namespace

cudaError_t launch_align(const AlignArgs &a, int n, cudaStream_t s) {
    if (n <= 0 || a.max_crops <= 0) return cudaSuccess;
    cudaError_t e = align_init();
    if (e != cudaSuccess) return e;
    k_align<<<dim3(a.max_crops, n), ALIGN_THREADS, 0, s>>>(a);
    return cudaGetLastError();
}

}  // namespace rf
