/* CPU oracle of cv2.remap on integer images -- test infrastructure only, like fd_oracle.c.
 *
 * The reference warps a neighbour slice with cv2.remap(reference, map_xy, None, INTER_LINEAR, BORDER_REPLICATE)
 * (src/flowdenoising.py:55-63). With an integer volume the image is 8U, 16U or 16S and OpenCV interpolates in that
 * type (imgwarp.cpp, remapBilinear):
 *   map        the float32 (H, W, 2) map is quantised as for float images: sx = cvRound(X * 32), ix = sx >> 5,
 *              fraction index (sy & 31) * 32 + (sx & 31) into the 1/32-px tables;
 *   8U         fixed point: table entry k = saturate_cast<short>(wy * wx * 32768) for the four taps, corrected so that the
 *              four sum to 32768 (initInterTab2D), result (sum w_k * p_k + 2^14) >> 15, saturated;
 *   16U / 16S  float32 weights wy * wx, the four products summed in tap order, then cvRound and saturate.
 * Taps outside the image take the nearest edge pixel (BORDER_REPLICATE).
 * Checked exhaustively against cv2 4.13.0 by tests/test_integer_volume_oracle.py.
 */
#include <math.h>
#include <stdint.h>
#include <string.h>

#define FDO_API __attribute__((visibility("default")))

enum { DT_U8 = 1, DT_U16 = 3, DT_S16 = 4 };   /* FDN_DTYPE_* of include/fdn_b200.h */

static short g_itab[1024][4];
static float g_ftab[1024][4];
static int g_init = 0;

static int clampi(int v, int lo, int hi) { return v < lo ? lo : v > hi ? hi : v; }

static void init_tables(void)
{
    if (g_init) return;
    for (int i = 0; i < 32; i++)
        for (int j = 0; j < 32; j++) {
            const float ty = i * (1.f / 32), tx = j * (1.f / 32);
            const float vy[2] = {1.f - ty, ty}, vx[2] = {1.f - tx, tx};
            short* it = g_itab[i * 32 + j];
            float* ft = g_ftab[i * 32 + j];
            int isum = 0;
            for (int k1 = 0; k1 < 2; k1++)
                for (int k2 = 0; k2 < 2; k2++) {
                    const float v = vy[k1] * vx[k2];
                    ft[k1 * 2 + k2] = v;
                    it[k1 * 2 + k2] = (short)clampi((int)lrintf(v * 32768.f), -32768, 32767);
                    isum += it[k1 * 2 + k2];
                }
            if (isum != 32768) {
                /* Only ax = ay = 0 gets here (32768 saturates to 32767, the sum falls 1 short). initInterTab2D looks for
                 * the smallest / largest tap in the 2x2 block that starts at tap (ksize/2, ksize/2): with ksize = 2 that
                 * is tap 3 (y1x1) and three places past this entry, still zero when it is built, so the missing unit
                 * lands on tap 3: {32767, 0, 0, 1}. (For 8-bit pixels every variant rounds to the same result.) */
                it[3] = (short)(it[3] - (isum - 32768));
            }
        }
    g_init = 1;
}

/* The 8U table as OpenCV builds it: out[1024][4] (entry (sy & 31) * 32 + (sx & 31), taps y0x0, y0x1, y1x0, y1x1). */
FDO_API void fdo_remap_table_8u(short* out)
{
    init_tables();
    memcpy(out, g_itab, sizeof g_itab);
}

/* cv2.remap(src, map, None, INTER_LINEAR, BORDER_REPLICATE) of a dense (H, W) image of dtype DT_U8 / DT_U16 / DT_S16;
 * map: (H, W, 2) float32 absolute coordinates (x first), dst: (H, W) of the same dtype. Returns 0, or -1 for a dtype
 * cv2.remap rejects. */
FDO_API int fdo_remap_typed(const void* src, int dtype, int H, int W, const float* map, void* dst)
{
    if (dtype != DT_U8 && dtype != DT_U16 && dtype != DT_S16) return -1;
    init_tables();
    for (int y = 0; y < H; y++)
        for (int x = 0; x < W; x++) {
            const size_t o = (size_t)y * W + x;
            const int sx = (int)lrintf(map[2 * o] * 32.f), sy = (int)lrintf(map[2 * o + 1] * 32.f);
            const int a = (sy & 31) * 32 + (sx & 31);
            const int ix = clampi(sx >> 5, -32768, 32767), iy = clampi(sy >> 5, -32768, 32767);
            const int x0 = clampi(ix, 0, W - 1), x1 = clampi(ix + 1, 0, W - 1);
            const int y0 = clampi(iy, 0, H - 1), y1 = clampi(iy + 1, 0, H - 1);
            const size_t i00 = (size_t)y0 * W + x0, i01 = (size_t)y0 * W + x1, i10 = (size_t)y1 * W + x0,
                         i11 = (size_t)y1 * W + x1;
            if (dtype == DT_U8) {
                const uint8_t* s = (const uint8_t*)src;
                const short* w = g_itab[a];
                const int v = s[i00] * w[0] + s[i01] * w[1] + s[i10] * w[2] + s[i11] * w[3];
                ((uint8_t*)dst)[o] = (uint8_t)clampi((v + (1 << 14)) >> 15, 0, 255);
            } else {
                const float* w = g_ftab[a];
                float p0, p1, p2, p3;
                if (dtype == DT_U16) {
                    const uint16_t* s = (const uint16_t*)src;
                    p0 = s[i00]; p1 = s[i01]; p2 = s[i10]; p3 = s[i11];
                } else {
                    const int16_t* s = (const int16_t*)src;
                    p0 = s[i00]; p1 = s[i01]; p2 = s[i10]; p3 = s[i11];
                }
                float t = p0 * w[0];
                t = t + p1 * w[1];
                t = t + p2 * w[2];
                t = t + p3 * w[3];
                const int r = (int)lrintf(t);
                if (dtype == DT_U16) ((uint16_t*)dst)[o] = (uint16_t)clampi(r, 0, 65535);
                else ((int16_t*)dst)[o] = (int16_t)clampi(r, -32768, 32767);
            }
        }
    return 0;
}
