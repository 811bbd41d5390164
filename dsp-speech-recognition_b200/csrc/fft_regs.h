// Register-resident FFT building blocks on packed frame pairs (shared by K1 and the pitch kernels).
// A cpx2 is one complex value for each of two frames: the .x halves belong to frame A, the .y halves to frame B,
// so every butterfly is one FADD2 / FMUL2 / FFMA2 on sm_100a.
#pragma once
#include "simt.h"

namespace dspfe {

struct cpx2 { float2 re, im; };  // one complex value for each of the two frames of a pair

DEVFN cpx2 cadd(cpx2 a, cpx2 b) { cpx2 r; r.re = f2add(a.re, b.re); r.im = f2add(a.im, b.im); return r; }
DEVFN cpx2 csub(cpx2 a, cpx2 b) { cpx2 r; r.re = f2sub(a.re, b.re); r.im = f2sub(a.im, b.im); return r; }
// a * (wr + i*wi), scalar twiddle shared by both frames
DEVFN cpx2 cmuls(cpx2 a, float wr, float wi) {
    cpx2 r;
    r.re = f2fmas(a.re, wr, f2muls(a.im, -wi));
    r.im = f2fmas(a.re, wi, f2muls(a.im, wr));
    return r;
}
DEVFN cpx2 cmul_negi(cpx2 a) { cpx2 r; r.re = a.im; r.im = f2neg(a.re); return r; }  // a * (-i)

// forward 4-point DFT (W4 = -i)
DEVFN void dft4(cpx2& a, cpx2& b, cpx2& c, cpx2& d) {
    cpx2 t0 = cadd(a, c), t1 = csub(a, c), t2 = cadd(b, d), t3 = cmul_negi(csub(b, d));
    a = cadd(t0, t2); c = csub(t0, t2); b = cadd(t1, t3); d = csub(t1, t3);
}

// forward 16-point DFT in registers, natural order in and out: X[k] = sum_n x[n] W16^{nk}
DEVFN void dft16(cpx2 (&x)[16]) {
    const float c1 = 0.92387953251128674f, s1 = 0.38268343236508977f, r2 = 0.70710678118654752f;
    // layer 1: for each n_b, DFT4 over n_a of x[4*n_a + n_b]; result k_a left at x[4*k_a + n_b]
#pragma unroll
    for (int nb = 0; nb < 4; ++nb) dft4(x[nb], x[4 + nb], x[8 + nb], x[12 + nb]);
    // twiddle W16^{n_b * k_a}
    x[5] = cmuls(x[5], c1, -s1);                                   // W^1
    { cpx2 t = x[6]; x[6].re = f2muls(f2add(t.re, t.im), r2); x[6].im = f2muls(f2sub(t.im, t.re), r2); }   // W^2
    x[7] = cmuls(x[7], s1, -c1);                                   // W^3
    { cpx2 t = x[9]; x[9].re = f2muls(f2add(t.re, t.im), r2); x[9].im = f2muls(f2sub(t.im, t.re), r2); }   // W^2
    x[10] = cmul_negi(x[10]);                                      // W^4
    { cpx2 t = x[11]; x[11].re = f2muls(f2sub(t.im, t.re), r2); x[11].im = f2muls(f2add(t.re, t.im), -r2); }  // W^6
    x[13] = cmuls(x[13], s1, -c1);                                 // W^3
    { cpx2 t = x[14]; x[14].re = f2muls(f2sub(t.im, t.re), r2); x[14].im = f2muls(f2add(t.re, t.im), -r2); }  // W^6
    x[15] = cmuls(x[15], -c1, s1);                                 // W^9
    // layer 2: for each k_a, DFT4 over n_b of x[4*k_a + n_b]; output k_b is X[k_a + 4*k_b]
#pragma unroll
    for (int ka = 0; ka < 4; ++ka) dft4(x[4 * ka], x[4 * ka + 1], x[4 * ka + 2], x[4 * ka + 3]);
    // x[4*k_a + k_b] now holds X[k_a + 4*k_b]: transpose the 4x4 register tile (pure renaming)
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = a + 1; b < 4; ++b) { cpx2 t = x[4 * a + b]; x[4 * a + b] = x[4 * b + a]; x[4 * b + a] = t; }
}

// 512-point complex FFT of a packed frame pair, one warp, 16 complex values per lane, 512 = 16 x 2 x 16:
//   element n = 32*n1 + 16*q + n2'  ->  lane 16*q + n2', register n1   (natural order: n = 32*register + lane)
// radix-16 in registers over n1, radix-2 across the two half-warps, twiddle, a 32x16 transpose over the warp through shared
// memory, radix-16 in registers over n2'.  With the radix-2 stage in the middle the output lands in the SAME layout
// (k = k1 + 16*kq + 32*k2' -> lane 16*kq + k1, register k2'), so one routine serves every transform of the chain and all
// pointwise tables are in natural order.  Forward DFT sum x[n] W512^{nk}; the unnormalised inverse is the same routine
// between two conjugations.
DEVFN cpx2 shfl_xor_c(cpx2 a, int m) {
    cpx2 r;
    r.re.x = simt::shfl32_xor(a.re.x, m); r.re.y = simt::shfl32_xor(a.re.y, m);
    r.im.x = simt::shfl32_xor(a.im.x, m); r.im.y = simt::shfl32_xor(a.im.y, m);
    return r;
}

// The radix-2 stage exchanges half the registers: b[kq][k1] = a0[k1] + (-1)^kq W32^k1 a1[k1] needs both half-warps' a at
// k1, so lane (q, n2') takes the butterflies of k1 = 8q + j, j < 8, and receives one value per j from lane (1 - q, n2'):
// q = 0 keeps a0[j] and sends a0[8 + j], q = 1 keeps W32^{8+j} a1[8 + j] and sends W32^j a1[j].  Each output is the same
// single rounding of the same two operands as a full exchange would give; q = 1 forms kp - r = -b[1] exactly and its
// twiddle carries the sign.  Afterwards register r of lane (q, n2') holds (kq, k1) = (r >> 3, 8q + (r & 7)).
// W32^k1 comes from immediates.  tws: [r*32 + lane] = W512^{n2' (k1 + 16 kq)} of that (kq, k1), negated for q = kq = 1
// (fill_fft512_twiddles).
// scr: kWarpScr float2 owned by the warp: the 32 x 16 tile, row 16 kq + k1 at a pitch of 17 float2.  Writes put a half-warp
// on 16 consecutive float2 of one row, reads a lane on its own row at column n2: row * 17 + n2 = row + n2 (mod 16) is
// distinct over each half-warp, so both 64-bit phases run without bank conflicts.
DEVFN void fft512(cpx2 (&x)[16], float2* scr, const float2* tws, int lane) {
    dft16(x);                                                   // over n1 -> k1
    const int q = lane >> 4;
    const float kC[16] = {1.0f, 0.98078528f, 0.923879533f, 0.831469612f, 0.707106781f, 0.555570233f, 0.382683432f, 0.195090322f, 6.123234e-17f, -0.195090322f, -0.382683432f, -0.555570233f, -0.707106781f, -0.831469612f, -0.923879533f, -0.98078528f};
    const float kS[16] = {-0.0f, -0.195090322f, -0.382683432f, -0.555570233f, -0.707106781f, -0.831469612f, -0.923879533f, -0.98078528f, -1.0f, -0.98078528f, -0.923879533f, -0.831469612f, -0.707106781f, -0.555570233f, -0.382683432f, -0.195090322f};
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const cpx2 us = cmuls(x[j], kC[j], kS[j]), uk = cmuls(x[8 + j], kC[8 + j], kS[8 + j]);   // W32^k1 a1[k1], taken on q = 1 only
        cpx2 snd, kp;
        snd.re = q ? us.re : x[8 + j].re; snd.im = q ? us.im : x[8 + j].im;
        kp.re = q ? uk.re : x[j].re; kp.im = q ? uk.im : x[j].im;
        const cpx2 r = shfl_xor_c(snd, 16);
        const float2 t0 = tws[j * 32 + lane], t1 = tws[(8 + j) * 32 + lane];
        x[j] = cmuls(cadd(kp, r), t0.x, t0.y);
        x[8 + j] = cmuls(csub(kp, r), t1.x, t1.y);
    }
    float2* wr = scr + 8 * q * 17 + (lane & 15);                // row 16 (r >> 3) + 8q + (r & 7), column n2'
    const float2* rd = scr + lane * 17;                         // row 16 kq + k1 = lane
#pragma unroll
    for (int r = 0; r < 16; ++r) wr[(16 * (r >> 3) + (r & 7)) * 17] = x[r].re;
    simt::warp_sync();
#pragma unroll
    for (int n2 = 0; n2 < 16; ++n2) x[n2].re = rd[n2];
    simt::warp_sync();
#pragma unroll
    for (int r = 0; r < 16; ++r) wr[(16 * (r >> 3) + (r & 7)) * 17] = x[r].im;
    simt::warp_sync();
#pragma unroll
    for (int n2 = 0; n2 < 16; ++n2) x[n2].im = rd[n2];
    simt::warp_sync();
    dft16(x);                                                   // over n2' -> k2'
}

}  // namespace dspfe
