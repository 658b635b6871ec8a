/* oracle/aux_fft128.h -- TEST INFRASTRUCTURE (checker), not product code.
 *
 * 128-point forward complex FFT standing in for CMSIS-DSP
 *     arm_cfft_f32(&arm_cfft_sR_f32_len128, buffer, 0, 1)         (AudioSDRpreProcessor.cpp:88)
 *     arm_cmplx_mag_squared_f32(buffer, buffer, 128)               (AudioSDRpreProcessor.cpp:89)
 * CMSIS-DSP (ARM, shipped with Teensyduino 1.5x as arm_math.h / libarm_cortexM7lfsp_math) is NOT part of the reference
 * tree, so its exact butterfly order cannot be pinned here.  PARITY UNPINNED for the rounding of the FFT: this file
 * restates the published transform (X[k] = sum x[n] exp(-2 pi i n k / 128), natural-order output) as a radix-2
 * decimation-in-frequency network in float32 with one rounding per operation; any correct float32 FFT agrees with
 * it to a few ulp of the largest line.  Everything the reference computes FROM the spectrum (AudioSDRpreProcessor.cpp:
 * 91-118) consumes it only through threshold compares, and
 * tests/test_aux_oracle.py::test_detector_decisions_do_not_hinge_on_fft_rounding checks the decisions against a float64
 * DFT as well.  The CUDA kernel evaluates the identical operation network, so CUDA == this file bit for bit.
 * tests/test_emu_pp_edges.py and tests/test_gpu_pp_edges.py pin the kernel to this network on purpose, with blocks one
 * rounding away from each decision, while parity with CMSIS stays unpinned.
 *
 * Used by oracle/sdr_aux_oracle.c (the restatement) and by oracle/shim/arm_math.h (so that the host-compiled
 * reference in oracle/_ref/refaux calls the same transform).
 */
#ifndef ORACLE_AUX_FFT128_H
#define ORACLE_AUX_FFT128_H
#include <stdint.h>
#include <string.h>

#ifndef AUX_TABLES_INCLUDED
#define AUX_TABLES_INCLUDED
#include "aux_tables.inc"
#endif

static inline float aux_tw(int i) { float f; memcpy(&f, &AUX_FFT_TW[i], 4); return f; }

/* in place on 128 interleaved (re, im) pairs; output in natural order */
static inline void aux_cfft128_forward(float *buf) {
  for (int half = 64; half >= 1; half >>= 1) {
    const int step = 64 / half;
    for (int base = 0; base < 128; base += 2 * half) {
      for (int j = 0; j < half; j++) {
        float *a = buf + 2 * (base + j), *b = buf + 2 * (base + j + half);
        const float ar = a[0], ai = a[1], br = b[0], bi = b[1];
        const float tr = ar - br, ti = ai - bi;
        const float wr = aux_tw(2 * j * step), wi = aux_tw(2 * j * step + 1);
        a[0] = ar + br;
        a[1] = ai + bi;
        const float p0 = tr * wr, p1 = ti * wi, p2 = tr * wi, p3 = ti * wr;
        b[0] = p0 - p1;
        b[1] = p2 + p3;
      }
    }
  }
  for (int i = 0; i < 128; i++) { /* 7-bit reversal */
    int r = 0;
    for (int k = 0; k < 7; k++) r |= ((i >> k) & 1) << (6 - k);
    if (r > i) {
      float t0 = buf[2 * i], t1 = buf[2 * i + 1];
      buf[2 * i] = buf[2 * r]; buf[2 * i + 1] = buf[2 * r + 1];
      buf[2 * r] = t0; buf[2 * r + 1] = t1;
    }
  }
}

/* the same network for n = 256 (spectrum tap on the grabber's snapshot, sdr_grabber_spectrum): in place, natural order */
static inline float aux_tw256(int i) { float f; memcpy(&f, &AUX_FFT_TW256[i], 4); return f; }
static inline void aux_cfft256_forward(float *buf) {
  for (int half = 128; half >= 1; half >>= 1) {
    const int step = 128 / half;
    for (int base = 0; base < 256; base += 2 * half) {
      for (int j = 0; j < half; j++) {
        float *a = buf + 2 * (base + j), *b = buf + 2 * (base + j + half);
        const float ar = a[0], ai = a[1], br = b[0], bi = b[1];
        const float tr = ar - br, ti = ai - bi;
        const float wr = aux_tw256(2 * j * step), wi = aux_tw256(2 * j * step + 1);
        a[0] = ar + br;
        a[1] = ai + bi;
        const float p0 = tr * wr, p1 = ti * wi, p2 = tr * wi, p3 = ti * wr;
        b[0] = p0 - p1;
        b[1] = p2 + p3;
      }
    }
  }
  for (int i = 0; i < 256; i++) { /* 8-bit reversal */
    int r = 0;
    for (int k = 0; k < 8; k++) r |= ((i >> k) & 1) << (7 - k);
    if (r > i) {
      float t0 = buf[2 * i], t1 = buf[2 * i + 1];
      buf[2 * i] = buf[2 * r]; buf[2 * i + 1] = buf[2 * r + 1];
      buf[2 * r] = t0; buf[2 * r + 1] = t1;
    }
  }
}

/* dst[i] = re^2 + im^2, two products and one sum in float32; dst may be src (arm_cmplx_mag_squared_f32 semantics) */
static inline void aux_cmplx_mag_squared(const float *src, float *dst, uint32_t n) {
  for (uint32_t i = 0; i < n; i++) {
    const float re = src[2 * i], im = src[2 * i + 1];
    const float a = re * re, b = im * im;
    dst[i] = a + b;
  }
}
#endif
