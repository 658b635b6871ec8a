/* sdr_types.h -- PODs shared by the host side (sdr_host.cpp) and the kernels (sdr_kernel.cu).
 *
 * HBM layout
 * ----------
 * state   : float/uint32 words, CHANNEL-FASTEST:  word w of channel c is state[w * ch_stride + c].
 *           A warp whose 32 lanes own 32 consecutive channels therefore touches one 128-byte line per
 *           state word.  The state IS the checkpoint: everything a channel carries from block to block.
 * cfg     : one SdrChanCfg per channel (array of structs; read once per launch per role).
 * groups  : one SdrGroup per CTA: 32 channel ids of one pipeline class (-1 = empty lane) and their plane rows.
 * planes  : caller-owned I/Q/audio, channel-major (include/sdr_batch.h).
 */
#ifndef SDR_TYPES_H
#define SDR_TYPES_H
#include <stdint.h>

#define SDR_LANES 32    /* channels per group (one warp lane each) */
#define SDR_TMAX 32     /* longest pipeline tile in samples (a launch's tile length is SdrLay::T: 32, 16 or 8; 128 / T tiles = one reference block) */
#define SDR_STAGES 14   /* pipeline stage ids (sdr_lay.h); a launch runs the subset its bucket needs, one warp each */
#define SDR_BAR_W 32    /* hand-over barriers per stage: stage s signals tile t on barrier (s, t % SDR_BAR_W) */
#define SDR_MAX_DEPS 4  /* hand-over rules per stage */
#define SDR_HQ_MIRROR 7 /* rows of the Hilbert Q ring repeated behind its end (sdr_pipeline.cuh, hq_at) */

/* ---- per-channel state words (reference member it stands for) ---- */
enum {
  W_IF_I = 0,        /* 16: _IFfilterStateI        H:191  {x1,x2,y1,y2} x 4 stages */
  W_IF_Q = 16,       /* 16: _IFfilterStateQ        H:192 */
  W_IMG_I = 32,      /* 16: _AMimage_stateI        H:193 */
  W_IMG_Q = 48,      /* 16: _AMimage_stateQ        H:194 */
  W_AUD = 64,        /* 16: _audio_filter_state    H:195 */
  W_PH_SSB = 80,     /* phase_SSB                  C:43 */
  W_PH_AM = 81,      /* phase_AM                   C:44 */
  W_AGC_GAIN = 82,   /* _agc_gain                  H:217 */
  W_AGC_OLD = 83,    /* _old_absVal                H:227 */
  W_AGC_HANG = 84,   /* _agc_hang_counter (u32)    H:229 */
  W_AGC_ACTIVE = 85, /* _agc_is_active (u32)       H:230 */
  W_AGC_CARRIER = 86,/* _agc_AMcarrierLevel        H:210 */
  W_SAM_YRE = 87,    /* yReal (function static)    C:690 */
  W_SAM_YIM = 88,    /* yImag                      C:691 */
  W_SAM_PREV = 89,   /* prev_phase_err_filt        C:692 */
  W_SAM_D0 = 90,     /* delay0                     H:270 */
  W_SAM_D1 = 91,     /* delay1 */
  W_SAM_PHASE = 92,  /* phase_est                  H:271 */
  W_SAM_FREQ = 93,   /* _PLLfreq                   H:273 */
  W_SAM_LOCKED = 94, /* _SAM_PLL_isLocked (u32)    H:274 */
  W_NB_AVG = 95,     /* _nb_AvgMag                 H:242 */
  W_NB_HIT = 96,     /* _nb_impulseDetected (u32)  H:246 */
  W_HQ = 128,        /* 256: the last 256 down-converted Q samples, oldest first (bufferQ, C:42) */
  W_HI = 384,        /* 128: the last 128 down-converted I samples (bufferI, C:41) */
  W_ALS_C = 512,     /* 128: _als_coeffs           H:202 */
  W_ALS_H = 640,     /* 128: the last 128 ALS inputs (_als_in[0..127] after the shift, H:201) */
  W_NB_MASK = 768,   /* 96 words = 384 byte codes: _mask, block slot (abs_block % 3), H:237 */
  W_NB_RING = 864,   /* 3 x 384: _BufferI, _BufferQ (H:235-236) and the envelope sqrt(I^2+Q^2) of every ring sample
                        (computed once on arrival instead of at each of its two scans), 3 block slots of 128, slot = abs_block % 3 */
  SDR_STATE_WORDS = 2016
};

/* noise-blanker mask codes (byte) -> value; code 0 must be 1.0 so that zeroed state == initBlanker() */
enum { MK_ONE = 0, MK_ZERO = 1, MK_933 = 2, MK_750 = 3, MK_500 = 4, MK_250 = 5, MK_067 = 6 };

/* ---- per-channel device configuration (resolved on the host from the setter shadow) ---- */
enum {
  CF_NB = 1u, CF_AUD = 2u, CF_AGC = 4u, CF_ALS = 8u, CF_ALS_NOTCH = 16u, CF_ALS_ADAPT = 32u, CF_MUTED = 64u,
  GF_LUT_GLOBAL = 0x10000u /* group summary only: some lane's AGC table is not among the 4 staged ones */
};
typedef struct {
  int32_t mode;            /* SDR_LSB..SDR_WSPR */
  uint32_t flags;          /* CF_* */
  float in_gain_i, in_gain_q, out_gain;
  float ssb_phase_inc;     /* (-_freq_shift) * (twoPI / fs), float ops as H:510 */
  int32_t if_set;          /* index into the IF coefficient sets {SSB, CW, WSPR, AM} */
  int32_t aud_set;         /* index into the audio sets (SDR_AUDIO_AM..SDR_AUDIO_3300) */
  float agc_a_att, agc_b_att, agc_a_rel, agc_b_rel, agc_static_gain;
  uint32_t agc_hang_count;
  int32_t agc_lut;         /* index into the handle's table of distinct 130-entry AGC tables */
  float nb_thr;
  int32_t als_m, als_delay;
  float als_lambda;
  uint32_t pad;
} SdrChanCfg;

/* ---- pipeline classes ---- */
enum { CLS_SSB = 0 /* LSB USB CW_LSB CW_USB WSPR: NCO + Hilbert */, CLS_ENV = 1 /* AM SAM: PLL + envelope */,
       CLS_ALS = 2 /* not a channel class: the plan of the ALS + output post-pass of a large bucket (sdr_lay.h, lay_build_als) */ };

#define SDR_LUT_SLOTS 4
typedef struct {
  int32_t cls;
  uint32_t feat;                 /* OR of the lanes' CF_* flags */
  int32_t cid[SDR_LANES];        /* channel id per lane, -1 = empty */
  int32_t lut_ids[SDR_LUT_SLOTS];/* up to 4 distinct AGC tables of this group, staged in shared memory (-1 = unused) */
  uint8_t lut_slot[SDR_LANES];   /* per lane: slot in lut_ids, or 255 = read the table from global memory */
  int32_t row[SDR_LANES];        /* per lane: the channel's row in the call's I/Q/audio planes and record columns (-1 = empty).
                                    Equal to cid in a call on every channel; the position of cid in the id list of a subset call */
} SdrGroup;

/* ---- constant tables in device memory ---- */
typedef struct {
  float if_sets[4][20];
  float aud_sets[10][20];
  float am_image[20];
  float hilbert[64];
  float sine[260];
  float pk_consts[8];      /* {1,1,-1,-1,-0,-0}: multiplicands / addends of the packed FMA forms, deliberately run-time data (sdr_pipeline.cuh, PkConst) */
} SdrTables;

/* ---- one hand-over rule: before tile t a stage waits until stage `stage` has finished tile t + k (kind 0) or the last tile
 * of t's block, t | (tpb - 1) (kind 1); tiles below 0 never block.  Built by lay_build() (sdr_lay.h). */
typedef struct { int8_t stage, kind; int16_t k; } SdrDep; /* `stage`: a barrier owner, SdrLay::bar_of */

/* ---- shared-memory plan + hand-over rules of one launch (one bucket = pipeline class x optional stages), sdr_lay.h ---- */
typedef struct {
  int32_t cls; uint32_t feat;        /* CLS_*, LF_* */
  int32_t T, tpb, tpb_sh, tile_f;    /* tile length in samples, tiles per block and its log2, floats per tile (T * 32) */
  int32_t n_hil;                     /* Hilbert warps (8 outputs of a tile each): T / 8 */
  int32_t nr, ni, na, nc, nz, nz2;   /* ring depths in tiles: input ring, Hilbert I delay, audio ring, AGC-out / ALS history ring, PLL-out ring, envelope work ring */
  int32_t hq_tiles, hq_rows;         /* Hilbert Q ring: tiles, rows of sample pairs (= hq_tiles * T / 2) */
  int32_t ins_row;                   /* floats per row of the input / output staging areas */
  int32_t o_sine, o_lut, o_ncot, o_cid, o_bar, o_flags, o_carr, o_nbs, o_mask, o_alsc, o_ins, o_outs, o_r, o_hq, o_hi, o_z, o_z2, o_a, o_c;
  int32_t smem_bytes, n_warps, dmax, error;
  uint8_t stage_of_warp[16];         /* physical warp -> (first) stage id */
  uint8_t prog[16][4];               /* physical warp -> the stages it runs each step, in this order (0xFF ends the list): one stage per warp
                                        except in the plans that merge light stages into one warp (sdr_lay.h, LF_SAM) */
  uint8_t active[16];                /* stage id -> runs in this launch */
  uint8_t bar_of[16];                /* stage id -> the stage whose barriers it signals: stages that always hand over together (the two IF rails,
                                        the Hilbert warps, the two image rails) share one barrier per tile, completed by all their arrivals */
  uint8_t bar_count[16];             /* arrivals that complete a barrier of that stage id */
  int32_t in_depth;                  /* input tiles requested ahead (landing buffers of the IN stage) */
  int32_t als_rows, als_mirror;      /* ALS post-pass plan (lay_build_als): rows of the tap array kept in shared memory; input ring kept twice */
  int8_t delay[16];                  /* the stage's delay in the lock-step schedule (documentation, deadlock-freedom proof, emulation) */
  SdrDep deps[SDR_STAGES][SDR_MAX_DEPS];
} SdrLay;

typedef struct {
  const void *in_i, *in_q;
  void *out;
  unsigned long long in_pitch, out_pitch; /* elements */
  int32_t in_fmt, out_fmt;
  uint32_t n_tiles;      /* n_blocks * lay.tpb */
  uint32_t blk0_mod3;    /* absolute index of the call's first block, mod 3 (noise-blanker ring slot) */
  const SdrChanCfg *cfg;
  float *state;
  unsigned long long ch_stride;
  const SdrGroup *groups; /* the launch's groups (CTA b runs groups[b]) */
  const float *agc_luts; /* [n_luts][132] */
  const SdrTables *tabs;
  uint32_t n_groups;
  uint32_t flags;        /* SDRL_CONTRACT: the handle asked for the contracting build (sdr_batch_desc.flags & SDR_BATCH_CONTRACT);
                            SDRL_RAW_OUT: first launch of a split ALS bucket -- the output stage writes the AGC output as it is (float32, no
                            ALS, gain, mute or truncation) to the scratch plane the ALS post-pass reads */
  float *raw;            /* split ALS bucket: scratch plane [group of the launch][sample of the call][lane] (float32), written by the
                            SDRL_RAW_OUT launch, read by the ALS post-pass (sdr_als_pass.cu) */
  uint32_t diag_skip;    /* diagnostics (profiling runs only): bit s set = stage s idles; results are then meaningless */
  unsigned long long *prof; /* optional [n_groups][SDR_PROF_SLOTS] (diagnostics twin): busy and waiting cycles per stage */
  uint32_t *bstat;       /* optional per-block status records of the launch's blocks (include/sdr_batch.h, SDR_BS_*): word
                            ((block * SDR_BS_FIELDS + field) * bs_stride + row); null = no records.  Written at the end of
                            each block by the stage that owns the field (sdr_pipeline.cuh, Ctx::bs_put) */
  unsigned long long bs_stride; /* = the call's row count (the handle's channel count, or the length of a subset call's id list) */
  SdrLay lay;
} SdrLaunch;

enum { SDRL_CONTRACT = 1u, SDRL_RAW_OUT = 2u };

/* default placement of the stages on the warps of a CTA (warp id % 4 = SM sub-partition, higher id = preferred by the
 * scheduler) for the launches that run all 14 stages; SDR_MAP_SSB / SDR_MAP_ENV (hex) override it for experiments */
#define SDR_MAP_SSB_DEFAULT 0xCBA435D8961720ull
#define SDR_MAP_SSB_NONB_DEFAULT 0xBC84627A3510D9ull /* SSB buckets without the blanker (BASELINE config 5): its three warps idle, so each of three
                                                         schedulers gets one Hilbert warp and one cascade / the output, the fourth two Hilbert
                                                         warps (tools/map_search.py --cls ssb --config 5: 1.496 -> 1.257 ms per 128 blocks) */
#define SDR_MAP_ENV_DEFAULT 0xA0D459B1328C67ull
#define SDR_MAP_ENV_NB_DEFAULT 0x19430DB7A258C6ull /* ENV buckets with the blanker (BASELINE config 4's AM and SAM buckets; its three warps work
                                                       there): tools/map_search.py --cls env --config 4 --split, 4.019 -> 3.685 ms per 64 blocks */
#define SDR_MAP_SSB_ALS_DEFAULT 0x4630127BC98DA5ull /* SSB buckets with the ALS filter: its stage (ALS + output) is by far the slowest and wants a
                                                        sub-partition where it wins the scheduler (tools/map_search.py --cls ssb --als) */
#define SDR_MAP_ENV_LEAN_DEFAULT 0x52980364BA7ull /* the 11-warp ENV plan on 16-sample tiles, two groups per SM (tools/map_search.py --cls envlean) */

#define SDR_PROF_SLOTS 64 /* [0..15] busy cycles per stage, [16..31] cycles waiting for other stages, [32] CTA cycles, [33] prologue (diagnostics twin only) */

#define SDR_AGC_LUT_STRIDE 132

#endif
