/* include/sdr_batch.h -- C ABI of the batched B200 receiver chain.
 *
 * Drop-in boundary for ONE path of DerekRowell/AudioSDR: the per-block receiver chain
 * AudioSDR::update() (reference SRC/AudioSDRlib/AudioSDR.cpp:39-168, "C:" below; class
 * declaration SRC/AudioSDRlib/AudioSDR.h:75-156, "H:" below).  One handle drives
 * n_channels independent receiver instances on one GPU; every instance behaves like one
 * `AudioSDR` object constructed in zeroed storage (the shipped sketch's global,
 * EXTRAS/BareBonesWSPR/BareBonesWSPR.ino:52) and fed one audio_block_t pair per block.
 *
 * What each entry point replaces in the reference:
 *   sdr_batch_create        AudioSDR::AudioSDR() -> init()                      H:77-79, C:174-185
 *   sdr_batch_set           any one public setter of the class                  H:88-152 (bodies C:187-311,356-398,498-566,653-682)
 *   sdr_batch_configure     a whole setter sequence per channel, e.g. the sketch's  INO:87-102,129
 *   sdr_batch_process[_*]   AudioStream::update_all() -> AudioSDR::update()     C:39-168
 *                            (receiveWritable(0/1) C:46-47 = the I/Q planes in; transmit(blockI,0/1) C:164-165 = the audio plane out)
 *   sdr_batch_get_status    the getters                                          C:224-230,255-273,295,371-381,495,507-512,568-600,660-665,752-757
 *   sdr_batch_*_status      process + the dynamic getters polled after every block (per-block status records, SDR_BS_*)
 *   sdr_batch_*_subset      process on the listed channels only; the others skip the call as update() does without input C:48-56
 *   sdr_batch_destroy       (object lifetime)
 *
 * Data layout: channel-major planes.  Sample t of channel c lives at plane[c*pitch + t]; pitch is
 * in ELEMENTS and must keep every row 16-byte aligned (pitch % 4 == 0 for float32, % 8 == 0 for
 * int16); t runs over 128*n_blocks samples of the call.  Wire formats:
 *   SDR_FMT_I16  int16 Q15, exactly the reference's audio_block_t::data (input scaling C:67-70,
 *                output truncation C:158-161) -- bit-for-bit the reference's boundary;
 *   SDR_FMT_F32  float32: input x stands for q/32767 and is scaled as (float)((double)x*gain)
 *                (identical to C:67-70 whenever the input gain is 1); output is the float product
 *                _output_gain*_audioOut of C:160 before the int16 truncation (0 when muted).
 *
 * Threading: process/set/configure are ordered on the stream given to process (set/configure are
 * host-side and take effect at the next process call, i.e. at a block boundary, as a setter
 * called between two update() ISRs does).  One handle must not be used from two host threads at
 * once; handles on different GPUs are independent (channels shard with no collective).
 *
 * Errors: every call returns 0 on success or a negative sdr_status; nothing throws across the ABI.
 * There is NO CPU fallback: if the CUDA device or kernel image is unavailable, create fails.
 */
#ifndef SDR_BATCH_H
#define SDR_BATCH_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SDR_BLOCK_SAMPLES 128      /* AUDIO_BLOCK_SAMPLES / n_block, H:73 */
#define SDR_SAMPLE_RATE 44100.0f   /* AUDIO_SAMPLE_RATE_EXACT on Teensy 4 */
#define SDR_ALL_CHANNELS 0xFFFFFFFFu

typedef enum {
  SDR_OK = 0,
  SDR_ERR_ARG = -1,        /* null pointer, bad channel id, bad pitch/alignment, n_blocks == 0 ... */
  SDR_ERR_MODE = -2,       /* demod mode / filter id / AGC mode outside the reference's enumerations */
  SDR_ERR_CUDA = -3,       /* CUDA runtime error; sdr_batch_last_error() has the text */
  SDR_ERR_NOMEM = -4,
  SDR_ERR_UNSUPPORTED = -5 /* ALS parameters that index before the reference's ring (M + delay > 129) */
} sdr_status;

/* Demodulation modes, H:44-50 (code numbering; the manual's table differs, SURVEY Q12). */
enum { SDR_LSB = 0, SDR_USB = 1, SDR_CW_LSB = 2, SDR_CW_USB = 3, SDR_AM = 4, SDR_SAM = 5, SDR_WSPR = 6 };
/* Audio band-pass selection, H:56-66. */
enum { SDR_AUDIO_AM = 0, SDR_AUDIO_CW, SDR_AUDIO_WSPR, SDR_AUDIO_2100, SDR_AUDIO_2300, SDR_AUDIO_2500,
       SDR_AUDIO_2700, SDR_AUDIO_2900, SDR_AUDIO_3100, SDR_AUDIO_3300, SDR_AUDIO_BYPASS };
/* AGC presets, H:68-71. */
enum { SDR_AGC_OFF = 0, SDR_AGC_FAST, SDR_AGC_MEDIUM, SDR_AGC_SLOW };
/* Wire formats. */
enum { SDR_FMT_I16 = 0, SDR_FMT_F32 = 1 };

/* The reference's public setter surface (H:88-152), one id per method; args as the method takes them. */
typedef enum {
  SDR_SET_setMute = 1,                 /* a0: 0/1                         C:249-253 */
  SDR_SET_setInputGain,                /* a0: gain, clamped to 0..10      C:232-238 */
  SDR_SET_setIQgainBalance,            /* a0: balance                     C:240-244 */
  SDR_SET_setDemodMode,                /* a0: mode; zeroes IF filter state C:187-222 */
  SDR_SET_enableAudioFilter,           /*                                 C:289-291 */
  SDR_SET_disableAudioFilter,          /*                                 C:292-294 */
  SDR_SET_setOutputGain,               /* a0: gain                        C:245-247 */
  SDR_SET_setAudioFilter,              /* a0: filter id; zeroes audio filter state C:298-311 */
  SDR_SET_enableALSfilter,             /* zeroes taps and history         C:384-391 */
  SDR_SET_disableALSfilter,            /*                                 C:356-358 */
  SDR_SET_setALSfilterNotch,           /*                                 C:359-361 */
  SDR_SET_setALSfilterPeak,            /*                                 C:362-364 */
  SDR_SET_setALSfilterAdaptive,        /*                                 C:365-367 */
  SDR_SET_setALSfilterStatic,          /*                                 C:368-370 */
  SDR_SET_setALSfilterParams,          /* a0: M (<=128), a1: lambda, a2: delay   C:393-398 */
  SDR_SET_enableAGC,                   /*                                 C:498-500 */
  SDR_SET_disableAGC,                  /*                                 C:501-503 */
  SDR_SET_setAGCthreshold,             /* a0: dB; rebuilds the table      C:514-517 */
  SDR_SET_setAGCslope,                 /* a0                              C:519-522 */
  SDR_SET_setAGCmode,                  /* a0: SDR_AGC_*                   C:524-544 */
  SDR_SET_setAGCkneeWidth,             /* a0: dB                          C:546-549 */
  SDR_SET_setAGCattackTime,            /* a0: ms                          C:551-555 */
  SDR_SET_setAGCreleaseTime,           /* a0: ms                          C:557-561 */
  SDR_SET_setAGChangTime,              /* a0: ms                          C:563-566 */
  SDR_SET_setAGCstaticGain,            /* a0                              C:504-506 */
  SDR_SET_enableNoiseBlanker,          /* zeroes the blanker rings        C:653-656 */
  SDR_SET_disableNoiseBlanker,         /*                                 C:657-659 */
  SDR_SET_setNoiseBlankerThreshold,    /* a0: ratio; zeroes the rings     C:666-669 */
  SDR_SET_setNoiseBlankerThresholdDb,  /* a0: dB;    zeroes the rings     C:671-674 */
  SDR_SET_init = 30                    /* AudioSDR::init()                C:174-185 */
} sdr_setter;

typedef struct sdr_batch sdr_batch_t;

typedef struct {
  uint32_t n_channels;          /* independent receiver instances on this handle */
  int32_t device;               /* CUDA device ordinal */
  uint32_t max_blocks_per_call; /* upper bound for n_blocks of one process call (0 = no bound) */
  uint32_t flags;               /* SDR_BATCH_* (0 = the default, bit-exact build) */
} sdr_batch_desc;

/* sdr_batch_desc.flags.  SDR_BATCH_CONTRACT: faster arithmetic in the linear sections of the chain (biquad cascades C:77,78,136,137,285,
 * Hilbert FIR C:88-112, NCO complex multiply H:515-518): fused multiply-adds and a different summation order.  Output is no
 * longer bit-identical to the reference's update(); it stays within 1e-4 of full scale (measured: profiles/, DESIGN.md). */
#define SDR_BATCH_CONTRACT 1u

/* One setter call addressed to one channel (or SDR_ALL_CHANNELS). */
typedef struct {
  uint32_t channel;
  uint32_t setter; /* sdr_setter */
  float a0, a1, a2;
} sdr_setter_call;

/* Per-channel read-back, the reference's getters. */
typedef struct {
  float tuning_offset;   /* getTuningOffset()        C:224-226 */
  float bpf_lower;       /* getBPFlower()            C:259-265 */
  float bpf_upper;       /* getBPFupper()            C:267-273 (WSPR keeps the reference's `+-` result) */
  float sam_frequency;   /* getSAMfrequency()        C:752-754 */
  float am_carrier;      /* getAMcarrierLevel()      C:495-497 */
  float agc_gain;        /* _agc_gain (for tests) */
  float nb_average;      /* _nb_AvgMag (for tests) */
  int32_t mode;          /* getDemodMode()           C:228-230 */
  int32_t audio_filter;  /* getAudioFilter()         C:295-297 */
  uint8_t muted;         /* getMute()                C:255-257 */
  uint8_t agc_enabled;   /* AGCisEnabled()           C:507-509 */
  uint8_t agc_active;    /* AGCisActive()            C:510-512 */
  uint8_t nb_enabled;    /* NoiseBlankerisEnabled()  C:660-662 */
  uint8_t nb_detected;   /* NoiseBlankerDetection()  C:663-665 */
  uint8_t sam_locked;    /* getSAMphaseLockStatus()  C:755-757 */
  uint8_t als_enabled;   /* ALSfilterIsEnabled()     C:371-373 */
  uint8_t als_notch;     /* ALSfilterIsNotch()       C:374-376 */
  uint8_t als_adaptive;  /* ALSfilterIsAdaptive()    C:380-382 */
  uint8_t audio_filter_enabled;
  uint8_t pad[2];
} sdr_channel_status;

/* Per-block status records: the dynamic getters after EVERY block of a process call, as the reference's sketch sees them when
 * it polls between two update() calls.  One 32-bit word per (block, field, channel), block-major:
 *     status[((size_t)b * SDR_BS_FIELDS + f) * n_channels + c]      b = block of the call, f = SDR_BS_*, c = channel
 * so that a run of blocks is one contiguous range.  Record (b, c) is what the getters (and _agc_gain / _nb_AvgMag) hold right
 * after channel c's update() for block b -- for every channel and every block, also fields whose stage does not run for the
 * channel (they keep their carried-over value).  The last record of a call equals sdr_batch_get_status after the call.
 * Flags are uint32 0 / 1, the other fields float32.  The buffer must be 16-byte aligned. */
enum { SDR_BS_AGC_GAIN = 0,     /* _agc_gain                            float */
       SDR_BS_AGC_ACTIVE,       /* AGCisActive()            C:510-512   uint32 0/1 */
       SDR_BS_AM_CARRIER,       /* getAMcarrierLevel()      C:495-497   float */
       SDR_BS_SAM_FREQUENCY,    /* getSAMfrequency()        C:752-754   float */
       SDR_BS_SAM_LOCKED,       /* getSAMphaseLockStatus()  C:755-757   uint32 0/1 */
       SDR_BS_NB_AVERAGE,       /* _nb_AvgMag                           float */
       SDR_BS_NB_DETECTED,      /* NoiseBlankerDetection()  C:663-665   uint32 0/1 */
       SDR_BS_FIELDS };

int sdr_batch_create(sdr_batch_t **out, const sdr_batch_desc *desc);
void sdr_batch_destroy(sdr_batch_t *h);

/* One reference setter on `n` channels (ids == NULL: all channels). */
int sdr_batch_set(sdr_batch_t *h, const uint32_t *channel_ids, uint32_t n, uint32_t setter, float a0, float a1, float a2);
/* A sequence of setter calls, applied in order (the order matters exactly as in the reference, SURVEY Q7). */
int sdr_batch_configure(sdr_batch_t *h, const sdr_setter_call *calls, uint32_t n_calls);

/* The hot path.  Device pointers; asynchronous on `cuda_stream` (a cudaStream_t, NULL = default stream).
 * in_fmt/out_fmt: SDR_FMT_*; pitches in elements.  Advances every channel by n_blocks blocks (the _subset forms below: the
 * listed channels only).
 * Device memory the handle owns besides the 7.9 KB of state per channel: a handle with more than 148 groups of 32
 * channels (4 736 channels or fewer, by mode mix) keeps a scratch plane for those that use the ALS filter, 4 bytes per ALS
 * channel and sample of the longest call so far, at most SDR_ALS_SCRATCH_MB (environment, default 4096) megabytes per kind
 * of channel (INTEGRATION.md, run-time switches). */
int sdr_batch_process_device(sdr_batch_t *h, const void *I, const void *Q, size_t in_pitch, int in_fmt,
                             void *audio, size_t out_pitch, int out_fmt, uint32_t n_blocks, void *cuda_stream);
/* The same call in its plainest form: float32 planes, rows densely packed (pitch = 128 * n_blocks elements). */
int sdr_batch_process(sdr_batch_t *h, const float *I, const float *Q, float *audio, uint32_t n_blocks, void *cuda_stream);
/* Same through HOST buffers (pinned or pageable): H2D copy, kernel, D2H copy, synchronous on return. */
int sdr_batch_process_host(sdr_batch_t *h, const void *I, const void *Q, size_t in_pitch, int in_fmt,
                           void *audio, size_t out_pitch, int out_fmt, uint32_t n_blocks);
/* The streaming form of the same call (the reference's update() is an endless stream of blocks, C:39-168: one interrupt per
 * 128 samples): submit_host queues the copies and launches and returns; wait_host returns when everything submitted so far
 * has landed in the callers' audio buffers.  Calls submitted back to back overlap -- the first copy-in of a call runs beside
 * the last kernel and copy-out of the call before -- so a stream of calls runs at the speed of the host link, without
 * the start-up and drain of each call.  Until wait_host returns, the input buffers must stay unchanged and the audio
 * buffers unread; host buffers must be pinned for the copies to be asynchronous.  Setter calls between two submits take
 * effect at that block boundary, as everywhere.  process_host == submit_host + wait_host. */
int sdr_batch_submit_host(sdr_batch_t *h, const void *I, const void *Q, size_t in_pitch, int in_fmt,
                          void *audio, size_t out_pitch, int out_fmt, uint32_t n_blocks);
int sdr_batch_wait_host(sdr_batch_t *h);
/* The three calls above with per-block status records (layout above: n_blocks * SDR_BS_FIELDS * n_channels words).
 * block_status == NULL makes each identical to the call without records.  _device_status: device memory, asynchronous on
 * the stream like the audio.  _host_status / submit_host_status: host memory (pinned for asynchronous copies); the
 * records land together with the call's audio, so wait_host_ticket(n) means the records of call n are there too. */
int sdr_batch_process_device_status(sdr_batch_t *h, const void *I, const void *Q, size_t in_pitch, int in_fmt,
                                    void *audio, size_t out_pitch, int out_fmt, uint32_t n_blocks, void *block_status,
                                    void *cuda_stream);
int sdr_batch_process_host_status(sdr_batch_t *h, const void *I, const void *Q, size_t in_pitch, int in_fmt,
                                  void *audio, size_t out_pitch, int out_fmt, uint32_t n_blocks, void *block_status);
int sdr_batch_submit_host_status(sdr_batch_t *h, const void *I, const void *Q, size_t in_pitch, int in_fmt,
                                 void *audio, size_t out_pitch, int out_fmt, uint32_t n_blocks, void *block_status);
/* One call at a time: sdr_batch_host_ticket() right after a submit_host (or process_host) names that call (1, 2, ...);
 * wait_host_ticket returns when that call's audio has landed, while later calls stay in flight -- a receiver that keeps
 * two calls queued drains call n while call n + 1 is being copied in and computed.  Calls complete in order. */
uint64_t sdr_batch_host_ticket(const sdr_batch_t *h);
int sdr_batch_wait_host_ticket(sdr_batch_t *h, uint64_t ticket);

/* The same calls on a chosen subset of the channels: the reference's update() returns without touching anything when an
 * input block is missing (C:48-56), so in a graph some objects skip a block period while others run.  The call advances
 * the n_ids channels channel_ids[0..n_ids) by n_blocks blocks each, bit for bit as update() would; every other channel is
 * untouched -- state, getters, no plane row and no record -- and its next processed block continues its own stream.  A
 * channel's output over any sequence of calls is therefore the reference run on that channel's own blocks, concatenated.
 *   channel_ids  host memory, read before the call returns; distinct ids below n_channels, n_ids >= 1.  NULL (with
 *                n_ids == n_channels) is exactly the call on every channel: the entry points above are these calls with NULL.
 *                Anything else returns SDR_ERR_ARG and queues nothing.
 *   planes       compact: row i of I, Q and audio belongs to channel channel_ids[i] (n_ids rows, any order of ids).
 *   block_status compact too: status[((size_t)b * SDR_BS_FIELDS + f) * n_ids + i] (NULL: no records).
 * Setters are unchanged: a setter on a channel that is not listed takes effect before that channel's next processed block,
 * as a setter between two ISRs does to an object that got no block.  get_status, export_state and import_state work on any
 * channel at any time; a blob exported from a channel that has skipped calls continues bit for bit wherever it is imported.
 * Grouping: the last subset's groups are kept and reused while its id list and the configuration stay the same, apart from
 * those of the calls on every channel (alternating the two forms re-plans neither). */
int sdr_batch_process_device_subset(sdr_batch_t *h, const uint32_t *channel_ids, uint32_t n_ids, const void *I, const void *Q,
                                    size_t in_pitch, int in_fmt, void *audio, size_t out_pitch, int out_fmt, uint32_t n_blocks,
                                    void *block_status, void *cuda_stream);
int sdr_batch_process_host_subset(sdr_batch_t *h, const uint32_t *channel_ids, uint32_t n_ids, const void *I, const void *Q,
                                  size_t in_pitch, int in_fmt, void *audio, size_t out_pitch, int out_fmt, uint32_t n_blocks,
                                  void *block_status);
/* ticketed like submit_host: sdr_batch_host_ticket() right after it names the call */
int sdr_batch_submit_host_subset(sdr_batch_t *h, const uint32_t *channel_ids, uint32_t n_ids, const void *I, const void *Q,
                                 size_t in_pitch, int in_fmt, void *audio, size_t out_pitch, int out_fmt, uint32_t n_blocks,
                                 void *block_status);

/* Getters for `n` channels (ids == NULL: channels 0..n-1).  Synchronises the handle's last stream. */
int sdr_batch_get_status(sdr_batch_t *h, const uint32_t *channel_ids, uint32_t n, sdr_channel_status *out);
/* getAGClookup(i) for one channel, C:595-597. */
int sdr_batch_get_agc_lookup(sdr_batch_t *h, uint32_t channel, float *out129);
/* Debug/test tap: raw per-channel state word (see audiosdr_b200/csrc/sdr_types.h). */
int sdr_batch_peek_state(sdr_batch_t *h, uint32_t channel, uint32_t word, float *out);

/* Checkpoint / migration.  A channel's whole carry-over -- the configuration its setters have built up (the members the
 * reference's setters write, H:164-330) and everything update() carries from block to block (filter delay lines H:191-195,
 * Hilbert rings and NCO phases C:41-44, AGC H:208-232, PLL C:690-694 / H:263-274, ALS taps and history H:198-205, blanker
 * rings, mask and average H:235-246) -- as one opaque blob of sdr_batch_state_bytes() bytes per channel.  Importing a blob
 * into any channel of any handle of the same library version (another GPU, another process, a handle that has run a
 * different number of blocks) continues the stream bit for bit.  Both calls synchronise the handle's last stream. */
size_t sdr_batch_state_bytes(void);
int sdr_batch_export_state(sdr_batch_t *h, const uint32_t *channel_ids, uint32_t n, void *blobs);
int sdr_batch_import_state(sdr_batch_t *h, const uint32_t *channel_ids, uint32_t n, const void *blobs);

/* Diagnostics: per-stage busy cycles of the pipeline kernel, summed over groups and launches since create.
 * Only recorded when the environment variable SDR_ROLE_PROFILE=1 was set at create (costs two clock reads per
 * stage per tile; the kernel timed in that mode writes no per-block status records).  busy[cls*14 + stage] (14 stages per pipeline class), total[cls] = summed CTA cycles,
 * groups[cls] = CTA launches counted. */
int sdr_batch_get_role_profile(sdr_batch_t *h, uint64_t *busy28, uint64_t *total2, uint64_t *groups2);

/* Kernels this handle has launched so far (for the benchmark's gpu_launches claim). */
uint64_t sdr_batch_launch_count(const sdr_batch_t *h);
const char *sdr_batch_last_error(void);
const char *sdr_batch_version(void);

#ifdef __cplusplus
}
#endif
#endif
