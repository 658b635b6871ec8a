/* include/sdr_aux.h -- C ABI of the two blocks either side of the receiver chain (SURVEY.md 8f rows 2 and 4), batched over
 * independent channels on one GPU.  Library: audiosdr_b200/libsdr_aux.so (CUDA, sm_100a; no CPU fallback).
 *
 *   sdr_preproc_*   replaces  class AudioSDRpreProcessor   AudioSDRpreProcessor.h:49-73, update() AudioSDRpreProcessor.cpp:46-138
 *   sdr_iqgen_*     replaces  class AudioIQgenerator       AudioIQgenerator.h:49-107,   update() AudioIQgenerator.cpp:33-87
 *   sdr_grabber_*   replaces  class AudioGrabberComplex256 AudioGrabberComplex256.h:46-64, update()/grab() AudioGrabberComplex256.cpp:50-91
 *
 * Planes are int16 (the reference's audio_block_t wire format), channel-major: sample s of channel c is plane[c*pitch + s],
 * pitch in elements.  Base pointers must be 16-byte aligned and pitches multiples of 8.  Output planes must not overlap the
 * input planes (the reference works in place on one block; a batched one-sample shift cannot).  Each process call advances
 * every channel by n_blocks blocks of 128 samples; all per-channel state lives in device memory between calls.
 *
 * Calls on a subset of the channels (*_subset): each class's update() starts by taking its input block(s) and returns
 * without touching any member when one is missing, as AudioSDR::update() does (AudioSDR.cpp:48-56).  For these three
 * classes the cited ranges are those of the whole update() (AudioSDRpreProcessor.cpp:46-138, AudioIQgenerator.cpp:33-87,
 * AudioGrabberComplex256.cpp:50-72); the exact lines of the early return are unchecked.  So in a graph some objects skip
 * a block period while others run.  The rules are those of sdr_batch_process_device_subset
 * (sdr_batch.h), so that one id list drives the whole graph:
 *   channel_ids  host memory, read before the call returns; distinct ids below n_channels, n_ids >= 1.  NULL (with
 *                n_ids == n_channels) is the call on every channel: the plain entry points are these calls with NULL.
 *                Anything else returns SDR_AUX_EINVAL and queues nothing: no state changes, no output is written.
 *   planes       compact: row i of every plane belongs to channel channel_ids[i] (n_ids rows, ids in any order).
 * Every unlisted channel is untouched and its next processed block continues its own stream; a channel's output over any
 * sequence of calls is the reference run on that channel's own blocks, concatenated.  Setters on an unlisted channel take
 * effect before that channel's next processed block.
 *
 * Checkpoint / migration (*_state_bytes, *_export_state, *_import_state): a channel's whole carry-over as one opaque blob
 * of *_state_bytes() bytes (channel_ids == NULL: channels 0..n-1).  A blob imports into any channel of any handle of the
 * same block and library version -- another GPU, a handle that has run a different number of blocks -- and the stream
 * continues bit for bit.  Both calls synchronise the device.
 * All functions return 0 (SDR_AUX_OK) or a negative error; sdr_aux_last_error() gives the text (thread local).
 */
#ifndef SDR_AUX_H
#define SDR_AUX_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

enum { SDR_AUX_OK = 0, SDR_AUX_EINVAL = -1, SDR_AUX_ECUDA = -2, SDR_AUX_ENOMEM = -3 };

/* ---------------------------------------------------------------- pre-processor ---- */
typedef struct sdr_preproc sdr_preproc_t;

/* setter ids = the reference's public functions (AudioSDRpreProcessor.h:54-59) */
typedef enum {
  SDR_PP_startAutoI2SerrorDetection = 1, /* AudioSDRpreProcessor.cpp:142-148 */
  SDR_PP_stopAutoI2SerrorDetection = 2,  /* AudioSDRpreProcessor.cpp:151-154 */
  SDR_PP_setI2SerrorCompensation = 3,    /* arg = -1, 0, +1;  AudioSDRpreProcessor.cpp:160-163 */
  SDR_PP_swapIQ = 4                      /* arg = 0 / 1;      AudioSDRpreProcessor.cpp:169 */
} sdr_preproc_setter;

typedef struct {
  int32_t auto_detect;   /* getAutoI2SerrorDetectionStatus(), AudioSDRpreProcessor.cpp:157 */
  int32_t correction;    /* getI2SerrorCompensation(),        AudioSDRpreProcessor.cpp:166 */
  int32_t failure_count; /* private members, for tests and checkpoints */
  int32_t success_count;
  int32_t saved_sample;
  int32_t swap;
} sdr_preproc_status;

int sdr_preproc_create(sdr_preproc_t **out, uint32_t n_channels, int device);
void sdr_preproc_destroy(sdr_preproc_t *h);
/* channels == NULL: every channel.  Setters take effect before the next processed block, in call order. */
int sdr_preproc_set(sdr_preproc_t *h, const uint32_t *channels, uint32_t n, uint32_t setter, int32_t arg);
int sdr_preproc_get_status(sdr_preproc_t *h, const uint32_t *channels, uint32_t n, sdr_preproc_status *out);
/* AudioSDRpreProcessor::update() for every channel, n_blocks times.  Device planes; asynchronous on `cuda_stream`. */
int sdr_preproc_process_device(sdr_preproc_t *h, const int16_t *I, const int16_t *Q, size_t in_pitch, int16_t *I_out,
                               int16_t *Q_out, size_t out_pitch, uint32_t n_blocks, void *cuda_stream);
/* ... host planes: copies in, runs, copies out, returns when the outputs are in host memory */
int sdr_preproc_process_host(sdr_preproc_t *h, const int16_t *I, const int16_t *Q, size_t in_pitch, int16_t *I_out,
                             int16_t *Q_out, size_t out_pitch, uint32_t n_blocks);
/* the same on the n_ids channels channel_ids[0..n_ids) (rules at the top of this file) */
int sdr_preproc_process_device_subset(sdr_preproc_t *h, const uint32_t *channel_ids, uint32_t n_ids, const int16_t *I, const int16_t *Q,
                                      size_t in_pitch, int16_t *I_out, int16_t *Q_out, size_t out_pitch, uint32_t n_blocks,
                                      void *cuda_stream);
int sdr_preproc_process_host_subset(sdr_preproc_t *h, const uint32_t *channel_ids, uint32_t n_ids, const int16_t *I, const int16_t *Q,
                                    size_t in_pitch, int16_t *I_out, int16_t *Q_out, size_t out_pitch, uint32_t n_blocks);
/* The same call, also returning the getters after every block: what a sketch polling getI2SerrorCompensation() and
 * getAutoI2SerrorDetectionStatus() after each update() sees, and so which output blocks were made under which correction and
 * at which block the detector stopped.  Ids, planes and checks are those of the *_subset calls, and the state the call
 * leaves is the same.
 *   block_status  int32 words, one per (block, field, row), block-major:
 *                 block_status[((size_t)b * SDR_PP_BS_FIELDS + f) * n_ids + i] = field f of row i's channel right after its
 *                 update() for block b, i.e. what sdr_preproc_get_status would return then (setters queued before the call
 *                 apply before block 0; the last block's record equals get_status after the call).  Fields in the order of
 *                 sdr_preproc_status; flags are 0 or 1, the saved sample is the int16 value sign-extended.  Every word of
 *                 [n_blocks][SDR_PP_BS_FIELDS][n_ids] is written, rows with the detector off included (their fields are
 *                 constant over the call except the saved sample, when the correction is +1 or -1).
 *                 Device memory for the device form.  Host memory (pageable or pinned) for the host form: the records are
 *                 staged on the device and copied out before the call returns.  Must be 16-byte aligned (SDR_AUX_EINVAL
 *                 otherwise, nothing queued).  NULL: the call without records (the four process entry points above are
 *                 these calls with NULL). */
enum { /* 0 .. 5, then the count */
  SDR_PP_BS_AUTO_DETECT, SDR_PP_BS_CORRECTION, SDR_PP_BS_FAILURE_COUNT, SDR_PP_BS_SUCCESS_COUNT, SDR_PP_BS_SAVED_SAMPLE, SDR_PP_BS_SWAP,
  SDR_PP_BS_FIELDS
};
int sdr_preproc_process_device_status(sdr_preproc_t *h, const uint32_t *channel_ids, uint32_t n_ids, const int16_t *I, const int16_t *Q,
                                      size_t in_pitch, int16_t *I_out, int16_t *Q_out, size_t out_pitch, uint32_t n_blocks,
                                      int32_t *block_status, void *cuda_stream);
int sdr_preproc_process_host_status(sdr_preproc_t *h, const uint32_t *channel_ids, uint32_t n_ids, const int16_t *I, const int16_t *Q,
                                    size_t in_pitch, int16_t *I_out, int16_t *Q_out, size_t out_pitch, uint32_t n_blocks,
                                    int32_t *block_status);
uint64_t sdr_preproc_launch_count(const sdr_preproc_t *h);
/* Blob: the PP.h:66-72 members (correction, savedSample, both detector counters, swap, detector flag).  Export applies queued
 * setters first, as get_status does; import replaces the channel's state including setters queued for it, and setters
 * called after the import apply on top of it. */
size_t sdr_preproc_state_bytes(void);
int sdr_preproc_export_state(sdr_preproc_t *h, const uint32_t *channel_ids, uint32_t n, void *blobs);
int sdr_preproc_import_state(sdr_preproc_t *h, const uint32_t *channel_ids, uint32_t n, const void *blobs);

/* ---------------------------------------------------------------- I/Q generator ---- */
typedef struct sdr_iqgen sdr_iqgen_t;

int sdr_iqgen_create(sdr_iqgen_t **out, uint32_t n_channels, int device);
void sdr_iqgen_destroy(sdr_iqgen_t *h);
/* AudioIQgenerator::setGainBalance (AudioIQgenerator.h:56-60): gainI = balance, gainQ = 1.0 / balance */
int sdr_iqgen_set_gain_balance(sdr_iqgen_t *h, const uint32_t *channels, uint32_t n, float balance);
/* AudioIQgenerator::update() for every channel, n_blocks times: X real input -> I (delayed 128 samples) and Q (Hilbert) */
int sdr_iqgen_process_device(sdr_iqgen_t *h, const int16_t *X, size_t in_pitch, int16_t *I_out, int16_t *Q_out,
                             size_t out_pitch, uint32_t n_blocks, void *cuda_stream);
int sdr_iqgen_process_host(sdr_iqgen_t *h, const int16_t *X, size_t in_pitch, int16_t *I_out, int16_t *Q_out,
                           size_t out_pitch, uint32_t n_blocks);
int sdr_iqgen_process_device_subset(sdr_iqgen_t *h, const uint32_t *channel_ids, uint32_t n_ids, const int16_t *X, size_t in_pitch,
                                    int16_t *I_out, int16_t *Q_out, size_t out_pitch, uint32_t n_blocks, void *cuda_stream);
int sdr_iqgen_process_host_subset(sdr_iqgen_t *h, const uint32_t *channel_ids, uint32_t n_ids, const int16_t *X, size_t in_pitch,
                                  int16_t *I_out, int16_t *Q_out, size_t out_pitch, uint32_t n_blocks);
uint64_t sdr_iqgen_launch_count(const sdr_iqgen_t *h);
/* Blob: the last 256 input samples (the filter's history, IQ.cpp:37-38) and (gainI, gainQ) */
size_t sdr_iqgen_state_bytes(void);
int sdr_iqgen_export_state(sdr_iqgen_t *h, const uint32_t *channel_ids, uint32_t n, void *blobs);
int sdr_iqgen_import_state(sdr_iqgen_t *h, const uint32_t *channel_ids, uint32_t n, const void *blobs);

/* ---------------------------------------------------------------- complex snapshot grabber ---- */
/* replaces class AudioGrabberComplex256 (AudioGrabberComplex256.h:46-64): every update() appends one block of interleaved
 * (re, im) samples to a two-block buffer; each time the buffer fills, it becomes the snapshot grab() hands out
 * (AudioGrabberComplex256.cpp:50-91).  No arithmetic: the batched form is a gather of the last complete pair of blocks. */
typedef struct sdr_grabber sdr_grabber_t;

int sdr_grabber_create(sdr_grabber_t **out, uint32_t n_channels, int device);
void sdr_grabber_destroy(sdr_grabber_t *h);
/* AudioGrabberComplex256::update() for every channel, n_blocks times; device planes as for the pre-processor */
int sdr_grabber_process_device(sdr_grabber_t *h, const int16_t *I, const int16_t *Q, size_t pitch, uint32_t n_blocks, void *cuda_stream);
/* the same on the n_ids channels channel_ids[0..n_ids).  Each channel keeps its own pair phase, _dataBufferValid and
 * new-data flag, so after calls on subsets the channels differ in all three. */
int sdr_grabber_process_device_subset(sdr_grabber_t *h, const uint32_t *channel_ids, uint32_t n_ids, const int16_t *I, const int16_t *Q,
                                      size_t pitch, uint32_t n_blocks, void *cuda_stream);
/* The same call, also returning every snapshot it publishes and/or its power spectrum: what a sketch polling
 * newDataAvailable() / grab() after every update() sees, one line per completed pair (a panadapter or waterfall per channel).
 * Ids, planes and checks are those of sdr_grabber_process_device_subset, and the state it leaves is the same.
 *   S = (n_blocks + 1) / 2 slots per row.  With p = the row's channel's pair phase before the call (its own blocks processed,
 *   mod 2), the row publishes counts[i] = (p + n_blocks) / 2 snapshots, in slots 0 .. counts[i]-1: slot k is the pair the
 *   call's block 2k + 1 - p (0-based) completes, the block after which the reference's newDataAvailable() turns true.  When
 *   p == 1, slot 0 starts with the block carried over from the channel's previous call (or from an imported blob).  Slots
 *   past counts[i] are not written (only when n_blocks is odd and p == 0).
 *   snapshots  device, int16 [n_ids][S][512] or NULL: each slot as grab() would have written it right after that block.
 *   power      device, float [n_ids][S][256] or NULL: each slot's spectrum, the same bins, order and bits as
 *              sdr_grabber_spectrum.
 *   counts     host, uint32 [n_ids] or NULL: filled before the call returns, without synchronising.
 * snapshots and power must be 16-byte aligned (SDR_AUX_EINVAL otherwise, nothing queued).  With all three NULL this is
 * sdr_grabber_process_device_subset.  Channel-major layout: a channel's waterfall for the call is one contiguous [S][256]. */
int sdr_grabber_process_device_snapshots(sdr_grabber_t *h, const uint32_t *channel_ids, uint32_t n_ids, const int16_t *I, const int16_t *Q,
                                         size_t pitch, uint32_t n_blocks, int16_t *snapshots, float *power, uint32_t *counts,
                                         void *cuda_stream);
/* newDataAvailable() of one channel: 1 / 0, negative on error */
int sdr_grabber_new_data_available(sdr_grabber_t *h, uint32_t channel);
/* grab() for the listed channels (NULL: all): 512 int16 per channel = 256 complex samples, to HOST memory
 * dest[i*512 .. i*512+511].  A channel before its first complete pair has no snapshot (the reference's _dataBufferValid):
 * its row is not written.  The call clears every listed channel's new-data flag.  Returns the number of rows written,
 * negative on error. */
int sdr_grabber_grab(sdr_grabber_t *h, const uint32_t *channels, uint32_t n, int16_t *dest);
/* all channels, device to device: dest[n_channels][512], rows of channels without a snapshot not written; clears every
 * new-data flag; returns 1 when some row was written, 0 when none */
int sdr_grabber_grab_device(sdr_grabber_t *h, int16_t *dest, void *cuda_stream);
/* Blob: the carried first block of an incomplete pair, the snapshot, the channel's pair phase, _dataBufferValid and the
 * new-data flag */
size_t sdr_grabber_state_bytes(void);
int sdr_grabber_export_state(sdr_grabber_t *h, const uint32_t *channel_ids, uint32_t n, void *blobs);
int sdr_grabber_import_state(sdr_grabber_t *h, const uint32_t *channel_ids, uint32_t n, const void *blobs);

/* Spectrum tap on the snapshots -- what the consumer of grab() does with them (the sketch's panadapter / S-meter; not part
 * of the library classes, SURVEY 8f row 3): the 256-point forward complex FFT of a channel's snapshot, samples taken as
 * floats (re, im) = (float)int16, and the power re^2 + im^2 per bin, natural bin order (bin k = k * 44100/256 Hz, bins 128..255
 * = negative frequencies).  power[i*256 + k] for the i-th listed channel (NULL: all channels); rows of channels without a
 * snapshot yet are not written.  Returns the number of rows written (host form) / 1 when some row was written (device
 * form), 0 when none, negative on error; the new-data flags are left alone (a spectrum is a view of the snapshot, not a
 * grab()). */
int sdr_grabber_spectrum(sdr_grabber_t *h, const uint32_t *channels, uint32_t n, float *power);
int sdr_grabber_spectrum_device(sdr_grabber_t *h, const uint32_t *d_channels, uint32_t n, float *d_power, void *cuda_stream);

/* ---------------------------------------------------------------- waterfall ---- */
/* Averaged waterfall lines per channel: the grabber's per-pair power spectra (sdr_grabber_process_device_snapshots' `power`,
 * bit for bit) averaged K at a time, in pair order, across calls.  Number the pairs a channel's grabber completes 0, 1, 2, ...
 * since the waterfall was created (or since the channel's blob was imported); line m of the channel is, per bin,
 *     acc = 0.0f;  for j in mK .. mK+K-1:  acc = acc + P_j     (float32, one rounding per add, in j order)
 *     line_m = acc / (float)K                                  (one IEEE division)
 * so with K == 1 the lines are the spectra themselves.  A channel's lines do not depend on how its blocks are cut into calls
 * or subsets, nor on a migration through export_state / import_state.  The waterfall holds each channel's partial sum (the
 * pairs held, < K) between calls; it is driven only through the grabber calls below. */
typedef struct sdr_waterfall sdr_waterfall_t;

int sdr_waterfall_create(sdr_waterfall_t **out, uint32_t n_channels, int device, uint32_t K); /* K >= 1 */
void sdr_waterfall_destroy(sdr_waterfall_t *w);
int sdr_waterfall_get_info(const sdr_waterfall_t *w, uint32_t *n_channels, int *device, uint32_t *K);
/* Blob: K, the pairs held and their partial sum (256 floats).  Imports only into a waterfall with the same K. */
size_t sdr_waterfall_state_bytes(void);
int sdr_waterfall_export_state(sdr_waterfall_t *w, const uint32_t *channel_ids, uint32_t n, void *blobs);
int sdr_waterfall_import_state(sdr_waterfall_t *w, const uint32_t *channel_ids, uint32_t n, const void *blobs);
/* sdr_grabber_process_device_subset on the listed channels (same ids, planes, checks and resulting grabber state), also
 * advancing the waterfall `wf` (same device and channel count as the grabber, else SDR_AUX_EINVAL) over the pairs it completes.
 *   Lmax = (K - 1 + (n_blocks + 1) / 2) / K line slots per row.
 *   lines   device, float [n_ids][Lmax][256], 16-byte aligned: row i's counts[i] lines completed by this call, oldest first,
 *           natural bin order.  Slots past counts[i] are not written.
 *   counts  host, uint32 [n_ids] or NULL: filled before the call returns, without synchronising.
 * A bad argument queues nothing: no state changes, nothing is written. */
int sdr_grabber_process_device_waterfall(sdr_grabber_t *gr, sdr_waterfall_t *wf, const uint32_t *channel_ids, uint32_t n_ids, const int16_t *I,
                                         const int16_t *Q, size_t pitch, uint32_t n_blocks, float *lines, uint32_t *counts, void *cuda_stream);
/* The same with row i's lines at slots first_line[i] .. first_line[i] + counts[i] - 1 of a row of line_pitch slots:
 * lines[((size_t)i * line_pitch + first_line[i] + m) * 256 + bin].  first_line: host, uint32 [n_ids] or NULL (zeros); a row
 * whose lines would run past line_pitch is SDR_AUX_EINVAL.  Lets a caller that cuts one call into several (sdr_graph.h)
 * gather each row's lines where the uncut call would have put them. */
int sdr_grabber_process_device_waterfall_at(sdr_grabber_t *gr, sdr_waterfall_t *wf, const uint32_t *channel_ids, uint32_t n_ids,
                                            const int16_t *I, const int16_t *Q, size_t pitch, uint32_t n_blocks, float *lines,
                                            size_t line_pitch, const uint32_t *first_line, uint32_t *counts, void *cuda_stream);

/* The channel count and device a handle was created with (for code that drives handles it did not create, e.g. sdr_graph.h) */
int sdr_preproc_get_info(const sdr_preproc_t *h, uint32_t *n_channels, int *device);
int sdr_iqgen_get_info(const sdr_iqgen_t *h, uint32_t *n_channels, int *device);
int sdr_grabber_get_info(const sdr_grabber_t *h, uint32_t *n_channels, int *device);

const char *sdr_aux_last_error(void);
const char *sdr_aux_version(void);

#ifdef __cplusplus
}
#endif
#endif
