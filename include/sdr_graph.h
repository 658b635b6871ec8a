/* include/sdr_graph.h -- the shipped sketch's receiver graph, streamed from HOST memory in one ticketed call.
 *
 * The sketch wires  I2S in -> AudioSDRpreProcessor -> AudioSDR -> I2S out, with AudioGrabberComplex256 tapping the
 * pre-processor's output (EXTRAS/BareBonesWSPR/BareBonesWSPR.ino:50-62, SURVEY 1); a single-ended front end has
 * AudioIQgenerator in place of the pre-processor.  A graph handle runs that graph over handles the caller created
 * (include/sdr_batch.h, include/sdr_aux.h) on int16 planes in host memory: per time chunk it copies the chunk's input up,
 * runs the blocks' existing device entry points on its own compute stream and copies the audio (and the optional records,
 * spectra and snapshots) down.  The corrected I/Q planes between the blocks never leave the device, so a call moves 6 bytes
 * per channel-sample over the host link (int16 I, Q in; int16 audio out) where the composition of the blocks' host calls
 * moves 14.  Library: audiosdr_b200/libsdr_graph.so (links libsdr_batch.so and libsdr_aux.so); no new kernel, no CPU path.
 *
 * A call equals, bit for bit, the composition of the blocks' device calls on the same ids, each over the whole call:
 *   sdr_preproc_process_device_status  or  sdr_iqgen_process_device_subset    (the front, if any)
 *   sdr_grabber_process_device_snapshots                                      (the tap, if any; on the front's output)
 *   sdr_batch_process_device_subset                                           (the receiver; int16 input)
 * -- every audio sample, record, snapshot, spectrum and count, and the state every member handle is left in (one exception,
 * which no output can see: the bytes of the grabber's carried block of a channel with no pair open, which its export_state
 * blob still holds, are those of the last open pair of a chunk rather than of the call).  The call is
 * cut into time chunks as sdr_batch_submit_host cuts its calls (SDR_HOST_CHUNKS, SDR_HOST_MIN_CHUNK; INTEGRATION.md); every
 * chunk but the last has an even number of blocks, so that each channel's grabber pair phase at a chunk's start is its phase
 * at the call's start.  The chunking does not change a single output bit.
 *
 * Member handles stay the caller's: setters on them between two submits take effect at that block boundary, as for the
 * device calls.  Getters, export_state and import_state on a member handle see every submitted call once sdr_graph_wait_host
 * has returned.  A caller who also drives a member handle directly (its own process or host calls) must call
 * sdr_graph_wait_host first: the pre-processor, generator and grabber do not order their own calls after work queued on
 * the graph's streams (the receiver does).  The graph does not own the members: destroy the graph before them.
 *
 * Errors: 0 or a negative sdr_status (sdr_batch.h); sdr_graph_last_error() has the text, thread local.  A bad argument is
 * found before anything is queued: the call then changes no state and writes no output.
 */
#ifndef SDR_GRAPH_H
#define SDR_GRAPH_H
#include <stddef.h>
#include <stdint.h>

#include "sdr_aux.h"
#include "sdr_batch.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sdr_graph sdr_graph_t;

typedef struct {
  sdr_batch_t *rx;       /* the receiver; required */
  sdr_preproc_t *pp;     /* the front: at most one of pp / gen; neither = the input I/Q go straight to the tap and receiver */
  sdr_iqgen_t *gen;
  sdr_grabber_t *grabber; /* optional tap on the receiver's input planes (the front's output) */
} sdr_graph_desc;        /* every handle on one device with the same n_channels, else SDR_ERR_ARG at create */

/* Optional outputs of a call: host memory (pinned for asynchronous copies), NULL = not wanted.  Layouts exactly as the
 * device calls define them, with n_ids rows (row i = channel ids[i]) and S = (n_blocks + 1) / 2.  The record, power and
 * snapshot buffers must be 16-byte aligned. */
typedef struct {
  void *rx_status;      /* [n_blocks][SDR_BS_FIELDS][n_ids] 32-bit words      sdr_batch_process_device_subset's block_status */
  int32_t *pp_status;   /* [n_blocks][SDR_PP_BS_FIELDS][n_ids]                sdr_preproc_process_device_status (pp front only) */
  float *power;         /* [n_ids][S][256]                                    sdr_grabber_process_device_snapshots (tap only) */
  int16_t *snapshots;   /* [n_ids][S][512]                                    (tap only) */
  uint32_t *counts;     /* [n_ids] slots written per row, filled before submit returns (tap only); slots past counts[i]
                         * are not written */
} sdr_graph_outputs;

int sdr_graph_create(sdr_graph_t **out, const sdr_graph_desc *desc);
/* Waits for the graph's calls in flight; the member handles are left alone. */
void sdr_graph_destroy(sdr_graph_t *g);

/* One call of the graph on the n_ids channels ids[0..n_ids) (NULL with n_ids == n_channels: every channel), n_blocks
 * blocks each.  Host planes, int16, row i = channel ids[i], pitches in elements (>= 128 * n_blocks):
 *   I_or_X, Q   the input: I and Q with the pre-processor front or none, the real input X with Q == NULL for the generator
 *   audio       SDR_FMT_I16 or SDR_FMT_F32 (out_fmt), as the receiver's wire formats (sdr_batch.h)
 * submit_host queues the call on the graph's streams and returns; calls submitted back to back overlap (the first copy-in
 * of a call runs beside the drain of the one before).  sdr_graph_host_ticket() right after a submit names that call; the
 * inputs must stay unchanged and every output unread until that call has been waited for (wait_host_ticket or wait_host).
 * process_host = submit_host + wait for that call.  n_blocks is bounded by the receiver's max_blocks_per_call (if any) and
 * by 2^24. */
int sdr_graph_submit_host(sdr_graph_t *g, const uint32_t *ids, uint32_t n_ids, const int16_t *I_or_X, const int16_t *Q,
                          size_t in_pitch, void *audio, size_t out_pitch, int out_fmt, uint32_t n_blocks, const sdr_graph_outputs *o);
int sdr_graph_process_host(sdr_graph_t *g, const uint32_t *ids, uint32_t n_ids, const int16_t *I_or_X, const int16_t *Q,
                           size_t in_pitch, void *audio, size_t out_pitch, int out_fmt, uint32_t n_blocks, const sdr_graph_outputs *o);
/* Waterfall lines from the grabber tap (sdr_waterfall_*, sdr_aux.h).  attach_waterfall gives a graph with a grabber a
 * waterfall handle on the same device with the same channel count (NULL detaches it; not while calls are in flight that
 * use it: attach waits for them).  While one is attached, the graph's calls are the _waterfall forms, which equal, bit for
 * bit, one sdr_grabber_process_device_waterfall over the whole call in place of the grabber's device call:
 *   lines        host, float [n_ids][Lmax][256], 16-byte aligned, Lmax = (K - 1 + (n_blocks + 1) / 2) / K: row i's lines of
 *                the call in slots 0 .. line_counts[i] - 1; later slots keep what they held.
 *   line_counts  host, uint32 [n_ids] or NULL, filled before submit returns.
 * The lines are gathered on the device and each chunk's completed line slots come down in one copy.  o->power, o->snapshots
 * and o->counts are not available with a waterfall (SDR_ERR_ARG); the plain calls are SDR_ERR_ARG while one is attached. */
int sdr_graph_attach_waterfall(sdr_graph_t *g, sdr_waterfall_t *wf);
int sdr_graph_submit_host_waterfall(sdr_graph_t *g, const uint32_t *ids, uint32_t n_ids, const int16_t *I_or_X, const int16_t *Q,
                                    size_t in_pitch, void *audio, size_t out_pitch, int out_fmt, uint32_t n_blocks, const sdr_graph_outputs *o,
                                    float *lines, uint32_t *line_counts);
int sdr_graph_process_host_waterfall(sdr_graph_t *g, const uint32_t *ids, uint32_t n_ids, const int16_t *I_or_X, const int16_t *Q,
                                     size_t in_pitch, void *audio, size_t out_pitch, int out_fmt, uint32_t n_blocks, const sdr_graph_outputs *o,
                                     float *lines, uint32_t *line_counts);
/* The latest call's ticket (1, 2, ...; 0 before the first).  Calls complete in order. */
uint64_t sdr_graph_host_ticket(const sdr_graph_t *g);
/* Returns when everything submitted so far has landed / when call `ticket` has landed (later calls stay in flight). */
int sdr_graph_wait_host(sdr_graph_t *g);
int sdr_graph_wait_host_ticket(sdr_graph_t *g, uint64_t ticket);

const char *sdr_graph_last_error(void);
const char *sdr_graph_version(void);

#ifdef __cplusplus
}
#endif
#endif
