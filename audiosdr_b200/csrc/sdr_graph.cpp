/* sdr_graph.cpp -- include/sdr_graph.h: the sketch's receiver graph streamed from host memory over existing block handles.
 *
 * No signal processing here: per time chunk the graph copies the chunk's input planes up on its H2D stream, runs the
 * blocks' own device entry points (libsdr_aux.so, libsdr_batch.so) on its compute stream and copies the outputs down on its
 * D2H stream.  Two staging sets alternate from chunk to chunk and from call to call, as in the receiver's host path
 * (sdr_host.cpp, host_call), so that the copy-in of chunk k + 1, the kernels of chunk k and the copy-out of chunk k - 1
 * overlap.  The intermediate I/Q planes are one set: every kernel that reads or writes them runs on the compute stream.
 */
#include <stdlib.h>
#include <string.h>

#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/sdr_graph.h"

namespace {

thread_local std::string g_err;
int fail(int code, const std::string &msg) { g_err = msg; return code; }

/* a member's error as a graph error, with the member's text */
int from_aux(int rc, const char *what) {
  if (rc == 0) return 0;
  const int code = rc == SDR_AUX_EINVAL ? SDR_ERR_ARG : rc == SDR_AUX_ENOMEM ? SDR_ERR_NOMEM : SDR_ERR_CUDA;
  return fail(code, std::string(what) + ": " + sdr_aux_last_error());
}
int from_rx(int rc) { return rc ? fail(rc, std::string("receiver: ") + sdr_batch_last_error()) : 0; }

#define CU(call)                                                                           \
  do {                                                                                     \
    cudaError_t e_ = (call);                                                               \
    if (e_ != cudaSuccess) return fail(SDR_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
  } while (0)

enum { GRAPH_TICKETS = 8 }; /* calls whose completion can be waited for one by one */

/* a device buffer that grows on demand */
struct Buf {
  void *p = nullptr; size_t cap = 0;
  int ensure(size_t n) {
    if (n <= cap) return 0;
    cudaFree(p); p = nullptr; cap = 0; /* (a failed allocation leaves no stale size behind) */
    if (cudaMalloc(&p, n) != cudaSuccess) { cudaGetLastError(); return fail(SDR_ERR_NOMEM, "cudaMalloc(graph staging) failed"); }
    cap = n;
    return 0;
  }
  void release() { cudaFree(p); p = nullptr; cap = 0; }
};

int env_positive(const char *name, int dflt) {
  const char *e = getenv(name);
  const int v = e ? atoi(e) : 0;
  return v > 0 ? v : dflt;
}

}  // namespace

struct sdr_graph {
  sdr_graph_desc d;
  uint32_t n_ch; int device; uint32_t max_blocks;
  cudaStream_t s_h2d, s_comp, s_d2h;
  cudaEvent_t ev_h2d[2], ev_comp[2], ev_d2h[2], ev_call[GRAPH_TICKETS];
  /* per staging set: input planes (I, Q or X), audio, receiver and pre-processor records, spectra, snapshots */
  Buf in_a[2], in_b[2], audio[2], rx_rec[2], pp_rec[2], power[2], snaps[2];
  Buf mid_i, mid_q; /* the front's output: the tap's and the receiver's input */
  uint64_t seq;     /* chunks queued since create: chunk n uses staging set n & 1 */
  uint64_t calls;   /* calls queued since create (= the latest ticket) */
  std::vector<uint8_t> mark;
  std::vector<uint32_t> counts, chunk_counts;
  sdr_waterfall_t *wf; /* attached waterfall or NULL */
  Buf wf_lines[2];     /* a whole call's lines [rows][Lmax][256], by call parity */
  std::vector<uint32_t> line_first; /* per row: lines of the call so far = the next chunk's first slot */
};

static int check_ids(sdr_graph *g, const uint32_t *ids, uint32_t n_ids) {
  if (!ids) return n_ids == g->n_ch ? 0 : fail(SDR_ERR_ARG, "ids == NULL needs n_ids == n_channels");
  if (n_ids == 0) return fail(SDR_ERR_ARG, "n_ids == 0");
  uint32_t i = 0;
  for (; i < n_ids && ids[i] < g->n_ch && !g->mark[ids[i]]; i++) g->mark[ids[i]] = 1;
  for (uint32_t k = 0; k < i; k++) g->mark[ids[k]] = 0;
  if (i == n_ids) return 0;
  return fail(SDR_ERR_ARG, ids[i] >= g->n_ch ? "channel id out of range" : "channel id listed twice");
}

static int drain(sdr_graph *g) {
  const cudaError_t a = cudaStreamSynchronize(g->s_d2h), b = cudaStreamSynchronize(g->s_comp), c = cudaStreamSynchronize(g->s_h2d);
  const cudaError_t e = a != cudaSuccess ? a : b != cudaSuccess ? b : c;
  return e == cudaSuccess ? 0 : fail(SDR_ERR_CUDA, std::string("graph streams: ") + cudaGetErrorString(e));
}

extern "C" void sdr_graph_destroy(sdr_graph_t *g) {
  if (!g) return;
  cudaSetDevice(g->device);
  if (g->s_comp) drain(g);
  /* the receiver orders its later calls, getters and destruction after the compute stream it last ran on: it must not
   * keep a stream destroyed here */
  if (g->s_comp) sdr_batch_release_stream(g->d.rx, g->s_comp);
  for (int k = 0; k < 2; k++) {
    for (Buf *b : {&g->in_a[k], &g->in_b[k], &g->audio[k], &g->rx_rec[k], &g->pp_rec[k], &g->power[k], &g->snaps[k]}) b->release();
    for (cudaEvent_t e : {g->ev_h2d[k], g->ev_comp[k], g->ev_d2h[k]}) if (e) cudaEventDestroy(e);
  }
  for (cudaEvent_t e : g->ev_call) if (e) cudaEventDestroy(e);
  g->mid_i.release(); g->mid_q.release(); g->wf_lines[0].release(); g->wf_lines[1].release();
  for (cudaStream_t s : {g->s_h2d, g->s_comp, g->s_d2h}) if (s) cudaStreamDestroy(s);
  delete g;
}

extern "C" int sdr_graph_create(sdr_graph_t **out, const sdr_graph_desc *desc) {
  if (!out || !desc || !desc->rx) return fail(SDR_ERR_ARG, "create: bad arguments (the receiver is required)");
  *out = nullptr;
  if (desc->pp && desc->gen) return fail(SDR_ERR_ARG, "create: at most one front (pre-processor or I/Q generator)");
  sdr_batch_desc rd;
  if (int rc = from_rx(sdr_batch_get_desc(desc->rx, &rd))) return rc;
  struct { const char *what; int rc; uint32_t n; int dev; } m[3] = {{"pre-processor", 0, 0, 0}, {"I/Q generator", 0, 0, 0}, {"grabber", 0, 0, 0}};
  if (desc->pp) m[0].rc = sdr_preproc_get_info(desc->pp, &m[0].n, &m[0].dev);
  if (desc->gen) m[1].rc = sdr_iqgen_get_info(desc->gen, &m[1].n, &m[1].dev);
  if (desc->grabber) m[2].rc = sdr_grabber_get_info(desc->grabber, &m[2].n, &m[2].dev);
  const bool used[3] = {desc->pp != nullptr, desc->gen != nullptr, desc->grabber != nullptr};
  for (int k = 0; k < 3; k++) {
    if (!used[k]) continue;
    if (int rc = from_aux(m[k].rc, m[k].what)) return rc;
    if (m[k].n != rd.n_channels) return fail(SDR_ERR_ARG, std::string("create: the ") + m[k].what + " has another channel count than the receiver");
    if (m[k].dev != rd.device) return fail(SDR_ERR_ARG, std::string("create: the ") + m[k].what + " is on another device than the receiver");
  }
  CU(cudaSetDevice(rd.device));
  sdr_graph *g = new sdr_graph();
  g->d = *desc; g->n_ch = rd.n_channels; g->device = rd.device; g->max_blocks = rd.max_blocks_per_call;
  g->s_h2d = g->s_comp = g->s_d2h = nullptr;
  for (int k = 0; k < 2; k++) g->ev_h2d[k] = g->ev_comp[k] = g->ev_d2h[k] = nullptr;
  for (auto &e : g->ev_call) e = nullptr;
  g->seq = g->calls = 0;
  g->wf = nullptr;
  g->mark.assign(g->n_ch, 0);
  int rc = 0;
  auto stream = [&](cudaStream_t *s) { if (!rc && cudaStreamCreateWithFlags(s, cudaStreamNonBlocking) != cudaSuccess) rc = fail(SDR_ERR_CUDA, "cudaStreamCreate failed"); };
  auto event = [&](cudaEvent_t *e) { if (!rc && cudaEventCreateWithFlags(e, cudaEventDisableTiming) != cudaSuccess) rc = fail(SDR_ERR_CUDA, "cudaEventCreate failed"); };
  /* non-blocking streams: the graph's work does not serialise with the legacy default stream (the aux blocks' host calls) */
  stream(&g->s_h2d); stream(&g->s_comp); stream(&g->s_d2h);
  for (int k = 0; k < 2; k++) { event(&g->ev_h2d[k]); event(&g->ev_comp[k]); event(&g->ev_d2h[k]); }
  for (auto &e : g->ev_call) event(&e);
  if (rc) { std::string keep = g_err; sdr_graph_destroy(g); g_err = keep; return rc; }
  *out = g;
  return SDR_OK;
}

extern "C" uint64_t sdr_graph_host_ticket(const sdr_graph_t *g) { return g ? g->calls : 0; }

extern "C" int sdr_graph_wait_host(sdr_graph_t *g) {
  if (!g) return fail(SDR_ERR_ARG, "wait_host: bad arguments");
  CU(cudaSetDevice(g->device));
  return drain(g);
}

extern "C" int sdr_graph_wait_host_ticket(sdr_graph_t *g, uint64_t ticket) {
  if (!g) return fail(SDR_ERR_ARG, "wait_host_ticket: bad arguments");
  if (ticket > g->calls) return fail(SDR_ERR_ARG, "wait_host_ticket: no such call yet");
  if (ticket == 0) return SDR_OK;
  CU(cudaSetDevice(g->device));
  /* copy-outs complete in the order of the calls: a ticket whose event has been reused is covered by the oldest one kept */
  const uint64_t oldest = g->calls >= GRAPH_TICKETS ? g->calls - GRAPH_TICKETS + 1 : 1;
  CU(cudaEventSynchronize(g->ev_call[(ticket < oldest ? oldest : ticket) % GRAPH_TICKETS]));
  return SDR_OK;
}

/* Chunk length in blocks: the receiver's host path's choice (about 6 chunks per streamed call, 12 per synchronous one, at
 * least SDR_HOST_MIN_CHUNK = 16 blocks; SDR_HOST_CHUNKS overrides the count), rounded up to an even number of blocks so
 * that every chunk but the last starts at an even block of the call. */
static uint32_t chunk_blocks(const sdr_graph *g, uint32_t n_blocks, bool streamed) {
  static const uint32_t env_chunks = (uint32_t)env_positive("SDR_HOST_CHUNKS", 0);
  static const uint32_t min_chunk = (uint32_t)env_positive("SDR_HOST_MIN_CHUNK", 16);
  const uint32_t want = env_chunks ? env_chunks : (streamed ? 6u : 12u);
  uint32_t c = (n_blocks + want - 1) / want;
  if (c < min_chunk) c = min_chunk;
  c += c & 1;
  if (g->max_blocks >= 2 && c > g->max_blocks) c = g->max_blocks & ~1u;
  return c < n_blocks ? c : n_blocks;
}

extern "C" int sdr_graph_attach_waterfall(sdr_graph_t *g, sdr_waterfall_t *wf) {
  if (!g) return fail(SDR_ERR_ARG, "attach_waterfall: bad arguments");
  if (wf) {
    if (!g->d.grabber) return fail(SDR_ERR_ARG, "attach_waterfall: the graph has no grabber");
    uint32_t n = 0, K = 0; int dev = 0;
    if (int rc = from_aux(sdr_waterfall_get_info(wf, &n, &dev, &K), "waterfall")) return rc;
    if (n != g->n_ch || dev != g->device) return fail(SDR_ERR_ARG, "attach_waterfall: the waterfall must have the graph's device and channel count");
  }
  CU(cudaSetDevice(g->device));
  if (int rc = drain(g)) return rc; /* calls in flight use the waterfall attached before */
  g->wf = wf;
  return SDR_OK;
}

static int graph_call(sdr_graph *g, const uint32_t *ids, uint32_t n_ids, const int16_t *I, const int16_t *Q, size_t in_pitch,
                      void *audio, size_t out_pitch, int out_fmt, uint32_t n_blocks, const sdr_graph_outputs *o, bool streamed,
                      bool with_lines, float *lines, uint32_t *line_counts) {
  /* ---- every argument, before anything is queued */
  if (!g || !I || !audio) return fail(SDR_ERR_ARG, "submit_host: bad arguments");
  if (with_lines != (g->wf != nullptr))
    return fail(SDR_ERR_ARG, g->wf ? "a graph with a waterfall takes the _waterfall calls" : "the _waterfall calls need an attached waterfall");
  uint32_t K = 1, Lmax = 0;
  if (g->wf) {
    uint32_t n = 0; int dev = 0;
    if (int rc = from_aux(sdr_waterfall_get_info(g->wf, &n, &dev, &K), "waterfall")) return rc;
    if (!lines || ((uintptr_t)lines & 15)) return fail(SDR_ERR_ARG, "lines must be non-NULL and 16-byte aligned");
    if (o && (o->power || o->snapshots || o->counts)) return fail(SDR_ERR_ARG, "power, snapshots and counts are not available with a waterfall");
    if (n_blocks) Lmax = (uint32_t)(((unsigned long long)K - 1 + (n_blocks + 1) / 2) / K);
  }
  if (int rc = check_ids(g, ids, n_ids)) return rc;
  if (n_blocks == 0) return fail(SDR_ERR_ARG, "n_blocks == 0");
  if (n_blocks > (1u << 24)) return fail(SDR_ERR_ARG, "n_blocks too large (at most 2^24 blocks per call)");
  if (g->max_blocks && n_blocks > g->max_blocks) return fail(SDR_ERR_ARG, "n_blocks > the receiver's max_blocks_per_call");
  if (g->d.gen ? Q != nullptr : Q == nullptr)
    return fail(SDR_ERR_ARG, g->d.gen ? "the I/Q generator front takes one real input plane: Q must be NULL" : "Q == NULL");
  if (out_fmt != SDR_FMT_I16 && out_fmt != SDR_FMT_F32) return fail(SDR_ERR_ARG, "unknown output format");
  const size_t ns = (size_t)n_blocks * 128;
  if (in_pitch < ns || out_pitch < ns) return fail(SDR_ERR_ARG, "pitch shorter than the call");
  const sdr_graph_outputs none = {nullptr, nullptr, nullptr, nullptr, nullptr};
  const sdr_graph_outputs &out = o ? *o : none;
  if (out.pp_status && !g->d.pp) return fail(SDR_ERR_ARG, "pp_status needs the pre-processor front");
  if ((out.power || out.snapshots || out.counts) && !g->d.grabber) return fail(SDR_ERR_ARG, "power, snapshots and counts need the grabber");
  if (((uintptr_t)out.rx_status | (uintptr_t)out.pp_status | (uintptr_t)out.power | (uintptr_t)out.snapshots) & 15)
    return fail(SDR_ERR_ARG, "record, power and snapshot buffers must be 16-byte aligned");
  CU(cudaSetDevice(g->device));

  /* ---- staging for one chunk */
  const uint32_t chunk = chunk_blocks(g, n_blocks, streamed), rows = n_ids;
  const size_t cs = (size_t)chunk * 128, cslots = (chunk + 1) / 2, oes = out_fmt == SDR_FMT_F32 ? 4 : 2;
  const size_t need[7] = {cs * 2 * rows, Q ? cs * 2 * rows : 0, cs * oes * rows, out.rx_status ? (size_t)chunk * SDR_BS_FIELDS * rows * 4 : 0,
                          out.pp_status ? (size_t)chunk * SDR_PP_BS_FIELDS * rows * 4 : 0, out.power ? cslots * 1024 * rows : 0,
                          out.snapshots ? cslots * 1024 * rows : 0};
  const size_t mid = g->d.pp || g->d.gen ? cs * 2 * rows : 0, lines_bytes = g->wf ? (size_t)(Lmax ? Lmax : 1) * 1024 * rows : 0;
  bool grow = mid > g->mid_i.cap || lines_bytes > g->wf_lines[0].cap;
  for (int k = 0; k < 2; k++) {
    const Buf *b[7] = {&g->in_a[k], &g->in_b[k], &g->audio[k], &g->rx_rec[k], &g->pp_rec[k], &g->power[k], &g->snaps[k]};
    for (int j = 0; j < 7; j++) grow |= need[j] > b[j]->cap;
  }
  if (grow) {
    if (int rc = drain(g)) return rc; /* the old buffers may still be read or written by calls in flight */
    for (int k = 0; k < 2; k++) {
      Buf *b[7] = {&g->in_a[k], &g->in_b[k], &g->audio[k], &g->rx_rec[k], &g->pp_rec[k], &g->power[k], &g->snaps[k]};
      for (int j = 0; j < 7; j++) if (int rc = b[j]->ensure(need[j])) return rc;
    }
    if (int rc = g->mid_i.ensure(mid)) return rc;
    if (int rc = g->mid_q.ensure(mid)) return rc;
    for (Buf &b : g->wf_lines) if (int rc = b.ensure(lines_bytes)) return rc;
  }

  /* ---- the chunks */
  const size_t S = (n_blocks + 1) / 2; /* slots per row of the caller's power / snapshots */
  if (g->d.grabber) { g->counts.assign(rows, 0); g->chunk_counts.assign(rows, 0); }
  int err = 0;
#define GR_TRY(expr) if ((err = (expr)) != 0) break
#define GR_CU(call) if ((call) != cudaSuccess) { err = fail(SDR_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(cudaGetLastError())); break; }
  /* Waterfall: each chunk's grabber call puts row r's lines at slot line_first[r] of the call's device buffer wl, where the
   * uncut call would put them.  After a chunk every row has completed the slots below the least line_first, and no later
   * chunk writes them: they come down in one copy.  A row's final count is at least Lmax - 1 (rows differ in their held
   * pairs, < K, and by at most one pair of their phase), so only slot Lmax - 1 may be left unwritten by some rows: it is
   * loaded with the caller's lines first, and the last chunk copies it down whole. */
  float *wl = g->wf ? (float *)g->wf_lines[(g->calls + 1) & 1].p : nullptr;
  const size_t lp = (size_t)Lmax * 1024; /* bytes per row of wl and of the caller's lines */
  uint32_t copied = 0;
  if (g->wf) {
    g->line_first.assign(rows, 0);
    do {
      /* wl was last read by the final copy of the call two before this one */
      if (g->calls >= 2) GR_CU(cudaStreamWaitEvent(g->s_h2d, g->ev_call[(g->calls - 1) % GRAPH_TICKETS], 0));
      if (Lmax) GR_CU(cudaMemcpy2DAsync(wl + (size_t)(Lmax - 1) * 256, lp, lines + (size_t)(Lmax - 1) * 256, lp, 1024, rows, cudaMemcpyHostToDevice, g->s_h2d));
    } while (0);
  }
  for (uint32_t done = 0; done < n_blocks && !err;) {
    const uint32_t nb = n_blocks - done < chunk ? n_blocks - done : chunk;
    const size_t w = (size_t)nb * 128;
    const int b = (int)(g->seq & 1);
    int16_t *in_a = (int16_t *)g->in_a[b].p, *in_b = (int16_t *)g->in_b[b].p;
    /* H2D of the chunk into set b: the kernels of chunk seq - 2 (of this call or the one before) must be done with it */
    if (g->seq >= 2) GR_CU(cudaStreamWaitEvent(g->s_h2d, g->ev_comp[b], 0));
    GR_CU(cudaMemcpy2DAsync(in_a, cs * 2, I + (size_t)done * 128, in_pitch * 2, w * 2, rows, cudaMemcpyHostToDevice, g->s_h2d));
    if (Q) GR_CU(cudaMemcpy2DAsync(in_b, cs * 2, Q + (size_t)done * 128, in_pitch * 2, w * 2, rows, cudaMemcpyHostToDevice, g->s_h2d));
    GR_CU(cudaEventRecord(g->ev_h2d[b], g->s_h2d));
    /* the blocks: they need the input, and the D2H of chunk seq - 2 must have drained output set b */
    GR_CU(cudaStreamWaitEvent(g->s_comp, g->ev_h2d[b], 0));
    if (g->seq >= 2) GR_CU(cudaStreamWaitEvent(g->s_comp, g->ev_d2h[b], 0));
    const int16_t *ri = in_a, *rq = in_b; /* the receiver's input: the front's output, or the call's input */
    if (g->d.pp) {
      GR_TRY(from_aux(sdr_preproc_process_device_status(g->d.pp, ids, n_ids, in_a, in_b, cs, (int16_t *)g->mid_i.p, (int16_t *)g->mid_q.p, cs, nb,
                                                        out.pp_status ? (int32_t *)g->pp_rec[b].p : nullptr, g->s_comp), "pre-processor"));
      ri = (const int16_t *)g->mid_i.p; rq = (const int16_t *)g->mid_q.p;
    } else if (g->d.gen) {
      GR_TRY(from_aux(sdr_iqgen_process_device_subset(g->d.gen, ids, n_ids, in_a, cs, (int16_t *)g->mid_i.p, (int16_t *)g->mid_q.p, cs, nb, g->s_comp),
                      "I/Q generator"));
      ri = (const int16_t *)g->mid_i.p; rq = (const int16_t *)g->mid_q.p;
    }
    if (g->wf) {
      GR_TRY(from_aux(sdr_grabber_process_device_waterfall_at(g->d.grabber, g->wf, ids, n_ids, ri, rq, cs, nb, wl, Lmax, g->line_first.data(),
                                                              g->chunk_counts.data(), g->s_comp), "grabber"));
    } else if (g->d.grabber) {
      GR_TRY(from_aux(sdr_grabber_process_device_snapshots(g->d.grabber, ids, n_ids, ri, rq, cs, nb, out.snapshots ? (int16_t *)g->snaps[b].p : nullptr,
                                                           out.power ? (float *)g->power[b].p : nullptr, g->chunk_counts.data(), g->s_comp),
                      "grabber"));
    }
    GR_TRY(from_rx(sdr_batch_process_device_subset(g->d.rx, ids, n_ids, ri, rq, cs, SDR_FMT_I16, g->audio[b].p, cs, out_fmt, nb,
                                                    out.rx_status ? g->rx_rec[b].p : nullptr, g->s_comp)));
    GR_CU(cudaEventRecord(g->ev_comp[b], g->s_comp));
    /* D2H of the chunk: audio, then the records (block-major: the chunk's blocks are one contiguous range of the caller's
     * buffer), then the spectra and snapshots (slots done/2 onward of every row) */
    GR_CU(cudaStreamWaitEvent(g->s_d2h, g->ev_comp[b], 0));
    GR_CU(cudaMemcpy2DAsync((char *)audio + (size_t)done * 128 * oes, out_pitch * oes, g->audio[b].p, cs * oes, w * oes, rows, cudaMemcpyDeviceToHost, g->s_d2h));
    if (out.rx_status) {
      const size_t rec = (size_t)SDR_BS_FIELDS * rows * 4;
      GR_CU(cudaMemcpyAsync((char *)out.rx_status + (size_t)done * rec, g->rx_rec[b].p, nb * rec, cudaMemcpyDeviceToHost, g->s_d2h));
    }
    if (out.pp_status) {
      const size_t rec = (size_t)SDR_PP_BS_FIELDS * rows * 4;
      GR_CU(cudaMemcpyAsync((char *)out.pp_status + (size_t)done * rec, g->pp_rec[b].p, nb * rec, cudaMemcpyDeviceToHost, g->s_d2h));
    }
    if (g->wf) {
      uint32_t lo = UINT32_MAX;
      for (uint32_t r = 0; r < rows; r++) { g->line_first[r] += g->chunk_counts[r]; lo = g->line_first[r] < lo ? g->line_first[r] : lo; }
      const uint32_t hi = done + nb == n_blocks ? Lmax : lo;
      if (hi > copied)
        GR_CU(cudaMemcpy2DAsync(lines + (size_t)copied * 256, lp, wl + (size_t)copied * 256, lp, (size_t)(hi - copied) * 1024, rows, cudaMemcpyDeviceToHost, g->s_d2h));
      copied = hi;
    } else if (g->d.grabber) {
      /* rows in runs of equal slot counts: a row writes (phase + nb) / 2 slots of the chunk, and the slot a row does not
       * write (an odd last chunk and phase 0) must keep what the caller's buffer holds */
      for (uint32_t r0 = 0; r0 < rows && !err;) {
        const uint32_t c = g->chunk_counts[r0];
        uint32_t r1 = r0 + 1;
        while (r1 < rows && g->chunk_counts[r1] == c) r1++;
        if (c) {
          /* the grabber lays the chunk's slots out as its own call of nb blocks: (nb + 1) / 2 per row */
          const size_t ks = (nb + 1) / 2, dst = (size_t)r0 * S + done / 2, src = (size_t)r0 * ks;
          if (out.power && cudaMemcpy2DAsync(out.power + dst * 256, S * 1024, (float *)g->power[b].p + src * 256, ks * 1024, c * 1024, r1 - r0,
                                             cudaMemcpyDeviceToHost, g->s_d2h) != cudaSuccess)
            err = fail(SDR_ERR_CUDA, std::string("copy of the spectra: ") + cudaGetErrorString(cudaGetLastError()));
          if (!err && out.snapshots && cudaMemcpy2DAsync(out.snapshots + dst * 512, S * 1024, (int16_t *)g->snaps[b].p + src * 512, ks * 1024, c * 1024,
                                                         r1 - r0, cudaMemcpyDeviceToHost, g->s_d2h) != cudaSuccess)
            err = fail(SDR_ERR_CUDA, std::string("copy of the snapshots: ") + cudaGetErrorString(cudaGetLastError()));
        }
        for (uint32_t r = r0; r < r1; r++) g->counts[r] += c;
        r0 = r1;
      }
      if (err) break;
    }
    GR_CU(cudaEventRecord(g->ev_d2h[b], g->s_d2h));
    done += nb; g->seq++;
  }
#undef GR_TRY
#undef GR_CU
  /* on a failure the streams are drained before returning: asynchronous copies into the caller's buffers must not outlive
   * the call */
  if (err) { drain(g); return err; }
  if (out.counts) memcpy(out.counts, g->counts.data(), 4 * (size_t)rows);
  if (line_counts) memcpy(line_counts, g->line_first.data(), 4 * (size_t)rows);
  /* the call's ticket: its last copy-out is the last thing in the D2H stream */
  g->calls++;
  CU(cudaEventRecord(g->ev_call[g->calls % GRAPH_TICKETS], g->s_d2h));
  return SDR_OK;
}

extern "C" int sdr_graph_submit_host(sdr_graph_t *g, const uint32_t *ids, uint32_t n_ids, const int16_t *I_or_X, const int16_t *Q, size_t in_pitch,
                                     void *audio, size_t out_pitch, int out_fmt, uint32_t n_blocks, const sdr_graph_outputs *o) {
  return graph_call(g, ids, n_ids, I_or_X, Q, in_pitch, audio, out_pitch, out_fmt, n_blocks, o, true, false, nullptr, nullptr);
}

extern "C" int sdr_graph_process_host(sdr_graph_t *g, const uint32_t *ids, uint32_t n_ids, const int16_t *I_or_X, const int16_t *Q, size_t in_pitch,
                                      void *audio, size_t out_pitch, int out_fmt, uint32_t n_blocks, const sdr_graph_outputs *o) {
  if (int rc = graph_call(g, ids, n_ids, I_or_X, Q, in_pitch, audio, out_pitch, out_fmt, n_blocks, o, false, false, nullptr, nullptr)) return rc;
  return sdr_graph_wait_host_ticket(g, g->calls);
}

extern "C" int sdr_graph_submit_host_waterfall(sdr_graph_t *g, const uint32_t *ids, uint32_t n_ids, const int16_t *I_or_X, const int16_t *Q,
                                               size_t in_pitch, void *audio, size_t out_pitch, int out_fmt, uint32_t n_blocks,
                                               const sdr_graph_outputs *o, float *lines, uint32_t *line_counts) {
  return graph_call(g, ids, n_ids, I_or_X, Q, in_pitch, audio, out_pitch, out_fmt, n_blocks, o, true, true, lines, line_counts);
}

extern "C" int sdr_graph_process_host_waterfall(sdr_graph_t *g, const uint32_t *ids, uint32_t n_ids, const int16_t *I_or_X, const int16_t *Q,
                                                size_t in_pitch, void *audio, size_t out_pitch, int out_fmt, uint32_t n_blocks,
                                                const sdr_graph_outputs *o, float *lines, uint32_t *line_counts) {
  if (int rc = graph_call(g, ids, n_ids, I_or_X, Q, in_pitch, audio, out_pitch, out_fmt, n_blocks, o, false, true, lines, line_counts)) return rc;
  return sdr_graph_wait_host_ticket(g, g->calls);
}

extern "C" const char *sdr_graph_last_error(void) { return g_err.c_str(); }
extern "C" const char *sdr_graph_version(void) { return "audiosdr_b200 graph 0.1 (sm_100a)"; }
