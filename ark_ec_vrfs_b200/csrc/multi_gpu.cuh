// Several GPUs of one node behind the C ABI (SURVEY.md 8e; included at the end of vrfs_b200.cu, host code only).
//
// Two deployment shapes share the device-side exchange of msm.cuh (PeerBox / PeerArgs / k_msm_final2 out_mode 2):
//  (1) one process per GPU (torch.distributed / torchrun): every rank owns an ordinary context, exports its mailbox as a CUDA
//      IPC handle (vrfs_ctx_peer_export), the 64-byte handles travel once over the caller's control plane (a host all-gather),
//      and vrfs_ctx_peer_connect maps the peers.  The *_allgather entry points are then collective calls: every rank computes
//      the partial commitment of its point range and the final kernel exchanges and folds the partials over NVLink.
//  (2) one caller, several GPUs (the `vrfs_ctx_create(const int* devices, int n_devices, ..)` of SURVEY 8b): vrfs_ctx_create_multi
//      owns one context per device, wires their mailboxes with plain peer access, shards verify batches by index range (no
//      collective) and runs the same MSM exchange with device 0 as the only folding rank.
// VRF batches never communicate; the MSM exchanges 144 bytes per column per rank.
#pragma once

// ---- peer group plumbing ------------------------------------------------------------------------------------------------------
static void peer_teardown(vrfs_ctx* ctx) {
  auto& P = ctx->peer;
  for (int r = 0; r < VRFS_MAX_PEERS; r++) {
    if (!P.box[r]) continue;
    if (r == P.rank && !P.ipc[r]) cudaFree(P.box[r]);
    else if (P.ipc[r]) cudaIpcCloseMemHandle(P.box[r]);
    P.box[r] = nullptr; P.ipc[r] = false;
  }
  if (P.timed_out) { cudaFreeHost(P.timed_out); P.timed_out = nullptr; }
  P.world = 0; P.epoch = 0;
}
// this rank's mailbox + the host-visible status word
static vrfs_status peer_alloc(vrfs_ctx* ctx, int rank, int world) {
  if (world < 1 || world > VRFS_MAX_PEERS || rank < 0 || rank >= world) return fail(ctx, VRFS_BAD_ARG, "need 0 <= rank < world <= %d", VRFS_MAX_PEERS);
  CU(cudaSetDevice(ctx->device));
  CU(cudaStreamSynchronize(ctx->stream));
  peer_teardown(ctx);
  auto& P = ctx->peer;
  void* box = nullptr;
  CU(cudaMalloc(&box, sizeof(PeerBox)));
  CU(cudaMemset(box, 0, sizeof(PeerBox)));
  CU(cudaHostAlloc((void**)&P.timed_out, sizeof(unsigned int), cudaHostAllocMapped | cudaHostAllocPortable));
  *P.timed_out = 0;
  CU(cudaDeviceSynchronize());
  P.rank = rank; P.box[rank] = (PeerBox*)box; P.ipc[rank] = false; P.epoch = 0;
  P.world = 0;                                         // not usable until connected
  return VRFS_OK;
}
extern "C" vrfs_status vrfs_ctx_peer_export(vrfs_ctx* ctx, int rank, int world, uint8_t* out_handle) {
  if (!ctx || !out_handle) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  static_assert(sizeof(cudaIpcMemHandle_t) == VRFS_PEER_HANDLE_BYTES, "cudaIpcMemHandle_t is 64 bytes");
  ST(peer_alloc(ctx, rank, world));
  cudaIpcMemHandle_t h;
  CU(cudaIpcGetMemHandle(&h, ctx->peer.box[rank]));
  memcpy(out_handle, &h, sizeof h);
  ctx->peer.world = -world;                            // exported, waiting for vrfs_ctx_peer_connect
  return VRFS_OK;
}
extern "C" vrfs_status vrfs_ctx_peer_connect(vrfs_ctx* ctx, const uint8_t* handles) {
  if (!ctx || !handles) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  auto& P = ctx->peer;
  if (P.world >= 0) return fail(ctx, VRFS_BAD_ARG, "vrfs_ctx_peer_export must come first");
  const int world = -P.world;
  CU(cudaSetDevice(ctx->device));
  for (int r = 0; r < world; r++) {
    if (r == P.rank) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, handles + (size_t)r * VRFS_PEER_HANDLE_BYTES, sizeof h);
    void* p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) return fail(ctx, VRFS_CUDA_ERROR, "cudaIpcOpenMemHandle of rank %d's mailbox failed: %s (the ranks must be GPUs of one node with peer access)", r, cudaGetErrorString(e));
    P.box[r] = (PeerBox*)p; P.ipc[r] = true;
  }
  P.world = world;
  return VRFS_OK;
}
extern "C" vrfs_status vrfs_ctx_peer_set_timeout_ms(vrfs_ctx* ctx, unsigned int ms) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  ctx->peer.timeout_ns = (unsigned long long)(ms ? ms : 1u) * 1000000ull;
  return VRFS_OK;
}
extern "C" int vrfs_ctx_peer_world(const vrfs_ctx* ctx) { return ctx && ctx->peer.world > 0 ? ctx->peer.world : 0; }

// arguments of this collective for the final kernel; every rank calls the collectives in the same order, so the epochs agree
static vrfs_status peer_begin(vrfs_ctx* ctx, int root, PeerArgs* A) {
  auto& P = ctx->peer;
  if (P.world <= 0) return fail(ctx, VRFS_BAD_ARG, "no peer group: vrfs_ctx_peer_export / vrfs_ctx_peer_connect first");
  P.epoch++;                                           // before anything that can fail: a failed call still consumes its epoch
  A->rank = P.rank; A->world = P.world; A->root = root; A->epoch = P.epoch; A->timeout_ns = P.timeout_ns;
  for (int r = 0; r < VRFS_MAX_PEERS; r++) A->box[r] = P.box[r];
  unsigned int* d = nullptr;
  CU(cudaHostGetDevicePointer((void**)&d, P.timed_out, 0));
  A->timed_out = d;
  return VRFS_OK;
}
static vrfs_status peer_check(vrfs_ctx* ctx) {          // after the stream was drained
  if (ctx->peer.timed_out && *ctx->peer.timed_out) {
    *ctx->peer.timed_out = 0;
    return fail(ctx, VRFS_CUDA_ERROR, "multi-GPU exchange timed out: a peer never delivered its partial sums (rank %d of %d)", ctx->peer.rank, ctx->peer.world);
  }
  return VRFS_OK;
}

// ---- collective entry points (one process per GPU) ------------------------------------------------------------------------------
// scalars of this rank's point range -> the FULL commitments on every rank
extern "C" vrfs_status vrfs_msm_g1_prepared_allgather(vrfs_ctx* ctx, const vrfs_msm_bases* h, const uint8_t* scalars, int n_columns, uint8_t* out) {
  if (!ctx || !h || h->ctx != ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  PeerArgs pa;
  ST(peer_begin(ctx, -1, &pa));
  if (n_columns < 1 || n_columns > VRFS_PEER_MAXCOL || !scalars || !out) return fail(ctx, VRFS_BAD_ARG, "bad argument");
  ST(begin_call(ctx, h->n));
  const uint8_t* d_s; uint8_t* d_o;
  ST(stage_in(ctx, BUF_IN1, scalars, h->n * 32 * (size_t)n_columns, &d_s));
  ST(stage_out(ctx, BUF_OUT0, (size_t)96 * n_columns, &d_o));
  ST(msm_prepared_dev(ctx, h, n_columns, 0, d_s, d_o, 2, &pa));
  ST(copy_out(ctx, out, d_o, (size_t)96 * n_columns));
  ST(finish_call(ctx));
  return peer_check(ctx);
}
// the ring commitment with the domain's rows split over the ranks (Lagrange-basis SRS): arguments as vrfs_ring_commit_rows_partial
extern "C" vrfs_status vrfs_ring_commit_rows_allgather(vrfs_ctx* ctx, const vrfs_msm_bases* srs_rows, size_t row_lo, size_t keyset_part_size, size_t n_keys,
                                                       const uint8_t* keys_rows, const uint8_t* padding, size_t n_tail, const uint8_t* tail, uint8_t* out_commitment) {
  if (!ctx || !srs_rows || srs_rows->ctx != ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  PeerArgs pa;
  ST(peer_begin(ctx, -1, &pa));
  if (!out_commitment) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  const size_t n = srs_rows->n;
  ST(begin_call(ctx, n));
  uint8_t *d_cols = nullptr, *d_o = nullptr;
  ST(ring_columns_dev(ctx, n, keyset_part_size, n_keys, keys_rows, padding, n_tail, tail, &d_cols, row_lo, false));
  ST(stage_out(ctx, BUF_OUT0, 3 * 96, &d_o));
  ST(msm_prepared_dev(ctx, srs_rows, 3, 1, d_cols, d_o, 2, &pa));
  ST(copy_out(ctx, out_commitment, d_o, 3 * 96));
  ST(finish_call(ctx));
  return peer_check(ctx);
}

// ---- one caller, several GPUs ------------------------------------------------------------------------------------------------
struct vrfs_mctx {
  int n = 0;
  vrfs_ctx* dev[VRFS_MAX_PEERS] = {nullptr};
  char err[600] = {0};
  std::mutex mu;
};
struct vrfs_multi_bases {
  vrfs_mctx* m;
  size_t n;
  size_t lo[VRFS_MAX_PEERS + 1];            // device g holds the bases [lo[g], lo[g+1])
  vrfs_msm_bases* part[VRFS_MAX_PEERS];
};
static vrfs_status mfail(vrfs_mctx* m, vrfs_status st, const char* fmt, ...) {
  if (m) { va_list ap; va_start(ap, fmt); vsnprintf(m->err, sizeof m->err, fmt, ap); va_end(ap); }
  return st;
}
// a failure on device g: keep its message
#define MST(m, g, call)                                                                                              \
  do {                                                                                                               \
    vrfs_status s_ = (call);                                                                                         \
    if (s_ != VRFS_OK) return mfail((m), s_, "device %d (cuda:%d): %s", (g), (m)->dev[g]->device, (m)->dev[g]->err); \
  } while (0)
extern "C" void vrfs_mctx_destroy(vrfs_mctx* m) {
  if (!m) return;
  for (int g = 0; g < m->n; g++) {
    if (!m->dev[g]) continue;
    // same-process mailboxes are plain pointers into the peers' allocations: forget them before the owners free them
    for (int r = 0; r < VRFS_MAX_PEERS; r++) if (r != m->dev[g]->peer.rank) m->dev[g]->peer.box[r] = nullptr;
  }
  for (int g = 0; g < m->n; g++) vrfs_ctx_destroy(m->dev[g]);
  delete m;
}
extern "C" vrfs_status vrfs_ctx_create_multi(const int* devices, int n_devices, vrfs_mctx** out) {
  if (!out) return VRFS_BAD_ARG;
  *out = nullptr;
  vrfs_mctx* m = new (std::nothrow) vrfs_mctx();
  if (!m) return VRFS_CUDA_ERROR;
  *out = m;                                 // returned even on failure so that vrfs_mctx_last_error can be read; destroy it either way
  if (!devices || n_devices < 1 || n_devices > VRFS_MAX_PEERS) return mfail(m, VRFS_BAD_ARG, "need 1..%d devices", VRFS_MAX_PEERS);
  for (int g = 0; g < n_devices; g++) for (int k = 0; k < g; k++) if (devices[g] == devices[k]) return mfail(m, VRFS_BAD_ARG, "device %d listed twice", devices[g]);
  for (int g = 0; g < n_devices; g++) {
    vrfs_status st = vrfs_ctx_create(devices[g], &m->dev[g]);
    m->n = g + 1;
    if (st != VRFS_OK) return mfail(m, st, "cuda:%d: %s", devices[g], m->dev[g] ? m->dev[g]->err : "context allocation failed");
  }
  // mailboxes + peer access between every pair (NVLink / NVSwitch on a B200 node)
  for (int g = 0; g < n_devices; g++) { CallGuard guard_(m->dev[g]); MST(m, g, peer_alloc(m->dev[g], g, n_devices)); }
  for (int g = 0; g < n_devices; g++) {
    cudaSetDevice(devices[g]);
    for (int r = 0; r < n_devices; r++) {
      if (r == g) continue;
      int can = 0;
      cudaDeviceCanAccessPeer(&can, devices[g], devices[r]);
      if (!can) return mfail(m, VRFS_CUDA_ERROR, "cuda:%d cannot access cuda:%d as a peer", devices[g], devices[r]);
      cudaError_t e = cudaDeviceEnablePeerAccess(devices[r], 0);
      if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
      else if (e != cudaSuccess) return mfail(m, VRFS_CUDA_ERROR, "cudaDeviceEnablePeerAccess(cuda:%d -> cuda:%d): %s", devices[g], devices[r], cudaGetErrorString(e));
      m->dev[g]->peer.box[r] = m->dev[r]->peer.box[r];
    }
    m->dev[g]->peer.world = n_devices;
  }
  return VRFS_OK;
}
extern "C" int vrfs_mctx_device_count(const vrfs_mctx* m) { return m ? m->n : 0; }
extern "C" vrfs_ctx* vrfs_mctx_device_ctx(vrfs_mctx* m, int i) { return (m && i >= 0 && i < m->n) ? m->dev[i] : nullptr; }
extern "C" const char* vrfs_mctx_last_error(const vrfs_mctx* m) { return m ? m->err : "null context"; }
extern "C" uint64_t vrfs_mctx_launch_count(const vrfs_mctx* m) {
  uint64_t t = 0;
  if (m) for (int g = 0; g < m->n; g++) t += m->dev[g]->launches;
  return t;
}
static inline size_t mshard(size_t n, int g, int G) { return (n * (size_t)g) / (size_t)G; }

// ietf::Verifier::verify over all devices: item range [n g / G, n (g+1) / G) on device g, everything enqueued on every device
// before anything is waited for, results written straight into the caller's arrays.  No collective.
extern "C" vrfs_status vrfs_multi_ietf_verify_batch(vrfs_mctx* m, vrfs_suite suite, size_t n, const uint8_t* pk, const uint8_t* input, const uint8_t* output,
                                                    const uint8_t* c, const uint8_t* s, const uint8_t* ad, const uint64_t* ad_off, uint8_t* out_ok, uint8_t* out_status) {
  if (!m || m->n < 1) return VRFS_BAD_ARG;
  std::lock_guard<std::mutex> lock_(m->mu);
  if (n == 0) return VRFS_OK;
  if (!pk || !input || !output || !c || !s || !out_ok) return mfail(m, VRFS_BAD_ARG, "null buffer");
  std::vector<std::unique_ptr<CallGuard>> guards;
  for (int g = 0; g < m->n; g++) guards.emplace_back(new CallGuard(m->dev[g]));
  for (int g = 0; g < m->n; g++) {
    const size_t lo = mshard(n, g, m->n), cnt = mshard(n, g + 1, m->n) - lo;
    if (!cnt) continue;
    MST(m, g, ietf_verify_host_enqueue(m->dev[g], suite, cnt, pk + lo * 64, input + lo * 64, output + lo * 64, c + lo * 32, s + lo * 32, ad,
                                       ad_off ? ad_off + lo : nullptr, out_ok + lo, out_status ? out_status + lo : nullptr));
  }
  for (int g = 0; g < m->n; g++) {
    vrfs_ctx* ctx = m->dev[g];
    cudaSetDevice(ctx->device);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { fail(ctx, VRFS_CUDA_ERROR, "cudaStreamSynchronize: %s", cudaGetErrorString(e)); return mfail(m, VRFS_CUDA_ERROR, "device %d (cuda:%d): %s", g, ctx->device, ctx->err); }
  }
  return VRFS_OK;
}

// RingContext's SRS over all devices: device g prepares the bases [n g / G, n (g+1) / G)
extern "C" void vrfs_multi_msm_g1_release(vrfs_multi_bases* h) {
  if (!h) return;
  for (int g = 0; g < VRFS_MAX_PEERS; g++) if (h->part[g]) vrfs_msm_g1_release(h->part[g]);
  delete h;
}
extern "C" vrfs_status vrfs_multi_msm_g1_prepare(vrfs_mctx* m, size_t n, const uint8_t* bases, vrfs_multi_bases** out) {
  if (!m || !out) return VRFS_BAD_ARG;
  std::lock_guard<std::mutex> lock_(m->mu);
  *out = nullptr;
  if (!bases || n < (size_t)m->n) return mfail(m, VRFS_BAD_ARG, "need at least one base per device");
  vrfs_multi_bases* h = new (std::nothrow) vrfs_multi_bases();
  if (!h) return mfail(m, VRFS_CUDA_ERROR, "out of host memory");
  h->m = m; h->n = n;
  for (int g = 0; g < VRFS_MAX_PEERS; g++) h->part[g] = nullptr;
  for (int g = 0; g <= m->n; g++) h->lo[g] = mshard(n, g, m->n);
  for (int g = 0; g < m->n; g++) {
    vrfs_status st = vrfs_msm_g1_prepare(m->dev[g], h->lo[g + 1] - h->lo[g], bases + h->lo[g] * 96, &h->part[g]);
    if (st != VRFS_OK) { mfail(m, st, "device %d (cuda:%d): %s", g, m->dev[g]->device, m->dev[g]->err); vrfs_multi_msm_g1_release(h); return st; }
  }
  *out = h;
  return VRFS_OK;
}
// wait for every device; the folding rank (device 0) reports a timed-out exchange
static vrfs_status multi_finish(vrfs_mctx* m) {
  vrfs_status ret = VRFS_OK;
  for (int g = 0; g < m->n; g++) {
    vrfs_ctx* ctx = m->dev[g];
    cudaSetDevice(ctx->device);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess && ret == VRFS_OK) { fail(ctx, VRFS_CUDA_ERROR, "cudaStreamSynchronize: %s", cudaGetErrorString(e)); ret = mfail(m, VRFS_CUDA_ERROR, "device %d (cuda:%d): %s", g, ctx->device, ctx->err); }
  }
  if (ret == VRFS_OK && peer_check(m->dev[0]) != VRFS_OK) ret = mfail(m, VRFS_CUDA_ERROR, "%s", m->dev[0]->err);
  return ret;
}
// n_columns commitments over the sharded SRS: device g reduces its point range, the partials meet in device 0's mailbox
extern "C" vrfs_status vrfs_multi_msm_g1_prepared(vrfs_mctx* m, const vrfs_multi_bases* h, const uint8_t* scalars, int n_columns, uint8_t* out) {
  if (!m || !h || h->m != m) return VRFS_BAD_ARG;
  std::lock_guard<std::mutex> lock_(m->mu);
  if (n_columns < 1 || n_columns > VRFS_PEER_MAXCOL || !scalars || !out) return mfail(m, VRFS_BAD_ARG, "bad argument");
  std::vector<std::unique_ptr<CallGuard>> guards;
  for (int g = 0; g < m->n; g++) guards.emplace_back(new CallGuard(m->dev[g]));
  // The folding device (0) is enqueued LAST: its final kernel spins until the other devices' partials arrive, and with peer access
  // enabled a cudaMalloc on ANY device has to update the page tables of its peers - it would block behind that spinning kernel
  // until the exchange timed out.  Enqueued last, device 0 only ever waits for work that is already in flight.
  for (int g = m->n - 1; g >= 0; g--) {
    vrfs_ctx* ctx = m->dev[g];
    const size_t lo = h->lo[g], cnt = h->lo[g + 1] - lo;
    PeerArgs pa;
    MST(m, g, peer_begin(ctx, 0, &pa));
    MST(m, g, begin_call(ctx, cnt));
    void* d_s = nullptr; uint8_t* d_o = nullptr;
    MST(m, g, ensure(ctx, BUF_IN1, cnt * 32 * (size_t)n_columns, &d_s));
    for (int col = 0; col < n_columns; col++) {          // column-major on the host: one strided piece per column
      cudaError_t e = cudaMemcpyAsync((uint8_t*)d_s + (size_t)col * cnt * 32, scalars + ((size_t)col * h->n + lo) * 32, cnt * 32, cudaMemcpyHostToDevice, ctx->stream);
      if (e != cudaSuccess) return mfail(m, VRFS_CUDA_ERROR, "device %d: cudaMemcpyAsync: %s", g, cudaGetErrorString(e));
    }
    MST(m, g, stage_out(ctx, BUF_OUT0, (size_t)96 * n_columns, &d_o));
    MST(m, g, msm_prepared_dev(ctx, h->part[g], n_columns, 0, (const uint8_t*)d_s, d_o, 2, &pa));
    if (g == 0) MST(m, g, copy_out(ctx, out, d_o, (size_t)96 * n_columns));
  }
  return multi_finish(m);
}
// the verifier key's commitment (cx, cy, selector) of a ring over a Lagrange-basis SRS sharded by rows (vrfs_ring_commit on G GPUs)
extern "C" vrfs_status vrfs_multi_ring_commit(vrfs_mctx* m, const vrfs_multi_bases* srs_lagrange, size_t keyset_part_size, size_t n_keys, const uint8_t* keys,
                                              const uint8_t* padding, size_t n_tail, const uint8_t* tail, uint8_t* out_commitment) {
  if (!m || !srs_lagrange || srs_lagrange->m != m) return VRFS_BAD_ARG;
  std::lock_guard<std::mutex> lock_(m->mu);
  const vrfs_multi_bases* h = srs_lagrange;
  if (!out_commitment) return mfail(m, VRFS_BAD_ARG, "null buffer");
  if (h->n & (h->n - 1)) return mfail(m, VRFS_BAD_ARG, "the SRS must span a power-of-two domain");
  if (n_keys > keyset_part_size || keyset_part_size + n_tail > h->n) return mfail(m, VRFS_BAD_ARG, "need n_keys <= keyset_part_size and keyset_part_size + n_tail <= domain size");
  std::vector<std::unique_ptr<CallGuard>> guards;
  for (int g = 0; g < m->n; g++) guards.emplace_back(new CallGuard(m->dev[g]));
  for (int g = m->n - 1; g >= 0; g--) {                  // the folding device last (see vrfs_multi_msm_g1_prepared)
    vrfs_ctx* ctx = m->dev[g];
    const size_t lo = h->lo[g], cnt = h->lo[g + 1] - lo;
    PeerArgs pa;
    MST(m, g, peer_begin(ctx, 0, &pa));
    MST(m, g, begin_call(ctx, cnt));
    uint8_t *d_cols = nullptr, *d_o = nullptr;
    MST(m, g, ring_columns_dev(ctx, cnt, keyset_part_size, n_keys, (keys && n_keys > lo) ? keys + lo * 64 : nullptr, padding, n_tail, tail, &d_cols, lo, false));
    MST(m, g, stage_out(ctx, BUF_OUT0, 3 * 96, &d_o));
    MST(m, g, msm_prepared_dev(ctx, h->part[g], 3, 1, d_cols, d_o, 2, &pa));
    if (g == 0) MST(m, g, copy_out(ctx, out_commitment, d_o, 3 * 96));
  }
  return multi_finish(m);
}
