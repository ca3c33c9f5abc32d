// worker_main.cc -- `tensor-fusion-worker`: the process the operator starts in the worker
// container (reference: internal/utils/compose.go:1304-1325)
//     ./tensor-fusion-worker -p 8000                        TCP transport, port "remote-vgpu"
//     ./tensor-fusion-worker -n shmem -m tf_shm -M 1024     shared-memory transport (local sidecar)
// Each accepted connection is one vGPU session: bytes read from the socket land in a pinned
// ring and go to the GPU through the C-ABI of libtfw_b200.so (include/tfw_worker.h); response
// frames go back on the same socket.  Environment contract: SURVEY.md App. D
// (TF_SHM_PATH, TF_CUDA_MEMORY_LIMIT [MiB], DISABLE_GPU_LIMITER, HYPERVISOR_IP/PORT, POD_NAME, ...).
#include <arpa/inet.h>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <netinet/in.h>
#include <netinet/tcp.h>
#include <poll.h>
#include <signal.h>
#include <sys/socket.h>
#include <unistd.h>

#include <atomic>
#include <cerrno>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <string>
#include <thread>
#include <vector>

#include "erl.h"
#include "hv_handshake.h"
#include "tfw_shm_ring.h"
#include "tfw_wire.h"
#include "tfw_worker.h"

namespace {

std::atomic<bool> g_stop{false};
int g_listen_fd = -1;

// SIGTERM (pod deletion) / SIGINT: stop accepting, let every session drain what it has and leave.
// Only async-signal-safe calls here.
void on_stop_signal(int) {
  g_stop.store(true);
  if (g_listen_fd >= 0) shutdown(g_listen_fd, SHUT_RDWR);  // wakes the blocking accept()
}
bool g_log = false;

void logf(const char* fmt, ...) __attribute__((format(printf, 1, 2)));
void logf(const char* fmt, ...) {
  if (!g_log) return;
  va_list ap;
  va_start(ap, fmt);
  fprintf(stderr, "[tensor-fusion-worker] ");
  vfprintf(stderr, fmt, ap);
  fputc('\n', stderr);
  va_end(ap);
}

bool send_all(int fd, const uint8_t* p, size_t n) {
  while (n) {
    ssize_t k = send(fd, p, n, MSG_NOSIGNAL);
    if (k < 0) { if (errno == EINTR) continue; return false; }
    p += k;
    n -= (size_t)k;
  }
  return true;
}

// Bootstrap handshake with the hypervisor (hv_handshake.h), best effort.
uint64_t g_vram_limit_from_hypervisor = 0;
uint32_t g_sm_percent_from_hypervisor = 0;  // hard isolation: computeUpLimit(tflops_limit / the GPU's max TFLOPS)
long g_auto_freeze_ttl_ms = 0;  // auto_freeze.freeze_to_mem_ttl of the hypervisor's pod info, or $TF_AUTO_FREEZE_TTL_MS

void hypervisor_handshake() {
  const tfhv::Result r = tfhv::handshake("tensorfusion-worker");  // pkg/constants/env.go:61
  if (!getenv("HYPERVISOR_IP")) return;
  if (!r.reached) { logf("hypervisor not reachable (continuing with env limits)"); return; }
  logf("hypervisor /api/v1/pod -> %.80s", r.pod_reply.c_str());
  g_vram_limit_from_hypervisor = r.vram_limit;
  if (r.auto_freeze_ttl_ms > 0 && !getenv("TF_AUTO_FREEZE_TTL_MS")) g_auto_freeze_ttl_ms = r.auto_freeze_ttl_ms;
  // hard isolation without an explicit SM limit from the operator: the share of the GPU the pod's TFLOPS limit
  // buys (B200 = 2250 dense bf16 TFLOPS, gpu-public-gpu-info.yaml:380-385)
  if (r.hard_isolation && r.tflops_limit > 0) {
    const char* mt = getenv("TF_GPU_MAX_TFLOPS");
    const double max_tflops = mt && atof(mt) > 0 ? atof(mt) : 2250.0;
    g_sm_percent_from_hypervisor = tferl::up_limit_percent(0, r.tflops_limit, max_tflops);
  }
  logf("pod info: vram_limit=%llu tflops_limit=%g isolation=%s auto_freeze_ttl_ms=%ld sm_percent=%u", (unsigned long long)r.vram_limit, r.tflops_limit,
       r.hard_isolation ? "hard" : "soft", r.auto_freeze_ttl_ms, g_sm_percent_from_hypervisor);
  logf("hypervisor /api/v1/process -> %.80s", r.process_reply.c_str());
}

// One vGPU session with the limits the operator put into the environment (SURVEY App. D).
tfw_worker* make_worker(int device) {
  tfw_config cfg{};
  cfg.struct_size = sizeof cfg;
  cfg.device = device;
  const char* shm = getenv("TF_SHM_PATH");
  const char* nolim = getenv("DISABLE_GPU_LIMITER");
  if (shm && *shm && !(nolim && *nolim) && access(shm, R_OK | W_OK) == 0) cfg.shm_path = shm;
  if (const char* m = getenv("TF_CUDA_MEMORY_LIMIT")) cfg.vram_limit_bytes = strtoull(m, nullptr, 10) << 20;  // MiB (compose.go:1287-1295)
  else if (g_vram_limit_from_hypervisor) cfg.vram_limit_bytes = g_vram_limit_from_hypervisor;                   // RemotePodInfo.vram_limit, bytes
  if (const char* sm = getenv("TF_CUDA_SM_PERCENT_LIMIT")) {  // hard compute limit (compose.go:1287-1295): an SM partition for this vGPU
    const long v = atol(sm);
    if (v > 0 && v < 100) cfg.sm_percent_limit = (uint32_t)v;
  } else if (g_sm_percent_from_hypervisor && g_sm_percent_from_hypervisor < 100) cfg.sm_percent_limit = g_sm_percent_from_hypervisor;
  tfw_worker* w = nullptr;
  const tfw_status rc = tfw_worker_create(&cfg, &w);
  if (rc != TFW_OK) {
    fprintf(stderr, "[tensor-fusion-worker] tfw_worker_create failed: %d%s\n", rc, rc == TFW_ERR_NO_DEVICE ? " (no CUDA device; there is no CPU fallback)" : "");
    return nullptr;
  }
  return w;
}

// What every session does, whatever the transport: the vGPU's control words and idle policy, submitting around a full
// response arena or ring, the window of spans whose DMA may still read client bytes, and the close-out.  The transports
// keep how bytes arrive, how responses leave and how the client's end is seen.
struct Session {
  struct Span { uint64_t ticket, upto; };
  tfw_worker* w;
  uint64_t* released = nullptr;  // where the end of a span is published once its DMA has completed (the rings' c2w_tail)
  std::deque<Span> inflight;     // oldest first
  timespec active{};             // the client's last activity, where the freeze-to-memory TTL starts
  uint64_t bytes_in = 0;

  Session(tfw_worker* worker, uint64_t* released_to = nullptr) : w(worker), released(released_to) { touch(); }
  void touch() { clock_gettime(CLOCK_MONOTONIC, &active); }
  // The provider's control words (AccelSnapshot / AccelResume / hard limits, DESIGN §7c): 0 running, 1 frozen by the
  // provider (nothing is read, so the client is back-pressured; responses keep leaving), 2 frozen by the idle policy.
  int control() { int frozen = 0; tfw_worker_poll_control(w, &frozen); return frozen; }
  // The client has sent bytes: a vGPU the idle policy froze comes back before any of them executes.  False while the HBM
  // is not available yet.
  bool thaw(int frozen) {
    if (frozen == 2 && tfw_worker_auto_resume(w) != TFW_OK) { usleep(2000); return false; }
    touch();
    return true;
  }
  // The client is quiet and the vGPU runs: once the TTL has passed it gives its HBM back (true), and the TTL starts over.
  bool freeze_if_idle() {
    if (g_auto_freeze_ttl_ms <= 0) return false;
    timespec now;
    clock_gettime(CLOCK_MONOTONIC, &now);
    if ((now.tv_sec - active.tv_sec) * 1000 + (now.tv_nsec - active.tv_nsec) / 1000000 < g_auto_freeze_ttl_ms) return false;
    uint64_t moved = 0;
    if (tfw_worker_auto_freeze(w, &moved) == TFW_OK) logf("idle for %ld ms: vGPU frozen to memory (%llu bytes)", g_auto_freeze_ttl_ms, (unsigned long long)moved);
    touch();
    return true;
  }
  // tfw_submit until the parser has taken what it can.  TFW_ERR_EXHAUSTED (the response arena or ring is full) calls
  // make_room(), then the frame is resumed where the parser stopped; make_room() false ends the attempt.
  template <class MakeRoom>
  tfw_status submit(const uint8_t* p, size_t n, size_t* used, MakeRoom make_room) {
    *used = 0;
    for (;;) {
      size_t u = 0;
      const tfw_status rc = tfw_submit(w, p + *used, n - *used, &u);
      *used += u;
      if (rc != TFW_ERR_EXHAUSTED) return rc;
      if (!make_room()) return TFW_ERR_FAILED;
    }
  }
  // Fence what has been submitted; past `window` spans in flight, wait for the oldest.
  bool fence(size_t window, uint64_t upto = 0) {
    uint64_t ticket = 0;
    if (tfw_fence(w, &ticket) != TFW_OK) return false;
    inflight.push_back({ticket, upto});
    return inflight.size() <= window || retire(true);
  }
  // Release the leading spans whose DMA has completed; `block` waits for the first.
  bool retire(bool block) {
    while (!inflight.empty()) {
      int done = 0;
      if (block) { if (tfw_fence_wait(w, inflight.front().ticket) != TFW_OK) return false; done = 1; }
      else if (tfw_fence_query(w, inflight.front().ticket, &done) != TFW_OK) return false;
      if (!done) break;
      if (released) __atomic_store_n(released, inflight.front().upto, __ATOMIC_RELEASE);
      inflight.pop_front();
      block = false;
    }
    return true;
  }
  // Unless the session failed, everything submitted executes and deliver() hands out what it produced; then the session's
  // log line, and the vGPU goes.
  template <class Deliver>
  void end(bool failed, Deliver deliver) {
    if (!failed) {
      tfw_flush(w);
      retire(true);
      deliver();
    }
    tfw_stats st{};
    tfw_get_stats(w, &st);
    logf("session closed: %llu bytes in, %llu frames, %llu payload bytes, %llu mover launches", (unsigned long long)bytes_in,
         (unsigned long long)st.frames, (unsigned long long)st.payload_bytes, (unsigned long long)st.mover_launches);
    tfw_worker_destroy(w);
  }
};

// A fresh header for rings of `total` bytes, published to clients last (magic, then worker_ready).
void init_ring_header(tfsr_header* hdr, uint64_t total) {
  std::memset(hdr, 0, sizeof *hdr);
  hdr->version = TFSR_VERSION;
  hdr->total_bytes = total;
  tfsr_layout(total, &hdr->c2w_off, &hdr->c2w_size, &hdr->w2c_off, &hdr->w2c_size);
  hdr->worker_pid = (uint32_t)getpid();
  hdr->session = 1;
  __atomic_store_n(&hdr->magic, TFSR_MAGIC, __ATOMIC_RELEASE);
  __atomic_store_n(&hdr->worker_ready, 1u, __ATOMIC_RELEASE);
}

void serve_rings(tfsr_header* hdr, uint8_t* base, uint64_t total_bytes, uint32_t session, int lock_fd, const std::string& ring_path, tfw_worker* w);

bool recv_exact(int fd, void* p, size_t n, int timeout_ms) {
  uint8_t* b = static_cast<uint8_t*>(p);
  while (n) {
    pollfd pf{fd, POLLIN, 0};
    const int pr = poll(&pf, 1, timeout_ms);
    if (pr < 0 && errno == EINTR) continue;
    if (pr <= 0) return false;
    const ssize_t k = recv(fd, b, n, 0);
    if (k < 0 && errno == EINTR) continue;
    if (k <= 0) return false;
    b += k;
    n -= (size_t)k;
  }
  return true;
}

// TFCS_OP_UPGRADE_SHM: a client on this node asks to continue on shared-memory rings it has created.  Returns true if
// the session was served (on the rings); false = stay on the socket (the refusal has been sent).
// `w`: the session's worker, created before the first frame was read; when this returns true the rings' session has used and destroyed it
bool try_upgrade_to_shm(int fd, const tfcs_frame_hdr& h, const std::string& name, tfw_worker* w) {
  auto refuse = [&](uint32_t code) {
    tfcs_frame_hdr r = h;
    r.opcode = TFCS_OP_RESP_ERROR;
    r.arg0 = code;
    r.arg1 = h.opcode;
    r.length = 0;
    send_all(fd, reinterpret_cast<const uint8_t*>(&r), sizeof r);
    return false;
  };
  if (getenv("TFW_NO_SHM_UPGRADE") || name.empty() || name.find('/') != std::string::npos || h.off0 < TFSR_MIN_BYTES || h.off0 > (8ull << 30)) return refuse(TFW_ERR_INVALID);
  const char* dir = getenv("TFW_SHM_DIR");
  const std::string path = std::string(dir && *dir ? dir : "/dev/shm") + "/" + name;
  const int sfd = open(path.c_str(), O_RDWR | O_NOFOLLOW);
  struct stat sb{};
  if (sfd < 0 || fstat(sfd, &sb) != 0 || !S_ISREG(sb.st_mode) || (uint64_t)sb.st_size != h.off0) {  // not our node's /dev/shm: another pod
    if (sfd >= 0) close(sfd);
    return refuse(TFW_ERR_NOT_FOUND);
  }
  const uint64_t total = h.off0;
  void* m = mmap(nullptr, total, PROT_READ | PROT_WRITE, MAP_SHARED, sfd, 0);
  if (m == MAP_FAILED) { close(sfd); return refuse(TFW_ERR_EXHAUSTED); }
  if (tfw_host_register(m, total) != TFW_OK) { munmap(m, total); close(sfd); return refuse(TFW_ERR_EXHAUSTED); }
  tfsr_header* hdr = static_cast<tfsr_header*>(m);
  init_ring_header(hdr, total);
  tfcs_frame_hdr r = h;
  r.opcode = TFCS_OP_RESP_ACK;
  r.length = 0;
  bool ok = send_all(fd, reinterpret_cast<const uint8_t*>(&r), sizeof r);
  for (int i = 0; ok && i < 10000 && __atomic_load_n(&hdr->client_pid, __ATOMIC_ACQUIRE) == 0; ++i) usleep(1000);  // the client attaches
  ok = ok && __atomic_load_n(&hdr->client_pid, __ATOMIC_ACQUIRE) != 0;
  if (ok) {
    logf("connection upgraded to shared-memory rings %s (%llu MiB)", path.c_str(), (unsigned long long)(total >> 20));
    serve_rings(hdr, static_cast<uint8_t*>(m), total, 1, sfd, path, w);
  }  // (else: the client never attached; the caller keeps the worker and finds the socket dead)
  __atomic_store_n(&hdr->worker_ready, 0u, __ATOMIC_RELEASE);
  tfw_host_unregister(m);
  munmap(m, total);
  close(sfd);
  unlink(path.c_str());
  return ok;
}

// One TCP connection: bytes are received into two pinned rings, responses go back on the socket; recv() <= 0 is the
// client's end.
void serve(int fd, int device) {
  int one = 1;
  setsockopt(fd, IPPROTO_TCP, TCP_NODELAY, &one, sizeof one);
  // bulk payloads: deep socket buffers (FORCE needs CAP_NET_ADMIN; the plain option is capped by net.core.*mem_max)
  int big = 32 << 20;
  if (setsockopt(fd, SOL_SOCKET, SO_RCVBUFFORCE, &big, sizeof big) != 0) setsockopt(fd, SOL_SOCKET, SO_RCVBUF, &big, sizeof big);
  if (setsockopt(fd, SOL_SOCKET, SO_SNDBUFFORCE, &big, sizeof big) != 0) setsockopt(fd, SOL_SOCKET, SO_SNDBUF, &big, sizeof big);
  // The vGPU first: a worker without a GPU closes the connection at once, whatever the client meant to say.
  tfw_worker* w = make_worker(device);
  if (!w) {
    close(fd);
    return;
  }
  // A client on this node may propose shared-memory rings with its very first frame (TFCS_OP_UPGRADE_SHM).
  {
    uint8_t peek[TFCS_HDR_BYTES];
    ssize_t k;
    do { k = recv(fd, peek, sizeof peek, MSG_PEEK | MSG_WAITALL); } while (k < 0 && errno == EINTR);
    tfcs_frame_hdr first{};
    if (k == (ssize_t)sizeof peek) {
      std::memcpy(&first, peek, sizeof first);
      if (first.magic == TFCS_MAGIC && first.opcode == TFCS_OP_UPGRADE_SHM && first.length <= 255) {
        char name[272] = {0};
        uint8_t skip[TFCS_HDR_BYTES];
        if (!recv_exact(fd, skip, sizeof skip, 5000) || !recv_exact(fd, name, (size_t)tfcs_pad16(first.length), 5000)) { tfw_worker_destroy(w); close(fd); return; }
        name[first.length] = 0;
        if (try_upgrade_to_shm(fd, first, name, w)) { close(fd); return; }  // (the rings' session took the worker)
      }
    }
  }
  // Two pinned rings: while the GPU still reads ring A (in-place DMA), the socket fills ring B.
  const size_t ring = 64u << 20;
  uint8_t* bufs[2] = {nullptr, nullptr};
  std::vector<uint8_t> out(16u << 20);
  if (tfw_host_alloc(ring, reinterpret_cast<void**>(&bufs[0])) != TFW_OK || tfw_host_alloc(ring, reinterpret_cast<void**>(&bufs[1])) != TFW_OK) {
    if (bufs[0]) tfw_host_free(bufs[0]);
    tfw_worker_destroy(w);
    close(fd);
    return;
  }
  Session s(w);
  int cur = 0;
  size_t fill = 0;
  auto drain = [&](bool block) {
    for (;;) {
      size_t m = 0;
      if (tfw_poll_responses(w, out.data(), out.size(), &m) != TFW_OK) return false;
      if (m && !send_all(fd, out.data(), m)) return false;
      if (!m || !block) return true;
    }
  };
  for (;;) {
    if (g_stop.load()) break;  // SIGTERM: finish what was submitted (the close-out below) and close
    const int frozen = s.control();
    if (frozen == 1) { if (!drain(false)) break; usleep(2000); continue; }  // the client is back-pressured by TCP
    // Responses (D2H payloads, SYNC acks) become ready asynchronously: while the client is quiet,
    // keep delivering them instead of blocking in recv().
    pollfd pf{fd, POLLIN, 0};
    const int pr = poll(&pf, 1, 2);
    if (pr == 0) {
      if (!drain(false)) break;
      if (!frozen) s.freeze_if_idle();
      continue;
    }
    if (pr < 0 && errno == EINTR) continue;
    if (!s.thaw(frozen)) continue;
    uint8_t* buf = bufs[cur];
    ssize_t n = recv(fd, buf + fill, ring - fill, 0);
    if (n < 0 && errno == EINTR) continue;
    if (n <= 0) break;
    // a bulk sender keeps the socket full: take what is already there (up to 16 MiB) before handing the span to the
    // GPU, so that one submit = one multi-MiB DMA instead of one per ~64 KiB read
    while ((size_t)n < (16u << 20) && fill + (size_t)n < ring) {
      const ssize_t k = recv(fd, buf + fill + n, ring - fill - (size_t)n, MSG_DONTWAIT);
      if (k <= 0) break;
      n += k;
    }
    s.bytes_in += (uint64_t)n;
    const size_t have = fill + (size_t)n;
    size_t used = 0;
    // response arena full: ship responses, then resume where the parser stopped
    const tfw_status rc = s.submit(buf, have, &used, [&] { tfw_flush(w); return drain(true); });
    if (rc != TFW_OK) { logf("submit failed: %d (%s)", rc, tfw_last_error(w)); break; }
    if (!s.fence(1)) break;  // one span in flight: the other ring, refilled next, has been read by the GPU
    cur ^= 1;
    fill = have - used;  // < 64 bytes: a partial header, moved to the front of the other ring
    std::memcpy(bufs[cur], buf + used, fill);
    if (!drain(false)) break;
  }
  s.end(false, [&] { drain(true); });
  tfw_host_free(bufs[0]);
  tfw_host_free(bufs[1]);
  close(fd);
}

// ---- shared-memory transport (include/tfw_shm_ring.h) -----------------------------------------------------
// How the worker waits for the client on the rings: spin, then 20 us naps, then 200 us naps once the client has been
// quiet for ~10 ms.
struct Backoff {
  int n = 0;
  void reset() { n = 0; }
  void pause() {
    ++n;
    if (n < 2000) { __builtin_ia32_pause(); return; }
    timespec ts{0, n < 2500 ? 20000 : 200000};
    nanosleep(&ts, nullptr);
  }
  bool probe_due() const { return n >= 5000 && n % 5000 == 0; }  // 5000 naps of 200 us = 1 s: time to probe the client's liveness
};

// One client session on the rings; `w` (may be null: worker_closed at once) is the session's vGPU and is destroyed here.
// Bytes are read in place from the client -> worker ring; responses are produced into the worker -> client ring by the
// library (the response sink); the client ends the session with client_closed, or is found gone through its liveness lock.
void serve_rings(tfsr_header* hdr, uint8_t* base, uint64_t total_bytes, uint32_t session, int lock_fd, const std::string& ring_path, tfw_worker* w) {
  if (!w) {
    __atomic_store_n(&hdr->worker_closed, session, __ATOMIC_RELEASE);
    return;
  }
  tfw_set_arena_prefix(w, ring_path.c_str());  // the client's page-locked memory: files <ring>.a<k> (TFCS_OP_HOST_REGISTER)
  // the layout comes from our own arithmetic, not from the header: the client can write to that page
  uint64_t c2w_off = 0, up = 0, w2c_off = 0, down = 0;
  tfsr_layout(total_bytes, &c2w_off, &up, &w2c_off, &down);
  uint8_t* c2w = base + c2w_off;
  // Responses are produced in the worker -> client ring itself: D2H payloads are written there by the copy
  // engine (the mapping is page-locked), the head cursor moves when the GPU is done with a piece.
  const tfw_response_sink sink{sizeof(tfw_response_sink), 0, base + w2c_off, down, &hdr->w2c_head, &hdr->w2c_tail};
  if (tfw_set_response_sink(w, &sink) != TFW_OK) {
    fprintf(stderr, "[tensor-fusion-worker] session %u: no response sink on the rings: %s\n", session, tfw_last_error(w));
    tfw_worker_destroy(w);
    __atomic_store_n(&hdr->worker_closed, session, __ATOMIC_RELEASE);
    return;
  }
  Session s(w, &hdr->c2w_tail);
  uint64_t rd = hdr->c2w_tail;  // read cursor; the shared tail trails it until the DMA of a span is done
  uint64_t wr = hdr->w2c_head;
  bool ring_full = false;
  auto closed = [&] { return __atomic_load_n(&hdr->client_closed, __ATOMIC_ACQUIRE) >= session; };
  // a client that died without saying so (include/tfw_shm_ring.h: liveness lock); probed once a second while silent
  auto client_gone = [&]() {
#ifdef TFSR_HAVE_LIVENESS
    return lock_fd >= 0 && __atomic_load_n(&hdr->client_lock_session, __ATOMIC_ACQUIRE) == session && !tfsr_client_alive(lock_fd);
#else
    (void)lock_fd;
    return false;
#endif
  };
  // publish the responses whose GPU work has completed; returns bytes published, -1 on error
  auto publish = [&]() -> long {
    size_t m = 0;
    if (tfw_poll_responses(w, nullptr, 0, &m) != TFW_OK) return -1;
    const uint64_t head = __atomic_load_n(&hdr->w2c_head, __ATOMIC_RELAXED);
    const long moved = (long)(head - wr);
    wr = head;
    ring_full = down - (head - __atomic_load_n(&hdr->w2c_tail, __ATOMIC_ACQUIRE)) < (1u << 20);
    return moved;
  };
  // the ring is full: publish what completes and wait for the client to consume, then the frame resumes
  auto make_room = [&]() {
    Backoff wait;
    const uint64_t tail0 = __atomic_load_n(&hdr->w2c_tail, __ATOMIC_ACQUIRE);
    while (__atomic_load_n(&hdr->w2c_tail, __ATOMIC_ACQUIRE) == tail0) {
      if (publish() < 0) return false;
      if (closed() || g_stop.load()) return false;  // nobody reads any more
      if (wait.probe_due() && client_gone()) return false;
      wait.pause();
    }
    return true;
  };
  alignas(16) uint8_t joined[TFCS_HDR_BYTES];
  Backoff idle;
  bool failed = false;

  for (;;) {
    if (g_stop.load()) break;  // SIGTERM: drain below, then worker_closed tells the client
    const int frozen = s.control();
    if (frozen == 1) { publish(); usleep(2000); continue; }
    if (frozen == 2) {
      if (__atomic_load_n(&hdr->c2w_head, __ATOMIC_ACQUIRE) == rd) {
        if (closed()) break;
        usleep(1000);
        continue;
      }
      if (!s.thaw(frozen)) continue;
    }
    bool progress = false;
    if (!s.inflight.empty()) {
      const size_t before = s.inflight.size();
      if (!s.retire(false)) { failed = true; break; }
      progress |= s.inflight.size() != before;
    }
    const uint64_t avail = __atomic_load_n(&hdr->c2w_head, __ATOMIC_ACQUIRE) - rd;
    if (avail) {
      const uint64_t pos = rd % up;
      const uint64_t span = std::min<uint64_t>(std::min<uint64_t>(avail, up - pos), 64u << 20);
      size_t used = 0;
      tfw_status rc = s.submit(c2w + pos, (size_t)span, &used, make_room);
      if (rc != TFW_OK) { logf("submit failed: %d (%s)", rc, tfw_last_error(w)); failed = true; break; }
      const uint64_t rest = span - used;  // < 64 bytes: the front of a header whose tail is not here yet ...
      if (rest && pos + span == up && avail - used >= TFCS_HDR_BYTES) {  // ... or wraps to the start of the ring
        std::memcpy(joined, c2w + pos + used, rest);
        std::memcpy(joined + rest, c2w, TFCS_HDR_BYTES - rest);
        size_t u2 = 0;
        rc = s.submit(joined, TFCS_HDR_BYTES, &u2, make_room);
        if (rc != TFW_OK || u2 != TFCS_HDR_BYTES) { logf("submit (wrapped header) failed: %d (%s)", rc, tfw_last_error(w)); failed = true; break; }
        used += TFCS_HDR_BYTES;
      }
      rd += used;
      s.bytes_in += used;
      if (used) {
        progress = true;
        if (!s.fence(6, rd)) { failed = true; break; }  // the fence ring holds 8
      }
    }
    const long moved = publish();
    if (moved < 0) { failed = true; break; }
    progress |= moved > 0;
    if (!avail && closed() && __atomic_load_n(&hdr->c2w_head, __ATOMIC_ACQUIRE) == rd) break;  // the client is done and everything it wrote has been consumed
    if (progress) { idle.reset(); s.touch(); }
    else {
      if (s.inflight.empty() && s.freeze_if_idle()) continue;
      idle.pause();
      if (idle.probe_due() && client_gone()) {
        logf("client of session %u is gone without closing: ending the session", session);
        break;
      }
    }
  }
  s.end(failed, [&] {
    // everything is ready after the flush; deliver it.  tfc_close keeps reading until worker_closed, a client
    // that died does not: give up after 2 s without progress.
    Backoff wait;
    timespec last;
    clock_gettime(CLOCK_MONOTONIC, &last);
    for (;;) {
      const long m = publish();
      if (m < 0 || !ring_full) break;
      timespec now;
      clock_gettime(CLOCK_MONOTONIC, &now);
      if (m > 0) { last = now; wait.reset(); }
      else if (now.tv_sec - last.tv_sec >= 2) break;
      wait.pause();
    }
  });
  __atomic_store_n(&hdr->c2w_tail, rd, __ATOMIC_RELEASE);
  __atomic_store_n(&hdr->worker_closed, session, __ATOMIC_RELEASE);
}

int run_shm(const std::string& name, long mb, int device) {
  if (name.empty() || name.find('/') != std::string::npos || mb < 2) {
    fprintf(stderr, "[tensor-fusion-worker] shmem transport needs -m <name without '/'> -M <MiB >= 2>\n");
    return 2;
  }
  const char* dir = getenv("TFW_SHM_DIR");
  const std::string path = std::string(dir && *dir ? dir : "/dev/shm") + "/" + name;  // pkg/constants/constants.go:291
  const uint64_t total = (uint64_t)mb << 20;
  int fd = open(path.c_str(), O_RDWR | O_CREAT, 0666);
  if (fd < 0 || ftruncate(fd, (off_t)total) != 0) { perror("tensor-fusion-worker: shm file"); return 2; }
  fchmod(fd, 0666);  // the client container runs as another user (compose.go:1316 chmods it too)
  void* m = mmap(nullptr, total, PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0);
  if (m == MAP_FAILED) { perror("tensor-fusion-worker: mmap"); close(fd); return 2; }  // fd stays open: liveness probes go through it
  tfsr_header* hdr = static_cast<tfsr_header*>(m);
  __atomic_store_n(&hdr->worker_ready, 0u, __ATOMIC_RELEASE);  // a stale header of a previous worker must not attract clients
  __atomic_store_n(&hdr->magic, 0u, __ATOMIC_RELEASE);
  // page-lock the rings: the copy engine reads H2D payloads in place
  const tfw_status reg = tfw_host_register(m, total);
  if (reg != TFW_OK) {
    fprintf(stderr, "[tensor-fusion-worker] cannot page-lock the shared rings: %d%s\n", reg,
            reg == TFW_ERR_NO_DEVICE ? " (no CUDA device; there is no CPU fallback)" : " (the file must live on a tmpfs such as /dev/shm)");
    munmap(m, total);
    close(fd);
    return 4;
  }
  init_ring_header(hdr, total);
  printf("tensor-fusion-worker serving shmem %s (%ld MiB)\n", path.c_str(), mb);
  fflush(stdout);
  const char* once = getenv("TFW_ONESHOT");
  int budget = once ? atoi(once) : -1;
  while (budget != 0 && !g_stop.load()) {
    if (__atomic_load_n(&hdr->client_pid, __ATOMIC_ACQUIRE) == 0) { usleep(500); continue; }
    const uint32_t session = hdr->session;
    logf("client %u attached (session %u)", hdr->client_pid, session);
    serve_rings(hdr, static_cast<uint8_t*>(m), total, session, fd, path, make_worker(device));
    // next client: cursors keep counting (they are monotonic); whatever the last client left unread or
    // unsent is discarded while nobody is attached
    hdr->c2w_tail = __atomic_load_n(&hdr->c2w_head, __ATOMIC_ACQUIRE);
    hdr->w2c_tail = hdr->w2c_head;
    hdr->session = session + 1;
    __atomic_store_n(&hdr->client_pid, 0u, __ATOMIC_RELEASE);
    if (budget > 0) --budget;
  }
  __atomic_store_n(&hdr->worker_ready, 0u, __ATOMIC_RELEASE);
  tfw_host_unregister(m);
  munmap(m, total);
  close(fd);
  return 0;
}

}  // namespace

int main(int argc, char** argv) {
  int port = 8000;  // pkg/constants/env.go:155-156
  std::string transport = "native", shm_name;
  long shm_mb = 0;
  for (int i = 1; i < argc; ++i) {
    if (!strcmp(argv[i], "-p") && i + 1 < argc) port = atoi(argv[++i]);
    else if (!strcmp(argv[i], "-n") && i + 1 < argc) transport = argv[++i];
    else if (!strcmp(argv[i], "-m") && i + 1 < argc) shm_name = argv[++i];
    else if (!strcmp(argv[i], "-M") && i + 1 < argc) shm_mb = atol(argv[++i]);
    else if (!strcmp(argv[i], "-h") || !strcmp(argv[i], "--help")) {
      printf("usage: tensor-fusion-worker -p <port> | -n shmem -m <name> -M <MiB>\n");
      return 0;
    }
  }
  g_log = getenv("TF_ENABLE_LOG") != nullptr;
  if (const char* e = getenv("TF_AUTO_FREEZE_TTL_MS")) g_auto_freeze_ttl_ms = atol(e);
  struct sigaction sa{};
  sa.sa_handler = on_stop_signal;
  sigaction(SIGTERM, &sa, nullptr);
  sigaction(SIGINT, &sa, nullptr);
  if (transport == "shmem") {
    hypervisor_handshake();
    return run_shm(shm_name, shm_mb, 0);
  }
  signal(SIGPIPE, SIG_IGN);
  hypervisor_handshake();
  int ls = socket(AF_INET, SOCK_STREAM, 0);
  g_listen_fd = ls;
  int one = 1;
  setsockopt(ls, SOL_SOCKET, SO_REUSEADDR, &one, sizeof one);
  sockaddr_in a{};
  a.sin_family = AF_INET;
  a.sin_port = htons((uint16_t)port);
  const char* bind_ip = getenv("TFW_BIND");
  a.sin_addr.s_addr = bind_ip ? inet_addr(bind_ip) : htonl(INADDR_ANY);
  if (bind(ls, (sockaddr*)&a, sizeof a) != 0 || listen(ls, 16) != 0) { perror("tensor-fusion-worker: bind/listen"); return 2; }
  socklen_t al = sizeof a;
  getsockname(ls, (sockaddr*)&a, &al);
  printf("tensor-fusion-worker listening on port %d\n", ntohs(a.sin_port));
  fflush(stdout);
  const char* once = getenv("TFW_ONESHOT");  // serve N connections, then exit (tests)
  int budget = once ? atoi(once) : -1;
  std::vector<std::thread> sessions;
  while (budget != 0) {
    int fd = accept(ls, nullptr, nullptr);
    if (fd < 0) { if (errno == EINTR && !g_stop.load()) continue; break; }
    sessions.emplace_back(serve, fd, 0);
    if (budget > 0) --budget;
  }
  for (auto& t : sessions) t.join();
  close(ls);
  return 0;
}
