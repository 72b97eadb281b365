// zkb_session (include/zkb200.h): the continuation segments of one session, proven on every device the session owns.  Built on the
// public C-ABI only (zkb_init, zkb_program_*, zkb_prover_*, zkb_prove_staged); the hot path is the prover's own CUDA proof, and what
// this file adds is the host side that keeps the GPUs fed: one queue, `inflight` worker threads per device, one program per device.
//
// Each worker owns a ctx and a staged prover, both created, driven and freed on its own thread.  A worker holds at most two segments on
// its prover's staging slots: the one it proves and one prefetched, whose upload runs on the device's shared FIFO copy stream while the
// first is proven.  Two ordering rules keep that pipeline full (DESIGN.md section 6):
//   (i)  uploads enter a device's copy stream in the order their segments left the queue: every segment draws a per-device turn when
//        it is dequeued and is staged in that turn, so a later segment's 1 GB upload never sits in front of an earlier one;
//   (ii) a worker does not prefetch a second segment while the queue is non-empty and another worker of its device has nothing staged:
//        that worker's first segment goes first.  Without it, pipeline fill was 169 ms per rank instead of about 60.
#include "common.cuh"
#include "circuit.hpp"
#include <array>
#include <condition_variable>
#include <deque>
#include <memory>
#include <mutex>
#include <thread>

namespace {

using zkb::Error;
using zkb::GROUP_ACCUM;
using zkb::GROUP_DATA;

// the message of a C-ABI call's error (empty on success), freed
std::string take(zkb_err e) {
  if (!e) return std::string();
  std::string m(e);
  zkb_free_error(e);
  return m;
}
void must(zkb_err e) {
  if (e) throw Error(take(e));
}

const char* const FREED = "zkb200: session freed before this segment's proof started";

struct Segment {
  uint64_t ticket = 0;
  int po2 = 0;
  std::vector<uint32_t> io;
  const void* data = nullptr;
  const void* accum = nullptr;
};
struct Result {
  bool done = false;
  std::string err;
  std::vector<uint32_t> seal;
};

struct Device;
struct Worker {
  Device* dev = nullptr;
  zkb_ctx* ctx = nullptr;
  zkb_prover* prover = nullptr;     // NULL after a failed renewal: the next segment tries again
  std::deque<Segment> staged;       // on the prover's staging slots, oldest first: the one being proven, then at most one prefetched
  std::string init_err;
  bool ready = false;
  std::thread th;
};
struct Device {
  int id = 0;
  zkb_program* prog = nullptr;
  std::vector<std::unique_ptr<Worker>> workers;
  int idle = 0;                     // workers with nothing staged, waiting for a segment (rule ii); guarded by the session's mu
  uint64_t turns_drawn = 0;         // rule (i); guarded by the session's mu
  std::mutex stage_mu;
  std::condition_variable stage_cv;
  uint64_t turn = 0;                // the turn being staged; guarded by stage_mu
};

}  // namespace

struct zkb_session {
  std::vector<uint32_t> blob;
  zkb::CircuitDef circuit;
  std::vector<std::unique_ptr<Device>> devs;
  std::mutex commit_mu;             // one zkb_session_commit at a time: every device commits the same po2 together
  std::mutex mu;                    // everything below, and Device::idle / turns_drawn
  std::condition_variable cv;       // any change of the state below
  std::deque<Segment> queue;
  std::map<uint64_t, Result> results;
  std::map<int, std::array<uint32_t, 9>> control_ids;     // committed po2 -> (po2, code root[8])
  uint64_t next_ticket = 1;
  bool go = false, stopping = false;
  int waiters = 0;                  // threads inside zkb_session_wait: the session is not deleted under them

  ~zkb_session() { shutdown(); }

  void finish(uint64_t ticket, std::string err, std::vector<uint32_t> seal) {      // under mu
    Result& r = results[ticket];
    r.done = true;
    r.err = std::move(err);
    r.seal = std::move(seal);
  }

  std::string renew(Worker& w) {
    if (w.prover) take(zkb_prover_free(w.prover));
    w.prover = nullptr;
    std::string e = take(zkb_prover_new(w.ctx, blob.data(), blob.size(), &w.prover));
    if (e.empty()) e = take(zkb_prover_set_program(w.prover, w.dev->prog));
    if (!e.empty() && w.prover) { take(zkb_prover_free(w.prover)); w.prover = nullptr; }
    return e;
  }

  // Stages s on w's prover in the device turn drawn now (rule i).  Called and returns with lk held; the stage itself runs without it.
  std::string stage(Worker& w, const Segment& s, std::unique_lock<std::mutex>& lk) {
    Device& d = *w.dev;
    const uint64_t my = d.turns_drawn++;
    lk.unlock();
    std::string e;
    {
      std::unique_lock<std::mutex> sl(d.stage_mu);
      d.stage_cv.wait(sl, [&] { return d.turn == my; });
      if (!w.prover) e = renew(w);
      if (e.empty()) e = take(zkb_prover_stage_traces(w.prover, s.po2, nullptr, s.data, s.accum));
      ++d.turn;
    }
    d.stage_cv.notify_all();
    lk.lock();
    return e;
  }

  // takes the queue's first segment onto w's prover; under mu
  void stage_next(Worker& w, std::unique_lock<std::mutex>& lk) {
    Segment s = std::move(queue.front());
    queue.pop_front();
    std::string e = stage(w, s, lk);
    if (e.empty()) w.staged.push_back(std::move(s));
    else finish(s.ticket, std::move(e), {});
    cv.notify_all();
  }

  void run(Worker& w) {
    Device& d = *w.dev;
    std::string err = take(zkb_init(d.id, &w.ctx));
    if (err.empty()) err = take(zkb_prover_new(w.ctx, blob.data(), blob.size(), &w.prover));
    std::unique_lock<std::mutex> lk(mu);
    w.init_err = err;
    w.ready = true;
    cv.notify_all();
    cv.wait(lk, [&] { return go || stopping; });
    while (!stopping) {
      if (w.staged.empty()) {
        ++d.idle;
        cv.wait(lk, [&] { return stopping || !queue.empty(); });
        --d.idle;
        if (!stopping) stage_next(w, lk);
        continue;
      }
      // rule (ii): the device's workers that have nothing staged take their first segment before this one prefetches a second
      cv.wait(lk, [&] { return stopping || queue.empty() || d.idle == 0; });
      if (stopping) break;
      if (!queue.empty()) stage_next(w, lk);

      const uint64_t ticket = w.staged.front().ticket;
      const uint32_t* io = w.staged.front().io.data();      // deque elements do not move while this thread alone changes w.staged
      lk.unlock();
      std::vector<uint32_t> seal;
      std::string e = take(zkb_prove_staged(w.prover, io));
      if (e.empty()) {
        size_t n = 0;
        e = take(zkb_prover_seal_words(w.prover, &n));
        seal.resize(n);
        if (e.empty()) e = take(zkb_prover_seal_copy(w.prover, seal.data()));
      }
      std::string renew_err;
      if (!e.empty()) renew_err = renew(w);     // a failed proof can leave its staging slot marked full: start over with a new prover
      lk.lock();
      finish(ticket, e, e.empty() ? std::move(seal) : std::vector<uint32_t>());
      w.staged.pop_front();
      if (!e.empty() && !w.staged.empty()) {     // the prefetched segment went with the old prover: stage it again on the new one
        std::string se = renew_err.empty() ? stage(w, w.staged.front(), lk) : renew_err;
        if (!se.empty()) { finish(w.staged.front().ticket, std::move(se), {}); w.staged.pop_front(); }
      }
      cv.notify_all();
    }
    for (const Segment& s : w.staged) finish(s.ticket, FREED, {});
    w.staged.clear();
    cv.notify_all();
    lk.unlock();
    if (w.prover) take(zkb_prover_free(w.prover));
    if (w.ctx) take(zkb_destroy(w.ctx));
    w.prover = nullptr;
    w.ctx = nullptr;
  }

  // Stops the workers (segments whose proof has not started fail), joins them, frees the programs, and returns once no thread is
  // inside zkb_session_wait.
  void shutdown() {
    {
      std::lock_guard<std::mutex> lk(mu);
      stopping = true;
      for (const Segment& s : queue) finish(s.ticket, FREED, {});
      queue.clear();
      cv.notify_all();
    }
    for (auto& d : devs)
      for (auto& w : d->workers)
        if (w->th.joinable()) w->th.join();
    for (auto& d : devs) {
      if (d->prog) take(zkb_program_free(d->prog));
      d->prog = nullptr;
    }
    std::unique_lock<std::mutex> lk(mu);
    cv.wait(lk, [&] { return waiters == 0; });
  }
};

extern "C" {

zkb_err zkb_session_new(const uint32_t* h_circuit, size_t circuit_words, const int* devices, size_t n_devices, int inflight,
                        zkb_session** out) {
  ZKB_API_BEGIN
  ZKB_REQUIRE(out != nullptr, "null out pointer");
  ZKB_REQUIRE(inflight >= 1 && inflight <= 8, "inflight must be in [1, 8], got " + std::to_string(inflight));
  std::unique_ptr<zkb_session> s(new zkb_session());
  s->circuit = zkb::CircuitDef::parse(h_circuit, circuit_words);
  s->blob.assign(h_circuit, h_circuit + circuit_words);
  int visible = 0;
  must(zkb_device_count(&visible));
  std::vector<int> ids;
  if (devices) ids.assign(devices, devices + n_devices);
  else for (int i = 0; i < visible; ++i) ids.push_back(i);
  ZKB_REQUIRE(!ids.empty(), "no device for the session");
  for (size_t i = 0; i < ids.size(); ++i) {
    ZKB_REQUIRE(ids[i] >= 0 && ids[i] < visible, "device " + std::to_string(ids[i]) + " is not visible (" + std::to_string(visible) + " devices)");
    for (size_t j = 0; j < i; ++j) ZKB_REQUIRE(ids[j] != ids[i], "device " + std::to_string(ids[i]) + " is listed twice");
  }
  for (int id : ids) {
    std::unique_ptr<Device> d(new Device());
    d->id = id;
    for (int k = 0; k < inflight; ++k) {
      d->workers.emplace_back(new Worker());
      d->workers.back()->dev = d.get();
    }
    s->devs.push_back(std::move(d));
  }
  zkb_session* sp = s.get();
  for (auto& d : s->devs)
    for (auto& w : d->workers) {
      Worker* wp = w.get();
      wp->th = std::thread([sp, wp] { sp->run(*wp); });     // on an exception here ~zkb_session joins the threads already started
    }
  std::string err;
  {
    std::unique_lock<std::mutex> lk(s->mu);
    for (auto& d : s->devs)
      for (auto& w : d->workers) {
        s->cv.wait(lk, [&] { return w->ready; });
        if (err.empty() && !w->init_err.empty()) err = w->init_err + " (device " + std::to_string(d->id) + ")";
      }
  }
  // The workers wait for `go`, so their ctxs and provers are not in use on their threads here.  The program is made from the device's
  // first worker ctx, which only names the device.  These calls select each device on the caller's thread: its device is restored.
  int caller_device = 0;
  ZKB_CUDA(cudaGetDevice(&caller_device));
  for (auto& d : s->devs) {
    if (err.empty()) err = take(zkb_program_new(d->workers[0]->ctx, s->blob.data(), s->blob.size(), &d->prog));
    for (auto& w : d->workers)
      if (err.empty()) err = take(zkb_prover_set_program(w->prover, d->prog));
  }
  cudaSetDevice(caller_device);
  if (!err.empty()) throw Error(err);     // ~zkb_session stops and joins the workers and frees what they and this call made
  {
    std::lock_guard<std::mutex> lk(s->mu);
    s->go = true;
    s->cv.notify_all();
  }
  *out = s.release();
  ZKB_API_END
}

zkb_err zkb_session_commit(zkb_session* s, int po2, const void* h_code, uint32_t* h_control_id) {
  ZKB_API_BEGIN
  ZKB_REQUIRE(s && h_control_id, "null argument");
  std::lock_guard<std::mutex> commit_lock(s->commit_mu);
  {
    std::lock_guard<std::mutex> lk(s->mu);
    ZKB_REQUIRE(!s->stopping, "the session is being freed");
    ZKB_REQUIRE(!s->control_ids.count(po2), "the session already holds a code commitment at po2 " + std::to_string(po2));
  }
  const size_t n = s->devs.size();
  std::vector<std::array<uint32_t, 9>> ids(n);
  std::vector<std::string> errs(n);
  std::vector<std::thread> ths;
  try {
    for (size_t i = 0; i < n; ++i)
      ths.emplace_back([&, i] { errs[i] = take(zkb_program_commit(s->devs[i]->prog, po2, h_code, 0, ids[i].data())); });
  } catch (...) {
    for (auto& t : ths) t.join();
    throw;
  }
  for (auto& t : ths) t.join();
  for (size_t i = 0; i < n; ++i)
    if (!errs[i].empty()) throw Error(errs[i] + " (device " + std::to_string(s->devs[i]->id) + ")");
  for (size_t i = 1; i < n; ++i)
    ZKB_REQUIRE(ids[i] == ids[0], "the code roots at po2 " + std::to_string(po2) + " differ between devices " + std::to_string(s->devs[0]->id) +
                                      " and " + std::to_string(s->devs[i]->id));
  memcpy(h_control_id, ids[0].data(), 9 * 4);
  std::lock_guard<std::mutex> lk(s->mu);
  s->control_ids[po2] = ids[0];
  ZKB_API_END
}

zkb_err zkb_session_control_ids(zkb_session* s, size_t* n, uint32_t* h_out) {
  ZKB_API_BEGIN
  ZKB_REQUIRE(s && n, "null argument");
  std::lock_guard<std::mutex> lk(s->mu);
  if (h_out) {
    ZKB_REQUIRE(*n >= s->control_ids.size(), "h_out holds " + std::to_string(*n) + " entries; the session has " + std::to_string(s->control_ids.size()));
    for (const auto& kv : s->control_ids) {
      memcpy(h_out, kv.second.data(), 9 * 4);
      h_out += 9;
    }
  }
  *n = s->control_ids.size();
  ZKB_API_END
}

zkb_err zkb_session_submit(zkb_session* s, int po2, const uint32_t* h_io, const void* h_data, const void* h_accum, uint64_t* ticket) {
  ZKB_API_BEGIN
  ZKB_REQUIRE(s && ticket, "null argument");
  const zkb::CircuitDef& c = s->circuit;
  ZKB_REQUIRE(h_io || c.out_size == 0, "null io");
  ZKB_REQUIRE(h_data || c.group_size[GROUP_DATA] == 0, "null data trace");
  ZKB_REQUIRE(h_accum || c.group_size[GROUP_ACCUM] == 0 || !c.wsteps.empty(),
              "null accum trace and the circuit blob carries no witness program to compute it");
  Segment seg;
  seg.po2 = po2;
  if (c.out_size) seg.io.assign(h_io, h_io + c.out_size);
  seg.data = h_data;
  seg.accum = h_accum;
  std::lock_guard<std::mutex> lk(s->mu);
  ZKB_REQUIRE(!s->stopping, "the session is being freed");
  ZKB_REQUIRE(s->control_ids.count(po2), "the session has no code commitment at po2 " + std::to_string(po2) + " (zkb_session_commit)");
  seg.ticket = s->next_ticket++;
  s->results[seg.ticket];
  *ticket = seg.ticket;
  s->queue.push_back(std::move(seg));
  s->cv.notify_all();
  ZKB_API_END
}

zkb_err zkb_session_wait(zkb_session* s, uint64_t ticket, uint32_t* h_seal, size_t* words) {
  ZKB_API_BEGIN
  ZKB_REQUIRE(s && words, "null argument");
  std::unique_lock<std::mutex> lk(s->mu);
  ++s->waiters;
  struct Leave {      // destroyed before lk, so under the lock
    zkb_session* s;
    ~Leave() { --s->waiters; s->cv.notify_all(); }
  } leave{s};
  auto it = s->results.find(ticket);
  for (;;) {
    ZKB_REQUIRE(it != s->results.end(), "unknown or released ticket " + std::to_string(ticket));
    if (it->second.done) break;
    s->cv.wait(lk);
    it = s->results.find(ticket);
  }
  Result& r = it->second;
  if (!r.err.empty()) {
    std::string e = std::move(r.err);
    s->results.erase(it);
    throw Error(e);
  }
  if (!h_seal) {
    *words = r.seal.size();
  } else {
    ZKB_REQUIRE(*words >= r.seal.size(), "h_seal holds " + std::to_string(*words) + " words; the seal has " + std::to_string(r.seal.size()));
    memcpy(h_seal, r.seal.data(), r.seal.size() * 4);
    *words = r.seal.size();
    s->results.erase(it);
  }
  ZKB_API_END
}

zkb_err zkb_session_free(zkb_session* s) {
  ZKB_API_BEGIN
  delete s;
  ZKB_API_END
}

}  // extern "C"
