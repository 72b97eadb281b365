// Host-side prover orchestration over the device operators: the B200 stand-in for risc0-zkp 1.2.5
// `prove::{Prover, poly_group::PolyGroup, merkle::MerkleTreeProver, fri::fri_prove, write_iop::WriteIOP}` and for the
// circuit crate's `prove_segment` driver (un-vendored; call site /root/reference/crates/guest-prover-r0/src/prover.rs:90).
// The ORDER of transcript operations follows SURVEY.md App. D exactly -- it is what makes Merkle roots, FRI
// commitments and seal words comparable with the reference.  What differs is where things run:
//   * every buffer stays on the device for the whole segment; the host only sees roots, top layers, the DEEP
//     evaluations, the 1024 final FRI coefficients and the query answers;
//   * the `poly_divide` step that risc0 1.2.x does on the CPU through `combos.view_mut` (a 16*(combos+1)*n-byte round
//     trip) is a device kernel (k_poly.cu);
//   * the query phase is 7 launches and one copy instead of ~6000 single-digest reads (k_query.cu);
//   * operators are stream-ordered; the host blocks only where Fiat-Shamir needs a value (one small copy per commit).
#include "ops.cuh"
#include "transcript.hpp"
#include <memory>
#include <mutex>
#include <time.h>

namespace zkb {

struct WriteIOP {
  std::vector<uint32_t> proof;
  HostRng rng;
  void write(const uint32_t* w, size_t n) { proof.insert(proof.end(), w, w + n); }
  void write_fp4(const std::vector<Fp4>& v) { for (const Fp4& x : v) for (int j = 0; j < 4; ++j) proof.push_back(x.c[j].v); }
  void commit(const Digest& d) { rng.mix(d); }
};

// ---- device memory helper (stream-ordered pool) ------------------------------------------------------------
struct DevBuf {
  zkb_ctx* ctx = nullptr; uint32_t* p = nullptr; size_t words = 0;
  DevBuf() {}
  DevBuf(zkb_ctx* c, size_t w) : ctx(c), words(w) { pool_alloc(c, &p, std::max<size_t>(w, 4) * 4); }
  DevBuf(const DevBuf&) = delete; DevBuf& operator=(const DevBuf&) = delete;
  DevBuf(DevBuf&& o) noexcept { *this = std::move(o); }
  DevBuf& operator=(DevBuf&& o) noexcept { reset(); ctx = o.ctx; p = o.p; words = o.words; o.p = nullptr; o.words = 0; return *this; }
  void reset() { if (p) cudaFreeAsync(p, ctx->stream); p = nullptr; words = 0; }
  ~DevBuf() { reset(); }
};
static void d2h(zkb_ctx* ctx, void* dst, const void* src, size_t bytes) {
  ZKB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  ZKB_CUDA(cudaStreamSynchronize(ctx->stream));
}
static void h2d(zkb_ctx* ctx, void* dst, const void* src, size_t bytes) {   // src is pageable: the runtime stages it before returning
  ZKB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
}

// ---- MerkleTreeParams / MerkleTreeProver (merkle.rs, prove/merkle.rs; App. D.2, D.5) ---------------------------
struct MerkleParams {
  size_t rows, cols, layers, top_layer, top_size;
  MerkleParams() : rows(0), cols(0), layers(0), top_layer(0), top_size(1) {}
  MerkleParams(size_t r, size_t c, size_t queries) : rows(r), cols(c) {
    layers = 0; while (((size_t)1 << layers) < r) ++layers;
    top_layer = 0;
    for (size_t i = 1; i < layers; ++i) { if (((size_t)1 << i) > queries) break; top_layer = i; }
    top_size = (size_t)1 << top_layer;
  }
  size_t path_len() const { return layers - top_layer; }
};
struct DeviceMerkle {
  MerkleParams params;
  const uint32_t* matrix = nullptr;   // cols x rows, not owned
  DevBuf nodes;                       // 2*rows digests
  Digest root;
  std::vector<uint32_t> top;          // the top layer, nodes[top_size .. 2*top_size), as commit() read it back
  void build(zkb_ctx* ctx, const uint32_t* m, size_t rows, size_t cols) {
    params = MerkleParams(rows, cols, QUERIES);
    matrix = m;
    nodes = DevBuf(ctx, 2 * rows * 8);
    hash_rows(ctx, nodes.p + rows * 8, m, rows, cols);
    merkle_build(ctx, nodes.p, rows);
  }
  // MerkleTreeProver::commit: write the top layer, then mix the root.  One small blocking copy.
  void commit(zkb_ctx* ctx, WriteIOP& iop) {
    read_top(ctx);
    write(iop);
  }
  // reads the top layer and the root back; blocks until the tree is built
  void read_top(zkb_ctx* ctx) {
    std::vector<uint32_t> upper(2 * params.top_size * 8);
    d2h(ctx, upper.data() + 8, nodes.p + 8, (2 * params.top_size - 1) * 32);    // nodes[1 .. 2*top_size)
    top.assign(upper.begin() + params.top_size * 8, upper.end());
    memcpy(root.w, upper.data() + 8, 32);
  }
  // the transcript actions of commit() for a tree committed before: the same top layer and root, no device work
  void write(WriteIOP& iop) const {
    iop.write(top.data(), top.size());
    iop.commit(root);
  }
  QueryTree query_tree(uint32_t out_offset) const {
    return QueryTree{matrix, nodes.p, (uint32_t)params.rows, (uint32_t)params.cols, (uint32_t)params.top_size, (uint32_t)params.path_len(), out_offset};
  }
  uint32_t query_words() const { return (uint32_t)(params.cols + params.path_len() * 8); }
};

// ---- PolyGroup (prove/poly_group.rs) ---------------------------------------------------------------------
struct PolyGroup {
  size_t count = 0, n = 0;
  DevBuf coeffs, evaluated;
  DeviceMerkle merkle;
  // takes ownership of bit-reversed coefficients (count x n).  The reference bit-reverses them here (poly_group.rs) because its DEEP
  // evaluation and mix read natural order; here `coeffs` STAYS bit-reversed -- batch_evaluate_any takes the order as a flag, the mix is
  // elementwise, and only the three combo polynomials are put in natural order afterwards (48 MB instead of 1.24 GB per segment).
  void build(zkb_ctx* ctx, DevBuf&& c, size_t count_, int po2) {
    count = count_; n = (size_t)1 << po2;
    coeffs = std::move(c);
    evaluated = DevBuf(ctx, count * n * INV_RATE);
    ntt_forward(ctx, evaluated.p, coeffs.p, count, po2 + 2, 2);
    merkle.build(ctx, evaluated.p, n * INV_RATE, count);
  }
};

struct FriRound { DevBuf evaluated; DeviceMerkle merkle; size_t domain = 0; };

// ZKB_PROFILE=1: synchronise at every phase boundary of a segment proof and print host-clocked phase times to stderr
// (diagnostics only; the extra synchronisations cost a little throughput).
struct PhaseTimer {
  zkb_ctx* ctx; bool on; double t0;
  static double now() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6; }
  explicit PhaseTimer(zkb_ctx* c) : ctx(c) { const char* e = getenv("ZKB_PROFILE"); on = e && e[0] == '1'; if (on) { cudaStreamSynchronize(ctx->stream); t0 = now(); } }
  void mark(const char* what) {
    if (!on) return;
    double host = now();
    cudaStreamSynchronize(ctx->stream);
    double t = now();
    fprintf(stderr, "zkb200 phase %-28s %8.3f ms (host returned after %8.3f ms)\n", what, t - t0, host - t0);
    t0 = t;
  }
};

// A completed commitment of the code group, i.e. of the program at one po2: a private copy of the trace (the witness program reads it,
// and a caller's buffer may change under the same pointer), the bit-reversed coefficients, the LDE matrix and the Merkle tree with its
// top layer and root (~640 MB at po2 20).  A prover keeps its last one (zkb_prover::code); a zkb_program keeps one per committed po2.
struct CodeCommit {
  int po2 = -1;                 // -1: empty
  DevBuf trace;
  PolyGroup group;
  // Prover::commit_group(code) without its transcript actions (group.merkle.write replays those): make_coeffs out of place, so that
  // the copy keeps the trace, PolyGroup::new, and the top-layer read-back.  `t` is the trace in device memory; `uploaded` is the buffer
  // it was uploaded into, taken over as the copy, or empty when `t` is the caller's buffer and has to be copied.
  void build(zkb_ctx* ctx, DevBuf&& uploaded, const uint32_t* t, size_t cols, int po2_, PhaseTimer& pt) {
    const size_t words = cols << po2_;
    if (uploaded.p) {
      trace = std::move(uploaded);
    } else {
      trace = DevBuf(ctx, words);
      if (words) ZKB_CUDA(cudaMemcpyAsync(trace.p, t, words * 4, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    DevBuf c(ctx, words);
    ntt_inverse(ctx, c.p, cols, po2_, true, trace.p);
    pt.mark("commit_group: iNTT+zk_shift");
    group.build(ctx, std::move(c), cols, po2_);
    pt.mark("commit_group: LDE+hash+merkle");
    group.merkle.read_top(ctx);
    pt.mark("commit_group: commit (d2h)");
    po2 = po2_;
  }
};

// zkb_program (include/zkb200.h): one circuit's code commitments, one per po2, built on a private ctx of the device (own stream and pool,
// so the storage depends on no caller's ctx) and read by any prover on that device.  An entry is complete when zkb_program_commit returns
// and is neither changed nor removed until the program is destroyed, so provers on other streams read it without synchronisation.
// Ownership is shared between the caller's handle and every prover holding the program; each holder synchronises its stream before it
// lets go (zkb_prover::release), so the last one frees memory no stream still reads.
struct Program {
  zkb_ctx* ctx = nullptr;
  std::vector<uint32_t> blob;
  CircuitDef circuit;
  std::mutex commit_mu;                     // one commit at a time on the private ctx
  mutable std::mutex map_mu;                // guards `entries` alone: provers look entries up while a new po2 is being committed
  std::map<int, std::unique_ptr<CodeCommit>> entries;
  const CodeCommit* find(int po2) const {
    std::lock_guard<std::mutex> lock(map_mu);
    auto it = entries.find(po2);
    return it == entries.end() ? nullptr : it->second.get();
  }
  ~Program() {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    entries.clear();                        // stream-ordered frees on the private stream
    zkb_free_error(zkb_destroy(ctx));       // synchronises that stream, then destroys its pool
  }
};
static std::string no_program_entry(int po2) { return "the attached program has no code commitment at po2 " + std::to_string(po2) + " (zkb_program_commit)"; }

}  // namespace zkb

struct zkb_program { std::shared_ptr<zkb::Program> s; };

using namespace zkb;

// ONE host->device copy stream per device, shared by every prover of the process: staged uploads are then served FIFO, each at the
// full link rate, in the order the workers asked for them (= the order their proofs need them).  With a stream per prover the DMA
// engine interleaves the three workers' 1.17 GB uploads, every one of them lands late, and on a link that is barely fast enough
// (23 GB/s against the 21.6 GB/s a GPU consumes: GPUs 0-3 of this pool when all eight upload) the proofs wait for their traces.
static cudaStream_t shared_copy_stream(int device) {
  static std::mutex mu;
  static std::map<int, cudaStream_t> streams;
  std::lock_guard<std::mutex> lock(mu);
  auto it = streams.find(device);
  if (it != streams.end()) return it->second;
  cudaStream_t s = nullptr;
  ZKB_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
  streams[device] = s;      // lives as long as the process (like the device's memory pool)
  return s;
}

static const char PROOF_SYSTEM_INFO[17] = "RISC0_STARK:v1__";
static Digest hash_protocol_info(const uint8_t* info) {
  uint32_t e[16];
  for (int i = 0; i < 16; ++i) e[i] = Fp::from(info[i]).v;
  return hash_words(e, 16);
}

struct zkb_prover {
  zkb_ctx* ctx = nullptr;
  std::vector<uint32_t> blob;
  CircuitDef circuit;
  std::unique_ptr<WriteIOP> iop;
  int po2 = 0; size_t n = 0;
  PolyGroup groups[3];            // this segment's accum and data groups; the code group is seg_code's or code's (see group())
  PolyGroup check_group;
  // The code group is the program: zkb_verify_segment accepts a seal only if its code root is one of the circuit's control IDs for
  // that po2, so every valid proof of a circuit at one po2 commits the same code trace.  The last code commit that completed is kept
  // across segments (reset() leaves it alone) and reused when the next code trace is equal to it word for word (~640 MB at po2 20).
  CodeCommit code;
  // zkb_prover_set_program: a NULL code argument proves from the attached program's commitment at the segment's po2.  The segment
  // holds the program it read from until reset(), so detaching mid-segment does not free what its finish still reads.
  std::shared_ptr<Program> program, seg_program;
  const CodeCommit* seg_code = nullptr;
  const PolyGroup& group(int g) const { return g != GROUP_CODE ? groups[g] : seg_code ? seg_code->group : code.group; }
  // lets go of a program: every read of its entries on this prover's stream must be done first
  void release(std::shared_ptr<Program>& h) {
    if (!h) return;
    ZKB_CUDA(cudaStreamSynchronize(ctx->stream));
    h.reset();
  }
  std::vector<std::unique_ptr<FriRound>> fri_rounds;
  std::vector<Digest> roots;
  std::vector<uint32_t> io, mix;
  bool begun = false, finished = false;

  // Double-buffered trace staging: segment k+1's host->device copy runs on `copy_stream` while segment k is proven on the
  // ctx stream (zkb_prover_stage_traces / zkb_prove_staged).
  struct TraceSlot {
    uint32_t* buf[3] = {nullptr, nullptr, nullptr};
    size_t words[3] = {0, 0, 0};
    cudaEvent_t uploaded[3] = {nullptr, nullptr, nullptr};      // one per trace group: a group's commit starts as soon as ITS bytes have landed
    cudaEvent_t consumed = nullptr;
    int po2 = -1;
    bool full = false;
    bool device_accum = false;      // no accum trace was staged: zkb_prove_staged fills the group with the circuit's witness program
    bool code_from_program = false; // no code trace was staged: the attached program's commitment is used, and nothing is uploaded for it
  };
  TraceSlot slots[2];
  cudaStream_t copy_stream = nullptr;
  bool own_copy_stream = false;
  int stage_idx = 0, prove_idx = 0;
  const cudaEvent_t* group_ready = nullptr;      // staged proof in progress: per-group upload events the commits wait on

  void stage_traces(int po2_, const void* const h_traces[3]) {
    ZKB_REQUIRE(po2_ >= 6 && po2_ + 2 <= MAX_PO2, "segment po2 out of range [6, 24]");
    const bool code_from_program = !h_traces[GROUP_CODE] && program;
    ZKB_REQUIRE(!code_from_program || program->find(po2_), no_program_entry(po2_));
    if (!copy_stream) {
      static const bool priv = [] { const char* e = getenv("ZKB_COPY_STREAM"); return e && !strcmp(e, "private"); }();      // measurement knob: one stream per prover (round-1 behaviour)
      if (priv) { ZKB_CUDA(cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking)); own_copy_stream = true; }
      else copy_stream = shared_copy_stream(ctx->device);
    }
    TraceSlot& sl = slots[stage_idx];
    ZKB_REQUIRE(!sl.full, "both staging slots are full: call zkb_prove_staged first");
    if (!sl.consumed) {
      for (int g = 0; g < 3; ++g) ZKB_CUDA(cudaEventCreateWithFlags(&sl.uploaded[g], cudaEventDisableTiming));
      ZKB_CUDA(cudaEventCreateWithFlags(&sl.consumed, cudaEventDisableTiming));
    } else {
      ZKB_CUDA(cudaStreamWaitEvent(copy_stream, sl.consumed, 0));    // the proof that last read this slot must be done with it
    }
    const size_t rows = (size_t)1 << po2_;
    // in commit order (code, data, accum): the proof of this segment can start when the 64 MB code group is in, and the data /
    // accum uploads run behind its first commits instead of in front of them
    static const int ORDER[3] = {GROUP_CODE, GROUP_DATA, GROUP_ACCUM};
    for (int k = 0; k < 3; ++k) {
      const int g = ORDER[k];
      size_t words = (size_t)circuit.group_size[g] * rows;
      if (sl.words[g] < words && !(g == GROUP_CODE && code_from_program)) {
        if (sl.buf[g]) { ZKB_CUDA(cudaStreamSynchronize(ctx->stream)); ZKB_CUDA(cudaStreamSynchronize(copy_stream)); ZKB_CUDA(cudaFree(sl.buf[g])); }
        ZKB_CUDA(cudaMalloc((void**)&sl.buf[g], std::max<size_t>(words, 4) * 4));
        sl.words[g] = words;
      }
      if (words && h_traces[g]) ZKB_CUDA(cudaMemcpyAsync(sl.buf[g], h_traces[g], words * 4, cudaMemcpyHostToDevice, copy_stream));
      ZKB_CUDA(cudaEventRecord(sl.uploaded[g], copy_stream));
    }
    sl.device_accum = h_traces[GROUP_ACCUM] == nullptr && circuit.group_size[GROUP_ACCUM] != 0;
    sl.code_from_program = code_from_program;
    sl.po2 = po2_; sl.full = true;
    stage_idx ^= 1;
  }
  void prove_staged(const uint32_t* h_io) {
    TraceSlot& sl = slots[prove_idx];
    ZKB_REQUIRE(sl.full, "no staged traces: call zkb_prover_stage_traces first");
    struct Guard { const cudaEvent_t*& r; ~Guard() { r = nullptr; } } guard{group_ready};      // also on an error path
    group_ready = sl.uploaded;
    segment_begin(sl.po2, h_io, sl.code_from_program ? nullptr : sl.buf[GROUP_CODE], sl.buf[GROUP_DATA], true, nullptr);
    if (sl.device_accum) {
      // the reference's prove_segment order: commit code + data, draw `mix`, CircuitHal::accumulate, commit accum -- with the witness
      // program of the circuit blob run on the device, so this group (14 % of SYN-280's trace bytes) never crosses the host link
      ZKB_CUDA(cudaMemsetAsync(sl.buf[GROUP_ACCUM], 0, sl.words[GROUP_ACCUM] * 4, ctx->stream));
      const uint32_t* code_trace = seg_code ? seg_code->trace.p : sl.buf[GROUP_CODE];      // the program's retained copy
      accumulate(ctx, circuit, sl.buf[GROUP_ACCUM], code_trace, sl.buf[GROUP_DATA], mix.data(), io.data(), sl.po2);
    }
    segment_finish(sl.buf[GROUP_ACCUM], true);
    ZKB_CUDA(cudaEventRecord(sl.consumed, ctx->stream));
    sl.full = false;
    prove_idx ^= 1;
  }
  void free_staging() {
    for (TraceSlot& sl : slots) {
      for (int g = 0; g < 3; ++g) { if (sl.buf[g]) cudaFree(sl.buf[g]); sl.buf[g] = nullptr; sl.words[g] = 0; }
      for (int g = 0; g < 3; ++g) if (sl.uploaded[g]) cudaEventDestroy(sl.uploaded[g]);
      if (sl.consumed) cudaEventDestroy(sl.consumed);
      sl = TraceSlot();
    }
    if (copy_stream && own_copy_stream) cudaStreamDestroy(copy_stream);
    copy_stream = nullptr; own_copy_stream = false;      // the shared per-device stream is not ours to destroy
  }

  void reset() {
    iop.reset(new WriteIOP());
    for (auto& g : groups) g = PolyGroup();
    check_group = PolyGroup();
    fri_rounds.clear(); roots.clear(); io.clear(); mix.clear();
    begun = finished = false;
    seg_code = nullptr;
    release(seg_program);
  }

  // Prover::commit_group: make_coeffs (interpolate + zk_shift), PolyGroup::new, merkle.commit
  void commit_group(int g, const void* trace, bool on_device) {
    PhaseTimer pt(ctx);
    size_t cols = circuit.group_size[g];
    if (group_ready) ZKB_CUDA(cudaStreamWaitEvent(ctx->stream, group_ready[g], 0));
    if (g == GROUP_CODE) { commit_code(trace, on_device, pt); return; }
    DevBuf c(ctx, cols * n);
    // a trace that is already on the device is read in place by the first iNTT pass (no device-to-device copy)
    if (cols && !on_device) ZKB_CUDA(cudaMemcpyAsync(c.p, trace, cols * n * 4, cudaMemcpyHostToDevice, ctx->stream));
    pt.mark("commit_group: upload");
    ntt_inverse(ctx, c.p, cols, po2, true, on_device ? (const uint32_t*)trace : nullptr);
    pt.mark("commit_group: iNTT+zk_shift");
    groups[g].build(ctx, std::move(c), cols, po2);
    pt.mark("commit_group: LDE+hash+merkle");
    groups[g].merkle.commit(ctx, *iop);
    pt.mark("commit_group: commit (d2h)");
    roots.push_back(groups[g].merkle.root);
  }

  // The code group.  From the program: replay the transcript actions of its commitment; the prover's own retained commitment is
  // neither read nor changed.  From a trace: with the trace in device memory, compare it with the retained one.  Equal: the commitment
  // is reused and only its transcript actions are replayed.  Different, or another po2: commit, then retain the result.
  void commit_code(const void* trace, bool on_device, PhaseTimer& pt) {
    if (seg_code) {
      seg_code->group.merkle.write(*iop);
      roots.push_back(seg_code->group.merkle.root);
      pt.mark("commit_group: code from program");
      return;
    }
    const size_t cols = circuit.group_size[GROUP_CODE], words = cols * n;
    DevBuf up;
    if (!on_device) {
      up = DevBuf(ctx, words);
      if (words) ZKB_CUDA(cudaMemcpyAsync(up.p, trace, words * 4, cudaMemcpyHostToDevice, ctx->stream));
      trace = up.p;
      pt.mark("commit_group: upload");
    }
    const uint32_t* t = (const uint32_t*)trace;
    if (code.po2 == po2 && words_equal(ctx, t, code.trace.p, words)) {
      code.group.merkle.write(*iop);
      roots.push_back(code.group.merkle.root);
      pt.mark("commit_group: code reused");
      return;
    }
    code = CodeCommit();          // dropped before the commit: an error in it leaves nothing retained, not a half-updated state
    CodeCommit next;
    next.build(ctx, std::move(up), t, cols, po2, pt);
    next.group.merkle.write(*iop);
    roots.push_back(next.group.merkle.root);
    code = std::move(next);
  }

  // code == NULL with a program attached: the program's commitment at po2_ is this segment's code group
  void segment_begin(int po2_, const uint32_t* h_io, const void* code, const void* data, bool on_device, uint32_t* h_mix_out) {
    ZKB_REQUIRE(po2_ >= 6 && po2_ + 2 <= MAX_PO2, "segment po2 out of range [6, 24]");
    const CodeCommit* from_program = nullptr;
    if (!code && program) {
      from_program = program->find(po2_);
      ZKB_REQUIRE(from_program, no_program_entry(po2_));
    }
    ZKB_REQUIRE(code || from_program || circuit.group_size[GROUP_CODE] == 0, "null code trace and no program attached");
    reset();
    if (from_program) { seg_program = program; seg_code = from_program; }
    po2 = po2_; n = (size_t)1 << po2;
    iop->commit(hash_protocol_info((const uint8_t*)PROOF_SYSTEM_INFO));
    iop->commit(hash_protocol_info(circuit.info));
    for (uint32_t i = 0; i < circuit.out_size; ++i) ZKB_REQUIRE(h_io[i] < P, "io word is not a canonical field element (must be < P)");
    io.assign(h_io, h_io + circuit.out_size);
    std::vector<uint32_t> hdr(io);
    hdr.push_back((uint32_t)po2);      // risc0 prove_segment appends Elem::from_u32_slice(&[po2]): the RAW word (a bytemuck cast), not enc(po2)
    iop->commit(hash_words(hdr.data(), hdr.size()));
    iop->write(hdr.data(), hdr.size());
    commit_group(GROUP_CODE, code, on_device);
    commit_group(GROUP_DATA, data, on_device);
    mix.resize(circuit.mix_size);
    for (uint32_t i = 0; i < circuit.mix_size; ++i) mix[i] = iop->rng.random_elem().v;
    if (h_mix_out && circuit.mix_size) memcpy(h_mix_out, mix.data(), 4 * circuit.mix_size);
    begun = true;
  }

  void segment_finish(const void* accum, bool on_device) {
    ZKB_REQUIRE(begun && !finished, "segment_finish called out of order");
    commit_group(GROUP_ACCUM, accum, on_device);
    finalize();
    finished = true;
  }

  // Prover::finalize (App. D.3) + fri_prove (D.4)
  void finalize() {
    const CircuitDef& c = circuit;
    WriteIOP& io_p = *iop;
    const size_t domain = n * INV_RATE;
    PhaseTimer pt(ctx);
    // 1. check polynomial
    Fp4 poly_mix = io_p.rng.random_ext_elem();
    {
      DevBuf check(ctx, EXT_SIZE * domain);
      const uint32_t* ev[3] = {group(0).evaluated.p, group(1).evaluated.p, group(2).evaluated.p};
      eval_check(ctx, check.p, c, ev, mix.data(), io.data(), poly_mix, po2);
      pt.mark("finalize: eval_check");
      ntt_inverse(ctx, check.p, EXT_SIZE, po2 + 2, false);
      check_group.build(ctx, std::move(check), CHECK_SIZE, po2);
    }
    check_group.merkle.commit(ctx, io_p);
    pt.mark("finalize: check group commit");
    roots.push_back(check_group.merkle.root);
    // 2. DEEP evaluations of every tap and of the 16 check polynomials, one device pass + one copy
    Fp4 z = io_p.rng.random_ext_elem();
    Fp back_one = inv(pow(Fp::from(137), (uint64_t)1 << (MAX_ROU_PO2 - po2)));   // ROU_REV[po2]
    const size_t tap_size = c.tap_size();
    std::vector<Fp4> all_xs(tap_size + CHECK_SIZE), eval_u(tap_size + CHECK_SIZE);
    std::vector<uint32_t> which(tap_size + CHECK_SIZE);
    Fp4 z_pow = pow(z, EXT_SIZE);
    for (size_t t = 0; t < tap_size; ++t) { which[t] = c.taps[t].column; all_xs[t] = z * pow(back_one, c.taps[t].back); }
    for (size_t i = 0; i < CHECK_SIZE; ++i) { which[tap_size + i] = (uint32_t)i; all_xs[tap_size + i] = z_pow; }
    {
      DevBuf d_which(ctx, which.size()), d_xs(ctx, 4 * all_xs.size()), d_out(ctx, 4 * all_xs.size());
      h2d(ctx, d_which.p, which.data(), which.size() * 4);
      h2d(ctx, d_xs.p, all_xs.data(), all_xs.size() * 16);
      for (uint32_t g = 0; g < 3; ++g) {
        size_t b = c.group_tap_begin(g), e = c.group_tap_end(g);
        batch_evaluate_any(ctx, group(g).coeffs.p, po2, d_which.p + b, d_xs.p + 4 * b, d_out.p + 4 * b, e - b, true);
      }
      batch_evaluate_any(ctx, check_group.coeffs.p, po2, d_which.p + tap_size, d_xs.p + 4 * tap_size, d_out.p + 4 * tap_size, CHECK_SIZE, true);
      d2h(ctx, eval_u.data(), d_out.p, eval_u.size() * 16);
    }
    pt.mark("finalize: DEEP evaluations");
    // 3. coeff_u: per-register interpolation (host, a few field ops), check evaluations appended
    std::vector<Fp4> coeff_u(tap_size + CHECK_SIZE);
    for (const RegisterDef& r : c.regs) poly_interpolate(&coeff_u[r.tap_pos], &all_xs[r.tap_pos], &eval_u[r.tap_pos], r.size);
    for (size_t i = 0; i < CHECK_SIZE; ++i) coeff_u[tap_size + i] = eval_u[tap_size + i];
    // 4.
    io_p.write_fp4(coeff_u);
    io_p.commit(hash_words((const uint32_t*)coeff_u.data(), coeff_u.size() * 4));
    Fp4 mix_c = io_p.rng.random_ext_elem();
    // 5. combos
    const size_t combos_size = c.combos_size();
    DevBuf combos(ctx, (combos_size + 1) * n * 4);
    ZKB_CUDA(cudaMemsetAsync(combos.p, 0, (combos_size + 1) * n * 16, ctx->stream));
    {
      std::vector<uint32_t> ids;
      for (const RegisterDef& r : c.regs) ids.push_back(r.combo_id);
      for (size_t i = 0; i < CHECK_SIZE; ++i) ids.push_back((uint32_t)combos_size);
      DevBuf d_ids(ctx, ids.size());
      h2d(ctx, d_ids.p, ids.data(), ids.size() * 4);
      Fp4 cur = Fp4::one();
      size_t off = 0;
      for (uint32_t g = 0; g < 3; ++g) {
        size_t cols = c.group_size[g];
        mix_poly_coeffs(ctx, combos.p, cur, mix_c, group(g).coeffs.p, d_ids.p + off, cols, n, (uint32_t)combos_size + 1);
        cur *= pow(mix_c, cols);
        off += cols;
      }
      mix_poly_coeffs(ctx, combos.p, cur, mix_c, check_group.coeffs.p, d_ids.p + off, CHECK_SIZE, n, (uint32_t)combos_size + 1);
      batch_bit_reverse_ext(ctx, combos.p, combos_size + 1, po2);      // the mix ran over bit-reversed coefficients: natural order from here on
    }
    pt.mark("finalize: coeff_u + mix_poly_coeffs");
    // 6. subtract the interpolants (touches only the lowest coefficients), then divide on the device
    {
      uint32_t max_sz = 1;
      for (const RegisterDef& r : c.regs) max_sz = std::max(max_sz, r.size);
      ZKB_REQUIRE(max_sz <= n, "more taps per register than rows");
      std::vector<Fp4> delta((combos_size + 1) * max_sz);
      Fp4 cur = Fp4::one();
      for (const RegisterDef& r : c.regs) {
        for (uint32_t i = 0; i < r.size; ++i) delta[r.combo_id * max_sz + i] += cur * coeff_u[r.tap_pos + i];
        cur *= mix_c;
      }
      for (size_t i = 0; i < CHECK_SIZE; ++i) { delta[combos_size * max_sz] += cur * coeff_u[tap_size + i]; cur *= mix_c; }
      size_t n_div = 1;
      for (auto& cb : c.combos) n_div += cb.size();
      DevBuf d_delta(ctx, delta.size() * 4), d_rem(ctx, n_div * 4);
      h2d(ctx, d_delta.p, delta.data(), delta.size() * 16);
      sub_small(ctx, combos.p, n, d_delta.p, (uint32_t)combos_size + 1, max_sz);
      size_t k = 0;
      for (size_t ci = 0; ci < combos_size; ++ci)
        for (uint32_t back : c.combos[ci]) poly_divide(ctx, combos.p + ci * n * 4, n, z * pow(back_one, back), d_rem.p + 4 * k++);
      poly_divide(ctx, combos.p + combos_size * n * 4, n, z_pow, d_rem.p + 4 * k++);
      std::vector<uint32_t> rem(4 * n_div);
      d2h(ctx, rem.data(), d_rem.p, rem.size() * 4);
      for (uint32_t w : rem) ZKB_REQUIRE(w == 0, "combo division left a remainder (inconsistent DEEP evaluations)");
    }
    pt.mark("finalize: divide");
    // 7. FRI
    DevBuf fin(ctx, EXT_SIZE * n);
    eltwise_sum_extelem(ctx, fin.p, combos.p, n, combos_size + 1);
    combos.reset();
    batch_bit_reverse(ctx, fin.p, EXT_SIZE, po2);
    fri_prove(std::move(fin));
    pt.mark("finalize: fri_prove + queries");
  }

  void fri_prove(DevBuf coeffs) {
    WriteIOP& io_p = *iop;
    size_t len = n;
    const size_t orig_domain = n * INV_RATE;
    while (len > FRI_MIN_DEGREE) {
      int lpo2 = 0; while (((size_t)1 << lpo2) < len) ++lpo2;
      std::unique_ptr<FriRound> r(new FriRound);
      r->domain = len * INV_RATE;
      r->evaluated = DevBuf(ctx, EXT_SIZE * r->domain);
      ntt_forward(ctx, r->evaluated.p, coeffs.p, EXT_SIZE, lpo2 + 2, 2);
      r->merkle.build(ctx, r->evaluated.p, r->domain / FRI_FOLD, FRI_FOLD * EXT_SIZE);
      r->merkle.commit(ctx, io_p);
      roots.push_back(r->merkle.root);
      Fp4 fold_mix = io_p.rng.random_ext_elem();
      DevBuf out(ctx, coeffs.words / FRI_FOLD);
      fri_fold(ctx, out.p, coeffs.p, fold_mix, out.words / EXT_SIZE);
      coeffs = std::move(out);
      len /= FRI_FOLD;
      fri_rounds.push_back(std::move(r));
    }
    {
      int lpo2 = 0; while (((size_t)1 << lpo2) < len) ++lpo2;
      batch_bit_reverse(ctx, coeffs.p, EXT_SIZE, lpo2);     // `coeffs` is not needed in bit-reversed order any more
      std::vector<uint32_t> fin(coeffs.words);
      d2h(ctx, fin.data(), coeffs.p, fin.size() * 4);
      io_p.write(fin.data(), fin.size());
      io_p.commit(hash_words(fin.data(), fin.size()));
    }
    // queries: all positions first (writes do not feed the rng), then one gather launch per tree and one copy
    int bits = 0; while (((size_t)1 << bits) < orig_domain) ++bits;
    const uint32_t n_trees = 4 + (uint32_t)fri_rounds.size();
    std::vector<uint32_t> idx((size_t)n_trees * QUERIES);
    for (size_t q = 0; q < QUERIES; ++q) {
      size_t pos = io_p.rng.random_bits(bits);
      for (uint32_t t = 0; t < 4; ++t) idx[t * QUERIES + q] = (uint32_t)pos;
      for (size_t r = 0; r < fri_rounds.size(); ++r) {
        size_t group = pos % (fri_rounds[r]->domain / FRI_FOLD);
        idx[(4 + r) * QUERIES + q] = (uint32_t)group;
        pos = group;
      }
    }
    std::vector<QueryTree> trees;
    uint32_t off = 0;
    const DeviceMerkle* gm[4] = {&group(0).merkle, &group(1).merkle, &group(2).merkle, &check_group.merkle};
    for (int t = 0; t < 4; ++t) { trees.push_back(gm[t]->query_tree(off)); off += gm[t]->query_words(); }
    for (auto& r : fri_rounds) { trees.push_back(r->merkle.query_tree(off)); off += r->merkle.query_words(); }
    const uint32_t words_per_query = off;
    DevBuf d_idx(ctx, idx.size()), d_out(ctx, (size_t)words_per_query * QUERIES);
    h2d(ctx, d_idx.p, idx.data(), idx.size() * 4);
    for (uint32_t t = 0; t < n_trees; ++t) gather_queries(ctx, d_out.p, words_per_query, trees[t], d_idx.p + (size_t)t * QUERIES, (uint32_t)QUERIES);
    size_t base = io_p.proof.size();
    io_p.proof.resize(base + (size_t)words_per_query * QUERIES);
    d2h(ctx, io_p.proof.data() + base, d_out.p, (size_t)words_per_query * QUERIES * 4);
  }

  // core/poly.rs poly_interpolate for the 1- and 2-point cases plus general Lagrange (host; a handful of taps)
  static void poly_interpolate(Fp4* out, const Fp4* x, const Fp4* fx, size_t size) {
    if (size == 1) { out[0] = fx[0]; return; }
    if (size == 2) {
      out[1] = (fx[0] - fx[1]) * inv(x[0] - x[1]);
      out[0] = fx[0] - out[1] * x[0];
      return;
    }
    std::vector<Fp4> ft(size + 1);
    ft[0] = Fp4::one();
    for (size_t i = 0; i < size; ++i) {
      for (size_t j = i + 1; j >= 1; --j) ft[j] = ft[j - 1] - x[i] * ft[j];
      ft[0] = Fp4::zero() - x[i] * ft[0];
    }
    for (size_t i = 0; i < size; ++i) out[i] = Fp4::zero();
    for (size_t i = 0; i < size; ++i) {
      // fr = ft / (x - x_i) by synthetic division (quotient in fr[0..size)), scaled so that fr(x_i) == fx_i
      std::vector<Fp4> fr(ft);
      Fp4 cur;
      for (size_t j = size + 1; j-- > 0;) { Fp4 next = x[i] * cur + fr[j]; fr[j] = cur; cur = next; }
      Fp4 at, pw = Fp4::one();
      for (size_t j = 0; j < size; ++j) { at += fr[j] * pw; pw *= x[i]; }
      Fp4 mul = fx[i] * inv(at);
      for (size_t j = 0; j < size; ++j) out[j] += mul * fr[j];
    }
  }
};

extern "C" {

zkb_err zkb_prover_new(zkb_ctx* ctx, const uint32_t* h_circuit, size_t circuit_words, zkb_prover** out) {
  ZKB_API_BEGIN
  use(ctx);
  ZKB_REQUIRE(out != nullptr, "null out pointer");
  std::unique_ptr<zkb_prover> p(new zkb_prover());
  p->ctx = ctx;
  p->circuit = CircuitDef::parse(h_circuit, circuit_words);
  p->blob.assign(h_circuit, h_circuit + circuit_words);
  p->reset();
  *out = p.release();
  ZKB_API_END
}
zkb_err zkb_prover_free(zkb_prover* p) {
  ZKB_API_BEGIN
  if (p) {
    use(p->ctx); p->reset(); p->code = CodeCommit(); cudaStreamSynchronize(p->ctx->stream); if (p->copy_stream) cudaStreamSynchronize(p->copy_stream); p->free_staging();
    p->program.reset();      // the stream is synchronised above
    delete p;
  }
  ZKB_API_END
}
zkb_err zkb_prover_set_program(zkb_prover* p, zkb_program* prog) {
  ZKB_API_BEGIN
  ZKB_REQUIRE(p != nullptr, "null prover");
  use(p->ctx);
  std::shared_ptr<Program> next;
  if (prog) {
    next = prog->s;
    ZKB_REQUIRE(next->ctx->device == p->ctx->device, "the program was made for another device than the prover's");
    ZKB_REQUIRE(next->blob == p->blob, "the program was made for another circuit blob than the prover's");
  }
  p->release(p->program);
  p->program = std::move(next);
  ZKB_API_END
}
zkb_err zkb_program_new(zkb_ctx* ctx, const uint32_t* h_circuit, size_t circuit_words, zkb_program** out) {
  ZKB_API_BEGIN
  use(ctx);
  ZKB_REQUIRE(out != nullptr, "null out pointer");
  std::shared_ptr<Program> s = std::make_shared<Program>();
  s->circuit = CircuitDef::parse(h_circuit, circuit_words);
  s->blob.assign(h_circuit, h_circuit + circuit_words);
  if (zkb_err e = zkb_init(ctx->device, &s->ctx)) { std::string m(e); zkb_free_error(e); throw Error(m); }
  *out = new zkb_program{std::move(s)};
  ZKB_API_END
}
zkb_err zkb_program_commit(zkb_program* prog, int po2, const void* code, int code_on_device, uint32_t* h_control_id) {
  ZKB_API_BEGIN
  ZKB_REQUIRE(prog != nullptr, "null program");
  Program& g = *prog->s;
  ZKB_REQUIRE(po2 >= 6 && po2 + 2 <= MAX_PO2, "segment po2 out of range [6, 24]");
  const size_t cols = g.circuit.group_size[GROUP_CODE], words = cols << po2;
  ZKB_REQUIRE((code || cols == 0) && h_control_id, "null argument");
  std::lock_guard<std::mutex> lock(g.commit_mu);
  ZKB_REQUIRE(!g.find(po2), "the program already holds a code commitment at po2 " + std::to_string(po2) + " (entries are immutable)");
  use(g.ctx);
  PhaseTimer pt(g.ctx);
  DevBuf up;
  if (!code_on_device) {
    up = DevBuf(g.ctx, words);
    if (words) ZKB_CUDA(cudaMemcpyAsync(up.p, code, words * 4, cudaMemcpyHostToDevice, g.ctx->stream));
    pt.mark("commit_group: upload");
  }
  const uint32_t* t = code_on_device ? (const uint32_t*)code : up.p;
  std::unique_ptr<CodeCommit> e(new CodeCommit());
  e->build(g.ctx, std::move(up), t, cols, po2, pt);      // ends in a blocking read-back: the entry is complete on return
  h_control_id[0] = (uint32_t)po2;
  memcpy(h_control_id + 1, e->group.merkle.root.w, 32);
  std::lock_guard<std::mutex> map_lock(g.map_mu);
  g.entries[po2] = std::move(e);
  ZKB_API_END
}
zkb_err zkb_program_control_ids(zkb_program* prog, size_t* n, uint32_t* h_out) {
  ZKB_API_BEGIN
  ZKB_REQUIRE(prog && n, "null argument");
  const Program& g = *prog->s;
  std::lock_guard<std::mutex> lock(g.map_mu);
  if (h_out) {
    ZKB_REQUIRE(*n >= g.entries.size(), "h_out holds " + std::to_string(*n) + " entries; the program has " + std::to_string(g.entries.size()));
    for (const auto& kv : g.entries) {
      *h_out++ = (uint32_t)kv.first;
      memcpy(h_out, kv.second->group.merkle.root.w, 32);
      h_out += 8;
    }
  }
  *n = g.entries.size();
  ZKB_API_END
}
zkb_err zkb_program_free(zkb_program* prog) {
  ZKB_API_BEGIN
  delete prog;
  ZKB_API_END
}
zkb_err zkb_prover_segment_begin(zkb_prover* p, int po2, const uint32_t* h_io, const void* code, const void* data, int traces_on_device, uint32_t* h_mix_out) {
  ZKB_API_BEGIN
  ZKB_REQUIRE(p != nullptr, "null prover");
  use(p->ctx);
  ZKB_REQUIRE((h_io || p->circuit.out_size == 0) && (code || p->program || p->circuit.group_size[GROUP_CODE] == 0) && (data || p->circuit.group_size[GROUP_DATA] == 0), "null argument");
  p->segment_begin(po2, h_io, code, data, traces_on_device != 0, h_mix_out);
  ZKB_API_END
}
zkb_err zkb_prover_segment_finish(zkb_prover* p, const void* accum, int trace_on_device) {
  ZKB_API_BEGIN
  ZKB_REQUIRE(p != nullptr, "null prover");
  use(p->ctx);
  ZKB_REQUIRE(accum || p->circuit.group_size[GROUP_ACCUM] == 0, "null accum trace");
  p->segment_finish(accum, trace_on_device != 0);
  ZKB_API_END
}
zkb_err zkb_prove_segment(zkb_prover* p, int po2, const uint32_t* h_io, const void* code, const void* data, const void* accum, int traces_on_device) {
  ZKB_API_BEGIN
  ZKB_REQUIRE(p != nullptr, "null prover");
  use(p->ctx);
  ZKB_REQUIRE((h_io || p->circuit.out_size == 0) && (code || p->program || p->circuit.group_size[GROUP_CODE] == 0) &&
              (data || p->circuit.group_size[GROUP_DATA] == 0) && (accum || p->circuit.group_size[GROUP_ACCUM] == 0), "null argument");
  p->segment_begin(po2, h_io, code, data, traces_on_device != 0, nullptr);
  p->segment_finish(accum, traces_on_device != 0);
  ZKB_API_END
}
zkb_err zkb_prover_stage_traces(zkb_prover* p, int po2, const void* h_code, const void* h_data, const void* h_accum) {
  ZKB_API_BEGIN
  ZKB_REQUIRE(p != nullptr, "null prover");
  use(p->ctx);
  const void* tr[3];
  tr[GROUP_ACCUM] = h_accum; tr[GROUP_CODE] = h_code; tr[GROUP_DATA] = h_data;
  for (int g = 0; g < 3; ++g) ZKB_REQUIRE(tr[g] || p->circuit.group_size[g] == 0 || (g == GROUP_ACCUM && !p->circuit.wsteps.empty()) || (g == GROUP_CODE && p->program),
                                          g == GROUP_ACCUM ? "null accum trace and the circuit blob carries no witness program to compute it" : "null trace");
  p->stage_traces(po2, tr);
  ZKB_API_END
}
zkb_err zkb_prover_stage_wait(zkb_prover* p) {
  ZKB_API_BEGIN
  ZKB_REQUIRE(p != nullptr, "null prover");
  use(p->ctx);
  if (p->copy_stream) ZKB_CUDA(cudaStreamSynchronize(p->copy_stream));
  ZKB_API_END
}
zkb_err zkb_prove_staged(zkb_prover* p, const uint32_t* h_io) {
  ZKB_API_BEGIN
  ZKB_REQUIRE(p != nullptr, "null prover");
  use(p->ctx);
  ZKB_REQUIRE(h_io || p->circuit.out_size == 0, "null io");
  p->prove_staged(h_io);
  ZKB_API_END
}
zkb_err zkb_prover_seal_words(zkb_prover* p, size_t* out) {
  ZKB_API_BEGIN
  ZKB_REQUIRE(p && out, "null argument");
  *out = p->iop->proof.size();
  ZKB_API_END
}
zkb_err zkb_prover_seal_copy(zkb_prover* p, uint32_t* h_out) {
  ZKB_API_BEGIN
  ZKB_REQUIRE(p && h_out, "null argument");
  memcpy(h_out, p->iop->proof.data(), p->iop->proof.size() * 4);
  ZKB_API_END
}
zkb_err zkb_prover_root_count(zkb_prover* p, size_t* out) {
  ZKB_API_BEGIN
  ZKB_REQUIRE(p && out, "null argument");
  *out = p->roots.size();
  ZKB_API_END
}
zkb_err zkb_prover_roots_copy(zkb_prover* p, uint32_t* h_out) {
  ZKB_API_BEGIN
  ZKB_REQUIRE(p && h_out, "null argument");
  memcpy(h_out, p->roots.data(), p->roots.size() * 32);
  ZKB_API_END
}

}  // extern "C"
