/* zkb200.h -- C ABI of libzkb200.so, the B200-native (sm_100a) STARK proving backend for the
 * `zktls prove -p r0` hot path.
 *
 * What this boundary replaces.  The reference reaches the prover through one call,
 * `risc0_zkvm::default_prover().prove_with_opts(..)` (/root/reference/crates/guest-prover-r0/src/prover.rs:79,90);
 * inside the pinned, un-vendored crates (risc0-zkp / risc0-core / risc0-sys 1.2.5, sppark 0.1.11 --
 * /root/reference/Cargo.lock:5057-5085, 5008-5017, 5045-5054, 6223-6230) the data-parallel work is done
 * through the risc0_zkp `Hal` / `CircuitHal` traits (risc0-zkp/src/hal/mod.rs), whose CUDA
 * implementation binds C functions `risc0_zkp_cuda_*` / `sppark_*` over FFI.  Each operator below names the
 * `Hal` method it stands in for; SURVEY.md App. C gives the exact semantics.
 *
 * Conventions (identical to risc0-sys so a Rust shim can reuse `ffi_wrap` verbatim):
 *   - every function returns `const char*`: NULL on success, otherwise a malloc'd NUL-terminated message that
 *     the caller releases with zkb_free_error() (plain free()).  Nothing unwinds or aborts across the ABI.
 *   - pointers named d_* / `void*` buffers are DEVICE pointers (from zkb_alloc, or any CUDA allocation on the
 *     ctx's device, 16-byte aligned); h_* are host pointers.  A sub-buffer is pointer + offset on the caller side.
 *   - Fp = one u32 Montgomery word (canonical, < P = 2013265921); Fp4 = 4 consecutive words; Digest = 8 words;
 *     matrices are column-major: column c of a (cols x rows) matrix is words [c*rows, (c+1)*rows).
 *   - operators are stream-ordered and asynchronous on the ctx stream; only zkb_d2h, zkb_sync, zkb_timer_stop and
 *     the prover calls block.  A ctx is bound to one device and driven by one host thread at a time (the Hal is
 *     !Send in the reference); several ctxs per process / per GPU are independent.
 *   - there is no CPU fallback: without a CUDA device zkb_init fails and nothing else is callable.
 */
#ifndef ZKB200_H
#define ZKB200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct zkb_ctx zkb_ctx;
typedef struct zkb_prover zkb_prover;
typedef struct zkb_program zkb_program;
typedef const char* zkb_err;

/* ---- lifecycle -------------------------------------------------------------------------------------- */
const char* zkb_version(void);
void zkb_free_error(const char* err);
zkb_err zkb_init(int device, zkb_ctx** out);                       /* owns a new non-blocking stream */
zkb_err zkb_init_on_stream(int device, void* cuda_stream, zkb_ctx** out);   /* borrows the caller's cudaStream_t */
zkb_err zkb_destroy(zkb_ctx* ctx);
zkb_err zkb_sync(zkb_ctx* ctx);
zkb_err zkb_device_info(zkb_ctx* ctx, int* sm_count, int* cc_major, int* cc_minor, size_t* total_mem);
/* CUDA devices visible to this process (segments are sharded over them, one ctx per device and worker: no ctx needed) */
zkb_err zkb_device_count(int* out);
/* number of kernels this ctx has launched so far (bench.py's `gpu_launches`) */
zkb_err zkb_kernel_launches(zkb_ctx* ctx, uint64_t* out);
/* CUDA-event timer on the ctx stream (the stream the kernels are launched on) */
zkb_err zkb_timer_start(zkb_ctx* ctx);
zkb_err zkb_timer_stop(zkb_ctx* ctx, float* ms);

/* ---- memory: Hal::{alloc_*, copy_from_*}, Buffer::{view, view_mut, get_at, to_vec} ----------------------- */
zkb_err zkb_alloc(zkb_ctx* ctx, size_t bytes, void** d_out);
zkb_err zkb_free(zkb_ctx* ctx, void* d_ptr);
zkb_err zkb_host_alloc(zkb_ctx* ctx, size_t bytes, void** h_out);     /* pinned host memory */
zkb_err zkb_host_free(zkb_ctx* ctx, void* h_ptr);
zkb_err zkb_memset0(zkb_ctx* ctx, void* d_ptr, size_t bytes);
zkb_err zkb_fill_u32(zkb_ctx* ctx, void* d_ptr, size_t n, uint32_t value);
zkb_err zkb_h2d(zkb_ctx* ctx, void* d_dst, const void* h_src, size_t bytes);   /* async if h_src is pinned */
zkb_err zkb_d2h(zkb_ctx* ctx, void* h_dst, const void* d_src, size_t bytes);   /* blocks until complete */
zkb_err zkb_d2d(zkb_ctx* ctx, void* d_dst, const void* d_src, size_t bytes);

/* ---- NTT family --------------------------------------------------------------------------------------- */
/* Hal::batch_interpolate_ntt(io, count): per column inverse NTT, natural-order evaluations -> bit-reversed
 * coefficients, scaled by 1/2^po2.  io: count x 2^po2. */
zkb_err zkb_batch_interpolate_ntt(zkb_ctx* ctx, void* d_io, size_t count, int po2);
/* Hal::zk_shift(io, count): io[c][i] *= 3^bitrev(i). */
zkb_err zkb_zk_shift(zkb_ctx* ctx, void* d_io, size_t count, int po2);
/* fused batch_interpolate_ntt + zk_shift (what Prover::commit_group's make_coeffs does back to back) */
zkb_err zkb_batch_interpolate_ntt_zk_shift(zkb_ctx* ctx, void* d_io, size_t count, int po2);
/* Hal::batch_expand(out, in, count): out[c][i] = in[c][i >> expand_bits]. */
zkb_err zkb_batch_expand(zkb_ctx* ctx, void* d_out, const void* d_in, size_t count, int in_po2, int expand_bits);
/* Hal::batch_evaluate_ntt(io, count, expand_bits): forward NTT skipping the first expand_bits levels,
 * bit-reversed in -> natural out.  io: count x 2^po2. */
zkb_err zkb_batch_evaluate_ntt(zkb_ctx* ctx, void* d_io, size_t count, int po2, int expand_bits);
/* Hal::batch_expand_into_evaluate_ntt(out, in, count, expand_bits): the LDE.  in: count x 2^in_po2 bit-reversed
 * coefficients; out: count x 2^(in_po2+expand_bits) natural-order evaluations. */
zkb_err zkb_batch_expand_into_evaluate_ntt(zkb_ctx* ctx, void* d_out, const void* d_in, size_t count, int in_po2, int expand_bits);
/* Hal::batch_bit_reverse(io, count). */
zkb_err zkb_batch_bit_reverse(zkb_ctx* ctx, void* d_io, size_t count, int po2);

/* ---- Poseidon2 hashing / Merkle ------------------------------------------------------------------------ */
/* Hal::hash_rows(out, matrix): out[r] = hash_elem_slice(row r of the column-major cols x rows matrix). */
zkb_err zkb_poseidon2_hash_rows(zkb_ctx* ctx, void* d_out_digests, const void* d_matrix, size_t rows, size_t cols);
/* Hal::hash_fold(io, input_size, output_size): io[output_size+i] = hash_pair(io[input_size+2i], io[input_size+2i+1]). */
zkb_err zkb_poseidon2_hash_fold(zkb_ctx* ctx, void* d_nodes, size_t input_size, size_t output_size);
/* all levels of MerkleTreeProver::new after hash_rows: nodes is the heap-indexed array of 2*rows digests with the
 * leaves already at [rows, 2*rows); fills [1, rows). */
zkb_err zkb_poseidon2_merkle_build(zkb_ctx* ctx, void* d_nodes, size_t rows);

/* ---- polynomial mixing / DEEP / FRI ---------------------------------------------------------------------- */
/* Hal::batch_evaluate_any(coeffs, poly_count, which, xs, out): out[j] = sum_i coeffs[which[j]][i] * xs[j]^i.
 * d_which: n_eval u32; d_xs / d_out: n_eval Fp4. */
zkb_err zkb_batch_evaluate_any(zkb_ctx* ctx, const void* d_coeffs, size_t poly_count, int po2, const void* d_which,
                               const void* d_xs, void* d_out, size_t n_eval);
/* Hal::mix_poly_coeffs(out, mix_start, mix, in, combos, input_size, count):
 * out[combos[i]*count + idx] += mix_start * mix^i * in[i*count + idx].  h_mix_start/h_mix: 4 host words each;
 * d_combos: input_size u32 on the device. */
zkb_err zkb_mix_poly_coeffs(zkb_ctx* ctx, void* d_out, const uint32_t* h_mix_start, const uint32_t* h_mix, const void* d_in,
                            const void* d_combos, size_t input_size, size_t count);
/* Device version of the host step in Prover::finalize (core/poly.rs poly_divide): synthetic division of the
 * Fp4 polynomial d_poly[0..n) by (x - z) in place; writes the remainder (4 words) to d_rem. */
zkb_err zkb_poly_divide(zkb_ctx* ctx, void* d_poly, size_t n, const uint32_t* h_z, void* d_rem);
/* The whole division step of Prover::finalize (SURVEY.md 8b `zkb_combos_divide`): d_combos holds n_combos Fp4 polynomials of n
 * coefficients each; division k < n_div divides polynomial h_combo[k] by (x - h_points[4k..4k+4)) in place, in the order given;
 * the n_div remainders (4 words each) are written to h_rem after one synchronisation. */
zkb_err zkb_combos_divide(zkb_ctx* ctx, void* d_combos, size_t n, size_t n_combos, const uint32_t* h_combo, const uint32_t* h_points,
                          size_t n_div, uint32_t* h_rem);
/* Hal::eltwise_sum_extelem(out, in): out[j*count+idx] = (sum_k in[k*count+idx])[j]. */
zkb_err zkb_eltwise_sum_extelem(zkb_ctx* ctx, void* d_out, const void* d_in, size_t count, size_t to_add);
/* Hal::fri_fold(out, in, mix): out_count = out.len/4; in.len = 64*out_count. */
zkb_err zkb_fri_fold(zkb_ctx* ctx, void* d_out, const void* d_in, const uint32_t* h_mix, size_t out_count);
/* Hal::eltwise_{add,copy,zeroize}_elem, gather_sample, prefix_products. */
zkb_err zkb_eltwise_add_elem(zkb_ctx* ctx, void* d_out, const void* d_a, const void* d_b, size_t n);
zkb_err zkb_eltwise_copy_elem(zkb_ctx* ctx, void* d_out, const void* d_in, size_t n);
zkb_err zkb_eltwise_zeroize_elem(zkb_ctx* ctx, void* d_io, size_t n);
zkb_err zkb_gather_sample(zkb_ctx* ctx, void* d_dst, const void* d_src, size_t idx, size_t size, size_t stride);
/* Batched gather_sample (SURVEY.md 8b "+ batched zkb_gather_rows"): the query phase of MerkleTreeProver::prove / fri_prove reads one
 * row per query; row q of dst (size elements) = gather_sample(src, h_idx[q], size, stride), all n_idx <= 65535 rows in one launch
 * instead of n_idx launches.  src_len = elements in src (every row is bounds-checked against it); h_idx is a host slice. */
zkb_err zkb_gather_rows(zkb_ctx* ctx, void* d_dst, const void* d_src, size_t src_len, const uint32_t* h_idx, size_t n_idx, size_t size, size_t stride);
zkb_err zkb_prefix_products(zkb_ctx* ctx, void* d_io_fp4, size_t n);
/* Hal::scatter(into, index, offsets, values) (witness-generation helper): for every row r < n_rows and k in
 * [h_index[r], h_index[r+1]): into[h_offsets[k]] = h_values[k].  index/offsets/values are host slices as in the trait;
 * an offset >= into_len is an error. */
zkb_err zkb_scatter(zkb_ctx* ctx, void* d_into, size_t into_len, const uint32_t* h_index, size_t n_rows, const uint32_t* h_offsets,
                    const uint32_t* h_values);

/* ---- CircuitHal::eval_check ------------------------------------------------------------------------------- */
/* check[j*4n + c] = (poly_fp(c) / ((3 w^c)^n - 1))[j] over the LDE domain (4n points).  The constraint system is
 * data: h_circuit is the circuit blob (TapSet + PolyExtStep program; layout in DESIGN.md).  d_accum/d_code/d_data
 * are the groups' evaluated matrices (cols x 4n); h_mix_g/h_out_g the globals; h_poly_mix 4 words. */
zkb_err zkb_eval_check(zkb_ctx* ctx, void* d_check, const uint32_t* h_circuit, size_t circuit_words, const void* d_accum,
                       const void* d_code, const void* d_data, const uint32_t* h_mix_g, const uint32_t* h_out_g,
                       const uint32_t* h_poly_mix, int po2);

/* The specialised (JIT-compiled) form of eval_check for a circuit: its generated source (host-only; writes up to cap bytes
 * NUL-terminated, full length to *needed) -- CUDA C++ for ordinary circuits, a CUDA C++ tile kernel + PTX unit functions for
 * heavy ones (>= 2000 constraints: the "flat" form, linked with nvJitLink) -- and an ahead-of-time compile into the on-disk cubin
 * cache: ZKB_CACHE_DIR, else `_jitcache/` next to the library, else $XDG_CACHE_HOME/zkb200 or ~/.cache/zkb200 (0700); directories
 * and files must be owned by the user (or root) and not group/world-writable; never a shared /tmp path.  The counterpart of the
 * reference compiling its generated poly_fp at crate build time. */
zkb_err zkb_eval_check_source(const uint32_t* h_circuit, size_t circuit_words, char* out, size_t cap, size_t* needed);
zkb_err zkb_eval_check_precompile(const uint32_t* h_circuit, size_t circuit_words);
/* CircuitHal::accumulate(ctrl, io, data, mix, accum, steps) (risc0-circuit-rv32im `prove/hal/{cpu,cuda}.rs`, run by
 * prove_segment between the data commit and the accum commit; in-tree call site crates/guest-prover-r0/src/prover.rs:90):
 * fills the accum group's columns on the device from the code (= ctrl) and data traces, the `mix` globals that
 * zkb_prover_segment_begin returned, and io.  Rows / columns the circuit's witness program does not write keep the caller's
 * contents.  The witness program is DATA: the `n_wsteps` section of the circuit blob (W_CONST .. W_PREFIX_PRODUCT, DESIGN.md 5),
 * JIT-compiled per phase; a circuit whose blob carries no witness program gets an error string. */
zkb_err zkb_accumulate(zkb_ctx* ctx, const uint32_t* h_circuit, size_t circuit_words, void* d_accum, const void* d_code,
                       const void* d_data, const uint32_t* h_mix, const uint32_t* h_io, int po2);

/* ---- Prover: risc0-zkp prove::Prover + the circuit's prove_segment driver (SURVEY.md App. D) ------------------ */
zkb_err zkb_prover_new(zkb_ctx* ctx, const uint32_t* h_circuit, size_t circuit_words, zkb_prover** out);
zkb_err zkb_prover_free(zkb_prover* p);
/* First half of prove_segment: transcript header, commit_group(code), commit_group(data), then draws the circuit's
 * `mix` globals (written to h_mix_out, mix_size words).  code/data: group_size x 2^po2 column-major trace
 * evaluations; `*_on_device` says whether the pointer is a device or a (preferably pinned) host pointer.  The
 * trace buffers are not modified.  code == NULL with a program attached (zkb_prover_set_program): the program's
 * commitment at po2 is the code group, as in zkb_prove_segment and zkb_prover_stage_traces. */
zkb_err zkb_prover_segment_begin(zkb_prover* p, int po2, const uint32_t* h_io, const void* code, const void* data,
                                 int traces_on_device, uint32_t* h_mix_out);
/* Second half: commit_group(accum), finalize (eval_check, DEEP, FRI, queries).  The seal is then available. */
zkb_err zkb_prover_segment_finish(zkb_prover* p, const void* accum, int trace_on_device);
zkb_err zkb_prover_seal_words(zkb_prover* p, size_t* out);
zkb_err zkb_prover_seal_copy(zkb_prover* p, uint32_t* h_out);
/* Merkle roots in commit order (code, data, accum, check, FRI rounds...), 8 words each */
zkb_err zkb_prover_root_count(zkb_prover* p, size_t* out);
zkb_err zkb_prover_roots_copy(zkb_prover* p, uint32_t* h_out);
/* One-shot convenience over the two calls above for traces whose accum group does not depend on `mix`. */
zkb_err zkb_prove_segment(zkb_prover* p, int po2, const uint32_t* h_io, const void* code, const void* data, const void* accum,
                          int traces_on_device);
/* Pipelined form for a queue of segments (the continuation segments of one session): zkb_prover_stage_traces starts the
 * host->device copy of a segment's three trace groups (pinned host memory recommended) on a separate copy stream into one of
 * two staging slots and returns at once; zkb_prove_staged proves the oldest staged segment (as zkb_prove_segment does).
 * Staging segment k+1 before proving segment k overlaps its upload with the proof.  At most two segments may be staged.
 * h_accum may be NULL when the circuit blob carries a witness program: zkb_prove_staged then runs CircuitHal::accumulate on
 * the device between the data commit and the accum commit (prove_segment's order), and the accum group is never uploaded. */
zkb_err zkb_prover_stage_traces(zkb_prover* p, int po2, const void* h_code, const void* h_data, const void* h_accum);
zkb_err zkb_prove_staged(zkb_prover* p, const uint32_t* h_io);
/* Blocks until every upload started by zkb_prover_stage_traces on this prover has landed (lets several provers that share
 * one PCIe link take turns instead of splitting its bandwidth).  It only synchronises the prover's copy stream, so -- unlike
 * every other call on a prover -- it may run on another host thread while zkb_prove_staged is in progress. */
zkb_err zkb_prover_stage_wait(zkb_prover* p);

/* ---- Program: a circuit's code commitments, made once per device and po2 ------------------------------------------------------
 * The code trace is the program: zkb_verify_segment accepts a seal only if (po2, code root) is one of the circuit's control IDs.
 * A program commits the code trace once per po2 on the device and holds the commitment read-only (trace copy, coefficients,
 * LDE matrix, Merkle tree: ~640 MB at po2 20, ~10 GB at po2 24); any number of provers on that device prove segments from it
 * given only their data and accum traces.
 *
 * With a program attached, a NULL code argument to zkb_prover_segment_begin, zkb_prove_segment or zkb_prover_stage_traces means
 * "the program's commitment at this po2".  The transcript is the one commit_group(code) writes (top layer written, root mixed,
 * root recorded), so seal and roots equal those the same segment gives when its code trace is passed.  On the staged path with
 * h_accum == NULL the witness program reads the program's copy of the code trace: only data (or data and accum) is uploaded.  A po2
 * the program has not committed is an error string naming it, returned before the transcript is touched or any device work
 * starts (in zkb_prover_stage_traces too); the prover stays usable.  A non-NULL code argument takes the trace path unchanged,
 * including the prover's own retained code commitment, which a segment proven from the program neither reads nor changes.
 *
 * Sharing and lifetime.  Entries are immutable once zkb_program_commit returns: provers on other ctxs and streams of the device
 * read them with no further synchronisation, and provers driven from different host threads may share one program (a commit of a
 * new po2 may run while they prove from existing entries).  Ownership is shared: the caller's handle and every prover holding the
 * program keep it alive, and its memory goes when the last of them lets go.  A prover lets go by detaching, by attaching another
 * program, or by zkb_prover_free; it synchronises its stream first, so no read of the entries is outstanding.  The storage lives on
 * a private stream and memory pool of the device, so it does not depend on the ctx passed to zkb_program_new. */
/* ctx names the device only: the program does not keep the ctx, and it may outlive it. */
zkb_err zkb_program_new(zkb_ctx* ctx, const uint32_t* h_circuit, size_t circuit_words, zkb_program** out);
/* Commits the code trace at po2 on the device: iNTT + zk_shift, x4 LDE, hash_rows, Merkle build.  This is exactly what
 * commit_group(code) computes.  Blocks until the commitment is complete.  Writes the control ID (po2, code root[8]) to
 * h_control_id (9 words).  A po2 that is already committed is an error: entries are immutable.  code: code_cols x 2^po2 words,
 * a device pointer (its contents complete before the call) when code_on_device, else a host pointer; it is not kept. */
zkb_err zkb_program_commit(zkb_program* prog, int po2, const void* code, int code_on_device, uint32_t* h_control_id);
/* The table zkb_verify_segment takes: *n entries of 9 words, ascending po2.  h_out == NULL only queries *n; otherwise *n is h_out's
 * capacity in entries on input (an error if smaller than the table) and the number written on return. */
zkb_err zkb_program_control_ids(zkb_program* prog, size_t* n, uint32_t* h_out);
zkb_err zkb_program_free(zkb_program* prog);   /* releases the caller's handle; provers holding the program keep it alive */
/* Attaches prog to p (NULL detaches).  The circuit blobs must be equal word for word, and both must be on the same device.
 * A segment begun from the program keeps it alive until the prover's next segment or zkb_prover_free. */
zkb_err zkb_prover_set_program(zkb_prover* p, zkb_program* prog);

/* ---- Session: the continuation segments of one session, proven on every device of the process ------------------------------------
 * A session owns `inflight` worker threads per device, each with its own ctx and staged prover, and one program per device.  The caller
 * commits the code trace once per po2, submits (po2, io, data[, accum]) per segment and collects seals by ticket; no per-device code
 * and no threads of its own.  One queue serves every device, so a session's tail is one segment, not one round.  A worker stages its
 * next segment while it proves the current one (zkb_prover_stage_traces / zkb_prove_staged, code from the program).  Within a device,
 * uploads enter the shared copy stream in the order their segments leave the queue, and a worker does not prefetch a second segment
 * while the queue is non-empty and another worker of its device has nothing staged (DESIGN.md section 6).  Device memory per device:
 * inflight x (segment working set + 2 staging slots without the code group) + the program.  submit, wait and commit may be called from
 * any host thread, concurrently; zkb_session_free must be the last call on a session. */
typedef struct zkb_session zkb_session;
/* devices == NULL: every visible device.  inflight: provers per device (1..8).  Starts inflight worker threads per device; each
 * creates its own ctx and prover on its own thread (a ctx is driven by one host thread).  On an error nothing stays running. */
zkb_err zkb_session_new(const uint32_t* h_circuit, size_t circuit_words, const int* devices, size_t n_devices, int inflight,
                        zkb_session** out);
/* Commits the code trace (host pointer) at po2 on every device of the session, in parallel, and writes the control ID (9 words).
 * The per-device roots must agree: a mismatch is an error.  A po2 already committed is an error. */
zkb_err zkb_session_commit(zkb_session* s, int po2, const void* h_code, uint32_t* h_control_id);
zkb_err zkb_session_control_ids(zkb_session* s, size_t* n, uint32_t* h_out);    /* same convention as zkb_program_control_ids */
/* Queues one segment; returns at once with a ticket (increasing in submit order).  h_io is copied.  h_data / h_accum (pinned
 * recommended; pageable works) must stay alive and unmodified until the ticket's seal has been collected or the session is freed.
 * h_accum == NULL: the circuit's witness program computes the accum group on the device.  Refused here, with nothing queued,
 * for: a po2 that has not been committed (named in the message), NULL data with data_cols > 0, NULL accum with no witness program
 * in the blob, or a session being freed.  A segment that fails later (e.g. an io word >= P) fails its own ticket only. */
zkb_err zkb_session_submit(zkb_session* s, int po2, const uint32_t* h_io, const void* h_data, const void* h_accum, uint64_t* ticket);
/* Blocks until the ticket's segment is proven.  h_seal == NULL: writes the seal length to *words and keeps the result.
 * Otherwise *words is h_seal's capacity on input (an error if smaller than the seal); copies the seal, sets *words, releases the
 * ticket.  A segment that failed returns its own error string, once, and the ticket is released.  Unknown or released
 * ticket: error. */
zkb_err zkb_session_wait(zkb_session* s, uint64_t ticket, uint32_t* h_seal, size_t* words);
/* Stops accepting segments.  Segments whose proof has not started (queued, or staged ahead on a worker) fail with "session freed".
 * Waits for the proofs in progress and for the threads inside zkb_session_wait, joins every worker thread, then frees the provers,
 * programs and ctxs. */
zkb_err zkb_session_free(zkb_session* s);

/* CPU verifier for a seal produced by the prover (risc0-zkp verify/*): checks the transcript, Merkle paths, FRI
 * and the constraint relation at the DEEP point.  Host-only, like the reference's verifier.
 * The code group's Merkle root identifies the PROGRAM (risc0: `check_code(po2, root)` against the control ID): it must equal
 * one of the `n_control_ids` entries of `h_control_ids` (9 words each: po2, code root[8]).  With n_control_ids == 0 the call
 * is refused unless `h_out_po2_code_root` (9 words, optional otherwise) is given: the caller then receives (po2, code root)
 * and MUST compare them itself -- a seal whose code trace the prover chose freely proves nothing. */
zkb_err zkb_verify_segment(const uint32_t* h_circuit, size_t circuit_words, const uint32_t* h_seal, size_t seal_words,
                           const uint32_t* h_control_ids, size_t n_control_ids, uint32_t* h_out_po2_code_root);

/* ---- poseidon_254 hash suite (first slice of SURVEY.md 8f-4: the suite identity_p254 / the Groth16 wrapper use) --------------------
 * Poseidon over the BN254 scalar field, t = 3, x^5, R_F = 8, R_P = 57 = circomlib's 2-input `poseidon`; constants regenerated from the
 * reference Grain LFSR and pinned by circomlib's public known answers.  Digests are 8 little-endian u32 words holding the canonical
 * field element.  hash_fold / merkle_build follow risc0's hash_pair (poseidon([0, a, b])[0]); hash_rows uses a PROVISIONAL packing of
 * the row (8 canonical BabyBear values per word in radix 2^31, rate 2, overwrite mode, zero padding) -- upstream's rule is not
 * recoverable offline (zktls_b200/csrc/k_poseidon254.cu). */
zkb_err zkb_poseidon254_hash_rows(zkb_ctx* ctx, void* d_out_digests, const void* d_matrix, size_t rows, size_t cols);
zkb_err zkb_poseidon254_hash_fold(zkb_ctx* ctx, void* d_nodes, size_t input_size, size_t output_size);
zkb_err zkb_poseidon254_merkle_build(zkb_ctx* ctx, void* d_nodes, size_t rows);
/* host-only known-answer hook: one permutation of three canonical field elements (3 x 8 words in, 3 x 8 words out) */
zkb_err zkb_poseidon254_permute_host(const uint32_t* h_in, uint32_t* h_out);

#ifdef __cplusplus
}
#endif
#endif /* ZKB200_H */
