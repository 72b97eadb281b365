// Internal (C++) entry points of the kernels, shared between translation units; the C-ABI wrappers and the prover
// both go through these.
#pragma once
#include "common.cuh"
#include "circuit.hpp"

namespace zkb {

// k_ntt.cu
// src (optional, device): read the evaluations from src instead of io (out of place; src is left untouched)
void ntt_inverse(zkb_ctx* ctx, uint32_t* io, size_t count, int k, bool zk_shift, const uint32_t* src = nullptr);
void ntt_forward(zkb_ctx* ctx, uint32_t* out, const uint32_t* in, size_t count, int k_out, int expand_bits);
// k_poseidon2.cu
void hash_rows(zkb_ctx* ctx, uint32_t* out, const uint32_t* matrix, size_t rows, size_t cols);
void hash_fold(zkb_ctx* ctx, uint32_t* nodes, size_t input_size, size_t output_size);
void merkle_build(zkb_ctx* ctx, uint32_t* nodes, size_t rows);
// k_poly.cu
void eltwise_add(zkb_ctx* ctx, uint32_t* o, const uint32_t* a, const uint32_t* b, size_t n);
void eltwise_zeroize(zkb_ctx* ctx, uint32_t* x, size_t n);
void fill_u32(zkb_ctx* ctx, uint32_t* x, size_t n, uint32_t v);
void gather_sample(zkb_ctx* ctx, uint32_t* dst, const uint32_t* src, size_t idx, size_t size, size_t stride);
void batch_expand(zkb_ctx* ctx, uint32_t* out, const uint32_t* in, size_t count, int in_po2, int expand_bits);
void batch_bit_reverse(zkb_ctx* ctx, uint32_t* io, size_t count, int po2);
void batch_bit_reverse_ext(zkb_ctx* ctx, uint32_t* io, size_t count, int po2);      // arrays of Fp4 (16-byte) elements
void zk_shift(zkb_ctx* ctx, uint32_t* io, size_t count, int po2);
void eltwise_sum_extelem(zkb_ctx* ctx, uint32_t* out, const uint32_t* in, size_t count, size_t to_add);
void fri_fold(zkb_ctx* ctx, uint32_t* out, const uint32_t* in, const Fp4& mix, size_t m);
void mix_poly_coeffs(zkb_ctx* ctx, uint32_t* out, const Fp4& mix_start, const Fp4& mix, const uint32_t* in, const uint32_t* d_combos,
                     size_t input_size, size_t count, uint32_t n_combo_slots);
// coeffs_bit_reversed: the columns hold their coefficients in bit-reversed order (as the iNTT leaves them); same results
void batch_evaluate_any(zkb_ctx* ctx, const uint32_t* coeffs, int po2, const uint32_t* d_which, const uint32_t* d_xs, uint32_t* d_out, size_t n_eval,
                        bool coeffs_bit_reversed = false);
void poly_divide(zkb_ctx* ctx, uint32_t* d_poly, size_t n, const Fp4& z, uint32_t* d_rem);
void prefix_products(zkb_ctx* ctx, uint32_t* d_io, size_t n);
// true if the n words at a and b are all equal: one device pass, one 4-byte read-back (synchronises the stream)
bool words_equal(zkb_ctx* ctx, const uint32_t* a, const uint32_t* b, size_t n);
// CircuitHal::accumulate: the circuit blob's witness program, phase by phase (k_accum.cu)
void accumulate(zkb_ctx* ctx, const CircuitDef& c, uint32_t* d_accum, const uint32_t* d_code, const uint32_t* d_data, const uint32_t* h_mix, const uint32_t* h_io, int po2);
// k_eval_check.cu
void eval_check(zkb_ctx* ctx, uint32_t* d_check, const CircuitDef& c, const uint32_t* const d_groups[3], const uint32_t* mix_g, const uint32_t* out_g,
                const Fp4& poly_mix, int po2);
// k_query.cu
struct QueryTree { const uint32_t* matrix; const uint32_t* nodes; uint32_t rows, cols, top_size, path_len, out_offset; };
void gather_queries(zkb_ctx* ctx, uint32_t* d_out, uint32_t words_per_query, const QueryTree& tree, const uint32_t* d_idx, uint32_t n_queries);
void sub_small(zkb_ctx* ctx, uint32_t* d_fp4_dst, size_t stride_fp4, const uint32_t* d_deltas, uint32_t rows, uint32_t per_row);

}  // namespace zkb
