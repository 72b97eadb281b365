// Element-wise, mixing, DEEP and FRI-fold kernels (sm_100a).
//
// Stand-ins for the risc0-zkp `Hal` methods eltwise_{add,copy,zeroize}_elem, eltwise_sum_extelem, fri_fold,
// mix_poly_coeffs, batch_evaluate_any, gather_sample, prefix_products, zk_shift, batch_expand,
// batch_bit_reverse (risc0-sys kernels/zkp/cuda/*.cu in the CudaHal; SURVEY.md 2.3, App. C.2-C.11) and for the
// host-side `poly_divide` step of Prover::finalize (core/poly.rs; App. C.13), which is kept on the device here.
// All are HBM-bound streaming kernels except the DEEP evaluation (4 modmul per coefficient).
#include "common.cuh"

namespace zkb {

struct Fp4Arg { uint32_t w[4]; };
__host__ __device__ inline Fp4 arg4(const Fp4Arg& a) { return Fp4::load(a.w); }
inline Fp4Arg to_arg(const Fp4& x) { Fp4Arg a; x.store(a.w); return a; }
inline Fp4Arg to_arg(const uint32_t* w) { Fp4Arg a; memcpy(a.w, w, 16); return a; }

constexpr int EW_BLOCK = 256;

// Lazy sums of products: a 64-bit accumulator takes unreduced 32 x 32-bit products (one IMAD.WIDE each); after every second
// product its high word is brought back below P, which keeps it below P * 2^32 + 2 P^2 < 2^64; fin_acc does the one
// Montgomery reduction at the end.
__device__ __forceinline__ uint64_t fixhi(uint64_t a) {       // high word < 2P  ->  high word < P (value mod P unchanged)
  uint32_t hi = (uint32_t)(a >> 32);
  uint32_t y = hi - P;
  hi = y < hi ? y : hi;
  return ((uint64_t)hi << 32) | (uint32_t)a;
}
__device__ __forceinline__ uint32_t fin_acc(uint64_t a) { return reduce_2p(mont_redc_lazy(fixhi(a))); }

// ---- trivial element-wise ----------------------------------------------------------------------------
__global__ void k_add(uint32_t* __restrict__ o, const uint32_t* __restrict__ a, const uint32_t* __restrict__ b, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) o[i] = add_mod(a[i], b[i]);
}
__global__ void k_zeroize(uint32_t* __restrict__ x, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && x[i] == INVALID) x[i] = 0;
}
__global__ void k_fill(uint32_t* __restrict__ x, size_t n, uint32_t v) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) x[i] = v;
}
__global__ void k_gather(uint32_t* __restrict__ dst, const uint32_t* __restrict__ src, size_t idx, size_t size, size_t stride) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < size) dst[i] = src[idx + i * stride];
}
// Hal::scatter: into[offsets[k]] = values[k] for k in [k0, k1)
__global__ void k_scatter(uint32_t* __restrict__ into, const uint32_t* __restrict__ offsets, const uint32_t* __restrict__ values, size_t count, size_t into_len, uint32_t* __restrict__ bad) {
  size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= count) return;
  uint32_t o = offsets[k];
  if (o < into_len) into[o] = values[k]; else atomicAdd(bad, 1u);
}
__global__ void k_expand(uint32_t* __restrict__ out, const uint32_t* __restrict__ in, size_t total_out, int expand_bits) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < total_out) out[i] = in[i >> expand_bits];     // columns are contiguous, so this holds across the batch
}
// in-place bit reversal of each column
__global__ void k_bit_reverse(uint32_t* __restrict__ io, int po2, size_t count) {
  size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t n = (size_t)1 << po2;
  if (g >= n * count) return;
  uint32_t i = (uint32_t)(g & (n - 1));
  uint32_t r = bit_rev32(i, po2);
  if (i < r) {
    uint32_t* col = io + (g - i);
    uint32_t a = col[i], b = col[r];
    col[i] = b; col[r] = a;
  }
}
// Tiled in-place bit reversal for po2 >= 2T: write i = (a, m, b) with a the top T bits and b the low T bits; then
// rev(i) = (rev(b), rev(m), rev(a)), so the 2^T x 2^T tile (a, b) of slice m lands, transposed and with both tile
// coordinates bit-reversed, in slice rev(m).  One CTA owns the pair of slices {m, rev(m)}: every global access is a row
// of 2^T consecutive words (128 / 256 bytes) and the permutation itself happens in shared memory.
template <int T, typename E = uint32_t>
__global__ void __launch_bounds__(256) k_bit_reverse_tiled(E* __restrict__ io, int po2) {
  constexpr int W = 1 << T;
  __shared__ E A[W][W + 1], B[W][W + 1];
  const int mid_bits = po2 - 2 * T;
  const uint32_t m = blockIdx.x & ((1u << mid_bits) - 1u);
  const uint32_t rm = bit_rev32(m, mid_bits);
  if (m > rm) return;
  E* base = io + ((size_t)(blockIdx.x >> mid_bits) << po2);
  const int hi_shift = po2 - T;
  const bool pair = m != rm;
  for (uint32_t e = threadIdx.x; e < W * W; e += 256) {
    uint32_t a = e >> T, b = e & (W - 1);
    A[a][b] = base[((size_t)a << hi_shift) | (m << T) | b];
    if (pair) B[a][b] = base[((size_t)a << hi_shift) | (rm << T) | b];
  }
  __syncthreads();
  for (uint32_t e = threadIdx.x; e < W * W; e += 256) {
    uint32_t a = e >> T, b = e & (W - 1);
    uint32_t ra = bit_rev32(a, T), rb = bit_rev32(b, T);
    base[((size_t)a << hi_shift) | (rm << T) | b] = A[rb][ra];
    if (pair) base[((size_t)a << hi_shift) | (m << T) | b] = B[rb][ra];
  }
}
// the same permutation over arrays of 16-byte elements (Fp4 coefficients), small sizes
__global__ void k_bit_reverse_ext(uint4* __restrict__ io, int po2, size_t count) {
  size_t n = (size_t)1 << po2;
  size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n * count) return;
  uint32_t i = (uint32_t)(g & (n - 1));
  uint32_t r = bit_rev32(i, po2);
  if (i < r) {
    uint4* col = io + (g - i);
    uint4 a = col[i], b = col[r];
    col[i] = b; col[r] = a;
  }
}
// io[c][i] *= 3^bitrev(i)
__global__ void k_zk_shift(uint32_t* __restrict__ io, int po2, size_t count) {
  size_t n = (size_t)1 << po2;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Fp s = pow(Fp::from(3), bit_rev32((uint32_t)i, po2));
  for (size_t c = 0; c < count; ++c) io[c * n + i] = mont_mul(io[c * n + i], s.v);
}

// ---- eltwise_sum_extelem / fri_fold ----------------------------------------------------------------------
__global__ void k_sum_extelem(uint32_t* __restrict__ out, const uint4* __restrict__ in, size_t count, size_t to_add) {
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= count) return;
  uint32_t t0 = 0, t1 = 0, t2 = 0, t3 = 0;
  for (size_t k = 0; k < to_add; ++k) {
    uint4 v = in[k * count + idx];
    t0 = add_mod(t0, v.x); t1 = add_mod(t1, v.y); t2 = add_mod(t2, v.z); t3 = add_mod(t3, v.w);
  }
  out[idx] = t0; out[count + idx] = t1; out[2 * count + idx] = t2; out[3 * count + idx] = t3;
}
__global__ void k_fri_fold(uint32_t* __restrict__ out, const uint32_t* __restrict__ in, Fp4Arg mix_arg, size_t m) {
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= m) return;
  Fp4 mix = arg4(mix_arg), tot, cur = Fp4::one();
#pragma unroll 4
  for (uint32_t i = 0; i < 16; ++i) {
    size_t r = (size_t)bit_rev32(i, 4) * m + idx;
    Fp4 v = Fp4::raw(in[r], in[16 * m + r], in[32 * m + r], in[48 * m + r]);
    tot += cur * v;
    cur *= mix;
  }
  out[idx] = tot.c[0].v; out[m + idx] = tot.c[1].v; out[2 * m + idx] = tot.c[2].v; out[3 * m + idx] = tot.c[3].v;
}

// ---- mix_poly_coeffs --------------------------------------------------------------------------------------
// pw[i] = start * mix^i
__global__ void k_mix_powers(uint4* __restrict__ pw, Fp4Arg start, Fp4Arg mix, uint32_t n) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Fp4 r = arg4(start) * pow(arg4(mix), i);
  pw[i] = st4(r);
}
// grid.y = combo id; each thread owns out[combo][idx] and sweeps the columns that map to this combo.  Per chunk of 256 columns warp 0
// compacts the matching column indices into shared memory, so the sweep is branch-free and keeps four coefficient loads in flight
// per thread.  (That alone changed nothing -- see k_mix_poly_coeffs4 below for what did; this form remains for counts that are not a multiple of 4.)
constexpr int MIX_CHUNK = 256;
__global__ void __launch_bounds__(EW_BLOCK) k_mix_poly_coeffs(uint4* __restrict__ out, const uint4* __restrict__ pw, const uint32_t* __restrict__ in,
                                                               const uint32_t* __restrict__ combos, uint32_t input_size, size_t count) {
  __shared__ uint4 s_pw[MIX_CHUNK];
  __shared__ uint32_t s_combo[MIX_CHUNK];
  __shared__ uint16_t s_list[MIX_CHUNK + 4];
  __shared__ uint32_t s_hits;
  const uint32_t combo = blockIdx.y, lane = threadIdx.x & 31;
  size_t idx = (size_t)blockIdx.x * EW_BLOCK + threadIdx.x;
  bool live = idx < count;
  // lazy 64-bit accumulation (see fixhi): one IMAD.WIDE per column and Fp4 component, one high-word fix per two columns
  uint64_t a0 = 0, a1 = 0, a2 = 0, a3 = 0;
  bool any = false;
  for (uint32_t base = 0; base < input_size; base += MIX_CHUNK) {
    uint32_t chunk = min((uint32_t)MIX_CHUNK, input_size - base);
    __syncthreads();
    for (uint32_t t = threadIdx.x; t < chunk; t += EW_BLOCK) { s_pw[t] = pw[base + t]; s_combo[t] = combos[base + t]; }
    __syncthreads();
    if (threadIdx.x < 32) {
      uint32_t cnt = 0;
      for (uint32_t t0 = 0; t0 < chunk; t0 += 32) {
        const uint32_t t = t0 + lane;
        const bool hit = t < chunk && s_combo[t] == combo;
        const uint32_t m = __ballot_sync(0xffffffffu, hit);
        if (hit) s_list[cnt + __popc(m & ((1u << lane) - 1u))] = (uint16_t)t;
        cnt += __popc(m);
      }
      if (lane == 0) s_hits = cnt;
    }
    __syncthreads();
    const uint32_t hits = s_hits;
    if (!live || hits == 0) continue;
    any = true;
    const uint32_t* col0 = in + (size_t)base * count + idx;
    for (uint32_t k = 0; k < hits; k += 4) {
      uint32_t v[4]; uint4 p[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const bool on = k + u < hits;
        const uint32_t t = on ? s_list[k + u] : 0u;
        v[u] = on ? __ldg(col0 + (size_t)t * count) : 0u;        // a zero coefficient adds nothing
        p[u] = s_pw[t];
      }
#pragma unroll
      for (int u = 0; u < 4; u += 2) {
        a0 += (uint64_t)v[u] * p[u].x; a1 += (uint64_t)v[u] * p[u].y; a2 += (uint64_t)v[u] * p[u].z; a3 += (uint64_t)v[u] * p[u].w;
        a0 += (uint64_t)v[u + 1] * p[u + 1].x; a1 += (uint64_t)v[u + 1] * p[u + 1].y; a2 += (uint64_t)v[u + 1] * p[u + 1].z; a3 += (uint64_t)v[u + 1] * p[u + 1].w;
        a0 = fixhi(a0); a1 = fixhi(a1); a2 = fixhi(a2); a3 = fixhi(a3);
      }
    }
  }
  if (live && any) {
    uint4* o = out + (size_t)combo * count + idx;
    uint4 cur = *o;
    Fp4 r = ld4(cur) + Fp4::raw(fin_acc(a0), fin_acc(a1), fin_acc(a2), fin_acc(a3));
    *o = st4(r);
  }
}

// Four consecutive coefficients per thread (one 128-bit load per column, 512 contiguous bytes per warp and column): with one word per
// thread every warp request was a lone 128-byte line 4 MB away from the previous one, and the sweep ran at the random-access rate of
// the HBM (1.9 TB/s): 0.51 -> 0.27 ms for 224 x 2^20 on B200.  Used when count is a multiple of 4 (every power-of-two size above 2).
__global__ void __launch_bounds__(EW_BLOCK) k_mix_poly_coeffs4(uint4* __restrict__ out, const uint4* __restrict__ pw, const uint32_t* __restrict__ in,
                                                                const uint32_t* __restrict__ combos, uint32_t input_size, size_t count) {
  __shared__ uint4 s_pw[MIX_CHUNK];
  __shared__ uint32_t s_combo[MIX_CHUNK];
  __shared__ uint16_t s_list[MIX_CHUNK + 2];
  __shared__ uint32_t s_hits;
  const uint32_t combo = blockIdx.y, lane = threadIdx.x & 31;
  const size_t idx = ((size_t)blockIdx.x * EW_BLOCK + threadIdx.x) * 4;
  const bool live = idx < count;
  uint64_t a[4][4];
#pragma unroll
  for (int r = 0; r < 4; ++r) { a[r][0] = a[r][1] = a[r][2] = a[r][3] = 0; }
  bool any = false;
  for (uint32_t base = 0; base < input_size; base += MIX_CHUNK) {
    uint32_t chunk = min((uint32_t)MIX_CHUNK, input_size - base);
    __syncthreads();
    for (uint32_t t = threadIdx.x; t < chunk; t += EW_BLOCK) { s_pw[t] = pw[base + t]; s_combo[t] = combos[base + t]; }
    __syncthreads();
    if (threadIdx.x < 32) {
      uint32_t cnt = 0;
      for (uint32_t t0 = 0; t0 < chunk; t0 += 32) {
        const uint32_t t = t0 + lane;
        const bool hit = t < chunk && s_combo[t] == combo;
        const uint32_t m = __ballot_sync(0xffffffffu, hit);
        if (hit) s_list[cnt + __popc(m & ((1u << lane) - 1u))] = (uint16_t)t;
        cnt += __popc(m);
      }
      if (lane == 0) s_hits = cnt;
    }
    __syncthreads();
    const uint32_t hits = s_hits;
    if (!live || hits == 0) continue;
    any = true;
    const uint32_t* col0 = in + (size_t)base * count + idx;
    for (uint32_t k = 0; k < hits; k += 2) {
      const bool on1 = k + 1 < hits;
      const uint32_t t0 = s_list[k], t1 = on1 ? s_list[k + 1] : 0u;
      const uint4 v0 = __ldg(reinterpret_cast<const uint4*>(col0 + (size_t)t0 * count));
      const uint4 v1 = on1 ? __ldg(reinterpret_cast<const uint4*>(col0 + (size_t)t1 * count)) : make_uint4(0u, 0u, 0u, 0u);      // a zero coefficient adds nothing
      const uint4 p0 = s_pw[t0], p1 = s_pw[t1];
      const uint32_t c0[4] = {v0.x, v0.y, v0.z, v0.w}, c1[4] = {v1.x, v1.y, v1.z, v1.w};
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        a[r][0] += (uint64_t)c0[r] * p0.x; a[r][1] += (uint64_t)c0[r] * p0.y; a[r][2] += (uint64_t)c0[r] * p0.z; a[r][3] += (uint64_t)c0[r] * p0.w;
        a[r][0] += (uint64_t)c1[r] * p1.x; a[r][1] += (uint64_t)c1[r] * p1.y; a[r][2] += (uint64_t)c1[r] * p1.z; a[r][3] += (uint64_t)c1[r] * p1.w;
        a[r][0] = fixhi(a[r][0]); a[r][1] = fixhi(a[r][1]); a[r][2] = fixhi(a[r][2]); a[r][3] = fixhi(a[r][3]);
      }
    }
  }
  if (live && any) {
    uint4* o = out + (size_t)combo * count + idx;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      uint4 cur = o[r];
      Fp4 v = ld4(cur) + Fp4::raw(fin_acc(a[r][0]), fin_acc(a[r][1]), fin_acc(a[r][2]), fin_acc(a[r][3]));
      o[r] = st4(v);
    }
  }
}

// ---- batch_evaluate_any (DEEP) -------------------------------------------------------------------------
// out[j] = sum_i coeffs[which[j]][i] * x_j^i with Fp coefficients and an Fp4 point.  Write i = slab * SLAB + m * 256 + t
// (t = thread, m = step): thread t of block (slab, j) accumulates sum_m c[..] * (x^256)^m LAZILY -- one IMAD.WIDE per
// coefficient and Fp4 component into a 64-bit accumulator whose high word is brought back below P after every second term
// (see fixhi) -- and only then multiplies by x^t, reduces over the block and scales by x^(slab * SLAB).  All powers come
// from per-point tables built by a small pre-kernel, so the main loop is 4 IMAD.WIDE + 2 fix-ups per coefficient
// (the canonical form costs 4 Montgomery multiplications + 4 modular additions).
// STEPS coefficients per thread: the block epilogue (an Fp4 product by x^t, the block reduction, an Fp4 product by x^(slab base)) costs as
// much multiplier-pipe time as ~45 coefficients, so large launches use 256 steps per thread (0.60 -> 0.535 ms for 448 points x 2^20 on B200),
// small ones 64 (more blocks, less predicated-off work).
constexpr int EVAL_THREADS = 256, EVAL_WARPS = EVAL_THREADS / 32;
// tables per evaluation point j: [x^t, t < 256][x^(256 m), m < steps][x^(slab * slab_size), slab < n_slabs]
__host__ __device__ inline size_t eval_table_stride(uint32_t steps, uint32_t n_slabs) { return (size_t)EVAL_THREADS + steps + n_slabs; }
// brev_po2 > 0: the coefficient array is in BIT-REVERSED order (position p holds the coefficient of x^rev(p), rev over brev_po2 bits).
// A position splits into disjoint bit fields p = t + 256 m + 256 steps slab, and rev(p) is the sum of the reversed fields, so the
// same three tables work with the exponents rev(t), rev(256 m), rev(256 steps slab) -- no data movement.
__global__ void k_eval_tables(uint4* __restrict__ tables, const uint4* __restrict__ xs, uint32_t steps, uint32_t n_slabs, uint32_t n_eval, int brev_po2) {
  const size_t stride = eval_table_stride(steps, n_slabs);
  size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= stride * n_eval) return;
  uint32_t j = (uint32_t)(g / stride), e = (uint32_t)(g % stride);
  uint4 xv = xs[j];
  uint64_t exp = e < EVAL_THREADS ? e : e < EVAL_THREADS + steps ? (uint64_t)(e - EVAL_THREADS) * EVAL_THREADS : (uint64_t)(e - EVAL_THREADS - steps) * EVAL_THREADS * steps;
  if (brev_po2 > 0) exp = (exp >> brev_po2) ? 0 : bit_rev32((uint32_t)exp, brev_po2);      // positions >= n are never read
  Fp4 r = pow(ld4(xv), exp);
  tables[g] = st4(r);
}
// acc + a * b as ONE IMAD.WIDE.  Spelled in PTX because `acc += (uint64_t)c * p` with c = (in range ? load : 0) made the compiler carry c
// as a 64-bit pair with a zero high word and emit a 64 x 32 bit product: an extra IMAD and add per term on the multiplier pipe the kernel
// is bound by (ncu: fmaheavy 79 %).
__device__ __forceinline__ uint64_t mad_wide(uint32_t a, uint32_t b, uint64_t acc) {
  uint64_t d;
  asm("mad.wide.u32 %0, %1, %2, %3;" : "=l"(d) : "r"(a), "r"(b), "l"(acc));
  return d;
}
// FULL: n is a multiple of the slab (every power-of-two n >= 256 * STEPS): no bounds checks in the loop
template <int STEPS, bool FULL>
__global__ void __launch_bounds__(EVAL_THREADS) k_eval_slabs(uint4* __restrict__ partial, const uint32_t* __restrict__ coeffs, size_t n,
                                                              const uint32_t* __restrict__ which, const uint4* __restrict__ tables, uint32_t n_slabs) {
  __shared__ uint4 s_pw[STEPS];
  __shared__ uint4 s_red[EVAL_WARPS];
  constexpr uint32_t SLAB = (uint32_t)EVAL_THREADS * STEPS;
  const uint32_t slab = blockIdx.x, j = blockIdx.y;
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint4* tab = tables + (size_t)j * eval_table_stride(STEPS, n_slabs);
  for (int i = threadIdx.x; i < STEPS; i += EVAL_THREADS) s_pw[i] = tab[EVAL_THREADS + i];
  __syncthreads();
  const uint32_t n32 = (uint32_t)n;                        // n <= 2^26
  const uint32_t base = slab * SLAB + threadIdx.x;
  const uint32_t* col = coeffs + (size_t)which[j] * n + base;
  uint64_t a0 = 0, a1 = 0, a2 = 0, a3 = 0;
#pragma unroll 8
  for (int m = 0; m < STEPS; m += 2) {
    const uint32_t o0 = (uint32_t)m * EVAL_THREADS, o1 = o0 + EVAL_THREADS;
    uint32_t c0, c1;
    if (FULL) { c0 = __ldg(col + o0); c1 = __ldg(col + o1); }
    else { c0 = base + o0 < n32 ? __ldg(col + o0) : 0u; c1 = base + o1 < n32 ? __ldg(col + o1) : 0u; }
    uint4 p0 = s_pw[m], p1 = s_pw[m + 1];
    a0 = mad_wide(c0, p0.x, a0); a1 = mad_wide(c0, p0.y, a1); a2 = mad_wide(c0, p0.z, a2); a3 = mad_wide(c0, p0.w, a3);
    a0 = mad_wide(c1, p1.x, a0); a1 = mad_wide(c1, p1.y, a1); a2 = mad_wide(c1, p1.z, a2); a3 = mad_wide(c1, p1.w, a3);
    a0 = fixhi(a0); a1 = fixhi(a1); a2 = fixhi(a2); a3 = fixhi(a3);
  }
  Fp4 acc = Fp4::raw(fin_acc(a0), fin_acc(a1), fin_acc(a2), fin_acc(a3));
  uint4 xt = tab[threadIdx.x];
  acc *= ld4(xt);
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    Fp4 o = Fp4::raw(__shfl_down_sync(0xffffffffu, acc.c[0].v, off), __shfl_down_sync(0xffffffffu, acc.c[1].v, off),
                     __shfl_down_sync(0xffffffffu, acc.c[2].v, off), __shfl_down_sync(0xffffffffu, acc.c[3].v, off));
    acc += o;
  }
  if (lane == 0) s_red[warp] = st4(acc);
  __syncthreads();
  if (threadIdx.x == 0) {
    Fp4 t;
    for (int w = 0; w < EVAL_WARPS; ++w) { uint4 v = s_red[w]; t += ld4(v); }
    uint4 xs = tab[EVAL_THREADS + STEPS + slab];
    t *= ld4(xs);
    partial[(size_t)j * n_slabs + slab] = st4(t);
  }
}
__global__ void k_eval_reduce(uint4* __restrict__ out, const uint4* __restrict__ partial, uint32_t n_slabs, uint32_t n_eval) {
  uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_eval) return;
  Fp4 t;
  for (uint32_t s = 0; s < n_slabs; ++s) { uint4 v = partial[(size_t)j * n_slabs + s]; t += ld4(v); }
  out[j] = st4(t);
}

// ---- poly_divide (synthetic division by x - z), Fp4 coefficients -----------------------------------------
// Recurrence: next = z*cur + p[i]; p[i] = cur  (i descending).  Parallelised by chunks of DIV_CHUNK: pass 1 computes
// each chunk's Horner total, the totals are divided recursively by (X - z^DIV_CHUNK) -- which yields exactly every
// chunk's carry-in and the global remainder -- and pass 2 replays each chunk from its carry.
constexpr int DIV_CHUNK = 8;      // 8 Fp4 = one 128-byte line per thread; n/8 threads keep the SMs full, 7 levels for n = 2^20
__global__ void __launch_bounds__(128) k_div_totals(uint4* __restrict__ totals, const uint4* __restrict__ p, size_t n, Fp4Arg z_arg) {
  size_t c = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t lo = c * DIV_CHUNK;
  if (lo >= n) return;
  Fp4 z = arg4(z_arg), acc;
  if (lo + DIV_CHUNK <= n) {
    uint4 v[DIV_CHUNK];
#pragma unroll
    for (int k = 0; k < DIV_CHUNK; ++k) v[k] = p[lo + k];
#pragma unroll
    for (int k = DIV_CHUNK - 1; k >= 0; --k) acc = acc * z + ld4(v[k]);
  } else {
    for (size_t i = n; i-- > lo;) { uint4 v = p[i]; acc = acc * z + ld4(v); }
  }
  totals[c] = st4(acc);
}
__global__ void __launch_bounds__(128) k_div_apply(uint4* __restrict__ p, const uint4* __restrict__ carries, size_t n, Fp4Arg z_arg) {
  size_t c = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t lo = c * DIV_CHUNK;
  if (lo >= n) return;
  Fp4 z = arg4(z_arg);
  uint4 cv = carries[c];
  Fp4 cur = ld4(cv);
  if (lo + DIV_CHUNK <= n) {
    uint4 v[DIV_CHUNK];
#pragma unroll
    for (int k = 0; k < DIV_CHUNK; ++k) v[k] = p[lo + k];
#pragma unroll
    for (int k = DIV_CHUNK - 1; k >= 0; --k) {
      Fp4 next = z * cur + ld4(v[k]);
      v[k] = st4(cur);
      cur = next;
    }
#pragma unroll
    for (int k = 0; k < DIV_CHUNK; ++k) p[lo + k] = v[k];
  } else {
    for (size_t i = n; i-- > lo;) {
      uint4 v = p[i];
      Fp4 next = z * cur + ld4(v);
      p[i] = st4(cur);
      cur = next;
    }
  }
}
__global__ void k_div_serial(uint4* __restrict__ p, size_t n, Fp4Arg z_arg, uint4* __restrict__ rem) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  Fp4 z = arg4(z_arg), cur;
  for (size_t i = n; i-- > 0;) {
    uint4 v = p[i];
    Fp4 next = z * cur + ld4(v);
    p[i] = st4(cur);
    cur = next;
  }
  *rem = st4(cur);
}

// ---- prefix_products (Fp4 inclusive product scan) -----------------------------------------------------
constexpr int PP_CHUNK = 64;
__global__ void k_pp_totals(uint4* __restrict__ totals, const uint4* __restrict__ io, size_t n) {
  size_t c = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t lo = c * PP_CHUNK;
  if (lo >= n) return;
  size_t hi = min(lo + (size_t)PP_CHUNK, n);
  Fp4 acc = Fp4::one();
  for (size_t i = lo; i < hi; ++i) { uint4 v = io[i]; acc *= ld4(v); }
  totals[c] = st4(acc);
}
__global__ void k_pp_apply(uint4* __restrict__ io, const uint4* __restrict__ scanned_totals, size_t n) {
  size_t c = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t lo = c * PP_CHUNK;
  if (lo >= n) return;
  size_t hi = min(lo + (size_t)PP_CHUNK, n);
  Fp4 acc = Fp4::one();
  if (c > 0) { uint4 v = scanned_totals[c - 1]; acc = ld4(v); }
  for (size_t i = lo; i < hi; ++i) {
    uint4 v = io[i];
    acc *= ld4(v);
    io[i] = st4(acc);
  }
}
__global__ void k_pp_serial(uint4* __restrict__ io, size_t n) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  Fp4 acc = Fp4::one();
  for (size_t i = 0; i < n; ++i) {
    uint4 v = io[i];
    acc *= ld4(v);
    io[i] = st4(acc);
  }
}

// ---- exact comparison: *differ = 1 if any element differs (V = uint4 when both arrays are 16-byte aligned) ----------------
__device__ __forceinline__ uint32_t bits_xor(uint32_t x, uint32_t y) { return x ^ y; }
__device__ __forceinline__ uint32_t bits_xor(const uint4& x, const uint4& y) { return (x.x ^ y.x) | (x.y ^ y.y) | (x.z ^ y.z) | (x.w ^ y.w); }
template <typename V>
__global__ void __launch_bounds__(EW_BLOCK) k_differ(const V* __restrict__ a, const V* __restrict__ b, size_t count,
                                                     const uint32_t* __restrict__ a_tail, const uint32_t* __restrict__ b_tail, uint32_t tail,
                                                     uint32_t* __restrict__ differ) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t d = i < count ? bits_xor(a[i], b[i]) : 0u;
  if (i < tail) d |= a_tail[i] ^ b_tail[i];
  if (__syncthreads_or(d != 0) && threadIdx.x == 0) *differ = 1u;
}

// ---- host-side launchers (shared with prover.cu) --------------------------------------------------------
void eltwise_add(zkb_ctx* ctx, uint32_t* o, const uint32_t* a, const uint32_t* b, size_t n) {
  if (!n) return;
  k_add<<<grid_for(n, EW_BLOCK), EW_BLOCK, 0, ctx->stream>>>(o, a, b, n); launched(ctx);
}
void eltwise_zeroize(zkb_ctx* ctx, uint32_t* x, size_t n) {
  if (!n) return;
  k_zeroize<<<grid_for(n, EW_BLOCK), EW_BLOCK, 0, ctx->stream>>>(x, n); launched(ctx);
}
void fill_u32(zkb_ctx* ctx, uint32_t* x, size_t n, uint32_t v) {
  if (!n) return;
  k_fill<<<grid_for(n, EW_BLOCK), EW_BLOCK, 0, ctx->stream>>>(x, n, v); launched(ctx);
}
// all queries of one tree in one launch: row q of dst = gather_sample(src, idx[q], size, stride)
__global__ void k_gather_rows(uint32_t* __restrict__ dst, const uint32_t* __restrict__ src, const uint32_t* __restrict__ idx, size_t size, size_t stride) {
  const size_t q = blockIdx.y, base = idx[q];
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < size; i += (size_t)gridDim.x * blockDim.x) dst[q * size + i] = src[base + i * stride];
}
void gather_rows(zkb_ctx* ctx, uint32_t* dst, const uint32_t* src, const uint32_t* d_idx, size_t n_idx, size_t size, size_t stride) {
  if (!size || !n_idx) return;
  dim3 grid((unsigned)std::min<size_t>(grid_for(size, EW_BLOCK), 1024), (unsigned)n_idx);
  k_gather_rows<<<grid, EW_BLOCK, 0, ctx->stream>>>(dst, src, d_idx, size, stride); launched(ctx);
}
void gather_sample(zkb_ctx* ctx, uint32_t* dst, const uint32_t* src, size_t idx, size_t size, size_t stride) {
  if (!size) return;
  k_gather<<<grid_for(size, EW_BLOCK), EW_BLOCK, 0, ctx->stream>>>(dst, src, idx, size, stride); launched(ctx);
}
void batch_expand(zkb_ctx* ctx, uint32_t* out, const uint32_t* in, size_t count, int in_po2, int expand_bits) {
  size_t total = (count << in_po2) << expand_bits;
  if (!total) return;
  k_expand<<<grid_for(total, EW_BLOCK), EW_BLOCK, 0, ctx->stream>>>(out, in, total, expand_bits); launched(ctx);
}
void batch_bit_reverse(zkb_ctx* ctx, uint32_t* io, size_t count, int po2) {
  size_t total = count << po2;
  if (!total || po2 == 0) return;
  if (po2 >= 12 && (count << (po2 - 12)) < (1u << 31)) {
    k_bit_reverse_tiled<6><<<(unsigned)(count << (po2 - 12)), 256, 0, ctx->stream>>>(io, po2); launched(ctx);
    return;
  }
  if (po2 >= 10 && (count << (po2 - 10)) < (1u << 31)) {
    k_bit_reverse_tiled<5><<<(unsigned)(count << (po2 - 10)), 256, 0, ctx->stream>>>(io, po2); launched(ctx);
    return;
  }
  k_bit_reverse<<<grid_for(total, EW_BLOCK), EW_BLOCK, 0, ctx->stream>>>(io, po2, count); launched(ctx);
}
// in-place bit reversal of `count` arrays of 2^po2 Fp4 elements
void batch_bit_reverse_ext(zkb_ctx* ctx, uint32_t* io, size_t count, int po2) {
  size_t total = count << po2;
  if (!total || po2 == 0) return;
  if (po2 >= 10 && (count << (po2 - 10)) < (1u << 31)) k_bit_reverse_tiled<5, uint4><<<(unsigned)(count << (po2 - 10)), 256, 0, ctx->stream>>>((uint4*)io, po2);
  else k_bit_reverse_ext<<<grid_for(total, EW_BLOCK), EW_BLOCK, 0, ctx->stream>>>((uint4*)io, po2, count);
  launched(ctx);
}
void zk_shift(zkb_ctx* ctx, uint32_t* io, size_t count, int po2) {
  size_t n = (size_t)1 << po2;
  if (!count) return;
  k_zk_shift<<<grid_for(n, EW_BLOCK), EW_BLOCK, 0, ctx->stream>>>(io, po2, count); launched(ctx);
}
void eltwise_sum_extelem(zkb_ctx* ctx, uint32_t* out, const uint32_t* in, size_t count, size_t to_add) {
  if (!count) return;
  k_sum_extelem<<<grid_for(count, EW_BLOCK), EW_BLOCK, 0, ctx->stream>>>(out, (const uint4*)in, count, to_add); launched(ctx);
}
void fri_fold(zkb_ctx* ctx, uint32_t* out, const uint32_t* in, const Fp4& mix, size_t m) {
  if (!m) return;
  k_fri_fold<<<grid_for(m, EW_BLOCK), EW_BLOCK, 0, ctx->stream>>>(out, in, to_arg(mix), m); launched(ctx);
}
void mix_poly_coeffs(zkb_ctx* ctx, uint32_t* out, const Fp4& mix_start, const Fp4& mix, const uint32_t* in, const uint32_t* d_combos,
                     size_t input_size, size_t count, uint32_t n_combo_slots) {
  if (!input_size || !count) return;
  uint4* pw = (uint4*)scratch(ctx, input_size * 16);
  k_mix_powers<<<grid_for(input_size, EW_BLOCK), EW_BLOCK, 0, ctx->stream>>>(pw, to_arg(mix_start), to_arg(mix), (uint32_t)input_size); launched(ctx);
  if (count % 4 == 0 && ((uintptr_t)in & 15) == 0) {
    dim3 grid(grid_for(count / 4, EW_BLOCK), n_combo_slots);
    k_mix_poly_coeffs4<<<grid, EW_BLOCK, 0, ctx->stream>>>((uint4*)out, pw, in, d_combos, (uint32_t)input_size, count);
  } else {
    dim3 grid(grid_for(count, EW_BLOCK), n_combo_slots);
    k_mix_poly_coeffs<<<grid, EW_BLOCK, 0, ctx->stream>>>((uint4*)out, pw, in, d_combos, (uint32_t)input_size, count);
  }
  launched(ctx);
}
void batch_evaluate_any(zkb_ctx* ctx, const uint32_t* coeffs, int po2, const uint32_t* d_which, const uint32_t* d_xs, uint32_t* d_out, size_t n_eval, bool coeffs_bit_reversed) {
  if (!n_eval) return;
  size_t n = (size_t)1 << po2;
  static int forced = [] { const char* e = getenv("ZKB_EVAL_STEPS"); return e ? atoi(e) : 0; }();
  // 256 steps only when that still leaves several blocks per SM (16 evaluation points of a 2^20 column: 256 blocks -- too few)
  const uint32_t steps = forced == 64 || forced == 256 ? (uint32_t)forced : (po2 >= 18 && n_eval * (n >> 16) >= 1024 ? 256u : 64u);
  const size_t slab = (size_t)EVAL_THREADS * steps;
  uint32_t n_slabs = (uint32_t)((n + slab - 1) / slab);
  const size_t stride = eval_table_stride(steps, n_slabs);
  uint4* partial = (uint4*)scratch(ctx, (n_eval * n_slabs + n_eval * stride) * 16);
  uint4* tables = partial + n_eval * n_slabs;
  k_eval_tables<<<grid_for(stride * n_eval, 128), 128, 0, ctx->stream>>>(tables, (const uint4*)d_xs, steps, n_slabs, (uint32_t)n_eval, coeffs_bit_reversed ? po2 : 0); launched(ctx);
  for (size_t j0 = 0; j0 < n_eval; j0 += 32768) {      // grid.y limit
    uint32_t nj = (uint32_t)std::min<size_t>(32768, n_eval - j0);
    dim3 grid(n_slabs, nj);
    const bool full = n % slab == 0;
#define ZKB_SLABS(ST, FL) k_eval_slabs<ST, FL><<<grid, EVAL_THREADS, 0, ctx->stream>>>(partial + j0 * n_slabs, coeffs, n, d_which + j0, tables + j0 * stride, n_slabs)
    if (steps == 256) { if (full) ZKB_SLABS(256, true); else ZKB_SLABS(256, false); }
    else { if (full) ZKB_SLABS(64, true); else ZKB_SLABS(64, false); }
#undef ZKB_SLABS
    launched(ctx);
  }
  k_eval_reduce<<<grid_for(n_eval, 128), 128, 0, ctx->stream>>>((uint4*)d_out, partial, n_slabs, (uint32_t)n_eval); launched(ctx);
}
// d_work: caller-provided device scratch of >= 2 * ceil(n / DIV_CHUNK) Fp4 (or nullptr to use a temporary)
void poly_divide(zkb_ctx* ctx, uint32_t* d_poly, size_t n, const Fp4& z, uint32_t* d_rem) {
  if (n <= 64) {
    k_div_serial<<<1, 32, 0, ctx->stream>>>((uint4*)d_poly, n, to_arg(z), (uint4*)d_rem); launched(ctx);
    return;
  }
  size_t chunks = (n + DIV_CHUNK - 1) / DIV_CHUNK;
  uint4* totals = nullptr;
  pool_alloc(ctx, &totals, chunks * 16);
  k_div_totals<<<grid_for(chunks, 128), 128, 0, ctx->stream>>>(totals, (const uint4*)d_poly, n, to_arg(z)); launched(ctx);
  poly_divide(ctx, (uint32_t*)totals, chunks, pow(z, DIV_CHUNK), d_rem);
  k_div_apply<<<grid_for(chunks, 128), 128, 0, ctx->stream>>>((uint4*)d_poly, totals, n, to_arg(z)); launched(ctx);
  pool_free(ctx, totals);
}
void prefix_products(zkb_ctx* ctx, uint32_t* d_io, size_t n) {
  if (n <= 4 * PP_CHUNK) {
    if (n) { k_pp_serial<<<1, 32, 0, ctx->stream>>>((uint4*)d_io, n); launched(ctx); }
    return;
  }
  size_t chunks = (n + PP_CHUNK - 1) / PP_CHUNK;
  uint4* totals = nullptr;
  pool_alloc(ctx, &totals, chunks * 16);
  k_pp_totals<<<grid_for(chunks, 128), 128, 0, ctx->stream>>>(totals, (const uint4*)d_io, n); launched(ctx);
  prefix_products(ctx, (uint32_t*)totals, chunks);
  k_pp_apply<<<grid_for(chunks, 128), 128, 0, ctx->stream>>>((uint4*)d_io, totals, n); launched(ctx);
  pool_free(ctx, totals);
}
bool words_equal(zkb_ctx* ctx, const uint32_t* a, const uint32_t* b, size_t n) {
  if (!n) return true;
  uint32_t* flag = nullptr;
  pool_alloc(ctx, &flag, 4);
  ZKB_CUDA(cudaMemsetAsync(flag, 0, 4, ctx->stream));
  if (aligned16(a) && aligned16(b)) {
    const size_t n4 = n / 4;
    const uint32_t tail = (uint32_t)(n % 4);
    k_differ<uint4><<<grid_for(std::max<size_t>(n4, tail), EW_BLOCK), EW_BLOCK, 0, ctx->stream>>>((const uint4*)a, (const uint4*)b, n4, a + 4 * n4, b + 4 * n4, tail, flag);
  } else {
    k_differ<uint32_t><<<grid_for(n, EW_BLOCK), EW_BLOCK, 0, ctx->stream>>>(a, b, n, a, b, 0, flag);
  }
  launched(ctx);
  uint32_t differ = 1;
  ZKB_CUDA(cudaMemcpyAsync(&differ, flag, 4, cudaMemcpyDeviceToHost, ctx->stream));
  ZKB_CUDA(cudaStreamSynchronize(ctx->stream));
  pool_free(ctx, flag);
  return differ == 0;
}

}  // namespace zkb

using namespace zkb;

static inline void check_po2(int po2) { ZKB_REQUIRE(po2 >= 0 && po2 <= MAX_PO2, "po2 out of range [0, 26]"); }

extern "C" {

zkb_err zkb_fill_u32(zkb_ctx* ctx, void* d_ptr, size_t n, uint32_t value) {
  ZKB_API_BEGIN use(ctx); ZKB_REQUIRE(d_ptr || !n, "null buffer"); fill_u32(ctx, (uint32_t*)d_ptr, n, value); ZKB_API_END
}
zkb_err zkb_eltwise_add_elem(zkb_ctx* ctx, void* d_out, const void* d_a, const void* d_b, size_t n) {
  ZKB_API_BEGIN use(ctx); ZKB_REQUIRE((d_out && d_a && d_b) || !n, "null buffer"); eltwise_add(ctx, (uint32_t*)d_out, (const uint32_t*)d_a, (const uint32_t*)d_b, n); ZKB_API_END
}
zkb_err zkb_eltwise_copy_elem(zkb_ctx* ctx, void* d_out, const void* d_in, size_t n) {
  ZKB_API_BEGIN use(ctx); ZKB_REQUIRE((d_out && d_in) || !n, "null buffer");
  if (n) ZKB_CUDA(cudaMemcpyAsync(d_out, d_in, n * 4, cudaMemcpyDeviceToDevice, ctx->stream));
  ZKB_API_END
}
zkb_err zkb_eltwise_zeroize_elem(zkb_ctx* ctx, void* d_io, size_t n) {
  ZKB_API_BEGIN use(ctx); ZKB_REQUIRE(d_io || !n, "null buffer"); eltwise_zeroize(ctx, (uint32_t*)d_io, n); ZKB_API_END
}
zkb_err zkb_gather_sample(zkb_ctx* ctx, void* d_dst, const void* d_src, size_t idx, size_t size, size_t stride) {
  ZKB_API_BEGIN use(ctx); ZKB_REQUIRE((d_dst && d_src) || !size, "null buffer"); gather_sample(ctx, (uint32_t*)d_dst, (const uint32_t*)d_src, idx, size, stride); ZKB_API_END
}
zkb_err zkb_gather_rows(zkb_ctx* ctx, void* d_dst, const void* d_src, size_t src_len, const uint32_t* h_idx, size_t n_idx, size_t size, size_t stride) {
  ZKB_API_BEGIN use(ctx);
  if (!n_idx || !size) return nullptr;
  ZKB_REQUIRE(d_dst && d_src && h_idx, "null buffer");
  ZKB_REQUIRE(n_idx <= 65535, "gather_rows: more than 65535 rows in one call");
  ZKB_REQUIRE(stride == 0 || (size - 1) <= (src_len ? src_len - 1 : 0) / stride, "gather_rows: a row reaches outside the source buffer");      // (no overflow in the product below)
  for (size_t q = 0; q < n_idx; ++q) ZKB_REQUIRE((size_t)h_idx[q] + (size - 1) * stride < src_len, "gather_rows: a row reaches outside the source buffer");
  uint32_t* d_idx = nullptr;
  pool_alloc(ctx, &d_idx, n_idx * 4);
  ZKB_CUDA(cudaMemcpyAsync(d_idx, h_idx, n_idx * 4, cudaMemcpyHostToDevice, ctx->stream));
  gather_rows(ctx, (uint32_t*)d_dst, (const uint32_t*)d_src, d_idx, n_idx, size, stride);
  ZKB_CUDA(cudaStreamSynchronize(ctx->stream));          // h_idx is the caller's (pageable) memory: done with it before returning
  pool_free(ctx, d_idx);
  ZKB_API_END
}
zkb_err zkb_scatter(zkb_ctx* ctx, void* d_into, size_t into_len, const uint32_t* h_index, size_t n_rows, const uint32_t* h_offsets, const uint32_t* h_values) {
  ZKB_API_BEGIN use(ctx);
  ZKB_REQUIRE(h_index || !n_rows, "null index");
  if (!n_rows) return nullptr;
  const uint32_t k0 = h_index[0], k1 = h_index[n_rows];
  for (size_t r = 0; r < n_rows; ++r) ZKB_REQUIRE(h_index[r] <= h_index[r + 1], "scatter: index must be non-decreasing");
  if (k1 == k0) return nullptr;
  ZKB_REQUIRE(d_into && h_offsets && h_values, "null buffer");
  const size_t count = k1 - k0;
  uint32_t* d_tmp = nullptr;
  pool_alloc(ctx, &d_tmp, (2 * count + 1) * 4);
  ZKB_CUDA(cudaMemcpyAsync(d_tmp, h_offsets + k0, count * 4, cudaMemcpyHostToDevice, ctx->stream));
  ZKB_CUDA(cudaMemcpyAsync(d_tmp + count, h_values + k0, count * 4, cudaMemcpyHostToDevice, ctx->stream));
  ZKB_CUDA(cudaMemsetAsync(d_tmp + 2 * count, 0, 4, ctx->stream));
  k_scatter<<<grid_for(count, EW_BLOCK), EW_BLOCK, 0, ctx->stream>>>((uint32_t*)d_into, d_tmp, d_tmp + count, count, into_len, d_tmp + 2 * count); launched(ctx);
  uint32_t bad = 0;
  ZKB_CUDA(cudaMemcpyAsync(&bad, d_tmp + 2 * count, 4, cudaMemcpyDeviceToHost, ctx->stream));
  ZKB_CUDA(cudaStreamSynchronize(ctx->stream));
  pool_free(ctx, d_tmp);
  ZKB_REQUIRE(bad == 0, "scatter: offset outside the destination buffer");
  ZKB_API_END
}
zkb_err zkb_prefix_products(zkb_ctx* ctx, void* d_io_fp4, size_t n) {
  ZKB_API_BEGIN use(ctx); ZKB_REQUIRE((d_io_fp4 && aligned16(d_io_fp4)) || !n, "null or misaligned buffer"); prefix_products(ctx, (uint32_t*)d_io_fp4, n); ZKB_API_END
}
zkb_err zkb_zk_shift(zkb_ctx* ctx, void* d_io, size_t count, int po2) {
  ZKB_API_BEGIN use(ctx); check_po2(po2); ZKB_REQUIRE(d_io || !count, "null buffer"); zk_shift(ctx, (uint32_t*)d_io, count, po2); ZKB_API_END
}
zkb_err zkb_batch_expand(zkb_ctx* ctx, void* d_out, const void* d_in, size_t count, int in_po2, int expand_bits) {
  ZKB_API_BEGIN use(ctx); check_po2(in_po2); ZKB_REQUIRE(expand_bits >= 0 && in_po2 + expand_bits <= MAX_PO2, "expand_bits out of range");
  ZKB_REQUIRE((d_out && d_in) || !count, "null buffer");
  batch_expand(ctx, (uint32_t*)d_out, (const uint32_t*)d_in, count, in_po2, expand_bits);
  ZKB_API_END
}
zkb_err zkb_batch_bit_reverse(zkb_ctx* ctx, void* d_io, size_t count, int po2) {
  ZKB_API_BEGIN use(ctx); check_po2(po2); ZKB_REQUIRE(d_io || !count, "null buffer"); batch_bit_reverse(ctx, (uint32_t*)d_io, count, po2); ZKB_API_END
}
zkb_err zkb_eltwise_sum_extelem(zkb_ctx* ctx, void* d_out, const void* d_in, size_t count, size_t to_add) {
  ZKB_API_BEGIN use(ctx); ZKB_REQUIRE((d_out && d_in && aligned16(d_in)) || !count, "null or misaligned buffer");
  eltwise_sum_extelem(ctx, (uint32_t*)d_out, (const uint32_t*)d_in, count, to_add);
  ZKB_API_END
}
zkb_err zkb_fri_fold(zkb_ctx* ctx, void* d_out, const void* d_in, const uint32_t* h_mix, size_t out_count) {
  ZKB_API_BEGIN use(ctx); ZKB_REQUIRE(((d_out && d_in) || !out_count) && h_mix, "null buffer");
  fri_fold(ctx, (uint32_t*)d_out, (const uint32_t*)d_in, Fp4::load(h_mix), out_count);
  ZKB_API_END
}
zkb_err zkb_mix_poly_coeffs(zkb_ctx* ctx, void* d_out, const uint32_t* h_mix_start, const uint32_t* h_mix, const void* d_in, const void* d_combos,
                            size_t input_size, size_t count) {
  ZKB_API_BEGIN use(ctx);
  ZKB_REQUIRE(d_out && d_in && d_combos && h_mix_start && h_mix, "null buffer");
  ZKB_REQUIRE(aligned16(d_out), "out must be 16-byte aligned");
  // combo slots present: read the ids back once (tiny) to size the grid
  std::vector<uint32_t> ids(input_size);
  ZKB_CUDA(cudaMemcpyAsync(ids.data(), d_combos, input_size * 4, cudaMemcpyDeviceToHost, ctx->stream));
  ZKB_CUDA(cudaStreamSynchronize(ctx->stream));
  uint32_t slots = 0;
  for (uint32_t v : ids) slots = std::max(slots, v + 1);
  ZKB_REQUIRE(slots <= 65535, "combo id too large");
  mix_poly_coeffs(ctx, (uint32_t*)d_out, Fp4::load(h_mix_start), Fp4::load(h_mix), (const uint32_t*)d_in, (const uint32_t*)d_combos, input_size, count, slots);
  ZKB_API_END
}
zkb_err zkb_batch_evaluate_any(zkb_ctx* ctx, const void* d_coeffs, size_t poly_count, int po2, const void* d_which, const void* d_xs, void* d_out, size_t n_eval) {
  ZKB_API_BEGIN use(ctx); check_po2(po2); (void)poly_count;
  ZKB_REQUIRE((d_coeffs && d_which && d_xs && d_out) || !n_eval, "null buffer");
  ZKB_REQUIRE(aligned16(d_xs) && aligned16(d_out), "xs/out must be 16-byte aligned");
  batch_evaluate_any(ctx, (const uint32_t*)d_coeffs, po2, (const uint32_t*)d_which, (const uint32_t*)d_xs, (uint32_t*)d_out, n_eval, false);
  ZKB_API_END
}
zkb_err zkb_poly_divide(zkb_ctx* ctx, void* d_poly, size_t n, const uint32_t* h_z, void* d_rem) {
  ZKB_API_BEGIN use(ctx);
  ZKB_REQUIRE(d_poly && h_z && d_rem && aligned16(d_poly) && aligned16(d_rem), "null or misaligned buffer");
  poly_divide(ctx, (uint32_t*)d_poly, n, Fp4::load(h_z), (uint32_t*)d_rem);
  ZKB_API_END
}
// SURVEY.md 8(b) `zkb_combos_divide`: the whole division step of Prover::finalize in one call -- division k divides combo polynomial
// h_combo[k] (n Fp4 coefficients at d_combos + 4 n h_combo[k] words) by (x - h_points[k]) in place, in the order given (a combo is divided
// once per tap offset it holds); the n_div remainders come back together (one synchronisation instead of one per quotient).
zkb_err zkb_combos_divide(zkb_ctx* ctx, void* d_combos, size_t n, size_t n_combos, const uint32_t* h_combo, const uint32_t* h_points, size_t n_div, uint32_t* h_rem) {
  ZKB_API_BEGIN use(ctx);
  if (!n_div) return nullptr;
  ZKB_REQUIRE(d_combos && h_combo && h_points && h_rem && aligned16(d_combos), "null or misaligned buffer");
  ZKB_REQUIRE(n >= 1, "combos_divide: empty polynomials");
  for (size_t k = 0; k < n_div; ++k) ZKB_REQUIRE(h_combo[k] < n_combos, "combos_divide: combo index out of range");
  uint32_t* d_rem = nullptr;
  pool_alloc(ctx, &d_rem, n_div * 16);
  for (size_t k = 0; k < n_div; ++k) poly_divide(ctx, (uint32_t*)d_combos + (size_t)h_combo[k] * n * 4, n, Fp4::load(h_points + 4 * k), d_rem + 4 * k);
  ZKB_CUDA(cudaMemcpyAsync(h_rem, d_rem, n_div * 16, cudaMemcpyDeviceToHost, ctx->stream));
  ZKB_CUDA(cudaStreamSynchronize(ctx->stream));
  pool_free(ctx, d_rem);
  ZKB_API_END
}

}  // extern "C"
