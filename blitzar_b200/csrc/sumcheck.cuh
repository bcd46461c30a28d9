// Sumcheck prover over the two sumcheck fields: sxt_prove_sumcheck / b200_prove_sumcheck_device.
//
// Replaces sxt/proof/sumcheck/{sum_gpu,fold_gpu,reduction_gpu,gpu_driver}.h for the gpu backend
// (dispatch: sxt/cbindings/backend/gpu_backend.cc:106-145). Protocol (cbindings/blitzar_api.h:133-183,
// sxt/proof/sumcheck/proof_computation.h), with mid = 2^(num_variables - 1 - round):
//   p(X) = sum_{i < mid} sum_k mult_k prod_{j in terms_k} (f_j[i] + (f_j[i + mid] - f_j[i]) X)
//   r    = callback(p)                          (host; the caller's transcript)
//   f_j' = (1 - r) f_j[i] + r f_j[i + mid]      (f_j[i + mid] = 0 past the current length)
// The MLEs stay resident in HBM for the whole proof; the host sees the round_degree + 1
// coefficients and returns r, one stream synchronisation per round.
//
// Element types: FSc25 (mod l, SXT_FIELD_SCALAR255: 32-byte plain integers in the ABI) and FGk
// (mod r of bn254, SXT_FIELD_GRUMPKIN: Montgomery limbs in the ABI, bit-identical to ours). On the
// device everything is Montgomery; plain inputs are converted as they are first read (one multiply
// by R^2), and the round coefficients are converted back before they leave the device.
#pragma once
#include <algorithm>
#include <vector>

#include "engine_api.cuh"

namespace b200 {

// longest product the kernels are specialised for (the reference's max_degree_v,
// sxt/proof/sumcheck/constant.h:25)
constexpr unsigned kSumcheckMaxLength = 5;
constexpr int kSumcheckCoeffs = kSumcheckMaxLength + 1;

// Descriptor checks (error code, 0 = valid); every non-zero code aborts the C-ABI call with the
// message below.
enum SumcheckCheck {
  kSumcheckOk = 0,
  kSumcheckNull = 1,           // a required pointer is null
  kSumcheckField = 2,          // field_id is neither SXT_FIELD_SCALAR255 nor SXT_FIELD_GRUMPKIN
  kSumcheckEmpty = 3,          // n == 0
  kSumcheckDegree = 4,         // round_degree == 0 (a round polynomial needs two coefficients)
  kSumcheckLengthZero = 5,     // a product of length 0
  kSumcheckLengthDegree = 6,   // a product longer than round_degree
  kSumcheckLengthCap = 7,      // a product longer than kSumcheckMaxLength
  kSumcheckTermCount = 8,      // sum of the product lengths != num_product_terms
  kSumcheckTermIndex = 9,      // a product term >= num_mles
};
inline const char* sumcheck_message(int code) {
  switch (code) {
  case kSumcheckNull: return "sumcheck: polynomials, evaluation_point, descriptor, its arrays and the "
                             "callback must not be null";
  case kSumcheckField: return "sumcheck: unsupported field_id (0 = scalar255, 1 = grumpkin)";
  case kSumcheckEmpty: return "sumcheck: n must be greater than zero";
  case kSumcheckDegree: return "sumcheck: round_degree must be at least 1";
  case kSumcheckLengthZero: return "sumcheck: every product_length must be at least 1";
  case kSumcheckLengthDegree: return "sumcheck: a product_length exceeds round_degree";
  case kSumcheckLengthCap: return "sumcheck: product_length above 5 is not supported";
  case kSumcheckTermCount: return "sumcheck: product lengths do not add up to num_product_terms";
  case kSumcheckTermIndex: return "sumcheck: a product term is not an MLE index (< num_mles)";
  default: return "sumcheck: invalid descriptor";
  }
}
// Byte stride of the product table: the reference's std::pair<FIELD, unsigned> is 36 bytes for
// scalar255 (alignment 1) and 40 for grumpkin (alignment 8); the length sits at byte 32 in both.
inline size_t sumcheck_table_stride(unsigned field_id) { return field_id == 0 ? 36 : 40; }
inline unsigned sumcheck_length(const sumcheck_descriptor& d, unsigned field_id, unsigned k) {
  unsigned len;
  std::memcpy(&len, (const unsigned char*)d.product_table + k * sumcheck_table_stride(field_id) + 32,
              sizeof len);
  return len;
}
inline int sumcheck_check(const void* polynomials, const void* evaluation_point, unsigned field_id,
                          const sumcheck_descriptor* d, const void* callback) {
  if (!polynomials || !evaluation_point || !d || !callback)
    return kSumcheckNull;
  if (field_id > 1)
    return kSumcheckField;
  if (d->n == 0)
    return kSumcheckEmpty;
  if (d->round_degree == 0)
    return kSumcheckDegree;
  if (!d->mles || (d->num_products && !d->product_table) || (d->num_product_terms && !d->product_terms))
    return kSumcheckNull;
  uint64_t total = 0;
  for (unsigned k = 0; k < d->num_products; ++k) {
    const unsigned len = sumcheck_length(*d, field_id, k);
    if (len == 0)
      return kSumcheckLengthZero;
    if (len > kSumcheckMaxLength)
      return kSumcheckLengthCap;
    if (len > d->round_degree)
      return kSumcheckLengthDegree;
    total += len;
  }
  if (total != d->num_product_terms)
    return kSumcheckTermCount;
  for (unsigned t = 0; t < d->num_product_terms; ++t)
    if (d->product_terms[t] >= d->num_mles)
      return kSumcheckTermIndex;
  return kSumcheckOk;
}

// ---- device side -------------------------------------------------------------------------------
template <class F> B200_HD void sc_load(typename F::E& v, const typename F::E* p, u64 i, bool plain) {
  v = p[i];
  if (plain)
    F::to_mont(v, v);
}
// The products of the polynomial: multipliers (Montgomery), lengths, and the concatenated terms.
template <class F> struct SumcheckProducts {
  const typename F::E* mult;
  const u32* lens;
  const u32* terms;
  u32 num_products;
};
// acc[0..L] += m prod_{t < L} (a_t + b_t X) at pair i, with a_t = f_j[i], b_t = f_j[i + mid] - a_t
// (f_j[i + mid] = 0 unless has_hi) and j = terms[t]: the factors are multiplied out one at a time,
// 2 + (L - 1)(L + 2) multiplications for a product of length L.
template <class F, int L>
B200_HD void sc_expand(typename F::E* acc, const typename F::E& m, const u32* terms,
                       const typename F::E* f, u64 stride, u64 i, u64 mid, bool has_hi,
                       bool plain) {
  typedef typename F::E E;
  E c[L + 1], a, b;
#pragma unroll
  for (int t = 0; t < L; ++t) {
    const u64 base = (u64)terms[t] * stride;
    sc_load<F>(a, f, base + i, plain);
    if (has_hi)
      sc_load<F>(b, f, base + i + mid, plain);
    else
      b = F::zero();
    F::sub(b, b, a);
    if (t == 0) {
      F::mul(c[0], m, a);
      F::mul(c[1], m, b);
    } else {
      F::mul(c[t + 1], c[t], b);
#pragma unroll
      for (int d = t; d >= 1; --d) {
        E u;
        F::mul(c[d], c[d], a);
        F::mul(u, c[d - 1], b);
        F::add(c[d], c[d], u);
      }
      F::mul(c[0], c[0], a);
    }
  }
#pragma unroll
  for (int d = 0; d <= L; ++d)
    F::add(acc[d], acc[d], c[d]);
}
template <class F>
B200_HD void sc_accumulate_pair(typename F::E* acc, const SumcheckProducts<F>& P,
                                const typename F::E* f, u64 stride, u64 i, u64 mid, bool has_hi,
                                bool plain) {
  u32 t = 0;
  for (u32 k = 0; k < P.num_products; ++k) {
    const u32 len = P.lens[k];
    const typename F::E m = P.mult[k];
    switch (len) {
    case 1: sc_expand<F, 1>(acc, m, P.terms + t, f, stride, i, mid, has_hi, plain); break;
    case 2: sc_expand<F, 2>(acc, m, P.terms + t, f, stride, i, mid, has_hi, plain); break;
    case 3: sc_expand<F, 3>(acc, m, P.terms + t, f, stride, i, mid, has_hi, plain); break;
    case 4: sc_expand<F, 4>(acc, m, P.terms + t, f, stride, i, mid, has_hi, plain); break;
    default: sc_expand<F, 5>(acc, m, P.terms + t, f, stride, i, mid, has_hi, plain); break;
    }
    t += len;
  }
}
template <class F>
B200_HD void sc_store_partials(typename F::E* partial, u64 threads, u64 t, u32 width,
                               const typename F::E* acc) {
#pragma unroll
  for (int c = 0; c < kSumcheckCoeffs; ++c)
    if ((u32)c < width)
      partial[c * threads + t] = acc[c];
}

// Round sum: thread t takes the pairs i = t, t + threads, ...
// (neighbouring threads read neighbouring elements) and leaves `width` partial coefficients,
// coefficient-major: partial[c * threads + t]. Column j of f starts at f + j * stride.
template <class F> struct SumcheckSumBody {
  static constexpr int kBlock = 128;
  typedef typename F::E E;
  const E* f;
  u64 stride, mid, hi;  // pairs i < mid; f_j[i + mid] exists for i < hi
  u64 threads;
  u32 width;
  bool plain;  // f holds plain values (scalar255 input)
  SumcheckProducts<F> P;
  E* partial;
  B200_HD void operator()(u64 t) const {
    E acc[kSumcheckCoeffs];
#pragma unroll
    for (int c = 0; c < kSumcheckCoeffs; ++c)
      acc[c] = F::zero();
    for (u64 i = t; i < mid; i += threads)
      sc_accumulate_pair<F>(acc, P, f, stride, i, mid, i < hi, plain);
    sc_store_partials<F>(partial, threads, t, width, acc);
  }
};

// Fold at the midpoint m of the previous round: out_j[q] = g_j[q] + r (g_j[q + m] - g_j[q]), one
// thread per (MLE j, position q < m). g: length gn, column stride gs; out: column stride m. It is its
// own launch before each later round's sum: on a B200 that beat folding inside the sum kernel by up
// to 15 % (DESIGN.md §12).
template <class F> struct SumcheckFoldBody {
  static constexpr int kBlock = 128;
  typedef typename F::E E;
  const E* g;
  u64 gs, gn;
  bool plain;  // g holds plain values (scalar255 input, first fold)
  E r;         // Montgomery
  E* out;
  u64 m;
  B200_HD void operator()(u64 t) const {
    const u64 j = t / m, q = t % m;
    E lo, hi;
    sc_load<F>(lo, g, j * gs + q, plain);
    if (q + m < gn)
      sc_load<F>(hi, g, j * gs + q + m, plain);
    else
      hi = F::zero();
    F::sub(hi, hi, lo);
    F::mul(hi, hi, r);
    F::add(out[j * m + q], lo, hi);
  }
};

// One reduction level: out[c * out_count + u] = sum of in[c * count + u * G ...] over G partials. The
// last level (out_count == 1) writes the round polynomial, in the ABI form of the field.
template <class F> struct SumcheckReduceBody {
  static constexpr int kBlock = 128;
  typedef typename F::E E;
  const E* in;
  u64 count, out_count;
  u32 G;
  bool to_plain;
  E* out;
  B200_HD void operator()(u64 t) const {
    const u64 c = t / out_count, u = t % out_count;
    const u64 b = u * G, e = std::min<u64>(b + G, count);
    E acc = F::zero();
    for (u64 k = b; k < e; ++k)
      F::add(acc, acc, in[c * count + k]);
    if (out_count == 1 && to_plain)
      F::from_mont(acc, acc);
    out[c * out_count + u] = acc;
  }
};

// ---- host driver ---------------------------------------------------------------------------------
typedef void (*SumcheckCallback)(void* r, void* context, const void* polynomial, unsigned len);

template <class F> struct Sumcheck {
  typedef typename F::E E;
  // Threads of a round with `mid` pairs: a grid-stride launch of at most kMaxThreads; once
  // mid <= kTailPairs a single block covers the round (the last rounds cost one small launch each
  // instead of a grid).
  static constexpr u64 kMaxThreads = 1ull << 17, kTailPairs = 1024;
  static constexpr u32 kGroup = 128;  // partials summed per thread of a reduction level
  static u64 round_threads(u64 mid) {
    if (mid <= kTailPairs)
      return std::min<u64>(mid, SumcheckSumBody<F>::kBlock);
    return std::min<u64>(mid, kMaxThreads);
  }
  static unsigned num_variables(unsigned n) {
    unsigned k = 0;
    while ((1ull << k) < n)
      ++k;
    return std::max(k, 1u);
  }

  // `plain`: the ABI form of the field is plain (scalar255). `mles_on_device`: d.mles is a device
  // pointer in the ABI layout, read in place and never written.
  static void prove(stream_t s, unsigned char* polynomials, unsigned char* evaluation_point,
                    bool plain, unsigned field_id, const sumcheck_descriptor& d,
                    SumcheckCallback callback, void* context, bool mles_on_device) {
    const u64 n = d.n, M = d.num_mles;
    const unsigned v = num_variables(d.n);
    const unsigned plen = d.round_degree + 1;
    u64 mid = 1ull << (v - 1);

    // products: Montgomery multipliers, lengths, terms
    std::vector<E> mult(d.num_products);
    std::vector<u32> lens(d.num_products), terms(d.product_terms, d.product_terms + d.num_product_terms);
    u32 width = 1;
    for (unsigned k = 0; k < d.num_products; ++k) {
      std::memcpy(&mult[k], (const unsigned char*)d.product_table + k * sumcheck_table_stride(field_id),
                  sizeof(E));
      if (plain)
        F::to_mont(mult[k], mult[k]);
      lens[k] = sumcheck_length(d, field_id, k);
      width = std::max(width, lens[k] + 1);
    }
    DevBuf<E> dmult(d.num_products + 1, s);
    DevBuf<u32> dlens(d.num_products + 1, s), dterms(d.num_product_terms + 1, s);
    copy_h2d(dmult.p, mult.data(), mult.size() * sizeof(E), s);
    copy_h2d(dlens.p, lens.data(), lens.size() * sizeof(u32), s);
    copy_h2d(dterms.p, terms.data(), terms.size() * sizeof(u32), s);
    const SumcheckProducts<F> P{dmult.p, dlens.p, dterms.p, d.num_products};

    // MLE storage: the input (n x M), its first fold (mid x M) and a second fold buffer
    // (mid/2 x M), which for host input is the upload buffer itself
    const u64 fold1 = v > 1 ? mid * M : 0, fold2 = v > 2 ? (mid / 2) * M : 0;
    const u64 T0 = round_threads(mid);
    u64 partial_elems = 0;
    for (u64 c = T0; c > 1; c = (c + kGroup - 1) / kGroup)
      partial_elems += c;
    partial_elems = width * (partial_elems + 1);
#ifndef B200_EMULATE
    {
      size_t free_b = 0, total_b = 0;
      B200_CUDA(cudaMemGetInfo(&free_b, &total_b));
      int dev = 0;
      B200_CUDA(cudaGetDevice(&dev));
      cudaMemPool_t pool;
      B200_CUDA(cudaDeviceGetDefaultMemPool(&pool, dev));
      uint64_t reserved = 0, used = 0;  // freed blocks the pool keeps cached are reusable
      B200_CUDA(cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReservedMemCurrent, &reserved));
      B200_CUDA(cudaMemPoolGetAttribute(pool, cudaMemPoolAttrUsedMemCurrent, &used));
      const double need = (double)sizeof(E) * ((mles_on_device ? fold2 : n * M) + fold1 + partial_elems);
      B200_REQUIRE(need <= (double)free_b + (double)(reserved - used),
                   "sumcheck: the MLEs and their first fold do not fit in free device memory");
    }
#endif
    DevBuf<E> upload(mles_on_device ? 0 : n * M, s), buf1(fold1, s),
        buf2(mles_on_device ? fold2 : 0, s);
    const E* in = (const E*)d.mles;
    if (!mles_on_device) {
      copy_h2d(upload.p, d.mles, n * M * sizeof(E), s);
      in = upload.p;
    }
    E* folds[2] = {buf1.p, mles_on_device ? buf2.p : upload.p};
    DevBuf<E> partial(partial_elems, s), poly(plen, s);
    dev_zero(poly.p, plen * sizeof(E), s);  // coefficients above the longest product stay zero

    const E* cur = in;  // MLEs of this round: length 2 mid (n in the first round), stride cur_stride
    u64 cur_len = n;
    std::vector<unsigned char> r_abi(sizeof(E));
    E r{};
    for (unsigned round = 0; round < v; ++round) {
      const u64 T = round_threads(mid);
      if (round == 0) {
        launch(SumcheckSumBody<F>{in, n, mid, n > mid ? n - mid : 0, T, width, plain, P, partial.p},
               T, s);
      } else {
        E* out = folds[(round - 1) & 1];
        launch(SumcheckFoldBody<F>{cur, cur_len, cur_len, plain && round == 1, r, out, 2 * mid},
               2 * mid * M, s);
        launch(SumcheckSumBody<F>{out, 2 * mid, mid, mid, T, width, false, P, partial.p}, T, s);
        cur = out;
        cur_len = 2 * mid;
      }
      // reduction levels: width x T partials -> the round polynomial
      E* src = partial.p;
      u64 count = T;
      do {
        const u64 out_count = (count + kGroup - 1) / kGroup;
        E* dst = out_count == 1 ? poly.p : src + width * count;
        launch(SumcheckReduceBody<F>{src, count, out_count, kGroup, plain, dst}, width * out_count, s);
        src = dst;
        count = out_count;
      } while (count > 1);
      unsigned char* slot = polynomials + (size_t)round * plen * sizeof(E);
      copy_d2h(slot, poly.p, plen * sizeof(E), s);
      stream_sync(s);
      callback(r_abi.data(), context, slot, plen);
      std::memcpy(evaluation_point + (size_t)round * sizeof(E), r_abi.data(), sizeof(E));
      std::memcpy(&r, r_abi.data(), sizeof(E));
      if (plain)
        F::to_mont(r, r);
      mid /= 2;
    }
    stream_sync(s);  // the buffers of this call are released stream-ordered
  }
};

}  // namespace b200
