// Type-erased per-curve entry points of the MSM engine. api.cu sees only this header, so the
// kernels of each curve are compiled exactly once, in that curve's own translation unit.
#pragma once
#include <cmath>
#include <cstdint>

#include "../../include/blitzar_b200.h"
#include "runtime.cuh"

namespace b200 {

struct MsmOptions {
  u32 window_bits = 0;  // 0 = choose from n
  u32 chunk1 = 0;       // chunk length of the first accumulation level (0 = 32, or 64 for big passes)
  u32 chunkn = 8;       // chunk length of the cascade levels
  u32 reduce_g1 = 16;   // bucket-reduction group size, first level (power of two)
  u32 reduce_gn = 4;    // bucket-reduction group size, later levels (power of two)
  u64 quad_threshold = 32768;  // launches with at most this many logical threads run 4 lanes each
  u64 max_group_entries = 1ull << 30;  // columns are grouped below this many (term, window) entries
  u64 max_range_entries = 1ull << 31;  // one sort pass holds at most this many entries: longer
                                       // columns are processed as several generator ranges
  int pair_levels = -1;  // batch-affine pair levels (Weierstrass): -1 = from the mean bucket load
  u32 pair_batch = 0;    // pairs per thread of a pair level (0 = 32)
  int range_skew = 0;   // piece schedule of a multi-range call (range_begin); set by the host layer
  u32 uniform_add = 2;  // gathering level: runs start from the identity (no divergent start path);
                        // 0 off, 1 on, 2 = ed25519 only
  u32 gens_normalized = 0;  // set per call: the generator array is a fixed-base table (Z = 1 entries)
  u32 lane_tail = 1;  // warp-cooperative (lane-sliced) Horner / encoding kernels for ed25519
  u32 scatter_window_major = 0;  // scatter with one thread per (window, term), window-major
  u32 table_policy = 0;  // fixed-base tables: 0 = cost model decides, 1 = whenever available, 2 = never
};

struct EngineCtx {
  stream_t s;
  MsmOptions opt;
  const void* builtin;  // device-resident built-in ristretto generators g(0..num_builtin)
  uint64_t num_builtin;
  stream_t tail = stream_t();  // optional second stream: cascade + merge of piece k under piece k+1
  // fixed-base table over the built-in generators (window w of generator i at builtin[w n + i]);
  // builtin_windows <= 1: plain generators only
  u32 builtin_window_bits = 0, builtin_windows = 0;
};

// sxt_multiexp_handle: generators of one curve resident in HBM, plus (when it pays and fits) the
// fixed-base table 2^(c w) G_i, w < windows, laid out window-major: entry w * n + i. Window 0 IS the
// generator array, so `gens` serves both the table mode and the variable-base fallback.
struct Handle {
  unsigned curve_id;
  unsigned n;
  void* gens;  // device array of the curve's generator layout, windows * n entries
  unsigned window_bits = 0, windows = 1;
};

// Window width of a fixed-base table over n generators: minimises (digit additions + bucket
// reduction) for one 256-bit output, subject to the table fitting in `budget_bytes` and in the
// 31-bit generator index of a sorted entry. Returns 0 when no table should be built.
inline unsigned table_window_bits(uint64_t n, size_t gen_bytes, double budget_bytes) {
  if (n < 1024)  // tiny handles: the variable-base path with a small window wins anyway
    return 0;
  unsigned best = 0;
  double best_cost = 1e300;
  for (unsigned c = 10; c <= 20; ++c) {
    const double W = 256 / c + 1;
    if (W * (double)n * (double)gen_bytes > budget_bytes || W * (double)n >= 2147483648.0)
      continue;
    const double cost = W * (double)n + 2.5 * (double)(1u << (c - 1));
    if (cost < best_cost) {
      best_cost = cost;
      best = c;
    }
  }
  return best;
}

template <class T> struct DevBuf {
  T* p = nullptr;
  stream_t s;
  DevBuf(size_t count, stream_t s_) : s(s_) { p = (T*)dev_alloc(count * sizeof(T), s); }
  ~DevBuf() { dev_free(p, s); }
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
};

// generator-range r of `num_ranges` over n terms starts here (shared by the engine and the C-ABI
// layer, which schedules the host-to-device copies of each range)
// skew > 0: pieces shrink towards the end (upload-bound calls: little work is left after the last
// byte has arrived); skew < 0: pieces grow (compute-bound calls: the first kernels start early);
// 0: equal pieces. begin(0) = 0, begin(num_ranges) = n, strictly monotone for n >= num_ranges.
inline uint64_t range_begin(uint64_t n, uint32_t r, uint32_t num_ranges, int skew = 0) {
  if (r == 0)
    return 0;
  if (r >= num_ranges)
    return n;
  if (skew == 0 || n < 64ull * num_ranges)
    return n * r / num_ranges;
  const double t = (double)r / (double)num_ranges;
  const double f = skew > 0 ? 1.0 - (1.0 - t) * std::sqrt(1.0 - t) : t * std::sqrt(t);
  uint64_t b = (uint64_t)((double)n * f);
  const uint64_t lo = r, hi = n - (num_ranges - r);  // keep every piece non-empty
  return b < lo ? lo : (b > hi ? hi : b);
}
// called on the host before the engine touches terms [begin, end) (e.g. make the compute stream wait
// for that range's copies)
typedef void (*range_wait_fn)(void* user, uint64_t begin, uint64_t end);

struct CurveVTable {
  unsigned curve_id, point_bytes, gen_bytes, abi_gen_bytes, abi_proj_bytes, abi_commit_bytes;
  void (*commit_device)(const EngineCtx&, void* out_commitments, void* out_partials, uint32_t num,
                        const sxt_sequence_descriptor* d, const void* generators_dev,
                        uint64_t offset_generators, uint32_t num_ranges, range_wait_fn wait,
                        void* wait_user);
  void (*fixed_device)(const EngineCtx&, void* out_res, void* out_partials, const Handle* h,
                       int mode, unsigned element_num_bytes, const unsigned* bit_table,
                       const unsigned* lengths, unsigned num_outputs, unsigned n,
                       const uint8_t* scalars_dev);
  void (*ingest_projective)(const EngineCtx&, const void* raw_dev, void* gens, uint64_t n);
  void (*gens_to_projective)(const EngineCtx&, const void* gens, void* out_dev, uint64_t n);
  void (*store)(const EngineCtx&, const void* pts, void* out_dev, uint64_t count, bool commit);
  void (*sum_parts)(const EngineCtx&, const void* parts, uint32_t nparts, uint32_t count,
                    void* out_pts);
  // synthetic generators (synth.cuh) in the ABI layout: projective structs or commit-stride affine
  void (*synth_generators)(const EngineCtx&, void* out_dev, uint64_t n, uint64_t first,
                           bool projective);
  unsigned abi_compact_bytes;
  // generators out of a reference partition-table image (device copy of the file's table)
  void (*ingest_compact_table)(const EngineCtx&, const void* table_dev, unsigned window_width,
                               void* gens, uint64_t n);
  // fills windows 1 .. windows-1 of a fixed-base table whose window 0 (n generators) is in place
  void (*build_table)(const EngineCtx&, void* table, uint64_t n, unsigned window_bits,
                      unsigned windows);
};
extern const CurveVTable kVTableEd25519, kVTableBls12381, kVTableBn254, kVTableGrumpkin;

// inner-product argument over ristretto255 (ipa.cuh); same contracts as the two sxt_* entry points
void ipa_prove(const EngineCtx& ctx, uint8_t* l_vector, uint8_t* r_vector, uint8_t* ap_value,
               uint8_t* transcript203, uint64_t n, uint64_t generators_offset,
               const uint8_t* a_vector, const uint8_t* b_vector);
int ipa_verify(const EngineCtx& ctx, uint8_t* transcript203, uint64_t n,
               uint64_t generators_offset, const uint8_t* b_vector, const uint8_t* product,
               const uint8_t* a_commit160, const uint8_t* l_vector, const uint8_t* r_vector,
               const uint8_t* ap_value);

// sumcheck prover (sumcheck.cuh); the contract of sxt_prove_sumcheck, descriptor->mles a device
// pointer when mles_on_device. Aborts with a message on an invalid descriptor.
void sumcheck_prove(const EngineCtx& ctx, void* polynomials, void* evaluation_point,
                    unsigned field_id, const sumcheck_descriptor* descriptor,
                    void* transcript_callback, void* transcript_context, bool mles_on_device);

// lane-sliced field arithmetic self-test (lanefield.cuh): number of mismatching checks over
// `warps` warps of pseudo-random / edge-case operands
unsigned selftest_lane_arithmetic(const EngineCtx& ctx, unsigned warps, unsigned seed);

// built-in ristretto generators g(first .. first+n) into the device generator layout
void launch_builtin_generators(const EngineCtx& ctx, void* gens, uint64_t first, uint64_t n);

}  // namespace b200
