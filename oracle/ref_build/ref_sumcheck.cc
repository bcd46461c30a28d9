// TEST INFRASTRUCTURE — not product code.
//
// The reference's cpu sumcheck prover (cbindings/sumcheck.cc + cpu_backend.cc:73-112) behind a C
// symbol, `ref_prove_sumcheck`. Built by sumcheck.mk into oracle/_ref/libblitzar_ref_sumcheck.so and
// linked against libblitzar_ref_cpu.so, which already holds the field arithmetic of both sumcheck
// fields; the prover itself is template-only in the reference (sxt/proof/sumcheck/*.h).
#include <cstddef>
#include <utility>

#include "sxt/base/num/ceil_log2.h"
#include "sxt/cbindings/backend/callback_sumcheck_transcript.h"
#include "sxt/fieldgk/realization/field.h"
#include "sxt/proof/sumcheck/cpu_driver.h"
#include "sxt/proof/sumcheck/proof_computation.h"
#include "sxt/scalar25/realization/field.h"

using namespace sxt;

// the product-table layouts the C ABI documents: 36-byte entries for scalar255, 40 for grumpkin
static_assert(sizeof(std::pair<s25t::element, unsigned>) == 36, "scalar255 product-table stride");
static_assert(sizeof(std::pair<fgkt::element, unsigned>) == 40, "grumpkin product-table stride");

// layout-compatible with sumcheck_descriptor (cbindings/blitzar_api.h:155-183)
struct ref_sumcheck_descriptor {
  const void* mles;
  const void* product_table;
  const unsigned* product_terms;
  unsigned n, num_mles, num_products, num_product_terms, round_degree;
};

template <class T>
static void prove(void* polynomials, void* evaluation_point, const ref_sumcheck_descriptor& d,
                  void* callback, void* context) {
  const auto num_variables = static_cast<size_t>(std::max(basn::ceil_log2(d.n), 1));
  cbnbck::callback_sumcheck_transcript<T> transcript{
      reinterpret_cast<typename cbnbck::callback_sumcheck_transcript<T>::callback_t>(callback),
      context};
  prfsk::cpu_driver<T> drv;
  auto fut = prfsk::prove_sum<T>(
      {static_cast<T*>(polynomials), (d.round_degree + 1u) * num_variables},
      {static_cast<T*>(evaluation_point), num_variables}, transcript, drv,
      {static_cast<const T*>(d.mles), static_cast<size_t>(d.n) * d.num_mles},
      {static_cast<const std::pair<T, unsigned>*>(d.product_table), d.num_products},
      {d.product_terms, d.num_product_terms}, d.n);
  (void)fut;
}

// field_id 0: s25t::element (SXT_FIELD_SCALAR255), 1: fgkt::element (SXT_FIELD_GRUMPKIN)
extern "C" void ref_prove_sumcheck(void* polynomials, void* evaluation_point, unsigned field_id,
                                   const ref_sumcheck_descriptor* descriptor, void* callback,
                                   void* context) {
  if (field_id == 0)
    prove<s25t::element>(polynomials, evaluation_point, *descriptor, callback, context);
  else
    prove<fgkt::element>(polynomials, evaluation_point, *descriptor, callback, context);
}
