// TEST INFRASTRUCTURE — never linked into the product.
//
// The sumcheck prover of blitzar_b200/csrc/sumcheck.cuh with its kernel bodies run as serial host
// loops (-DB200_EMULATE, see emul.cpp), linked into the same emulation library.
#include "emul_prefix.h"
#include "../../blitzar_b200/csrc/sumcheck.cuh"

using namespace b200;

// same contract as sxt_prove_sumcheck (the descriptor is assumed valid: see emul_sumcheck_check)
extern "C" void emul_prove_sumcheck(void* polynomials, void* evaluation_point, unsigned field_id,
                                    const sumcheck_descriptor* d, void* callback, void* context) {
  auto cb = reinterpret_cast<SumcheckCallback>(callback);
  auto* polys = static_cast<unsigned char*>(polynomials);
  auto* point = static_cast<unsigned char*>(evaluation_point);
  if (field_id == 0)
    Sumcheck<FSc25>::prove(0, polys, point, true, field_id, *d, cb, context, false);
  else
    Sumcheck<FGk>::prove(0, polys, point, false, field_id, *d, cb, context, false);
}
// the descriptor checks of sxt_prove_sumcheck as a return code (0 = valid, see SumcheckCheck)
extern "C" int emul_sumcheck_check(const void* polynomials, const void* evaluation_point,
                                   unsigned field_id, const sumcheck_descriptor* d,
                                   const void* callback) {
  return sumcheck_check(polynomials, evaluation_point, field_id, d, callback);
}
