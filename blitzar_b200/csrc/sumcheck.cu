// Instantiates the sumcheck prover (sumcheck.cuh) for both sumcheck fields.
#include "sumcheck.cuh"
namespace b200 {
void sumcheck_prove(const EngineCtx& ctx, void* polynomials, void* evaluation_point,
                    unsigned field_id, const sumcheck_descriptor* descriptor,
                    void* transcript_callback, void* transcript_context, bool mles_on_device) {
  const int code =
      sumcheck_check(polynomials, evaluation_point, field_id, descriptor, transcript_callback);
  B200_REQUIRE(code == kSumcheckOk, sumcheck_message(code));
  auto cb = reinterpret_cast<SumcheckCallback>(transcript_callback);
  auto* polys = static_cast<unsigned char*>(polynomials);
  auto* point = static_cast<unsigned char*>(evaluation_point);
  if (field_id == SXT_FIELD_SCALAR255)
    Sumcheck<FSc25>::prove(ctx.s, polys, point, true, field_id, *descriptor, cb, transcript_context,
                           mles_on_device);
  else
    Sumcheck<FGk>::prove(ctx.s, polys, point, false, field_id, *descriptor, cb, transcript_context,
                         mles_on_device);
}
}  // namespace b200
