"""Sumcheck timing on the GPU (sxt_prove_sumcheck host-to-host, b200_prove_sumcheck_device on MLEs
already in HBM, per-round device time) beside the reference cpu backend at small n.

Shape of the reference's benchmark (benchmark/sumcheck/benchmark.m.cc): num_products products of
length `degree` over n x (degree * num_products) MLEs, product_terms = iota, random multipliers.
Traffic and field multiplications are counted from the shapes (`round_counts`); the achieved rate
is set against the HBM bandwidth and an integer-multiply issue bound (see `bounds`).

    python tests/sumcheck_timing.py [--log2n 16 18 20 22 24] [--degrees 2 3 5] [--products 1 2 4]
                                    [--fields 0 1] [--reps 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import blitzar_b200 as bb  # noqa: E402
from tests.test_sumcheck import Challenger  # noqa: E402

HBM_BYTES_PER_S = 7.7e12  # HGX B200 data sheet, one GPU
SMS = 148
IMAD_PER_CLK_SM = 64  # 32-bit integer multiply-add issue rate per SM (one per lane of two SMSPs)
IMADS_PER_MUL = 2 * 8 * 8 + 8  # 8-limb CIOS Montgomery product: a*b and m*p wide products + m
ELEM = 32
HOST_LIMIT = 1 << 31  # host-to-host runs only where the MLEs take at most 2 GiB of host memory


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True).stdout
    name, power, clock = [x.strip() for x in q.splitlines()[0].split(",")]
    return name, power, float(clock.split()[0]) * 1e6


def round_counts(n, degree, num_products, field_id):
    """Per round: (HBM bytes read + written, field multiplications), from the shapes. Round 0 sums
    the uploaded MLEs; round k >= 1 folds the previous MLEs (4 mid elements per MLE in, 2 mid out,
    one multiplication per folded element) and then sums the folded MLEs (2 mid elements per MLE
    read again)."""
    m = degree * num_products
    v = max((n - 1).bit_length(), 1)
    per_pair = num_products * (2 + (degree - 1) * (degree + 2))
    out = []
    for k in range(v):
        mid = 1 << (v - 1 - k)
        if k == 0:
            hbm = n * m * ELEM
            muls = mid * per_pair + (2 * mid * m if field_id == 0 else 0)  # scalar255: to Montgomery
        else:
            prev = n if k == 1 else 4 * mid
            hbm = (prev + 4 * mid) * m * ELEM
            muls = mid * per_pair + 2 * mid * m + (prev * m if (k == 1 and field_id == 0) else 0)
        out.append((hbm, muls))
    return out


def bounds(counts, clock_hz):
    hbm = sum(c[0] for c in counts) / HBM_BYTES_PER_S
    mul = sum(c[1] for c in counts) * IMADS_PER_MUL / (SMS * IMAD_PER_CLK_SM * clock_hz)
    return hbm, mul


def inputs(n, degree, num_products, field_id, seed):
    m = degree * num_products
    g = torch.Generator(device="cuda").manual_seed(seed)
    mles = torch.randint(0, 256, (m, n, ELEM), dtype=torch.uint8, device="cuda", generator=g)
    mles[:, :, ELEM - 1] &= 0x0F  # < 2^252: canonical for both fields
    rng = np.random.default_rng(seed)
    table = []
    for _ in range(num_products):
        mult = rng.integers(0, 256, ELEM, dtype=np.uint8)
        mult[-1] &= 0x0F
        table.append((mult.tobytes(), degree))
    return mles, table, list(range(m))


class RoundClock(Challenger):
    """The test callback plus a CUDA event on the library's stream at every round boundary (the
    stream is idle while the callback runs)."""

    def __init__(self, field_id, stream):
        super().__init__(field_id)
        self.stream, self.events = stream, []
        self.mark()

    def mark(self):
        e = torch.cuda.Event(enable_timing=True)
        e.record(self.stream)
        self.events.append(e)

    def __call__(self, polynomial):
        r = super().__call__(polynomial)
        self.mark()
        return r

    def round_ms(self):
        self.events[-1].synchronize()
        return [a.elapsed_time(b) for a, b in zip(self.events, self.events[1:])]


def run(args):
    name, power, clock = card()
    print(f"card: {name}, power limit {power}, max SM clock {clock / 1e6:.0f} MHz", flush=True)
    assert bb.sxt_init() == 0
    stream = torch.cuda.ExternalStream(bb.stream_ptr())
    results = []
    for field_id in args.fields:
        for logn in args.log2n:
            for degree in args.degrees:
                for num_products in args.products:
                    n = 1 << logn
                    mles, table, terms = inputs(n, degree, num_products, field_id, seed=logn)
                    torch.cuda.synchronize()
                    m = mles.shape[0]

                    def device_call(clock_cb=None):
                        ch = clock_cb or Challenger(field_id)
                        return bb.prove_sumcheck_device(field_id, mles.data_ptr(), n, m, table,
                                                        terms, ch)

                    device_call()  # warm-up: module load, pool growth
                    dev_ms = []
                    for _ in range(args.reps):
                        t0 = time.perf_counter()
                        polys, point = device_call()
                        dev_ms.append((time.perf_counter() - t0) * 1e3)
                    rc = RoundClock(field_id, stream)
                    device_call(rc)
                    rounds = rc.round_ms()
                    counts = round_counts(n, degree, num_products, field_id)
                    hbm_s, mul_s = bounds(counts, clock)
                    dev = min(dev_ms)
                    row = dict(field=field_id, log2n=logn, degree=degree, products=num_products,
                               mles=m, device_ms=round(dev, 3),
                               rounds_ms=[round(x, 4) for x in rounds],
                               round0_ms=round(rounds[0], 4),
                               hbm_bytes=sum(c[0] for c in counts),
                               field_muls=sum(c[1] for c in counts),
                               hbm_bound_ms=round(hbm_s * 1e3, 4),
                               mul_bound_ms=round(mul_s * 1e3, 4),
                               bound="hbm" if hbm_s >= mul_s else "multiply",
                               share_of_bound=round(max(hbm_s, mul_s) * 1e3 / sum(rounds), 3))
                    if m * n * ELEM <= HOST_LIMIT:
                        host = mles.cpu().numpy()
                        bb.prove_sumcheck(field_id, host, table, terms, Challenger(field_id))
                        t0 = time.perf_counter()
                        hp, hpt = bb.prove_sumcheck(field_id, host, table, terms,
                                                    Challenger(field_id))
                        row["host_ms"] = round((time.perf_counter() - t0) * 1e3, 3)
                        assert np.array_equal(hp, polys) and np.array_equal(hpt, point)
                        if logn <= args.ref_max_log2n:
                            from oracle import refsumcheck
                            t0 = time.perf_counter()
                            rp, rpt = refsumcheck.prove_sumcheck(field_id, host, table, terms,
                                                                 Challenger(field_id))
                            row["reference_cpu_ms"] = round((time.perf_counter() - t0) * 1e3, 3)
                            row["same_as_reference"] = bool(np.array_equal(rp, polys) and
                                                            np.array_equal(rpt, point))
                    results.append(row)
                    print(json.dumps(row), flush=True)
                    del mles
                    torch.cuda.empty_cache()
    summary = dict(card=name, power_limit=power, max_sm_clock_mhz=clock / 1e6, results=results)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(summary, f, indent=1)
    return summary


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2n", type=int, nargs="+", default=[16, 18, 20, 22, 24])
    ap.add_argument("--degrees", type=int, nargs="+", default=[2, 3, 5])
    ap.add_argument("--products", type=int, nargs="+", default=[1, 2, 4])
    ap.add_argument("--fields", type=int, nargs="+", default=[1, 0])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--ref-max-log2n", type=int, default=16,
                    help="time the reference cpu backend up to this n")
    ap.add_argument("--out", default=None, help="JSON file for the results")
    run(ap.parse_args())
