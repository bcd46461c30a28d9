#!/usr/bin/env python3
"""bench.py — MSM throughput (scalar.point terms / second) on the BASELINE configs.

    python bench.py [--gpus N] [--steps K] [--warmup W]             # headline: C2, weak scaling
    python bench.py --workload {c1,c2,c3,c4,c5} [--scaling {weak,strong}] [...]
    python bench.py --impl reference [...]                          # the reference's CPU path
    python bench.py --dump-outputs DIR [...]                        # also write the results (.npy)

Workloads (SURVEY §8d; inputs are the reference benchmarks' own, generated in HBM by
b200_synthetic_generators_device):
  c1  ristretto255, built-in generators (generators == NULL), 1 column, n = 2^16
  c2  ristretto255, explicit generators g(i), 252-bit scalars, n = 2^20        <- BASELINE metric
  c3  bls12-381 G1, per-index generate_random_element points (distinct), 255-bit scalars, n = 2^22
  c4  64 columns x n = 2^20 ristretto255 over shared generators, columns sharded over the GPUs
  c5  bn254 G1 fixed-base MSM through an sxt_multiexp_handle, n = 2^24, generator range sharded
A "step" is one complete MSM (one call of the hot path) over the synthetic batch.
  value  device-resident: inputs already in HBM in the ABI layout; CUDA events on the library stream
  e2e    the same metric through the reference-facing C ABI with HOST (pinned) buffers: H2D of the
         inputs and D2H of the result inside the timed region
N > 1 (torchrun, one process per GPU). weak: every rank owns a full-size generator-range shard
(c2: 2^20 terms per GPU) of one N-times larger MSM; strong: the config's n is split over the ranks.
The only exchange is an NCCL all-gather of one partial point per column and rank, then N-1 point
additions (SURVEY §8e). c4 shards by column: no exchange at all.

With no --workload the headline line (c2, weak) also carries an "extras" object: short runs of the
other BASELINE configs at this N (N = 1: c3, the per-GPU shares of c4 and c5, pageable-memory e2e, the
reference's own GPU kernels on the same inputs; N > 1: strong-scaling c2, c4, c5).

--dump-outputs DIR writes, on rank 0, what the last timed device-resident step of the measured
workload returned, so that two builds can be compared output for output (the inputs depend only on
the arguments): DIR/commitments.npy (c1-c4: the commitment of every column) or
DIR/projective_results.npy (c5: the projective MSM result), float64 [columns, bytes] holding the
specified bytes of each result, one byte value per element.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "MSM throughput (scalar*point terms/sec), ristretto255, n=2^20 per GPU"
# name -> (curve id, log2 n, columns, bytes per term (SURVEY §8d), top-byte mask, description)
WORKLOADS = {
    "c1": (0, 16, 1, 192, 0x0F, "C1: ristretto255 Pedersen commitment, built-in generators, 1 column, n=2^16"),
    "c2": (0, 20, 1, 192, 0x0F, "C2: ristretto255 MSM, random 252-bit scalars, n=2^20"),
    "c3": (1, 22, 1, 136, 0x7F, "C3: bls12-381 G1 MSM, random 255-bit scalars, n=2^22, distinct generators"),
    "c4": (0, 20, 64, 52, 0x0F, "C4: multi-commitment, 64 columns x n=2^20 ristretto255"),
    "c5": (2, 24, 1, 96, 0x3F, "C5: bn254 G1 fixed-generator MSM (sxt_fixed_multiexponentiation), n=2^24"),
}
KERNEL_NAMES = {0: "Ed25519", 1: "Bls12381G1", 2: "Bn254G1", 3: "GrumpkinG"}


def read_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index):
        self.rows = []
        self.dev = device_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "25",
                 "-i", str(self.dev)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                    "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(mx)) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def make_scalars(n, seed, top_mask=0x0F, nbytes=32):
    """Uniform random bytes with the top byte masked (SURVEY §8d: < 2^252 / 2^255 / 2^254)."""
    rng = np.random.default_rng(seed)
    s = rng.integers(0, 256, (n, nbytes), dtype=np.uint8)
    s[:, nbytes - 1] &= top_mask
    return s


# ---------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation on the host cores
# ---------------------------------------------------------------------------------------------------
_REF_CACHE = {}


def _ref_worker(args):
    """One single-threaded reference MSM of n ristretto terms; returns (seconds inside the MSM call,
    commitment bytes). Input generation is outside the timed span."""
    n, seed, use_ref = args
    if use_ref:
        from oracle import refcpu as o
    else:
        from oracle import port as o
    if n not in _REF_CACHE:
        _REF_CACHE[n] = o.ristretto_generators(n, 0)
    g = _REF_CACHE[n]
    s = make_scalars(n, seed)
    t = time.perf_counter()
    out = o.commit(0, [(s, 0)], g)
    return time.perf_counter() - t, out.tobytes()


def cpu_baseline_sample(n_sample, procs, seed=100, warm=True):
    """`procs` independent reference MSMs of n_sample terms running concurrently (the reference cpu
    backend is single-threaded per call: README.md:89-92). Returns (terms/s, kind, results)."""
    import multiprocessing as mp
    from oracle import refcpu
    use_ref = refcpu.available()
    ctx = mp.get_context("spawn")
    with ctx.Pool(procs) as pool:
        if warm:
            pool.map(_ref_worker, [(min(n_sample, 1 << 12), 7 + i, use_ref) for i in range(procs)])
        res = pool.map(_ref_worker, [(n_sample, seed + i, use_ref) for i in range(procs)])
    return procs * n_sample / max(r[0] for r in res), ("reference" if use_ref else "port"), res


def run_reference(args, rank, world):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    # per process and step; a 20-step run stays within a few minutes. The reference's cpu throughput
    # falls slowly with n (BASELINE.md §3), so a 2^16-term column is close to the 2^20 workload.
    n_sample = 1 << 16
    from oracle import refcpu
    use_ref = refcpu.available()
    kind = "reference" if use_ref else "port"
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    steps = args.steps  # ~1.5-2 s per step on a 128-core host
    with ctx.Pool(cores) as pool:
        pool.map(_ref_worker, [(1 << 12, i, use_ref) for i in range(cores)])  # load + page in
        for _ in range(max(1, min(args.warmup, 1))):
            pool.map(_ref_worker, [(n_sample, i, use_ref) for i in range(cores)])
        wall = 0.0
        for k in range(steps):
            wall += max(r[0] for r in pool.map(_ref_worker, [(n_sample, 1000 * k + i, use_ref)
                                                             for i in range(cores)]))
    terms = steps * cores * n_sample
    value = terms / wall
    sample = (f"{cores} concurrent single-threaded reference MSMs of n=2^16 ristretto terms per step, "
              f"{steps} timed steps (the reference cpu backend is serial per call; a 2^20-term column "
              f"per core is out of reach of a bounded run — see cpu_baseline_same_config in the CUDA "
              f"arm's line for one full-size single-core MSM)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "terms/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * wall / steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64 (radix-2^51 limbs, integer)", "data": "synthetic",
        "config": {"workload": WORKLOADS["c2"][5] + " per GPU",
                   "reference_sample_terms_per_step": cores * n_sample},
        "cpu_baseline": {"value": value, "unit": "terms/s", "cores": cores, "kind": kind,
                         "sample": sample},
        "e2e": {"value": value, "unit": "terms/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# CUDA arm
# ---------------------------------------------------------------------------------------------------
class Env:
    """Per-process CUDA / NCCL context shared by the workloads."""

    def __init__(self, rank, local_rank, world):
        import torch
        import blitzar_b200 as bb
        self.torch, self.bb = torch, bb
        self.rank, self.local_rank, self.world = rank, local_rank, world
        self.dist = None
        torch.cuda.set_device(local_rank)
        if world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            self.dist = dist
        assert bb.sxt_init(device=local_rank) == 0
        # the library's stream as a torch stream: NCCL collectives issued under it are ordered against
        # the engine's kernels on the device, without host synchronisation
        self.lib_stream = torch.cuda.ExternalStream(bb.stream_ptr(),
                                                    device=torch.device("cuda", local_rank))

    def barrier(self):
        self.bb.synchronize()
        self.torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def pinned(self, shape):
        return self.torch.empty(shape, dtype=self.torch.uint8).pin_memory()

    def dev(self, shape):
        return self.torch.empty(shape, dtype=self.torch.uint8, device="cuda")

    def max_over_ranks(self, *vals):
        if self.dist is None:
            return vals
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return tuple(float(x) for x in t)


def run_workload(env, name, scaling, steps, warmup, with_e2e=True, sampler=None):
    """Times one BASELINE workload at env.world GPUs. Returns a dict (rank 0) of measurements; every
    rank must call it."""
    torch, bb, dist, world, rank = env.torch, env.bb, env.dist, env.world, env.rank
    curve, logn, ncol_total, bytes_per_term, mask, desc = WORKLOADS[name]
    n_cfg = 1 << logn
    pb = bb.point_bytes(curve)
    gen_stride = {0: 160, 1: 104, 2: 72, 3: 72}[curve]
    proj_stride = {0: 160, 1: 144, 2: 96, 3: 96}[curve]
    out_bytes = {0: 32, 1: 48, 2: 72, 3: 72}[curve]
    fixed = name.startswith("c5")
    by_column = name.startswith("c4")
    if by_column:  # columns are sharded; every rank holds all generators
        assert ncol_total % world == 0
        ncol, n, first = ncol_total // world, n_cfg, 0
        scaling = "strong"
    else:
        ncol = ncol_total
        if scaling == "weak":
            n, first = n_cfg, rank * n_cfg
        else:
            assert n_cfg % world == 0
            n, first = n_cfg // world, rank * (n_cfg // world)
    global_terms = (n * ncol) * world if not by_column else n * ncol_total
    builtin = name == "c1"

    # ---- synthetic inputs, generated where they will be used ---------------------------------------
    d_gens = None
    if not builtin:
        stride = proj_stride if fixed else gen_stride
        d_gens = env.dev((n, stride))
        bb.synthetic_generators_device(curve, d_gens.data_ptr(), n, first, projective=fixed)
    scal_host = [env.pinned((n, 32)) for _ in range(ncol)]
    for j, sh in enumerate(scal_host):
        col_id = j + (rank * ncol if by_column else 0)
        sh.numpy()[:] = make_scalars(n, 12345 + 1000 * col_id + (0 if by_column else rank), mask)
    d_scal = [env.dev((n, 32)) for _ in range(ncol)]
    for d, h in zip(d_scal, scal_host):
        d.copy_(h)
    gens_host = None
    if not builtin and not fixed and with_e2e:
        gens_host = env.pinned((n, gen_stride))
        gens_host.copy_(d_gens)
    handle, t_handle = None, None
    if fixed:
        bb.synchronize()
        t0 = time.perf_counter()
        handle = bb.MultiexpHandle(curve, device_ptr=d_gens.data_ptr(), n=n)
        bb.synchronize()
        t_handle = time.perf_counter() - t0
    torch.cuda.synchronize()
    bb.synchronize()
    d_partial = torch.zeros((ncol, pb), dtype=torch.uint8, device="cuda")
    d_all = torch.zeros((world, ncol, pb), dtype=torch.uint8, device="cuda")
    res_stride = proj_stride if fixed else out_bytes
    d_out = torch.zeros((ncol * res_stride + 64,), dtype=torch.uint8, device="cuda")
    shapes = [(n, 32, 0)] * ncol
    scal_ptrs = [d.data_ptr() for d in d_scal]
    exchange = world > 1 and not by_column

    def combine():
        with torch.cuda.stream(env.lib_stream):
            dist.all_gather_into_tensor(d_all.view(-1), d_partial.view(-1))
        if fixed:
            bb.combine_partials_projective_device(curve, d_out.data_ptr(), d_all.data_ptr(), world, ncol)
        else:
            bb.combine_partials_device(curve, d_out.data_ptr(), d_all.data_ptr(), world, ncol)

    def step_device():
        out_ptr, part_ptr = (None, d_partial.data_ptr()) if exchange else (d_out.data_ptr(), None)
        if fixed:
            bb.fixed_msm_device(handle, out_ptr, part_ptr, 32, 1, n, scal_ptrs[0])
        else:
            bb.commit_device(curve, shapes, scal_ptrs, d_gens.data_ptr() if d_gens is not None else None,
                             out_ptr, part_ptr, first if builtin else 0)
        if exchange:
            combine()

    out_host = env.pinned((ncol * res_stride + 64,))

    def step_e2e(columns=None, gens=None):
        """host buffers in, host result out — the plugin call a consumer makes (per rank: the same
        pipelined upload path, partial points, then the exchange)"""
        cols = columns if columns is not None else [(h.numpy(), 0) for h in scal_host]
        g = gens if gens is not None else (gens_host.numpy() if gens_host is not None else None)
        if not exchange:
            if fixed:
                return handle.fixed_multiexponentiation(32, 1, n, cols[0][0])
            return bb.compute_pedersen_commitments(curve, cols, g, first if builtin else 0)
        if fixed:
            bb.fixed_msm_host_partials(handle, d_partial.data_ptr(), 32, 1, n, cols[0][0])
        else:
            bb.commit_host_partials(curve, cols, g, d_partial.data_ptr(), first if builtin else 0)
        combine()
        bb.lib().b200_memcpy_d2h(C.c_void_p(out_host.data_ptr()), C.c_void_p(d_out.data_ptr()),
                                 C.c_uint64(ncol * res_stride))
        return out_host.numpy()[:ncol * res_stride].reshape(ncol, res_stride).copy()

    # ---- device-resident timing --------------------------------------------------------------------
    for _ in range(warmup):
        step_device()
    env.barrier()
    bb.profile_accumulate(True)
    bb.profile_read()
    launches0 = bb.launch_count()
    e0, e1 = bb.Event(), bb.Event()
    env.barrier()
    e0.record()
    for _ in range(steps):
        step_device()
    e1.record()
    ms = e0.elapsed_ms(e1)
    env.barrier()
    launches = bb.launch_count() - launches0
    acc_ms, acc_launches = bb.profile_read()
    bb.profile_accumulate(False)
    dev_result = d_out.cpu().numpy()[:ncol * res_stride].reshape(ncol, res_stride).copy()

    # ---- end-to-end timing -------------------------------------------------------------------------
    t_e2e, e2e_result = None, None
    if with_e2e:
        for _ in range(max(1, warmup // 2)):
            step_e2e()
        env.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            e2e_result = step_e2e()
        bb.synchronize()
        t_e2e = time.perf_counter() - t0
        env.barrier()
        k = {0: 32, 1: 48, 2: 65, 3: 65}[curve]
        if not fixed:
            assert np.array_equal(np.asarray(e2e_result)[:, :k], dev_result[:, :k]), \
                f"{name}: device-resident and end-to-end paths disagree"
    ms, t_e2e_m = env.max_over_ranks(ms, t_e2e or 0.0)

    res = {
        "workload": desc, "scaling": scaling, "n_per_gpu": n, "columns_per_gpu": ncol,
        "global_terms": global_terms, "steps": steps, "warmup": warmup,
        "ms_per_step": ms / steps, "value": global_terms * steps / (ms * 1e-3), "unit": "terms/s",
        "gpu_launches": int(launches),
        "_state": dict(dev_result=dev_result, e2e_step=step_e2e, scal_host=scal_host,
                       gens_host=gens_host, first=first, n=n, curve=curve, mask=mask, fixed=fixed),
    }
    if with_e2e:
        h2d = n * 32 * ncol + (0 if (builtin or fixed) else n * gen_stride)
        res["e2e"] = {"value": global_terms * steps / t_e2e_m, "unit": "terms/s",
                      "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": ncol * res_stride,
                      "ms_per_step": 1e3 * t_e2e_m / steps, "host_memory": "pinned"}
    if acc_launches:
        acc_avg_ms = acc_ms / acc_launches
        per_launch_terms = n * ncol * steps / acc_launches  # several launches per step: pieces / groups
        peak, peak_src = read_peaks()
        achieved = bytes_per_term * per_launch_terms / (acc_avg_ms * 1e-3) / 1e9
        res["roofline"] = {
            "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": None, "peak_source": peak_src,
            "kernel": f"level-1 bucket accumulation ({KERNEL_NAMES[curve]})",
            "kernel_ms": acc_avg_ms, "launches_per_step": acc_launches / steps,
            "kernel_share_of_step": acc_ms / ms,
            "algorithmic_bytes_per_launch": bytes_per_term * per_launch_terms,
            "bytes_per_term": bytes_per_term}
    if t_handle is not None:
        res["handle_new_s"] = t_handle
    return res


def dump_outputs(directory, st):
    """The device-resident result of the last timed step as float64 byte values (see the module
    docstring); struct padding is left out."""
    from tests import common
    os.makedirs(directory, exist_ok=True)
    k = st["dev_result"].shape[1] if st["fixed"] else common.CMP[st["curve"]]
    name = "projective_results" if st["fixed"] else "commitments"
    np.save(os.path.join(directory, name + ".npy"), st["dev_result"][:, :k].astype(np.float64))


def release(res):
    st = res.pop("_state", None)
    return st


def check_against_reference(env, res, st):
    """Parity of the bench's own result, not only self-consistency (ADVICE r1): Weierstrass workloads
    through the closed form over the reference's generators, with ONE reference scalar multiplication."""
    from oracle import refcpu
    from tests import common
    if not refcpu.available() or st["curve"] == 0 or env.world != 1:
        return None
    s = st["scal_host"][0].numpy()
    want = common.closed_form_commitment(refcpu, st["curve"], s, st["first"])
    got = st["dev_result"][:1]
    if st["fixed"]:
        got = refcpu.normalize(st["curve"], np.ascontiguousarray(got))
    return bool(common.same(st["curve"], got, want))


def run_cuda(args, rank, local_rank, world):
    env = Env(rank, local_rank, world)
    bb = env.bb
    headline = args.workload or "c2"
    scaling = args.scaling or "weak"
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    main = run_workload(env, headline, scaling, args.steps, args.warmup)
    clocks = sampler.stop() if rank == 0 else None
    st = release(main)
    curve = st["curve"]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, st)

    extras = {}
    cpu, cpu_same = None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, kind, _ = cpu_baseline_sample(1 << 17, 1)
        cpu = {"value": v, "unit": "terms/s", "cores": 1, "kind": kind,
               "sample": "one reference cpu-backend MSM of n=2^17 ristretto terms (same generator / "
                         "scalar distribution as the workload), 1 thread — the reference cpu backend "
                         "is serial"}
    if args.workload is None and not args.no_extras:
        # ---- the other BASELINE configs, short runs ------------------------------------------------
        xs, xw = 5, 3
        if world == 1:
            if headline == "c2" and rank == 0 and not args.no_cpu_baseline:
                # same-config single-core reference MSM on the bench's own inputs: the CPU number at
                # the metric's n AND the oracle check of the GPU result
                from oracle import refcpu
                o = refcpu if refcpu.available() else __import__("oracle.port", fromlist=["port"])
                s = st["scal_host"][0].numpy()
                t0 = time.perf_counter()
                want = o.commit(0, [(s, 0)], st["gens_host"].numpy())
                dt = time.perf_counter() - t0
                ok = bool(np.array_equal(want[:, :32], st["dev_result"][:, :32]))
                assert ok, "C2 result differs from the reference cpu backend"
                cpu_same = {"value": st["n"] / dt, "unit": "terms/s", "cores": 1,
                            "kind": "reference" if refcpu.available() else "port", "seconds": dt,
                            "sample": "ONE reference cpu-backend MSM on the bench's own C2 inputs "
                                      "(n=2^20); its commitment equals the CUDA result",
                            "matches_cuda_result": ok}
                # pageable host memory (what a Rust Vec is)
                cols = [(np.array(h.numpy()), 0) for h in st["scal_host"]]
                gens = np.array(st["gens_host"].numpy())
                for _ in range(2):
                    st["e2e_step"](cols, gens)
                t0 = time.perf_counter()
                for _ in range(xs):
                    st["e2e_step"](cols, gens)
                dt = (time.perf_counter() - t0) / xs
                extras["e2e_pageable"] = {"value": st["n"] / dt, "unit": "terms/s", "ms_per_step": dt * 1e3,
                                          "host_memory": "pageable (numpy arrays)"}
                from oracle import refgpu
                if refgpu.available():
                    best = (1e9, 1e9)
                    for _ in range(2):
                        _, whole, kern = refgpu.bucket_msm(st["gens_host"].numpy(), s)
                        best = min(best, (whole, kern))
                    extras["refgpu"] = {"kernels_ms": best[1], "with_copies_ms": best[0],
                                        "what": "the reference's own bucket-method CUDA kernels compiled "
                                                "for sm_100a (oracle/_ref/libblitzar_ref_gpu.so), same "
                                                "C2 inputs, same GPU; kernels only, not its host pipeline"}
            del st
            for nm in ("c3", "c4_share", "c5_share", "c1"):
                if nm == "c4_share":
                    WORKLOADS[nm] = (0, 20, 8, 52, 0x0F, "C4 per-GPU share: 8 columns x n=2^20 ristretto255")
                if nm == "c5_share":
                    WORKLOADS[nm] = (2, 21, 1, 96, 0x3F, "C5 per-GPU share: bn254 fixed-base MSM, n=2^21")
                r = run_workload(env, nm, "strong", xs, xw)
                s2 = release(r)
                if rank == 0 and nm in ("c3", "c5_share"):
                    s2["fixed"] = nm == "c5_share"
                    r["matches_reference_closed_form"] = check_against_reference(env, r, s2)
                del s2
                extras[nm] = r
        else:
            del st
            r = run_workload(env, "c2", "strong", xs, xw)
            release(r)
            extras["c2_strong"] = r
            if 64 % world == 0:
                r = run_workload(env, "c4", "strong", xs, xw)
                release(r)
                extras["c4"] = r
            r = run_workload(env, "c5", "strong", xs, xw)
            release(r)
            extras["c5"] = r

    if rank == 0:
        roof = main.get("roofline")
        if roof is not None and curve == 0:
            roof["note"] = ("integer-ALU bound (about 16 point additions of 8 field multiplications "
                            "per term); see DESIGN.md")
            roof["secondary"] = imad_roofline(main["n_per_gpu"], roof["kernel_ms"] * roof["launches_per_step"],
                                              clocks)
            prof = os.path.join(ROOT, "profiles", "r02_accumulate_traffic.json")
            if os.path.exists(prof):
                try:
                    j = json.load(open(prof))
                    roof["traffic"] = j.get("dram_bytes_per_launch")
                    roof["traffic_source"] = "profiles/r02_accumulate_traffic.json (ncu --set full capture)"
                except Exception:
                    pass
        line = {
            "metric": METRIC if headline == "c2" else "MSM throughput (terms/s), " + main["workload"],
            "value": main["value"], "unit": "terms/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": main["ms_per_step"],
            "higher_is_better": True, "scaling": main["scaling"], "vs_baseline": None,
            "dtype": "u32 limbs (integer modular arithmetic)", "data": "synthetic",
            "config": {"workload": main["workload"] + (" per GPU (generator-range shard per rank)"
                                                       if main["scaling"] == "weak" else ""),
                       "global_terms": main["global_terms"], "curve": KERNEL_NAMES[curve],
                       "cache": "inputs per step exceed the 126 MB L2",
                       "parallelism": f"generator-range x{world}" if headline != "c4" else f"columns x{world}"},
            "e2e": main.get("e2e"),
            "gpu_launches": main["gpu_launches"],
            "clocks": clocks,
            "roofline": roof,
            "cpu_baseline": cpu,
        }
        if cpu_same:
            line["cpu_baseline_same_config"] = cpu_same
        if extras:
            line["extras"] = extras
        print(json.dumps(line), flush=True)
    if env.dist is not None:
        env.dist.destroy_process_group()


def imad_roofline(n, kernel_ms, clocks):
    """The bound that actually limits the accumulation kernel: the 32x32->64 multiplier. One term
    has 16 signed 16-bit digits (252-bit scalars), i.e. 16 bucket entries; every entry except the
    first of a bucket run is one cached-form addition = 8 field multiplications = 8 x (64 + 8)
    IMAD.WIDE.U32 (schoolbook 8x8 limbs + the 2^256 = 38 fold). Peak = 29.2 lane-ops/clk/SM measured
    on B200 for the multiply-accumulate-with-carry form this kernel issues (tests/micro/pipes.cu;
    plain IMAD.WIDE 23.0, IMAD.HI 24.6) x 148 SMs x the SM clock sampled during the run."""
    windows, nbuckets = 16, 1 << 15
    entries = windows * n * (1.0 - 2.0 ** -16)  # zero digits are skipped
    runs = windows * nbuckets * (1.0 - (1.0 - 1.0 / nbuckets) ** (entries / windows))
    imads = (entries - runs) * 8 * 72
    mhz = (clocks or {}).get("sm_mhz") or 1965.0
    peak = 29.2 * 148 * mhz * 1e6
    achieved = imads / (kernel_ms * 1e-3)
    return {"bound": "imad_wide", "achieved": achieved, "peak": peak, "unit": "IMAD.WIDE lane-ops/s",
            "frac": achieved / peak, "imad_wide_per_step": imads}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=None, choices=["c1", "c2", "c3", "c4", "c5"])
    ap.add_argument("--scaling", default=None, choices=["weak", "strong"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result of the last timed step to DIR as .npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_cuda(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
