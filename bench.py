#!/usr/bin/env python
"""bench.py — BLS12-377 G1 MSM points/s (headline) and Fr NTT elements/s (secondary) on N B200s.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference CPU algorithms (oracle port)
    python bench.py ... --dump-outputs DIR                   # also write the last step's outputs as DIR/*.npy

One "step" = one pass of the hot path over one batch of synthetic input:
  * product arm: one 2^lg-point VariableBase::msm per GPU (weak scaling: every rank owns 2^lg points;
    at N > 1 the per-rank window sums are all-gathered over NCCL and added on the device) — `value` is
    measured with bases and scalars resident in HBM; `e2e` goes through the reference-facing C ABI with
    PAGEABLE host buffers (what a Rust Vec is): H2D of points + scalars and D2H of the result inside the
    timed region (`e2e_pinned`: the same call on pinned buffers).
  * reference arm: the CPU restatement of batched::msm (oracle/oracle.c, OpenMP over all host cores) on a
    bounded sample of the same workload — the Rust reference cannot be built here (no cargo/rustc).

Every timed result is CHECKED outside the timed region: the bases are h(seed, i)·G, so
Σ s_i·P_i = (Σ s_i·h_i mod r)·G — one dot product and one scalar multiplication by the oracle — for the
single-GPU MSM, the sharded result at every N, the 2^26-total sharded run and the KZG commitment; the NTT
output is compared with the oracle's fft_in_place element by element.  `checked` in the JSON line says so.

Prints ONE JSON line on rank 0.  Timing: CUDA events on the launching stream, barrier + synchronize on
both sides, max over ranks; inputs (≥ 2.2 GB per step) are far larger than L2 so no flush is needed.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

ALGO_BYTES_PER_POINT = 128      # SURVEY §8(d): 96 B affine (x, y) + 32 B scalar, each touched once
ALGO_BYTES_PER_ELEMENT = 64     # NTT: 32 B read + 32 B write per element per TRANSFORM
FALLBACK_HBM_GBS = 6650.0       # /opt/skills/guides/B200_PROFILING.md
R_MOD = 8444461749428370424248824938781546531375899335154063827935233455917409239041
R_LIMBS = np.array([(R_MOD >> (64 * i)) & (2**64 - 1) for i in range(4)], dtype=np.uint64)


def load_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def load_traffic(key):
    """dram bytes per launch of the dominant kernel from the committed ncu --set full summary, or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get(key)
    except Exception:
        return None


def random_scalars(n, seed):
    """Uniform integers in [0, r): draw 4 limbs, clear the top REPR_SHAVE_BITS = 3 bits, reject ≥ r — the reference's own
    sampler (fields/src/macros.rs:40-56).  Also used for Montgomery images (any value < r is one)."""
    rng = np.random.default_rng(seed)
    out = np.empty((n, 4), dtype=np.uint64)
    todo = np.arange(n)
    while todo.size:
        x = rng.integers(0, 2**64, size=(todo.size, 4), dtype=np.uint64)
        x[:, 3] &= np.uint64((1 << 61) - 1)
        lt = np.zeros(todo.size, dtype=bool)
        eq = np.ones(todo.size, dtype=bool)
        for i in (3, 2, 1, 0):
            lt |= eq & (x[:, i] < R_LIMBS[i])
            eq &= x[:, i] == R_LIMBS[i]
        out[todo[lt]] = x[lt]
        todo = todo[~lt]
    return out


def base_multipliers(seed, n):
    """h(seed, i) of snarkvm_b200_generate_bases_device (csrc/msm.cu): P_i = h·G, as canonical uint64 [n, 4]."""
    def sm(x):
        x = x + np.uint64(0x9E3779B97F4A7C15)
        x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return x ^ (x >> np.uint64(31))
    with np.errstate(over="ignore"):
        k = sm(np.uint64(seed & ((1 << 64) - 1)) ^ sm(np.arange(n, dtype=np.uint64)))
    k[k == 0] = 1
    ks = np.zeros((n, 4), dtype=np.uint64)
    ks[:, 0] = k
    return ks


def u64_as_f64(a):
    """uint64 limbs → their little-endian 32-bit words as float64 (last axis doubles); exact, every word is < 2^32"""
    return np.ascontiguousarray(a, dtype=np.uint64).view(np.uint32).astype(np.float64)


def dump_outputs(d, arrays):
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, f"{name}.npy"), a)


def limbs_to_int(a):
    return sum(int(v) << (64 * i) for i, v in enumerate(np.asarray(a).reshape(-1)[:4]))


def int_to_limbs(v):
    return np.array([(v >> (64 * i)) & (2**64 - 1) for i in range(4)], dtype=np.uint64)


class Checker:
    """The oracle used as the CHECKER, outside every timed region (never as the thing measured)."""

    def __init__(self):
        from oracle import bls12_377 as py, cpu
        cpu.build()
        try:
            cpu.set_num_threads(len(os.sched_getaffinity(0)))     # torchrun exports OMP_NUM_THREADS=1
        except AttributeError:
            cpu.set_num_threads(os.cpu_count() or 1)
        self.cpu, self.py = cpu, py
        self.g = np.frombuffer(py.affine_bytes(py.G1_GENERATOR), dtype=np.uint8).copy()

    def dot(self, scalars, seed):
        """Σ s_i·h(seed, i) mod r as a Python int (scalars canonical)"""
        return limbs_to_int(self.cpu.fr_dot_canonical(scalars, base_multipliers(seed, scalars.shape[0])))

    def point(self, k):
        """(k mod r)·G as the normalised projective image uint64[18]"""
        return self.cpu.g1_mul(self.g, int_to_limbs(k % R_MOD))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.proc = None

    def start(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            parts = [p.strip() for p in s.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0])); mx = float(parts[1])
            except ValueError:
                continue
            for nm, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def workload_config(args, world):
    """The workload both arms name (identical dict in the product and the reference line)."""
    return {"workload": f"bls12_377_g1_msm_2^{args.lg}_points_per_gpu", "points_per_gpu": 1 << args.lg,
            "scalars": "uniform in [0, r)", "bases": "h(seed,i)*G, affine 104 B stride",
            "parallelism": f"points sharded over {world} GPU(s); one all-gather of window sums" if world > 1 else "single GPU"}


# ------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle (CPU restatement of the reference algorithms)
# ------------------------------------------------------------------------------------------------
def cpu_msm_points_per_s(cpu, bases_host, scal):
    t = time.perf_counter()
    cpu.msm(bases_host, scal, cpu.BATCHED)
    dt = time.perf_counter() - t
    return scal.shape[0] / dt, dt


def cpu_ntt_elements_per_s(cpu, lg_sample):
    """Best over a few OpenMP team sizes: the port's per-stage parallel-for (standing in for rayon's chunked
    butterflies, fft/domain.rs:667-688) stops scaling — and can slow down — on very wide hosts."""
    x = random_scalars(1 << lg_sample, 778)
    allc = cpu.num_threads()
    best = None
    for th in sorted({allc, min(allc, 64), min(allc, 32), min(allc, 16)}, reverse=True):
        cpu.set_num_threads(th)
        cpu.ntt(x[:1 << 12], cpu.FORWARD, cpu.STANDARD)          # spin the team up
        t = time.perf_counter()
        cpu.ntt(x, cpu.FORWARD, cpu.STANDARD)
        dt = time.perf_counter() - t
        if best is None or dt < best[0]:
            best = (dt, th)
    cpu.set_num_threads(allc)
    return (1 << lg_sample) / best[0], best[0], best[1]


def cpu_bases(n):
    """Valid subgroup points for the CPU legs, built with the oracle's batched affine addition."""
    from oracle import bls12_377 as py, cpu
    bases = np.zeros((n, 104), dtype=np.uint8)
    bases[0] = np.frombuffer(py.affine_bytes(py.g1_mul(py.G1_GENERATOR, 0xB200)), dtype=np.uint8)
    cur = 1
    while cur < n:
        m = min(cur, n - cur)
        step = np.frombuffer(py.affine_bytes(py.g1_mul(py.G1_GENERATOR, cur)), dtype=np.uint8)
        bases[cur:cur + m] = cpu.batch_affine_add(bases[:m], np.tile(step, (m, 1)))
        cur += m
    return bases


def run_reference(args, rank, world):
    if rank != 0:
        return
    chk = Checker()
    cpu = chk.cpu
    lg = args.ref_lg
    if lg <= 0:
        # the workload's own size when the whole run stays within a few minutes (≈ 0.75 µs per point on 64 cores), else the
        # largest smaller power of two that does: 2^24 for ≤ 12 timed steps, 2^23 for ≤ 24, 2^22 beyond
        lg = args.lg
        while lg > 16 and args.steps * (1 << lg) * 0.75e-6 > 150.0:
            lg -= 1
    bases = cpu_bases(1 << lg)
    threads = cpu.num_threads()
    scal = random_scalars(1 << lg, 777)
    for _ in range(args.warmup):
        cpu.msm(bases[: 1 << min(lg, 16)], scal[: 1 << min(lg, 16)], cpu.BATCHED)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu.msm(bases, scal, cpu.BATCHED)
    dt = (time.perf_counter() - t0) / args.steps
    value = (1 << lg) / dt
    ntt_v, ntt_dt, ntt_th = cpu_ntt_elements_per_s(cpu, args.ref_ntt_lg)
    sample = (f"each step = one 2^{lg}-point batched::msm (a bounded sample of the 2^{args.lg}-point workload: points/s of this algorithm "
              f"grows only slowly with n) on {threads} OpenMP threads, one task per window as rayon in batched.rs:400-401")
    line = {
        "impl": "reference", "metric": "bls12_377_g1_msm_points_per_sec", "value": value, "unit": "points/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64 limbs (CPU)", "data": "synthetic",
        "config": workload_config(args, world),
        "note": "C restatement of the reference CPU (rayon) path — Rust toolchain unavailable",
        "cpu_baseline": {"value": value, "unit": "points/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "ntt": {"metric": "fr_ntt_elements_per_sec", "value": ntt_v, "unit": "elements/s",
                "sample": f"one 2^{args.ref_ntt_lg} forward fft_in_place, best of 16/32/64/{threads} threads = {ntt_th}", "ms": ntt_dt * 1e3},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# product arm
# ------------------------------------------------------------------------------------------------
def run_product(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    from snarkvm_b200 import _lib, cuda as shim, device, sharded

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback exists)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    n = 1 << args.lg
    peak, peak_src = load_peak()
    chk = Checker()
    checks = {}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks_mod_r(v):
        """Σ over ranks of a Python int, mod r (the closed-form dot products of the shards)"""
        if world == 1:
            return v % R_MOD
        objs = [None] * world
        dist.all_gather_object(objs, int(v))
        return sum(objs) % R_MOD

    def timed(fn, steps, collect=None):
        """K calls of fn bracketed by barrier + synchronize, CUDA events on the launching stream, max over ranks → ms per step;
        `collect` (if given) turns what the K calls returned into results INSIDE the timed region"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        outs = [fn() for _ in range(steps)]
        if collect is not None:
            outs = [collect(o) for o in outs]
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)) / steps, outs

    def wall_timed(fn, steps):
        barrier()
        t0 = time.perf_counter()
        outs = [fn() for _ in range(steps)]
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3
        barrier()
        return max_over_ranks(ms) / steps, outs

    # ---- inputs: per-rank shard, generated in HBM ----
    seed = 0xB200 + rank
    bases = device.generate_bases(n, seed=seed, device=dev)
    scal_np = random_scalars(n, 1234 + rank)
    scalars = torch.from_numpy(scal_np.view(np.int64)).to(dev)
    torch.cuda.synchronize()
    expect = chk.point(sum_over_ranks_mod_r(chk.dot(scal_np, seed)))          # closed form of the whole job's sum

    if world > 1:
        def step_device():
            return sharded.msm_sharded_async(bases, scalars, plan_npoints=n)
        collect = lambda p: p.result()                                         # noqa: E731
    else:
        def step_device():
            return device.msm(bases, scalars)
        collect = None

    first = step_device()
    first = collect(first) if collect else first
    checks["msm_value"] = bool((first == expect).all())
    assert checks["msm_value"], "device-resident MSM differs from the closed form (Σ s_i·h_i)·G"

    # ---- `value`: device-resident MSM, K steps ----
    for _ in range(args.warmup):
        o = step_device()
        if collect:
            collect(o)
    _lib.profile_enable(True)
    for k in (0, 1, 2, 3):
        _lib.profile_collect(k)
    sampler = ClockSampler(local_rank)
    launches0 = _lib.launch_count()
    if rank == 0:
        sampler.start()
    ms_per_step, outs = timed(step_device, args.steps, collect)
    clocks = sampler.stop() if rank == 0 else None
    launches = _lib.launch_count() - launches0
    acc_ms, acc_n = _lib.profile_collect(_lib.PROF_MSM_ACCUMULATE)
    sort_ms, _ = _lib.profile_collect(_lib.PROF_MSM_SORT)
    red_ms, _ = _lib.profile_collect(_lib.PROF_MSM_REDUCE)
    _lib.profile_enable(False)
    assert all((o == expect).all() for o in outs), "MSM result changed between steps"
    dumps = {"msm": u64_as_f64(outs[-1])}                # normalised projective X, Y, Z (Montgomery limbs) of the last step
    ms_total = ms_per_step * args.steps
    value = n * world / (ms_per_step * 1e-3)
    acc_ms_per_step = acc_ms / max(1, args.steps)           # the whole accumulation phase of one MSM (several kernels)
    achieved = ALGO_BYTES_PER_POINT * n / (acc_ms_per_step * 1e-3) / 1e9

    # ---- `e2e`: through the reference-facing call with HOST buffers (H2D + D2H inside the timing) ----
    # pageable = what a Rust Vec<G1Affine> / Vec<BigInteger256> is; pinned = the best a caller could do
    bases_pin = torch.empty((n, 104), dtype=torch.uint8).pin_memory()
    bases_pin.copy_(bases)
    torch.cuda.synchronize()
    scal_pin = torch.from_numpy(scal_np.view(np.int64)).pin_memory()
    b_pin, s_pin = bases_pin.numpy(), scal_pin.numpy().view(np.uint64)
    b_page = np.empty((n, 104), dtype=np.uint8); b_page[:] = b_pin       # plain malloc'd arrays
    s_page = np.empty((n, 4), dtype=np.uint64); s_page[:] = scal_np
    e2e_steps = max(1, min(args.steps, args.e2e_steps))

    def make_e2e(bh, sh):
        if world == 1:
            return (lambda: shim.msm(bh, sh)), None                       # snarkvm_msm: H2D points+scalars, MSM, D2H 144 B
        return (lambda: sharded.msm_sharded_async(bh, sh, plan_npoints=n, dev=dev)), (lambda p: p.result())

    e2e = {}
    for name, bh, sh in (("pageable", b_page, s_page), ("pinned", b_pin, s_pin)):
        fn, col = make_e2e(bh, sh)
        r = fn(); r = col(r) if col else r
        ok = bool((r == expect).all())
        checks[f"msm_e2e_{name}"] = ok
        assert ok, f"e2e ({name}) result differs from the closed form"
        ms, _ = wall_timed((lambda: col(fn())) if col else fn, e2e_steps)
        e2e[name] = ms
    e2e_ms = e2e["pageable"]
    e2e_value = n * world / (e2e_ms * 1e-3)
    del b_page, s_page
    e2e_resident = None
    if world == 1 and not args.skip_registered:
        # same call, SRS-style usage: the bases slice was registered once (snarkvm_b200_register_bases), only the
        # 32 B/point scalars cross PCIe per call
        shim.register_bases(b_pin)
        assert (shim.msm(b_pin, s_pin) == expect).all()
        r_ms, _ = wall_timed(lambda: shim.msm(b_pin, s_pin), e2e_steps)
        shim.unregister_bases(b_pin)
        e2e_resident = {"value": n / (r_ms * 1e-3), "unit": "points/s", "ms_per_step": r_ms, "h2d_bytes_per_step": n * 32,
                        "d2h_bytes_per_step": 144, "api": "snarkvm_msm after snarkvm_b200_register_bases (bases resident)"}
        # and with the fixed-base tables of the registered slice built once (snarkvm_b200_register_bases_precomputed);
        # an extra, never the headline: a failure here (e.g. not enough HBM for the tables) is reported, not fatal
        try:
            t0 = time.perf_counter()
            shim.register_bases_precomputed(b_pin)
            setup_s = time.perf_counter() - t0
            try:
                assert (shim.msm(b_pin, s_pin) == expect).all()
                p_ms, _ = wall_timed(lambda: shim.msm(b_pin, s_pin), e2e_steps)
            finally:
                shim.unregister_bases(b_pin)
            e2e_resident["precomputed_tables"] = {"value": n / (p_ms * 1e-3), "unit": "points/s", "ms_per_step": p_ms,
                                                  "one_time_setup_s": setup_s,
                                                  "api": "snarkvm_msm after snarkvm_b200_register_bases_precomputed"}
        except Exception as exc:  # noqa: BLE001
            e2e_resident["precomputed_tables"] = {"error": repr(exc)}
    del bases_pin, b_pin

    # ---- BASELINE config 5a: 2^total_lg points sharded over the N GPUs (strong scaling: total work fixed) ----
    strong = None
    if args.total_lg and not args.skip_strong:
        tn = 1 << args.total_lg
        lo, hi = sharded.shard_range(tn, rank, world)
        shard_n = hi - lo
        plan_n = (tn + world - 1) // world
        sseed = 0x5A00 + rank
        sb = bases if shard_n == n else device.generate_bases(shard_n, seed=sseed, device=dev)
        if shard_n == n:
            sseed = seed
        ssc_np = scal_np if shard_n == n else random_scalars(shard_n, 4321 + rank)
        ssc = scalars if shard_n == n else torch.from_numpy(ssc_np.view(np.int64)).to(dev)
        sexpect = chk.point(sum_over_ranks_mod_r(chk.dot(ssc_np, sseed)))
        sfn = lambda: sharded.msm_sharded_async(sb, ssc, plan_npoints=plan_n)      # noqa: E731
        got = sfn().result()
        checks["msm_sharded_total"] = bool((got == sexpect).all())
        assert checks["msm_sharded_total"], "sharded 2^total MSM differs from the closed form"
        ssteps = max(2, min(args.steps, 5))
        s_ms, souts = timed(sfn, ssteps, lambda p: p.result())
        assert all((o == sexpect).all() for o in souts)
        strong = {"metric": "bls12_377_g1_msm_points_per_sec", "value": tn / (s_ms * 1e-3), "unit": "points/s", "scaling": "strong",
                  "workload": f"2^{args.total_lg} points in total, ⌈n/N⌉ per GPU, NCCL all-gather of window sums + device point-reduce",
                  "points_per_gpu": shard_n, "ms_per_step": s_ms, "steps": ssteps, "checked": True}
        del sb, ssc

    # ---- secondary metric: Fr NTT elements/s (per-GPU replicas; BASELINE config 3) ----
    ntt = None
    if not args.skip_ntt:
        from snarkvm_b200.cuda import NTTDirection, NTTType
        nn = 1 << args.ntt_lg
        x_np = random_scalars(nn, 99 + rank)
        x = torch.from_numpy(x_np.view(np.int64)).to(dev)
        scratch = torch.empty_like(x)
        y = device.ntt_(x.clone(), NTTDirection.Forward, NTTType.Standard, scratch)
        if rank == 0:
            checks["ntt_vs_oracle"] = bool((y.cpu().numpy().view(np.uint64) == chk.cpu.ntt(x_np, chk.cpu.FORWARD, chk.cpu.STANDARD)).all())
            assert checks["ntt_vs_oracle"], "NTT output differs from the oracle's fft_in_place"
        back = device.ntt_(y.clone(), NTTDirection.Inverse, NTTType.Standard, scratch)
        checks["ntt_round_trip"] = bool(torch.equal(back, x))
        assert checks["ntt_round_trip"]
        del y, back
        for _ in range(3):
            device.ntt_(x, NTTDirection.Forward, NTTType.Standard, scratch)
        _lib.profile_enable(True)
        _lib.profile_collect(_lib.PROF_NTT_PASS)
        reps = 10
        ntt_ms, _ = timed(lambda: device.ntt_(x, NTTDirection.Forward, NTTType.Standard, scratch), reps)
        pass_ms, pass_n = _lib.profile_collect(_lib.PROF_NTT_PASS)
        _lib.profile_enable(False)
        if args.dump_outputs:
            # x now holds the last timed transform's output: a fixed, seeded sample of its rows (Montgomery limbs)
            rows = np.sort(np.random.default_rng(0).choice(nn, size=min(nn, 1 << 16), replace=False))
            dumps["ntt_rows"] = rows.astype(np.float64)
            dumps["ntt"] = u64_as_f64(x[torch.from_numpy(rows).to(dev)].cpu().numpy().view(np.uint64))
        xs_page = np.empty((nn, 4), dtype=np.uint64); xs_page[:] = random_scalars(nn, 5)
        xs_pin_t = torch.from_numpy(xs_page.view(np.int64).copy()).pin_memory()
        xs_pin = xs_pin_t.numpy().view(np.uint64)
        ntt_e2e = {}
        e2e_in = torch.from_numpy(xs_page.view(np.int64)).to(dev)
        e2e_want = device.ntt_(e2e_in, NTTDirection.Forward, NTTType.Standard, scratch).cpu().numpy().view(np.uint64)   # the path checked against the oracle above
        del e2e_in
        for name, buf in (("pageable", xs_page), ("pinned", xs_pin)):
            shim.NTT(nn, buf, shim.NTTInputOutputOrder.NN, shim.NTTDirection.Forward, shim.NTTType.Standard)
            checks["ntt_e2e_" + name] = bool((buf == e2e_want).all())
            assert checks["ntt_e2e_" + name], "snarkvm_ntt (host buffer) differs from the device-resident transform"
            ms, _ = wall_timed(lambda: shim.NTT(nn, buf, shim.NTTInputOutputOrder.NN, shim.NTTDirection.Forward, shim.NTTType.Standard), 2)
            ntt_e2e[name] = ms
        per_pass_ms = pass_ms / max(1, pass_n)
        npass = pass_n // reps if reps else None
        ach = ALGO_BYTES_PER_ELEMENT * nn / (ntt_ms * 1e-3) / 1e9
        ntt = {
            "metric": "fr_ntt_elements_per_sec", "value": nn * world / (ntt_ms * 1e-3), "unit": "elements/s",
            "workload": f"forward NN NTT of 2^{args.ntt_lg} Fr elements per GPU (replicas, no collective)",
            "ms_per_transform": ntt_ms, "passes_per_transform": npass,
            "e2e": {"value": nn * world / (ntt_e2e["pageable"] * 1e-3), "unit": "elements/s", "h2d_bytes_per_step": nn * 32,
                    "d2h_bytes_per_step": nn * 32, "ms_per_step": ntt_e2e["pageable"], "api": "snarkvm_ntt (pageable host buffer)"},
            "e2e_pinned": {"value": nn * world / (ntt_e2e["pinned"] * 1e-3), "unit": "elements/s", "ms_per_step": ntt_e2e["pinned"]},
            "roofline": {"bound": "hbm", "kernel": "k_ntt_pass x%d (one transform)" % (npass or 0), "achieved": ach, "peak": peak, "unit": "GB/s",
                         "frac": ach / peak, "traffic": load_traffic("ntt_transform"), "per_launch_ms": ntt_ms,
                         "per_pass": {"ms": per_pass_ms, "achieved": ALGO_BYTES_PER_ELEMENT * nn / (per_pass_ms * 1e-3) / 1e9},
                         "note": "SURVEY §8(d): 64 B per element per TRANSFORM over the whole transform's duration; the butterflies are "
                                 "bound by the INT32 multiplier (1 Fr mul each), not by HBM"},
        }
        del x, scratch

    # ---- BASELINE config 4: KZG10 commit at 2^22 coefficients with hiding_bound = Some(1), operands resident ----
    kzg = None
    if not args.skip_kzg:
        nk = 1 << args.kzg_lg
        c_np = random_scalars(nk, 4242 + rank)                                   # Montgomery images of random coefficients
        b_np2 = random_scalars(3, 4343 + rank)                                   # blinding polynomial: degree hiding_bound + 1
        coeffs = torch.from_numpy(c_np.view(np.int64)).to(dev)
        blind = torch.from_numpy(b_np2.view(np.int64)).to(dev)
        powers = bases[:nk] if nk <= n else device.generate_bases(nk, seed=seed, device=dev)
        gseed = 0x6A00 + rank
        gamma = device.generate_bases(8, seed=gseed, device=dev)
        kexpect = chk.point(chk.dot(chk.cpu.fr_from_mont(c_np), seed) + chk.dot(chk.cpu.fr_from_mont(b_np2), gseed))
        kfn = lambda: device.kzg_commit_hiding(powers, coeffs, gamma, blind)     # noqa: E731
        checks["kzg_commit_hiding"] = bool((kfn() == kexpect).all())
        assert checks["kzg_commit_hiding"], "KZG hiding commitment differs from the closed form"
        for _ in range(2):
            kfn()
        kzg_ms, _ = timed(kfn, 5)
        kzg = {"metric": "kzg10_commit_coefficients_per_sec", "value": nk * world / (kzg_ms * 1e-3), "unit": "coefficients/s",
               "ms_per_commit": kzg_ms, "checked": True,
               "workload": f"KZG10::commit of a 2^{args.kzg_lg}-coefficient polynomial, hiding_bound = Some(1) (3 blinding terms in the same pass), "
                           f"powers resident in HBM, per GPU"}
        # a round of 8 commitments of 2^20 coefficients in ONE pass (sonic_pc/mod.rs:177-257)
        nb = 1 << 20
        if nb <= nk:
            polys = [coeffs[i * (nk // 8): i * (nk // 8) + nb] if (i * (nk // 8) + nb) <= nk else coeffs[:nb] for i in range(8)]
            polys = [p.contiguous() for p in polys]
            want0 = device.kzg_commit(powers, polys[0])
            got = device.kzg_commit_batch(powers, polys)
            checks["kzg_batch_vs_single"] = bool((got[0] == want0).all() and (got[7] == device.kzg_commit(powers, polys[7])).all())
            assert checks["kzg_batch_vs_single"]
            b_ms, _ = timed(lambda: device.kzg_commit_batch(powers, polys), 5)
            o_ms, _ = timed(lambda: device.kzg_commit(powers, polys[0]), 5)
            kzg["round_batch"] = {"value": 8 * nb * world / (b_ms * 1e-3), "unit": "coefficients/s", "ms_per_round": b_ms,
                                  "workload": "8 polynomials × 2^20 coefficients, one pass over the resident powers",
                                  "one_by_one_ms": 8 * o_ms, "single_2^20_ms": o_ms}
        if not args.skip_precomputed:
            t0 = time.perf_counter()
            pre = device.PrecomputedBases(powers)
            torch.cuda.synchronize()
            pre_s = time.perf_counter() - t0
            assert (pre.kzg_commit(coeffs) == device.kzg_commit(powers, coeffs)).all()
            for _ in range(2):
                pre.kzg_commit(coeffs)
            pre_ms, _ = timed(lambda: pre.kzg_commit(coeffs), 5)
            kzg["precomputed_tables"] = {"value": nk * world / (pre_ms * 1e-3), "unit": "coefficients/s", "ms_per_commit": pre_ms,
                                         "window_bits": pre.c, "windows": pre.nwin, "table_bytes": pre.table_bytes,
                                         "one_time_precompute_s": pre_s, "note": "plain (non-hiding) commitment over the tables"}
            if nb <= nk:
                gotp = pre.kzg_commit_batch(polys)
                checks["kzg_batch_tables_vs_single"] = bool((gotp[0] == want0).all() and (gotp[7] == device.kzg_commit(powers, polys[7])).all())
                assert checks["kzg_batch_tables_vs_single"]
                pb_ms, _ = timed(lambda: pre.kzg_commit_batch(polys), 5)
                kzg["precomputed_tables"]["round_batch"] = {"value": 8 * nb * world / (pb_ms * 1e-3), "unit": "coefficients/s", "ms_per_round": pb_ms,
                                                            "workload": "8 polynomials × 2^20 coefficients, one pass over the tables"}
            pre.free()
        # UniversalParams::lagrange_basis: iFFT over G1 points (data_structures.rs:68-72)
        ng = 1 << args.g1_ntt_lg
        gp = powers.reshape(-1)[: ng * 104].contiguous()
        device.lagrange_basis(gp)
        lb_ms, _ = timed(lambda: device.lagrange_basis(gp), 1)
        kzg["lagrange_basis"] = {"ms": lb_ms, "workload": f"ifft of 2^{args.g1_ntt_lg} G1 points per GPU", "unit": "ms"}

    # ---- BASELINE config 5b: Varuna prover rounds + round commitments on a synthetic R1CS, polynomials resident (SURVEY §8 f3) ----
    varuna_line = None
    if world == 1 and args.varuna_lg > 0:
        import importlib.util
        spec = importlib.util.spec_from_file_location("bench_varuna", os.path.join(ROOT, "tools", "bench_varuna.py"))
        bv = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(bv)
        varuna_line = bv.run(args.varuna_lg, reps=2)
        # the whole prove_batch-shaped pipeline: hiding mode, SonicKZG10 commits with degree / hiding bounds, linear combinations, openings
        varuna_line["prove"] = bv.run_prove(args.varuna_lg, reps=1)

    # ---- G2 (north_star "G1/G2"): VariableBase::msm over Affine<G2>, standard::msm semantics, closed-form check ----
    g2_line = None
    if world == 1 and args.g2_lg > 0:
        from oracle import g2 as og2
        ng2 = 1 << args.g2_lg
        g2seed = 0x62 + rank
        g2b = device.generate_bases_g2(ng2, g2seed, device=dev)
        g2s = random_scalars(ng2, 777)
        g2sd = torch.from_numpy(g2s.view(np.int64)).to(dev)
        got2 = device.msm_g2(g2b, g2sd)
        want2 = np.frombuffer(og2.g2_projective_bytes_normalised(og2.g2_mul(og2.G2_GEN, chk.dot(g2s, g2seed))), dtype=np.uint64)
        checks["g2_msm"] = bool((got2 == want2).all())
        assert checks["g2_msm"], "G2 MSM differs from the closed form"
        g2_ms, _ = timed(lambda: device.msm_g2(g2b, g2sd), 3)
        g2_line = {"metric": "bls12_377_g2_msm_points_per_sec", "value": ng2 / (g2_ms * 1e-3), "unit": "points/s", "ms_per_msm": g2_ms,
                   "checked": True, "workload": f"2^{args.g2_lg}-point VariableBase::msm over Affine<G2> (Fq2 coordinates, 200-byte images), resident"}
        del g2b, g2sd

    # ---- the same MSM at the sizes a prover calls it with (Varuna commits 2^12 … 2^21 coefficients): resident inputs, whole call
    #      (sort, accumulate, quad-lane reduction tail, D2H of the window sums, host Horner), each checked by the closed form ----
    sizes_line = None
    if world == 1 and not args.skip_sizes:
        sizes_line = {}
        for lg_s in (12, 14, 16, 18, 20, 22):
            if lg_s >= args.lg:
                continue
            ns = 1 << lg_s
            bs, ss = bases[:ns], scalars[:ns]
            got_s = device.msm(bs, ss)
            ok_s = bool((got_s == chk.point(chk.dot(scal_np[:ns], seed))).all())
            checks[f"msm_2^{lg_s}"] = ok_s
            assert ok_s, f"2^{lg_s}-point MSM differs from the closed form"
            reps_s = 20 if lg_s <= 18 else 5
            for _ in range(3):
                device.msm(bs, ss)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(reps_s):
                device.msm(bs, ss)
            ms_s = (time.perf_counter() - t0) / reps_s * 1e3
            sizes_line[f"2^{lg_s}"] = {"ms_per_msm": ms_s, "points_per_s": ns / (ms_s * 1e-3)}

    if rank != 0:
        return

    # ---- cpu_baseline: the oracle port on this box's host cores, bounded sample (N = 1 only) ----
    cpu_baseline = None
    if world == 1 and not args.skip_cpu:
        cpu = chk.cpu
        lg_s = min(args.cpu_lg, args.lg)
        hb = bases[: 1 << lg_s].cpu().numpy()
        v, dt = cpu_msm_points_per_s(cpu, hb, scal_np[: 1 << lg_s])
        cpu_baseline = {"value": v, "unit": "points/s", "cores": cpu.num_threads(), "kind": "port",
                        "sample": f"one 2^{lg_s}-point batched::msm ({dt:.1f} s) on the first 2^{lg_s} points and scalars of the GPU's input — "
                                  f"C restatement of the reference CPU path, OpenMP task per window"}
        if ntt is not None:
            nv, ndt, nth = cpu_ntt_elements_per_s(cpu, args.cpu_ntt_lg)
            ntt["cpu_baseline"] = {"value": nv, "unit": "elements/s", "cores": nth, "kind": "port",
                                   "sample": f"one 2^{args.cpu_ntt_lg} forward fft_in_place ({ndt:.2f} s), best team size of 16/32/64/all"}

    plan = device.msm_plan(n)
    plan_levels = plan["levels"]
    cfg = workload_config(args, world)
    line = {
        "metric": "bls12_377_g1_msm_points_per_sec", "value": value, "unit": "points/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u32 limbs (Montgomery integer arithmetic, IMAD pipe)",
        "data": "synthetic", "config": cfg,
        "plan": {"window_bits": plan["c"], "windows": plan["nwin"], "pair_levels": plan_levels,
                 "l2": f"inputs ({n * 136 / 1e9:.2f} GB/step) plus {n * plan['nwin'] * 96 / 1e9:.1f} GB of scattered level-0 records and the dense "
                       f"pair-level scratch stream through the 126 MB L2 every step — no flush needed"},
        "checked": all(checks.values()), "checks": checks,
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "points/s", "h2d_bytes_per_step": n * (104 + 32) * world,
                "d2h_bytes_per_step": (144 if world == 1 else plan["nwin"] * 192) * world, "ms_per_step": e2e_ms, "steps": e2e_steps,
                "host_memory": "pageable (plain malloc, what a Rust Vec is); staged through the library's pinned ring",
                "api": "snarkvm_msm (drop-in C-ABI)" if world == 1 else "sharded.msm_sharded_async on host buffers (snarkvm_b200_msm_window_sums_host + NCCL)"},
        "e2e_pinned": {"value": n * world / (e2e["pinned"] * 1e-3), "unit": "points/s", "ms_per_step": e2e["pinned"],
                       "host_memory": "pinned (cudaHostAlloc)"},
        "e2e_registered_bases": e2e_resident,
        "sharded_total": strong,
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "kernel": "bucket accumulation phase: k_pair_level2 x%d + k_bucket_accumulate%s (level-0 records written by k_scatter_records in the sort phase)" % (
                         plan_levels, "_dense" if plan_levels else ""),
                     "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": load_traffic("msm_bucket_accumulation_phase") if args.lg == 24 else None,
                     "peak_source": peak_src, "per_launch_ms": acc_ms_per_step,
                     "share_of_step": {"sort": sort_ms / ms_total, "accumulate": acc_ms / ms_total, "reduce": red_ms / ms_total},
                     "note": "algorithmic 128 B/point over the phase's duration; the phase is bound by the INT32 multiplier (fmaheavy pipe, "
                             "profiles/), not by HBM"},
        "cpu_baseline": cpu_baseline,
        "ntt": ntt,
        "kzg_commit": kzg,
        "varuna": varuna_line,
        "g2_msm": g2_line,
        "msm_sizes": sizes_line,
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dumps)
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--lg", type=int, default=24, help="log2 points per GPU (BASELINE configs[1]: 2^20/2^22/2^24)")
    ap.add_argument("--total-lg", type=int, default=26, help="BASELINE config 5a: total points of the strong-scaling sharded MSM (0 = skip)")
    ap.add_argument("--ntt-lg", type=int, default=24)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-lg", type=int, default=24, help="cpu_baseline sample size (bounded: 2^24 points ≈ 12 s on 64 cores)")
    ap.add_argument("--cpu-ntt-lg", type=int, default=22)
    ap.add_argument("--ref-lg", type=int, default=0, help="--impl reference: log2 points per step (0 = the workload's size if the run stays within a few minutes, else the largest bounded sample that does)")
    ap.add_argument("--ref-ntt-lg", type=int, default=22)
    ap.add_argument("--kzg-lg", type=int, default=22)
    ap.add_argument("--varuna-lg", type=int, default=18, help="log2 constraints of the Varuna prover-rounds extra (0 = skip)")
    ap.add_argument("--g2-lg", type=int, default=16, help="log2 points of the G2 MSM extra (0 = skip)")
    ap.add_argument("--g1-ntt-lg", type=int, default=16, help="size of the G1 iFFT (lagrange_basis) timed inside the KZG extra")
    ap.add_argument("--skip-kzg", action="store_true")
    ap.add_argument("--skip-sizes", action="store_true")
    ap.add_argument("--skip-ntt", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-strong", action="store_true")
    ap.add_argument("--skip-registered", action="store_true")
    ap.add_argument("--skip-precomputed", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step returned as DIR/<name>.npy: msm.npy (the G1 MSM result) and, "
                         "unless --skip-ntt, ntt.npy (a seeded sample of 2^16 rows of the last timed NTT output, their indices in "
                         "ntt_rows.npy); uint64 limbs are stored as their little-endian 32-bit words in float64, which is exact")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs records the product path (--impl b200)")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_product(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
