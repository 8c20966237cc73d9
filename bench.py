#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 hot path (see BASELINE.json / SURVEY.md 8d).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload NAME] [--batch B] [--dump-outputs DIR]

A "step" is one pass of the hot path -- CKKS Evaluator::multiply + relinearize_inplace -- over one batch of synthetic
uniform-random ciphertexts (as native/bench does: bench.h:195-270) that is already resident in HBM.  Under torchrun
every rank processes its own shard of the batch on its own GPU (weak scaling, no data-path collective; rank 0 broadcasts
the relinearization key once at setup and gathers per-ciphertext digests at the end, both NCCL).  Rank 0 prints ONE JSON line.

  value     whole-job ciphertexts/s, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e       same metric through the host-buffer C-ABI call (pinned host buffers, H2D + D2H inside the timed region)
  verified  sampled outputs of the TIMED run (both sides of a key-switching chunk boundary, first and last ciphertext) compared
            word for word with the reference's own Evaluator (oracle/_ref); a mismatch aborts the run with a non-zero status
  roofline  SURVEY 8(d) accounting: compulsory bytes of the fused operation (6*L*n*8 per ciphertext + one pass over the key per
            B_reuse ciphertexts) over the measured time, the DRAM traffic of the whole step from the committed ncu capture
            (step_traffic), plus the second ceiling (integer-multiply issue rate: 64-bit and 32-bit butterflies / multiply-accumulates)
            measured in process
  configs   BASELINE.json configs[1..3] (cfg2 batch multiply+relinearize, cfg3 depth-8 chain, cfg4 rotate sweep) and the shape the
            metric text names (n=65536, 16 primes): device-resident and end-to-end rates, each with its own verification (N=1 only)
  cpu_baseline  the reference's own CPU implementation (oracle/_ref, i.e. SEAL 4.4.3 compiled from its sources, HEXL off)
                on this box's host cores, bounded sample, best of {physical cores, all hardware threads}

--impl reference times that CPU implementation alone, on the same workload/metric.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOADS = {
    # BASELINE.json configs[4] (the config the metric is quoted on): CKKS n=65536, 32 primes, multiply+relinearize;
    # 8192 ciphertexts over 8 GPUs = 1024 per GPU.  Fits one GPU: 2 x 33.3 GB in + 33.3 GB out + scratch.
    "ckks_n65536_k32": dict(scheme=2, n=65536, bits=[55] * 32, batch=1024, e2e_batch=64, cpu_reps=1),
    # BASELINE.json configs[1]
    "ckks_n8192_k4": dict(scheme=2, n=8192, bits=[54] * 4, batch=1024, e2e_batch=256, cpu_reps=200),
    # metric text "n=2^16, L=16 primes"
    "ckks_n65536_k16": dict(scheme=2, n=65536, bits=[55] * 16, batch=1024, e2e_batch=32, cpu_reps=2),
    # diagnostic shape: the headline's prime count at a degree whose rows are 8x shorter (same bytes per step at 8x the batch)
    "ckks_n8192_k32": dict(scheme=2, n=8192, bits=[55] * 32, batch=2048, e2e_batch=64, cpu_reps=8),
    "ckks_n32768_k16": dict(scheme=2, n=32768, bits=[55] * 15 + [56], batch=256, e2e_batch=64, cpu_reps=4),
    # tiny shape for the CPU contract test of the reference arm (tests/test_bench_contract.py); not a bench line
    "smoke": dict(scheme=2, n=4096, bits=[40, 40, 40], batch=8, e2e_batch=4, cpu_reps=4),
}
METRIC = "CKKS multiply+relinearize ciphertexts/s"
UNIT = "ciphertexts/s"


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel):
    """dram bytes per launch of a kernel from the committed ncu capture summary (and the batch it was captured at), or None"""
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            return json.load(f).get(kernel)
    except Exception:
        return None


# ---------------------------------------------------------------------------------------------- host facts ----
def host_threads():
    """threads this process may really use: the affinity mask, bounded by the cgroup CPU quota"""
    n = len(os.sched_getaffinity(0))
    try:
        q = open("/sys/fs/cgroup/cpu.max").read().split()
        if q[0] != "max":
            n = max(1, min(n, int(float(q[0]) / float(q[1]))))
    except Exception:
        pass
    return n


def cpu_facts():
    """(model name, physical cores inside the affinity mask, hardware threads usable)"""
    model, cores = "unknown", set()
    allowed = os.sched_getaffinity(0)
    try:
        cur = {}
        for line in open("/proc/cpuinfo"):
            if ":" in line:
                k, v = [x.strip() for x in line.split(":", 1)]
                cur[k] = v
            elif cur:
                if int(cur.get("processor", -1)) in allowed:
                    cores.add((cur.get("physical id", "0"), cur.get("core id", cur.get("processor"))))
                    model = cur.get("model name", model)
                cur = {}
        if cur and int(cur.get("processor", -1)) in allowed:
            cores.add((cur.get("physical id", "0"), cur.get("core id", cur.get("processor"))))
    except Exception:
        pass
    t = host_threads()
    return model, max(1, min(len(cores) or t, t)), t


def cpu_reference_rate(rc, op, L, reps):
    """reference throughput on the host: best of {one thread per physical core, every hardware thread}; HEXL off"""
    model, phys, threads = cpu_facts()
    rc.time_op(op, L, min(4, threads), 1)  # warm the code paths and the thread-local pools' first touch
    sweep = []
    for t in sorted({phys, threads}):
        secs = rc.time_op(op, L, t, reps)
        sweep.append({"threads": t, "value": t * reps / secs, "per_thread": reps / secs})
    best = max(sweep, key=lambda s: s["value"])
    return {"value": best["value"], "unit": UNIT, "cores": best["threads"], "kind": "reference", "cpu_model": model,
            "physical_cores": phys, "hardware_threads": threads, "per_thread": best["per_thread"], "sweep": sweep,
            "sample": f"{best['threads'] * reps} ciphertexts, {best['threads']} threads x {reps}, SEAL 4.4.3 built from its own sources "
                      f"(oracle/_ref), HEXL off (not installable here)"}


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            self.p.kill()
            out = ""
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        # median of the upper half = clocks under load (idle samples before/after the region pull the plain median down)
        load = sm[len(sm) // 2:] if sm else []
        return {"sm_mhz": (load[len(load) // 2] if load else None), "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def gpu_numa_cpus(dev):
    """(node, cpus) of the NUMA node the GPU's PCIe root port hangs off, or (None, None) when the box does not say"""
    try:
        import torch

        p = torch.cuda.get_device_properties(dev)
        addr = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{addr}/numa_node").read())
        if node < 0:
            return None, None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        return (node, cpus) if cpus else (None, None)
    except Exception:
        return None, None


def run_reference(args, wl, rank, world):
    """--impl reference: the reference's own CPU implementation (oracle/_ref) on the host cores."""
    if rank != 0:
        return
    import refseal as R

    if not R.available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libsealref.so missing (build it with oracle/Makefile)"}))
        return
    mods = R.coeff_modulus_create(wl["n"], wl["bits"])
    L = len(mods) - 1
    t0 = time.time()
    rc = R.RefContext(wl["scheme"], wl["n"], mods)
    rc.relin_key()
    setup_s = time.time() - t0
    reps = wl["cpu_reps"]
    model, phys, threads = cpu_facts()
    rc.time_op(0, L, min(4, threads), 1)
    # pick the better thread count once (one untimed probe each), then time K steps with it
    probe = {t: t * reps / rc.time_op(0, L, t, reps) for t in sorted({phys, threads})} if args.warmup > 0 else {threads: 0.0}
    cores = max(probe, key=probe.get)
    total_t, total_ops = 0.0, 0
    for _ in range(args.steps):
        total_t += rc.time_op(0, L, cores, reps)
        total_ops += cores * reps
    v = total_ops / total_t
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total_t / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
        "data": "synthetic", "config": {"workload": args.workload, "n": wl["n"], "coeff_modulus_primes": len(mods), "L": L,
                                        "ops": "Evaluator::multiply_inplace + relinearize_inplace", "step": f"{cores} threads x {reps} ciphertexts"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "reference", "cpu_model": model, "physical_cores": phys,
                         "hardware_threads": threads, "per_thread": v / cores,
                         "thread_sweep": [{"threads": t, "value": r} for t, r in sorted(probe.items())],
                         "sample": f"{total_ops} ciphertexts on {cores} threads (SEAL 4.4.3 from oracle/_ref, HEXL off: not installable here); "
                                   f"setup {setup_s:.1f}s excluded; thread count = best of one probe at {sorted(probe)}"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ shared helpers ----
def device_rand(torch, mods, n, shape_prefix, L, gen):
    """uniform residues in [0, q_i) per RNS row, generated on the device: [*shape_prefix][L][n]"""
    t = torch.empty((*shape_prefix, L, n), dtype=torch.int64, device="cuda")
    for i in range(L):
        t[..., i, :] = torch.randint(0, mods[i], (*shape_prefix, n), generator=gen, dtype=torch.int64, device="cuda")
    return t


def to_np(t):
    import numpy as np

    return t.cpu().numpy().view(np.uint64)


def fail(msg):
    sys.stderr.write("bench.py: VERIFICATION FAILED: " + msg + "\n")
    sys.stderr.flush()
    os._exit(3)


def dump_outputs(path, out, np, max_ciphertexts=8, max_coeffs=4096):
    """Write a fixed sample of the device-resident result out[batch][2][L][n] (residue words below 2^63) to path/*.npy, so that
    two builds can be compared output for output: the same seeded ciphertext and coefficient indices on every run, the first and
    last ciphertext always among them.  float64 holds 53 bits, so each word is stored exactly as its high and low 32 bits
    (multiply_relinearize_hi32.npy, multiply_relinearize_lo32.npy, shape [ciphertexts][2][L][coefficients]); the sampled indices
    are written beside them.  At most 8 x 2 x L x 4096 words, 32 MB for L = 31."""
    import torch

    B, n = out.shape[0], out.shape[-1]
    rng = np.random.default_rng(0xD0)
    inner = rng.choice(np.arange(1, B - 1), size=min(max(B - 2, 0), max_ciphertexts - 2), replace=False)
    cts = sorted({0, B - 1} | {int(i) for i in inner})
    cols = np.sort(rng.choice(n, size=min(n, max_coeffs), replace=False))
    sample = out[torch.tensor(cts, device=out.device)][..., torch.from_numpy(cols).to(out.device)]
    words = sample.cpu().numpy().view(np.uint64)
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "multiply_relinearize_hi32.npy"), (words >> np.uint64(32)).astype(np.float64))
    np.save(os.path.join(path, "multiply_relinearize_lo32.npy"), (words & np.uint64(0xFFFFFFFF)).astype(np.float64))
    np.save(os.path.join(path, "sample_ciphertexts.npy"), np.array(cts, dtype=np.float64))
    np.save(os.path.join(path, "sample_coefficients.npy"), cols.astype(np.float64))


def timed(torch, fn, steps, warmup=1):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps * 1e-3


# ------------------------------------------------------------------- BASELINE.json configs[1..3] (N = 1) ----
def run_cfg2(S, R, torch, np):
    """CKKS n=8192, 4 primes, batch 1024: multiply + relinearize"""
    n, batch, L = 8192, 1024, 3
    mods = R.coeff_modulus_create(n, [54] * 4)
    rc = R.RefContext(R.CKKS, n, mods)
    ctx = S.Context(S.CKKS, n, mods)
    rk = ctx.load_key(rc.relin_key())
    g = torch.Generator(device="cuda")
    g.manual_seed(2)
    a, b = device_rand(torch, mods, n, (batch, 2), L, g), device_rand(torch, mods, n, (batch, 2), L, g)
    out = torch.empty_like(a)
    sec = timed(torch, lambda: ctx.d_multiply_relinearize(a, b, rk, out, L, batch), 5, 2)
    ha, hb, ho = a.cpu().pin_memory(), b.cpu().pin_memory(), torch.empty_like(a, device="cpu").pin_memory()
    na, nb, no = (x.numpy().view(np.uint64) for x in (ha, hb, ho))

    def e2e():
        S._check(S.lib().sb200_multiply_relinearize_host(ctx.h, L, batch, S._hp(na), S._hp(nb), rk.h, S._hp(no)))

    e2e()
    t0 = time.perf_counter()
    for _ in range(3):
        e2e()
    e2e_sec = (time.perf_counter() - t0) / 3
    idx = [0, 1, batch // 2, batch - 1]
    for i in idx:
        want = rc.multiply_relin(L, to_np(a[i]), to_np(b[i]))
        if not (to_np(out[i]) == want).all() or not (no[i] == want).all():
            fail(f"cfg2 ciphertext {i}")
    return {"config": "CKKS n=8192, 4 primes, batch 1024, multiply+relinearize", "value": batch / sec, "unit": UNIT,
            "e2e": {"value": batch / e2e_sec, "unit": UNIT, "h2d_bytes_per_step": int(ha.nbytes + hb.nbytes), "d2h_bytes_per_step": int(ho.nbytes)},
            "verified": {"indices": idx, "ok": True, "against": "oracle/_ref (reference Evaluator), device-resident and host-buffer results"}}


def run_k16(S, R, torch, np):
    """the shape BASELINE.json's metric text names ("n=2^16, L=16 primes"): CKKS n=65536, 16 primes, batch 512: multiply + relinearize"""
    n, batch = 65536, 512
    mods = R.coeff_modulus_create(n, [55] * 16)
    L = len(mods) - 1
    rc = R.RefContext(R.CKKS, n, mods)
    ctx = S.Context(S.CKKS, n, mods)
    free_b, _ = torch.cuda.mem_get_info()
    ctx.set_limit(ctx.LIMIT_SCRATCH_BYTES, int(max(8 << 30, min(free_b - (40 << 30), 64 << 30))))
    rk = ctx.load_key(rc.relin_key())
    g = torch.Generator(device="cuda")
    g.manual_seed(16)
    a, b = device_rand(torch, mods, n, (batch, 2), L, g), device_rand(torch, mods, n, (batch, 2), L, g)
    out = torch.empty_like(a)
    sec = timed(torch, lambda: ctx.d_multiply_relinearize(a, b, rk, out, L, batch), 3, 2)
    idx = [0, batch - 1]
    for i in idx:
        if not (to_np(out[i]) == rc.multiply_relin(L, to_np(a[i]), to_np(b[i]))).all():
            fail(f"k16 ciphertext {i}")
    return {"config": "CKKS n=65536, 16 primes, batch 512, multiply+relinearize (device-resident)", "value": batch / sec, "unit": UNIT,
            "ciphertexts_per_key_pass": ctx.keyswitch_chunk(L, batch, True),
            "verified": {"indices": idx, "ok": True, "against": "oracle/_ref (reference Evaluator)"}}


def run_cfg3(S, R, torch, np):
    """CKKS n=32768, 16 primes, batch 256: a <- rescale(relin(a*b)); b <- mod_switch_to_next(b), depth 8 (SURVEY 8d)"""
    n, batch, depth = 32768, 256, 8
    mods = R.coeff_modulus_bfv_default(n)
    L0 = len(mods) - 1
    rc = R.RefContext(R.CKKS, n, mods)
    ctx = S.Context(S.CKKS, n, mods)
    rk = ctx.load_key(rc.relin_key())
    g = torch.Generator(device="cuda")
    g.manual_seed(3)
    a0, b0 = device_rand(torch, mods, n, (batch, 2), L0, g), device_rand(torch, mods, n, (batch, 2), L0, g)
    # level buffers allocated once: the chain itself allocates nothing
    bufs = [[torch.empty((batch, 2, L0 - d, n), dtype=torch.int64, device="cuda") for d in range(depth + 1)] for _ in range(2)]
    prod = torch.empty((batch, 2, L0, n), dtype=torch.int64, device="cuda")

    def chain(a_in, b_in):
        a, b, L = a_in, b_in, L0
        for d in range(depth):
            p = prod.view(-1)[: batch * 2 * L * n].view(batch, 2, L, n)
            ctx.d_multiply_relinearize(a, b, rk, p, L, batch)
            na_, nb_ = bufs[0][d + 1], bufs[1][d + 1]
            ctx.d_rescale_to_next(p, na_, L, batch)
            ctx.d_mod_switch_to_next(b, nb_, L, batch)
            a, b, L = na_, nb_, L - 1
        return a, b

    sec = timed(torch, lambda: chain(a0, b0), 3, 1)
    ra, rb = chain(a0, b0)
    torch.cuda.synchronize()
    ra, rb = ra.clone(), rb.clone()
    # end to end: operands start in pinned host memory, the two results end there; the chain stays on the device in between.
    # The batch flows in 4 slices: the H2D copy of slice k+1 and the D2H copy of slice k-1 run on their own streams while the
    # device works on slice k (every slice has its own level buffers).
    ha, hb = a0.cpu().pin_memory(), b0.cpu().pin_memory()
    hra, hrb = torch.empty_like(ra, device="cpu").pin_memory(), torch.empty_like(rb, device="cpu").pin_memory()
    nsl = 4
    per = batch // nsl
    s_in, s_out, s_cmp = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.current_stream()
    sl_in = [(torch.empty((per, 2, L0, n), dtype=torch.int64, device="cuda"), torch.empty((per, 2, L0, n), dtype=torch.int64, device="cuda"))
             for _ in range(nsl)]
    sl_bufs = [[[torch.empty((per, 2, L0 - d, n), dtype=torch.int64, device="cuda") for d in range(depth + 1)] for _ in range(2)] for _ in range(nsl)]
    sl_prod = torch.empty((per, 2, L0, n), dtype=torch.int64, device="cuda")

    def chain_slice(k):
        a, b, L = sl_in[k][0], sl_in[k][1], L0
        for d in range(depth):
            p = sl_prod.view(-1)[: per * 2 * L * n].view(per, 2, L, n)
            ctx.d_multiply_relinearize(a, b, rk, p, L, per)
            na_, nb_ = sl_bufs[k][0][d + 1], sl_bufs[k][1][d + 1]
            ctx.d_rescale_to_next(p, na_, L, per)
            ctx.d_mod_switch_to_next(b, nb_, L, per)
            a, b, L = na_, nb_, L - 1
        return a, b

    def e2e():
        ups, dones = [], []
        for k in range(nsl):
            with torch.cuda.stream(s_in):
                sl_in[k][0].copy_(ha[k * per:(k + 1) * per], non_blocking=True)
                sl_in[k][1].copy_(hb[k * per:(k + 1) * per], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(s_in)
                ups.append(ev)
        for k in range(nsl):
            s_cmp.wait_event(ups[k])
            xa, xb = chain_slice(k)
            ev = torch.cuda.Event()
            ev.record(s_cmp)
            with torch.cuda.stream(s_out):
                s_out.wait_event(ev)
                hra[k * per:(k + 1) * per].copy_(xa, non_blocking=True)
                hrb[k * per:(k + 1) * per].copy_(xb, non_blocking=True)
        torch.cuda.synchronize()

    e2e()
    t0 = time.perf_counter()
    for _ in range(2):
        e2e()
    e2e_sec = (time.perf_counter() - t0) / 2
    idx = [0, batch - 1]
    for i in idx:
        wa, wb, L = to_np(a0[i]), to_np(b0[i]), L0
        for _ in range(depth):
            wa = rc.rescale(L, rc.multiply_relin(L, wa, wb))
            wb = rc.mod_switch(L, wb)
            L -= 1
        if not ((to_np(ra[i]) == wa).all() and (to_np(rb[i]) == wb).all() and (hra[i].numpy().view(np.uint64) == wa).all()):
            fail(f"cfg3 chain, ciphertext {i}")
    return {"config": "CKKS n=32768, 16 primes, batch 256, depth-8 chain of multiply+relinearize+rescale (+ mod_switch_to_next of b)",
            "value": batch * depth / sec, "unit": "chain steps (multiply+relinearize+rescale)/s", "chains_per_s": batch / sec,
            "e2e": {"value": batch * depth / e2e_sec, "unit": "chain steps/s", "h2d_bytes_per_step": int(ha.nbytes + hb.nbytes),
                    "d2h_bytes_per_step": int(hra.nbytes + hrb.nbytes), "e2e_over_device": sec / e2e_sec, "slices": nsl,
                    "note": "host operands in, host results out; copies of neighbouring slices overlap the chain of the current one"},
            "verified": {"indices": idx, "ok": True, "against": "oracle/_ref: the same 8-level chain on the reference Evaluator"}}


def run_cfg4(S, R, torch, np):
    """BFV n=16384, 8 primes, batch 512: rotate_rows over every Galois element of create_galois_keys()"""
    n, batch, L = 16384, 512, 7
    mods = R.coeff_modulus_create(n, [54] * 8)
    t = R.plain_modulus_batching(n, 20)
    rb = R.RefContext(R.BFV, n, mods, t)
    ctx = S.Context(S.BFV, n, mods, t)
    steps = [0] + [s * (1 << k) for k in range(13) for s in (1, -1) if (1 << k) < n // 2]
    elts = sorted({rb.galois_elt_from_step(s) for s in steps})
    keys = {e: ctx.load_key(rb.galois_key(e)) for e in elts}
    g = torch.Generator(device="cuda")
    g.manual_seed(4)
    a = device_rand(torch, mods, n, (batch, 2), L, g)
    out = torch.empty_like(a)

    def sweep():
        for e in elts:
            ctx.d_apply_galois(a, e, keys[e], out, L, batch)

    sec = timed(torch, sweep, 2, 1)
    ha, ho = a.cpu().pin_memory(), torch.empty_like(a, device="cpu").pin_memory()
    na, no = ha.numpy().view(np.uint64), ho.numpy().view(np.uint64)
    sub = elts[:: max(1, len(elts) // 4)][:4]  # the end-to-end leg runs a few of the elements (every call moves the whole batch both ways)
    S._check(S.lib().sb200_apply_galois_host(ctx.h, L, batch, S._hp(na), sub[0], keys[sub[0]].h, S._hp(no)))
    t0 = time.perf_counter()
    for e in sub:
        S._check(S.lib().sb200_apply_galois_host(ctx.h, L, batch, S._hp(na), e, keys[e].h, S._hp(no)))
    e2e_sec = (time.perf_counter() - t0) / len(sub)
    checked = []
    for e in (elts[0], elts[len(elts) // 2], elts[-1]):
        ctx.d_apply_galois(a, e, keys[e], out, L, batch)
        torch.cuda.synchronize()
        for i in (0, batch - 1):
            if not (to_np(out[i]) == rb.apply_galois(L, to_np(a[i]), e)).all():
                fail(f"cfg4 galois element {e}, ciphertext {i}")
        checked.append(e)
    return {"config": f"BFV n=16384, 8 primes, batch 512, rotate_rows sweep over all {len(elts)} Galois elements",
            "value": batch * len(elts) / sec, "unit": "rotations/s", "sweeps_per_s": 1.0 / sec,
            "e2e": {"value": batch / e2e_sec, "unit": "rotations/s", "h2d_bytes_per_step": int(ha.nbytes), "d2h_bytes_per_step": int(ho.nbytes),
                    "elements_timed": len(sub)},
            "verified": {"galois_elements": checked, "indices": [0, batch - 1], "ok": True, "against": "oracle/_ref Evaluator::apply_galois"}}


def run_cpp_harness():
    """end-to-end figures measured through the C++ drop-in class (tests/cpp/chain_bench.cpp, built where the reference headers are)"""
    exe = os.path.join(ROOT, "tests", "cpp", "_bin", "chain_bench")
    if not os.path.exists(exe):
        return {"unavailable": "tests/cpp/_bin/chain_bench not built"}
    try:
        r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
        for line in reversed(r.stdout.strip().splitlines()):
            if line.startswith("{"):
                return json.loads(line)
        return {"unavailable": f"no result line (rc {r.returncode}): {(r.stdout + r.stderr)[-300:]}"}
    except Exception as e:  # noqa: BLE001
        return {"unavailable": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="ckks_n65536_k32", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="ciphertexts per GPU per step (default: the workload's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the BASELINE.json cfg2-cfg4 lines and the C++ harness")
    ap.add_argument("--no-verify", action="store_true", help="skip the comparison with the reference (profiling runs only)")
    ap.add_argument("--ks-algo", type=int, default=None, choices=[0, 1, 2],
                    help="key switching: 0 = 64-bit digit transforms, 1 = automatic (library default: the integer convolution on auxiliary "
                         "primes from 6 digits on), 2 = the integer path at every level")
    ap.add_argument("--scratch-gib", type=float, default=0.0, help="key-switching scratch budget (0: what the device has left, at most 64 GiB)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a fixed sample of the last timed step's output ciphertexts to DIR/*.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    wl = dict(WORKLOADS[args.workload])
    if args.batch:
        wl["batch"] = args.batch
        wl["e2e_batch"] = min(wl["e2e_batch"], args.batch)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, wl, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    import refseal as R
    import seal_b200 as S

    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n, B = wl["n"], wl["batch"]
    mods = S.coeff_modulus_create(n, wl["bits"])
    k, L = len(mods), len(mods) - 1
    ctx = S.Context(wl["scheme"], n, mods, device=local)
    if args.ks_algo is not None:
        ctx.set_limit(ctx.LIMIT_KS_ALGORITHM, args.ks_algo)
    aux_primes = ctx.ksint_primes() if (args.ks_algo != 0 and (L >= 6 or args.ks_algo == 2)) else []
    g = torch.Generator(device="cuda")
    g.manual_seed(0x5EA1 + rank)

    # ---- the key: the reference's own relinearization key when the reference library is here (so that the timed outputs can be
    #      compared with the reference Evaluator), generated on rank 0 and broadcast; uniform residues otherwise
    use_ref = R.available() and not args.no_verify
    rc = None
    key_dev = torch.empty((L, 2, k, n), dtype=torch.int64, device="cuda")
    if rank == 0:
        if use_ref:
            rc = R.RefContext(wl["scheme"], n, mods)
            key_dev.copy_(torch.from_numpy(rc.relin_key().view(np.int64)))
        else:
            key_dev.copy_(device_rand(torch, mods, n, (L, 2), k, g))
    if world > 1:
        dist.broadcast(key_dev, 0)  # "tables + keys replicated (one broadcast from rank 0 at setup)", SURVEY 8(e)
    key_np = to_np(key_dev)
    rk = ctx.load_key(key_np)
    del key_dev
    if use_ref or args.no_verify or rank != 0:
        key_np = None
    a, b = device_rand(torch, mods, n, (B, 2), L, g), device_rand(torch, mods, n, (B, 2), L, g)
    out = torch.empty((B, 2, L, n), dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    # key-switching scratch: what the device has left after the batch is resident (180 GB HBM3e), so that one pass over the 1 GB key
    # serves as many ciphertexts as possible (B_reuse of SURVEY 8d); the library default is 8 GiB
    free_b, _ = torch.cuda.mem_get_info()
    scratch_budget = int(args.scratch_gib * 2**30) if args.scratch_gib > 0 else int(max(8 << 30, min(free_b - (6 << 30), 64 << 30)))
    ctx.set_limit(ctx.LIMIT_SCRATCH_BYTES, scratch_budget)

    def step():
        ctx.d_multiply_relinearize(a, b, rk, out, L, B)

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    launches0 = ctx.launch_count
    ctx.profile(True)
    sampler = ClockSampler(local) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    clocks = sampler.stop() if sampler else None
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    launches = ctx.launch_count - launches0
    prof = ctx.profile_read_work32()
    ctx.profile(False)

    # ---- verification of the timed run's outputs against the reference Evaluator (rank 0's shard; the other ranks run the
    #      same library on their own inputs and contribute their digests below)
    chunk = ctx.keyswitch_chunk(L, B, True)
    verified = None
    if rank == 0 and not args.no_verify:
        idx = sorted({0, min(chunk, B) - 1, min(chunk, B - 1), B - 1})
        if rc is not None:
            from concurrent.futures import ThreadPoolExecutor

            ins = [(to_np(a[i]), to_np(b[i])) for i in idx]
            with ThreadPoolExecutor(len(idx)) as ex:
                wants = list(ex.map(lambda p: rc.multiply_relin(L, p[0], p[1]), ins))
            against = "oracle/_ref: Evaluator::multiply_inplace + relinearize_inplace of the unmodified reference, same key and inputs"
        else:
            import oracle as O  # the reference library did not travel: the plain-C restatement checks one ciphertext

            idx = idx[:1]
            oc = O.Oracle(wl["scheme"], n, mods)
            wants = [oc.multiply_relin(L, to_np(a[i]), to_np(b[i]), key_np) for i in idx]
            against = "oracle/liboracle.so (plain-C restatement; oracle/_ref absent), synthetic key"
        for i, want in zip(idx, wants):
            if not (to_np(out[i]) == want).all():
                fail(f"{args.workload} ciphertext {i} of the timed run differs from the reference")
        verified = {"indices": idx, "ok": True, "chunk": chunk, "chunks_per_step": -(-B // chunk), "against": against}
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, out, np)

    # end-of-run gather (the only collective besides the key broadcast): one 64-bit digest per ciphertext of this rank's last step
    from seal_b200.shard import digest as ct_digest, gather_digests

    digests = gather_digests(ct_digest(out), rank, world)  # NCCL over NVLink when world > 1
    torch.cuda.synchronize()
    assert rank != 0 or digests.numel() == B * world

    # ---- second headline metric: NTT GB/s vs the HBM roofline (Evaluator::transform_from_ntt_inplace + transform_to_ntt_inplace
    #      over the whole input slab, the reference bench's NTTForward/NTTInverse cases; 2*n*8 algorithmic bytes per row per transform)
    nb = min(B, 64)
    ntt_rows = nb * 2 * L
    ctx.d_ntt_inverse(a, L, 2, nb)
    ctx.d_ntt_forward(a, L, 2, nb)
    torch.cuda.synchronize()
    n0, n1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n0.record()
    for _ in range(args.steps):
        ctx.d_ntt_inverse(a, L, 2, nb)
        ctx.d_ntt_forward(a, L, 2, nb)  # restores the slab exactly (checked by the parity tests)
    n1.record()
    torch.cuda.synchronize()
    ntt_ms = n0.elapsed_time(n1) / (2 * args.steps)
    ntt_gbps = ntt_rows * 2 * n * 8 / (ntt_ms * 1e-3) / 1e9

    # ---- the second ceiling, measured now, in this process (SURVEY 8d): butterflies / multiply-accumulates on registers only
    ceil = None
    if rank == 0:
        ceil = {"fwd_col_shape": ctx.selftest_rate(0), "fwd_fused_shape": ctx.selftest_rate(1), "inverse": ctx.selftest_rate(2),
                "mac": ctx.selftest_rate(3)}
        if aux_primes:  # the integer key-switching path: 32-bit butterflies and 32x32->64 multiply-accumulates
            # mac32: the product kernel's own form and launch shape (two products per accumulator and digit pair, 512 threads x 1 CTA)
            ceil.update({"bfly32_fwd": ctx.selftest_rate(10), "bfly32_inv": ctx.selftest_rate(11), "mac32": ctx.selftest_rate(15),
                         "mac32_unpaired_128x4": ctx.selftest_rate(12)})

    # ---- e2e through the host-buffer C-ABI entry point (pinned host memory, H2D + D2H inside the timed region)
    e2e = None
    if not args.no_e2e:
        Be = wl["e2e_batch"]
        # staging buffers on the GPU's own NUMA node (first touch by a thread bound there): every rank's H2D / D2H traffic then
        # stays on its socket instead of crossing the inter-socket link; the affinity is restored before the CPU baseline runs
        all_cpus = os.sched_getaffinity(0)
        numa_node, numa_cpus = gpu_numa_cpus(local)
        if numa_cpus:
            os.sched_setaffinity(0, numa_cpus)
        ha = torch.empty((Be, 2, L, n), dtype=torch.int64).pin_memory()
        hb = torch.empty((Be, 2, L, n), dtype=torch.int64).pin_memory()
        ho = torch.empty((Be, 2, L, n), dtype=torch.int64).pin_memory()
        ha.copy_(a[:Be])
        hb.copy_(b[:Be])
        torch.cuda.synchronize()
        na, nb_, no = ha.numpy().view(np.uint64), hb.numpy().view(np.uint64), ho.numpy().view(np.uint64)

        def e2e_step():
            S._check(S.lib().sb200_multiply_relinearize_host(ctx.h, L, Be, S._hp(na), S._hp(nb_), rk.h, S._hp(no)))

        e2e_step()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e_step()  # returns after the D2H copy has completed
        my_t = time.perf_counter() - t0
        t = torch.tensor([my_t], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        if not (ho.cuda() == out[:Be]).all():
            fail("e2e (host pipeline) result differs from the device-resident result of the timed run")
        os.sched_setaffinity(0, all_cpus)
        h2d, d2h = int(ha.nbytes + hb.nbytes), int(ho.nbytes)
        # per-rank staging facts (VERDICT r1: e2e scaling): NUMA node of each rank's GPU and its own copy rates
        mine = torch.tensor([float(numa_node if numa_node is not None else -1), h2d * args.steps / my_t / 1e9, d2h * args.steps / my_t / 1e9,
                             Be * args.steps / my_t], dtype=torch.float64, device="cuda")
        allr = [torch.zeros_like(mine) for _ in range(world)]
        if world > 1:
            dist.all_gather(allr, mine)
        else:
            allr = [mine]
        e2e = {"value": world * Be * args.steps / float(t.item()), "unit": UNIT, "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "batch_per_step": Be, "host_numa_node": numa_node,
               "per_rank": [{"rank": r, "gpu_numa_node": int(x[0].item()), "h2d_GBps": round(x[1].item(), 2), "d2h_GBps": round(x[2].item(), 2),
                             "ct_per_s": round(x[3].item(), 1)} for r, x in enumerate(allr)],
               "note": "2 x 32.5 MB in + 32.5 MB out per ciphertext: the host link (PCIe Gen5 x16 per GPU) bounds this figure"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    value = world * B * args.steps / (ms_total / 1e3)
    peak, peak_src = measured_peak()
    # ---- roofline, SURVEY 8(d): compulsory bytes of the fused operation = 6*L*n*8 per ciphertext (4 polynomials in, 2 out; the third
    #      product polynomial is never materialised) + one pass over the key (2*L*(L+1)*n*8) per B_reuse ciphertexts (= the chunk)
    ct_bytes = 6 * L * n * 8
    key_bytes = 2 * L * k * n * 8
    nchunks = -(-B // chunk)
    step_bytes = B * ct_bytes + nchunks * key_bytes
    b_reuse = B / nchunks
    prof.sort(key=lambda r: -r[1])
    tot_prof_ms = sum(r[1] for r in prof) or 1.0
    top = prof[0]
    top_launch_ms = top[1] / max(top[2], 1)
    sm_hz = (clocks or {}).get("sm_mhz") or (clocks or {}).get("sm_max_mhz") or 1965.0
    sm_hz *= 1e6
    smsp = torch.cuda.get_device_properties(local).multi_processor_count * 4

    def alu_entry(r):
        """second ceiling for one kernel: time the measured butterfly / multiply-accumulate rates would need vs the time it took"""
        name, kms, launches_, _, bf, mc, b32, m32 = r
        if bf <= 0 and mc <= 0 and b32 <= 0 and m32 <= 0:
            return None
        inv = name.startswith(("ks_target_intt", "ks_top_intt", "rescale_top", "ntt_inv", "ks_prod_intt", "modswitch_top"))
        rate_b = ceil["inverse"] if inv else (ceil["fwd_fused_shape"] if name == "ks_local_mac" else ceil["fwd_col_shape"])
        floor_s = bf / 32 / rate_b + mc / 32 / ceil["mac"]
        rate32 = None
        if b32 > 0 or m32 > 0:
            rate32 = ceil["bfly32_inv"] if name.startswith("ks32_inv") else ceil["bfly32_fwd"]
            floor_s += b32 / 32 / rate32 + m32 / 32 / ceil["mac32"]
        e = {"kernel": name, "frac_of_alu_ceiling": floor_s / (kms * 1e-3), "floor_ms": floor_s * 1e3}
        if bf > 0:
            e["achieved_clk_per_warp_bfly"] = kms * 1e-3 * sm_hz * smsp / (bf / 32)
            e["floor_clk_per_warp_bfly"] = sm_hz * smsp / rate_b
        if b32 > 0:
            e["achieved_clk_per_warp_bfly32"] = kms * 1e-3 * sm_hz * smsp / (b32 / 32)
            e["floor_clk_per_warp_bfly32"] = sm_hz * smsp / rate32
        if m32 > 0:
            e["achieved_clk_per_warp_mac32"] = kms * 1e-3 * sm_hz * smsp / (m32 / 32)
            e["floor_clk_per_warp_mac32"] = sm_hz * smsp / ceil["mac32"]
        return e

    alu = [e for e in (alu_entry(r) for r in prof) if e]
    whole_floor = sum(e["floor_ms"] for e in alu) * 1e-3
    traffic = ncu_traffic(top[0])
    # DRAM traffic of ALL kernels of one key-switching chunk (committed ncu capture, one launch each) against the compulsory bytes of
    # that chunk: what the intermediates of the path cost in HBM traffic
    step_traffic = None
    per_kernel = [ncu_traffic(r[0]) for r in prof]
    if all(per_kernel) and len({t_["batch"] for t_ in per_kernel}) == 1:
        cb = per_kernel[0]["batch"]
        tot_b = sum(t_["dram_bytes_per_launch"] for t_ in per_kernel)
        step_traffic = {"ciphertexts_per_chunk": cb, "dram_bytes_per_chunk": tot_b, "dram_bytes_per_ciphertext": tot_b / cb,
                        "ratio_to_compulsory": tot_b / (cb * ct_bytes + key_bytes),
                        "avg_dram_GBps_at_measured_speed": tot_b / cb * value / 1e9, "frac_of_hbm_peak": tot_b / cb * value / 1e9 / peak}
    alg_per_launch = step_bytes * args.steps / max(top[2], 1)  # the operation's compulsory bytes behind one launch of the dominant kernel
    achieved = alg_per_launch / (top_launch_ms * 1e-3) / 1e9
    roofline = {
        "bound": "hbm", "kernel": top[0], "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
        "traffic": traffic["dram_bytes_per_launch"] if traffic else None,
        "traffic_ratio": (traffic["dram_bytes_per_launch"] / (traffic.get("batch", chunk) * ct_bytes + key_bytes)) if traffic else None,
        "traffic_source": traffic.get("source") if traffic else None, "step_traffic": step_traffic,
        "peak_source": peak_src, "share_of_step": top[1] / tot_prof_ms, "launches": top[2], "avg_launch_ms": top_launch_ms,
        "bytes_basis": "SURVEY 8(d): the whole operation's compulsory bytes (6*L*n*8 per ciphertext + key per B_reuse) are attributed to "
                       "the dominant kernel's launches; intermediates (digits, accumulated products) are not counted",
        "alg_bytes_per_ciphertext": ct_bytes, "key_bytes": key_bytes, "B_reuse": b_reuse, "key_passes_per_step": nchunks,
        "key_bytes_device_format": (len(aux_primes) * 4 * 2 * L * k * n) if aux_primes else key_bytes,
        "alu": {"unit": "clocks per warp-butterfly per SM sub-partition (32 butterflies, one sub-partition)",
                "ceiling_source": "sb200_selftest_rate in this process, same clocks: the path's butterfly / multiply-accumulate code on registers only",
                "ceilings_warp_ops_per_s": ceil, "sm_hz_used": sm_hz, "kernels": alu,
                "step_frac_of_alu_ceiling": whole_floor / (tot_prof_ms * 1e-3)},
        "note": ("key switching = exact integer convolution modulo %d auxiliary 29-bit primes (32-bit butterflies, 32x32->64 multiply-accumulates), "
                 "CRT back to the q_i; both ceilings of SURVEY 8(d) are reported" % len(aux_primes)) if aux_primes else
                "integer-multiply-issue bound path (64-bit modular butterflies on 32-bit multipliers); both ceilings of SURVEY 8(d) are reported",
        "kernels": [{"name": r[0], "ms": round(r[1], 3), "launches": r[2], "share": round(r[1] / tot_prof_ms, 4)} for r in prof]}
    op_gbps = step_bytes * args.steps / (ms_total * 1e-3) / 1e9 / 1.0  # per GPU: every rank runs the same step
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        if R.available():
            if rc is None:
                rc = R.RefContext(wl["scheme"], n, mods)
            rc.relin_key()
            cpu = cpu_reference_rate(rc, 0, L, wl["cpu_reps"])
        else:
            cpu = {"value": None, "unit": UNIT, "cores": host_threads(), "kind": "reference", "sample": "oracle/_ref/libsealref.so not present"}
    configs = None
    if world == 1 and not args.no_configs and R.available():
        del a, b, out
        torch.cuda.empty_cache()
        configs = {}
        for name, fn in (("cfg2", run_cfg2), ("cfg3", run_cfg3), ("cfg4", run_cfg4), ("n65536_k16", run_k16)):
            t0 = time.time()
            configs[name] = fn(S, R, torch, np)
            configs[name]["wall_s"] = round(time.time() - t0, 1)
            torch.cuda.empty_cache()
        configs["cpp"] = run_cpp_harness()
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
        "data": "synthetic",
        "config": {"workload": args.workload, "scheme": "CKKS", "n": n, "coeff_modulus_primes": k, "L": L, "prime_bits": wl["bits"][0],
                   "batch_per_gpu": B, "global_batch": B * world, "ops": "Evaluator::multiply + relinearize_inplace (fused call)",
                   "l2": f"inputs {2 * B * 2 * L * n * 8 / 2**30:.1f} GiB per GPU >> 126 MB L2 (no flush needed)",
                   "scratch_budget_GiB": round(scratch_budget / 2**30, 1), "ciphertexts_per_key_pass": chunk,
                   "key_switching": ("integer convolution, auxiliary primes %s" % aux_primes) if aux_primes else "64-bit digit transforms",
                   "parallelism": f"batch sharded x{world}, no data-path collective"},
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "verified": verified, "roofline": roofline,
        "ntt": {"metric": "negacyclic NTT GB/s (2*n*8 B per row per transform)", "rows_per_transform_call": ntt_rows, "n": n,
                "ms_per_call": ntt_ms, "achieved_GBps": ntt_gbps, "peak_GBps": peak, "frac_of_hbm_peak": ntt_gbps / peak,
                "alu_ceiling_GBps": (ceil["fwd_col_shape"] + ceil["inverse"]) / 2 * 32 / (n / 2 * (n.bit_length() - 1)) * 2 * n * 8 / 1e9,
                "note": "16 butterfly stages per 16 bytes moved: the transform is bound by the integer-multiply issue rate (alu_ceiling_GBps), not by HBM"},
        "op_roofline": {"alg_bytes_per_step": step_bytes, "achieved_GBps_per_gpu": op_gbps, "frac_of_hbm_peak": op_gbps / peak},
        "cpu_baseline": cpu, "configs": configs,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
