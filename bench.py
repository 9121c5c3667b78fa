#!/usr/bin/env python
"""bench.py -- headline benchmark: secp256k1 ECDSA verifies/s at batch 2^20 per GPU, plus (at N = 1) the
other BASELINE.json configurations as a `workloads` object on the same JSON line.

Usage:
  python bench.py --gpus N --steps K --warmup W          # this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K --warmup W   # reference CPU arm
One JSON line on stdout from rank 0.  Every timed loop runs exactly K steps.  --dump-outputs DIR writes what the
timed paths returned in their last step as DIR/<name>.npy (float32), so that two builds can be compared on the same
seeded inputs.

* headline workload: BASELINE.json configs[1] -- 2^20 random (msgHash, sig, pub) triples per GPU
  (benchdata.gen_secp256k1_verify: 4096 keys, 1/64 corrupted), weak scaling: rank g verifies its own
  shard (seed 0xE1110500+g for N>1), statuses gathered over NCCL.
* `value`: inputs already resident in HBM; a step = prep kernel + verify kernel over the whole shard
  (+ the NCCL gather of 1 B/item when N>1).
* `e2e`: the same metric through the public host-buffer call (C ABI eb200_ecdsa_verify_batch via
  elliptic_b200.ec.EC.verify_batch_packed) with HOST buffers: H2D + kernels + D2H inside the timed
  region; `e2e.pageable` repeats it with ordinary (unpinned) numpy buffers.
* `workloads` (N = 1 only): ed25519 verify 2^20, curve25519 derive 2^20, p256 / p384 verify 2^20, p521
  verify 2^18 -- each with the device-resident rate, the end-to-end rate through the host-buffer ABI, its
  roofline entry, an equality assert of every status (and every derived x) against the generator's
  expectation, and a spot check of >= 512 items against the Python oracle (outside the timed regions).
* `roofline`: the binding resource is the integer multiplier (fma pipe), not HBM; the denominator is
  the IMAD.WIDE.U32 rate measured on this pool by bench_micro/imad_peak.cu (profiles/r0*_imad_peak.json).
  `roofline_hbm` gives the contract's HBM view of the same kernel.
* `cpu_baseline` / --impl reference: Node.js is not installed in this image (nor on the GPU box), so the
  reference's own JS cannot run; the CPU arm is oracle/c/k256_ref.c, a C restatement of the reference's
  algorithm (kind "port"), timed on one thread and on every schedulable host thread.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MAC32_PER_VERIFY_REF = 301376     # BASELINE.md section 2: 2216 fm x 136 MAC32 (reference algorithm)
ALG_BYTES_PER_VERIFY = 161        # SURVEY 8d: e,r,s,x,y in + 1 status byte out
LOG2_BATCH = 20
CACHE = os.environ.get("EB200_CACHE", "/tmp/eb200_cache")
DUMP_MAX_BYTES = 64 << 20
DUMP_DERIVE_ROWS = 1 << 16        # fixed, seeded sample of the 2^20 derived x (all of them would be 128 MB as float32)
DUMP_SEED = 0xE111D
WORKLOAD = "secp256k1 batch ECDSA verify, 2^20 random sigs per GPU (BASELINE.json configs[1])"

# (key, log2 n, MAC32 per unit of the REFERENCE algorithm (SURVEY 8d), algorithmic bytes per unit, seed)
# p521: 13.61 field mults per scalar bit (the p256 / p384 figures) x 521 bits x (2*17^2 + 17) MAC32
EXTRA = [
    ("ed25519_verify", 20, 816680, 129, 0xE1110003),
    ("curve25519_derive", 20, 554336, 97, 0xE1110004),
    ("p256_verify", 20, 473688, 161, 0xE1110256),
    ("p384_verify", 20, 1567800, 241, 0xE1110384),
    ("p521_verify", 18, 4218550, 331, 0xE1110521),
]


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_quota():
    """CPU bandwidth limit of this container in cores (cgroup v2 cpu.max), or None when unlimited / unknown.
    The GPU boxes expose every host thread in the affinity mask but cap the container's CPU time, which is
    why the all-thread rate is far below cores x per_core (r01: 143 k/s on one box, 716 k/s on another)."""
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        return None if q == "max" else float(q) / float(per)
    except Exception:
        return None


def load_peaks():
    hbm, how = 6650.0, "fallback"
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            hbm, how = float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    imad = 18.46   # T MAC32/s: plain IMAD.WIDE.U32 (measured on this pool)
    for name in ("r02_imad_peak.json", "r01_imad_peak.json"):
        q = os.path.join(ROOT, "profiles", name)
        if os.path.exists(q):
            try:
                d = json.load(open(q))
                d = d.get("packed_field", d)
                imad = max(v for k, v in d.items() if k.startswith("wide_") and not k.startswith("wide_cc"))
                break
            except Exception:
                pass
    return hbm, how, imad


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.samples, self.reasons, self.max = [], set(), None
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            try:
                self.samples.append(float(f[0]))
                self.max = float(f[1])
                for nm, v in zip(names, f[3:7]):
                    if v.lower().startswith("active"):
                        self.reasons.add(nm)
            except Exception:
                pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        s = sorted(self.samples)
        load = [x for x in s if self.max and x > 0.5 * self.max] or s
        return {"sm_mhz": load[len(load) // 2] if load else None, "sm_max_mhz": self.max,
                "samples": len(s), "reasons": sorted(self.reasons)}


def dataset(rank, world):
    import benchdata
    seed = 0xE1110002 if world == 1 else 0xE1110500 + rank
    return benchdata.gen_secp256k1_verify(1 << LOG2_BATCH, seed=seed, cache_dir=CACHE)


# ---------------------------------------------------------------------------------------------
# CPU arm: oracle/c/k256_ref.c (the checker; only ever executed here, outside the GPU's timed regions)
def cpu_rates(ds, threads, sample_all=1 << 16, sample_one=1 << 11, reps=3):
    """(all-thread rate, one-thread rate, items used).  Dynamic 64-item chunks inside the C driver keep one
    slow core from stretching the batch; the median of `reps` runs is reported."""
    from oracle import c_oracle
    c_oracle.build()
    n = ds["e"].shape[0]
    sample_all, sample_one = min(n, sample_all), min(n, sample_one)

    def run(m, th, lo=0):
        sl = slice(lo, lo + m)
        t = time.perf_counter()
        st = c_oracle.verify_batch(ds["e"][sl], ds["r"][sl], ds["s"][sl], ds["pub"][sl], th)
        dt = time.perf_counter() - t
        assert np.array_equal(st, ds["expected"][sl]), "CPU restatement disagrees with the generator"
        return m / dt

    run(4096, threads)                                           # warm-up: tables, thread stacks
    total = sorted(run(sample_all, threads, (k * sample_all) % max(1, n - sample_all + 1)) for k in range(reps))[reps // 2]
    one = sorted(run(sample_one, 1, k * sample_one) for k in range(reps))[reps // 2]
    return total, one, sample_all


def run_reference(args):
    """--impl reference: the reference's CPU path (C restatement; Node.js absent)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ds = dataset(0, 1)
    threads = host_threads()
    from oracle import c_oracle
    c_oracle.build()
    sample = 1 << 16
    n = 1 << LOG2_BATCH
    for _ in range(max(1, args.warmup)):
        c_oracle.verify_batch(ds["e"][:8192], ds["r"][:8192], ds["s"][:8192], ds["pub"][:8192], threads)
    t0 = time.perf_counter()
    for k in range(args.steps):
        lo = (k * sample) % n
        sl = slice(lo, lo + sample)
        st = c_oracle.verify_batch(ds["e"][sl], ds["r"][sl], ds["s"][sl], ds["pub"][sl], threads)
        assert np.array_equal(st, ds["expected"][sl])
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"secp256k1_verify_status": st})
    value = args.steps * sample / dt
    _, one, _ = cpu_rates(ds, threads, reps=1)
    line = {
        "impl": "reference", "metric": "secp256k1 ECDSA verifies/sec", "value": value, "unit": "verifies/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 limbs (integer, exact)",
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample_per_step": sample},
        "cpu_baseline": {"value": value, "unit": "verifies/s", "cores": threads, "kind": "port",
                         "per_core": one, "total": value, "effective_cores": value / one,
                         "cgroup_cpu_quota_cores": cpu_quota(),
                         "sample": "%d signatures/step x %d steps of the same 2^20 workload, oracle/c/k256_ref.c (C "
                                   "restatement of the reference's GLV+JSF+wNAF algorithm; Node.js not installed); "
                                   "per_core = the same code on one thread" % (sample, args.steps)},
        "e2e": {"value": value, "unit": "verifies/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ---------------------------------------------------------------------------------------------
# oracle spot checks for the extra workloads (worker processes; never inside a timed region)
def _spot_ecdsa(args):
    name, rows = args
    from oracle.ref_py.ec import EC
    ec = EC(name)
    out = []
    for e, r, s, pub in rows:
        ln = len(e)
        ev = int.from_bytes(e, "big")
        if ev >= ec.n:
            ev -= ec.n                     # what _truncateToN leaves for a len-byte array (the ABI takes it reduced or not)
        rv, sv = int.from_bytes(r, "big"), int.from_bytes(s, "big")
        if not (1 <= rv < ec.n and 1 <= sv < ec.n):
            out.append(0)
            continue
        out.append(int(ec.verify(ev, {"r": rv, "s": sv},
                                 {"x": int.from_bytes(pub[:ln], "big"), "y": int.from_bytes(pub[ln:], "big")})))
    return out


def _spot_ed(rows):
    from oracle.ref_py.eddsa import EDDSA
    from oracle.ref_py.bn import RefError
    ed = EDDSA()
    out = []
    for R, S, A, M in rows:
        try:
            out.append(int(ed.verify(M, R + S, A)))
        except RefError as ex:
            out.append({"invalid point": 2, "Assertion failed": 5}[ex.args[0]])
    return out


def _spot_x(rows):
    from oracle.ref_py import curves
    from oracle.ref_py.bn import RefError
    from oracle.ref_py.ec import EC, KeyPair
    ec, c = EC("curve25519"), curves.get("curve25519").curve
    out = []
    for k, x in rows:
        try:
            out.append((1, KeyPair(ec, priv=int.from_bytes(k, "big")).derive(c.point(int.from_bytes(x, "big"), 1))))
        except RefError as ex:
            out.append(({"Assertion failed": 5, "public point not validated": 3}[ex.args[0]], 0))
    return out


def spot_indices(n, count=512, corrupt_every=64):
    step = max(1, n // (count - 64))
    idx = list(range(0, n, step))[:count - 64]
    bad = list(range(corrupt_every - 1, n, corrupt_every))                  # corrupted / twist items
    idx += bad[::max(1, len(bad) // 64)][:64]
    return sorted(set(idx))


def pmap(fn, rows, wrap=None):
    import benchdata
    chunks = [rows[i:i + 16] for i in range(0, len(rows), 16)]
    res = benchdata._pmap(fn, [wrap(c) for c in chunks] if wrap else chunks, min_items=2)
    return [x for part in res for x in part]


def run_extra(key, log2n, mac32, alg_bytes, seed, lib, nat, dev, steps, imad_peak, outputs=None):
    """One of the non-headline BASELINE configurations on a single GPU.  `outputs` (a dict) receives what the
    device-resident call returned in its last timed step."""
    import torch
    import benchdata
    n = 1 << log2n
    t_gen = time.time()
    stream = torch.cuda.current_stream().cuda_stream
    out_host = None
    if key.endswith("_verify") and key != "ed25519_verify":
        name = key.split("_")[0]
        cid, ln = {"p256": (nat.CURVE_P256, 32), "p384": (nat.CURVE_P384, 48), "p521": (nat.CURVE_P521, 66)}[name]
        ds = benchdata.gen_ecdsa_verify(name, n, seed=seed, n_keys=1024, cache_dir=CACHE)
        cols = ("e", "r", "s", "pub")
        d = {k: torch.from_numpy(ds[k]).to(dev) for k in cols}
        d_status = torch.empty(n, dtype=torch.uint8, device=dev)
        d_ws = torch.empty(lib.eb200_ecdsa_verify_workspace_bytes(cid, n), dtype=torch.uint8, device=dev)

        def step():
            nat.check(lib.eb200_ecdsa_verify_batch_dev(cid, n, d["e"].data_ptr(), d["r"].data_ptr(), d["s"].data_ptr(),
                                                       d["pub"].data_ptr(), nat.PUB_XY, d_status.data_ptr(), d_ws.data_ptr(), stream))
        from elliptic_b200.ec import EC
        ec = EC(name, device=dev.index)
        h = {k: torch.from_numpy(ds[k]).pin_memory().numpy() for k in cols}
        e2e_call = lambda: ec.verify_batch_packed(h["e"], h["r"], h["s"], h["pub"])
        h2d, d2h = n * 5 * ln, n
        api = "EC('%s').verify_batch_packed -> eb200_ecdsa_verify_batch" % name
        idx = spot_indices(n)
        spot = lambda: pmap(_spot_ecdsa, [(ds["e"][i].tobytes(), ds["r"][i].tobytes(), ds["s"][i].tobytes(), ds["pub"][i].tobytes()) for i in idx],
                            wrap=lambda c: (name, c))
        kernel = "sw_verify_kernel<%s>" % name.upper()
    elif key == "ed25519_verify":
        ds = benchdata.gen_ed25519_verify(n, seed=seed, cache_dir=CACHE, with_msgs=True)
        cols = ("R", "S", "A", "h")
        d = {k: torch.from_numpy(ds[k]).to(dev) for k in cols}
        d_status = torch.empty(n, dtype=torch.uint8, device=dev)
        d_ws = torch.empty(lib.eb200_eddsa_verify_workspace_bytes(n), dtype=torch.uint8, device=dev)

        def step():
            nat.check(lib.eb200_eddsa_verify_batch_dev(n, d["R"].data_ptr(), d["S"].data_ptr(), d["A"].data_ptr(), d["h"].data_ptr(),
                                                       d_status.data_ptr(), d_ws.data_ptr(), stream))
        from elliptic_b200.eddsa import EDDSA
        ed = EDDSA(device=dev.index)
        h = {k: torch.from_numpy(ds[k]).pin_memory().numpy() for k in ("R", "S", "A")}
        hm = torch.from_numpy(ds["msgs"].reshape(-1)).pin_memory().numpy()
        off = np.arange(n + 1, dtype=np.uint64) * 32
        e2e_call = lambda: ed.verify_batch_msgs_packed(h["R"], h["S"], h["A"], hm, off)     # raw messages: SHA-512 on the GPU too
        h2d, d2h = n * 128 + (n + 1) * 8, n
        api = "EDDSA().verify_batch_msgs_packed -> eb200_eddsa_verify_batch_msgs (R, S, A, 32-byte messages; SHA-512 on the GPU)"
        idx = spot_indices(n)
        spot = lambda: pmap(_spot_ed, [(ds["R"][i].tobytes(), ds["S"][i].tobytes(), ds["A"][i].tobytes(), ds["msgs"][i].tobytes()) for i in idx])
        kernel = "ed25519_verify_kernel"
    else:
        ds = benchdata.gen_x25519_derive(n, seed=seed, cache_dir=CACHE)
        d = {k: torch.from_numpy(ds[k]).to(dev) for k in ("priv", "pubx")}
        d_status = torch.empty(n, dtype=torch.uint8, device=dev)
        d_out = torch.empty((n, 32), dtype=torch.uint8, device=dev)

        def step():
            nat.check(lib.eb200_x25519_derive_batch_dev(n, d["priv"].data_ptr(), d["pubx"].data_ptr(), d_out.data_ptr(),
                                                        d_status.data_ptr(), stream))
        from elliptic_b200.ec import EC
        ec = EC("curve25519", device=dev.index)
        h = {k: torch.from_numpy(ds[k]).pin_memory().numpy() for k in ("priv", "pubx")}
        out_host = {}
        h_out = torch.empty((n, 32), dtype=torch.uint8).pin_memory().numpy()         # the caller owns (and reuses) the result buffers
        h_st = torch.empty(n, dtype=torch.uint8).pin_memory().numpy()

        def e2e_call():
            out_host["x"], st = ec.derive_batch_packed(h["priv"], h["pubx"], out=h_out, status=h_st)
            return st
        h2d, d2h = n * 64, n * 33
        api = "EC('curve25519').derive_batch_packed -> eb200_x25519_derive_batch"
        idx = spot_indices(n, corrupt_every=256)
        spot = lambda: pmap(_spot_x, [(ds["priv"][i].tobytes(), ds["pubx"][i].tobytes()) for i in idx])
        kernel = "x25519_derive_kernel"
    gen_s = time.time() - t_gen
    expected = torch.from_numpy(ds["expected"]).to(dev)

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    assert bool((d_status == expected).all()), key + ": GPU statuses differ from the generator's expectation"
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        step()
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / steps
    k_ms = nat.last_timing()["main_kernel_ms"]
    if outputs is not None:
        outputs[key + "_status"] = d_status.cpu().numpy()
        if key == "curve25519_derive":
            rows = np.sort(np.random.default_rng(DUMP_SEED).choice(n, DUMP_DERIVE_ROWS, replace=False))
            outputs[key + "_x_sample"] = d_out[torch.from_numpy(rows).to(dev)].cpu().numpy()
    for _ in range(2):
        st = e2e_call()
    assert np.array_equal(st, ds["expected"]), key + ": host-buffer call differs from the generator's expectation"
    t0 = time.perf_counter()
    for _ in range(steps):
        st = e2e_call()
    e2e_dt = (time.perf_counter() - t0) / steps
    # ---- checks (outside the timed regions): oracle on >= 512 items, output bytes for derive
    verdicts = spot()
    st_np = d_status.cpu().numpy()
    checked = {"spot_items": len(idx), "statuses_equal_generator": True}
    if key == "curve25519_derive":
        out_np = d_out.cpu().numpy()
        assert np.array_equal(out_np, out_host["x"]), "derive: device-resident and host-buffer outputs differ"
        for i, (stv, x) in zip(idx, verdicts):
            assert int(st_np[i]) == stv, (key, i, int(st_np[i]), stv)
            if stv == 1:
                assert out_np[i].tobytes() == x.to_bytes(32, "big"), (key, i)
        # agreement: every valid item's shared x is a valid x again (derive(k', x_out) does not throw) is implied
        # by the oracle check above; a checksum of the 2^20 outputs pins the run
        import hashlib
        checked["out_sha256"] = hashlib.sha256(out_np.tobytes()).hexdigest()
        checked["oracle_output_bytes_equal"] = True
    else:
        for i, v in zip(idx, verdicts):
            assert int(st_np[i]) == v, (key, i, int(st_np[i]), v)
    checked["oracle_equal"] = True
    ach = n * mac32 / (k_ms * 1e-3) / 1e12
    return {
        "n": n, "value": n / (ms * 1e-3), "unit": "derives/s" if key.endswith("derive") else "verifies/s",
        "ms_per_step": ms, "steps": steps, "kernel_ms": k_ms, "gen_s": round(gen_s, 1),
        "e2e": {"value": n / e2e_dt, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": steps, "api": api},
        "roofline": {"bound": "int32-multiplier (fma pipe)", "kernel": kernel, "achieved": ach, "peak": imad_peak,
                     "unit": "T MAC32/s", "frac": ach / imad_peak, "mac32_per_unit_reference_algorithm": mac32,
                     "hbm_gbs_algorithmic": n * alg_bytes / (k_ms * 1e-3) / 1e9},
        "checks": checked,
    }


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from elliptic_b200 import _native as nat
    from elliptic_b200.ec import EC

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node %d" % args.gpus)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # communicator lines (rank count, transport) go to stderr; stdout carries the one JSON line
        # (NCCL's debug level is set in main(), before torch is imported)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    lib = nat.init(local)
    ds = dataset(rank, world)
    n = 1 << LOG2_BATCH
    ec = EC("secp256k1", device=local)

    # ---- device-resident arm --------------------------------------------------
    d = {k: torch.from_numpy(ds[k]).to(dev) for k in ("e", "r", "s", "pub")}
    d_status = torch.empty(n, dtype=torch.uint8, device=dev)
    ws_bytes = lib.eb200_ecdsa_verify_workspace_bytes(nat.CURVE_SECP256K1, n)
    d_ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    gathered = torch.empty(n * world, dtype=torch.uint8, device=dev) if world > 1 else None
    expected = torch.from_numpy(ds["expected"]).to(dev)

    def step():
        st = torch.cuda.current_stream().cuda_stream
        nat.check(lib.eb200_ecdsa_verify_batch_dev(
            nat.CURVE_SECP256K1, n, d["e"].data_ptr(), d["r"].data_ptr(), d["s"].data_ptr(), d["pub"].data_ptr(),
            nat.PUB_XY, d_status.data_ptr(), d_ws.data_ptr(), st))
        if world > 1:
            dist.all_gather_into_tensor(gathered, d_status)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    warm = max(args.warmup, 3)
    for _ in range(warm):
        step()
    barrier()
    assert bool((d_status == expected).all()), "GPU statuses differ from the generator's expectation"
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    main_ms = []
    barrier()
    ev0.record()
    for _ in range(args.steps):
        step()
    ev1.record()
    barrier()
    total_ms = ev0.elapsed_time(ev1)
    outputs = {}
    if args.dump_outputs and rank == 0:
        outputs["secp256k1_verify_status"] = (gathered if world > 1 else d_status).cpu().numpy()
    # per-launch duration of the dominant kernel (events on the launch stream), last timed step
    tm_last = nat.last_timing()
    main_ms.append(tm_last["main_kernel_ms"])
    launches_per_step = tm_last["launches"]
    # as many individually timed launches again for the roofline average
    for _ in range(args.steps):
        step()
        torch.cuda.synchronize()
        main_ms.append(nat.last_timing()["main_kernel_ms"])
    t = torch.tensor([total_ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    value = n * world / (ms_per_step * 1e-3)

    # ---- end-to-end arm: host buffers through the public API --------------------------------
    def e2e(hn, steps):
        for _ in range(2):
            st_host = ec.verify_batch_packed(hn["e"], hn["r"], hn["s"], hn["pub"])
        assert np.array_equal(st_host, ds["expected"])
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            st_host = ec.verify_batch_packed(hn["e"], hn["r"], hn["s"], hn["pub"])
        dt = time.perf_counter() - t0
        tm = nat.last_timing()
        tt = torch.tensor([dt], device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return n * world * steps / float(tt.item()), tm

    e2e_steps = args.steps
    hp = {k: torch.from_numpy(ds[k]).pin_memory() for k in ("e", "r", "s", "pub")}
    e2e_value, e2e_tm = e2e({k: v.numpy() for k, v in hp.items()}, e2e_steps)
    e2e_pageable, _ = e2e({k: np.array(ds[k], copy=True) for k in ("e", "r", "s", "pub")}, e2e_steps)
    clocks = sampler.stop() if rank == 0 else None

    if rank == 0:
        hbm_peak, hbm_how, imad_peak = load_peaks()
        k_ms = float(np.mean(main_ms))
        ach_mac = n * MAC32_PER_VERIFY_REF / (k_ms * 1e-3) / 1e12
        ach_gbs = n * ALG_BYTES_PER_VERIFY / (k_ms * 1e-3) / 1e9
        line = {
            "metric": "secp256k1 ECDSA verifies/sec", "value": value, "unit": "verifies/s", "n_gpus": world,
            "steps": args.steps, "warmup": warm, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u32 limbs (integer, exact)", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "batch_per_gpu": n, "keys": 4096, "corrupted": "1/64", "pub_format": "x||y (64 B)",
                       "l2": "inputs (168 MB) + per-item tables (805 MB) exceed the 126 MB L2; no flush needed",
                       "parallelism": "shard per GPU, NCCL all_gather of 1 B/item" if world > 1 else "single GPU"},
            "e2e": {"value": e2e_value, "unit": "verifies/s", "h2d_bytes_per_step": n * 160, "d2h_bytes_per_step": n,
                    "steps": e2e_steps, "h2d_ms": e2e_tm["h2d_ms"], "kernel_ms": e2e_tm["kernel_ms"],
                    "d2h_ms": e2e_tm["d2h_ms"], "pageable": e2e_pageable,
                    "api": "elliptic_b200.ec.EC.verify_batch_packed -> eb200_ecdsa_verify_batch (value: pinned host "
                           "buffers; pageable: ordinary numpy buffers)"},
            "gpu_launches": int(launches_per_step) * args.steps,   # prep + verify + exact-replay kernels per step
            "roofline": {"bound": "int32-multiplier (fma pipe)", "kernel": "k256_verify_kernel",
                         "achieved": ach_mac, "peak": imad_peak, "unit": "T MAC32/s", "frac": ach_mac / imad_peak,
                         "traffic": None, "kernel_ms": k_ms,
                         "note": "achieved = 2^20 x 301376 MAC32 (the reference algorithm's 2216 field mults x 136, "
                                 "BASELINE.md s2) / kernel time; peak = measured IMAD.WIDE.U32 rate "
                                 "(bench_micro/imad_peak.cu, profiles/r0*_imad_peak.json)"},
            "roofline_hbm": {"bound": "hbm", "achieved": ach_gbs, "peak": hbm_peak, "unit": "GB/s",
                             "frac": ach_gbs / hbm_peak, "traffic": None, "peak_source": hbm_how + " (MEASURED_PEAKS.json)",
                             "note": "161 algorithmic bytes per verify; the path is not HBM-bound"},
            "clocks": clocks,
        }
        for name in ("r02_traffic.json", "r01_traffic.json"):
            tr = os.path.join(ROOT, "profiles", name)
            if os.path.exists(tr):
                try:
                    tj = json.load(open(tr))
                    line["roofline"]["traffic"] = tj.get("dram_bytes_per_launch")
                    line["roofline_hbm"]["traffic"] = tj.get("dram_bytes_per_launch")
                    break
                except Exception:
                    pass
        if world == 1:
            threads = host_threads()
            total, one, used = cpu_rates(ds, threads)
            line["cpu_baseline"] = {
                "value": total, "unit": "verifies/s", "cores": threads, "kind": "port", "per_core": one, "total": total,
                "effective_cores": total / one, "cgroup_cpu_quota_cores": cpu_quota(),
                "sample": "%d signatures of the same workload on %d threads (median of 3), 2048 on one thread; "
                          "oracle/c/k256_ref.c (C restatement of the reference algorithm, 64-bit limbs; Node.js is not "
                          "installed so the JS itself cannot run)" % (used, threads)}
            if not args.no_workloads:
                del d, d_ws, hp
                torch.cuda.empty_cache()
                wl = {}
                for key, log2n, mac32, alg_bytes, seed in EXTRA:
                    if args.only and key not in args.only.split(","):
                        continue
                    wl[key] = run_extra(key, log2n, mac32, alg_bytes, seed, lib, nat, dev, args.steps, imad_peak,
                                        outputs if args.dump_outputs else None)
                    torch.cuda.empty_cache()
                line["workloads"] = wl
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def run_single_process(args):
    """--single-process: ONE host process drives N GPUs through the library's own sharding
    (eb200_init(devices[], N) + eb200_ecdsa_verify_batch over the whole N x 2^20 batch).  The per-GPU shards and
    seeds are those of the torchrun launch; statuses come home with each device's own D2H copy (the library's
    gather), so no NCCL communicator is involved in this mode."""
    import torch
    from elliptic_b200 import _native as nat
    from elliptic_b200.ec import EC
    N = args.gpus
    assert torch.cuda.device_count() >= N, "not enough GPUs"
    lib = nat.init_devices(list(range(N)))
    n = 1 << LOG2_BATCH
    shards = [dataset(g, N) for g in range(N)]
    cols = ("e", "r", "s", "pub")
    big = {k: np.concatenate([d[k] for d in shards]) for k in cols}
    expected = np.concatenate([d["expected"] for d in shards])
    ec = EC("secp256k1", device=0)
    # ---- device-resident arm: each GPU holds its shard; one host thread enqueues on all of them
    dev = [torch.device("cuda", g) for g in range(N)]
    d = [{k: torch.from_numpy(shards[g][k]).to(dev[g]) for k in cols} for g in range(N)]
    d_status = [torch.empty(n, dtype=torch.uint8, device=dev[g]) for g in range(N)]
    ws_bytes = lib.eb200_ecdsa_verify_workspace_bytes(nat.CURVE_SECP256K1, n)
    d_ws = [torch.empty(ws_bytes, dtype=torch.uint8, device=dev[g]) for g in range(N)]
    streams = [torch.cuda.current_stream(dev[g]).cuda_stream for g in range(N)]

    def step():
        for g in range(N):
            nat.check(lib.eb200_ecdsa_verify_batch_dev(
                nat.CURVE_SECP256K1, n, d[g]["e"].data_ptr(), d[g]["r"].data_ptr(), d[g]["s"].data_ptr(), d[g]["pub"].data_ptr(),
                nat.PUB_XY, d_status[g].data_ptr(), d_ws[g].data_ptr(), streams[g]))

    def sync():
        for g in range(N):
            torch.cuda.synchronize(dev[g])

    warm = max(args.warmup, 3)
    for _ in range(warm):
        step()
    sync()
    for g in range(N):
        assert np.array_equal(d_status[g].cpu().numpy(), shards[g]["expected"]), "GPU %d statuses differ" % g
    sampler = ClockSampler(0)
    sampler.start()
    ev = []
    for g in range(N):
        with torch.cuda.device(dev[g]):
            ev.append((torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)))
            ev[g][0].record()
    for _ in range(args.steps):
        step()
    for g in range(N):
        with torch.cuda.device(dev[g]):
            ev[g][1].record()
    sync()
    total_ms = max(ev[g][0].elapsed_time(ev[g][1]) for g in range(N))        # max over GPUs, device clocks
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"secp256k1_verify_status": np.concatenate([s.cpu().numpy() for s in d_status])})
    ms_per_step = total_ms / args.steps
    value = n * N / (ms_per_step * 1e-3)
    # ---- end-to-end arm: one host call over the whole batch, host buffers, library-internal sharding
    def e2e(hn, steps):
        for _ in range(2):
            st = ec.verify_batch_packed(hn["e"], hn["r"], hn["s"], hn["pub"])
        assert np.array_equal(st, expected)
        t0 = time.perf_counter()
        for _ in range(steps):
            st = ec.verify_batch_packed(hn["e"], hn["r"], hn["s"], hn["pub"])
        return n * N * steps / (time.perf_counter() - t0), nat.last_timing()
    e2e_steps = args.steps
    hp = {k: torch.from_numpy(big[k]).pin_memory() for k in cols}
    e2e_value, tm = e2e({k: v.numpy() for k, v in hp.items()}, e2e_steps)
    e2e_pageable, _ = e2e(big, e2e_steps)
    clocks = sampler.stop()
    _, _, imad_peak = load_peaks()
    k_ms = tm["main_kernel_ms"]
    line = {
        "metric": "secp256k1 ECDSA verifies/sec", "value": value, "unit": "verifies/s", "n_gpus": N, "steps": args.steps,
        "warmup": warm, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32 limbs (integer, exact)", "data": "synthetic",
        "config": {"workload": WORKLOAD, "batch_per_gpu": n, "launch": "single process, eb200_init(devices[], %d)" % N,
                   "parallelism": "contiguous blocks over %d GPUs inside eb200_ecdsa_verify_batch, one host thread per GPU" % N},
        "e2e": {"value": e2e_value, "unit": "verifies/s", "h2d_bytes_per_step": n * N * 160, "d2h_bytes_per_step": n * N,
                "steps": e2e_steps, "pageable": e2e_pageable, "slowest_gpu_kernel_span_ms": k_ms,
                "api": "one EC.verify_batch_packed -> eb200_ecdsa_verify_batch call over %d x 2^20 items" % N},
        "gpu_launches": int(tm["launches"]) * 0 + 5 * N * args.steps, "clocks": clocks,
    }
    emit(line)


_JSON_OUT = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version line to fd 1
    whatever NCCL_DEBUG_FILE says; child processes inherit fd 1), so fd 1 is pointed at stderr for the whole run and
    the JSON line goes to a private duplicate of the original stdout."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def dump_outputs(path, arrays):
    """--dump-outputs: each array as <path>/<name>.npy in float32 (statuses and bytes are small integers: exact)."""
    arrays = {k: np.asarray(v, np.float32) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_MAX_BYTES, "outputs to dump: %d bytes > %d" % (total, DUMP_MAX_BYTES)
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


def emit(line):
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError("must be at least 1")
    return v


def main():
    claim_stdout()
    # communicator lines (rank count, transport: NVLS / P2P) are part of the evidence.  Set before anything can load
    # NCCL; it writes to fd 1, which now is stderr.  The GPU boxes preset VERSION, which hides them: raise that too.
    if int(os.environ.get("WORLD_SIZE", "1")) > 1 and os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "INFO"
        os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=20, help="timed steps of every timed loop")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-workloads", action="store_true", help="headline only (development)")
    ap.add_argument("--only", default="", help="comma-separated subset of the extra workloads (development)")
    ap.add_argument("--single-process", action="store_true",
                    help="drive all --gpus N devices from this one process through the library's own sharding")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what they returned in their last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    elif args.single_process:
        run_single_process(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
