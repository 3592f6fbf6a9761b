#!/usr/bin/env python3
"""bench.py — the headline metric of BASELINE.json: credential Ed25519 verifies/s (512 B payload) at N B200s.

    python bench.py --gpus N --steps K --warmup W                (N > 1: launched by torch.distributed.run, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W   (the reference's CPU path: oracle C port, all host threads)
    python bench.py --soak 60 --gpus N                            (BASELINE configs[4]: sustained mixed ingest, own JSON line)
    python bench.py --steps K --dump-outputs DIR                  (also writes the last timed step's result bitmap as DIR/verify_ok.npy)

A "step" is one pass of the hot path over one batch: per GPU, configs[1] of BASELINE.json — batched Ed25519 verify of
1 M x 512 B credentials (K = 1024 key pairs, 1 % corrupted so the kernel cannot short-circuit; SURVEY.md §8d).  Weak
scaling: every rank verifies its own 1 M batch, no collective on the data path (§8e).

  value      verifies/s with inputs resident in HBM (CUDA events on the launching stream, max over ranks).  Every step starts from
             an EMPTY issuer-key cache: de-duplication, the 1024 per-key tables and all 10^6 verifications happen inside the step
  e2e        the same work through the C-ABI host call (afc_ed25519_verify_batch): pinned host buffers (allocated after the rank is
             bound to its GPU's NUMA node), H2D of all inputs and D2H of the result bitmap inside the timed region
  roofline   the dominant kernel against the measured HBM peak, algorithmic bytes = 609 B / credential (frac), and the whole
             step against the same peak (frac_step)
  cpu_baseline  the oracle's C port of Go's algorithm on this box's host cores, bounded sample (rank 0, N = 1 only); OpenSSL beside it
  cfg4       BASELINE configs[3]: 2^22 Ed25519 signatures + RFC 6962 audit append, leaves in contiguous 2^k-aligned ranges over
             the ranks, local subtree roots ALL-GATHERED OVER NCCL and folded on every rank; the global root is checked against a
             single-rank recomputation (root_ok)
  cfg3       BASELINE configs[2]: HMAC-SHA256 over 10 M x 256 B webhook bodies (N = 1)
  warm_keycache / no_keycache / keyed / issuer_mix   secondary figures of the verify path

Only the `cpu_baseline` legs and `--impl reference` execute anything under oracle/.
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
sys.dont_write_bytecode = True          # the benchmark leaves the tree untouched (it may be read-only); only --dump-outputs writes

N_ITEMS = 1_000_000
MSG_LEN = 512
N_KEYS = 1024
ALGO_BYTES = 609            # 512 msg + 32 pk + 64 sig read, 1 result byte written (SURVEY.md §8d)
METRIC = "credential Ed25519 verifies/sec (512B payload)"
UNIT = "verifies/s"
# identical in the b200 and the reference arm: the workload, not how an arm runs it
CONFIG = {"workload": "batched Ed25519 verify, 1 M x 512 B credentials per GPU (BASELINE.json configs[1])", "items_per_gpu_per_step": N_ITEMS,
          "msg_len": MSG_LEN, "keys": N_KEYS, "key_of_item": "i mod 1024",
          "corrupted": "1% (i%100==0: message bit (i/100 mod 4096) flipped; i%100==50: bit 3 of signature byte 33 flipped)"}
CFG4_LEAVES = 1 << 22
CFG3_ITEMS = 10_000_000


def host_threads():
    """CPU threads this process may actually use: affinity mask, capped by the cgroup CPU quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for qf, pf in (("/sys/fs/cgroup/cpu.max", None), ("/sys/fs/cgroup/cpu/cpu.cfs_quota_us", "/sys/fs/cgroup/cpu/cpu.cfs_period_us")):
        try:
            if pf is None:
                q, per = open(qf).read().split()
            else:
                q, per = open(qf).read().strip(), open(pf).read().strip()
            if q not in ("max", "-1"):
                n = max(1, min(n, int(float(q) / float(per) + 0.999)))
            break
        except Exception:
            continue
    return n


def bind_to_gpu_numa_node(index):
    """Pin this rank to the CPUs next to its GPU BEFORE any pinned host memory is allocated (Linux allocates, and CUDA pins, pages
    on the node of the allocating thread).  Round 1 left ranks wherever the launcher put them: at 8 GPUs the host-call figure fell
    to 0.70 of linear because half of the staging buffers sat on the other socket.  Returns what was done, for the JSON line."""
    info = {"bound": False}
    try:
        allowed = os.sched_getaffinity(0)
        bind_to_gpu_numa_node.original = set(allowed)
        cpus = None
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(index)
            words = (max(allowed) // 64) + 1
            mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
            cpus = {w * 64 + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1}
            info["source"] = "nvmlDeviceGetCpuAffinity"
            try:
                info["numa_node"] = int(pynvml.nvmlDeviceGetNumaNodeId(h))
            except Exception:
                pass
        except Exception:
            cpus = None
        if cpus:
            use = cpus & allowed
            if use and use != allowed:
                os.sched_setaffinity(0, use)
                info["bound"] = True
            info["cpus"] = len(use or allowed)
            info["cpus_before"] = len(allowed)
    except Exception as ex:
        info["error"] = repr(ex)
    return info


def unbind_for_cpu_legs():
    """The CPU baselines use every host thread the process may use: undo the NUMA binding of the GPU sections first."""
    orig = getattr(bind_to_gpu_numa_node, "original", None)
    if orig:
        try:
            os.sched_setaffinity(0, orig)
        except OSError:
            pass


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        # NVML in a thread (no process start-up latency, so short timed regions still get samples); nvidia-smi -lms as fallback
        try:
            import pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.nv, self.stop_flag = pynvml, False
            self.th = threading.Thread(target=self._nvml_loop, daemon=True)
            self.th.start()
            return
        except Exception:
            self.nv = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _nvml_loop(self):
        nv = self.nv
        bits = (("hw_slowdown", nv.nvmlClocksThrottleReasonHwSlowdown), ("hw_thermal_slowdown", nv.nvmlClocksThrottleReasonHwThermalSlowdown),
                ("sw_thermal_slowdown", nv.nvmlClocksThrottleReasonSwThermalSlowdown), ("sw_power_cap", nv.nvmlClocksThrottleReasonSwPowerCap))
        try:
            mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        except Exception:
            mx = 0
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append("%d, %d, 0, %s" % (sm, mx, ", ".join("Active" if (r & b) else "Not Active" for _, b in bits)))
            except Exception:
                pass
            time.sleep(0.02)

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if getattr(self, "nv", None):
            self.stop_flag = True
            self.th.join(timeout=2)
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                pass
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        # median of the upper half = clocks under load (idle samples at the edges are dropped)
        s = sorted(sm)
        load = s[len(s) // 2:]
        return {"sm_mhz": load[len(load) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def make_workload(ctx, dev, rank, n_keys=N_KEYS, n=N_ITEMS, distinct_tail=0, seed=0xAF02):
    """cfg2 inputs, generated on the device (synthetic): returns device tensors + expected bitmap.  key of item i = i mod n_keys;
    with distinct_tail > 0 the last `distinct_tail` items each carry a key of their own (the cold half of a hot/cold mix)."""
    import torch
    g = torch.Generator(device=dev)
    g.manual_seed(seed + rank)
    rng = np.random.default_rng(seed)
    nk_total = n_keys + distinct_tail
    kseeds = torch.from_numpy(rng.integers(0, 256, (nk_total, 32), dtype=np.uint8)).to(dev)
    d_exp = torch.empty((nk_total, 96), dtype=torch.uint8, device=dev)
    ctx.expand_dev(kseeds, nk_total, d_exp)
    d_msgs = torch.randint(0, 256, (n, MSG_LEN), dtype=torch.uint8, device=dev, generator=g)
    idx = torch.arange(n, device=dev)
    ki = idx % n_keys
    if distinct_tail:
        ki = torch.where(idx >= n - distinct_tail, n_keys + (idx - (n - distinct_tail)), ki)
    d_ki = ki.to(torch.int32)
    d_off = torch.arange(n + 1, device=dev, dtype=torch.int64) * MSG_LEN
    d_sigs = torch.empty((n, 64), dtype=torch.uint8, device=dev)
    ctx.sign_expanded_dev(d_exp, d_ki, d_msgs.view(-1), d_off, n, d_sigs)
    d_pks = d_exp[:, 64:][d_ki.long()].contiguous()
    flip_msg, flip_s = idx % 100 == 0, idx % 100 == 50
    bitpos = (idx // 100) % (MSG_LEN * 8)
    rows, cols = idx[flip_msg], bitpos[flip_msg] // 8
    d_msgs[rows, cols] = d_msgs[rows, cols] ^ (1 << (bitpos[flip_msg] % 8)).to(torch.uint8)
    srows = idx[flip_s]
    d_sigs[srows, 33] = d_sigs[srows, 33] ^ 0x08
    expect = (~(flip_msg | flip_s)).to(torch.uint8)
    torch.cuda.synchronize()
    return d_pks, d_sigs, d_msgs.view(-1), d_off, expect


def cpu_sample(m, threads, CO, rng, kseeds, kpks):
    """m credentials of the cfg2 workload on the host, corrupted exactly like the GPU arm's."""
    idx = np.arange(m)
    ki = idx % N_KEYS
    msgs = rng.integers(0, 256, (m, MSG_LEN), dtype=np.uint8)
    off = np.arange(m + 1, dtype=np.uint64) * MSG_LEN
    sigs = CO.ed25519_sign_batch(kseeds[ki].copy(), msgs.reshape(-1), off, threads)
    fm = idx[idx % 100 == 0]
    bit = (fm // 100) % (MSG_LEN * 8)
    msgs[fm, bit // 8] ^= (1 << (bit % 8)).astype(np.uint8)
    sigs[idx % 100 == 50, 33] ^= 0x08
    expect = m - int(((idx % 100 == 0) | (idx % 100 == 50)).sum())
    return kpks[ki].copy(), sigs, msgs.reshape(-1), off, expect


def cpu_reference_rate(threads, budget_s=12.0, impl="oracle"):
    """Oracle C port (Go's algorithm: 51-bit limbs, NAF-5/NAF-8 vartime double-scalar mult) — or OpenSSL through the same batch
    driver — on `threads` host threads over a bounded sample of the same workload.  Returns (verifies/s, sample size)."""
    from oracle import c_oracle as CO
    rng = np.random.default_rng(0xAF02)
    kseeds = rng.integers(0, 256, (N_KEYS, 32), dtype=np.uint8)
    kpks = CO.ed25519_pubkey_batch(kseeds, threads)
    pk, sg, ms, off, _ = cpu_sample(4096 * max(1, threads // 8), threads, CO, rng, kseeds, kpks)
    t0 = time.perf_counter()
    CO.ed25519_verify_batch(pk[:2048], sg[:2048], ms, off[:2049], 1, impl=impl)
    cpu_reference_rate.single_thread = 2048 / (time.perf_counter() - t0)
    t0 = time.perf_counter()
    CO.ed25519_verify_batch(pk, sg, ms, off, threads, impl=impl)
    rate0 = (len(off) - 1) / (time.perf_counter() - t0)
    m = int(min(N_ITEMS, max(8192, rate0 * budget_s)))
    pk, sg, ms, off, expect = cpu_sample(m, threads, CO, rng, kseeds, kpks)
    t0 = time.perf_counter()
    ok = CO.ed25519_verify_batch(pk, sg, ms, off, threads, impl=impl)
    dt = time.perf_counter() - t0
    assert int(ok.sum()) == expect
    return m / dt, m


def cpu_baseline_block(threads, budget_s=12.0):
    rate, sample = cpu_reference_rate(threads, budget_s)
    single = cpu_reference_rate.single_thread
    blk = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
           "sample": "%d credentials of the same workload (same key schedule and corruption pattern); oracle/afc_oracle.c (C restatement of Go "
                     "crypto/ed25519: 51-bit limbs, NAF vartime double-scalar mult), %d pthreads (one thread alone: %.0f/s); the Go toolchain is "
                     "absent, so the reference itself cannot run" % (sample, threads, single)}
    try:        # BASELINE.md §3 B1: OpenSSL 3 through the same batch driver (oracle/afc_openssl.c), a second, independent CPU figure
        orate, osample = cpu_reference_rate(threads, min(budget_s, 6.0), impl="openssl")
        blk["openssl"] = {"value": orate, "unit": UNIT, "cores": threads,
                          "sample": "%d credentials, EVP_DigestVerify (OpenSSL 3), %d pthreads" % (osample, threads),
                          "single_thread": cpu_reference_rate.single_thread}
    except Exception as ex:
        blk["openssl"] = {"error": repr(ex)}
    return blk


def run_reference(args, rank, world):
    if rank != 0:
        return
    threads = host_threads()
    # each step = one bounded sample; scale the per-step budget so warmup+steps end within a few minutes
    budget = max(2.0, min(12.0, 150.0 / max(1, args.steps + args.warmup)))
    rates, sample = [], 0
    for i in range(args.warmup + args.steps):
        r, sample = cpu_reference_rate(threads, budget)
        if i >= args.warmup:
            rates.append(r)
    value = float(np.mean(rates))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * sample / value, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
        "data": "synthetic", "config": dict(CONFIG),
        "run": {"sample_per_step": sample, "threads": threads},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": "%d credentials of that workload per step (bounded CPU sample); oracle/afc_oracle.c (C restatement of Go crypto/ed25519: "
                                   "51-bit limbs, NAF vartime double-scalar mult), %d pthreads (one thread alone: %.0f/s); Go toolchain absent so the "
                                   "reference itself cannot run" % (sample, threads, cpu_reference_rate.single_thread)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------------
def pinned_like(lib, t):
    """A pinned host copy of device tensor t, allocated through the library (afc_alloc_pinned) AFTER the NUMA binding."""
    import ctypes as C
    import torch
    nbytes = t.numel() * t.element_size()
    p = lib.afc_alloc_pinned(max(nbytes, 1))
    if not p:
        raise MemoryError("afc_alloc_pinned(%d)" % nbytes)
    buf = (C.c_uint8 * nbytes).from_address(p)
    h = torch.frombuffer(buf, dtype=torch.uint8).view(t.dtype).view(t.shape)
    h.copy_(t)
    return h, p


def timed_loop(fn, steps, barrier):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    barrier()
    return e0.elapsed_time(e1)


def dump_outputs(out_dir, arrays):
    """Write device tensors as out_dir/<name>.npy in float32.  The inputs are seeded, so the files of two builds run with the same
    arguments can be compared item by item."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy().astype(np.float32))


def cfg4_block(ctx, dev, rank, world, barrier, reps=3):
    """BASELINE configs[3]: 2^22 sign + RFC 6962 append over the ranks, NCCL all-gather of the subtree roots, fold; timed on the
    device (max over ranks), then checked against a single-rank recomputation of the whole log on rank 0."""
    import torch
    import torch.distributed as dist
    import agentfield_b200 as afb
    n_total = CFG4_LEAVES
    per = n_total // world                     # 2^22 / {1,2,4,8}: contiguous, 2^k-aligned ranges (agentfield_b200/shard.py)
    rng = np.random.default_rng(0xAF04)
    kseeds = torch.from_numpy(rng.integers(0, 256, (N_KEYS, 32), dtype=np.uint8)).to(dev)
    d_exp = torch.empty((N_KEYS, 96), dtype=torch.uint8, device=dev)
    ctx.expand_dev(kseeds, N_KEYS, d_exp)

    def shard_msgs(g):
        gen = torch.Generator(device=dev); gen.manual_seed(0xAF0400 + g)
        return torch.randint(0, 256, (per, MSG_LEN), dtype=torch.uint8, device=dev, generator=gen)
    msgs = shard_msgs(rank)
    off = torch.arange(per + 1, device=dev, dtype=torch.int64) * MSG_LEN
    ki = ((torch.arange(per, device=dev) + rank * per) % N_KEYS).to(torch.int32)
    sigs = torch.empty((per, 64), dtype=torch.uint8, device=dev)
    soff = torch.arange(per + 1, device=dev, dtype=torch.int64) * 64
    local = torch.zeros(32, dtype=torch.uint8, device=dev)
    allr = torch.zeros(world * 32, dtype=torch.uint8, device=dev)
    groot = torch.zeros(32, dtype=torch.uint8, device=dev)
    aud, top = afb.Auditor(ctx), afb.Auditor(ctx)
    empty = aud.save()

    def once():
        aud.load(empty); top.load(empty)
        ctx.sign_expanded_dev(d_exp, ki, msgs.view(-1), off, per, sigs)          # E1: 2^22 / world signatures
        aud.append_dev(sigs.view(-1), soff, per)                                  # M1: leaf = the 64-byte signature
        aud.root_dev(local)
        if world > 1:
            dist.all_gather_into_tensor(allr, local)                              # the one exchange step: world x 32 bytes over NCCL
        else:
            allr.copy_(local)
        top.append_hashes_dev(allr, world)                                        # every rank folds the top log2(world) levels itself
        top.root_dev(groot)
    once(); torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(); once(); e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        times.append(float(t.item()))
    ms = min(times)
    root = bytes(groot.cpu().tolist())
    # the same with the other fixed-base multiplication for the nonces (default: constant time; the fast path gathers from the
    # radix-65536 table at addresses made of nonce digits) — same signatures, same root
    mode = ctx.sign_mode()
    ctx.sign_configure(mode != "constant-time")
    once(); torch.cuda.synchronize()
    other = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(); once(); e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        other.append(float(t.item()))
    other_same_root = bytes(groot.cpu().tolist()) == root
    ctx.sign_configure(mode == "constant-time")
    # every rank must hold the same global root
    same = True
    if world > 1:
        r0 = groot.clone(); dist.broadcast(r0, 0)
        flag = torch.tensor([int(torch.equal(r0, groot))], device=dev); dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        same = bool(flag.item())
    blk = {"leaves_total": n_total, "leaves_per_gpu": per, "sign_mode": mode, "ms": ms, "signs_plus_appends_per_s": n_total / (ms * 1e-3),
           ("fast_variable_time_ms" if mode == "constant-time" else "constant_time_ms"): min(other), "other_mode_same_root": other_same_root,
           "root": root.hex(),
           "same_root_on_every_rank": same,
           "collective": "ncclAllGather of %d x 32 B subtree roots (torch.distributed, NCCL over NVLink)" % world if world > 1
           else "none (single GPU: the fold of one root)", "hbm_frac": 640.0 * per / (ms * 1e-3) / 1e9 / peaks()[0]}
    # single-rank recomputation of the whole log (rank 0, outside the timed region): shard by shard through ONE log
    if rank == 0:
        ref = afb.Auditor(ctx)
        for g in range(world):
            m = msgs if g == rank else shard_msgs(g)
            k2 = ((torch.arange(per, device=dev) + g * per) % N_KEYS).to(torch.int32)
            s2 = torch.empty((per, 64), dtype=torch.uint8, device=dev)
            ctx.sign_expanded_dev(d_exp, k2, m.view(-1), off, per, s2)
            ref.append_dev(s2.view(-1), soff, per)
            torch.cuda.synchronize()
            del s2
        r2 = torch.zeros(32, dtype=torch.uint8, device=dev)
        ref.root_dev(r2); torch.cuda.synchronize()
        blk["root_ok"] = bool(bytes(r2.cpu().tolist()) == root) and same
        ref.close()
    aud.close(); top.close()
    return blk


def cfg3_block(ctx, dev):
    """BASELINE configs[2]: HMAC-SHA256 over 10 M x 256 B bodies with one 32-byte secret per message (worst case), one GPU."""
    import torch
    n = CFG3_ITEMS
    g = torch.Generator(device=dev); g.manual_seed(0xAF03)
    bodies = torch.randint(0, 256, (n, 256), dtype=torch.uint8, device=dev, generator=g)
    keys = torch.randint(0, 256, (n, 32), dtype=torch.uint8, device=dev, generator=g)
    off = torch.arange(n + 1, device=dev, dtype=torch.int64) * 256
    koff = (torch.arange(n + 1, device=dev, dtype=torch.int64) * 32).to(torch.int32)
    tags = torch.empty((n, 32), dtype=torch.uint8, device=dev)
    fn = lambda: ctx.hmac_sha256_dev(keys.view(-1), koff, bodies.view(-1), off, n, tags)
    fn(); torch.cuda.synchronize()
    ms = timed_loop(fn, 5, torch.cuda.synchronize) / 5
    # spot check against hashlib
    import hashlib
    import hmac
    pick = [0, 1, n // 2, n - 1]
    hb, hk, ht = bodies[pick].cpu().numpy(), keys[pick].cpu().numpy(), tags[pick].cpu().numpy()
    ok = all(hmac.new(bytes(hk[i]), bytes(hb[i]), hashlib.sha256).digest() == bytes(ht[i]) for i in range(len(pick)))
    return {"items": n, "body_len": 256, "key_len": 32, "ms": ms, "msgs_per_s": n / (ms * 1e-3), "hbm_frac": 320.0 * n / (ms * 1e-3) / 1e9 / peaks()[0],
            "spot_check_ok": ok}


def issuer_mix_block(ctx, dev, rank, steps):
    """How the verify call degrades when the issuers do not fit the round-1 sweet spot: 4096 issuers x 244 credentials (all hot,
    4x the tables to build), and a 50/50 mix — half of the batch from 512 hot issuers, half from keys that appear once (cold,
    generic kernel in the same call).  Cache emptied before every step, as in the headline."""
    import torch
    out = {}
    for name, kw in (("4096_issuers", dict(n_keys=4096)), ("half_hot_half_distinct", dict(n_keys=512, distinct_tail=N_ITEMS // 2))):
        d_pks, d_sigs, d_msgs, d_off, expect = make_workload(ctx, dev, rank, seed=0xAF07, **kw)
        d_ok = torch.empty(N_ITEMS, dtype=torch.uint8, device=dev)

        def step():
            ctx.keycache_clear()
            ctx.verify_dev(d_pks, d_sigs, d_msgs, d_off, N_ITEMS, d_ok)
        step(); step(); torch.cuda.synchronize()
        assert torch.equal(d_ok, expect), name
        ms = timed_loop(step, steps, torch.cuda.synchronize) / steps
        st = ctx.keycache_stats()
        out[name] = {"ms_per_step": ms, "value": N_ITEMS / (ms * 1e-3), "unit": UNIT, "hot": st["last_hot"], "cold": st["last_cold"],
                     "tables_built": st["last_built"]}
        del d_pks, d_sigs, d_msgs, d_off, d_ok
    out["note"] = "per-key decision on the device: cached or frequent keys through tables, the rest through the generic kernel in the same call"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="headline + cfg4 only (quick A/B runs)")
    ap.add_argument("--ab", action="store_true", help="headline + warm_keycache + keyed only (kernel A/B runs)")
    ap.add_argument("--soak", type=float, default=0.0, help="BASELINE configs[4]: sustained mixed ingest for this many seconds (own JSON line)")
    ap.add_argument("--soak-rate", type=float, default=100_000.0, help="whole-job target rate of --soak, actions/s")
    ap.add_argument("--extras", action="store_true", help="also time sign / canonical form / microbenchmarks")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (the 1 M-entry verify bitmap, 4 MB) as DIR/verify_ok.npy "
                         "in float32; rank 0 only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3

    numa = bind_to_gpu_numa_node(local_rank)           # before torch / CUDA allocate anything pinned
    # NCCL's own init lines (ranks, transports) go to stderr so that a reader of the run can see how many ranks joined;
    # stdout carries the one JSON line only
    nccl_log = None
    if world > 1:
        # (NCCL writes its debug lines to STDOUT unless told otherwise, and /dev/stderr as NCCL_DEBUG_FILE was ignored on the pool's
        # boxes: each rank logs to a file of its own and copies it to stderr once the communicator is up)
        nccl_log = "/tmp/afc_nccl_rank%d_%d.log" % (rank, os.getpid())
        os.environ["NCCL_DEBUG"] = os.environ.get("AFC_NCCL_DEBUG", "INFO")
        os.environ["NCCL_DEBUG_SUBSYS"] = os.environ.get("AFC_NCCL_DEBUG_SUBSYS", "INIT")
        os.environ["NCCL_DEBUG_FILE"] = nccl_log
    import torch
    import torch.distributed as dist
    import agentfield_b200 as afb

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    ctx = afb.Context(local_rank)
    info = ctx.device_info()
    numa["library"] = ctx.numa_info()                  # what the library's own staging pools bind to (sysfs local_cpulist of the GPU)
    bad = ctx.selftest(200)
    if bad:
        raise SystemExit("PTX field self-test failed on %d threads" % bad)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if world > 1:
        barrier()                                      # the first collective creates the communicator: its init lines are in the log now
        try:
            with open(nccl_log) as f:
                for ln in f:
                    if rank == 0 or "Init COMPLETE" in ln or "nranks" in ln.lower():
                        sys.stderr.write(ln)
            sys.stderr.flush()
        except OSError as ex:
            sys.stderr.write("bench.py: NCCL log %s not readable: %r\n" % (nccl_log, ex))

    if args.soak > 0:
        soak(args, ctx, dev, rank, world, barrier, numa)
        if world > 1:
            dist.destroy_process_group()
        return

    d_pks, d_sigs, d_msgs, d_off, expect = make_workload(ctx, dev, rank)
    n = N_ITEMS
    d_ok = torch.empty(n, dtype=torch.uint8, device=dev)

    # ---------------- device-resident timing (value)
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    ctx.verify_dev(d_pks, d_sigs, d_msgs, d_off, n, d_ok)          # cold: the issuer-key cache is empty, tables get built in this call
    c1.record()
    torch.cuda.synchronize()
    cold_ms = c0.elapsed_time(c1)

    def step():
        # Nothing is carried from one step to the next: the issuer-key cache is emptied first, so de-duplication, the 1024
        # per-key tables and all 10^6 verifications are redone inside every timed step.
        ctx.keycache_clear()
        ctx.verify_dev(d_pks, d_sigs, d_msgs, d_off, n, d_ok)

    for _ in range(args.warmup):
        step()
    barrier()
    assert torch.equal(d_ok, expect), "verify bitmap differs from the corruption pattern"
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = ctx.launch_count()
    ctx.profile_begin(64 + 32 * args.steps)      # per-kernel CUDA events on the launching stream (one pair per launch, claimed lazily)
    ms_total = timed_loop(step, args.steps, barrier)
    prof = ctx.profile_end()
    launches = ctx.launch_count() - launches0
    clocks = sampler.stop()
    assert torch.equal(d_ok, expect)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"verify_ok": d_ok})
    t_ms = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_step = float(t_ms.item()) / args.steps
    value = world * n / (ms_step * 1e-3)

    # ---------------- end to end through the C-ABI host call (pinned host buffers, H2D + D2H inside)
    lib, H = afb._abi.load(), ctx.handle
    hp = [pinned_like(lib, t) for t in (d_pks, d_sigs, d_msgs, d_off)]
    h_pks, h_sigs, h_msgs, h_off = (h for h, _ in hp)
    h_ok, p_ok = pinned_like(lib, d_ok)

    def e2e_step():
        ctx.keycache_clear()
        rc = lib.afc_ed25519_verify_batch(H, h_pks.data_ptr(), h_sigs.data_ptr(), h_msgs.data_ptr(), h_off.data_ptr(), n, h_ok.data_ptr())
        if rc != 0:
            raise afb.AfcError(rc, lib.afc_last_cuda_error(H).decode())

    e2e_step()
    assert torch.equal(h_ok, expect.cpu())
    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    t_e = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
    e2e_value = world * n * args.steps / float(t_e.item())
    h2d = n * (32 + 64 + MSG_LEN) + (n + 1) * 8
    d2h = n
    # the transfer floor of that call: the same pinned buffers copied to the device with nothing else going on
    scratch = [torch.empty_like(t, device=dev) for t in (h_pks, h_sigs, h_msgs, h_off)]
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    for rep in range(3):
        if rep == 1:
            c0.record()
        for dst, src in zip(scratch, (h_pks, h_sigs, h_msgs, h_off)):
            dst.copy_(src, non_blocking=True)
    c1.record(); torch.cuda.synchronize()
    t_h = torch.tensor([c0.elapsed_time(c1) / 2], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_h, op=dist.ReduceOp.MAX)
    h2d_only_ms = float(t_h.item())
    del scratch
    e2e_extra = {"ms_per_step": 1e3 * float(t_e.item()) / args.steps, "h2d_only_ms": h2d_only_ms, "pcie_h2d_GBps": h2d / h2d_only_ms / 1e6,
                 "numa": numa,
                 "note": "h2d_only_ms = the step's inputs copied from the same pinned buffers with no compute, all ranks at once (max over ranks): "
                         "the transfer floor of the host call"}

    # ---------------- roofline of the dominant kernel
    hbm_peak, peak_src = peaks()
    zero = {"avg_ms": float("nan"), "count": 0, "total_ms": 0.0}
    dom = max(("k_ed_verify_cached_dyn", "k_ed_verify_cached", "k_ed_verify_quad", "k_ed_verify"), key=lambda k: prof.get(k, zero)["total_ms"])
    kv = prof.get(dom, zero)
    achieved = ALGO_BYTES * n / (kv["avg_ms"] * 1e-3) / 1e9 if kv["count"] else float("nan")
    traffic, traffic_src = None, None
    for cand in ("r02_ncu_traffic.json", "r01_e_ncu_traffic.json"):     # dram__bytes_read.sum + dram__bytes_write.sum from the committed ncu --set full capture
        try:
            tk = json.load(open(os.path.join(ROOT, "profiles", cand)))["kernels"]
            if dom in tk:
                traffic, traffic_src = tk[dom].get("traffic_bytes"), "profiles/" + cand
                break
        except Exception:
            pass
    step_gbs = ALGO_BYTES * n / (ms_total / args.steps * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "algorithmic_bytes_per_launch": ALGO_BYTES * n,
                "kernel_avg_ms": kv["avg_ms"], "kernel_launches_timed": kv["count"], "kernel_share_of_step": kv["total_ms"] / max(ms_total, 1e-9),
                "achieved_step": step_gbs, "frac_step": step_gbs / hbm_peak,
                "other_kernels_ms": {k: v["avg_ms"] for k, v in prof.items() if k != dom and v["count"] and k != "(untimed)"},
                "untimed_launches": prof.get("(untimed)", {}).get("count", 0),
                "note": "integer-multiplier (IMAD.WIDE) bound: see DESIGN.md section 4; HBM fraction reported because the metric asks for it. "
                        "frac charges all 609 B to the dominant kernel, frac_step to the whole step (hashing + table build + verify); kernels on the "
                        "side streams overlap the hashing, so the per-kernel times add up to more than the step"}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": dict(CONFIG),
        "run": {"l2": "inputs (609 MB per step) larger than L2 (126 MB)",
                "parallelism": ("independent shards, no collective on the verify path; cfg4 all-gathers the audit roots over NCCL" if world > 1
                                else "single GPU"), "sm_count": info["sm_count"], "keycache": "emptied before every step"},
        "clocks": clocks, "e2e": dict({"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h}, **e2e_extra),
        "gpu_launches": int(launches), "roofline": roofline, "impl": "b200",
    }
    del h_pks, h_sigs, h_msgs, h_off, h_ok
    for _, p in hp:
        lib.afc_free_pinned(p)
    lib.afc_free_pinned(p_ok)
    del hp

    # ---------------- BASELINE configs[3]: 2^22 sign + audit append sharded over the ranks, NCCL all-gather of the roots
    try:
        line["cfg4"] = cfg4_block(ctx, dev, rank, world, barrier) if not args.ab else {"skipped": "--ab"}
    except Exception as ex:
        line["cfg4"] = {"error": repr(ex)}
    torch.cuda.empty_cache()

    if not args.no_secondary:
        # ---------------- secondary: steady state of a long-running verifier (tables of known issuers stay cached between calls)
        try:
            for _ in range(max(5, args.warmup)):             # the sections before this one leave the SMs mostly idle: let the clocks settle
                ctx.verify_dev(d_pks, d_sigs, d_msgs, d_off, n, d_ok)
            wms = timed_loop(lambda: ctx.verify_dev(d_pks, d_sigs, d_msgs, d_off, n, d_ok), args.steps, barrier) / args.steps
            assert torch.equal(d_ok, expect)
            line["warm_keycache"] = {"value": world * n / (wms * 1e-3), "unit": UNIT, "ms_per_step": wms,
                                     "note": "same call without clearing the issuer-key cache between steps (tables of the 1024 issuers reused)"}
        except Exception as ex:
            line["warm_keycache"] = {"error": repr(ex)}

        # ---------------- secondary: the generic double-scalar kernel alone (issuer-key cache disabled: what a batch of all-distinct keys costs)
        kc_info = ctx.keycache_stats()
        kc_info["cold_first_call_ms"] = cold_ms       # first call on an empty cache (1 M credentials, 1024 tables built inside it)
        line["keycache"] = kc_info
        try:
            if args.ab:
                raise RuntimeError("skipped (--ab)")
            ctx.keycache_configure(0)
            for _ in range(2):
                ctx.verify_dev(d_pks, d_sigs, d_msgs, d_off, n, d_ok)
            barrier()
            assert torch.equal(d_ok, expect)
            gsteps = max(3, min(args.steps, 20))
            gms = timed_loop(lambda: ctx.verify_dev(d_pks, d_sigs, d_msgs, d_off, n, d_ok), gsteps, barrier) / gsteps
            line["no_keycache"] = {"value": world * n / (gms * 1e-3), "unit": UNIT, "ms_per_step": gms,
                                   "hbm_frac": ALGO_BYTES * n / (gms * 1e-3) / 1e9 / hbm_peak,
                                   "note": "same call with afc_keycache_configure(ctx, 0): generic Straus kernel, no per-key tables"}
        except Exception as ex:
            line["no_keycache"] = {"error": repr(ex)}
        finally:
            ctx.keycache_configure(kc_info["max_keys"])
            kc_info["note"] = ("value and e2e empty the issuer-key cache before every step (tables rebuilt inside the timed region); "
                               "warm_keycache keeps them between steps; no_keycache disables the cache (generic kernel); cold_first_call_ms "
                               "additionally includes the one-time device allocations")

        # ---------------- secondary: the same batch verified against a registered key set (identity cache, SURVEY.md §8f N1)
        try:
            t0 = time.perf_counter()
            kpks = d_pks[:N_KEYS].cpu().numpy()                      # key i occupies rows i, i + K, ... (key_i = i mod K)
            ks = afb.KeySet([bytes(p) for p in kpks], ctx)
            build_s = time.perf_counter() - t0
            d_ki = (torch.arange(n, device=dev) % N_KEYS).to(torch.int32)
            for _ in range(2):
                ks.verify_dev(d_ki, d_sigs, d_msgs, d_off, n, d_ok)
            barrier()
            assert torch.equal(d_ok, expect), "keyed verify bitmap differs"
            kms = timed_loop(lambda: ks.verify_dev(d_ki, d_sigs, d_msgs, d_off, n, d_ok), args.steps, barrier) / args.steps
            line["keyed"] = {"value": world * n / (kms * 1e-3), "unit": UNIT, "ms_per_step": kms, "keyset_build_s": build_s,
                             "table_bytes": ks.info()["table_bytes"], "hbm_frac": ALGO_BYTES * n / (kms * 1e-3) / 1e9 / hbm_peak,
                             "note": "afc_ed25519_verify_keyed_batch_dev: issuer keys registered once (per-key radix-256 tables), same inputs and bitmap"}
            ks.close()
        except Exception as ex:     # secondary figure only
            line["keyed"] = {"error": repr(ex)}
        del d_pks, d_sigs, d_msgs, d_off, d_ok
        torch.cuda.empty_cache()
        if world == 1 and not args.ab:
            try:
                line["issuer_mix"] = issuer_mix_block(ctx, dev, rank, max(3, min(args.steps, 10)))
            except Exception as ex:
                line["issuer_mix"] = {"error": repr(ex)}
            torch.cuda.empty_cache()
            try:
                line["cfg3"] = cfg3_block(ctx, dev)
            except Exception as ex:
                line["cfg3"] = {"error": repr(ex)}
            torch.cuda.empty_cache()

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        unbind_for_cpu_legs()
        line["cpu_baseline"] = cpu_baseline_block(host_threads(), 12.0)
    if args.extras:
        line["extras"] = extras(ctx, dev, world, rank)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def soak(args, ctx, dev, rank, world, barrier, numa):
    """BASELINE configs[4]: open-loop Poisson arrivals at --soak-rate actions/s over the whole job (rate / world per GPU), each
    action = Ed25519 sign (512 B) + HMAC-SHA256 (256 B) + one audit-log leaf, through the native dispatcher (csrc/afc_ingest.cu);
    the per-rank audit roots are all-gathered over NCCL at the end.  The CPU leg: the oracle's C port doing the same three
    operations per action on all host threads, bounded sample (rank 0)."""
    import torch
    import torch.distributed as dist
    import agentfield_b200 as afb
    from agentfield_b200 import shard
    rng = np.random.default_rng(0xAF05)
    ing = afb.Ingest(ctx.expand(rng.integers(0, 256, (64, 32), dtype=np.uint8)), ctx, batch_max=4096, linger_us=500, max_msg=512, max_key=32, max_body=256)
    ing.soak(args.soak_rate / world, 1.0, producers=2, seed=0xAF05 + rank)            # warm-up second
    barrier()
    res = ing.soak(args.soak_rate / world, args.soak, producers=4, seed=0xAF0500 + rank)
    barrier()
    peak = ing.soak(1_000_000, min(5.0, args.soak), producers=8, seed=0xAF0550 + rank)   # what one GPU sustains when pushed
    st = ing.stats()
    ing.close()
    vals = torch.tensor([res["achieved_rate"], res["p50_us"], res["p99_us"], res["max_us"], res["late_submits"], res["completed"], peak["achieved_rate"],
                         peak["p99_us"]], dtype=torch.float64, device=dev)
    if world > 1:
        summed = vals.clone(); dist.all_reduce(summed, op=dist.ReduceOp.SUM)
        maxed = vals.clone(); dist.all_reduce(maxed, op=dist.ReduceOp.MAX)
        roots = shard.allgather_roots(bytes.fromhex(st["log_root"]))
        global_root = afb.fold_roots(np.frombuffer(b"".join(roots), dtype=np.uint8), ctx).hex()
    else:
        summed, maxed, global_root = vals, vals, st["log_root"]
    if rank != 0:
        return
    line = {"metric": "sustained mixed ingest, agent-actions/s (Ed25519 sign 512 B + HMAC-SHA256 256 B + audit append)", "value": float(summed[0]),
            "unit": "actions/s", "n_gpus": world, "seconds": args.soak, "target_rate": args.soak_rate, "higher_is_better": True, "scaling": "strong",
            "data": "synthetic", "impl": "b200", "dtype": "u32",
            "config": {"workload": "BASELINE.json configs[4]: sustained mixed ingest, %g actions/s over %d GPU(s), %g s" % (args.soak_rate, world, args.soak),
                       "arrivals": "open-loop Poisson, 4 producer threads per GPU", "batch_max": 4096, "linger_us": 500},
            "latency_us": {"p50_max_over_ranks": float(maxed[1]), "p99_max_over_ranks": float(maxed[2]), "max": float(maxed[3])},
            "late_submits": int(summed[4]), "completed": int(summed[5]), "audit_root_of_rank_logs": global_root,
            "collective": "ncclAllGather of the %d per-rank audit roots" % world if world > 1 else "none",
            "pushed": {"target_rate_per_gpu": 1_000_000, "achieved_rate": float(summed[6]), "p99_us_max_over_ranks": float(maxed[7])}, "numa": numa}
    if not args.no_cpu_baseline:
        unbind_for_cpu_legs()
        line["cpu_baseline"] = cpu_ingest_rate(host_threads())
    print(json.dumps(line), flush=True)


def cpu_ingest_rate(threads, budget_s=10.0):
    """The same action on the host: sign (from the seed, as the reference does per VC) + HMAC + RFC 6962 leaf hash, oracle C port."""
    from oracle import c_oracle as CO
    rng = np.random.default_rng(0xAF05)
    m = 2048 * max(1, threads // 4)
    seeds = rng.integers(0, 256, (64, 32), dtype=np.uint8)

    def run(m):
        msgs = rng.integers(0, 256, (m, MSG_LEN), dtype=np.uint8); off = np.arange(m + 1, dtype=np.uint64) * MSG_LEN
        bodies = rng.integers(0, 256, (m, 256), dtype=np.uint8); boff = np.arange(m + 1, dtype=np.uint64) * 256
        keys = rng.integers(0, 256, (m, 32), dtype=np.uint8); koff = np.arange(m + 1, dtype=np.uint32) * 32
        sd = seeds[np.arange(m) % 64].copy()
        t0 = time.perf_counter()
        sigs = CO.ed25519_sign_batch(sd, msgs.reshape(-1), off, threads)
        CO.hmac_sha256_batch(keys.reshape(-1), koff, bodies.reshape(-1), boff, threads)
        CO.merkle_root(sigs.reshape(-1), np.arange(m + 1, dtype=np.uint64) * 64, threads)
        return m / (time.perf_counter() - t0)
    r0 = run(m)
    m2 = int(min(2_000_000, max(m, r0 * budget_s)))
    r = run(m2)
    return {"value": r, "unit": "actions/s", "cores": threads, "kind": "port",
            "sample": "%d actions (sign from seed + HMAC + Merkle root over the signatures), oracle/afc_oracle.c on %d pthreads" % (m2, threads)}


def extras(ctx, dev, world, rank):
    """Further secondary figures (not the headline): SHA-256, sign, Merkle append alone, canonical form, register-only microbenchmarks."""
    import torch
    import agentfield_b200 as afb
    out = {}
    g = torch.Generator(device=dev); g.manual_seed(0xAF03 + rank)

    def timed(fn, reps=3):
        fn(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    hbm_peak, _ = peaks()
    n = 4_000_000
    bodies = torch.randint(0, 256, (n, 256), dtype=torch.uint8, device=dev, generator=g)
    off = torch.arange(n + 1, device=dev, dtype=torch.int64) * 256
    dig = torch.empty((n, 32), dtype=torch.uint8, device=dev)
    ms = timed(lambda: ctx.sha256_dev(bodies.view(-1), off, n, dig))
    out["sha256_256B"] = {"msgs_per_s": n / (ms * 1e-3), "ms": ms, "hbm_frac": 288 * n / (ms * 1e-3) / 1e9 / hbm_peak}
    del bodies, dig
    n = 1 << 19
    rng = np.random.default_rng(0xAF04)
    kseeds = torch.from_numpy(rng.integers(0, 256, (N_KEYS, 32), dtype=np.uint8)).to(dev)
    d_exp = torch.empty((N_KEYS, 96), dtype=torch.uint8, device=dev)
    ctx.expand_dev(kseeds, N_KEYS, d_exp)
    msgs = torch.randint(0, 256, (n, MSG_LEN), dtype=torch.uint8, device=dev, generator=g)
    off = torch.arange(n + 1, device=dev, dtype=torch.int64) * MSG_LEN
    ki = (torch.arange(n, device=dev) % N_KEYS).to(torch.int32)
    sigs = torch.empty((n, 64), dtype=torch.uint8, device=dev)
    ms_sign = timed(lambda: ctx.sign_expanded_dev(d_exp, ki, msgs.view(-1), off, n, sigs))
    out["sign_512B_expanded_keys"] = {"signs_per_s": n / (ms_sign * 1e-3), "ms": ms_sign}
    seeds_full = kseeds[ki.long()].contiguous()
    ms_sign2 = timed(lambda: ctx.sign_dev(seeds_full, msgs.view(-1), off, n, sigs), reps=2)
    out["sign_512B_from_seeds"] = {"signs_per_s": n / (ms_sign2 * 1e-3), "ms": ms_sign2}
    soff = torch.arange(n + 1, device=dev, dtype=torch.int64) * 64
    root_dev = torch.empty(32, dtype=torch.uint8, device=dev)
    aud = afb.Auditor(ctx)
    empty_log = aud.save()

    def append_ms():
        aud.load(empty_log)                                   # same log object every time: its level buffers are allocated once
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        aud.append_dev(sigs.view(-1), soff, n)
        aud.root_dev(root_dev)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)
    append_ms()
    ms_m = min(append_ms() for _ in range(3))
    aud.close()
    out["merkle_append_64B_leaves"] = {"leaves_per_s": n / (ms_m * 1e-3), "ms": ms_m}
    # canonical form on the device: 2^19 VCDocument-shaped documents (23 values of 32 bytes), values as in real credentials (DIDs,
    # base64url hashes, timestamps: nothing to escape) and with 6 % of the bytes being characters Go escapes
    try:
        from agentfield_b200 import canonical as CA
        tmpl = CA.vc_document_template(False, ctx)
        F, flen = tmpl.n_fields, 32
        lib, P, st = afb._abi.load(), afb._abi.ptr, torch.cuda.current_stream().cuda_stream
        plain = list(b"abcdefghijklmnopqrstuvwxyzABCDEFGHIJKLMNOPQRSTUVWXYZ0123456789-_:/")
        kinds_t = torch.tensor(tmpl.kinds, device=dev)
        raw_cols = torch.nonzero(kinds_t == CA.RAW).flatten()
        d_voff = torch.arange(n * F + 1, device=dev, dtype=torch.int64) * flen
        res = {}
        for label, alphabet in (("plain_values", plain), ("6pct_escaped", plain + [0x22, 0x3c, 0x0a, 0x5c])):
            table = torch.tensor(alphabet, dtype=torch.uint8, device=dev)
            d_vals = table[torch.randint(0, table.numel(), (n * F * flen,), device=dev, generator=torch.Generator(device=dev).manual_seed(5))]
            d_vals.view(n, F, flen)[:, raw_cols, :] = 0x31          # RAW members must be valid JSON on their own: digits
            d_doc, d_doff = tmpl.fill_dev(d_vals, d_voff, n)
            total = int(d_doff[-1].item())

            def both_passes():                               # output buffers allocated once, as a long-running issuer would
                lib.afc_json_fill_sizes_dev(ctx.handle, P(tmpl.d_segs), P(tmpl.d_seg_off), P(tmpl.d_kinds), F, P(d_vals), P(d_voff), n, P(d_doff), None, st)
                lib.afc_json_fill_dev(ctx.handle, P(tmpl.d_segs), P(tmpl.d_seg_off), P(tmpl.d_kinds), F, P(d_vals), P(d_voff), n, P(d_doff), P(d_doc), st)
            both_passes(); torch.cuda.synchronize()
            ctx.profile_begin()                               # per-kernel CUDA events over the same launches the total is taken from
            ms_c = timed(both_passes, reps=5)
            kms = {k: v["avg_ms"] for k, v in ctx.profile_end().items()}
            res[label] = {"docs_per_s": n / (ms_c * 1e-3), "ms": ms_c, "kernels_ms": kms, "bytes_out": total, "bytes_in": int(d_vals.numel()),
                          "hbm_frac": (total + d_vals.numel() * 2 + 8 * (n * F + n)) / (ms_c * 1e-3) / 1e9 / hbm_peak}
            del d_doc, d_doff, d_vals
        res["note"] = "sizes pass + scan + fill pass into preallocated buffers; values are read twice; one document per thread"
        out["canonical_form_vc_documents"] = res
    except Exception as ex:
        out["canonical_form_vc_documents"] = {"error": repr(ex)}
    mb = {}
    for name, which, iters in (("fe_mul", 0, 4000), ("fe_sq", 1, 4000), ("fe_addsub", 2, 20000), ("fe_mul_portable", 5, 2000),
                               ("fe_sq_via_mul", 6, 4000), ("fe_mul_schoolbook", 7, 4000), ("sha256_compress", 3, 2000), ("sha512_compress", 4, 1000),
                               ("pipe_imad32_x16", 11, 20000), ("pipe_alu_x16", 12, 20000)):
        ops, ms = ctx.microbench(which, iters)
        mb[name] = {"ops_per_s": ops, "ms": ms}
    out["microbench"] = mb
    return out


if __name__ == "__main__":
    main()
