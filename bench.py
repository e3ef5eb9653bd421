#!/usr/bin/env python
"""bench.py — routing decisions/s of the prefix-cache-aware Endpoint Picker hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--cfg 2|3|4|5] [--mode replicas|sharded] [--scale F] [--dump-outputs DIR]

One "step" = one pass of the hot path (hash → index lookup → weighted score → argmax)
over one batch of synthetic requests.  Default workload = BASELINE.json's headline
config 3: 16 384 requests × 1 024 endpoints × 4 096-token prompts (SURVEY.md §8d).

Prints ONE JSON line (rank 0):
  value     whole-job decisions/s with inputs already resident in HBM (device-timed,
            CUDA events on the launching stream, max over ranks)
  e2e       the same metric through the public C-ABI call with HOST (pinned) buffers:
            H2D of the prompts and D2H of the picks inside the timed region
  roofline  dominant kernel: algorithmic bytes per launch ÷ its CUDA-event duration,
            against MEASURED_PEAKS.json's HBM copy bandwidth
  cpu_baseline  the CPU oracle (C++ restatement of the upstream algorithm; the
            reference's Go path is neither in /root/reference nor compilable here,
            SURVEY.md §0 F1/F2) timed on a bounded sample on the host cores

Multi-GPU (torchrun, one rank per GPU): --mode replicas (default: the 1 024-endpoint
pool fits one GPU, so every GPU is an independent replica serving its own batches —
SURVEY.md §8e) or --mode sharded (configs 4/5: endpoint-range shards + the library's
exchange of presence masks and (score, endpoint) pairs — in-kernel peer-memory stores over
NVLink by default, FI_EPP_EXCHANGE=nccl for the two-all-gather path).
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
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from

import numpy as np  # noqa: E402

METRIC = "routing decisions/sec (4K-tok prompts x 1024 endpoints); achieved HBM GB/s"
ORACLE_LABEL = ("C++ restatement of the upstream EPP v1.2.1 algorithm (oracle/epp_oracle.cpp); the reference's Go "
                "path is not in /root/reference and cannot be compiled here (SURVEY.md F1/F2); parity unpinned by "
                "reference tests")


def log(*a):
    if int(os.environ.get("RANK", "0")) == 0:
        print("[bench]", *a, file=sys.stderr, flush=True)


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (copy, read+write)"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md); MEASURED_PEAKS.json absent"


class ClockSampler:
    """SM clock + throttle reasons around and DURING the timed region: in-process NVML, one sample right
    before the region, one every 10 ms inside it (the default run's region is ~30 ms — too short for
    `nvidia-smi -lms`), one right after; nvidia-smi as fallback.  Only the rank that prints the line samples
    (its own GPU), and sparsely: NVML calls contend with kernel launches on the driver — every rank polling at
    2 kHz took a 4-rank sharded step from 0.29 to 0.78 ms, rank 0 alone at 500 Hz still to 0.43 ms."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None
        self.nvml = None
        self.samples = []  # (sm_mhz, reasons bitmask)
        self.max_mhz = None
        self.stop_flag = False

    def start(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.gpu]) if vis and vis.split(",")[self.gpu].isdigit() else self.gpu
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            self._sample()  # right before the timed region (the warm-up has just run: clocks are at load level)
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _sample(self):
        n = self.nvml
        mhz = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
        try:
            rs = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
        except Exception:
            rs = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
        self.samples.append((mhz, rs))

    def _poll(self):
        while not self.stop_flag:
            time.sleep(0.010)
            if self.stop_flag:
                break
            try:
                self._sample()
            except Exception:
                pass

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.nvml is None and self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "source": "not sampled on this rank"}
        if self.nvml is not None:
            self.stop_flag = True
            self.t.join(timeout=2)
            try:
                self._sample()  # right after the last timed kernel
            except Exception:
                pass
            n = self.nvml
            bits = {"hw_slowdown": getattr(n, "nvmlClocksEventReasonHwSlowdown", 0x8),
                    "hw_thermal_slowdown": getattr(n, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                    "sw_thermal_slowdown": getattr(n, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                    "sw_power_cap": getattr(n, "nvmlClocksEventReasonSwPowerCap", 0x4)}
            sm = [a for a, _ in self.samples]
            reasons = sorted(k for k, b in bits.items() if any(r & b for _, r in self.samples))
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.max_mhz, "reasons": reasons,
                    "samples": len(sm), "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


def build_config(wl, cfg_id, begin, count, device, max_batch, mode, lru_capacity=0, base=None):
    from fusioninfer_b200 import make_config, synth

    profiles, pd = synth.baseline_profiles(cfg_id)
    slots = 4096
    mult = int(os.environ.get("FI_BENCH_SLOT_MULT", "2"))  # index load factor <= 1/mult
    # an endpoint-range shard is a directory of the WHOLE pool's keys (membership rows for its own endpoints)
    while slots < mult * (wl.E if mode == "sharded" else count) * wl.lru_capacity:
        slots *= 2
    return make_config(num_endpoints=wl.E, block_bytes=wl.block_bytes, max_blocks=wl.max_blocks, lru_capacity=lru_capacity,
                       max_batch=max_batch, max_prompt_bytes=max_batch * wl.T * 4, index_slots=slots, device=device,
                       endpoint_begin=begin, endpoint_count=count, profiles=profiles, pd=pd, base=base)


def algorithmic_bytes(wl, picks_nprobe_total, R, E_local, hashed_requests=None):
    """SURVEY.md §8d: A = 4·T + N_probe·(8 + E_local/8) + 16 per decision (hashed_requests: the requests THIS
    GPU hashes — R/world when a sharded pool splits the hashing)."""
    hr = R if hashed_requests is None else hashed_requests
    return {"hash_blocks": hr * 4 * wl.T, "match_pick": picks_nprobe_total * (8 + E_local / 8.0) + 16.0 * R}


def load_traffic():
    """dram bytes per launch of the dominant kernels from the committed ncu summary, if any."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        with open(p) as f:
            return json.load(f)
    except Exception:
        return {}


def host_cores():
    """Cores the CPU legs may use: the affinity mask capped by the cgroup CPU quota (os.cpu_count() ignores both)."""
    from oracle import epp_oracle as eo

    try:
        aff = len(os.sched_getaffinity(0))
    except Exception:
        aff = os.cpu_count() or 1
    return {"usable": eo.usable_cores(), "affinity": aff, "os_cpu_count": os.cpu_count() or 1}


def build_oracle(wl, cfg_id, ops_iter, log_label="oracle"):
    """The CPU restatement with the given index content; its configuration is filled by the oracle library."""
    from oracle import epp_oracle as eo

    t0 = time.time()
    o = eo.Oracle(build_config(wl, cfg_id, 0, wl.E, 0, max(wl.R, 1), "replicas", base=eo.default_config()))
    o.update_endpoints(wl.endpoint_states())
    for ops in ops_iter:
        o.index_apply(ops)
    log(f"{log_label} index built in {time.time() - t0:.1f}s")
    return o


def run_reference(args, wl, cfg_id):
    """--impl reference: the CPU restatement on the box's host cores, bounded sample per step.  Nothing of the
    product library is loaded in this process."""
    from fusioninfer_b200 import synth

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = host_cores()
    ncores = cores["usable"]
    o = build_oracle(wl, cfg_id, [], "oracle (empty)")
    o.index_reserve(wl.E * wl.lru_capacity)
    t0 = time.time()
    for ops in wl.index_ops(chunk_endpoints=128):
        o.index_apply(ops)
    log(f"oracle index built in {time.time() - t0:.1f}s")
    S = args.cpu_sample
    sub = synth.Workload(**{**wl.__dict__, "R": S})
    tok, offs = sub.prompts(batch=100)
    # Every thread walks its shard `rep` times per step (persistent worker pool, no thread spawn per call):
    # calibrate rep for up to ~1 s of wall time per step.
    t0 = time.perf_counter()
    o.pick_batch_repeat(tok, offs, wl.h0, nthreads=ncores, repeat=2)
    per_pass = (time.perf_counter() - t0) / 2
    target = min(1.0, 60.0 / max(args.steps + args.warmup, 1))
    rep = int(max(1, min(64, target / max(per_pass, 1e-6))))
    for _ in range(args.warmup):
        o.pick_batch_repeat(tok, offs, wl.h0, nthreads=ncores, repeat=rep)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        o.pick_batch_repeat(tok, offs, wl.h0, nthreads=ncores, repeat=rep)
    dt = time.perf_counter() - t0
    val = S * rep * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "decisions/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": workload_config(wl, cfg_id, "cpu"),
        "cpu_baseline": {"value": val, "unit": "decisions/s", "cores": ncores, "cores_detail": cores, "kind": "port",
                         "sample": f"{S} requests x {rep} passes of the same workload per step, full {wl.E}-endpoint index "
                                   f"({wl.E * wl.lru_capacity} entries), {ncores} persistent worker threads; {ORACLE_LABEL}"},
        "e2e": {"value": val, "unit": "decisions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


class stdout_to_stderr:
    """Point file descriptor 1 at stderr for the duration (native libraries print to fd 1 directly)."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


def workload_config(wl, cfg_id, parallelism):
    return {
        "workload": f"cfg{cfg_id}: {wl.R} req x {wl.E} endpoints x {wl.T}-token prompts (uint32), "
                    f"{wl.block_bytes} B blocks, <= {wl.max_blocks} blocks, {wl.lru_capacity} index entries/endpoint",
        "global_batch": wl.R, "endpoints": wl.E, "prompt_tokens": wl.T, "parallelism": parallelism,
        "l2": f"inputs larger than L2: {wl.R * wl.T * 4 / 2**20:.0f} MiB of prompts per step, rotating batches; "
              f"index {wl.E * wl.lru_capacity / 1e6:.1f} M entries",
    }


def bind_to_gpu_numa(local):
    """Run this rank on the cores of its GPU's NUMA node while it allocates and fills its pinned host buffers
    (pages are placed where the allocating thread runs), so that they are local to the GPU's PCIe root: on the
    8-GPU node GPUs 4-7 hang off NUMA node 1 (round 1: e2e 6.19 ms/step at N = 8 vs 5.04 at N = 1).
    Returns (note for the JSON line, function that restores the original affinity)."""
    try:
        original = os.sched_getaffinity(0)
    except Exception:  # noqa: BLE001
        return "numa: affinity not available", (lambda: None)

    def restore():
        try:
            os.sched_setaffinity(0, original)
        except Exception:  # noqa: BLE001
            pass

    try:
        import torch

        bus = torch.cuda.get_device_properties(local).pci_bus_id
        dom = torch.cuda.get_device_properties(local).pci_domain_id
        dev = torch.cuda.get_device_properties(local).pci_device_id
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0/numa_node"
        with open(path) as f:
            node = int(f.read().strip())
        if node < 0:
            return "numa: single node", restore
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
            return f"numa: pinned buffers allocated from node {node} ({len(allowed)} cpus), the node of GPU {local}", restore
        return f"numa: node {node} has no allowed cpu", restore
    except Exception as e:  # noqa: BLE001
        return f"numa: not bound ({type(e).__name__})", restore


def measure_h2d_gbs(src_ptr, nbytes):
    """The PCIe yardstick of the e2e leg: plain cudaMemcpyAsync calls from the SAME pinned buffer the e2e leg
    feeds from, in this process — one copy of the whole buffer, and the buffer in 8 back-to-back slices (what the
    library's host path does); best of 6 each, the better of the two."""
    import ctypes

    import torch

    rt = None
    for name in ("libcudart.so.12", "libcudart.so"):
        try:
            rt = ctypes.CDLL(name)
            break
        except OSError:
            continue
    if rt is None:
        return None
    rt.cudaMemcpyAsync.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p]
    dst = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    best = 0.0
    for slices in (1, 8):
        per = (nbytes + slices - 1) // slices
        for _ in range(6):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for k in range(slices):
                n = min(per, nbytes - k * per)
                if n > 0 and rt.cudaMemcpyAsync(dst.data_ptr() + k * per, src_ptr + k * per, n, 1, stream) != 0:
                    return None
            e1.record()
            torch.cuda.synchronize()
            best = max(best, nbytes / (e0.elapsed_time(e1) * 1e-3) / 1e9)
    del dst
    return best


class Scenario:
    """One workload on one picker: index build, device-resident timing, per-kernel split, sampled parity."""

    def __init__(self, args, cfg_id, mode, rank, world, local, order="chain", R_override=None, batches=None):
        from fusioninfer_b200 import synth

        self.args, self.cfg_id, self.mode, self.rank, self.world, self.local, self.order = args, cfg_id, mode, rank, world, local, order
        self.wl = synth.baseline_workload(cfg_id)
        if R_override:
            self.wl.R = R_override
        self.nb = batches or max(1, args.batches)
        self.split_hash = False  # sharded pools: every rank hashes every prompt (the library default); True = split + all-gather

    # -- sampled requests whose picks the oracle re-derives (known BEFORE the index is built, so that every rank
    # can keep just the index entries those requests can touch: for them that is equivalent to the full index)
    def _plan_sample(self, tok0, S):
        from oracle import epp_oracle as eo

        wl = self.wl
        self.sample_idx = np.linspace(0, wl.R - 1, S).astype(np.int64)
        o = eo.Oracle(build_config(wl, self.cfg_id, 0, wl.E, 0, S, "replicas", base=eo.default_config()))
        sub_offs = np.arange(S + 1, dtype=np.uint64) * np.uint64(wl.T * 4)
        self.sample_tok = np.ascontiguousarray(tok0[self.sample_idx])
        self.sample_offs = sub_offs
        ch, _ = o.hash_batch(self.sample_tok, sub_offs, wl.h0)
        self.needed = np.unique(ch)
        self.kept_ops = []

    def build(self, sample=0):
        import torch

        from fusioninfer_b200 import EndpointPicker
        from fusioninfer_b200 import dist as fdist

        wl, rank, world, local, mode = self.wl, self.rank, self.world, self.local, self.mode
        t0 = time.time()
        self.begin, self.count = fdist.shard_range(wl.E, rank, world) if mode == "sharded" else (0, wl.E)
        churn = self.order == "churned"
        cfg = build_config(wl, self.cfg_id, self.begin, self.count, local, wl.R, mode, lru_capacity=wl.lru_capacity if churn else 0)
        self.picker = EndpointPicker(cfg)
        if mode == "sharded" and world > 1:
            uid = EndpointPicker.comm_unique_id() if rank == 0 else None
            with stdout_to_stderr():  # the library's own communicator
                self.picker.comm_init(fdist.broadcast_bytes(uid, 128), rank, world)
        self.exchange = self.picker.comm_exchange()
        self.picker.update_endpoints(wl.endpoint_states())
        # request batches: replicas serve different batches per rank, shards all see the same requests
        self.d_tok, self.d_off, self.host0 = [], [], None
        for b in range(self.nb):
            bid = b if mode == "sharded" else rank * self.nb + b
            tok, offs = wl.prompts(batch=bid)
            self.d_tok.append(torch.from_numpy(tok.view(np.int32)).cuda())
            self.d_off.append(torch.from_numpy(offs.view(np.int64)).cuda())
            if b == 0:
                self.host0 = (tok, offs)
        if sample:
            self._plan_sample(self.host0[0], min(sample, wl.R))
        n_ops = 0
        rng = np.random.default_rng(0xF051 + self.cfg_id)
        if churn:
            n_ops = self._build_through_lru()
        else:
            for ops in wl.index_ops(ep_lo=self.begin, ep_hi=self.begin + self.count, chunk_endpoints=128):
                if sample:
                    self.kept_ops.append(ops[np.isin(ops["hash"], self.needed)])
                if self.order == "shuffled":
                    ops = ops[rng.permutation(len(ops))]
                self.picker.index_apply(ops)
                n_ops += len(ops)
        self.picker.index_sync()
        ist = self.picker.index_stats()
        self.index_stats = {"entries": int(n_ops), "keys": int(ist.used - ist.tombstones), "slots": int(ist.slots),
                            "tombstones": int(ist.tombstones), "rebuilds": int(ist.rebuilds)}
        R, P = wl.R, self.picker.n_profiles
        self.P = P
        self.d_h0 = torch.full((R,), int(np.uint64(wl.h0).astype(np.int64)), dtype=torch.int64, device="cuda")
        self.d_out = torch.zeros(R * P * 16, dtype=torch.uint8, device="cuda")
        self.d_outs = [torch.zeros(R * P * 16, dtype=torch.uint8, device="cuda") for _ in range(2)]
        self.stream = torch.cuda.current_stream().cuda_stream
        log(f"rank {rank}: cfg{self.cfg_id}/{mode}/{self.order}: {n_ops} index entries -> {ist.used} keys in {ist.slots} slots, "
            f"{self.nb} batch(es) of {R} requests resident ({time.time() - t0:.1f}s)")
        return self

    def _build_through_lru(self):
        """An AGED index: the initial state enters through the host LRU (filler first, then the shared group
        chains), then K pick + indexer.Add(chain, picked endpoint) rounds evict filler and scatter new chains over
        retired nodes' successors — what a live picker's index looks like (tombstones, maybe a rebuild)."""
        wl, pk = self.wl, self.picker
        nb = wl.n_blocks
        n = 0
        for ops in wl.index_ops(ep_lo=self.begin, ep_hi=self.begin + self.count, chunk_endpoints=64):
            # one pseudo-request per run of <= n_blocks ops of one endpoint, filler before the group chains
            e = ops["endpoint"]
            h = ops["hash"]
            out_e, rows = [], []
            for ep in np.unique(e):
                he = h[e == ep]
                grp, fil = he[: wl.groups_per_endpoint * nb], he[wl.groups_per_endpoint * nb:]
                seq = np.concatenate([fil, grp])
                pad = (-len(seq)) % nb
                seq = np.concatenate([seq, np.zeros(pad, dtype=np.uint64)])
                rows.append(seq.reshape(-1, nb))
                out_e.append(np.full(rows[-1].shape[0], ep, dtype=np.uint32))
            ch = np.concatenate(rows)
            ee = np.concatenate(out_e)
            valid = (ch != 0).sum(axis=1).astype(np.uint32)  # the padded tail row of an endpoint carries fewer hashes
            pk.index_add_chains(ee, ch, valid)
            n += int(valid.sum())
        for k in range(self.args.churn_rounds):
            tok, offs = wl.prompts(batch=1000 + k)
            picks, chains = pk.pick_batch(tok, offs, wl.h0, want_chains=True)
            pk.index_add_chains(picks[:, 0]["endpoint"], chains, picks[:, 0]["n_blocks"])
        return n

    # -- timing -------------------------------------------------------------------------------------
    def step(self, i):
        b = i % self.nb
        wl = self.wl
        self.picker.pick_batch_device(self.d_tok[b].data_ptr(), self.d_off[b].data_ptr(), self.d_h0.data_ptr(), wl.R,
                                      wl.R * wl.T * 4, self.d_out.data_ptr(), 0, self.stream)

    def submit(self, i):
        b = i % self.nb
        wl = self.wl
        self.picker.pick_submit(self.d_tok[b].data_ptr(), self.d_off[b].data_ptr(), self.d_h0.data_ptr(), wl.R,
                                wl.R * wl.T * 4, self.d_outs[i & 1].data_ptr(), self.stream)

    def run_steps(self, k, pipelined=False):
        if pipelined:
            t0 = time.perf_counter()
            for i in range(k):
                self.submit(i)
            self.submit_us = (time.perf_counter() - t0) * 1e6 / max(k, 1)  # host time per submit (launch-bound if ~ the step)
            self.picker.pick_wait(self.stream)
        else:
            for i in range(k):
                self.step(i)

    def time_steps(self, steps, warmup, pipelined=False, clocks=None):
        """-> (ms per step: CUDA events on the launching stream, max over ranks; launches of this library)"""
        import torch

        from fusioninfer_b200 import dist as fdist

        self.run_steps(max(warmup, 3), pipelined)
        torch.cuda.synchronize()
        fdist.barrier()
        torch.cuda.synchronize()
        self.picker.reset_stats()
        if clocks is not None:
            clocks.start()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        self.run_steps(steps, pipelined)
        ev1.record()
        torch.cuda.synchronize()
        fdist.barrier()
        ms = fdist.max_over_ranks(ev0.elapsed_time(ev1)) / steps
        return ms, int(self.picker.stats().kernel_launches)

    def kernel_split(self, steps):
        """per-kernel CUDA-event durations + N_probe from a profiled pass (not part of any reported step time)"""
        import torch

        pk = self.picker
        pk.reset_stats()
        pk.set_profiling(True)
        n = min(steps, 8)
        for i in range(n):
            self.step(i)
        torch.cuda.synchronize()
        st = pk.stats()
        pk.set_profiling(False)
        kern = {"hash_blocks": (st.ms_hash_blocks, st.n_hash_blocks), "chain_finalize": (st.ms_chain_probe, st.n_chain_probe),
                "match_pick": (st.ms_match_pick, st.n_match_pick), "other": (st.ms_other, st.n_other)}
        # "other" counts the sharded step's two chain all-gathers as launches without time: per-launch average
        # only over launches that were timed
        avg = {k: (v[0] / v[1] if v[1] else 0.0) for k, v in kern.items()}
        return avg, st.probed_blocks / max(n, 1)

    def last_picks(self, steps, pipelined):
        """the picks [R, P] the last of `steps` timed steps wrote (run_steps: step i of the pipelined path writes
        d_outs[i & 1], every stream-ordered step writes d_out)"""
        import torch

        from fusioninfer_b200 import PICK_DTYPE

        buf = self.d_outs[(steps - 1) & 1] if pipelined else self.d_out
        torch.cuda.synchronize()
        return buf.cpu().numpy().view(PICK_DTYPE).reshape(self.wl.R, self.P)

    def picks_of_batch0(self):
        """the device path's picks of batch 0, as records [R, P] (+ the chains)"""
        import torch

        wl = self.wl
        d_chain = torch.zeros(wl.R * wl.max_blocks, dtype=torch.int64, device="cuda")
        self.picker.pick_batch_device(self.d_tok[0].data_ptr(), self.d_off[0].data_ptr(), self.d_h0.data_ptr(), wl.R,
                                      wl.R * wl.T * 4, self.d_out.data_ptr(), d_chain.data_ptr(), self.stream)
        torch.cuda.synchronize()
        picks = self.d_out.cpu().numpy().view(np.dtype(
            [("endpoint", "<u4"), ("match_blocks", "<u2"), ("n_blocks", "<u2"), ("score", "<f8")])).reshape(wl.R, self.P)
        return picks, d_chain.cpu().numpy().view(np.uint64).reshape(wl.R, wl.max_blocks)

    def sampled_parity(self):
        """bit-exact check of the sampled requests' picks against the oracle (whole pool, unsharded).  Sharded:
        the ranks' kept index entries are gathered on rank 0."""
        from fusioninfer_b200 import dist as fdist

        picks, _ = self.picks_of_batch0()
        kept = np.concatenate(self.kept_ops) if self.kept_ops else np.zeros(0, dtype=self.kept_ops_dtype())
        if self.mode == "sharded" and self.world > 1:
            import torch.distributed as dist

            parts = [None] * self.world
            dist.all_gather_object(parts, kept)
            kept = np.concatenate(parts)
        if self.rank != 0:
            return None
        o = build_oracle(self.wl, self.cfg_id, [kept], f"cfg{self.cfg_id} sample oracle")
        want = o.pick_batch(self.sample_tok, self.sample_offs, self.wl.h0, nthreads=host_cores()["usable"])
        same = picks[self.sample_idx].tobytes() == want.tobytes()
        if not same:
            log(f"PARITY FAILURE cfg{self.cfg_id} {self.mode}")
        return {"checked_requests": int(len(self.sample_idx)), "bit_exact": bool(same)}

    @staticmethod
    def kept_ops_dtype():
        from fusioninfer_b200 import _abi as abi

        return abi.np_dtypes()[1]

    def close(self):
        import torch

        self.picker.close()
        self.d_tok = self.d_off = None
        self.d_out = self.d_outs = self.d_h0 = None
        torch.cuda.empty_cache()


def sub_record(sc, steps, warmup, peak, with_parity=True):
    """A compact result of one extra configuration (BASELINE.json configs 2, 4, 5) for the line's roofline dict."""
    wl = sc.wl
    ms, _ = sc.time_steps(steps, warmup)
    avg, nprobe = sc.kernel_split(steps)
    hashed = None
    if sc.mode == "sharded" and sc.world > 1 and sc.split_hash:
        hashed = wl.R / sc.world
    alg = algorithmic_bytes(wl, nprobe, wl.R, sc.count, hashed)
    step_alg = alg["hash_blocks"] + alg["match_pick"]
    units = wl.R * (sc.world if sc.mode == "replicas" else 1)
    rec = {
        "workload": workload_config(wl, sc.cfg_id, f"{sc.mode}{sc.world}")["workload"],
        "decisions_per_s": units / (ms * 1e-3), "ms_per_step": ms, "kernel_ms": avg,
        "n_probe_per_decision": nprobe / wl.R,
        "algorithmic_bytes_per_step_per_gpu": step_alg,
        "step_algorithmic_gbs_per_gpu": step_alg / (ms * 1e-3) / 1e9,
        "frac": step_alg / (ms * 1e-3) / 1e9 / peak,
        "index": sc.index_stats, "exchange": sc.exchange,
    }
    if with_parity:
        rec["parity"] = sc.sampled_parity()
    return rec


DUMP_BYTES = 60_000_000  # array data of --dump-outputs; with the .npy headers under 64 MB in all


def dump_outputs(out_dir, picks):
    """Write the picks [R, P] as DIR/<field>.npy (float64, exact for every field of fi_pick) plus DIR/request.npy,
    the request index of each row.  Above DUMP_BYTES in all, the rows are a fixed seeded sample of the requests."""
    R = picks.shape[0]
    per_request = 8 * (1 + len(picks.dtype.names) * picks.shape[1])
    rows = np.arange(R)
    if R * per_request > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(R, DUMP_BYTES // per_request, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "request.npy"), rows.astype(np.float64))
    for name in picks.dtype.names:
        np.save(os.path.join(out_dir, f"{name}.npy"), picks[rows][name].astype(np.float64))
    log(f"picks of the last timed step ({len(rows)} of {R} requests) written to {out_dir}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cfg", type=int, default=3, choices=[2, 3, 4, 5])
    ap.add_argument("--mode", default=None, choices=["replicas", "sharded"])
    ap.add_argument("--pipeline", dest="pipeline", action="store_true", default=True,
                    help="(default) time the pipelined device API: fi_epp_pick_submit per batch, one fi_epp_pick_wait at the end "
                         "of the K steps — two batches in flight, batch k+1 is hashed while batch k is matched")
    ap.add_argument("--no-pipeline", dest="pipeline", action="store_false",
                    help="time stream-ordered fi_epp_pick_batch_device calls instead (reported as roofline.stream_ordered anyway)")
    ap.add_argument("--scale", type=float, default=1.0, help="shrink R (debug only; the JSON line says so)")
    ap.add_argument("--batches", type=int, default=2, help="distinct request batches rotated through")
    ap.add_argument("--cpu-sample", type=int, default=4096)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--e2e-steps", type=int, default=0, help="0 = same as --steps (capped at 10)")
    ap.add_argument("--no-e2e", action="store_true", help="skip the e2e leg (tuning runs only)")
    ap.add_argument("--extras", default="auto", choices=["auto", "none"],
                    help="auto: the default cfg-3 run also measures BASELINE.json's other configs into the roofline dict — "
                         "N = 1: cfg 2, cfg 5 on one GPU, and cfg 3 on a shuffled and on an LRU-aged index; N > 1: cfg 4 and "
                         "cfg 5 with the index sharded by endpoint range (peer-memory and NCCL pick exchange, split and "
                         "replicated hashing)")
    ap.add_argument("--index-order", default="chain", choices=["chain", "shuffled", "churned"],
                    help="how the main run's index was built (the default run reports all three in roofline.index_order)")
    ap.add_argument("--churn-rounds", type=int, default=6, help="pick + indexer.Add rounds that age the 'churned' index")
    ap.add_argument("--extra-steps", type=int, default=30)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the picks of the last one as DIR/<field>.npy (float64; rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the picks of the GPU path (--impl ours)")

    from fusioninfer_b200 import synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        log(f"note: WORLD_SIZE={world} but --gpus {args.gpus}; using the launched world size")
        args.gpus = world
    cfg_id = args.cfg
    mode = args.mode or ("sharded" if cfg_id in (4, 5) and world > 1 else "replicas")
    wl = synth.baseline_workload(cfg_id)
    if args.scale != 1.0:
        wl.R = max(64, int(wl.R * args.scale))

    if args.impl == "reference":
        run_reference(args, wl, cfg_id)
        return

    import torch

    from fusioninfer_b200 import PinnedBuffer
    from fusioninfer_b200 import dist as fdist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the pick path has no CPU fallback (use --impl reference "
                         "for the CPU arm)")
    if world > 1:
        # stdout carries exactly one JSON line: keep NCCL's version banner off it
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        # NCCL prints its banner when the first communicator is created (lazily, at the first collective):
        # do that now with fd 1 pointing at stderr, whatever the debug settings of the box are
        with stdout_to_stderr():
            fdist.init_process_group("nccl")
            torch.cuda.set_device(local)
            fdist.barrier()
            torch.cuda.synchronize()
    torch.cuda.set_device(local)
    numa_note, numa_restore = bind_to_gpu_numa(local)
    peak, peak_src = measured_peak_gbs()

    # ---- main scenario (untimed set-up) ------------------------------------------------------------
    sc = Scenario(args, cfg_id, mode, rank, world, local, order=args.index_order, R_override=wl.R if args.scale != 1.0 else None)
    sc.split_hash = os.environ.get("FI_EPP_SHARD_HASH", "replicated") == "split"
    sc.build()
    picker, R, P = sc.picker, sc.wl.R, sc.P
    wl = sc.wl
    pipelined = args.pipeline and not (mode == "sharded" and world > 1)

    # ---- timed region: exactly K steps, device events on the launching stream -----------------
    clocks = ClockSampler(local)
    ms_step, launches = sc.time_steps(args.steps, args.warmup, pipelined,
                                      clocks if (rank == 0 and os.environ.get("FI_BENCH_NO_CLOCKS") != "1") else None)
    clk = clocks.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, sc.last_picks(args.steps, pipelined))
    units = R * (world if mode == "replicas" else 1)
    value = units / (ms_step * 1e-3)
    stream_ordered = None
    pinfo = picker.pipeline_info() if pipelined else None
    if pinfo is not None:
        pinfo["host_us_per_submit"] = round(getattr(sc, "submit_us", 0.0), 1)
    if pipelined:  # the same K steps through the stream-ordered call, for reference
        ms_so, _ = sc.time_steps(min(args.steps, 50), 3, False)
        stream_ordered = {"decisions_per_s": units / (ms_so * 1e-3), "ms_per_step": ms_so,
                          "how": "fi_epp_pick_batch_device, one call per step (each call orders the caller's stream behind its result)"}

    # ---- per-kernel durations + N_probe (profiled pass, not part of the number above) -----------
    avg_ms, nprobe_per_step = sc.kernel_split(args.steps)
    hashed = R / world if (mode == "sharded" and world > 1 and sc.split_hash) else None
    alg = algorithmic_bytes(wl, nprobe_per_step, R, sc.count, hashed)
    dom = max(("hash_blocks", "match_pick"), key=lambda k: avg_ms[k])
    achieved = alg[dom] / (avg_ms[dom] * 1e-3) / 1e9 if avg_ms[dom] else 0.0
    traffic = load_traffic() if (cfg_id == 3 and mode == "replicas" and args.scale == 1.0) else {}  # captured for cfg 3 only
    step_alg = alg["hash_blocks"] + alg["match_pick"]
    roofline = {
        "bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
        "frac": achieved / peak if peak else None, "traffic": traffic.get(dom),
        "peak_source": peak_src + " (burst figure: kernel timed alone with CUDA events)",
        "algorithmic_bytes_per_launch": alg[dom],
        "kernel_ms": avg_ms, "n_probe_per_decision": nprobe_per_step / R,
        "step_algorithmic_gbs": step_alg / (ms_step * 1e-3) / 1e9,
        "step_frac": step_alg / (ms_step * 1e-3) / 1e9 / peak,
        "other_kernels": {k: {"achieved": (alg[k] / (avg_ms[k] * 1e-3) / 1e9 if avg_ms[k] else 0.0),
                              "traffic": traffic.get(k)} for k in ("hash_blocks", "match_pick") if k != dom},
        "index": sc.index_stats, "index_order_of_value": args.index_order, "stream_ordered": stream_ordered,
    }

    # ---- e2e: public C-ABI call with host (pinned) buffers, H2D + D2H inside ---------------------
    tok0, offs0 = sc.host0
    pin_tok = PinnedBuffer(tok0.nbytes)
    pin_off = PinnedBuffer(offs0.nbytes)
    pin_h0 = PinnedBuffer(8 * R)
    pin_out = PinnedBuffer(16 * R * P)
    pin_tok.array(np.uint32)[:] = tok0.reshape(-1)
    pin_off.array(np.uint64)[:] = offs0
    pin_h0.array(np.uint64)[:] = np.uint64(wl.h0)
    e2e_steps = args.e2e_steps or min(args.steps, 10)
    if args.no_e2e:
        e2e_steps = 1
    for _ in range(2):
        picker.pick_batch_raw(pin_tok.ptr, pin_off.ptr, pin_h0.ptr, R, pin_out.ptr)
    fdist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        picker.pick_batch_raw(pin_tok.ptr, pin_off.ptr, pin_h0.ptr, R, pin_out.ptr)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    dt = fdist.max_over_ranks(dt)
    h2d_bytes = int(tok0.nbytes + offs0.nbytes + 8 * R)
    h2d_gbs = measure_h2d_gbs(pin_tok.ptr, int(tok0.nbytes)) if not args.no_e2e else None
    h2d_gbs_min = -fdist.max_over_ranks(-h2d_gbs) if h2d_gbs else None
    e2e = {"value": units * e2e_steps / dt, "unit": "decisions/s",
           "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": int(16 * R * P),
           "ms_per_step": 1e3 * dt / e2e_steps, "steps": e2e_steps,
           "how": "fi_epp_pick_batch on pinned host buffers: H2D prompts+offsets+seeds, kernels, D2H picks, per step",
           "roofline": {"bound": "pcie", "h2d_gbs_measured": h2d_gbs_min, "unit": "GB/s",
                        "achieved": h2d_bytes / (dt / e2e_steps) / 1e9,
                        "frac": (h2d_bytes / (dt / e2e_steps) / 1e9 / h2d_gbs_min) if h2d_gbs_min else None,
                        "how": "achieved = H2D bytes of a step / its wall time (host clock, D2H of the picks and the last slice's "
                               "kernels included); yardstick = bare cudaMemcpyAsync of the same pinned prompt buffer in this "
                               "process (CUDA events; whole and in 8 slices, best of 6, slowest rank)"},
           "numa": numa_note}
    e2e_picks = pin_out.array(np.uint8).copy().view(np.dtype(
        [("endpoint", "<u4"), ("match_blocks", "<u2"), ("n_blocks", "<u2"), ("score", "<f8")])).reshape(R, P)
    numa_restore()  # the CPU leg below may use every core again

    # ---- cpu_baseline (rank 0, bounded sample) + parity of the e2e picks on that sample ---------------
    cpu = None
    parity = None
    if rank == 0 and not args.no_cpu and args.index_order == "chain":
        cores = host_cores()
        ncores = cores["usable"]
        o = build_oracle(wl, cfg_id, [], "oracle (empty)")
        S = min(args.cpu_sample, R)
        # the FULL index, not just the sampled requests' hashes: a tiny index would make the CPU
        # lookups unrealistically cache-friendly
        o.index_reserve(wl.E * wl.lru_capacity)
        t0 = time.time()
        for ops in wl.index_ops(chunk_endpoints=128):
            o.index_apply(ops)
        log(f"oracle index built in {time.time() - t0:.1f}s")
        want = o.pick_batch(tok0[:S], offs0[: S + 1], wl.h0, nthreads=ncores)
        # timing: every worker walks its shard `rep` times (persistent pool); ~10-20 s of CPU work in total
        t1 = time.perf_counter()
        o.pick_batch_repeat(tok0[:S], offs0[: S + 1], wl.h0, nthreads=ncores, repeat=2)
        per_pass = (time.perf_counter() - t1) / 2
        rep = int(max(1, min(64, 0.15 / max(per_pass, 1e-6))))
        t1 = time.perf_counter()
        o.pick_batch_repeat(tok0[:S], offs0[: S + 1], wl.h0, nthreads=ncores, repeat=rep)
        tn = (time.perf_counter() - t1) / rep
        same = e2e_picks[:S].tobytes() == want.tobytes()
        parity = {"checked_requests": S, "bit_exact": bool(same)}
        if not same:
            log("PARITY FAILURE on the cpu_baseline sample")
        # single-thread figure on a smaller slice
        S1 = min(S, 512)
        t0 = time.perf_counter()
        o.pick_batch(tok0[:S1], offs0[: S1 + 1], wl.h0, nthreads=1)
        t1s = time.perf_counter() - t0
        cpu = {"value": S / tn, "unit": "decisions/s", "cores": ncores, "cores_detail": cores, "kind": "port",
               "single_thread_value": S1 / t1s,
               "sample": f"first {S} requests of batch 0 x {rep} passes (full {wl.E * wl.lru_capacity}-entry index), "
                         f"{ncores} persistent worker threads sharded by request; single-thread figure on the first {S1}; {ORACLE_LABEL}"}
        del o
    sc.close()

    # ---- BASELINE.json's other configurations, into the roofline dict ---------------------------------
    extras = args.extras == "auto" and cfg_id == 3 and mode == "replicas" and args.scale == 1.0 and args.index_order == "chain"
    if extras and world == 1:
        others = {}
        for cid in (2, 5):
            x = Scenario(args, cid, "replicas", rank, world, local, batches=2 if cid == 2 else 1).build(sample=512)
            others[f"cfg{cid}"] = sub_record(x, args.extra_steps, 3, peak)
            x.close()
        roofline["configs"] = others
        order = {"chain": {"decisions_per_s": value, "ms_per_step": ms_step, "match_pick_ms": avg_ms["match_pick"]}}
        for od in ("shuffled", "churned"):
            x = Scenario(args, 3, "replicas", rank, world, local, order=od, batches=1).build()
            ms, _ = x.time_steps(args.extra_steps, 3, pipelined)  # the same API as the headline
            av, _ = x.kernel_split(8)
            order[od] = {"decisions_per_s": R / (ms * 1e-3), "ms_per_step": ms, "match_pick_ms": av["match_pick"], "index": x.index_stats}
            x.close()
        order["how"] = ("chain: every endpoint's chains bulk-loaded back to back (the headline); shuffled: the same entries in a "
                        f"random order; churned: the state entered through the host LRU, then {args.churn_rounds} rounds of pick + "
                        "indexer.Add(chain, picked endpoint) with evictions before timing")
        roofline["index_order"] = order
    if extras and world > 1:
        sharded = {}
        for cid in (4, 5):
            x = Scenario(args, cid, "sharded", rank, world, local, batches=1)
            x.build(sample=512)
            rec = sub_record(x, args.extra_steps, 3, peak)
            variants = {}
            # variants: the NCCL all-gather of the picks instead of the peer-memory exchange; split hashing (every rank
            # hashes R/world prompts and the chains are all-gathered) instead of every rank hashing every prompt
            for name, opts in (("nccl_exchange", {"exchange": 2}), ("split_hash", {"shard_hash": 1})):
                try:
                    for k, v in opts.items():
                        x.picker.set_option(k, v)
                    x.split_hash = "shard_hash" in opts
                    ms, _ = x.time_steps(args.extra_steps, 3)
                    av, _ = x.kernel_split(8)
                    variants[name] = {"decisions_per_s": x.wl.R / (ms * 1e-3), "ms_per_step": ms, "kernel_ms": av}
                except Exception as e:  # noqa: BLE001
                    variants[name] = {"error": str(e)[:200]}
                finally:
                    try:
                        x.picker.set_option("exchange", 1 if x.exchange == "peer" else 2)
                        x.picker.set_option("shard_hash", 0)
                        x.split_hash = False
                    except Exception:  # noqa: BLE001
                        pass
            rec["variants"] = variants
            rec["bound_decisions_per_s"] = {"how": "SURVEY.md §8d worst case per GPU (every GPU hashes every prompt, all blocks hit) at "
                                                   "the measured HBM peak, lock-step over the ranks",
                                            "value": peak * 1e9 / (4 * x.wl.T + x.wl.n_blocks * (8 + x.count / 8.0) + 16)}
            sharded[f"cfg{cid}"] = rec
            x.close()
        roofline["sharded"] = sharded

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "decisions/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": dict(workload_config(wl, cfg_id, f"{mode}{world}"), exchange=sc.exchange,
                           pipeline=((f"fi_epp_pick_submit/pick_wait on a partitioned GPU (green contexts): batch k matched and "
                                      f"batch k+2 hashed on {pinfo['main_sms']} SMs while batch k+1's chains are walked on "
                                      f"{pinfo['walk_sms']} SMs, 3 batches in flight; all K batches complete inside the timed region; "
                                      f"host time per submit {pinfo['host_us_per_submit']} us on this rank")
                                     if pinfo and pinfo["partitioned"] else
                                     ("fi_epp_pick_submit/pick_wait: 2 batches in flight, batch k+1 hashed while batch k "
                                      "is matched; all K batches complete inside the timed region")) if pipelined
                           else "stream-ordered fi_epp_pick_batch_device calls"),
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "clocks": clk, "gpu_launches": int(launches),
            "parity": parity,
        }
        if args.scale != 1.0:
            line["config"]["workload"] += f" [DEBUG scale={args.scale}: NOT the headline config]"
        print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist

        dist.destroy_process_group()


if __name__ == "__main__":
    main()
