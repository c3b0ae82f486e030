#!/usr/bin/env python
"""bench.py — mel-frames/sec through the CFM DiT estimator (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config cfg1|cfg2|cfg3|cfg4] [--impl reference] [--dump-outputs DIR]

A "step" is one complete ``CFMDecoder.forward`` ODE solve over one batch of synthetic inputs
(SURVEY.md §8d): weights = reference-style init under manual_seed(0) with the adaLN gates re-drawn
N(0, 0.3²); inputs under manual_seed(1); z unmasked; CFG strength 3.
  value  : frames/s with every rank's batch slice already resident in its HBM (device timed, max over ranks)
  e2e    : the same metric through ``CFMDecoder.solve_host`` = ``st_solve_host`` of the C ABI with PINNED HOST
           buffers — the H2D copies of (mu, mask, c, z), the solve, the D2H read of the mel and the stream
           synchronisation are inside the call and inside the timed region, per rank
  roofline: the tcgen05 conv-GEMM class (dominant kernel): algorithmic FLOPs / CUDA-event time of
           every launch in one instrumented solve, against MEASURED_PEAKS.json's sustained bf16 peak
  cpu_baseline / --impl reference: the reference's own CPU path — the genuine modules staged under
           baseline/_ref (kind "reference"; oracle port if nothing is staged) — on host cores, bounded sample
  parity : utterances {first, second, middle, last} of the measured batch re-solved on the CPU (checker only)
  --dump-outputs DIR: the mel the timed solve returned in its last step, as DIR/mel.npy (see dump_outputs)
Multi-GPU (torchrun, one rank per GPU): weak scaling, the per-GPU batch is fixed, every rank owns its slice
(value / e2e); the rank-0-owns-everything NCCL scatter/gather variant is timed beside it (root_scatter_gather,
with the scatter+gather alone reported separately); at N = 8 BASELINE cfg4 as written (1024 = 128 per GPU)
rides along under the key "cfg4".
"""
from __future__ import annotations

import argparse
import atexit
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    "cfg0": dict(B=1, T=300, n_steps=10, method="euler", cfg=3.0, lengths=None,
                 desc="batch=1, ~300-frame mel (64 phonemes), 10-step Euler + CFG — the reference's CPU-runnable plumbing case"),
    # name: per-GPU batch, T, steps, method, cfg, description (BASELINE.json configs[1..4])
    "cfg1": dict(B=32, T=1000, n_steps=10, method="euler", cfg=3.0, lengths=None,
                 desc="batch=32/GPU, n_mel=80, T=1000, 10-step Euler + CFG"),
    "cfg2": dict(B=256, T=500, n_steps=25, method="dopri5_fixed", cfg=None, lengths=None,
                 desc="batch=256, n_mel=80, T=500, 25 fixed Dormand-Prince steps (6 evals/step, NFE=150), no CFG"),
    "cfg3": dict(B=128, T=None, n_steps=10, method="euler", cfg=None, lengths="uniform200-2000",
                 desc="bucketed variable-length batch=128 (T in [200,2000]), 10-step Euler, masked attention"),
    "cfg4": dict(B=128, T=1000, n_steps=10, method="euler", cfg=3.0, lengths=None,
                 desc="batch=128/GPU (1024 over 8 GPUs), n_mel=80, T=1000, 10-step Euler + CFG"),
}
N_MEL = 80
NFE_PER_STEP = {"euler": 1, "midpoint": 2, "rk4": 4, "dopri5_fixed": 6}


def flops_per_frame_call(T: int, n_mel: int = N_MEL) -> float:
    """BASELINE.md §3: F_call(T) = 32.948e6 + 6144·T for M=80 (2·MAC)."""
    H, F, L = 256, 1024, 6
    return 2.0 * ((3 * n_mel * F + 3 * F * F + 3 * F * H) + (n_mel + H) * H + L * (4 * H * H + 2 * T * H + 6 * H * F)
                  + 3 * (6 * H * H) + H * n_mel)


COND_FLOPS = 2.0 * (3 * N_MEL * 1024 + 3 * 1024 * 1024 + 3 * 1024 * 256)    # 8.356 MFLOP/frame, hoistable


def make_model(device):
    from stabletts_b200 import CFMDecoder
    torch.manual_seed(0)
    m = CFMDecoder(N_MEL, N_MEL, 256, N_MEL, 1024, 4, 6, 3, 0.1, 256).eval()
    with torch.no_grad():
        for i in range(6):
            node = m.estimator._modules["blocks"]._modules[str(i)]._modules["block"]._modules["adaLN_modulation"]._modules["2"]
            torch.nn.init.normal_(node.weight, std=0.3)
            torch.nn.init.normal_(node.bias, std=0.3)
    return m.to(device) if device is not None else m


def make_inputs(cfgd, B, seed=1):
    """CPU tensors (global generator, manual_seed(seed)) in the reference's boundary layout."""
    torch.manual_seed(seed)
    if cfgd["lengths"] is None:
        T = cfgd["T"]
        lens = torch.full((B,), T, dtype=torch.long)
    else:
        lens = torch.randint(200, 2001, (B,))
        lens, _ = torch.sort(lens)
        T = int(lens.max())
    mask = (torch.arange(T)[None, :] < lens[:, None]).float().unsqueeze(1)
    mu = torch.randn(B, N_MEL, T) * mask
    c = torch.randn(B, 256)
    z = torch.randn(B, N_MEL, T)
    fs, fc = torch.randn(1, 256), torch.randn(1, N_MEL, 1)
    return dict(mu=mu, mask=mask, c=c, z=z, fs=fs, fc=fc, lens=lens, T=T)


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.QUERY}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
            atexit.register(self.proc.kill)         # a run that dies before stop() must not leave the sampler behind
        except Exception:
            self.proc = None
            return
        # nvidia-smi takes seconds to initialise NVML on an 8-GPU host and its first query stalls the driver for
        # hundreds of ms: wait for the first sample so that this start-up never lands inside a timed region
        t0 = time.perf_counter()
        while time.perf_counter() - t0 < 20.0:
            try:
                if os.path.getsize(self.path) > 0:
                    break
            except OSError:
                pass
            time.sleep(0.1)

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        rows = []
        try:
            for line in open(self.path):
                p = [x.strip() for x in line.split(",")]
                if len(p) >= 9 and p[1].isdigit():
                    rows.append(p)
        finally:
            try:
                os.unlink(self.path)
            except OSError:
                pass
        if rows:
            clocks = [int(r[1]) for r in rows]
            busy = [c for c, r in zip(clocks, rows) if float(r[3]) > 250.0] or clocks
            out["sm_mhz"] = statistics.median(busy)
            out["sm_max_mhz"] = int(rows[0][2])
            out["power_w_max"] = max(float(r[3]) for r in rows)
            out["samples"] = len(rows)
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for j, n in enumerate(names):
                if any(r[5 + j].lower().startswith("active") for r in rows):
                    out["reasons"].append(n)
        return out


def cpu_threads() -> int:
    """Host threads actually usable: min(affinity mask, cgroup CPU quota) — see oracle.usable_cpus()."""
    from oracle import usable_cpus
    return usable_cpus()


class CpuArm:
    """The reference's CPU path for this workload (BASELINE.md §4): the GENUINE ``models.flow_matching.CFMDecoder`` /
    ``models.estimator.Decoder`` staged unmodified under baseline/_ref (oracle/stage_reference.py; ``kind`` =
    "reference") with the fixed-grid stepping of the absent torchdiffeq restated, or — when nothing is staged — the
    oracle port (``kind`` = "port").  One of the two places bench.py executes anything under oracle/ (the other is the
    parity check)."""

    def __init__(self, state):
        from oracle import stage_reference as SR
        self.state = state
        self.kind = "port"
        self.model = None
        if SR.available():
            try:
                _, RefCFM = SR.load_reference()
                m = RefCFM(N_MEL, N_MEL, 256, N_MEL, 1024, 4, 6, 3, 0.1, 256).eval()
                m.estimator.load_state_dict(state, strict=True)
                self.model, self.kind = m, "reference"
            except Exception as e:                     # noqa: BLE001 — fall back to the port, say why
                self.note = f"staged reference failed to import ({e}); oracle port used"

    def estimator_call(self, inp):
        from oracle import estimator_ref as R
        with torch.inference_mode():
            if self.model is not None:
                return self.model.estimator(torch.tensor(0.5), inp["z"], inp["mask"], inp["mu"], inp["c"])
            return R.estimator_forward(self.state, torch.tensor(0.5), inp["z"], inp["mask"], inp["mu"], inp["c"])

    def solve(self, inp, steps, method, kw):
        """CFMDecoder.forward semantics with the noise injected (the reference draws randn_like(mu) from the global RNG:
        the draw is replaced by the workload's z through a one-shot patch of torch.randn_like)."""
        from oracle import estimator_ref as R
        if self.model is None:
            return R.cfm_forward(self.state, inp["mu"], inp["mask"], steps, inp["z"], inp["c"], method, kw)
        orig = torch.randn_like
        torch.randn_like = lambda *_a, **_k: inp["z"].clone()
        try:
            with torch.inference_mode():
                return self.model(inp["mu"], inp["mask"], steps, 1.0, inp["c"], method, kw)
        finally:
            torch.randn_like = orig


def take_rows(inp, rows):
    idx = torch.as_tensor(rows)
    out = {k: inp[k][idx].contiguous() for k in ("mu", "mask", "c", "z")}
    out["lens"] = inp["lens"][idx]
    Tm = int(out["lens"].max())
    Tc = min(inp["T"], Tm + 4)                  # >= 4 pad frames: crop-invariant with and without CFG
    for k in ("mu", "mask", "z"):
        out[k] = out[k][:, :, :Tc].contiguous()
    out["T"] = Tc
    return out


def cpu_reference_solve(arm, inp, cfgd, rows, budget_s=25.0):
    """The CPU arm on a BOUNDED sample: the utterances ``rows`` of the workload; if a probe evaluation predicts that
    the full-NFE solve exceeds ``budget_s`` first the row set is halved (keeping first and last), then the number of ODE
    steps is cut and the throughput scaled to the full NFE.  Returns (rows used, output or None if truncated,
    seconds-equivalent for the FULL solve of those rows, note)."""
    kw = None if cfgd["cfg"] is None else dict(fake_speaker=inp["fs"], fake_content=inp["fc"], cfg_strength=cfgd["cfg"])
    per_step = NFE_PER_STEP[cfgd["method"]] * (2 if kw else 1)
    rows = list(rows)
    while True:
        sub = take_rows(inp, rows)
        t0 = time.perf_counter()
        arm.estimator_call(sub)
        probe = time.perf_counter() - t0
        if probe * per_step * cfgd["n_steps"] <= budget_s or len(rows) <= 2:
            break
        rows = [rows[0], rows[-1]]
    steps = cfgd["n_steps"]
    if probe * per_step * steps > budget_s:
        steps = max(1, int(budget_s / (probe * per_step)))
    t0 = time.perf_counter()
    out = arm.solve(sub, steps, cfgd["method"], kw)
    dt = time.perf_counter() - t0
    if steps == cfgd["n_steps"]:
        return rows, out, dt, f"full NFE={per_step * steps}"
    return rows, None, dt * cfgd["n_steps"] / steps, f"{steps} of {cfgd['n_steps']} ODE steps timed ({dt:.1f} s), scaled to the full NFE"


def sample_rows(B):
    """first, second, middle and last utterance of a batch (a batch-offset bug in the later rows must show)."""
    return sorted(set([0, min(1, B - 1), B // 2, B - 1]))


def run_reference(args, cfgd, rank):
    if rank != 0:
        return
    threads = cpu_threads()
    torch.set_num_threads(threads)
    model = make_model(None)
    state = {k: v.detach().clone() for k, v in model.estimator.state_dict().items()}
    arm = CpuArm(state)
    inp = make_inputs(cfgd, cfgd["B"])
    set_cfg_params(inp, cfgd)
    rows = sample_rows(cfgd["B"])
    budget = max(5.0, 150.0 / max(args.steps + max(args.warmup, 0) / 4 + 1, 1))          # whole run within a few minutes
    if args.warmup > 0:
        cpu_reference_solve(arm, inp, cfgd, rows, budget_s=budget / 4)
    t, note, used, frames = 0.0, "", rows, 0
    for _ in range(args.steps):
        used, _, dt, note = cpu_reference_solve(arm, inp, cfgd, rows, budget_s=budget)
        t += dt
        frames += int(inp["lens"][torch.as_tensor(used)].sum())
    val = frames / t
    sample = (f"utterances {used} of the workload (B={len(used)}, BASELINE.md §4) per step; {note}; {threads} torch threads; "
              f"{'genuine reference modules from baseline/_ref' if arm.kind == 'reference' else 'oracle port'}")
    line = {"impl": "reference", "metric": "mel-frames/sec through CFM DiT estimator (ODE solve, all evaluations)",
            "value": val, "unit": "frames/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.config}: {cfgd['desc']} (CPU sample: {sample})"},
            "cpu_baseline": {"value": val, "unit": "frames/s", "cores": threads, "kind": arm.kind, "sample": sample},
            "e2e": {"value": val, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def set_cfg_params(inp, cfgd):
    """fake_* are model parameters (models/model.py:43-44): replicated like the weights, same on every rank."""
    if cfgd["cfg"] is not None:
        g = torch.Generator().manual_seed(2)
        inp["fs"], inp["fc"] = torch.randn(1, 256, generator=g), torch.randn(1, N_MEL, 1, generator=g)


_CPU_REF_CACHE = {}      # (config name, rows) -> (rows, ref, seconds, note, kind): the CPU arm runs once per config, not once per precision


def run_config(args, name, model, dev, rank, world, steps, warmup, flush, *, full=True, precision="ffn_fp16x2"):
    """Measures one BASELINE config on this process group.  Every rank generates the same seeded GLOBAL batch on the
    host and keeps its own contiguous slice (pinned): a one-process-per-GPU server owns its requests' buffers.
      value  : every rank's slice resident in its HBM, no collective in the timed region ("per_rank_inputs")
      e2e    : every rank uploads its own pinned slice and downloads its own mel through CFMDecoder.solve_host
               (= st_solve_host of the C ABI: H2D + solve + D2H + stream sync inside the call)
      root_scatter_gather (N > 1): rank 0 owns the global batch in HBM, NCCL scatter -> solve -> gather inside the timed
               region; the scatter+gather alone is timed separately (SURVEY.md §8d cfg4)."""
    import torch.distributed as dist
    from stabletts_b200 import _lib, shard
    model.estimator.set_precision(precision)
    cfgd = CONFIGS[name]
    Bper = cfgd["B"]
    Bglob = Bper * world
    inp = make_inputs(cfgd, Bglob)
    set_cfg_params(inp, cfgd)
    T = inp["T"]
    sl = slice(rank * Bper, (rank + 1) * Bper)
    kw = kw_host = None
    if cfgd["cfg"] is not None:
        kw_host = dict(fake_speaker=inp["fs"], fake_content=inp["fc"], cfg_strength=cfgd["cfg"])
        kw = dict(fake_speaker=inp["fs"].to(dev), fake_content=inp["fc"].to(dev), cfg_strength=cfgd["cfg"])
    pinned = {k: inp[k][sl].contiguous().pin_memory() for k in ("mu", "mask", "c", "z")}
    local = {k: pinned[k].to(dev) for k in pinned}
    lens_local = [int(v) for v in inp["lens"][sl]]
    out_pinned = torch.empty(Bper, N_MEL, T, dtype=torch.float32).pin_memory()
    frames_global = int(inp["lens"].sum())
    bucketed = cfgd["lengths"] is not None

    def solve_one(mu, mask, c, z):
        return model(mu, mask, cfgd["n_steps"], 1.0, c, cfgd["method"], kw, z=z)

    def solve(mu, mask, c, z, lens=None):
        if not bucketed:
            return solve_one(mu, mask, c, z)
        lens = lens if lens is not None else mask.sum(dim=(1, 2)).long().tolist()    # host-visible lengths (bucketing is host logic)
        return shard.bucketed_solve(solve_one, mu, mask, c, z, lens, n_buckets=4)

    def step_device():
        return solve(local["mu"], local["mask"], local["c"], local["z"], lens_local)

    # bucketed workloads: requests are batched per length bucket on the host BEFORE they are submitted (that is what a
    # bucketing server does); each bucket owns pinned input / output buffers cropped to its own maximum + 4 pad frames
    e2e_buckets = []
    if bucketed:
        for idx in shard.length_buckets(lens_local, 4):
            Tb = min(T, max(lens_local[i] for i in idx) + 4)
            sel = torch.as_tensor(idx)
            e2e_buckets.append(dict(
                mu=pinned["mu"][sel][:, :, :Tb].contiguous().pin_memory(), mask=pinned["mask"][sel][:, :, :Tb].contiguous().pin_memory(),
                c=pinned["c"][sel].contiguous().pin_memory(), z=pinned["z"][sel][:, :, :Tb].contiguous().pin_memory(),
                out=torch.empty(len(idx), N_MEL, Tb, dtype=torch.float32).pin_memory()))

    def step_e2e():
        if not bucketed:
            return model.solve_host(pinned["mu"], pinned["mask"], cfgd["n_steps"], 1.0, pinned["c"], cfgd["method"], kw_host,
                                    z=pinned["z"], out=out_pinned)
        for bk in e2e_buckets:                                       # one H2D + solve + D2H per bucket, results stay per bucket
            model.solve_host(bk["mu"], bk["mask"], cfgd["n_steps"], 1.0, bk["c"], cfgd["method"], kw_host, z=bk["z"], out=bk["out"])
        return e2e_buckets[-1]["out"]

    glob = None
    if world > 1 and rank == 0:
        glob = {k: inp[k].to(dev) for k in ("mu", "mask", "c", "z")}

    def step_sg(fn=None):
        a = (glob["mu"], glob["mask"], glob["c"], glob["z"]) if rank == 0 else (None,) * 4
        return shard.sharded_solve(fn or solve, *a, device=dev, batch=Bglob, n_mel=N_MEL, T=T, gin=256)

    def timed(fn, n):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(n + 1)]
        ev[0].record()
        out = None
        for i in range(n):
            flush.zero_()
            out = fn()
            ev[i + 1].record()
        torch.cuda.synchronize()
        ms = torch.tensor([ev[0].elapsed_time(ev[n])], device=dev)
        per = [round(ev[i].elapsed_time(ev[i + 1]), 2) for i in range(n)]    # diagnostics (this rank)
        if world > 1:
            dist.barrier()
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), out, per

    remeasured = []

    def timed_checked(fn, n, tag):
        """K timed steps; if one step is an outlier (> 1.5x the median: a host stall or a driver hiccup starves the GPU
        for tens of ms about once in a dozen runs) the whole K-step region is measured ONCE more and the repeat is kept;
        the JSON line says so.  The decision is rank 0's, broadcast, so every rank repeats or none does."""
        ms, out, per = timed(fn, n)
        med = sorted(per)[len(per) // 2]
        again = torch.tensor([1 if (n >= 3 and max(per) > 1.5 * med) else 0], device=dev)
        if world > 1:
            dist.broadcast(again, 0)
        if int(again.item()) and not args.ncu_mode:
            remeasured.append({"region": tag, "first_attempt_step_ms": per[:32]})
            ms, out, per = timed(fn, n)
        return ms, out, per

    # warm-up: at least W untimed steps AND ~2 s of load (under the 1 kW cap the SM clock needs about a second to
    # settle); the extra count is decided on rank 0 and broadcast so every rank does the same.
    tw0 = time.perf_counter()
    for _ in range(warmup):
        flush.zero_()                   # same ops as a timed step: torch lazy-loads its fill kernel's module on first use
        step_device()
    torch.cuda.synchronize()
    el = time.perf_counter() - tw0
    extra = 0 if args.ncu_mode else int(max(0.0, 2.0 - el) / max(el / max(warmup, 1), 1e-4)) + 1
    if world > 1:
        ex_t = torch.tensor([extra], device=dev)
        dist.broadcast(ex_t, 0)
        extra = int(ex_t.item())
    for _ in range(extra):
        flush.zero_()
        step_device()
    timed(step_device, 1)               # one untimed pass through the timing harness itself (events, all_reduce)
    n_warm = warmup + extra + 1
    torch.cuda.synchronize()
    th0 = time.perf_counter()
    step_device()                       # host-side enqueue time of one step (no sync): launch-bound check
    host_ms = (time.perf_counter() - th0) * 1e3
    torch.cuda.synchronize()
    l0 = model.estimator.launch_count()
    ms_dev, out_dev, per_dev = timed_checked(step_device, steps, "value")
    launches = (model.estimator.launch_count() - l0) // (2 if any(r["region"] == "value" for r in remeasured) else 1)
    res = {"name": name, "cfgd": cfgd, "Bglob": Bglob, "T": T, "frames": frames_global, "ms_dev": ms_dev, "per_dev": per_dev,
           "out_dev": out_dev if (full and not bucketed) else None, "out_last": out_dev if args.dump_outputs else None,
           "launches": int(launches), "host_ms": host_ms, "n_warm": n_warm, "remeasured": remeasured, "inp": inp}
    if args.ncu_mode:
        return res
    step_e2e()
    ms_e2e, _, per_e2e = timed_checked(step_e2e, steps, "e2e")
    if bucketed:
        h2d_loc = sum(bk[k].numel() * 4 for bk in e2e_buckets for k in ("mu", "mask", "c", "z"))
        d2h_loc = sum(bk["out"].numel() * 4 for bk in e2e_buckets)
    else:
        h2d_loc, d2h_loc = sum(pinned[k].numel() * 4 for k in pinned), Bper * N_MEL * T * 4
    res.update(ms_e2e=ms_e2e, per_e2e=per_e2e, h2d=h2d_loc * world, d2h=d2h_loc * world)
    out_global = None
    if world > 1:
        n_sg = min(steps, 3)
        step_sg()
        ms_sg, out_global, per_sg = timed_checked(step_sg, n_sg, "root_scatter_gather")
        ident = lambda mu, mask, c, z: z                 # scatter + gather alone (no solve)
        step_sg(ident)
        ms_only, _, _ = timed(lambda: step_sg(ident), n_sg)
        res["sg"] = {"ms_per_step": ms_sg / n_sg, "value": frames_global * n_sg / (ms_sg * 1e-3), "steps": n_sg,
                     "scatter_gather_only_ms": ms_only / n_sg, "step_ms": per_sg,
                     "what": "rank 0 owns the global batch in HBM; NCCL P2P scatter of (mu, mask, c, z), solve, gather of the mel, all inside the timed region"}

    # parity: first / second / middle / last utterance re-solved by the CPU arm (the checker) — on the gathered global
    # batch when N > 1 (rank 0), so a wrong slice offset on ANY rank would show
    if rank == 0 and not args.no_cpu_baseline:
        threads = cpu_threads()
        torch.set_num_threads(threads)
        state = {k: v.detach().cpu().clone() for k, v in model.estimator.state_dict().items()}
        arm = CpuArm(state)
        got = out_global if out_global is not None else out_dev
        nb = Bglob if out_global is not None else Bper
        key = (name, tuple(sample_rows(nb)))
        if key not in _CPU_REF_CACHE:
            _CPU_REF_CACHE[key] = cpu_reference_solve(arm, inp, cfgd, sample_rows(nb), budget_s=args.cpu_budget)
        rows, ref, dt, note = _CPU_REF_CACHE[key]
        fr = int(inp["lens"][torch.as_tensor(rows)].sum())
        if world == 1 and full and precision == args.precision:
            res["cpu_baseline"] = {"value": fr / dt, "unit": "frames/s", "cores": threads, "kind": arm.kind,
                                   "sample": f"utterances {rows} of the batch (T={T}); {note}; os.cpu_count()={os.cpu_count()}"}
        if ref is not None:
            Tc = ref.shape[-1]
            d = got[torch.as_tensor(rows, device=got.device)][:, :, :Tc].cpu().double() - ref.double()
            res["parity"] = {"max_rel": float(d.abs().max() / ref.abs().max()), "l2_rel": float(d.norm() / ref.double().norm()),
                             "rows": rows, "vs": f"CPU {arm.kind} on the same inputs, full solve, utterances {rows} of the "
                                                 f"{'gathered global' if out_global is not None else 'measured'} batch"}
        else:
            res["parity"] = {"max_rel": None, "note": f"full-NFE CPU solve exceeds --cpu-budget ({note})"}

    # instrumented solve: per-class CUDA-event timing of every launch (roofline) — rank 0's slice, no collectives
    if full and rank == 0:
        lib, h = _lib.load_library(), model.estimator._handle
        lib.st_profile_begin(h)
        step_device()
        n = _lib.ST_PROF_NCAT
        ms_a, fl_a, by_a, ln_a = (C.c_double * n)(), (C.c_double * n)(), (C.c_double * n)(), (C.c_int64 * n)()
        lib.st_profile_end(h, ms_a, fl_a, by_a, ln_a)
        is_a = (C.c_double * n)()
        lib.st_profile_issued(h, is_a)
        prof = {nm: dict(ms=ms_a[i], flops=fl_a[i], bytes=by_a[i], launches=int(ln_a[i]), issued=is_a[i]) for i, nm in enumerate(_lib.ST_PROF_NAMES)}
        prof["gemm"] = {k: sum(v[k] for n_, v in prof.items() if n_.startswith("gemm_")) for k in ("ms", "flops", "bytes", "launches", "issued")}
        res["prof"] = prof
    if world > 1:
        dist.barrier()
    del local, glob
    torch.cuda.empty_cache()
    return res


def run_vocoder(args, dev, mel, flush, steps=5):
    """SURVEY.md §8 row f4: the vocoder hand-off (api.py:76) on the mel the solve just produced — Vocos at the reference's
    VocosConfig / MelConfig sizes (dim 768, 12 ConvNeXt blocks, n_fft 2048, hop 512, 44.1 kHz) with input width n_mel = 80,
    seeded synthetic weights.  Reports vocoder frames/s and audio-seconds/s, and the parity of two utterances vs the oracle."""
    from stabletts_b200 import Vocos
    from oracle import vocoder_ref as V
    st = V.make_state(input_channels=N_MEL)
    d = dict(V.DIMS); d["input_channels"] = N_MEL
    voc = Vocos(**d).eval()
    voc.load_state_dict(st, strict=True)
    voc = voc.to(dev)
    voc.set_engine(args.engine)
    B, _, T = mel.shape
    for _ in range(3):
        audio = voc(mel)
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    ev[0].record()
    for i in range(steps):
        flush.zero_()
        audio = voc(mel)
        ev[i + 1].record()
    torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[steps]) / steps
    out = {"workload": f"Vocos (dim 768, 12 blocks, n_fft 2048, hop 512) on the solve's mel: B={B}, n_mel={N_MEL}, T={T}",
           "ms_per_step": ms, "frames_per_s": B * T / (ms * 1e-3), "audio_seconds_per_s": B * T * 512 / 44100.0 / (ms * 1e-3),
           "sample_rate": 44100, "gflop_per_frame": 0.088, "tflops": B * T * 88.0e6 / (ms * 1e-3) / 1e12,
           "gpu_launches_per_step": None}
    if not args.no_cpu_baseline:
        rows = [0, B - 1]
        with torch.inference_mode():
            ref = V.vocos_forward(st, mel[rows].cpu())
        dlt = audio[rows].cpu().double() - ref.double()
        out["parity"] = {"max_rel": float(dlt.abs().max() / ref.abs().max()), "l2_rel": float(dlt.norm() / ref.double().norm()),
                         "vs": f"oracle/vocoder_ref.py (pinned against the unmodified reference Vocos) on utterances {rows}"}
    return out


DUMP_BYTES = 60_000_000            # the .npy header and rounding stay well inside 64 MB


def dump_outputs(out_dir, mel):
    """Writes the (B, n_mel, T) mel the timed solve returned in its last step as out_dir/mel.npy in float32, so that
    two builds run with the same arguments (hence the same seeded inputs) can be compared output for output.  A batch
    larger than DUMP_BYTES is cut to a fixed, seeded sample of utterances, kept in batch order."""
    import numpy as np
    mel = mel.detach().float().cpu()
    if mel.numel() * 4 > DUMP_BYTES:
        n = DUMP_BYTES // (mel[0].numel() * 4)
        rows = torch.randperm(mel.shape[0], generator=torch.Generator().manual_seed(0))[:n].sort().values
        mel = mel[rows]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "mel.npy"), mel.numpy())


def work_flops(cfgd, lens):
    nfe = cfgd["n_steps"] * NFE_PER_STEP[cfgd["method"]] * (2 if cfgd["cfg"] is not None else 1)
    lens = lens.double()
    hoisted = float(((nfe * (32.948e6 - COND_FLOPS) + COND_FLOPS) * lens + nfe * 6144.0 * lens * lens).sum())
    faithful = float((nfe * (32.948e6 * lens + 6144.0 * lens * lens)).sum())
    return nfe, hoisted, faithful


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg1", choices=list(CONFIGS))
    ap.add_argument("--engine", default="tcgen05", choices=["tcgen05", "simt"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-budget", type=float, default=30.0, help="seconds of CPU work for the cpu_baseline / parity leg")
    ap.add_argument("--no-cfg4", action="store_true", help="at N=8 skip the additional BASELINE cfg4 block (128/GPU = 1024 global)")
    ap.add_argument("--no-vocoder", action="store_true", help="skip the vocoder hand-off block (row f4)")
    ap.add_argument("--precision", default="ffn_fp16x2", choices=["ffn_fp16x2", "bf16x3"],
                    help="operand precision of the headline run: ffn_fp16x2 (the library default: split-bf16 x 3 everywhere except the FFN "
                         "convs, fp16 activations x fp16 hi/lo weights in 2 passes) or bf16x3 (3 passes everywhere); at N = 1 the OTHER mode "
                         "is measured beside it and reported under 'other_precision'")
    ap.add_argument("--no-second-precision", action="store_true", help="skip the secondary precision block")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps write the mel the last timed step returned "
                                                          "(rank 0's batch slice) as DIR/mel.npy, float32, at most 64 MB")
    ap.add_argument("--ncu-mode", action="store_true",
                    help="for `ncu` launch lists only: honours --warmup < 3, skips e2e / instrumented / CPU legs (numbers printed under a profiler are never bench values)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the CUDA path computed (--impl ours)")
    cfgd = CONFIGS[args.config]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, cfgd, rank)
        return
    if args.warmup < 3 and not args.ncu_mode:
        args.warmup = 3
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    import torch.distributed as dist
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    model = make_model(dev)
    model.estimator.set_engine(args.engine)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                 # started BEFORE warm-up: nvidia-smi start-up stalls the driver for ~100 ms
    r = run_config(args, args.config, model, dev, rank, world, args.steps, args.warmup, flush, full=True, precision=args.precision)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, r.pop("out_last"))
    if args.ncu_mode:
        if rank == 0:
            print(json.dumps({"ncu_mode": True, "ms_per_step_under_profiler": r["ms_dev"] / args.steps, "gpu_launches": r["launches"]}))
        if world > 1:
            dist.destroy_process_group()
        return
    # the other precision mode on the same box, same inputs (decide-with-evidence block: throughput, parity, GEMM roofline)
    other = None
    if world == 1 and not args.no_second_precision and args.engine == "tcgen05":
        other_name = "bf16x3" if args.precision == "ffn_fp16x2" else "ffn_fp16x2"
        try:
            other = run_config(args, args.config, model, dev, rank, world, min(args.steps, 4), 3, flush, full=True, precision=other_name)
            other["precision"] = other_name
        except Exception as e:                              # noqa: BLE001
            other = {"error": repr(e)[:300], "precision": other_name}
        model.estimator.set_precision(args.precision)
    vocoder = None
    if rank == 0 and world == 1 and not args.no_vocoder and r.get("out_dev") is not None:
        try:
            vocoder = run_vocoder(args, dev, r["out_dev"], flush)
        except Exception as e:                              # noqa: BLE001 — the headline must not die with the extra block
            vocoder = {"error": repr(e)[:300]}
    # BASELINE cfg4 AS WRITTEN (batch 1024 over 8 GPUs = 128 per GPU) rides along in the N = 8 run of the default config
    r4 = None
    if world == 8 and args.config == "cfg1" and not args.no_cfg4:
        r4 = run_config(args, "cfg4", model, dev, rank, world, min(args.steps, 3), 3, flush, full=False, precision=args.precision)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = float(peaks.get("bf16_tflops_sustained", 1400.0))
    peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained)" if peaks else "fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)"
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "gemm_traffic.json")))["dram_bytes_per_launch_avg"]
    except Exception:
        pass
    prof = r["prof"]
    gm = prof["gemm"]
    ach_tf = gm["flops"] / (gm["ms"] * 1e-3) / 1e12 if gm["ms"] > 0 else 0.0
    nfe, hoisted, faithful = work_flops(cfgd, r["inp"]["lens"])
    sec_step = r["ms_dev"] * 1e-3 / args.steps
    value = r["frames"] * args.steps / (r["ms_dev"] * 1e-3)
    e2e_val = r["frames"] * args.steps / (r["ms_e2e"] * 1e-3)

    def block(rr, n_steps):
        b = {"workload": f"{rr['name']}: {rr['cfgd']['desc']}", "global_batch": rr["Bglob"], "T": rr["T"], "frames_per_step": rr["frames"],
             "steps": n_steps, "value": rr["frames"] * n_steps / (rr["ms_dev"] * 1e-3), "ms_per_step": rr["ms_dev"] / n_steps,
             "e2e": {"value": rr["frames"] * n_steps / (rr["ms_e2e"] * 1e-3), "ms_per_step": rr["ms_e2e"] / n_steps,
                     "h2d_bytes_per_step": rr["h2d"], "d2h_bytes_per_step": rr["d2h"]},
             "root_scatter_gather": rr.get("sg"), "parity": rr.get("parity"), "step_ms": rr["per_dev"], "unit": "frames/s"}
        return b

    line = {
        "metric": "mel-frames/sec through CFM DiT estimator (ODE solve, all evaluations)",
        "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "warmup_steps_run": r["n_warm"],
        "ms_per_step": 1e3 * sec_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": ("f32" if args.engine != "tcgen05" else
                  "f32 (split-bf16x3 tensor-core operands, fp32 accumulate)" if args.precision == "bf16x3" else
                  "f32 (split-bf16x3 tensor-core operands; FFN convs fp16 activations x fp16 hi/lo weights, 2 passes; fp32 accumulate)"),
        "data": "synthetic",
        "config": {"workload": f"{args.config}: {cfgd['desc']}", "global_batch": r["Bglob"], "T": r["T"], "nfe": nfe,
                   "frames_per_step": r["frames"], "parallelism": f"batch-shard x{world}",
                   "inputs": "every rank owns its contiguous batch slice (value: resident in its HBM; e2e: its own pinned host buffers); "
                             "the rank-0 NCCL scatter/gather variant is reported under root_scatter_gather",
                   "l2": "256 MiB flush between steps; per-eval working set (~1.5 GB) exceeds the 126 MB L2",
                   "engine": args.engine},
        "clocks": {"sm_mhz": clocks["sm_mhz"], "sm_max_mhz": clocks["sm_max_mhz"], "reasons": clocks["reasons"],
                   "samples": clocks["samples"], "power_w_max": clocks.get("power_w_max")},
        "e2e": {"value": e2e_val, "unit": "frames/s", "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"],
                "ms_per_step": r["ms_e2e"] / args.steps,
                "api": "CFMDecoder.solve_host -> st_solve_host (C ABI): pinned host buffers, H2D + solve + D2H + stream sync inside the call, per rank"},
        "root_scatter_gather": r.get("sg"),
        "gpu_launches": r["launches"], "host_enqueue_ms_per_step": round(r["host_ms"], 2),
        "step_ms": {"value": r["per_dev"][:32], "e2e": r["per_e2e"][:32]}, "remeasured": r["remeasured"],
        "roofline": {"bound": "tensor", "kernel": "gemm_tc2_kernel / gemm_tc_kernel (tcgen05 split-bf16 conv-GEMM, all launches of one solve)",
                     "achieved": ach_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach_tf / peak_tf, "traffic": traffic,
                     "traffic_note": "dram__bytes_read+write per launch, mean over the ncu --set full capture in profiles/gemm_traffic.json",
                     "achieved_per_launch_gflop": gm["flops"] / max(gm["launches"], 1) / 1e9,
                     "issued_tflops": gm.get("issued", 0.0) / max(gm["ms"], 1e-9) / 1e9,
                     "issued_frac": gm.get("issued", 0.0) / max(gm["ms"], 1e-9) / 1e9 / peak_tf,
                     "issued_note": "tensor-core FLOPs actually issued (MMA passes x algorithmic, st_profile_issued) / the same time / the same "
                                    "peak: the tensor-pipe utilisation behind the algorithmic `frac`",
                     "peak_source": peak_src, "launches": gm["launches"], "kernel_ms_per_step": gm["ms"],
                     "note": "algorithmic FLOPs (2*rows*N*K*taps); the bf16x3 split issues 3 MMAs per algorithmic MAC"
                             + (", the FFN convs 2 (fp16 activations x fp16 hi/lo weights)" if args.precision == "ffn_fp16x2" else ""),
                     "precision": args.precision},
        "breakdown_ms_per_step": {k: round(v["ms"], 3) for k, v in prof.items()},
        "breakdown_tflops": {k: round(v["flops"] / max(v["ms"], 1e-9) / 1e9, 1) for k, v in prof.items() if v["flops"] > 0},
        "attention": {"tflops": prof["attention"]["flops"] / max(prof["attention"]["ms"], 1e-9) / 1e9},
        "ln": {"gbs": prof["ln"]["bytes"] / max(prof["ln"]["ms"], 1e-9) / 1e6, "hbm_peak_gbs": peaks.get("hbm_gbs")},
        "work": {"hoisted_tflop_per_step": hoisted / 1e12, "faithful_tflop_per_step": faithful / 1e12,
                 "whole_solve_tflops_hoisted": hoisted / 1e12 / sec_step / max(world, 1) * 1.0},
        "cpu_baseline": r.get("cpu_baseline"), "parity": r.get("parity"),
    }
    if r4 is not None:
        line["cfg4"] = block(r4, min(args.steps, 3))
    if vocoder is not None:
        line["vocoder"] = vocoder
    if other is not None:
        if "error" in other:
            line["other_precision"] = other
        else:
            n2 = min(args.steps, 4)
            og = other["prof"]["gemm"]
            o_tf = og["flops"] / (og["ms"] * 1e-3) / 1e12 if og["ms"] > 0 else 0.0
            line["other_precision"] = {
                "precision": other["precision"], "value": other["frames"] * n2 / (other["ms_dev"] * 1e-3), "unit": "frames/s",
                "ms_per_step": other["ms_dev"] / n2, "e2e_ms_per_step": other["ms_e2e"] / n2, "parity": other.get("parity"),
                "roofline": {"achieved": o_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": o_tf / peak_tf,
                             "issued_frac": og.get("issued", 0.0) / max(og["ms"], 1e-9) / 1e9 / peak_tf,
                             "note": "same algorithmic FLOPs; the FFN and long-skip convs issue 2 MMAs per MAC in ffn_fp16x2 mode, 3 in bf16x3"},
                "breakdown_ms_per_step": {k: round(v["ms"], 3) for k, v in other["prof"].items()},
                "note": "the other st_set_precision mode measured on the same box right after the headline run; the headline (value, e2e) is the --precision mode"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
