#!/usr/bin/env python
"""Benchmark of the hot path: realizations/s of 67-pulsar ng15-shaped EFAC/EQUAD + ECORR + red noise
+ HD-correlated GWB residuals (BASELINE.json metric), on N GPUs of one node.

    python bench.py --gpus N --steps K --warmup W            # our arm (torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K ...   # CPU arm: the UNMODIFIED reference on host cores
    python bench.py --config 3|4|5|exact ...                  # the other BASELINE configs as the headline workload
    python bench.py ... --dump-outputs DIR                    # + the last timed step's result rows, DIR/residuals.npy

A step = one batch of R realizations (default 1000) of the whole 67-pulsar array through
``PulsarBatch.generate`` (throughput mode: in-kernel Philox; outputs stay in HBM).  ``value`` = realizations of
all ranks / max-over-ranks device time.  ``e2e`` = the same metric through ``ptar_run_job_to_host``: per-step
noise parameters are copied host->device from pinned memory and every residual is copied back to pinned host
memory inside the timed region.  ``roofline`` is for the dominant kernel (the fused generator): algorithmic
bytes = 8 B x sum(N_toa) x realizations per launch (SURVEY.md 8d), duration from CUDA events around every
launch in the timed region, peak = MEASURED_PEAKS.json ``hbm_gbs``.

The default run (what the driver records) also carries, at N = 1: ``other_configs`` (BASELINE configs 3 and 4
and the literal F @ a generator, ``exact_epochs``), ``variants`` (two white draws per TOA like the reference;
library-accurate and float64 Box-Muller builds), ``cpu_baseline`` (the unmodified reference and the numpy port
on the host cores) and ``setup_s``; at N > 1: ``config5`` (BASELINE config 5: 100k realizations of ng15-epoch
strong-scaled over the ranks with the final NCCL all-gather chunked and overlapped with generation, timed with
and without the collective).
"""
from __future__ import annotations

import argparse
import atexit
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "realizations/sec (67-psr ng15 GWB+RN+ECORR)"
FALLBACK_HBM_GBS = 6650.0
SEED = 20250922
DUMP_BYTES = 60_000_000      # --dump-outputs writes at most this much (under 64 MB with the .npy header)
NVLINK_PEER_GBS = 770.0      # B200_PROFILING.md: measured peer copy per direction per GPU (900 nominal)
CGW3 = dict(gwtheta=1.5707963267948966, gwphi=2.5, mc=1e9, dist=5.0, fgw=1e-8, phase0=0.5, psi=1.5, inc=0.7853981633974483,
            pdist=1.0, psrTerm=True, evolve=True, tref=53000 * 86400)   # the reference test's source (tests/...:48-53)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        with open(p) as fh:
            d = json.load(fh)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


def source_hash():
    """sha256 over the generator kernel's device code (ptar_generate.cuh, ptar_rng.cuh): stamps the ncu capture that
    `roofline.traffic` comes from, so a figure captured from an older generator is visibly stale."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "pta_replicator_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f in ("ptar_generate.cuh", "ptar_rng.cuh"):      # the device code of the captured kernel (gen_kernel)
            with open(os.path.join(d, f), "rb") as fh:
                h.update(fh.read())
    return h.hexdigest()[:16]


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag, self.proc = index, [], False, None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.terminate)      # also when the run fails before finish(): no nvidia-smi left behind
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.samples.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc is not None:
            self.proc.terminate()
        sm = sorted(float(s[0]) for s in self.samples if s and s[0].replace(".", "").isdigit())
        mx = [float(s[1]) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()]
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------ CPU arms
def cpu_arms(psrs, noise, seconds, want_port=True):
    """The reference's own CPU path on this box's host cores (bounded samples):
    kind "reference" = the unmodified functions under the stub harness (oracle/refrecipe.py; staged bytecode from
    oracle/_ref when /root/reference is absent), kind "port" = the numpy restatement (oracle/recipe.py)."""
    from oracle import recipe, refrecipe, refstubs
    from pta_replicator_b200.distributed import usable_cores
    cores = usable_cores()
    res = {"cores": cores, "cores_how": "len(sched_getaffinity) capped by the cgroup cpu quota", "os_cpu_count": os.cpu_count()}
    if refstubs.available():
        ds = refrecipe.dataset_from_pulsars(psrs, noise)
        _, one = refrecipe.timed_realizations(ds, 1, 1)
        done, wall = refrecipe.timed_realizations(ds, cores * 8, cores, budget_s=seconds)
        res["reference"] = {"value": done / wall, "single_core": 1.0 / one, "realizations": done, "wall_s": wall,
                            "root": "staged bytecode (oracle/_ref)" if refstubs.available() != refstubs.REFERENCE_ROOT else "/root/reference"}
    if want_port:
        ds = recipe.dataset_from_pulsars(psrs, noise)
        _, one = recipe.timed_realizations(ds, 1, 1)
        done, wall = recipe.timed_realizations(ds, cores * 8, cores, budget_s=min(seconds, 10.0))
        res["port"] = {"value": done / wall, "single_core": 1.0 / one, "realizations": done, "wall_s": wall}
    return res


def cpu_baseline_block(arms):
    kind = "reference" if "reference" in arms else "port"
    a = arms[kind]
    what = ("the UNMODIFIED reference functions add_measurement_noise / add_jitter / add_red_noise / add_gwb under the "
            "stub harness (PINT's adjust_TOAs / Residuals are no-ops: flatters the reference)") if kind == "reference" else \
           "numpy oracle port (no PINT, no dense U: faster than the unmodified reference)"
    blk = {"value": a["value"], "unit": "realizations/s", "cores": arms["cores"], "kind": kind,
           "single_core_value": a["single_core"],
           "sample": f"{a['realizations']} realizations of the same workload in {a['wall_s']:.1f} s, one single-threaded process per "
                     f"usable core ({arms['cores']}; os.cpu_count() = {arms['os_cpu_count']}); {what}"}
    if kind == "reference" and "port" in arms:
        blk["port"] = {"value": arms["port"]["value"], "single_core_value": arms["port"]["single_core"],
                       "note": "numpy restatement of the same recipe (oracle/recipe.py), same pool"}
    return blk


def run_reference(args):
    """The reference arm: the reference's own CPU implementation of the path on all usable host cores;
    a step = one realization per core (pool start-up and one warm-up realization per worker untimed)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import recipe, refrecipe, refstubs
    from pta_replicator_b200 import synthetic
    from pta_replicator_b200.distributed import usable_cores
    psrs, noise = synthetic.make_ng15_like(args.kind)
    cores = usable_cores()
    use_ref = bool(refstubs.available())
    mod = refrecipe if use_ref else recipe
    ds = mod.dataset_from_pulsars(psrs, noise)
    _, one = mod.timed_realizations(ds, 1, 1)
    per_step = cores
    budget = max(20.0, 150.0 / max(args.steps, 1))
    done_total, wall = 0, 0.0
    for _ in range(args.steps):
        done, w = mod.timed_realizations(ds, per_step, cores, budget_s=budget)
        done_total += done
        wall += w
    value = done_total / wall
    ntoa = sum(p.toas.ntoas for p in psrs)
    kind = "reference" if use_ref else "port"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "realizations/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"ng15-{args.kind}: 67 psr, sum N_toa={ntoa}, EFAC/EQUAD+ECORR(1s)+RN(30 comp)+HD GWB(npts=600,howml=10)",
                       "realizations_per_step": per_step},
            "cpu_baseline": {"value": value, "unit": "realizations/s", "cores": cores, "kind": kind,
                             "single_core_value": 1.0 / one,
                             "sample": f"{per_step} realizations/step x {args.steps} steps ({done_total} completed), one single-threaded process "
                                       f"per usable core ({cores}; os.cpu_count() = {os.cpu_count()}); "
                                       + ("UNMODIFIED reference functions under the stub harness, "
                                          + ("staged bytecode oracle/_ref" if refstubs.available() != refstubs.REFERENCE_ROOT else "/root/reference")
                                          + " (PINT stubs: flatters the reference)" if use_ref else "numpy oracle port")},
            "e2e": {"value": value, "unit": "realizations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ GPU arm
def aniso_clm(psrs, lmax=6, seed=SEED):
    """BASELINE config 4 (SURVEY.md 8d): clm[0] = sqrt(4 pi), clm[1:] ~ 0.05 N(0,1), redrawn until the ORF is PD."""
    import numpy as np
    from pta_replicator_b200 import orf as orf_mod
    radec = orf_mod.psrlocs_from_pulsars(psrs)
    locs = np.stack([radec[:, 0], np.pi / 2.0 - radec[:, 1]], axis=1)
    basis = orf_mod.correlated_basis(locs, lmax)
    rng = np.random.default_rng(seed)
    for _ in range(100):
        clm = np.r_[np.sqrt(4 * np.pi), 0.05 * rng.standard_normal((lmax + 1) ** 2 - 1)]
        orf = 2.0 * sum(c * b for c, b in zip(clm, basis))
        if np.all(np.linalg.eigvalsh(orf) > 0):
            return list(clm)
    raise RuntimeError("no positive-definite anisotropic ORF in 100 draws")


def make_batch(cfg, args, merged=True, exact=False, psrs_noise=None):
    """cfg '2': EFAC/EQUAD + ECORR + RN + HD GWB (the metric config); '3': + CGW; '4': anisotropic GWB lmax = 6;
    '5': config 2's recipe on ng15-epoch (one TOA per epoch)."""
    from pta_replicator_b200 import synthetic
    from pta_replicator_b200.engine import PulsarBatch
    t0 = time.perf_counter()
    kind = "epoch" if cfg == "5" else args.kind
    psrs, noise = psrs_noise if psrs_noise is not None else synthetic.make_ng15_like(kind)
    b = PulsarBatch(psrs, rn_taylor_tol=args.taylor_tol, exact_epochs=exact)
    b.white_merged = merged
    synthetic.ng15_recipe(b, noise, gwb=(cfg != "4"))
    if cfg == "3":
        b.add_cgw(**CGW3)
    if cfg == "4":
        b.set_gwb(-14.6733, 13.0 / 3.0, lmax=6, clm=aniso_clm(psrs))
    if args.chunk:
        b.default_chunk = args.chunk
    b.split_epoch = bool(args.split)
    b.compile()
    return b, psrs, noise, time.perf_counter() - t0, kind


def workload_name(cfg, kind, b, exact=False):
    extra = {"2": "", "3": " + CGW", "4": " (anisotropic ORF, lmax=6)", "5": ""}[cfg]
    gw = "GWB(npts=600,howml=10)" if cfg == "4" else "HD GWB(npts=600,howml=10)"
    return (f"ng15-{kind}: 67 psr, sum N_toa={b.n_toa_total}, EFAC/EQUAD+ECORR(1s)+RN(30 comp)+{gw}{extra}"
            + (", exact_epochs (one epoch per TOA: the literal F @ a)" if exact else ""))


def dump_outputs(dirpath, out):
    """``--dump-outputs``: write ``dirpath/residuals.npy``, the rows (realizations) of ``out`` [rows, ld] (fp64, packed
    engine order, as ``PulsarBatch.generate`` returns it) at a fixed, seeded choice of row indices; as many rows as fit in
    DUMP_BYTES.  Same arguments, same rows: two builds can be compared output for output."""
    import numpy as np
    import torch
    n_rows, ld = out.shape
    rows = np.sort(np.random.default_rng(SEED).choice(n_rows, size=min(n_rows, DUMP_BYTES // (8 * ld)), replace=False))
    os.makedirs(dirpath, exist_ok=True)
    np.save(os.path.join(dirpath, "residuals.npy"), out[torch.from_numpy(rows).to(out.device)].cpu().numpy())


def timed_steps(b, R, steps, warmup, rc, world=1, rank=0, dist=None, k0=0, dump=None):
    """W untimed + K timed steps bracketed by barrier + synchronize; returns (ms max over ranks, per-kernel dict).
    ``dump(out)`` (optional) receives the output buffer as the last timed step left it."""
    import numpy as np
    import torch
    out = getattr(b, "_bench_out", None)
    if out is None or out.shape[0] != R:
        out = torch.zeros((R, b.ld), dtype=torch.float64, device=b.device)
        b._bench_out = out

    def step(k, timers=None):
        real0 = (((k0 + k) * world + rank) * R + 3) // 4 * 4     # rank-major blocks of global ids
        b.generate(R, seed=SEED, real0=real0, out=out, rc=rc, timers=timers)

    for k in range(warmup):
        step(k)
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for k in range(steps):
        step(warmup + k)
    e1.record()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    ms = e0.elapsed_time(e1)
    if dump is not None:
        dump(out)
    timers = {}
    for k in range(steps):     # same K steps again with CUDA events around every launch (same stream, same schedule)
        step(warmup + steps + k, timers)
    torch.cuda.synchronize()
    tms = torch.tensor([ms], dtype=torch.float64, device=b.device)
    if dist is not None:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    per = {}
    for name, a, z in timers["events"]:
        per.setdefault(name, []).append(a.elapsed_time(z))
    kern = {k: {"launches": len(v), "avg_ms": float(np.mean(v)), "total_ms": float(np.sum(v))} for k, v in per.items()}
    return float(tms.item()), kern, step


def roofline_of(b, kern, R, steps, hbm, how):
    gen = kern["generate"]
    n_gen = gen["launches"]
    alg = 8.0 * b.n_toa_total * (R * steps / n_gen)
    achieved = alg / (gen["avg_ms"] * 1e-3) / 1e9
    total = sum(k["total_ms"] for k in kern.values())
    return {"bound": "hbm", "kernel": "gen_kernel (fused white+ECORR+red+GWB-interp generator)", "achieved": achieved,
            "peak": hbm, "unit": "GB/s", "frac": achieved / hbm, "traffic": None, "peak_source": how,
            "algorithmic_bytes_per_launch": alg, "avg_launch_ms": gen["avg_ms"], "share_of_step": gen["total_ms"] / total,
            "whole_step_frac": 8.0 * b.n_toa_total * R * steps / (total * 1e-3) / 1e9 / hbm}


def short_line(b, R, rc, hbm, how, steps=3, warmup=2):
    ms, kern, _ = timed_steps(b, R, steps, warmup, rc)
    rf = roofline_of(b, kern, R, steps, hbm, how)
    return {"value": R * steps / (ms * 1e-3), "unit": "realizations/s", "ms_per_step": ms / steps, "realizations_per_step": R,
            "kernels_ms_per_step": {k: v["total_ms"] / steps for k, v in kern.items()},
            "roofline_frac": rf["frac"], "whole_step_frac": rf["whole_step_frac"], "algorithmic_GBps": rf["achieved"]}


def config5_block(args, world, rank, dist, hbm, steps=1, warmup=1, dump=None):
    """BASELINE config 5: 100k realizations of ng15-epoch strong-scaled over the ranks, final all-gather chunked
    (C realizations per rank per chunk) and overlapped with generation on a second stream; timed with and without
    the collective on the identical schedule (``warmup`` untimed + ``steps`` timed runs each; ms per run); one gathered
    chunk is checked bit for bit against local regeneration.  ``dump(full)`` (optional) receives the gathered result of
    the last timed run."""
    import torch
    from pta_replicator_b200 import distributed as D
    b, psrs, noise, setup_s, kind = make_batch("5", args)
    nreal, chunk = args.c5_nreal, args.c5_chunk
    C, n_chunks, padded = D.gather_plan(nreal, world, chunk)
    full = torch.zeros((padded, b.ld), dtype=torch.float64, device=b.device)   # the packed axis' alignment tail is never written
    comm = torch.cuda.Stream(b.device) if world > 1 else None

    def run(gather):
        D.generate_gathered(b, nreal, seed=SEED, chunk=chunk, out=full, gather=gather, comm_stream=comm)

    res = {}
    for gather in (False, True):
        for _ in range(warmup):
            run(gather)                               # warm-up (also creates the NCCL channels)
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(steps):
            run(gather)
        e1.record()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        t = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device=b.device)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        res[gather] = float(t.item())
    if dump is not None:
        dump(full)
    p2p = None
    if world > 1:   # the same delivery by peer pushes (CUDA IPC + copy engines) instead of the NCCL collective
        try:
            p2p = {"how": "every rank maps the other ranks' result buffers (CUDA IPC) and pushes its chunks into them with the copy "
                          "engines over NVLink on side streams (one per peer) while the next chunk is generated; no SMs, no staging; timed "
                          "by the host clock from the first launch to the final stream sync (max over ranks)", "runs": {}}
            for ch in (chunk, 2048):
                Cp, ncp, padp = D.gather_plan(nreal, world, ch)
                if padp > full.shape[0]:
                    full = torch.empty((padp, b.ld), dtype=torch.float64, device=b.device)
                full.zero_()
                dl = D.PeerDelivery(full, n_streams=world - 1)
                for rep in range(2):
                    torch.cuda.synchronize()
                    dist.barrier()
                    t0 = time.perf_counter()
                    D.generate_gathered_p2p(b, nreal, seed=SEED, chunk=ch, out=full, delivery=dl)
                    torch.cuda.synchronize()
                    wall = time.perf_counter() - t0
                t = torch.tensor([wall * 1e3], dtype=torch.float64, device=b.device)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                other, c = (rank + 1) % world, ncp // 2
                r0 = D.chunk_ids(c, other, world, Cp)
                okp = int(torch.equal(b.generate(Cp, seed=SEED, real0=r0), full[r0:r0 + Cp]))
                tt = torch.tensor([okp], dtype=torch.int32, device=b.device)
                dist.all_reduce(tt, op=dist.ReduceOp.MIN)
                p2p["runs"][str(Cp)] = {"value_with_gather": padp / (float(t.item()) * 1e-3), "ms": float(t.item()),
                                        "shard_bitwise_ok": bool(int(tt.item())), "chunks": ncp,
                                        "recv_GBps_per_gpu": (world - 1) * padp / world * b.ld * 8.0 / (float(t.item()) * 1e-3) / 1e9}
                dl.close()
            best = max(p2p["runs"].values(), key=lambda v: v["value_with_gather"])
            p2p.update({k: best[k] for k in ("value_with_gather", "ms", "shard_bitwise_ok", "recv_GBps_per_gpu")})
            if full.shape[0] != padded:
                full = torch.empty((padded, b.ld), dtype=torch.float64, device=b.device)
        except Exception as e:  # noqa: BLE001 - report, keep the NCCL numbers
            p2p = {"error": str(e)[:300]}
    ok = 1
    if world > 1:   # rows another rank generated, as received here, against regenerating them on this GPU
        run(True)
        other, c = (rank + 1) % world, n_chunks // 2
        r0 = D.chunk_ids(c, other, world, C)
        mine = b.generate(C, seed=SEED, real0=r0)
        ok = int(torch.equal(mine, full[r0:r0 + C]))
        t = torch.tensor([ok], dtype=torch.int32, device=b.device)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        ok = int(t.item())
    recv = (world - 1) * padded / world * b.ld * 8.0           # bytes every GPU receives
    sweep = {}
    if world > 1:      # how the overlapped gather depends on the chunk size (same work, same ownership pattern)
        for ch in (128, 2048):
            Cs, ncs, pads = D.gather_plan(nreal, world, ch)
            if pads > full.shape[0]:
                full = torch.empty((pads, b.ld), dtype=torch.float64, device=b.device)
            for rep in range(2):
                torch.cuda.synchronize()
                dist.barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                D.generate_gathered(b, nreal, seed=SEED, chunk=ch, out=full, gather=True, comm_stream=comm)
                e1.record()
                torch.cuda.synchronize()
                dist.barrier()
            t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=b.device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            sweep[str(Cs)] = {"value_with_gather": pads / (float(t.item()) * 1e-3), "ms": float(t.item()), "chunks": ncs}
    blk = {"workload": workload_name("5", kind, b) + f"; {nreal} realizations strong-scaled over {world} GPU(s), chunk-interleaved ownership, "
                       f"{C} realizations per rank per chunk x {n_chunks} chunks ({padded} generated)",
           "value_without_gather": padded / (res[False] * 1e-3), "value_with_gather": padded / (res[True] * 1e-3),
           "ms_without_gather": res[False], "ms_with_gather": res[True], "unit": "realizations/s",
           "gathered_bytes_per_gpu": b.ld * 8.0 * padded, "gather_overlap": "NCCL all_gather_into_tensor of chunk c on a second stream while "
           "chunk c+1 is generated (two staging buffers)", "shard_bitwise_ok": bool(ok)}
    if world > 1:
        blk["p2p_push"] = p2p
        blk["chunk_sweep"] = sweep
        blk["nccl"] = {"high_priority_stream": os.environ.get("TORCH_NCCL_HIGH_PRIORITY", "")}
        blk["recv_GBps_per_gpu"] = recv / (res[True] * 1e-3) / 1e9
        blk["nvlink_frac_of_measured_peer_copy"] = blk["recv_GBps_per_gpu"] / NVLINK_PEER_GBS
        blk["gather_bound_ceiling"] = {"realizations_per_s": padded / (recv / (NVLINK_PEER_GBS * 1e9)),
                                       "note": f"every GPU must receive (G-1)/G of the result over NVLink: {recv / 1e9:.2f} GB at the measured "
                                               f"{NVLINK_PEER_GBS:.0f} GB/s peer-copy rate (B200_PROFILING.md)"}
    del full
    return blk


def bm_variant(lib, args):
    """Throughput of an alternative Box-Muller build of the library (PTAR_B200_LIB), in a fresh process."""
    env = dict(os.environ, PTAR_B200_LIB=lib)
    cmd = [sys.executable, os.path.abspath(__file__), "--steps", "3", "--warmup", "3", "--nreal", str(args.nreal), "--kind", args.kind,
           "--taylor-tol", str(args.taylor_tol), "--bare"]
    try:
        r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=300)
        d = json.loads(r.stdout.strip().splitlines()[-1])
        return {"value": d["value"], "unit": "realizations/s", "roofline_frac": d["roofline"]["frac"], "ms_per_step": d["ms_per_step"]}
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)[:200]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="2", choices=["2", "3", "4", "5", "exact"],
                    help="BASELINE.json configs: 2 = the metric config (default), 3 = + CGW, 4 = anisotropic lmax 6, "
                         "5 = ng15-epoch 100k realizations with the overlapped all-gather, exact = config 2 with one epoch per TOA")
    ap.add_argument("--nreal", type=int, default=1000, help="realizations per step per GPU")
    ap.add_argument("--kind", default="full", choices=["full", "epoch"])
    ap.add_argument("--rc", type=int, default=0)
    ap.add_argument("--chunk", type=int, default=0)
    ap.add_argument("--two-draws", action="store_true", help="two Philox normals per TOA (w1 z1 + w2 z2, like the reference) instead "
                                                             "of one merged N(0, w1^2+w2^2) draw")
    ap.add_argument("--e2e-nreal", type=int, default=256)
    ap.add_argument("--cpu-seconds", type=float, default=20.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-variants", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip other_configs / config5 blocks")
    ap.add_argument("--bare", action="store_true", help="headline measurement only (used for the library-variant sub-runs)")
    ap.add_argument("--split", action="store_true", help="epoch kernel + TOA kernel (two launches) instead of the fused generator")
    ap.add_argument("--taylor-tol", type=float, default=1e-13,
                    help="PulsarBatch(rn_taylor_tol=...): remainder bound of the in-epoch Taylor step, relative to the red-noise rms")
    ap.add_argument("--c5-nreal", type=int, default=100000)
    ap.add_argument("--c5-chunk", type=int, default=512)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed (rank 0's result rows, fp64, a fixed "
                         "seeded sample of at most 60 MB) to DIR/residuals.npy")
    args = ap.parse_args()
    if args.bare:
        args.no_cpu = args.no_variants = args.no_extras = True
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs needs the GPU arm (--impl ours)")
        return run_reference(args)

    import torch
    import __graft_entry__ as ge
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    from pta_replicator_b200 import distributed as D
    affinity0 = os.sched_getaffinity(0)
    numa = D.bind_to_gpu_numa(local)      # before any pinned allocation: staging buffers on the GPU's NUMA node
    dist = None
    if world > 1:
        import torch.distributed as dist
        # the NCCL kernels of the overlapped all-gather run next to a generator that fills every SM: give them a
        # high-priority stream so their CTAs are scheduled as soon as generator CTAs retire
        os.environ.setdefault("TORCH_NCCL_HIGH_PRIORITY", "1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    # the library is the one build() compiled into the tree: nothing is compiled here (the tree may be read-only)

    cfg = "2" if args.config == "exact" else args.config
    exact = args.config == "exact"
    hbm, how = peaks()
    dump = (lambda out: dump_outputs(args.dump_outputs, out)) if args.dump_outputs and rank == 0 else None
    if cfg == "5":               # config 5 as the headline: value = with the gather
        blk = config5_block(args, world, rank, dist, hbm, steps=args.steps, warmup=args.warmup, dump=dump)
        if rank == 0:
            print(json.dumps({"metric": METRIC, "value": blk["value_with_gather"], "unit": "realizations/s", "n_gpus": world,
                              "steps": args.steps, "warmup": args.warmup, "ms_per_step": blk["ms_with_gather"], "higher_is_better": True,
                              "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                              "config": {"workload": blk["workload"]}, "config5": blk}), flush=True)
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return

    b, psrs, noise, setup_s, kind = make_batch(cfg, args, merged=not args.two_draws, exact=exact)
    st = b.compile()
    R = args.nreal
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()          # samples span warm-up, the timed region and a short soak of the same steps
        t_wait = time.time()
        while not sampler.samples and time.time() - t_wait < 8.0:
            time.sleep(0.05)     # nvidia-smi can take a second to deliver its first sample
    ms_max, kern, step = timed_steps(b, R, args.steps, args.warmup, args.rc, world, rank, dist, dump=dump)
    if sampler:
        # the timed region lasts ~10-20 ms, shorter than nvidia-smi's 100 ms period: keep the identical load
        # running for ~0.7 s so that the clock / throttle record is taken under this load
        n0, t_soak, k = len(sampler.samples), time.time(), 0
        while time.time() - t_soak < 0.7:
            step(args.warmup + 2 * args.steps + k)
            torch.cuda.synchronize()
            k += 1
        clocks = sampler.finish()
        clocks["window"] = "warm-up + timed region + %d soak steps of the same load (%d samples before the soak)" % (k, n0)
    else:
        clocks = None
    value = world * R * args.steps / (ms_max * 1e-3)
    roof = roofline_of(b, kern, R, args.steps, hbm, how)
    n_gen = kern["generate"]["launches"]
    for prof in sorted(f for f in os.listdir(os.path.join(ROOT, "profiles")) if f.endswith("_traffic.json"))[::-1]:
        with open(os.path.join(ROOT, "profiles", prof)) as fh:
            tj = json.load(fh)
        cap_real = float(tj.get("gen_kernel_realizations_per_launch", 512))
        cap_bytes = float(tj.get("gen_kernel_dram_bytes_per_launch", 0.0))
        roof["traffic"] = cap_bytes / cap_real * (R * args.steps / n_gen)
        stale = tj.get("source_hash") != source_hash()
        roof["traffic_note"] = ("dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture (profiles/%s) of a %d-realization "
                                "launch (%.4g B; algorithmic %.4g B), scaled per realization; capture source hash %s, this build %s%s"
                                % (prof, cap_real, cap_bytes, 8.0 * b.n_toa_total * cap_real, tj.get("source_hash"), source_hash(),
                                   " -- STALE: the kernels changed since the capture" if stale else ""))
        roof["traffic_stale"] = bool(stale)
        break

    line = {"metric": METRIC, "value": value, "unit": "realizations/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(cfg, kind, b, exact),
                       "realizations_per_step_per_gpu": R,
                       "rng": "in-kernel Philox4x32-10 keyed on (seed, global realization id), fp32 MUFU Box-Muller (measured: "
                              "tests/test_gpu_statistics.py); all residual arithmetic fp64",
                       "white_draws_per_toa": 2 if args.two_draws else 1, "gwb_chunk": min(R, b.default_chunk),
                       "rn_taylor_tol": args.taylor_tol, "schedule": "epoch kernel + TOA kernel" if args.split else "fused generator",
                       "l2": f"output per step {R * b.ld * 8 / 1e9:.2f} GB > L2 (126 MB); no flush needed",
                       "parallelism": f"realization-sharded x{world}, no data-path collective in `value` (config5 block: with the all-gather)"},
            "kernels": kern, "kernels_timing": "second pass of the same K steps with CUDA events around every launch (same stream, same schedule)",
            "roofline": roof, "clocks": clocks, "setup_s": setup_s,
            "setup_note": "synthetic data set + PulsarBatch + recipe + plan() + compile() (host planning, uploads, Fourier basis, ORF Cholesky, "
                          "GWB factor QR), once per recipe; not in `value`",
            "gpu_launches": int(sum(k["launches"] for k in kern.values())), "source_hash": source_hash(), "numa_binding": numa}

    extras = world == 1 and rank == 0 and not args.no_extras
    # ---- variants (N == 1): the reference's two draws per TOA; library-accurate / float64 Box-Muller builds
    if world == 1 and not args.no_variants:
        var = {}
        b1, *_ = make_batch(cfg, args, merged=bool(args.two_draws), exact=exact, psrs_noise=(psrs, noise))
        v = short_line(b1, R, args.rc, hbm, how)
        v["note"] = ("w1 z1 + w2 z2 with two Philox normals per TOA, as the reference consumes them" if not args.two_draws else
                     "one merged N(0, w1^2 + w2^2) draw per TOA (same Gaussian law)")
        var["two_white_draws" if not args.two_draws else "merged_white_draw"] = v
        del b1
        for name, lib in (("box_muller_fp32_accurate", ge.LIB_BM1), ("box_muller_fp64", ge.LIB_BM2), ("philox4x32_7_rounds", ge.LIB_PHILOX7)):
            if os.path.isfile(lib) and not os.environ.get("PTAR_B200_LIB"):
                var[name] = bm_variant(lib, args)
        line["variants"] = var
    if extras:
        oc = {}
        for name, c, ex in (("config3_cgw", "3", False), ("config4_aniso_lmax6", "4", False), ("exact_epochs", "2", True)):
            if (c, ex) == (cfg, exact):
                continue
            bb, *_rest = make_batch(c, args, merged=not args.two_draws, exact=ex, psrs_noise=(psrs, noise))
            Rx = min(R, 256) if ex else R
            oc[name] = short_line(bb, Rx, args.rc, hbm, how)
            oc[name]["workload"] = workload_name(c, kind, bb, ex)
            oc[name]["setup_s"] = _rest[2]
            del bb
            torch.cuda.empty_cache()
        line["other_configs"] = oc

    # ---- e2e through the C ABI with host buffers (rank-local; aggregated like `value`)
    Re = min(args.e2e_nreal, R)
    pinned_out = torch.empty((Re, b.ld), dtype=torch.float64, pin_memory=True)
    host_in = {k: st[k].cpu().pin_memory() for k in ("w1", "w2", "wm", "ep_ecorr", "rn_scale") if k in st}
    h2d = int(sum(v.numel() * v.element_size() for v in host_in.values()))

    def e2e_step(k):
        for name, h in host_in.items():
            st[name].copy_(h, non_blocking=True)        # this step's noise parameters, pinned host -> device
        b.generate_to_host(Re, seed=SEED + 1, real0=4 * k * Re, out_host=pinned_out, chunk=32, rc=args.rc)

    for k in range(2):
        e2e_step(k)
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    ne2e = max(2, min(args.steps, 5))
    t0 = time.perf_counter()
    for k in range(ne2e):
        e2e_step(2 + k)
    torch.cuda.synchronize()
    te = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=b.device)
    if dist is not None:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    line["e2e"] = {"value": world * Re * ne2e / float(te.item()), "unit": "realizations/s", "h2d_bytes_per_step": h2d,
                   "d2h_bytes_per_step": int(Re * b.ld * 8), "realizations_per_step_per_gpu": Re, "steps": ne2e,
                   "d2h_GBps_per_gpu": Re * ne2e * b.ld * 8 / float(te.item()) / 1e9,
                   "path": "ptar_run_job_to_host: pinned H2D of noise parameters, generate in chunks of 32, D2H of every residual overlapped on a "
                           "second stream; the process is bound to its GPU's NUMA node before the pinned buffers are allocated"}
    del pinned_out

    if not args.no_extras:
        del b._bench_out
        torch.cuda.empty_cache()
        line["config5"] = config5_block(args, world, rank, dist, hbm)

    # ---- CPU baseline (rank 0, N == 1 only): the reference's own code on the host cores, bounded sample
    if rank == 0 and world == 1 and not args.no_cpu:
        os.sched_setaffinity(0, affinity0)     # the CPU arm may use every core this process was given
        line["cpu_baseline"] = cpu_baseline_block(cpu_arms(psrs, noise, args.cpu_seconds))
    if rank == 0:
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
