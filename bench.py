#!/usr/bin/env python
"""bench.py -- SHA-256 witness-generation throughput (blocks/s, bit-exact cells) on N B200s, next to the CPU path.

    python bench.py --gpus N --steps K --warmup W [--workload cfg2] [--impl reference] [--dump-outputs DIR]

A pass of the hot path over one batch of synthetic messages generates every advice / lookup / spread cell of every
instance into HBM (column-major Fr, Montgomery form) plus digests and cell checksums.  A timed step is L such passes back
to back (--launches-per-step; by default as many as make one step take >= 30 ms), and exactly K steps are timed.
--dump-outputs DIR writes what the last timed step computed to DIR (see dump_outputs).
At N=1 the workload is BASELINE.json configs[1] (1024 random 55-byte messages, one block each); with N>1 every
rank generates its own shard of the same size (weak scaling, no data-path collective; digests and checksums are
gathered over NCCL after the timed region).

JSON keys (one line, rank 0): see the task contract; `value` = whole-job blocks/s with inputs resident in HBM,
`e2e` = the same through the public C-ABI call with HOST message buffers (H2D inside, digests+checksums D2H),
`roofline` for k_expand (HBM-write bound) and `cpu_baseline` = the oracle (C restatement of the reference's
witness generation; the Rust crate cannot be built here) on this box's host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "SHA-256 blocks/sec witness-gen (bit-exact cells)"
UNIT = "blocks/s"
DUMP_BYTES_PER_ARRAY = 12 << 20   # --dump-outputs: five arrays, at most 60 MiB in all
DUMP_SEED = 0


def dump_outputs(out_dir, arrays):
    """Writes each output tensor as out_dir/<name>.npy without losing a bit: uint8 arrays as float32, 64-bit words as two
    float64 values each (low 32 bits first), one row per digest / per instance's checksums / per 32-byte cell.  An output
    larger than DUMP_BYTES_PER_ARRAY is a sample of its rows, drawn with a fixed seed and sorted; the row numbers (of the
    tensor flattened to rows) go to out_dir/<name>_rows.npy.  Equal arguments to bench.py give equal inputs, so the files of
    two builds compare entry for entry."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        rows = t.reshape(-1, t.shape[-1])
        row_bytes = rows.shape[1] * (4 if t.dtype == torch.uint8 else 16)
        if rows.shape[0] * row_bytes > DUMP_BYTES_PER_ARRAY:
            m = DUMP_BYTES_PER_ARRAY // (row_bytes + 8)
            idx = np.sort(np.random.default_rng(DUMP_SEED).choice(rows.shape[0], m, replace=False))
            rows = rows[torch.from_numpy(idx).to(rows.device)]
            np.save(os.path.join(out_dir, f"{name}_rows.npy"), idx.astype(np.float64))
        h = rows.cpu().numpy()
        h = h.astype(np.float32) if h.dtype == np.uint8 else h.view(np.uint32).astype(np.float64)
        np.save(os.path.join(out_dir, f"{name}.npy"), h)


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy read+write)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """Samples clocks / throttle reasons with one `nvidia-smi -lms 100` process running across the timed region."""

    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw,clocks.mem"

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.gpu), "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        lines = []
        if self.proc is not None:
            self.proc.terminate()
            try:
                out, _ = self.proc.communicate(timeout=5)
                lines = out.strip().splitlines()
            except Exception:
                self.proc.kill()
        sm, mx, reasons, pw, mem = [], 0, set(), [], []
        for ln in lines:
            s = [x.strip() for x in ln.split(",")]
            try:
                sm.append(float(s[0])); mx = max(mx, float(s[1]))
            except Exception:
                continue
            try:
                pw.append(float(s[6])); mem.append(float(s[7]))
            except Exception:
                pass
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], s[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm),
                "power_w": float(np.median(pw)) if pw else None, "mem_mhz": float(np.median(mem)) if mem else None}


def cpu_baseline(workload, sample_instances: int, n_threads: int, first: int = 0):
    """Times the oracle (CPU restatement of the reference's witness generation) on a bounded sample."""
    from oracle import oracle as O
    import __graft_entry__ as ge
    S = ge.load_package_module("synthetic")
    O.build()
    ocfg = O.OracleConfig(max_variable_byte_sizes=tuple(workload.max_variable_byte_sizes))
    blob, offs, lens = S.generate(workload, first, sample_instances)
    blob = np.concatenate([blob, np.zeros(1, np.uint8)])
    # layout: take it from one synthesized region
    reg = O.synthesize(ocfg, [bytes(blob[int(offs[0]):int(offs[0]) + int(lens[0])])], record_shape=False)
    lay = reg.layout()
    t0 = time.perf_counter()
    out = O.batch_packed(ocfg, lay, sample_instances, blob, offs, lens, np.zeros(sample_instances, np.uint32), want_cells=False, n_threads=n_threads)
    dt = time.perf_counter() - t0
    blocks = sample_instances * workload.blocks_per_instance
    return blocks / dt, dt, out


def make_config(w, lay, per_gpu):
    """`config` of the JSON line; the GPU arm and the reference arm print the same dict for the same workload."""
    return {"workload": f"{w.name}: {w.description}", "instances_per_gpu": per_gpu, "blocks_per_instance": lay.n_blocks,
            "cells_per_instance": lay.cells_per_instance, "bytes_per_instance": lay.cells_per_instance * 32,
            "l2": f"outputs {per_gpu * lay.bytes_per_instance / 1e9:.2f} GB per launch, larger than the 126 MB L2 (no flush needed)",
            "sharding": "independent instances per rank, no data-path collective"}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path.  The Rust crate cannot be built in this image
    (no cargo/rustc, git dependencies, no network), so this times the oracle port on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import __graft_entry__ as ge
    S = ge.load_package_module("synthetic")
    w = S.WORKLOADS[args.workload]
    cores = os.cpu_count() or 1
    sample = min(w.n_instances, max(cores * 4, int(args.cpu_sample)))
    # layout numbers of `config` from the oracle itself (this arm never loads the engine's library)
    from types import SimpleNamespace

    from oracle import oracle as O
    reg = O.synthesize(O.OracleConfig(max_variable_byte_sizes=tuple(w.max_variable_byte_sizes)), [b""] * len(w.max_variable_byte_sizes), record_shape=False)
    ol = reg.layout()
    cells = reg.n_gate + len(reg.lookup_idx) + 2 * reg.dense.shape[0]
    lay = SimpleNamespace(n_blocks=w.blocks_per_instance, cells_per_instance=cells,
                          bytes_per_instance=32 * (ol.n_gate_cols * ol.gate_col_rows + ol.n_lookup_cols * ol.lookup_col_rows + 4 * ol.spread_rows))
    per_gpu_nominal = args.instances or min(w.n_instances, int(0.6 * 170e9) // lay.bytes_per_instance)
    for _ in range(args.warmup):
        cpu_baseline(w, min(sample, cores), cores)
    vals, times = [], []
    for k in range(args.steps):
        v, dt, _ = cpu_baseline(w, sample, cores, first=0)
        vals.append(v); times.append(dt)
    value = float(np.mean(vals)) if vals else 0.0
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * float(np.mean(times)) if times else None, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u64 (BN254 Fr, 4x64-bit Montgomery limbs)", "data": "synthetic",
        "config": make_config(w, lay, per_gpu_nominal),
        "sample_instances": sample,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{sample} of {w.n_instances} instances of {w.name} per step, oracle/h2sha_oracle.c on {cores} threads"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def measure_full(ctx, w, min_seconds=0.5, max_steps=64, mem_frac=0.6, split=True, verify=8, limit_instances=0, steps=0):
    """A WHOLE configuration (or, with limit_instances, its first instances) sharded by instance over the ranks and streamed through
    each GPU's HBM in chunks: a step = every instance of the shard generated once (the witness of a chunk is overwritten by the next
    chunk, as a prover that consumes chunk by chunk would allow; digests and per-instance checksums of all instances are kept).
    Times `steps` steps (0: >= min_seconds of them, at most max_steps) with CUDA events on the launching stream (max over ranks),
    samples clocks during them, then checks digests against hashlib, the last chunk's witness under the device-side MockProver pass and `verify` instances against the oracle."""
    import hashlib

    import torch
    pkg, S, sh, dist = ctx["pkg"], ctx["S"], ctx["sh"], ctx["dist"]
    rank, world, local_rank, dev = ctx["rank"], ctx["world"], ctx["local_rank"], ctx["dev"]
    cfg = pkg.Sha256DynamicConfig.configure(list(w.max_variable_byte_sizes), device=local_rank)
    lay = cfg.layout
    n_total = min(w.n_instances, limit_instances) if limit_instances else w.n_instances
    lo, hi = sh.shard_range(n_total, rank, world) if split else (rank * n_total, (rank + 1) * n_total)
    shard = hi - lo
    torch.cuda.empty_cache()
    free_b, _ = torch.cuda.mem_get_info(dev)
    cap = max(1, int(mem_frac * free_b) // lay.bytes_per_instance)
    n_chunks = (shard + cap - 1) // cap
    csz = (shard + n_chunks - 1) // n_chunks
    gate, lookup, spread = cfg.alloc_outputs(csz, zero=True)
    d_digests = torch.zeros((shard, 32), dtype=torch.uint8, device=dev)
    d_cks = torch.zeros((shard, 4), dtype=torch.int64, device=dev)
    chunks = []
    for c0 in range(0, shard, csz):
        n = min(csz, shard - c0)
        blob, offs, lens = S.generate(w, lo + c0, n)
        chunks.append((c0, n, torch.from_numpy(np.concatenate([blob, np.zeros(16, np.uint8)])).to(dev), int(blob.size), offs, lens))
    stream = torch.cuda.current_stream(dev); sp = stream.cuda_stream

    def step():
        for c0, n, d_blob, nbytes, offs, lens in chunks:
            cfg.digest_batch_raw(n, d_blob.data_ptr(), True, nbytes, offs, lens, None, gate_ptr=gate.data_ptr(), lookup_ptr=lookup.data_ptr(),
                                 spread_ptr=spread.data_ptr(), digests_dev_ptr=d_digests[c0:].data_ptr(), checksums_dev_ptr=d_cks[c0:].data_ptr(), stream=sp)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # one warm-up step, timed on the device to size the timed region
    w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    step(); stream.synchronize()
    w0.record(stream); step(); w1.record(stream); w1.synchronize()
    est_ms = max(w0.elapsed_time(w1), 1e-3)
    steps = steps or int(min(max_steps, max(1, np.ceil(min_seconds * 1e3 / est_ms))))
    if world > 1:
        t = torch.tensor([steps], dtype=torch.int64, device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); steps = int(t.item())
    barrier()
    sampler = ClockSampler(local_rank); sampler.start()
    t_warm = time.perf_counter()
    while time.perf_counter() - t_warm < 0.3:     # let the clock sampler see the load the steps are timed under
        step(); stream.synchronize()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(steps):
        step()
    ev1.record(stream)
    barrier()
    clocks = sampler.stop()
    t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    ms_per_step = total_ms / steps
    # ---- checks ----
    dig = d_digests.cpu().numpy()
    n_dig = 0
    for i in range(0, shard, max(1, shard // 128)):
        assert hashlib.sha256(S.message(w, lo + i)).digest() == bytes(dig[i]), f"digest mismatch at instance {lo + i}"
        n_dig += 1
    c0, n, d_blob, nbytes, offs, lens = chunks[-1]
    viol = cfg.check_batch(pkg.BatchResult(None, None, gate[:n], lookup[:n], spread[:n]), d_digests[c0:].data_ptr())
    assert sum(viol.values()) == 0, viol
    nv = min(verify, n)
    if nv:
        from oracle import oracle as O
        ocfg = O.OracleConfig(max_variable_byte_sizes=tuple(w.max_variable_byte_sizes))
        olay = O.Layout(lay.n_gate_cols, lay.gate_col_rows, lay.n_lookup_cols, lay.lookup_col_rows, lay.spread_rows)
        blob_h = d_blob.cpu().numpy()
        ref = O.batch_packed(ocfg, olay, nv, blob_h, offs[:nv], lens[:nv], np.zeros(nv, np.uint32), want_cells=True, n_threads=min(nv, os.cpu_count() or 1))
        assert (gate[:nv].cpu().numpy().view(np.uint64) == ref["gate"]).all() and (lookup[:nv].cpu().numpy().view(np.uint64) == ref["lookup"]).all()
        assert (spread[:nv].cpu().numpy().view(np.uint64) == ref["spread"]).all()
        assert (d_cks[c0:c0 + nv].cpu().numpy().view(np.uint64) == ref["checksums"]).all()
    _, _, job_ck = sh.gather_results(d_digests, d_cks, world)
    peak, peak_src = measured_peak_gbs()
    n_job = n_total if split else n_total * world
    blocks = n_job * lay.n_blocks
    value = blocks / (ms_per_step * 1e-3)
    gbs = n_job * lay.cells_per_instance * 32 / (ms_per_step * 1e-3) / 1e9 / world
    out = {"workload": f"{w.name}: {w.description}", "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "ms_per_step": ms_per_step,
           "timed_region_s": total_ms * 1e-3, "scaling": "strong" if split else "weak", "instances_total": n_job, "instances_per_gpu": shard,
           "chunks_per_gpu": n_chunks, "instances_per_chunk": csz, "blocks_per_instance": lay.n_blocks, "cells_per_instance": lay.cells_per_instance,
           "witness_bytes_total": n_job * lay.cells_per_instance * 32, "cells_per_s": value * lay.cells_per_instance / lay.n_blocks,
           "hbm_write_gbs_per_gpu": gbs, "frac_of_peak_per_gpu": gbs / peak, "peak_gbs": peak, "peak_source": peak_src, "clocks": clocks,
           "gpu_launches": 2 * n_chunks * steps,
           "checked": {"digests_vs_hashlib": n_dig, "device_mock_prover_instances": n, "violations": viol, "oracle_instances": nv},
           "job_checksum": job_ck}
    cfg.close()
    del gate, lookup, spread, d_digests, d_cks, chunks
    torch.cuda.empty_cache()
    return out


def measure_latency_cfg1(ctx):
    """Latency of ONE digest (BASELINE configs[0] and the reference's own bench shape, benches/digest.rs:102-129: `[0x01; 56]`,
    max_variable_byte_size 1024 -> 16 blocks, 9 gate columns): host message -> h2sha_digest_batch -> every cell in HBM, digest and
    checksums back on the host, host waits.  Wall clock per call (median / min of 200) and the device time of the two kernels."""
    import hashlib

    import torch
    pkg, local_rank, dev = ctx["pkg"], ctx["local_rank"], ctx["dev"]
    out = {}
    shapes = (("bench_shape_56B_max1024", [1024], b"\x01" * 56), ("cfg1_64B_max128", [128], bytes(range(64))))
    # block_parts = 0: the engine as the throughput runs configure it (3 jobs per compression); 24: the latency setting of
    # h2sha_config_t.block_parts (>= 12 cuts a compression into 8-instance jobs for as many SMs)
    for name, sizes, msg, parts in [(n_ + suffix, s_, m_, p_) for (n_, s_, m_) in shapes for (suffix, p_) in (("", 0), ("_latency_tuned", 24))]:
        cfg = pkg.Sha256DynamicConfig.configure(sizes, device=local_rank, block_parts=parts)
        lay = cfg.layout
        gate, lookup, spread = cfg.alloc_outputs(1, zero=True)
        blob, offs, lens = pkg.pack_messages([[msg]])
        h_blob = torch.from_numpy(np.concatenate([blob, np.zeros(16, np.uint8)])).pin_memory()
        hd = torch.zeros((1, 32), dtype=torch.uint8).pin_memory(); hc = torch.zeros((1, 4), dtype=torch.int64).pin_memory()
        stream = torch.cuda.current_stream(dev)

        def call(timed=False):
            cfg.digest_batch_raw(1, h_blob.data_ptr(), False, int(blob.size), offs, lens, None, gate_ptr=gate.data_ptr(), lookup_ptr=lookup.data_ptr(),
                                 spread_ptr=spread.data_ptr(), digests_host_ptr=hd.data_ptr(), checksums_host_ptr=hc.data_ptr(), stream=stream.cuda_stream,
                                 time_kernels=timed)
            stream.synchronize()

        for _ in range(20):
            call()
        ts = []
        for _ in range(200):
            t0 = time.perf_counter(); call(); ts.append(time.perf_counter() - t0)
        km = []
        for _ in range(20):
            call(timed=True); km.append(cfg.last_kernel_ms())
        assert bytes(hd.numpy()[0]) == hashlib.sha256(msg).digest()
        out[name] = {"wall_us_median": 1e6 * float(np.median(ts)), "wall_us_min": 1e6 * float(np.min(ts)), "k_trace_us": 1e3 * float(np.median([k[0] for k in km])),
                     "k_expand_us": 1e3 * float(np.median([k[1] for k in km])), "blocks": lay.n_blocks, "cells": lay.cells_per_instance,
                     "gate_columns": lay.n_gate_cols, "block_parts": parts or 3}
        cfg.close()
        del gate, lookup, spread
    out["note"] = ("one instance per call, host buffers in, digest + checksums out, host synchronises after every call (latency, not throughput); "
                   "small batches take the warp-per-message trace kernel; *_latency_tuned = an engine created with block_parts = 24")
    return out


def _gpu_context(args):
    """Process-wide setup shared by the bench modes: package, device, (for N > 1) the NCCL process group."""
    import torch
    import torch.distributed as dist

    import __graft_entry__ as ge
    ge.build()
    pkg = ge.load_package()
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL prints its version banner (NCCL_DEBUG=VERSION on these boxes) on stdout when the communicator is created:
        # send fd 1 to stderr while that happens so that stdout carries nothing but the one JSON line
        sys.stdout.flush(); saved_fd = os.dup(1); os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.all_reduce(torch.zeros(1, device=dev)); torch.cuda.synchronize()
        finally:
            sys.stdout.flush(); os.dup2(saved_fd, 1); os.close(saved_fd)
    return {"pkg": pkg, "S": ge.load_package_module("synthetic"), "sh": ge.load_package_module("sharding"), "dist": dist, "ge": ge,
            "rank": rank, "world": world, "local_rank": local_rank, "dev": dev}


def run_full_workload(args):
    """--full-workload: the WHOLE BASELINE configuration (all its instances, e.g. 2^16 x 5 blocks or 2^18 x 33 blocks), see measure_full."""
    ctx = _gpu_context(args)
    w = ctx["S"].WORKLOADS[args.workload]
    r = measure_full(ctx, w, steps=args.steps)
    if ctx["rank"] == 0:
        print(json.dumps({
            "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": ctx["world"], "steps": r["steps"], "warmup": 1, "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64 (BN254 Fr, 4x64-bit Montgomery limbs; u32 SHA-256 words)",
            "data": "synthetic",
            "config": {"workload": r["workload"] + " -- the whole configuration", "instances_total": r["instances_total"], "instances_per_gpu": r["instances_per_gpu"],
                       "chunks_per_gpu": r["chunks_per_gpu"], "instances_per_chunk": r["instances_per_chunk"], "blocks_per_instance": r["blocks_per_instance"],
                       "cells_per_instance": r["cells_per_instance"], "witness_bytes_total": r["witness_bytes_total"],
                       "l2": "every chunk writes far more than the 126 MB L2"},
            "cells_per_s": r["cells_per_s"], "clocks": r["clocks"], "gpu_launches": r["gpu_launches"],
            "roofline": {"bound": "hbm", "achieved": r["hbm_write_gbs_per_gpu"], "peak": r["peak_gbs"], "unit": "GB/s", "frac": r["frac_of_peak_per_gpu"], "traffic": None,
                         "kernel": "k_trace + k_expand (whole step)", "peak_source": r["peak_source"]},
            "checked": r["checked"], "job_checksum": r["job_checksum"]}), flush=True)
    if ctx["world"] > 1:
        ctx["dist"].destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2")
    ap.add_argument("--instances", type=int, default=0, help="instances per GPU per step (0 = workload default, capped by HBM)")
    ap.add_argument("--split-total", action="store_true",
                    help="divide the workload's instances over the ranks (rank r takes [r*n/N, (r+1)*n/N): strong scaling) instead of "
                         "one full-size shard per rank; e.g. --workload cfg4 --gpus 8 = 2^16 messages on 8 GPUs, 8192 each")
    ap.add_argument("--full-workload", action="store_true",
                    help="generate the WHOLE configuration (all instances, sharded over the ranks, streamed through HBM in chunks) "
                         "instead of one HBM-sized batch per step; e.g. --workload cfg5 = 2^18 messages x 33 blocks = 22.5 TB of witness")
    ap.add_argument("--launches-per-step", type=int, default=0,
                    help="passes over the batch per timed step (0 = as many as make one step take >= 30 ms)")
    ap.add_argument("--no-north-star", action="store_true", help="skip the north-star block (config 4 split over the ranks), the other configurations and the config-1 latency")
    ap.add_argument("--cpu-sample", type=int, default=1024, help="instances in the CPU-baseline sample")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-witness-d2h", action="store_true", help="skip the extra end-to-end leg that copies the whole witness to the host")
    ap.add_argument("--verify", type=int, default=8, help="instances per rank checked cell-for-cell against the oracle after timing")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed on rank 0 (digests, checksums, gate / lookup / spread "
                         "cells; a seeded sample of the larger ones) as DIR/<name>.npy in float32 / float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.full_workload):
        ap.error("--dump-outputs applies to the default GPU mode")

    if args.impl == "reference":
        run_reference(args)
        return
    if args.full_workload:
        run_full_workload(args)
        return

    import torch

    ctx = _gpu_context(args)
    pkg, S, ge, dist = ctx["pkg"], ctx["S"], ctx["ge"], ctx["dist"]
    rank, world, local_rank, dev = ctx["rank"], ctx["world"], ctx["local_rank"], ctx["dev"]

    w = S.WORKLOADS[args.workload]
    cfg = pkg.Sha256DynamicConfig.configure(list(w.max_variable_byte_sizes), device=local_rank)
    lay = cfg.layout
    # instances per GPU per launch: the whole workload if it fits in ~60% of free HBM, else a chunk (ring reuse)
    free_b, _ = torch.cuda.mem_get_info(dev)
    cap = max(1, int((0.75 if args.split_total else 0.6) * free_b) // lay.bytes_per_instance)
    if args.split_total:
        sh0 = ctx["sh"]
        if w.n_instances % world:
            raise SystemExit("--split-total needs the workload's instance count to be a multiple of the number of GPUs")
        lo, hi = sh0.shard_range(w.n_instances, rank, world)
        if hi - lo > cap:
            raise SystemExit(f"--split-total: {hi - lo} instances per GPU need {(hi - lo) * lay.bytes_per_instance / 1e9:.0f} GB, more than fits ({cap} instances)")
        per_gpu, first = hi - lo, lo
    else:
        per_gpu = args.instances or min(w.n_instances, cap)
        per_gpu = min(per_gpu, cap)
        first = rank * per_gpu
    blob, offs, lens = S.generate(w, first, per_gpu)
    n_msgs = per_gpu
    blocks_per_launch = per_gpu * lay.n_blocks

    gate, lookup, spread = cfg.alloc_outputs(per_gpu, zero=True)
    d_digests = torch.zeros((n_msgs, 32), dtype=torch.uint8, device=dev)
    d_cks = torch.zeros((per_gpu, 4), dtype=torch.int64, device=dev)
    h_blob = torch.from_numpy(np.concatenate([blob, np.zeros(16, np.uint8)])).pin_memory()
    RING = 3   # result buffers of the end-to-end leg: step k's digests + checksums are read by the host while steps k+1, k+2 are in flight
    h_digests = [torch.zeros((n_msgs, 32), dtype=torch.uint8).pin_memory() for _ in range(RING)]
    h_cks = [torch.zeros((per_gpu, 4), dtype=torch.int64).pin_memory() for _ in range(RING)]
    d_blob = h_blob.to(dev)
    stream = torch.cuda.current_stream(dev)
    sp = stream.cuda_stream

    def launch_resident(first_call=False, timed=False):
        cfg.digest_batch_raw(per_gpu, d_blob.data_ptr(), True, int(blob.size), offs, lens, None, gate_ptr=gate.data_ptr(),
                             lookup_ptr=lookup.data_ptr(), spread_ptr=spread.data_ptr(), digests_dev_ptr=d_digests.data_ptr(),
                             checksums_dev_ptr=d_cks.data_ptr(), stream=sp, reuse_inputs=not first_call, time_kernels=timed)

    def launch_e2e(slot):
        cfg.digest_batch_raw(per_gpu, h_blob.data_ptr(), False, int(blob.size), offs, lens, None, gate_ptr=gate.data_ptr(),
                             lookup_ptr=lookup.data_ptr(), spread_ptr=spread.data_ptr(), digests_host_ptr=h_digests[slot].data_ptr(),
                             checksums_host_ptr=h_cks[slot].data_ptr(), stream=sp)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- device-resident leg (`value`) ----
    launch_resident(first_call=True)
    for _ in range(max(args.warmup, 3)):
        launch_resident()
    stream.synchronize()
    # A step = L back-to-back passes of the hot path over the batch, L chosen so that one step takes >= ~30 ms (0.6 s for the default
    # 20 steps): a pass over the default batch takes under a millisecond on a B200, too short a window to time on its own
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record(stream)
    for _ in range(8):
        launch_resident()
    p1.record(stream); p1.synchronize()
    est_launch_ms = max(p0.elapsed_time(p1) / 8, 1e-3)
    L = args.launches_per_step or int(min(4096, max(1, np.ceil(30.0 / est_launch_ms))))
    if world > 1:
        t = torch.tensor([L], dtype=torch.int64, device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); L = int(t.item())
    blocks_per_step = L * blocks_per_launch
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    t_warm = time.perf_counter()
    while time.perf_counter() - t_warm < 0.3:   # let the sampler see this same load before, during and after the timed steps
        launch_resident()
    stream.synchronize()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kernel_ms = []
    ev0.record(stream)
    for _ in range(args.steps * L):
        launch_resident()
    ev1.record(stream)
    barrier()
    total_ms = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"digests": d_digests, "checksums": d_cks, "gate": gate, "lookup": lookup, "spread": spread})
    # per-kernel durations, measured live with CUDA events on the launching stream over the same launches (>= 0.5 s of them)
    t_loop = time.perf_counter()
    while len(kernel_ms) < args.steps or time.perf_counter() - t_loop < 0.5:
        launch_resident(timed=True)
        kernel_ms.append(cfg.last_kernel_ms())
    clocks = sampler.stop()
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    value = world * blocks_per_step / (ms_per_step * 1e-3)
    trace_ms = float(np.mean([k[0] for k in kernel_ms])); expand_ms = float(np.mean([k[1] for k in kernel_ms]))

    # ---- end-to-end leg through the public call with host buffers: every launch copies its messages from pinned host memory
    # (H2D inside h2sha_digest_batch) and delivers digests + checksums to host memory, which the host reads (a word of every
    # result) before that result buffer is reused RING launches later.  The call only enqueues, so the host runs ahead of the device.
    done = [torch.cuda.Event() for _ in range(RING)]
    sink = 0

    def e2e_launches(n):
        nonlocal sink
        for k in range(n):
            slot = k % RING
            if k >= RING:
                done[slot].synchronize()
                sink += int(h_cks[slot][0, 3]) + int(h_digests[slot][0, 0])
            launch_e2e(slot)
            done[slot].record(stream)
        for k in range(max(0, n - RING), n):
            done[k % RING].synchronize()
            sink += int(h_cks[k % RING][0, 3]) + int(h_digests[k % RING][0, 0])

    e2e_launches(2 * RING)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    t0 = time.perf_counter()
    e2e_launches(args.steps * L)
    e1.record(stream)
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    e2e_ms = max(e0.elapsed_time(e1), wall_ms)  # the slower of the device and wall clocks
    t = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * blocks_per_step / (float(t.item()) / args.steps * 1e-3)
    h2d = L * (int(blob.size) + offs.nbytes + lens.nbytes + 4 * n_msgs)
    d2h = L * (n_msgs * 32 + per_gpu * 32)

    # ---- extra datapoint: the same end-to-end launches with a host synchronisation after every one (what round 1 reported as e2e)
    e2e_sync = None
    if world == 1:
        n_s = min(args.steps * L, 200)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for k in range(n_s):
            launch_e2e(0); stream.synchronize()
        e2e_sync = {"value": n_s * blocks_per_launch / (time.perf_counter() - t0), "unit": UNIT, "launches": n_s,
                    "note": "as e2e, but the host waits for every launch before it issues the next (no overlap of the next batch's H2D + trace kernel)"}

    # ---- extra datapoint: the same end-to-end launches alternating TWO engine handles on two streams (round 1's way to hide the
    # per-call host wait; with the asynchronous call a single handle should now match it) ----
    e2e_two = None
    if world == 1 and per_gpu * lay.bytes_per_instance <= (8 << 30):
        try:
            cfg2_ = pkg.Sha256DynamicConfig.configure(list(w.max_variable_byte_sizes), device=local_rank)
            out2 = cfg2_.alloc_outputs(per_gpu, zero=True)
            s2 = torch.cuda.Stream(dev)
            hd2 = torch.zeros((n_msgs, 32), dtype=torch.uint8).pin_memory(); hc2 = torch.zeros((per_gpu, 4), dtype=torch.int64).pin_memory()
            lanes = [(cfg, (gate, lookup, spread), stream, h_digests[0], h_cks[0]), (cfg2_, out2, s2, hd2, hc2)]

            def step_lane(k):
                c_, o_, st_, hd_, hc_ = lanes[k & 1]
                st_.synchronize()      # the launch that used this lane before has delivered its digests + checksums
                c_.digest_batch_raw(per_gpu, h_blob.data_ptr(), False, int(blob.size), offs, lens, None, gate_ptr=o_[0].data_ptr(), lookup_ptr=o_[1].data_ptr(),
                                    spread_ptr=o_[2].data_ptr(), digests_host_ptr=hd_.data_ptr(), checksums_host_ptr=hc_.data_ptr(), stream=st_.cuda_stream)

            for k in range(4):
                step_lane(k)
            torch.cuda.synchronize(dev)
            n_two = min(args.steps * L, 400)
            t0 = time.perf_counter()
            for k in range(n_two):
                step_lane(k)
            torch.cuda.synchronize(dev)
            dt = time.perf_counter() - t0
            assert (hd2.numpy() == h_digests[0].numpy()).all() and (hc2.numpy() == h_cks[0].numpy()).all()
            e2e_two = {"value": n_two * blocks_per_launch / dt, "unit": UNIT, "launches": n_two, "note": "as e2e, two engine handles on two streams alternating (wall clock)"}
            cfg2_.close(); del out2
        except Exception as ex:
            e2e_two = {"error": str(ex)}

    # ---- extra datapoint: the same end-to-end launch when the consumer is a CPU prover, i.e. the whole witness is also copied
    # to pinned host memory every launch (PCIe-bound; single GPU and small batches only) ----
    e2e_witness = None
    witness_bytes = per_gpu * lay.bytes_per_instance
    if world == 1 and witness_bytes <= (4 << 30) and not args.no_witness_d2h:
        h_gate = torch.empty(gate.shape, dtype=gate.dtype).pin_memory()
        h_lookup = torch.empty(lookup.shape, dtype=lookup.dtype).pin_memory()
        h_spread = torch.empty(spread.shape, dtype=spread.dtype).pin_memory()

        def step_witness():
            launch_e2e(0)
            h_gate.copy_(gate, non_blocking=True); h_lookup.copy_(lookup, non_blocking=True); h_spread.copy_(spread, non_blocking=True)
            stream.synchronize()

        step_witness()
        n_w = 4
        t0 = time.perf_counter()
        for _ in range(n_w):
            step_witness()
        dt = (time.perf_counter() - t0) / n_w
        e2e_witness = {"value": blocks_per_launch / dt, "unit": UNIT, "d2h_bytes_per_launch": n_msgs * 32 + per_gpu * 32 + h_gate.nbytes + h_lookup.nbytes + h_spread.nbytes,
                       "launches": n_w, "note": "as e2e, plus every advice/lookup/spread column copied to pinned host memory each launch (what a CPU "
                                                 "prover would need); PCIe-bound, not the headline"}
        del h_gate, h_lookup, h_spread

    # ---- the same hand-off in its compact form: the launch writes only the dictionary of distinct values (27 % of the cells), that
    # is copied to pinned host memory, and the host rebuilds the columns with 32-byte copies (h2sha_expand_compact) ----
    e2e_compact = None
    if world == 1 and not args.no_witness_d2h:
        try:
            ci = cfg.compact_info()
            d_dict = torch.empty((per_gpu, ci["dict_cells_per_instance"], 4), dtype=torch.int64, device=dev)
            h_dict = torch.empty(d_dict.shape, dtype=torch.int64).pin_memory()

            def step_compact():
                cfg.digest_batch_raw(per_gpu, h_blob.data_ptr(), False, int(blob.size), offs, lens, None, digests_host_ptr=h_digests[0].data_ptr(),
                                     checksums_host_ptr=h_cks[0].data_ptr(), compact_dict_ptr=d_dict.data_ptr(), stream=sp)
                h_dict.copy_(d_dict, non_blocking=True)
                stream.synchronize()

            step_compact()
            n_c = 6
            t0 = time.perf_counter()
            for _ in range(n_c):
                step_compact()
            dt_wire = (time.perf_counter() - t0) / n_c
            assert (h_cks[0].numpy() == h_cks[1].numpy()).all(), "the compact launch changes the cell checksums"
            # host-side expansion into [instance][column][2^k] vectors (what halo2's prover holds), on a slice that fits in host memory
            k_rows = 1 << int(np.ceil(np.log2(max(lay.gate_col_rows, lay.lookup_col_rows, lay.spread_rows))))
            n_x = int(max(1, min(per_gpu, (3 << 30) // (cfg.n_columns() * k_rows * 32))))
            cores = os.cpu_count() or 1
            h_cols = np.zeros((n_x, cfg.n_columns(), k_rows, 4), dtype=np.uint64)
            cfg.expand_compact(h_dict[:n_x].numpy(), n_x, k_rows, out=h_cols, zero_fill=False)
            t0 = time.perf_counter()
            reps = 0
            while reps < 2 or time.perf_counter() - t0 < 1.0:
                cfg.expand_compact(h_dict[:n_x].numpy(), n_x, k_rows, out=h_cols, zero_fill=False); reps += 1
            dt_x = (time.perf_counter() - t0) / reps / n_x
            # bit-exactness of the whole chain on the slice: expander(dictionary) == the cells of the batch buffers
            gate_h = gate[:n_x].cpu().numpy().view(np.uint64)
            rg = min(k_rows, lay.gate_col_rows)
            assert (h_cols[:, : lay.n_gate_cols, :rg] == gate_h[:, :, :rg]).all(), "expander(compact) differs from the gate cells"
            e2e_compact = {"wire": {"value": blocks_per_launch / dt_wire, "unit": UNIT, "d2h_bytes_per_launch": n_msgs * 32 + per_gpu * 32 + h_dict.nbytes,
                                    "launches": n_c, "note": "host messages -> h2sha_digest_batch(compact_dict only) -> dictionary in pinned host memory"},
                           "expand_on_host": {"value": lay.n_blocks / dt_x, "unit": UNIT, "threads": cores, "instances": n_x, "rows_per_column": k_rows,
                                              "note": "h2sha_expand_compact: dictionary -> [instance][column][2^k] Fr vectors, 32-byte copies only"},
                           "dict_bytes_per_instance": ci["dict_bytes_per_instance"], "cell_bytes_per_instance": lay.cells_per_instance * 32,
                           "ratio": lay.cells_per_instance * 32 / ci["dict_bytes_per_instance"]}
            del d_dict, h_dict, h_cols
        except Exception as ex:
            e2e_compact = {"error": str(ex)}

    # ---- correctness inside the bench: digests vs hashlib for all, cells vs oracle on a sample, gather over NCCL ----
    import hashlib
    last = (args.steps * L - 1) % RING          # result buffers of the last end-to-end launch
    dig = h_digests[last].numpy()
    h_cks_last = h_cks[last]
    for i in range(0, per_gpu, max(1, per_gpu // 64)):
        m = bytes(blob[int(offs[i]):int(offs[i]) + int(lens[i])])
        assert hashlib.sha256(m).digest() == bytes(dig[i]), f"digest mismatch at instance {first + i}"
    verified = 0
    mock_prover_instances = 0
    if args.verify:
        from oracle import oracle as O
        ocfg = O.OracleConfig(max_variable_byte_sizes=tuple(w.max_variable_byte_sizes))
        olay = O.Layout(lay.n_gate_cols, lay.gate_col_rows, lay.n_lookup_cols, lay.lookup_col_rows, lay.spread_rows)
        nv = min(args.verify, per_gpu)
        ref = O.batch_packed(ocfg, olay, nv, np.concatenate([blob, np.zeros(1, np.uint8)]), offs[:nv], lens[:nv], np.zeros(nv, np.uint32),
                             want_cells=True, n_threads=min(nv, os.cpu_count() or 1))
        assert (gate[:nv].cpu().numpy().view(np.uint64) == ref["gate"]).all(), "gate cells differ from oracle"
        assert (lookup[:nv].cpu().numpy().view(np.uint64) == ref["lookup"]).all(), "lookup cells differ from oracle"
        assert (spread[:nv].cpu().numpy().view(np.uint64) == ref["spread"]).all(), "spread cells differ from oracle"
        assert (h_cks_last.numpy().view(np.uint64)[:nv] == ref["checksums"]).all(), "checksums differ from oracle"
        for r_ in range(RING):
            assert (h_cks[r_].numpy() == h_cks_last.numpy()).all() and (h_digests[r_].numpy() == dig).all(), "end-to-end launches delivered different results"
        verified = nv
        # MockProver-style pass on one sampled instance of the GPU output with the product's own shape plan:
        # every gate, copy constraint, range / spread lookup, and the digest bytes (reference lib.rs:525-526)
        from oracle import mock_prover as MP
        shp_cfg = pkg.Sha256DynamicConfig.configure(list(w.max_variable_byte_sizes), device=-1, build_shape=True)
        sh, brk = shp_cfg.shape(), shp_cfg.breaks()
        i0 = nv - 1
        g = gate[i0].cpu().numpy().view(np.uint64); lk = lookup[i0].cpu().numpy().view(np.uint64); spc = spread[i0].cpu().numpy().view(np.uint64)
        ends = list(brk[1:]) + [lay.n_gate_cells]
        stream_cells = np.concatenate([g[c, : int(e_) - int(s_)] for c, (s_, e_) in enumerate(zip(brk, ends))])
        nc = lay.n_spread_cols // 2
        nl = np.arange(lay.n_spread_limbs)
        consts_mont = np.array([O.int_to_mont(int(a) | int(b_) << 64 | int(c) << 128 | int(d_) << 192) for a, b_, c, d_ in sh.fixed], dtype=np.uint64)
        msg0 = bytes(blob[int(offs[i0]):int(offs[i0]) + int(lens[i0])])
        MP.verify(gate=stream_cells, selectors=sh.selectors, breaks=brk, lookup_idx=sh.lookup_src, dense=spc[nl % nc, nl // nc],
                  spread=spc[nc + nl % nc, nl // nc], limb_gate_dense=sh.limb_dense_src, limb_gate_spread=sh.limb_spread_src, copies=sh.copies,
                  consts=consts_mont, lookup_bits=16, limb_bits=8, max_rows=(1 << 17) - 9, output_bytes_idx=[shp_cfg.handles(0).output_bytes],
                  expected_digests=[hashlib.sha256(msg0).digest()])
        assert (np.concatenate([lk[c] for c in range(lay.n_lookup_cols)])[: lay.n_lookup_cells] == stream_cells[sh.lookup_src]).all()
        mock_prover_instances = 1
    # MockProver-style check of EVERY instance of the step's output on the device (gates, copy constraints, both lookups,
    # digest bytes): h2sha_check_batch; all ranks, violations summed over the job
    res_all = pkg.BatchResult(None, None, gate, lookup, spread)
    t_chk = time.perf_counter()
    viol = cfg.check_batch(res_all, d_digests.data_ptr())
    t_chk = time.perf_counter() - t_chk
    vt = torch.tensor([viol[k] for k in ("gates", "copies", "range_lookups", "spread_lookups", "digest_bytes")], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(vt)
    device_check = {"instances": world * per_gpu, "violations": dict(zip(("gates", "copies", "range_lookups", "spread_lookups", "digest_bytes"), vt.tolist())),
                    "seconds_rank0": t_chk, "note": "h2sha_check_batch: every gate, copy constraint, range / spread lookup and digest byte of every "
                                                    "instance, on the device (first call includes building the shape plan)"}
    assert int(vt.sum().item()) == 0, f"constraint violations in the generated witness: {device_check}"
    # the only collective: gather digests + checksums (64 B / instance) after the hot path -- through the C-ABI
    # (h2sha_gather on an ncclComm_t created here from libnccl; torch.distributed only ships the 128-byte unique id), cross-checked
    # against torch.distributed.all_gather
    sh = ctx["sh"]
    _, cks_t, job_ck = sh.gather_results(d_digests, d_cks, world)
    collective = "none (1 GPU)"
    if world > 1:
        all_d, all_c, job_ck_abi = sh.gather_results_cabi(pkg, d_digests, d_cks, rank, world, stream)
        assert job_ck_abi == job_ck and torch.equal(all_c, cks_t), "h2sha_gather and torch.distributed.all_gather disagree"
        collective = "h2sha_gather (ncclAllGather through the C-ABI), cross-checked against torch.distributed.all_gather"

    # ---- reference points for the roofline, measured live on this GPU (rank 0): (a) the plainest writer of incompressible
    # cells (coalesced 256-bit stores, nothing else) over a buffer larger than L2, (b) k_expand timed alone after an idle
    # gap (burst clocks; the figures above are from back-to-back launches under the power cap) ----
    store_ceiling = None
    int_ceiling = None
    burst_ms = None
    if rank == 0:
        try:
            free_now, _ = torch.cuda.mem_get_info(dev)
            pb = int(min(4 << 30, free_now // 2)) // 4096 * 4096
            probe = torch.empty(pb, dtype=torch.uint8, device=dev)
            ts = []
            for _ in range(6):
                a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a_.record(stream); cfg.store_probe(probe.data_ptr(), pb, sp); b_.record(stream); b_.synchronize()
                ts.append(a_.elapsed_time(b_))
            # the same writer back to back for ~1.5 s (the power-capped regime the timed steps run in), then 10 timed launches
            t_s = time.perf_counter()
            while time.perf_counter() - t_s < 1.5:
                for _ in range(20):
                    cfg.store_probe(probe.data_ptr(), pb, sp)
                stream.synchronize()
            a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a_.record(stream)
            for _ in range(10):
                cfg.store_probe(probe.data_ptr(), pb, sp)
            b_.record(stream); b_.synchronize()
            store_ceiling = {"gbs": pb / (min(ts[1:]) * 1e-3) / 1e9, "gbs_sustained": 10 * pb / (a_.elapsed_time(b_) * 1e-3) / 1e9, "bytes": pb,
                             "how": "k_store_probe: coalesced st.global.v8.b32 of incompressible 32-byte cells; gbs = best of 5 single launches, "
                                    "gbs_sustained = 10 launches after 1.5 s of back-to-back launches"}
            del probe
            # (a') integer-ALU ceiling: IMAD/LOP3 dependency chains, no memory traffic
            scratch = torch.zeros(148 * 8 * 256 * 2, dtype=torch.int32, device=dev)
            ti = []
            for _ in range(4):
                a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a_.record(stream); n_int = cfg.int_probe(scratch.data_ptr(), 1 << 14, sp); b_.record(stream); b_.synchronize()
                ti.append(a_.elapsed_time(b_))
            int_ceiling = {"ginst_s": n_int / (min(ti[1:]) * 1e-3) / 1e9, "how": "k_int_probe: 8 independent IMAD+LOP3 chains per thread, 8 CTAs x 256 threads per SM, best of 3"}
            time.sleep(0.5)
            bm = []
            for _ in range(3):
                launch_resident(timed=True)
                bm.append(cfg.last_kernel_ms()[1])
                time.sleep(0.2)
            burst_ms = min(bm)
        except Exception as ex:   # measurement extras must not take the bench line down
            store_ceiling = {"error": str(ex)}

    # ---- extra datapoint: lookup-argument pre-work on the witness that is in HBM (not part of `value`): multiplicities of
    # every instance of the step, permuted (A', S') pairs of a 64-instance slice (64 B written per usable row) ----
    prework = None
    if rank == 0:
        try:
            usable = (1 << 17) - 6
            info = cfg.lookup_info()
            res_view = pkg.BatchResult(None, None, gate, lookup, spread)
            if usable >= info["min_usable_rows"]:
                n_mult = min(per_gpu, 4096)
                rv = pkg.BatchResult(None, None, gate[:n_mult], lookup[:n_mult], spread[:n_mult])
                tm = []
                for _ in range(4):
                    a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a_.record(stream); mult, bad = cfg.lookup_multiplicities(rv, usable); b_.record(stream); b_.synchronize()
                    tm.append(a_.elapsed_time(b_))
                assert bad == 0, "witness cells outside the lookup tables"
                # the same multiplicities counted by the expansion kernel itself while it writes the cells (no second pass over HBM)
                fused = torch.empty_like(mult); fbad = torch.zeros(1, dtype=torch.int32, device=dev)
                tf, tplain = [], []
                for _ in range(6):
                    cfg.digest_batch_raw(n_mult, d_blob.data_ptr(), True, int(blob.size), offs, lens, None, gate_ptr=gate.data_ptr(), lookup_ptr=lookup.data_ptr(),
                                         spread_ptr=spread.data_ptr(), lookup_mult_ptr=fused.data_ptr(), mult_usable_rows=usable, mult_bad_ptr=fbad.data_ptr(),
                                         stream=sp, time_kernels=True)
                    tf.append(cfg.last_kernel_ms()[1])
                    cfg.digest_batch_raw(n_mult, d_blob.data_ptr(), True, int(blob.size), offs, lens, None, gate_ptr=gate.data_ptr(), lookup_ptr=lookup.data_ptr(),
                                         spread_ptr=spread.data_ptr(), stream=sp, time_kernels=True)
                    tplain.append(cfg.last_kernel_ms()[1])
                assert torch.equal(fused, mult) and int(fbad.item()) == 0, "fused multiplicities differ from the second pass"
                fused_extra_ms = float(np.median(tf[1:]) - np.median(tplain[1:]))
                # permuted (A', S') pairs: 64 B written per usable row and instance; outputs preallocated, the C-ABI call timed with CUDA events
                # (range lookup = lookup 0; the first spread lookup needs a theta: any reduced field element serves for timing)
                import ctypes as C_
                Lc = pkg.load_library()
                n_perm = int(min(n_mult, 256, int(0.25 * torch.cuda.mem_get_info(dev)[0]) // (2 * usable * 32)))
                pa = torch.empty((n_perm, usable, 4), dtype=torch.int64, device=dev); ps = torch.empty_like(pa)
                theta = np.array([3, 5, 7, 11], dtype=np.uint64)
                perm_ms = {}
                for name, lidx, th in (("range", 0, None), ("spread", info["n_range_lookups"], theta.ctypes.data)):
                    tp = []
                    for _ in range(4):
                        a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        a_.record(stream)
                        rc_ = Lc.h2sha_permute_lookup(cfg._h, n_perm, lidx, C_.c_void_p(mult.data_ptr()), usable, C_.c_void_p(th), C_.c_void_p(pa.data_ptr()),
                                                      C_.c_void_p(ps.data_ptr()), None, C_.c_void_p(sp))
                        b_.record(stream); b_.synchronize()
                        assert rc_ == 0, Lc.h2sha_last_error().decode()
                        tp.append(a_.elapsed_time(b_))
                    perm_ms[name] = min(tp[1:])
                # the same permuted pair without any dense multiplicity array: k_expand leaves the raw value lists (keep_lookup_raw), the
                # permutation bins the one lookup it needs on the fly
                traw = []
                for _ in range(6):
                    cfg.digest_batch_raw(n_mult, d_blob.data_ptr(), True, int(blob.size), offs, lens, None, gate_ptr=gate.data_ptr(), lookup_ptr=lookup.data_ptr(),
                                         spread_ptr=spread.data_ptr(), keep_lookup_raw=True, stream=sp, time_kernels=True)
                    traw.append(cfg.last_kernel_ms()[1])
                raw_extra_ms = float(np.median(traw[1:]) - np.median(tplain[1:]))
                pa2 = torch.empty_like(pa); ps2 = torch.empty_like(ps)
                tp = []
                for _ in range(4):
                    a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a_.record(stream)
                    rc_ = Lc.h2sha_permute_lookup_from_raw(cfg._h, 0, n_perm, 0, usable, None, C_.c_void_p(pa2.data_ptr()), C_.c_void_p(ps2.data_ptr()), None, C_.c_void_p(sp))
                    b_.record(stream); b_.synchronize()
                    assert rc_ == 0, Lc.h2sha_last_error().decode()
                    tp.append(a_.elapsed_time(b_))
                rc_ = Lc.h2sha_permute_lookup(cfg._h, n_perm, 0, C_.c_void_p(mult.data_ptr()), usable, None, C_.c_void_p(pa.data_ptr()), C_.c_void_p(ps.data_ptr()), None, C_.c_void_p(sp))
                assert rc_ == 0 and torch.equal(pa, pa2) and torch.equal(ps, ps2), "permuted pair from the raw lists differs"
                perm_ms["range_from_raw"] = min(tp[1:])
                del pa2, ps2
                read_b = n_mult * (lay.n_lookup_cells + 2 * lay.n_spread_limbs) * 32
                prework = {"usable_rows": usable, "multiplicities_fused_extra_ms": fused_extra_ms, "k_expand_with_multiplicities_ms": float(np.median(tf[1:])),
                           "k_expand_plain_ms": float(np.median(tplain[1:])),
                           "multiplicities_second_pass_ms": min(tm[1:]), "multiplicities_instances": n_mult,
                           "multiplicities_second_pass_read_gbs": read_b / (min(tm[1:]) * 1e-3) / 1e9,
                           "permute_instances": n_perm,
                           "permute_range_lookup_ms": perm_ms["range"], "permute_range_write_gbs": n_perm * usable * 64 / (perm_ms["range"] * 1e-3) / 1e9,
                           "permute_spread_lookup_ms": perm_ms["spread"], "permute_spread_write_gbs": n_perm * usable * 64 / (perm_ms["spread"] * 1e-3) / 1e9,
                           "raw_lists_extra_ms": raw_extra_ms, "permute_range_from_raw_ms": perm_ms["range_from_raw"],
                           "permute_range_from_raw_write_gbs": n_perm * usable * 64 / (perm_ms["range_from_raw"] * 1e-3) / 1e9,
                           "note": "multiplicities: fused = counted by k_expand while it writes the cells (+ k_mult_from_raw), second pass = h2sha_lookup_multiplicities over the witness in HBM "
                                   "(incl. its memset and the allocation of the output); permute = h2sha_permute_lookup (scan + fill kernels) into preallocated outputs, CUDA events; "
                                   "raw lists = keep_lookup_raw (no dense multiplicities at all) + h2sha_permute_lookup_from_raw, output checked equal"}
                del mult, pa, ps, fused
            del res_view
        except Exception as ex:
            prework = {"error": str(ex)}

    # ---- the north-star run and the other named configurations, measured in this same process ----
    north_star = other_configs = latency_cfg1 = None
    if not args.no_north_star:
        cfg.close()
        del gate, lookup, spread, d_digests, d_cks, res_all
        torch.cuda.empty_cache()
        # BASELINE config 4: 2^16 256-byte messages (5 blocks each, 853 GB of witness) split by instance over the N ranks; each rank
        # streams its shard through HBM in chunks when it does not fit
        north_star = measure_full(ctx, S.WORKLOADS["cfg4"], min_seconds=0.6, max_steps=64, mem_frac=0.6, split=True, verify=4)
        north_star["note"] = ("BASELINE.json configs[3] / north_star: 2^16 instances of 256-byte messages sharded by instance across the ranks "
                              "(strong scaling: the job is fixed, N GPUs share it); value = whole-job blocks/s, max over ranks, >= 0.5 s timed")
        if world == 1:
            other_configs = {}
            for name, lim in (("cfg3", 1024), ("cfg5", 512)):
                try:
                    r_ = measure_full(ctx, S.WORKLOADS[name], min_seconds=0.6, max_steps=96, mem_frac=0.5, split=True, verify=2, limit_instances=lim)
                    r_["note"] = f"the first {lim} instances of the configuration (one HBM-sized shard); the whole configuration: bench.py --workload {name} --full-workload"
                    other_configs[name] = r_
                except Exception as ex:
                    other_configs[name] = {"error": str(ex)}
            try:
                latency_cfg1 = measure_latency_cfg1(ctx)
            except Exception as ex:
                latency_cfg1 = {"error": str(ex)}

    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        traffic = None   # dram__bytes_read + dram__bytes_write of one k_expand launch, from the committed ncu capture of this workload
        int_insts = None  # thread-level integer instructions of one k_expand launch, same capture
        try:
            with open(os.path.join(ROOT, "profiles", "k_expand_traffic.json")) as f:
                tj = json.load(f)
            if tj["workload"] == w.name and tj["instances_per_launch"] == per_gpu:
                traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
                int_insts = tj.get("int_thread_insts")
        except Exception:
            pass
        int_roof = None
        if int_insts and int_ceiling and "ginst_s" in int_ceiling:
            ach = int_insts / (expand_ms * 1e-3) / 1e9
            int_roof = {"achieved": ach, "peak": int_ceiling["ginst_s"], "unit": "Ginst/s (thread-level integer instructions)", "frac": ach / int_ceiling["ginst_s"],
                        "instructions_per_launch": int_insts, "peak_source": int_ceiling["how"],
                        "note": "the other roofline the north star names; HBM write is the slower (binding) one"}
        alg_bytes = per_gpu * lay.cells_per_instance * 32
        achieved = alg_bytes / (expand_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if args.split_total else "weak", "vs_baseline": None,
            "dtype": "u64 (BN254 Fr, 4x64-bit Montgomery limbs; u32 SHA-256 words)", "data": "synthetic",
            "config": make_config(w, lay, per_gpu),
            "launches_per_step": L, "ms_per_launch": ms_per_step / L, "timed_region_s": total_ms * 1e-3,
            "cells_per_s": value * lay.cells_per_instance / lay.n_blocks,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "note": f"every launch: pinned host message buffer -> h2sha_digest_batch (H2D inside) -> digests + checksums in host memory, read by the host "
                            f"before the result buffer is reused {RING} launches later; one engine handle, one stream; the call only enqueues, so the next batch's "
                            "H2D copy and trace kernel overlap this batch's expansion.  The witness stays in HBM for a device-side prover "
                            "(e2e_witness_to_host: what a CPU prover sees)"},
            "e2e_sync_every_launch": e2e_sync,
            "e2e_two_handles": e2e_two,
            "e2e_witness_to_host": e2e_witness,
            "e2e_witness_to_host_compact": e2e_compact,
            "gpu_launches": 2 * args.steps * L,
            "kernels_ms": {"k_trace": trace_ms, "k_expand": expand_ms},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "kernel": "k_expand", "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg_bytes,
                         "store_ceiling": store_ceiling,
                         "frac_of_store_ceiling": (achieved / store_ceiling["gbs"]) if store_ceiling and "gbs" in store_ceiling else None,
                         "frac_of_sustained_store_ceiling": (achieved / store_ceiling["gbs_sustained"]) if store_ceiling and "gbs_sustained" in store_ceiling else None,
                         "int_alu": int_roof,
                         "k_expand_burst_ms": burst_ms,
                         "achieved_burst": (alg_bytes / (burst_ms * 1e-3) / 1e9) if burst_ms else None},
            "lookup_prework": prework,
            "device_mock_prover": device_check,
            "verified_instances_vs_oracle": verified, "mock_prover_instances": mock_prover_instances, "job_checksum": job_ck,
            "collective": collective,
            "north_star": north_star, "other_configs": other_configs, "latency_cfg1": latency_cfg1,
        }
        if not args.no_cpu:
            cores = os.cpu_count() or 1
            sample = min(w.n_instances, args.cpu_sample)
            # bounded sample: repeat it until ~12 s of CPU work (cores x wall) have been timed
            reps, wall, blocks = 0, 0.0, 0
            while reps < 1 or (wall * cores < 12.0 and reps < 64):
                _, dt, _ = cpu_baseline(w, sample, cores)
                wall += dt; blocks += sample * w.blocks_per_instance; reps += 1
            line["cpu_baseline"] = {"value": blocks / wall, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": f"{reps} x {sample} instances of {w.name} ({blocks} blocks, {wall:.1f} s wall = {wall * cores:.0f} core-seconds), "
                                              f"oracle/h2sha_oracle.c (C restatement; the Rust crate cannot be built here) on {cores} threads"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    sys.dont_write_bytecode = True   # the bench writes nothing into the tree it runs from (which may be read-only)
    main()
