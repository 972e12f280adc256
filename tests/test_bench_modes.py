"""bench.py's arms: the CPU reference arm prints its one JSON line without a GPU; on a GPU the whole-configuration mode
streams a configuration through HBM in chunks and checks what it produced."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, timeout=600):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=timeout, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    lines = [ln for ln in out.stdout.strip().splitlines() if ln.strip()]
    assert len(lines) == 1, f"stdout must be exactly one JSON line, got {len(lines)}"
    return json.loads(lines[0])


def test_reference_arm_prints_one_json_line():
    d = _run("--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-sample", "8")
    assert d["impl"] == "reference" and d["unit"] == "blocks/s" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["gpu_launches"] == 0


def _words(a):
    """float64 (low, high) 32-bit halves of a dump -> the uint64 words."""
    h = a.astype(np.uint64)
    return h[:, 0::2] | (h[:, 1::2] << np.uint64(32))


def test_dump_outputs_is_lossless_bounded_and_seeded(tmp_path):
    import torch

    import bench
    rng = np.random.default_rng(1)
    dig = rng.integers(0, 256, (5, 32), dtype=np.uint8)
    cks = rng.integers(-2**63, 2**63 - 1, (5, 4), dtype=np.int64)
    cells = rng.integers(-2**63, 2**63 - 1, (3, 2, 40000, 4), dtype=np.int64)     # 15 MB: more than one array may take
    arrays = {"digests": torch.from_numpy(dig), "checksums": torch.from_numpy(cks), "gate": torch.from_numpy(cells)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    names = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert names == ["checksums.npy", "digests.npy", "gate.npy", "gate_rows.npy"]
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b)
        assert (tmp_path / "a" / n).stat().st_size <= bench.DUMP_BYTES_PER_ARRAY + 1024
    assert np.array_equal(np.load(tmp_path / "a" / "digests.npy"), dig)
    assert np.array_equal(_words(np.load(tmp_path / "a" / "checksums.npy")), cks.view(np.uint64))
    rows = np.load(tmp_path / "a" / "gate_rows.npy").astype(np.int64)
    assert len(rows) == bench.DUMP_BYTES_PER_ARRAY // 72 and (np.diff(rows) > 0).all() and rows[-1] < 240000
    assert np.array_equal(_words(np.load(tmp_path / "a" / "gate.npy")), cells.reshape(-1, 4).view(np.uint64)[rows])


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(tmp_path):
    """Two runs with different step counts dump the same results; they are the digests of the workload's messages and the
    oracle's cells and checksums."""
    import hashlib

    import __graft_entry__ as ge
    from oracle import oracle as O
    quick = ("--warmup", "1", "--no-north-star", "--no-cpu", "--no-witness-d2h")
    d = _run("--steps", "3", *quick, "--dump-outputs", str(tmp_path / "a"))
    assert d["steps"] == 3 and d["gpu_launches"] == 2 * 3 * d["launches_per_step"]
    _run("--steps", "1", *quick, "--dump-outputs", str(tmp_path / "b"))
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert {"digests.npy", "checksums.npy", "gate.npy", "lookup.npy", "spread.npy"} <= set(files)
    assert sum((tmp_path / "a" / f).stat().st_size for f in files) <= 64 << 20
    for f in files:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)), f
    S = ge.load_package_module("synthetic")
    w = S.WORKLOADS["cfg2"]
    n = d["config"]["instances_per_gpu"]
    blob, offs, lens = S.generate(w, 0, n)
    dig = np.load(tmp_path / "a" / "digests.npy")
    assert dig.shape == (n, 32)
    for i in range(n):
        assert bytes(dig[i].astype(np.uint8)) == hashlib.sha256(bytes(blob[int(offs[i]):int(offs[i]) + int(lens[i])])).digest()
    # cells and checksums of the first instances against the oracle
    k = 4
    ocfg = O.OracleConfig(max_variable_byte_sizes=w.max_variable_byte_sizes)
    reg = O.synthesize(ocfg, [bytes(blob[: int(lens[0])])], record_shape=False)
    ref = O.batch_packed(ocfg, reg.layout(), k, np.concatenate([blob, np.zeros(1, np.uint8)]), offs[:k], lens[:k], np.zeros(k, np.uint32),
                         want_cells=True)
    assert np.array_equal(_words(np.load(tmp_path / "a" / "checksums.npy"))[:k], ref["checksums"])
    n_checked = 0
    for name in ("gate", "lookup", "spread"):
        got = _words(np.load(tmp_path / "a" / f"{name}.npy"))
        want = ref[name].reshape(-1, 4)                       # rows of the first k instances come first in the flattened output
        if f"{name}_rows.npy" in files:
            rows = np.load(tmp_path / "a" / f"{name}_rows.npy").astype(np.int64)
            sel = rows < len(want)
            got, want = got[sel], want[rows[sel]]
        else:
            got = got[: len(want)]
        assert len(got) and np.array_equal(got, want), name
        n_checked += len(got)
    assert n_checked > 100


@pytest.mark.gpu
def test_full_workload_mode_streams_config3_in_chunks():
    d = _run("--workload", "cfg3", "--full-workload", "--steps", "1")
    assert d["config"]["instances_total"] == 4096 and d["config"]["blocks_per_instance"] == 17
    assert d["config"]["chunks_per_gpu"] >= 2                      # 181 GB of witness do not fit in one pass
    assert sum(d["checked"]["violations"].values()) == 0 and d["checked"]["oracle_instances"] == 8
    assert d["value"] > 1e5 and 0 < d["roofline"]["frac"] < 1.2
