"""bench.py contract checks on the CPU: the JSON line, and the N>1 launch path under torchrun with gloo (world size 2).

The kernels run through the test-only emulation build (DOT_RING_B200_BENCH_DRYRUN=1); the line is marked `dry_run`
and is never a measurement.  The real bench refuses a non-CUDA library."""

import hashlib
import json
import os
import random
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
KA1_ROOT_SHA256_PREFIX = "963f1e262eba87d5"  # ring 1023 root of the unmodified reference (tests/golden/ring1023_reference.json)

REQUIRED = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
            "config", "e2e", "gpu_launches", "clocks", "roofline"]  # fmt: skip


def _start(cmd):
    env = dict(os.environ, DOT_RING_B200_BENCH_DRYRUN="1")
    return subprocess.Popen(cmd, cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)


def _finish(proc, timeout=1500):
    out, err = proc.communicate(timeout=timeout)
    assert proc.returncode == 0, err[-2000:]
    lines = [ln for ln in out.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, out
    return json.loads(lines[0]), err


def _last_proof_sha(err):
    """The prefix of sha256(last proof of the last timed step) that bench.py prints on stderr."""
    shas = [ln.split()[-1] for ln in err.splitlines() if ln.startswith("[bench] last proof sha256 ")]
    assert len(shas) == 1, err[-2000:]
    return shas[0]


def _sha(row):
    return hashlib.sha256(row.astype(np.uint8).tobytes()).hexdigest()[:16]


def _check_line(line, n_gpus, total, steps, scaling):
    for key in REQUIRED:
        assert key in line, key
    assert line["metric"] == "ring_vrf_proofs_per_s" and line["unit"] == "proofs/s"
    assert line["n_gpus"] == n_gpus and line["steps"] == steps and line["scaling"] == scaling
    assert len(line["step_ms_rank0"]) == steps
    parity = line["config"]["parity"]
    assert parity["ring_root_sha256"] == KA1_ROOT_SHA256_PREFIX and parity["equal"] is True and parity["golden_proofs"] == 2 and parity["verified_sample"] >= 1
    assert line["config"]["total_proofs_per_step"] == total
    assert abs(line["value"] * line["ms_per_step"] * 1e-3 - total) < 1e-6 * total
    assert line["gpu_launches"] > 0
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic", "algorithmic_reduction"} <= set(line["roofline"])
    assert 0 < line["roofline"]["frac"] < 1.2 and line["roofline"]["kernel_launches_per_step"] == 3
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(line["e2e"])
    assert line["e2e"]["value"] <= line["value"] * 1.001


def _dumped(out_dir, name, indices):
    proofs, index = np.load(out_dir / f"{name}.npy"), np.load(out_dir / f"{name}_index.npy")
    assert proofs.dtype == np.float32 and proofs.shape == (len(indices), 784)
    assert index.dtype == np.float64 and index.tolist() == indices
    assert np.array_equal(proofs, np.round(proofs)) and proofs.min() >= 0 and proofs.max() <= 255
    return proofs


def test_bench_lines_dry_run(tmp_path):
    """The three launch modes of bench.py, run side by side (each builds an emulated 6145-point window table, ~1.5 minutes):
    one process / one device (weak, --batch), torchrun with two gloo ranks (strong: one batch of 3 proofs sharded 2 + 1), and
    one process driving two emulated devices through EnginePool (strong).  Each dumps the proofs of its last timed step."""
    single = _start([sys.executable, "bench.py", "--steps", "2", "--warmup", "1", "--batch", "1", "--window-bits", "4", "--no-cpu-baseline",
                     "--dump-outputs", str(tmp_path / "single")])  # fmt: skip
    ranks = _start([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", "29617",
                    "bench.py", "--gpus", "2", "--steps", "1", "--warmup", "1", "--total", "3", "--window-bits", "4", "--dump-outputs", str(tmp_path / "ranks")])  # fmt: skip
    pool = _start([sys.executable, "bench.py", "--gpus", "2", "--steps", "1", "--warmup", "1", "--total", "2", "--window-bits", "4",
                   "--dump-outputs", str(tmp_path / "pool")])  # fmt: skip
    line, err = _finish(single)
    _check_line(line, 1, 1, 2, "weak")
    assert _sha(_dumped(tmp_path / "single", "proofs", [0])[-1]) == _last_proof_sha(err)
    line, err = _finish(ranks)
    _check_line(line, 2, 3, 1, "strong")
    assert line["config"]["launch"].startswith("torchrun")
    assert "cpu_baseline" not in line  # rank 0 at N=1 only
    rank0 = _dumped(tmp_path / "ranks", "proofs_rank0", [0, 1])
    _dumped(tmp_path / "ranks", "proofs_rank1", [2])
    assert _sha(rank0[-1]) == _last_proof_sha(err)  # only rank 0 prints its last proof
    line, err = _finish(pool)
    _check_line(line, 2, 2, 1, "strong")
    assert "EnginePool" in line["config"]["launch"]
    # proofs 0 and 1 of step 0 have the same inputs in both strong-scaling runs, whichever way the batch is split
    pool_rows = _dumped(tmp_path / "pool", "proofs", [0, 1])
    assert _sha(pool_rows[-1]) == _last_proof_sha(err)
    assert np.array_equal(pool_rows, rank0)


def test_dump_outputs_shares_the_limit_over_ranks_and_samples_with_a_fixed_seed(tmp_path):
    import bench

    rng = random.Random(5)
    proofs = [bytes(rng.randrange(256) for _ in range(784)) for _ in range(40)]
    limit = 2 * (bench.NPY_HEADERS_BYTES + 10 * (784 * 4 + 8))  # room for 10 rows per rank at world size 2
    shards = ((0, 25), (25, 40))
    for rank, (lo, hi) in enumerate(shards):
        bench.dump_outputs(tmp_path / "ranks", proofs[lo:hi], lo, f"proofs_rank{rank}", 2, limit)
    assert sum(f.stat().st_size for f in (tmp_path / "ranks").iterdir()) <= limit
    for rank, (lo, hi) in enumerate(shards):
        rows = np.load(tmp_path / "ranks" / f"proofs_rank{rank}.npy")
        index = np.load(tmp_path / "ranks" / f"proofs_rank{rank}_index.npy")
        assert rows.dtype == np.float32 and rows.shape == (10, 784) and index.shape == (10,)
        assert np.all(np.diff(index) > 0) and lo <= index[0] and index[-1] < hi
        assert [r.astype(np.uint8).tobytes() for r in rows] == [proofs[int(i)] for i in index]
    bench.dump_outputs(tmp_path / "again", proofs[:25], 0, "proofs_rank0", 2, limit)
    assert np.array_equal(np.load(tmp_path / "again" / "proofs_rank0_index.npy"), np.load(tmp_path / "ranks" / "proofs_rank0_index.npy"))
    # within its share a rank writes every row, in batch order
    bench.dump_outputs(tmp_path / "all", proofs[:10], 7, "proofs", 1, limit)
    assert np.load(tmp_path / "all" / "proofs_index.npy").tolist() == list(range(7, 17))
    assert [r.astype(np.uint8).tobytes() for r in np.load(tmp_path / "all" / "proofs.npy")] == proofs[:10]


def test_bench_refuses_zero_steps():
    out = subprocess.run([sys.executable, "bench.py", "--steps", "0"], cwd=ROOT, capture_output=True, text=True, timeout=60)
    assert out.returncode == 2 and "--steps" in out.stderr


def test_bench_refuses_cpu_library_without_dryrun():
    """Without a usable CUDA device (none visible here) the real bench exits with an error and prints no line: it never
    falls back to the CPU emulation build, which only DOT_RING_B200_BENCH_DRYRUN=1 selects."""
    env = {k: v for k, v in os.environ.items() if k != "DOT_RING_B200_BENCH_DRYRUN"}
    env["CUDA_VISIBLE_DEVICES"] = ""  # no usable GPU, also on a machine that has one
    out = subprocess.run([sys.executable, "bench.py", "--steps", "1", "--warmup", "0", "--batch", "1"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode != 0 and "{" not in out.stdout  # the product path must fail loudly, not fall back
