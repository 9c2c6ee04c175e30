"""bench.py --dump-outputs writes the compressed stream of the last timed step as float32 .npy -- whole when it is short, the
bytes at a fixed seeded set of positions when it is long, at most 64 MB over all ranks -- so that the outputs of two builds can
be compared array for array."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_short_stream_is_whole(tmp_path):
    comp = torch.arange(1000).remainder(256).to(torch.uint8)
    bench.dump_outputs(str(tmp_path), comp)
    a = np.load(tmp_path / "compressed.npy")
    assert a.dtype == np.float32 and np.array_equal(a, comp.numpy())
    size = np.load(tmp_path / "compressed_size.npy")
    assert size.dtype == np.float64 and size.tolist() == [1000.0]


def test_dump_outputs_long_stream_is_a_fixed_sample(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 64)
    comp = torch.arange(250).to(torch.uint8)  # byte p holds p: the sample shows the positions it was taken at
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), comp)
    a, b = (np.load(tmp_path / d / "compressed.npy") for d in ("a", "b"))
    assert a.dtype == np.float32 and a.shape == (64,) and np.array_equal(a, b)
    assert np.load(tmp_path / "a" / "compressed_size.npy").tolist() == [250.0]
    assert (np.diff(a) > 0).all() and 0 <= a[0] and a[-1] < 250  # distinct positions, in stream order
    assert a[-1] - a[0] > 125 and not np.array_equal(a, np.arange(64))  # spread over the stream, not its head


@pytest.mark.parametrize("world", [1, 2, 8])
def test_dump_outputs_stay_within_64_mb_over_all_ranks(tmp_path, world):
    comp = torch.from_numpy(np.random.default_rng(1).integers(0, 256, 9_000_000, dtype=np.uint8))  # > DUMP_MAX_BYTES
    for rank in range(world):
        bench.dump_outputs(str(tmp_path), comp, rank, world)
    names = sorted(os.listdir(tmp_path))
    assert len(names) == 2 * world
    if world > 1:
        assert all(n.startswith("rank") for n in names) and "rank%d_compressed.npy" % (world - 1) in names
    assert sum(os.path.getsize(tmp_path / n) for n in names) <= 64_000_000


def test_dump_outputs_refused_for_the_reference_arm(tmp_path):
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(out)],
                       capture_output=True, text=True)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr
    assert not out.exists()


@pytest.mark.gpu
def test_bench_dumps_the_stream_of_its_last_timed_step(tmp_path):
    """A short bench run: the dumped stream is the one the benchmark reports and decodes to the benchmark's input."""
    from oracle.harness import sys_decompress
    from tools import datagen
    nbytes = 2_000_000
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "1", "--bytes", str(nbytes),
                        "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    comp = np.load(tmp_path / "compressed.npy")
    assert np.load(tmp_path / "compressed_size.npy").tolist() == [float(line["compressed_bytes"])] == [float(comp.size)]
    assert comp.size < bench.DUMP_MAX_BYTES  # the whole stream, not a sample
    assert sys_decompress(comp.astype(np.uint8).tobytes(), nbytes) == datagen.enwik_like(nbytes, seed=8)
