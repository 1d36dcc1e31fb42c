"""CPU checks of bench.py's host logic: the shard layouts its ring-parity protocol uses are the reference's
(test/test_burst.py:44-58, via the oracle), the FLOP counts are the ones SURVEY.md 8(d) states, the ncu-traffic
lookup never invents a number, and the reference arm prints a well-formed line without a GPU."""
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from oracle import attention_oracle as orc  # noqa: E402


def test_bench_shards_match_the_reference_layouts():
    t = torch.arange(2 * 48 * 3 * 4, dtype=torch.float32).reshape(2, 48, 3, 4)
    for world in (1, 2, 4):
        for layout in ("contiguous", "zigzag", "striped"):
            for rank in range(world):
                assert torch.equal(bench._shard(t, rank, world, layout), orc.shard(t, rank, world, layout)), (world, layout)


def test_flop_counts_are_surveys():
    assert abs(bench.flops(262144, "fwd") - 1.1259e15) / 1.1259e15 < 1e-3
    assert abs(bench.flops(262144, "fwd_bwd") - 3.9406e15) / 3.9406e15 < 1e-3
    assert abs(bench.flops(65536, "fwd") - 7.037e13) / 7.037e13 < 1e-3


def test_traffic_lookup_is_a_table_not_a_literal():
    assert bench.ncu_traffic("bwd_chunk_kernel", 12345, 678, 9, False) == (None, None)
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(path):
        tab = json.load(open(path))
        key = next(iter(tab))
        kern, sq, sk, hh, c = key.split(":")
        got, src = bench.ncu_traffic(kern, int(sq[3:]), int(sk[3:]), int(hh[2:]), bool(int(c[-1])))
        assert got == tab[key]["dram_bytes"] and src == tab[key]["source"]


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ, RANK="0")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                          "--warmup", "0"], capture_output=True, text=True, timeout=600, env=env)
    assert res.returncode == 0, res.stderr[-2000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["value"] > 0 and line["unit"] == "TFLOPS/s"
    assert line["steps"] == 2
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0
    # non-zero ranks of a torchrun launch exit without work
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference"],
                         capture_output=True, text=True, timeout=120, env=dict(os.environ, RANK="1"))
    assert res.returncode == 0 and res.stdout.strip() == ""


def test_dump_outputs_is_a_fixed_float32_sample_within_64_mb(tmp_path):
    import numpy as np
    S_loc, Hh, Dd = 4096, 2, 8
    outs = [torch.randn(1, S_loc, Hh, Dd).to(torch.bfloat16) for _ in range(4)]
    full = [t.float() for t in outs]
    bench.dump_outputs(str(tmp_path / "a"), outs, 0, 1)
    bench.dump_outputs(str(tmp_path / "b"), outs, 0, 1)
    rows = None
    for name, ref in zip(("o", "dq", "dk", "dv"), full):
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype == np.float32 and a.shape == (1, bench.DUMP_ROWS, Hh, Dd) and np.array_equal(a, b)
        # every dumped row is a row of the output, at the same positions in every output
        hit = [int(torch.nonzero((ref[0] == torch.from_numpy(r)).all(-1).all(-1))[0]) for r in a[0]]
        assert rows is None or hit == rows
        rows = hit
    assert rows == sorted(set(rows))
    assert 4 * bench.DUMP_ROWS * bench.H * bench.D * 4 <= 64 << 20
    bench.dump_outputs(str(tmp_path / "r"), outs, 1, 4)  # per-rank files, the row budget shared by the ranks
    assert np.load(tmp_path / "r" / "dv_rank1.npy").shape == (1, bench.DUMP_ROWS // 4, Hh, Dd)


def test_argument_errors():
    for extra, msg in ((["--steps", "0"], "--steps must be >= 1"),
                       (["--dump-outputs", "d", "--configs", "65536"], "not --configs"),
                       (["--dump-outputs", "d", "--impl", "reference"], "--impl reference")):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True,
                             text=True, timeout=120, cwd=ROOT)
        assert res.returncode == 2 and msg in res.stderr, (extra, res.stderr[-500:])


def test_default_ring_transport(monkeypatch):
    """copy engines when every rank of the job is on this node (torchrun's LOCAL_WORLD_SIZE == world size), NCCL
    otherwise; BA_RING_TRANSPORT always wins."""
    sys.path.insert(0, os.path.join(ROOT, "burst-attention_b200"))
    from burst_attn import comm
    monkeypatch.delenv("BA_RING_TRANSPORT", raising=False)
    for world, local, want in ((8, "8", "ce"), (8, "4", "nccl"), (8, None, "nccl"), (1, "1", "nccl"), (2, "x", "nccl")):
        monkeypatch.setattr(comm, "get_world_size", lambda g=None, w=world: w)
        if local is None:
            monkeypatch.delenv("LOCAL_WORLD_SIZE", raising=False)
        else:
            monkeypatch.setenv("LOCAL_WORLD_SIZE", local)
        assert comm.default_transport() == want, (world, local)
    monkeypatch.setenv("BA_RING_TRANSPORT", "nccl")
    monkeypatch.setenv("LOCAL_WORLD_SIZE", "8")
    assert comm.default_transport() == "nccl"
