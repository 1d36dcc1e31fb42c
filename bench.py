#!/usr/bin/env python
"""bench.py -- attention TFLOPS/s (fwd+bwd, and fwd) at seq=262144, H=32, d=128, bf16,
bs=1 on N B200s (BASELINE.json metric), strong scaling: the global sequence is
fixed and sharded over the N ranks (contiguous shards, non-causal -- the C2/C3
configurations; N=1 is the local kernel with no ring).

  python bench.py --gpus N --steps K --warmup W            (N>1: launched under torchrun)
  python bench.py --impl reference ...                     CPU arm: the oracle port of the
                                                           reference's path on the host cores
  python bench.py ... --dump-outputs DIR                   also write a sample of what the last
                                                           timed step returned (dump_outputs)

One "step" = one forward + one backward of burst_attn_func on synthetic
N(0,1) bf16 inputs already resident in HBM (`value`), and the same through the
public API from pinned HOST buffers with the H2D/D2H copies inside the timed
region (`e2e`).  FLOPs per benchmarks/benchmark.py:17-20 of the reference:
fwd 4*B*S^2*H*D, bwd 2.5x, fwd+bwd 3.5x.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "burst-attention_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

H, D, B = 32, 128, 1
METRIC = "attention fwd+bwd TFLOPS/s (bs=1, H=32, d=128, bf16; seq in config, default 262144), aggregate over GPUs"


def flops(S, mode, batch=None):
    f = 4.0 * (B if batch is None else batch) * S * S * H * D
    return {"fwd": f, "bwd": 2.5 * f, "fwd_bwd": 3.5 * f}[mode]


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(burst=p["bf16_tflops"], sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                    hbm=p["hbm_gbs"], source="MEASURED_PEAKS.json")
    return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


# --------------------------------------------------------------------------- #
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for t, line in self.rows:
            if t < t0 or t > t1:
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "samples": len(sm),
                "reasons": sorted(reasons)}


# --------------------------------------------------------------------------- #
def _ref_shim():
    """baseline/ref_shim.py: the UNMODIFIED reference from the git-ignored baseline/_ref (None if that install did
    not travel to this box)."""
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    try:
        import ref_shim
        if ref_shim.available():
            ref_shim.load()
            return ref_shim
    except Exception as e:  # noqa: BLE001
        sys.stderr.write(f"bench.py: reference in baseline/_ref not usable ({e!r}); CPU arm falls back to the oracle port\n")
    return None


def cpu_ref_step(shim, S, Hc, Dc, dtype, W, threads):
    """One fwd+bwd of the reference's own device-agnostic chunk path (inter_normal_attn / _backward,
    burst_utils.py:42-100) over a W-rank ring simulated on the host cores.  Returns (s_fwd, s_bwd, flops_fwd)."""
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(0)
    q, k, v, do = (torch.randn(1, Hc, S, Dc, generator=g).to(dtype) for _ in range(4))
    *_, tf, tb = shim.cpu_ring_step(q, k, v, do, W, Dc ** -0.5)
    return tf, tb, 4.0 * S * S * Hc * Dc


def cpu_port_step(S, threads, Hc=8, Dc=D):
    """Fallback when baseline/_ref is absent: the oracle's restatement of the same path (4 simulated ring
    rounds, fp32).  Returns (s_fwd+bwd, flops_fwd+bwd)."""
    from oracle import attention_oracle as orc
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(0)
    W = 4
    q, k, v, do = (torch.randn(1, S, Hc, Dc, generator=g) for _ in range(4))
    sh = lambda t: [orc.shard(t, r, W, "contiguous") for r in range(W)]
    qs, ks, vs, dos = sh(q), sh(k), sh(v), sh(do)
    t0 = time.time()
    os_, lses = orc.ring_forward(qs, ks, vs, Dc ** -0.5, "none", torch.float32)
    orc.ring_backward(qs, ks, vs, os_, lses, dos, Dc ** -0.5, "none", torch.float32)
    dt = time.time() - t0
    return dt, 3.5 * 4.0 * S * S * Hc * Dc


def best_cpu_threads(shim):
    """torch's CPU kernels do not scale to every hardware thread of a big host on these shapes (128 threads
    were 10x slower than 8 on the round-1 box); probe a few thread counts on a small sample and keep the best."""
    n = os.cpu_count() or 1
    best, best_rate = n, 0.0
    for t in sorted({n, min(n, 64), min(n, 32), min(n, 16), min(n, 8)}, reverse=True):
        if shim is not None:
            cpu_ref_step(shim, 512, 8, 64, torch.float32, 1, t)
            tf, tb, fl = cpu_ref_step(shim, 2048, 8, 64, torch.float32, 1, t)
            rate = 3.5 * fl / (tf + tb)
        else:
            cpu_port_step(512, t)
            dt, fl = cpu_port_step(2048, t)
            rate = fl / dt
        if rate > best_rate:
            best, best_rate = t, rate
    return best


def cpu_baseline():
    """BASELINE.json configs[0] (C1): bs=1 seq=4096 H=8 d=64, the reference's CPU-runnable case, through the
    reference's own functions, fp32 and bf16, W in {1, 4} simulated ranks (BASELINE.md 3): 1 warm-up + 3 timed reps."""
    shim = _ref_shim()
    threads = best_cpu_threads(shim)
    if shim is None:
        dt, fl = cpu_port_step(4096, threads, 8, 64)
        return {"value": fl / dt / 1e12, "unit": "TFLOPS/s", "cores": threads, "kind": "port",
                "sample": f"oracle port (torch CPU fp32) of the reference path, C1: fwd+bwd bs=1 S=4096 H=8 d=64, "
                          f"4 simulated ring rounds, {dt:.1f} s (baseline/_ref absent on this box)"}
    S, Hc, Dc = 4096, 8, 64
    detail = {}
    t_all = time.time()
    for dtype, name in ((torch.float32, "fp32"), (torch.bfloat16, "bf16")):
        for W in (1, 4):
            cpu_ref_step(shim, S, Hc, Dc, dtype, W, threads)
            tf = tb = 0.0
            for _ in range(3):
                a, b, fl = cpu_ref_step(shim, S, Hc, Dc, dtype, W, threads)
                tf, tb = tf + a / 3, tb + b / 3
            detail[f"{name}_W{W}"] = {"fwd_ms": 1e3 * tf, "bwd_ms": 1e3 * tb, "fwd_gflops": fl / tf / 1e9,
                                      "bwd_gflops": 2.5 * fl / tb / 1e9, "fwd_bwd_gflops": 3.5 * fl / (tf + tb) / 1e9}
    main = detail["fp32_W4"]
    return {"value": main["fwd_bwd_gflops"] / 1e3, "unit": "TFLOPS/s", "cores": threads,
            "host_threads_available": os.cpu_count(), "kind": "reference",
            "sample": "reference inter_normal_attn/_backward (burst_utils.py:42-100, unmodified, from baseline/_ref) on the "
                      f"host cores, C1: bs=1 S=4096 H=8 d=64, fwd+bwd; value = fp32, 4 simulated ring ranks; 1 warm-up + "
                      f"3 reps per cell, {time.time() - t_all:.1f} s in total",
            "detail_gflops": detail}


def run_reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path on this box's host cores, on a BOUNDED
    sample of the bench workload (same d=128, bf16, non-causal; H=8 instead of 32, S=4096 instead of 262144)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    shim = _ref_shim()
    threads = best_cpu_threads(shim)
    S, Hc = 4096, 8
    warm = max(0, min(args.warmup, 1))
    steps = args.steps
    t = 0.0
    if shim is not None:
        for _ in range(warm):
            cpu_ref_step(shim, S, Hc, D, torch.bfloat16, 4, threads)
        for _ in range(steps):
            tf, tb, fl1 = cpu_ref_step(shim, S, Hc, D, torch.bfloat16, 4, threads)
            t += tf + tb
        fl, kind, dt_name = 3.5 * fl1, "reference", "bf16"
        what = ("reference inter_normal_attn/_backward (burst_utils.py:42-100, unmodified, baseline/_ref), torch CPU bf16, "
                f"{threads} threads")
    else:
        for _ in range(warm):
            cpu_port_step(S, threads)
        for _ in range(steps):
            dt, fl = cpu_port_step(S, threads)
            t += dt
        kind, dt_name = "port", "f32"
        what = f"oracle port of the reference path (torch CPU fp32, {threads} threads; baseline/_ref absent)"
    val = fl * steps / t / 1e12
    sample = f"{what}: fwd+bwd bs=1 S={S} H={Hc} d=128 non-causal, 4 simulated ring ranks per step"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "TFLOPS/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": 1e3 * t / steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": dt_name, "data": "synthetic",
        "config": {"workload": "bounded CPU sample of the bench workload: " + sample},
        "cpu_baseline": {"value": val, "unit": "TFLOPS/s", "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": "TFLOPS/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# --------------------------------------------------------------------------- #
# ring parity before timing: the reference's own protocol (test/test_burst.py:159-219: b=2, s=256*W, d=128, fp16
# rtol=1e-3/atol=1e-2; bf16 at this repo's stated rtol=1.6e-2/atol=2e-2) for non-causal / zigzag / striped shards,
# fwd + bwd, against a PLAIN PyTorch fp32 dense attention computed on the GPU (the oracle is not used here).
# --------------------------------------------------------------------------- #
def _shard(t, rank, world, layout):
    if layout == "contiguous":
        return t.chunk(world, dim=1)[rank].contiguous()
    if layout == "zigzag":  # halves {i, 2W-1-i} (reference test/test_burst.py:46-52)
        c = t.chunk(2 * world, dim=1)
        return torch.cat([c[rank], c[2 * world - 1 - rank]], dim=1).contiguous()
    return t[:, rank::world].contiguous()  # striped: tokens {i, i+W, ...} (:55-58)


def _dense_fp32(q, k, v, do, causal):
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        q, k, v = (t.float().permute(0, 2, 1, 3).detach().requires_grad_() for t in (q, k, v))
        s = (q @ k.transpose(-1, -2)) * q.shape[-1] ** -0.5
        if causal:
            S = s.shape[-1]
            s = s.masked_fill(~torch.ones(S, S, dtype=torch.bool, device=s.device).tril(), float("-inf"))
        o = torch.softmax(s, -1) @ v
        g = torch.autograd.grad(o, (q, k, v), do.float().permute(0, 2, 1, 3))
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    return [t.permute(0, 2, 1, 3) for t in (o, *g)]


def _ring_transport():
    from burst_attn import comm
    return comm.default_transport()


def ring_parity(world, rank, dev, double_group):
    from burst_attn import burst_attn_func, burst_attn_func_striped
    cases, failed, worst = 0, [], 0.0
    for dtype, tol in ((torch.float16, (1e-3, 1e-2)), (torch.bfloat16, (1.6e-2, 2e-2))):
        for name, func, causal, layout in (("none", burst_attn_func, False, "contiguous"),
                                           ("zigzag", burst_attn_func, True, "zigzag"),
                                           ("striped", burst_attn_func_striped, True, "striped")):
            g = torch.Generator().manual_seed(7)  # identical full tensors on every rank
            q, k, v, do = (torch.randn(2, 256 * world, 8, D, generator=g).to(dtype).to(dev) for _ in range(4))
            ref = _dense_fp32(q, k, v, do, causal)
            ql, kl, vl = (_shard(t, rank, world, layout).requires_grad_() for t in (q, k, v))
            o = func(ql, kl, vl, None, "cuda", causal, True, False, None, double_group)
            grads = torch.autograd.grad(o, (ql, kl, vl), _shard(do, rank, world, layout))
            ok = True
            for got, r in zip((o, *grads), ref):
                r = _shard(r, rank, world, layout)
                err = (got.float() - r).abs()
                ok &= bool((err <= tol[1] + tol[0] * r.abs()).all().item())
                worst = max(worst, float(err.max().item()))
            flag = torch.tensor([0 if ok else 1], device=dev)
            if world > 1:
                dist.all_reduce(flag)
            cases += 1
            if flag.item() != 0:
                failed.append(f"{name}/{str(dtype).split('.')[-1]}")
    w = torch.tensor([worst], device=dev)
    if world > 1:
        dist.all_reduce(w, op=dist.ReduceOp.MAX)
    return {"W": world, "protocol": "b=2 s=256*W h=8 d=128; none/zigzag/striped x fp16 (rtol 1e-3, atol 1e-2) / bf16 "
            "(1.6e-2, 2e-2); O,dQ,dK,dV vs plain PyTorch fp32 dense attention on the GPU",
            "cases": cases, "ok": not failed, "failed": failed, "max_abs_err": float(w.item())}


def ref_ratio(world, S, causal, value):
    """value / the UNMODIFIED reference's fwd+bwd TFLOPS/s on the same kind of box at the same (N, S, causal), as
    measured by tools/ref_on_b200.py and committed in profiles/ref_on_b200_r02.json (None if not measured)."""
    path = os.path.join(ROOT, "profiles", "ref_on_b200_r02.json")
    if not os.path.exists(path):
        return None
    for ln in open(path):
        try:
            r = json.loads(ln)
        except Exception:  # noqa: BLE001
            continue
        if r.get("n_gpus") == world and r.get("seq") == S and bool(r.get("causal")) == bool(causal):
            return {"ratio": value / r["fwd_bwd_tflops"], "reference_tflops": r["fwd_bwd_tflops"],
                    "source": "profiles/ref_on_b200_r02.json (tools/ref_on_b200.py, separate box of the same pool)"}
    return None


def ncu_traffic(kernel, Sq, Sk, Hh, causal):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of `kernel` at this launch shape from the
    ncu --set full summary that tools/profile.sh regenerates (profiles/ncu_traffic.json); None when that shape was
    never captured -- never a literal."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(path):
        return None, None
    try:
        tab = json.load(open(path))
    except Exception:  # noqa: BLE001
        return None, None
    key = f"{kernel}:Sq={Sq}:Sk={Sk}:H={Hh}:causal={int(bool(causal))}"
    ent = tab.get(key)
    return (ent["dram_bytes"], ent.get("source")) if ent else (None, None)


DUMP_ROWS = 512  # token positions over all ranks: 4 outputs x 512 x H x D x fp32 = 32 MiB at H=32, d=128


def dump_outputs(dirname, outs, rank, world):
    """Write (O, dQ, dK, dV) of one step, each [B, S_local, H, D], as <dirname>/{o,dq,dk,dv}.npy in float32, at
    DUMP_ROWS // world token positions (all batch rows, heads and dims) drawn with a fixed seed.  The inputs are seeded
    too, so the same arguments give the same positions of the same computation in every run: two builds can be
    compared output for output.  With N > 1 ranks each writes a sample of its own shard as <name>_rank<r>.npy."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    S_loc = outs[0].shape[1]
    n = min(S_loc, max(1, DUMP_ROWS // world))
    idx = torch.randperm(S_loc, generator=torch.Generator().manual_seed(0))[:n].sort().values.to(outs[0].device)
    suffix = "" if world == 1 else f"_rank{rank}"
    for name, t in zip(("o", "dq", "dk", "dv"), outs):
        np.save(os.path.join(dirname, f"{name}{suffix}.npy"), t.detach().index_select(1, idx).float().cpu().numpy())


# --------------------------------------------------------------------------- #
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--seq", type=int, default=262144, help="global sequence length")
    ap.add_argument("--causal", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the ring parity protocol that runs before timing")
    ap.add_argument("--ab-comm", action="store_true", help="(default for N > 1; kept for older command lines)")
    ap.add_argument("--no-ab-comm", action="store_true",
                    help="skip the A/B partner of multi-GPU runs: the step with the ring replaced by a local buffer swap "
                         "(BA_RING_TRANSPORT=local), which isolates exposed ring-communication time (comm_ab in the JSON line)")
    ap.add_argument("--configs", default="", help="comma list of extra runs in the same process group, e.g. "
                    "'262144,524288c,1048576' (c = causal zigzag); one JSON line each (multi-GPU sessions are "
                    "expensive to start)")
    ap.add_argument("--double-ring", type=int, default=0, metavar="L",
                    help="run over the hierarchical (double) ring with intra-node rings of L consecutive ranks "
                         "(reference benchmarks/benchmark.py --double_ring); default 0 = flat ring")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (O, dQ, dK, dV) as DIR/<name>.npy, "
                         "float32, at a fixed seeded sample of token positions (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and args.configs:
        ap.error("--dump-outputs takes the one configuration of --seq / --causal, not --configs")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computed; --impl reference times a CPU sample instead")

    if args.impl == "reference":
        return run_reference_arm(args)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback in the product path)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    W = max(3, args.warmup)
    K = args.steps

    from burst_attn import burst_attn_func
    from burst_attn import chunk_ops, native
    native.check(native.lib().ba_device_check(), "ba_device_check")
    ops = chunk_ops.get_ops()

    args.double_group = [None, None]
    if args.double_ring and world > 1:
        L = args.double_ring
        os.environ["BA_DOUBLE_RING"] = "1"
        assert world % L == 0 and 1 < L < world, "--double-ring L needs 1 < L < world and L | world"
        rows = [list(range(n * L, (n + 1) * L)) for n in range(world // L)]
        mk_groups = lambda ranks: dist.new_subgroups_by_enumeration(ranks, backend="nccl")[0]  # noqa: E731
        args.double_group = [mk_groups(rows), mk_groups([list(c) for c in zip(*rows)])]

    args.parity = None if args.no_parity else ring_parity(world, rank, dev, args.double_group)
    runs = [(args.seq, args.causal, B)]
    if args.configs:  # "<seq>[c][b<batch>]", e.g. 262144, 524288c, 65536b4 (the reference README's two sweeps)
        import re
        runs = []
        for c in args.configs.split(","):
            m = re.fullmatch(r"(\d+)(c?)(?:b(\d+))?", c.strip())
            assert m, f"bad config token {c!r}"
            runs.append((int(m.group(1)), bool(m.group(2)), int(m.group(3) or B)))
    for seq_i, causal_i, batch_i in runs:
        args.seq, args.causal, args.batch = seq_i, causal_i, batch_i
        _bench_one(args, world, rank, local, dev, W, K, ops, burst_attn_func)
        torch.cuda.empty_cache()
    if world > 1:
        dist.barrier()
        from burst_attn import comm as _comm
        _comm.destroy_rings()
        dist.destroy_process_group()


def _bench_one(args, world, rank, local, dev, W, K, ops, burst_attn_func):
    S = args.seq
    Bn = getattr(args, "batch", B)
    S_loc = S // world
    layout = "zigzag" if args.causal else "contiguous"
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    mk = lambda: torch.randn(Bn, S_loc, H, D, device=dev, generator=gen, dtype=torch.float32).to(torch.bfloat16)
    q, k, v, do = mk(), mk(), mk(), mk()

    def step(qd, kd, vd, dod):
        qq, kk, vv = qd.detach().requires_grad_(), kd.detach().requires_grad_(), vd.detach().requires_grad_()
        o = burst_attn_func(qq, kk, vv, None, "cuda", args.causal, True, False, None, args.double_group)
        dq, dk, dv = torch.autograd.grad(o, (qq, kk, vv), dod)
        return o, dq, dk, dv

    # --dump-outputs keeps each step's results alive until the next step has returned; the warm-up does the same, so
    # the extra memory is in the allocator's cache before the timed steps start
    last = []

    def bench_step():
        res = step(q, k, v, do)
        if args.dump_outputs:
            last[:] = res

    def fwd_only(qd, kd, vd):
        with torch.no_grad():
            return burst_attn_func(qd, kd, vd, None, "cuda", args.causal, True, False, None, args.double_group)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) / n

    # ---- warm-up (also builds the NCCL ring)
    for _ in range(W):
        bench_step()
    torch.cuda.synchronize()

    # ---- timed: fwd+bwd, inputs resident in HBM; per-kernel events on the launching stream
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)
    ops.enable_timing(True)
    launches0 = ops.launches
    t_wall0 = time.time()
    ms_step = timed(bench_step, K)
    t_wall1 = time.time()
    launches = ops.launches - launches0
    torch.cuda.synchronize()
    kms = ops.kernel_ms()
    ops.enable_timing(False)
    clocks = sampler.stop(t_wall0, t_wall1)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last, rank, world)
        last.clear()
    ms_fwd = timed(lambda: fwd_only(q, k, v), max(1, min(K, 3)))

    causal_div = 2.0 if args.causal else 1.0
    fl_step = flops(S, "fwd_bwd", Bn) / causal_div
    value = fl_step / (ms_step * 1e-3) / 1e12
    fwd_tflops = flops(S, "fwd", Bn) / causal_div / (ms_fwd * 1e-3) / 1e12

    # ---- roofline of the dominant kernel (backward tile kernel: 2.5x the forward FLOPs)
    pk = peaks()
    roof = None
    if "bwd_chunk_kernel" in kms:
        n_l, tot_ms = kms["bwd_chunk_kernel"]
        # algorithmic FLOPs per launch = this rank's share of the step's backward FLOPs (5 GEMMs:
        # 10*Sq*Sk*H*D per round) / launches per step; non-causal: exactly 10*S_loc^2*H*D per ring round
        fl_launch = flops(S, "bwd", Bn) / causal_div / world / (n_l / K)
        ach = fl_launch / (tot_ms / n_l * 1e-3) / 1e12
        # DRAM traffic per launch: read from the per-shape ncu --set full summary tools/profile.sh regenerates
        # (profiles/ncu_traffic.json), for the launch shape this run actually used; None if never captured
        shp = ops.dominant_shape("bwd_chunk_kernel")
        traffic, traffic_src = ncu_traffic("bwd_chunk_kernel", *shp) if shp else (None, None)
        roof = {"kernel": "bwd_chunk_kernel", "bound": "tensor", "achieved": ach, "peak": pk["sustained"],
                "unit": "TFLOP/s", "frac": ach / pk["sustained"], "traffic": traffic, "traffic_source": traffic_src,
                "launch_shape": {"Sq": shp[0], "Sk": shp[1], "H": shp[2], "causal": shp[3]} if shp else None,
                "algorithmic_bytes": (2 * shp[0] + 2 * shp[1]) * shp[2] * D * 2 * Bn + (shp[0] + 2 * shp[1]) * shp[2] * D * 4 * 2 * Bn
                if shp else None,
                "peak_source": pk["source"] + " bf16_tflops_sustained (of measured)",
                "launches": n_l, "avg_launch_ms": tot_ms / n_l}
        if "fwd_chunk_kernel" in kms:
            n_f, tot_f = kms["fwd_chunk_kernel"]
            fl_f = flops(S, "fwd", Bn) / causal_div / world / (n_f / K)
            roof["fwd_kernel"] = {"achieved": fl_f / (tot_f / n_f * 1e-3) / 1e12, "launches": n_f,
                                  "avg_launch_ms": tot_f / n_f,
                                  "frac": fl_f / (tot_f / n_f * 1e-3) / 1e12 / pk["sustained"]}

    # ---- how much of the step is NOT inside one of our kernels on the compute stream: torch memsets /
    # allocations, launch gaps and any ring-communication time the kernels did not hide (upper bound
    # on exposed comm; target < 5 %)
    overlap = None
    if kms:
        k_ms = sum(t for _, t in kms.values()) / K
        overlap = {"kernel_ms_per_step": k_ms, "non_kernel_ms_per_step": ms_step - k_ms,
                   "non_kernel_frac": (ms_step - k_ms) / ms_step,
                   "per_kernel_ms_per_step": {n: t / K for n, (c, t) in kms.items()}}

    # ---- e2e: same step through the public API from pinned host buffers
    e2e = None
    if not args.no_e2e:
        hq, hk, hv, hdo = (t.cpu().pin_memory() for t in (q, k, v, do))
        ho = [torch.empty_like(hq).pin_memory() for _ in range(4)]

        copy_s = torch.cuda.Stream(device=dev)

        def e2e_step():
            # what a user of the public API can overlap with streams: dO rides up under the forward, O rides down
            # under the backward; Q/K/V up and dQ/dK/dV down stay exposed (the drivers take whole device tensors)
            cur = torch.cuda.current_stream(dev)
            dq_, dk_, dv_ = (h.to(dev, non_blocking=True) for h in (hq, hk, hv))
            with torch.cuda.stream(copy_s):
                ddo_ = hdo.to(dev, non_blocking=True)
                ev_do = torch.cuda.Event()
                ev_do.record(copy_s)
            ddo_.record_stream(cur)
            qq, kk, vv = dq_.requires_grad_(), dk_.requires_grad_(), dv_.requires_grad_()
            o = burst_attn_func(qq, kk, vv, None, "cuda", args.causal, True, False, None, args.double_group)
            ev_o = torch.cuda.Event()
            ev_o.record(cur)
            with torch.cuda.stream(copy_s):
                copy_s.wait_event(ev_o)
                ho[0].copy_(o.detach(), non_blocking=True)
            o.record_stream(copy_s)
            cur.wait_event(ev_do)
            grads = torch.autograd.grad(o, (qq, kk, vv), ddo_)
            for h, t in zip(ho[1:], grads):
                h.copy_(t, non_blocking=True)
            cur.wait_stream(copy_s)
        def e2e_step_host():
            # one rank: hand the pinned HOST tensors to the public API; its L2-blocked drivers stream K/V blocks and dO
            # up and O / dQ / dK / dV blocks down under the kernels (burst_attn/host_stream.py)
            qq, kk, vv = (h.detach().requires_grad_() for h in (hq, hk, hv))
            o = burst_attn_func(qq, kk, vv, None, "cuda", args.causal, True, False, None, args.double_group)
            return (o,) + tuple(torch.autograd.grad(o, (qq, kk, vv), hdo))

        if world == 1:
            e2e_step = e2e_step_host  # noqa: F811
        e2e_step()
        e2e_step()
        ms_e2e = timed(e2e_step, K)
        nbytes = hq.numel() * hq.element_size()
        e2e = {"value": fl_step / (ms_e2e * 1e-3) / 1e12, "unit": "TFLOPS/s", "ms_per_step": ms_e2e,
               "h2d_bytes_per_step": 4 * nbytes * world, "d2h_bytes_per_step": 4 * nbytes * world,
               "how": ("burst_attn_func on pinned host tensors (host-resident operands: copies stream under the "
                       "L2-blocked sub-launches)" if world == 1 else
                       "pinned host buffers -> device tensors -> burst_attn_func; dO up under the forward, O down under "
                       "the backward on a copy stream")}

    # ---- A/B: the same step with the ring replaced by a local buffer swap -> exposed ring-communication time
    ab = None
    if not args.no_ab_comm and world > 1:
        prev_tr = os.environ.get("BA_RING_TRANSPORT")
        os.environ["BA_RING_TRANSPORT"] = "local"
        try:
            step(q, k, v, do)
            ms_local = timed(lambda: step(q, k, v, do), K)
        finally:
            if prev_tr is None:
                os.environ.pop("BA_RING_TRANSPORT", None)
            else:
                os.environ["BA_RING_TRANSPORT"] = prev_tr
        ab = {"ms_per_step_ring": ms_step, "ms_per_step_local_swap": ms_local,
              "exposed_comm_frac": max(0.0, (ms_step - ms_local) / ms_step),
              "how": "BA_RING_TRANSPORT=local: every hop is a device-local copy src->dst on the compute stream"}

    tot_launch = torch.tensor([launches], device=dev, dtype=torch.int64)
    if world > 1:
        dist.all_reduce(tot_launch)

    if rank == 0:
        cpu = None if (args.no_cpu or world > 1) else cpu_baseline()  # reported on rank 0 at N=1 only
        # BASELINE.md: the reference's README publishes 191 TFLOPS/s/GPU fwd+bwd at S=262144 on 8 GPUs (8xA100)
        vs = value / (191.0 * 8) if (world == 8 and S == 262144 and not args.causal) else None
        line = {
            "metric": METRIC, "value": value, "unit": "TFLOPS/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": vs,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"burst_attn_func fwd+bwd, bs={Bn} S={S} (S_local={S_loc}) H=32 d=128 bf16 "
                                   f"{'causal zigzag' if args.causal else 'non-causal contiguous'} shards, "
                                   f"{'local kernel, no ring' if world == 1 else f'{world}-rank ring over ' + ('copy engines + CUDA IPC' if _ring_transport() == 'ce' else 'NCCL')}"
                                   f"{f' (double ring, intra {args.double_ring})' if args.double_ring and world > 1 else ''}",
                       "global_batch": Bn, "seq_len": S, "parallelism": f"sp{world}",
                       "l2": "inputs (>= 256 MiB per tensor per rank) exceed the 126 MB L2; no flush needed"},
            "value_per_gpu": value / world, "fwd_tflops": fwd_tflops, "fwd_ms": ms_fwd,
            "gpu_launches": int(tot_launch.item()), "clocks": clocks, "e2e": e2e, "roofline": roof, "overlap": overlap,
            "cpu_baseline": cpu, "parity": getattr(args, "parity", None), "comm_ab": ab,
            "vs_reference_on_b200": ref_ratio(world, S, args.causal, value),
        }
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
