"""Generate golden vectors by RUNNING THE REFERENCE (MayDomine/Burst-Attention at
/root/reference) on CPU in the build container.  The reference cannot travel to
the GPU box, so its outputs are committed as small .npz fixtures next to this
script; tests/test_oracle_golden.py pins oracle/attention_oracle.py to them.

The reference imports `bmtrain` (absent here) at module scope
(burst_attn_interface.py:1, comm.py:2-5); a stub module is injected -- no
reference source is modified or copied.

Run:  python tests/golden/make_golden.py      (needs /root/reference)

`ring` writes reference_cpu_ring.npz: the reference's whole CPU ring step (its own
inter_normal_attn / inter_normal_attn_backward over a simulated ring, through
baseline/ref_shim.py), which tests/test_oracle_golden.py pins the oracle's dense
attention to.  It needs the reference installed in baseline/_ref, which build()
makes where the reference's source is available.

      python tests/golden/make_golden.py ring
"""
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"

# inputs of the ring vectors: torch.manual_seed(RING_SEED), then q, k, v, dO = randn(RING_SHAPE) in that order,
# layout [B, H, S, D]; of each 512 KB output RING_PER_ROW elements of every (b, h, s) row are stored, at columns
# drawn with a fixed seed, so an error confined to a few rows (a chunk edge, say) is still seen
RING_SEED, RING_SHAPE, RING_WORLDS, RING_PER_ROW = 0, (1, 4, 512, 64), (1, 4), 2


def ring_inputs():
    torch.manual_seed(RING_SEED)
    return [torch.randn(*RING_SHAPE) for _ in range(4)]


def ring_sample_index():
    """Flat indices into a contiguous RING_SHAPE tensor, sorted."""
    rows, D = int(np.prod(RING_SHAPE[:-1])), RING_SHAPE[-1]
    g = torch.Generator().manual_seed(RING_SEED + 1)
    cols = torch.rand(rows, D, generator=g).argsort(dim=1)[:, :RING_PER_ROW]
    return (torch.arange(rows).unsqueeze(1) * D + cols).flatten().sort().values


def _stub_bmtrain():
    bmt = types.ModuleType("bmtrain")
    bmt.init = types.SimpleNamespace(is_initialized=lambda: False)
    bmt.config = {}
    bmt.print_rank = print
    sys.modules["bmtrain"] = bmt
    d = types.ModuleType("bmtrain.distributed"); sys.modules["bmtrain.distributed"] = d
    ops = types.ModuleType("bmtrain.distributed.ops"); ops.ncclSend = ops.ncclRecv = None
    sys.modules["bmtrain.distributed.ops"] = ops
    nccl = types.ModuleType("bmtrain.nccl")
    for n in ("commCount", "groupEnd", "groupStart", "allReduce", "commRank"):
        setattr(nccl, n, None)
    sys.modules["bmtrain.nccl"] = nccl
    bmt.distributed, bmt.nccl = d, nccl


def main():
    _stub_bmtrain()
    sys.path.insert(0, REF)
    import burst_attn.burst_utils as bu
    import burst_attn.burst_attn_interface as bi

    torch.manual_seed(20260922)
    out = {}

    # ---- 1. chunked forward chain through inter_normal_attn (burst_utils.py:42-74)
    B, H, S, D, W = 1, 2, 256, 64, 4
    scale = 1.0 / D ** 0.5
    q = torch.randn(B, H, S, D)
    k = torch.randn(B, H, S, D)
    v = torch.randn(B, H, S, D)
    m_i = lse_i = acc_o = None
    for c in range(W):
        ks = k.chunk(W, dim=2)[c]
        vs = v.chunk(W, dim=2)[c]
        acc_o, m_i, lse_i = bu.inter_normal_attn(q, ks, vs, m_i, lse_i, acc_o, scale, None)
    o_final = acc_o * torch.exp(m_i - lse_i)  # burst_attn_interface.py:246-248
    out.update(fwd_q=q, fwd_k=k, fwd_v=v, fwd_acc_o=acc_o, fwd_m=m_i, fwd_lse=lse_i,
               fwd_o=o_final, fwd_W=torch.tensor(W), fwd_scale=torch.tensor(scale))

    # ---- 2. chunk backward through inter_normal_attn_backward (burst_utils.py:77-100)
    do = torch.randn(B, H, S, D)
    delta = (o_final * do).sum(-1, keepdim=True)
    dq_tot = torch.zeros_like(q)
    dk_parts, dv_parts = [], []
    for c in range(W):
        ks = k.chunk(W, dim=2)[c]
        vs = v.chunk(W, dim=2)[c]
        dq = torch.empty_like(q)
        dk = torch.zeros_like(ks)
        dv = torch.zeros_like(vs)
        bu.inter_normal_attn_backward(do, q, ks, vs, delta, lse_i, dq, dk, dv, scale, None)
        dq_tot += dq
        dk_parts.append(dk)
        dv_parts.append(dv)
    out.update(bwd_do=do, bwd_delta=delta, bwd_dq=dq_tot,
               bwd_dk=torch.cat(dk_parts, 2), bwd_dv=torch.cat(dv_parts, 2))

    # ---- 3. LSE merge cuda_scale_out_lse_helper (burst_utils.py:20-33)
    Bm, Sm, Hm, Dm = 2, 48, 3, 16
    o = torch.randn(Bm, Sm, Hm, Dm)
    lse = torch.randn(Bm, Sm, Hm, 1) * 3
    o_new = torch.randn(Bm, Sm, Hm, Dm)
    lse_new = torch.randn(Bm, Hm, Sm) * 3
    mo, ml = bu.cuda_scale_out_lse_helper(o, lse, o_new, lse_new)
    out.update(merge_o=o, merge_lse=lse, merge_o_i=o_new, merge_lse_i=lse_new,
               merge_out_o=mo, merge_out_lse=ml)

    # ---- 4. get_partition_id (burst_attn_interface.py:20-37) single + double ring
    L, M = 4, 2  # 2 "nodes" of 4 (test/test_burst.py:129-138)
    table = np.zeros((L * M, L * M), dtype=np.int64)  # [rank, r-1]
    single = np.array([bi.get_partition_id([None, None], r) if False else r - 1
                       for r in range(1, L * M + 1)], dtype=np.int64)
    saved = (bi.get_rank, bi.get_world_size)
    try:
        for rank in range(L * M):
            intra, inter = rank % L, rank // L
            bi.get_rank = lambda g=None: {"intra": intra, "inter": inter}.get(g, rank)
            bi.get_world_size = lambda g=None: {"intra": L, "inter": M}.get(g, L * M)
            for r in range(1, L * M + 1):
                table[rank, r - 1] = bi.get_partition_id(("intra", "inter"), r)
        # single ring through the real function
        bi.get_rank = lambda g=None: 0
        bi.get_world_size = lambda g=None: L * M
        single = np.array([bi.get_partition_id([None, None], r) for r in range(1, L * M + 1)],
                          dtype=np.int64)
    finally:
        bi.get_rank, bi.get_world_size = saved
    out.update(pid_double=torch.from_numpy(table), pid_single=torch.from_numpy(single),
               pid_L=torch.tensor(L), pid_M=torch.tensor(M))

    # ---- 5. whole-op forward on CPU, W=1, flash=None ("normal" path, [B,H,S,D])
    try:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29577")
        dist.init_process_group("gloo", rank=0, world_size=1)
        qq = torch.randn(1, 2, 128, 32)
        kk = torch.randn(1, 2, 128, 32)
        vv = torch.randn(1, 2, 128, 32)
        oo = bi.burst_attn_func(qq, kk, vv, None, None, False)
        out.update(op_q=qq, op_k=kk, op_v=vv, op_o=oo)
        dist.destroy_process_group()
    except Exception as e:  # pragma: no cover - recorded in the fixture
        print("whole-op CPU forward not runnable:", repr(e))

    np.savez_compressed(os.path.join(HERE, "reference_vectors.npz"),
                        **{k_: v_.detach().cpu().numpy() for k_, v_ in out.items()})
    print("wrote", os.path.join(HERE, "reference_vectors.npz"), sorted(out))


def ring():
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(HERE)), "baseline"))
    import ref_shim
    q, k, v, do = ring_inputs()
    idx = ring_sample_index()
    out = {"idx": idx.numpy().astype(np.int32)}
    out.update({f"in_{n}": t.flatten()[idx].numpy() for n, t in zip(("q", "k", "v", "do"), (q, k, v, do))})
    for W in RING_WORLDS:
        o, dq, dk, dv, _, _ = ref_shim.cpu_ring_step(q, k, v, do, W, RING_SHAPE[-1] ** -0.5)
        out.update({f"W{W}_{n}": t.flatten()[idx].numpy() for n, t in zip(("o", "dq", "dk", "dv"), (o, dq, dk, dv))})
    path = os.path.join(HERE, "reference_cpu_ring.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, sorted(out))


if __name__ == "__main__":
    if sys.argv[1:] == ["ring"]:
        ring()
    else:
        main()
