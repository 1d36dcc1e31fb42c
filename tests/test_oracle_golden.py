"""Pin oracle/attention_oracle.py to vectors produced by the reference itself
(tests/golden/make_golden.py ran the reference's own functions on CPU)."""
import torch

from oracle import attention_oracle as orc


def T(a):
    return torch.from_numpy(a)


def test_unnormalised_chunk_chain_matches_reference(golden):
    q, k, v = T(golden["fwd_q"]), T(golden["fwd_k"]), T(golden["fwd_v"])
    W, scale = int(golden["fwd_W"]), float(golden["fwd_scale"])
    m = lse = acc = None
    for c in range(W):
        acc, m, lse = orc.chunk_forward_unnormalised(
            q, k.chunk(W, 2)[c], v.chunk(W, 2)[c], m, lse, acc, scale)
    torch.testing.assert_close(acc, T(golden["fwd_acc_o"]), rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(m, T(golden["fwd_m"]), rtol=0, atol=0)
    torch.testing.assert_close(lse, T(golden["fwd_lse"]), rtol=1e-6, atol=1e-6)


def test_carried_state_chunk_forward_matches_reference_output(golden):
    """The product's state convention (normalised O + lse, exact log) must give
    the reference's final O; the reference's +1e-5-in-log fudge
    (burst_utils.py:71,73) bounds agreement at ~1e-5 relative."""
    q, k, v = (T(golden[n]).permute(0, 2, 1, 3) for n in ("fwd_q", "fwd_k", "fwd_v"))
    W, scale = int(golden["fwd_W"]), float(golden["fwd_scale"])
    o = lse = None
    for c in range(W):
        o, lse = orc.chunk_forward(q, k.chunk(W, 1)[c], v.chunk(W, 1)[c], o, lse, scale)
    ref_o = T(golden["fwd_o"]).permute(0, 2, 1, 3).double()
    torch.testing.assert_close(o, ref_o, rtol=1e-4, atol=2e-5)
    ref_lse = T(golden["fwd_lse"]).squeeze(-1).double()
    torch.testing.assert_close(lse, ref_lse, rtol=1e-4, atol=2e-5)
    # and against the dense definition, tightly
    od, lsed = orc.dense_attention(q, k, v, scale)
    torch.testing.assert_close(o, od, rtol=1e-10, atol=1e-10)
    torch.testing.assert_close(lse, lsed, rtol=1e-10, atol=1e-10)


def test_chunk_backward_matches_reference(golden):
    q, k, v, do = (T(golden[n]).permute(0, 2, 1, 3) for n in ("fwd_q", "fwd_k", "fwd_v", "bwd_do"))
    W, scale = int(golden["fwd_W"]), float(golden["fwd_scale"])
    lse = T(golden["fwd_lse"]).squeeze(-1)
    delta = T(golden["bwd_delta"]).squeeze(-1)
    dq = torch.zeros_like(q, dtype=torch.float64)
    dks, dvs = [], []
    for c in range(W):
        a, b, c_ = orc.chunk_backward(do, q, k.chunk(W, 1)[c], v.chunk(W, 1)[c], delta, lse, scale)
        dq += a
        dks.append(b)
        dvs.append(c_)
    ref = lambda n: T(golden[n]).permute(0, 2, 1, 3).double()
    torch.testing.assert_close(dq, ref("bwd_dq"), rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(torch.cat(dks, 1), ref("bwd_dk"), rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(torch.cat(dvs, 1), ref("bwd_dv"), rtol=1e-4, atol=1e-5)


def test_lse_merge_matches_reference(golden):
    """chunk_forward's merge == cuda_scale_out_lse_helper (burst_utils.py:20-33)."""
    o, lse = T(golden["merge_o"]).double(), T(golden["merge_lse"]).double()
    o_i, lse_i = T(golden["merge_o_i"]).double(), T(golden["merge_lse_i"]).double()
    lse_bhs = lse.squeeze(-1).permute(0, 2, 1)
    new_lse = torch.logaddexp(lse_bhs, lse_i)
    w0 = torch.exp(lse_bhs - new_lse).permute(0, 2, 1).unsqueeze(-1)
    w1 = torch.exp(lse_i - new_lse).permute(0, 2, 1).unsqueeze(-1)
    torch.testing.assert_close(w0 * o + w1 * o_i, T(golden["merge_out_o"]).double(), rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(new_lse.permute(0, 2, 1).unsqueeze(-1),
                               T(golden["merge_out_lse"]).double(), rtol=1e-5, atol=1e-5)


def test_partition_ids_match_reference(golden):
    L, M = int(golden["pid_L"]), int(golden["pid_M"])
    W = L * M
    assert [orc.get_partition_id_single(r) for r in range(1, W + 1)] == golden["pid_single"].tolist()
    for rank in range(W):
        got = [orc.get_partition_id_double(r, rank % L, rank // L, L, M) for r in range(1, W + 1)]
        assert got == golden["pid_double"][rank].tolist()


def test_whole_op_forward_matches_reference(golden):
    q, k, v = (T(golden[n]).permute(0, 2, 1, 3) for n in ("op_q", "op_k", "op_v"))
    o, _ = orc.dense_attention(q, k, v)
    torch.testing.assert_close(o, T(golden["op_o"]).permute(0, 2, 1, 3).double(), rtol=1e-4, atol=2e-5)


def test_oracle_matches_the_installed_reference_cpu_ring():
    """Second pin (besides the chunk-level vectors above): the UNMODIFIED reference, driven through its own
    inter_normal_attn / inter_normal_attn_backward over a simulated 1- and 4-rank ring (baseline/ref_shim.cpu_ring_step),
    against the oracle's dense attention.  The reference's outputs are stored at a seeded sample of positions in
    tests/golden/reference_cpu_ring.npz (`python tests/golden/make_golden.py ring` regenerates it)."""
    import os
    import sys

    import numpy as np
    here = os.path.dirname(os.path.abspath(__file__))
    sys.path.insert(0, os.path.join(here, "golden"))
    import make_golden as mg
    ring = np.load(os.path.join(here, "golden", "reference_cpu_ring.npz"))
    q, k, v, do = mg.ring_inputs()
    idx = torch.from_numpy(ring["idx"]).long()
    for name, t in zip(("q", "k", "v", "do"), (q, k, v, do)):  # the inputs the reference ran on
        assert torch.equal(t.flatten()[idx], T(ring[f"in_{name}"])), name
    p = lambda t: t.permute(0, 2, 1, 3)  # noqa: E731  reference "normal" layout [B,H,S,D] <-> oracle [B,S,H,D]
    refs = orc.dense_attention_bwd(p(q), p(k), p(v), p(do))
    for W in mg.RING_WORLDS:
        for name, ref in zip(("o", "dq", "dk", "dv"), (refs[0],) + refs[2:]):
            # floor: the reference's own +1e-5 inside log (burst_utils.py:71,73) and fp32 arithmetic
            torch.testing.assert_close(T(ring[f"W{W}_{name}"]).double(), p(ref).flatten()[idx], rtol=1e-4, atol=2e-5)
