"""CPU: the oracle against what the UNMODIFIED reference computed on inputs and seeds that are NOT the other
fixtures — the oracle is pinned to the reference on a second, independent set of inputs.  The reference's
outputs are tests/golden/reference_live.npz (oracle/gen_golden_live.py, which also checked the oracle
bit for bit against the reference when it wrote them; large outputs are kept as a fixed sample of
elements, `gen_golden_live.sample`).  Integer outputs must match exactly; floating-point ones to TOL of
their largest magnitude, which only absorbs a different CPU's oneDNN/MKL kernel choice."""
import numpy as np
import pytest
import torch

from oracle import gen_golden_live as L

TOL = 1e-5


@pytest.fixture(scope="module")
def ref(golden):
    return golden("reference_live.npz")


def _close(ours, ref, key, tol=TOL):
    """`ours` (whole) against the reference's output `key` (whole or sampled) of the golden file."""
    assert tuple(ours.shape) == tuple(ref[f"{key}_shape"])
    ours, want = L.sample(ours).astype(np.float64), ref[key].astype(np.float64)
    assert float(np.abs(ours - want).max()) <= tol * max(1.0, float(np.abs(want).max())), float(np.abs(ours - want).max())


def test_propagation_ops_live(ref, prop_sd, fuse_sd):
    from oracle import stm_oracle as O
    images, mask = L.ops_inputs()
    frame = images[:, 1]
    for name, a in zip(("f16", "f8", "f4", "k16", "v16"), O.get_query_values(prop_sd, frame)):
        _close(a, ref, f"ops_{name}")
    mk, mv = O.memorize(prop_sd, frame, mask[1:])
    _close(mk, ref, "ops_mem_k")
    _close(mv, ref, "ops_mem_v")
    qv = O.get_query_values(prop_sd, images[:, 2])
    seg = O.segment_with_query(prop_sd, mk, mv, *qv, top_k=20)
    _close(seg, ref, "ops_seg")
    agg = O.aggregate_wbg(seg, keep_bg=True)
    _close(agg, ref, "ops_agg")
    assert float(np.abs(O.aggregate_wbg_f64(seg.numpy(), keep_bg=True) - agg.numpy()).max()) <= 5e-7
    pos, neg = (mask[1:2] - seg[0:1]).clamp(0, 1), (seg[0:1] - mask[1:2]).clamp(0, 1)
    at = O.get_attention(None, mk[0:1], pos, neg, qv[3])
    _close(at, ref, "ops_attn")
    assert float(np.abs(O.get_attention_f64(mk[0:1].numpy(), pos.numpy(), neg.numpy(), qv[3].numpy()) - at.numpy()).max()) <= 2e-6
    dist = torch.tensor([[0.25, 0.75]])
    _close(O.fusion_net(fuse_sd, images[:, 2], seg[0:1], agg[1:2], at, dist), ref, "ops_fuse")


def test_inference_core_live(ref, prop_sd, fuse_sd):
    """Whole interact() runs, two interactions (the second one fuses): bank trace is not observable in the
    reference, so probabilities and masks are compared."""
    from oracle import stm_oracle as O
    images, inters = L.core_inputs()
    oc = O.OracleInferenceCore(prop_sd, fuse_sd, images, 2, mem_freq=2, top_k=20)
    for j, (m, idx) in enumerate(inters, 1):
        om = oc.interact(m, idx)
        assert (om == ref[f"core_masks{j}"]).all() and om.shape == (7, 64, 88)
        _close(oc.prob, ref, f"core_prob{j}")
    _close(oc.certain_mem_k, ref, "core_certain_k")


def test_s2m_live(ref):
    from oracle import s2m_oracle as S, weights as Wt
    sd = Wt.make_s2m_state_dict()
    x, image, prev, scr = L.s2m_inputs()
    _close(S.s2m_forward(sd, x), ref, "s2m_logits")
    _close(S.s2m_controller_interact(sd, image, prev, scr, 1), ref, "s2m_controller")


def test_egress_live(ref):
    from oracle import egress_oracle as EO
    assert np.array_equal(ref["egress_palette"], EO.color_map())
    image, mask = L.egress_inputs()
    for alpha in L.EGRESS_ALPHAS:
        a = int(round(alpha * 100))
        assert np.array_equal(ref[f"egress_overlay_a{a}"], EO.overlay_davis(image, mask, alpha))
        assert np.array_equal(ref[f"egress_fade_a{a}"], EO.overlay_davis(image, mask, alpha, fade=True))


def test_fusion_generator_flow_live(ref, prop_sd):
    """SURVEY §8f-1: the client flow restated in tests/test_gpu_clients.py (what the GPU test drives our
    PropagationNetwork through) equals what the reference's real FusionGenerator class returned."""
    import types
    from oracle import stm_oracle as O
    from test_gpu_clients import fusion_generator_flow
    images, soft = L.fusion_generator_inputs()
    api = types.SimpleNamespace(pad_divide_by=O.pad_divide_by, aggregate_wbg=O.aggregate_wbg,
                                memorize=lambda f, m: O.memorize(prop_sd, f, m),
                                get_query_values=lambda f: O.get_query_values(prop_sd, f),
                                segment_with_query=lambda *a: O.segment_with_query(prop_sd, *a, top_k=50))
    prob = fusion_generator_flow(api, images, soft, 2, 0, 4, mem_freq=2)  # [K+1, T, 1, nh, nw], padded 168 -> 176
    assert prob.shape == (3, 5, 1, 128, 176)
    _close(prob[:, :, 0, :, 4:-4].contiguous(), ref, "fusion_generator_prob")  # the reference returns it unpadded


def test_attention_read_network_live(ref, prop_sd):
    """SURVEY §8f-2: AttentionReadNetwork.forward (model/attn_network.py:48-80) on a fresh batch."""
    from oracle import stm_oracle as O
    o1, o2 = O.attention_read_network(prop_sd, *L.attn_inputs())
    _close(o1, ref, "attn1")
    _close(o2, ref, "attn2")
