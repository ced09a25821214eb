"""Golden vectors for tests/test_reference_live.py and the IoU test of tests/test_dropin_callers_cpu.py:
what the UNMODIFIED reference (imported through oracle/refshim.py) computes on inputs and seeds that are
NOT those of the other fixtures, so that the oracle stays pinned to the reference on a second,
independent set of inputs.  Every case first checks that the oracle equals the reference bit for bit on
this host, then keeps the reference's outputs — whole where they are small, a fixed sample of at most
SAMPLE elements (`sample`) where they are not, so that the file stays small — in
tests/golden/reference_live.npz.  The input recipes below are the ones the tests rebuild.
Run where a checkout of the reference is available:  python -m oracle.gen_golden_live

TEST INFRASTRUCTURE (see oracle/stm_oracle.py)."""
from __future__ import annotations

import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import weights as Wt  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "reference_live.npz")
SAMPLE = 2048


def sample(a, n: int = SAMPLE) -> np.ndarray:
    """`n` elements of `a` (flattened) at evenly spread positions; the whole array when it has no more.
    Positions depend on the size only, so the generator and the tests pick the same elements."""
    a = np.asarray(a).reshape(-1)
    if a.size <= n:
        return a.copy()
    return a[np.linspace(0, a.size - 1, n).round().astype(np.int64)]


# ------------------------------------------------------------------------------------- input recipes
def ops_inputs():
    return Wt.synthetic_clip(3, 64, 96, 3, seed=2024)  # three objects: the "others" channel sums two masks


def core_inputs():
    images, mask = Wt.synthetic_clip(7, 64, 88, 2, seed=77)  # 88 -> padded to 96
    return images, ((mask, 1), (mask.flip(-1).contiguous(), 6))  # the second interaction fuses


def s2m_inputs():
    x = torch.randn((2, 6, 64, 80), generator=torch.Generator().manual_seed(5))
    image = torch.randn((1, 3, 64, 80), generator=torch.Generator().manual_seed(6))
    prev = torch.zeros((1, 64, 80), dtype=torch.int64)
    prev[:, 10:30, 10:40] = 1
    scr = np.full((60, 75), 255, dtype=np.uint8)  # unpadded: the controller pads the scribble maps
    scr[20:22, 5:50] = 1
    scr[40:42, 30:70] = 0
    return x, image, prev, scr


EGRESS_ALPHAS = (0.5, 0.37)


def egress_inputs():
    rng = np.random.default_rng(9)
    image = rng.integers(0, 256, size=(40, 52, 3), dtype=np.uint8)
    mask = rng.integers(0, 7, size=(40, 52), dtype=np.uint8) * (rng.random((40, 52)) > 0.6)
    return image, mask.astype(np.uint8)


def fusion_generator_inputs():
    images, mask = Wt.synthetic_clip(5, 128, 168, 2, seed=31)
    return images, mask[1:] * 0.8 + 0.05


def attn_inputs():
    g = torch.Generator().manual_seed(123)
    image, query = torch.randn((1, 3, 48, 80), generator=g), torch.randn((1, 3, 48, 80), generator=g)
    m11, m21, m12, m22 = (torch.rand((1, 1, 48, 80), generator=g) for _ in range(4))
    return image, m11, m21, m12, m22, query


def iou_inputs():
    rng = np.random.default_rng(3)
    seg_np, gt_np = rng.random((40, 50)) > 0.5, rng.random((40, 50)) > 0.6
    scores = torch.from_numpy(rng.random((4, 40, 50)).astype(np.float32))
    gt_soft = torch.from_numpy(rng.random((3, 1, 40, 50)).astype(np.float32))
    lab, lab2 = rng.integers(0, 4, (40, 50)), rng.integers(0, 4, (40, 50))
    return seg_np, gt_np, scores, gt_soft, lab, lab2


def iou_values(tu):
    """The IoU helpers of a `util.tensor_util` module on iou_inputs(), as float64 values."""
    seg_np, gt_np, scores, gt_soft, lab, lab2 = iou_inputs()
    seg_t, gt_t = torch.from_numpy(seg_np), torch.from_numpy(gt_np)
    vals = [*tu.compute_tensor_iu(seg_t, gt_t), tu.compute_tensor_iou(seg_t, gt_t), *tu.compute_np_iu(seg_np, gt_np),
            tu.compute_np_iou(seg_np, gt_np), tu.compute_multi_class_iou(scores, gt_soft),
            tu.compute_multi_class_iou_idx(lab, gt_soft[:, 0].numpy()), tu.compute_multi_class_iou_both_idx(lab, lab2)]
    return np.array([float(v) for v in vals], dtype=np.float64)


# ------------------------------------------------------------------------------------- reference outputs
def _eq(a, b):
    assert torch.equal(torch.as_tensor(a), torch.as_tensor(b)), "oracle differs from the reference"


def _reference_outputs(ref, prop_sd, fuse_sd):
    from oracle import egress_oracle as EO, refshim, s2m_oracle as S, stm_oracle as O
    from oracle.gen_golden_egress import load_reference_utils
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_gpu_clients import fusion_generator_flow
    g = {}

    net, fuse = ref.build_prop(prop_sd, top_k=20), ref.build_fusion(fuse_sd)
    images, mask = ops_inputs()
    frame = images[:, 1]
    for name, a, b in zip(("f16", "f8", "f4", "k16", "v16"), O.get_query_values(prop_sd, frame), net.get_query_values(frame)):
        _eq(a, b)
        g[f"ops_{name}"] = b
    mk, mv = net.memorize(frame, mask[1:])
    ok, ov = O.memorize(prop_sd, frame, mask[1:])
    _eq(ok, mk)
    _eq(ov, mv)
    qv = net.get_query_values(images[:, 2])
    seg = net.segment_with_query(mk, mv, *qv)
    _eq(O.segment_with_query(prop_sd, mk, mv, *qv, top_k=20), seg)
    agg = ref.aggregate_wbg(seg, keep_bg=True)
    _eq(O.aggregate_wbg(seg, keep_bg=True), agg)
    pos, neg = (mask[1:2] - seg[0:1]).clamp(0, 1), (seg[0:1] - mask[1:2]).clamp(0, 1)
    at = net.get_attention(mk[0:1], pos, neg, qv[3])
    _eq(O.get_attention(None, mk[0:1], pos, neg, qv[3]), at)
    fu = fuse(images[:, 2], seg[0:1], agg[1:2], at, torch.tensor([[0.25, 0.75]]))
    _eq(O.fusion_net(fuse_sd, images[:, 2], seg[0:1], agg[1:2], at, torch.tensor([[0.25, 0.75]])), fu)
    g.update(ops_mem_k=mk, ops_mem_v=mv, ops_seg=seg, ops_agg=agg, ops_attn=at, ops_fuse=fu)

    images, inters = core_inputs()
    rc = ref.InferenceCore(net, fuse, images, 2, mem_profile=0, mem_freq=2, device="cpu")
    oc = O.OracleInferenceCore(prop_sd, fuse_sd, images, 2, mem_freq=2, top_k=20)
    for j, (m, idx) in enumerate(inters, 1):
        rm = rc.interact(m, idx)
        assert (rm == oc.interact(m, idx)).all()
        _eq(oc.prob, rc.prob)
        g[f"core_masks{j}"], g[f"core_prob{j}"] = rm.astype(np.uint8), rc.prob.clone()
    _eq(oc.certain_mem_k, rc.certain_mem_k)
    g["core_certain_k"] = rc.certain_mem_k

    sd = Wt.make_s2m_state_dict()
    x, image, prev, scr = s2m_inputs()
    with refshim.reference_on_path():
        from interact.s2m_controller import S2MController
        from model.s2m.s2m_network import deeplabv3plus_resnet50 as S2M
        s2m = S2M().eval()
        s2m.load_state_dict(sd, strict=True)
        logits = s2m(x)
        ctrl = S2MController(s2m, 1, ignore_class=255, device="cpu").interact(image, prev, scr)
    _eq(S.s2m_forward(sd, x), logits)
    _eq(S.s2m_controller_interact(sd, image, prev, scr, 1), ctrl)
    g.update(s2m_logits=logits, s2m_controller=ctrl)

    iu, pal = load_reference_utils()
    g["egress_palette"] = pal.pal_color_map().astype(np.uint8)
    assert np.array_equal(g["egress_palette"], EO.color_map())
    image, mask = egress_inputs()
    for alpha in EGRESS_ALPHAS:
        a = int(round(alpha * 100))
        g[f"egress_overlay_a{a}"], g[f"egress_fade_a{a}"] = iu.overlay_davis(image, mask, alpha), iu.overlay_davis_fade(image, mask, alpha)
        assert np.array_equal(g[f"egress_overlay_a{a}"], EO.overlay_davis(image, mask, alpha))
        assert np.array_equal(g[f"egress_fade_a{a}"], EO.overlay_davis(image, mask, alpha, fade=True))

    images, soft = fusion_generator_inputs()
    net50 = ref.build_prop(prop_sd, top_k=50)
    with refshim.reference_on_path():
        import importlib
        FusionGenerator = importlib.import_module("generation.fusion_generator").FusionGenerator
        for k in [k for k in sys.modules if k == "generation" or k.startswith("generation.")]:
            sys.modules.pop(k)
    gen = FusionGenerator(net50, images, mem_freq=2)
    gen.reset(2)
    ref_prob = gen.interact_mask(soft, 2, 0, 4)  # [K+1, T, h, w], unpadded
    api = types.SimpleNamespace(pad_divide_by=O.pad_divide_by, aggregate_wbg=O.aggregate_wbg,
                                memorize=lambda f, m: O.memorize(prop_sd, f, m),
                                get_query_values=lambda f: O.get_query_values(prop_sd, f),
                                segment_with_query=lambda *a: O.segment_with_query(prop_sd, *a, top_k=50))
    _eq(fusion_generator_flow(api, images, soft, 2, 0, 4, mem_freq=2)[:, :, 0, :, 4:-4], ref_prob)
    g["fusion_generator_prob"] = ref_prob

    a1, a2 = ref.build_attn(prop_sd)(*attn_inputs())
    o1, o2 = O.attention_read_network(prop_sd, *attn_inputs())
    _eq(o1, a1)
    _eq(o2, a2)
    g.update(attn1=a1, attn2=a2)

    from util import tensor_util as ours
    with refshim.reference_on_path():
        import importlib
        ref_tu = importlib.import_module("util.tensor_util")
    g["iou"] = iou_values(ref_tu)
    assert np.array_equal(iou_values(ours), g["iou"])
    g["iou_tensor_iu_dtype"] = np.array(str(ref_tu.compute_tensor_iu(*map(torch.from_numpy, iou_inputs()[:2]))[0].dtype))
    return g


def main():
    from oracle import GOLDEN_THREADS, refshim
    torch.set_grad_enabled(False)
    torch.set_num_threads(GOLDEN_THREADS)
    ref = refshim.load_reference()
    try:
        g = _reference_outputs(ref, Wt.make_prop_state_dict(1234), Wt.make_fusion_state_dict(4321))
    finally:
        ref._restore()
    g = {k: v.numpy() if isinstance(v, torch.Tensor) else v for k, v in g.items()}
    sampled = [k for k, v in g.items() if v.dtype.kind == "f" and k != "iou"]  # every float output but the IoU values
    g.update({f"{k}_shape": np.array(g[k].shape) for k in sampled})
    g.update({k: sample(g[k]) for k in sampled})
    np.savez_compressed(OUT, **g)
    print(f"{OUT}: {os.path.getsize(OUT)} bytes, {len(g)} arrays, torch {torch.__version__}")


if __name__ == "__main__":
    main()
