"""CPU: UNCHANGED caller files of the reference, loaded straight from a checkout of it, running on top of
THIS repository's import-path shims (`model.propagation.prop_net`, `model.aggregate`,
`model.s2m.s2m_network`, `util.tensor_util` resolve to mivos_b200) — the drop-in claim of SURVEY §8(b)
exercised literally.  The networks run over the emulated C-ABI operators (tests/abi_emulator.py); the
same callers run on the real kernels wherever a B200 and the reference tree are both present.

  * generation/fusion_generator.py   FusionGenerator (second client of the propagation surface, §8f-1)
  * interact/s2m_controller.py       S2MController (per-object loop over `s2m_net(inputs)`, §8f-3)
  * interact/interaction.py          ScribbleInteraction.predict (GUI: controller + aggregate_wbg(hard))
  * davis_processor.py               DAVISProcessor.interact (DAVIS interactive track)
Those tests execute the reference's own source, which this repository does not contain: they run where a
checkout of the reference is given (oracle/refshim.py) and skip elsewhere.  The import-path overlay and the
IoU helpers are checked everywhere, against a stand-in checkout and the reference's stored results.
"""
import importlib.util
import os
import sys
import types

import numpy as np
import pytest
import torch

import abi_emulator
from oracle import refshim

needs_reference = pytest.mark.skipif(not refshim.available(),
                                     reason="runs the reference's own caller files: needs a checkout of the reference")
REF = refshim.REF_ROOT


def _load(relpath, name):
    spec = importlib.util.spec_from_file_location(name, os.path.join(REF, relpath))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.fixture()
def rt(monkeypatch):
    return abi_emulator.install_host_runtime(monkeypatch)


@needs_reference
def test_reference_fusion_generator_runs_on_our_surface(rt, prop_sd):
    from oracle import stm_oracle as O, weights as Wt
    from test_gpu_clients import fusion_generator_flow
    import model.propagation.prop_net as shim
    assert shim.PropagationNetwork is rt.PropagationNetwork  # the caller's import resolves to this repository
    fg = _load("generation/fusion_generator.py", "_ref_caller_fusion_generator")
    assert fg.PropagationNetwork is rt.PropagationNetwork and fg.aggregate_wbg is rt.aggregate_wbg
    net = rt.PropagationNetwork(top_k=50, act_dtype=torch.float32)
    net.load_state_dict(prop_sd, strict=True)
    images, mask = Wt.synthetic_clip(5, 128, 168, 2, seed=31)
    soft = mask[1:] * 0.8 + 0.05
    gen = fg.FusionGenerator(net, images, mem_freq=2)
    gen.reset(2)
    out = gen.interact_mask(soft, 2, 0, 4)
    assert out.shape == (3, 5, 128, 168)
    api = types.SimpleNamespace(pad_divide_by=O.pad_divide_by, aggregate_wbg=O.aggregate_wbg,
                                memorize=lambda f, m: O.memorize(prop_sd, f, m),
                                get_query_values=lambda f: O.get_query_values(prop_sd, f),
                                segment_with_query=lambda *a: O.segment_with_query(prop_sd, *a, top_k=50))
    want = fusion_generator_flow(api, images, soft, 2, 0, 4, mem_freq=2)[:, :, 0, :, 4:-4]
    d = (out - want).abs()
    assert float(d.max()) <= 3e-2 and float(d.mean()) <= 1e-3


@needs_reference
def test_reference_s2m_controller_runs_on_our_network(rt, golden):
    from oracle import weights as Wt
    ctl = _load("interact/s2m_controller.py", "_ref_caller_s2m_controller")
    assert ctl.S2M is rt.s2m.deeplabv3plus_resnet50  # `from model.s2m.s2m_network import deeplabv3plus_resnet50 as S2M`
    net = ctl.S2M()
    net.act_dtype = torch.float32
    net.load_state_dict(Wt.make_s2m_state_dict(), strict=True)
    g = golden("s2m_controller.npz")
    c = ctl.S2MController(net, int(g["k"]), ignore_class=255, device="cpu")
    m = c.interact(torch.from_numpy(g["image"]), torch.from_numpy(g["prev"]), g["scr"])
    assert m.shape == g["mask"].shape and float((m - torch.from_numpy(g["mask"])).abs().max()) <= 2e-2


@needs_reference
def test_reference_scribble_interaction_runs_on_our_surface(rt, golden, monkeypatch):
    """interact/interaction.py ScribbleInteraction: strokes drawn with cv2 -> controller.interact ->
    aggregate_wbg(hard=True), with our S2MController / S2MNetwork / aggregate behind the reference's imports."""
    from oracle import s2m_oracle as S, stm_oracle as O, weights as Wt
    from oracle.gen_golden_egress import load_reference_utils
    iu, _ = load_reference_utils()
    monkeypatch.setitem(sys.modules, "interact.interactive_utils", iu)  # the one reference module our interact/ shim lacks
    inter = _load("interact/interaction.py", "_ref_caller_interaction")
    assert inter.aggregate_wbg is rt.aggregate_wbg
    sd = Wt.make_s2m_state_dict()
    net = rt.S2MNetwork(act_dtype=torch.float32)
    net.load_state_dict(sd, strict=True)
    K, h, w = 2, 60, 90  # padded to 64 x 96
    image = torch.randn((1, 3, 64, 96), generator=torch.Generator().manual_seed(4))
    prev = torch.zeros((1, 64, 96), dtype=torch.uint8)
    si = inter.ScribbleInteraction(image, prev, (h, w), rt.S2MController(net, K, ignore_class=255, device="cpu"), K)
    for k, pts in ((1, [(10, 12), (40, 14), (60, 30)]), (2, [(20, 50), (70, 52)]), (0, [(5, 5), (30, 6)])):
        for x, y in pts:
            si.push_point(x, y, k)
        si.end_path()
    out = si.predict()
    assert out.shape == (K + 1, 1, 64, 96) and float((out.sum(0) - 1).abs().max()) <= 1e-5
    prob = S.s2m_controller_interact(sd, image, prev.long(), si.drawn_map, K)
    want = O.aggregate_wbg(prob, keep_bg=True, hard=True)
    assert float((out.argmax(0) != want.argmax(0)).float().mean()) <= 1e-2
    assert float((si.out_prob - prob).abs().max()) <= 2e-2


# the modules the overlay test imports, at their places in the reference's tree (every package has an __init__.py)
_CHECKOUT_FILES = ("inference_core.py", "interact/__init__.py", "interact/s2m_controller.py", "interact/timer.py",
                   "util/__init__.py", "util/tensor_util.py", "util/palette.py", "util/hyper_para.py", "model/__init__.py",
                   "model/aggregate.py", "model/fusion_net.py", "model/attn_network.py", "model/s2m/__init__.py",
                   "model/s2m/s2m_network.py", "model/propagation/__init__.py", "model/propagation/prop_net.py")


def test_pythonpath_overlay_resolves_modules_as_documented(tmp_path):
    """INTEGRATION.md §1: with this repository BEFORE the reference checkout on PYTHONPATH, the modules this
    repository provides resolve here and every other module of the same packages still resolves to the
    reference (the shim packages extend their __path__ over later sys.path entries).  The checkout is a
    stand-in with the reference's layout: empty modules at the reference's paths, same-named ones included."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    checkout = tmp_path / "reference"
    for rel in _CHECKOUT_FILES:
        (checkout / rel).parent.mkdir(parents=True, exist_ok=True)
        (checkout / rel).touch()
    (tmp_path / "cwd").mkdir()
    code = (
        "import inference_core, interact.s2m_controller as a, interact.timer as t, util.tensor_util as u, util.palette as p\n"
        "import model.aggregate as ag, model.fusion_net as fn, model.attn_network as an, model.s2m.s2m_network as sn\n"
        "import model.propagation.prop_net as pn, util.hyper_para as hp\n"
        "from util.tensor_util import pad_divide_by, unpad, unpad_3dim, compute_tensor_iou  # davis_processor.py:9, interactive_gui.py:35\n"
        "from util.palette import pal_color_map  # interactive_gui.py:36\n"
        "for m in (inference_core, a, u, p, ag, fn, an, sn, pn): print('ours', m.__file__)\n"
        "for m in (t, hp): print('ref', m.__file__)\n")
    env = dict(os.environ, PYTHONPATH=root + os.pathsep + str(checkout))
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=tmp_path / "cwd", timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = r.stdout.strip().splitlines()
    assert len(lines) == 11
    for ln in lines:
        kind, path = ln.split(" ", 1)
        assert path.startswith(root if kind == "ours" else str(checkout)), ln


def test_iou_helpers_equal_the_reference(golden):
    """Every IoU helper on the inputs of oracle/gen_golden_live.py equals what the reference's
    util/tensor_util.py returned for them (tests/golden/reference_live.npz)."""
    from oracle import gen_golden_live as L
    from util import tensor_util as ours
    ref = golden("reference_live.npz")
    assert np.array_equal(L.iou_values(ours), ref["iou"])
    seg_np, gt_np = L.iou_inputs()[:2]
    for a in ours.compute_tensor_iu(torch.from_numpy(seg_np), torch.from_numpy(gt_np)):
        assert str(a.dtype) == str(ref["iou_tensor_iu_dtype"])
    empty = np.zeros((4, 4), dtype=bool)
    assert ours.compute_np_iou(empty, empty) == 1.0  # 0/0 -> (0 + eps) / (0 + eps)


def _scribble(t, idx, label_map):
    """What DavisInteractiveSession hands out: one non-empty entry per interaction; our stand-in for
    davisinteractive.utils.scribbles.scribbles2mask returns the label map stored in it."""
    s = [[] for _ in range(t)]
    s[idx] = [label_map]
    return {"scribbles": s}


def _fake_davisinteractive(monkeypatch):
    pkg, utils, scr = types.ModuleType("davisinteractive"), types.ModuleType("davisinteractive.utils"), types.ModuleType(
        "davisinteractive.utils.scribbles")
    scr.scribbles2mask = lambda scribble, size: [scribble["scribbles"][0][0]]
    pkg.utils, utils.scribbles = utils, scr
    for name, mod in (("davisinteractive", pkg), ("davisinteractive.utils", utils), ("davisinteractive.utils.scribbles", scr)):
        monkeypatch.setitem(sys.modules, name, mod)


@needs_reference
def test_reference_davis_processor_runs_on_our_surface(rt, ref_outputs, prop_sd, fuse_sd, monkeypatch):
    """davis_processor.py UNCHANGED (the junction between the DAVIS interactive track and InferenceCore:
    S2M per object -> aggregate_wbg(hard) -> update_mask_only x2 -> interact), once on the reference's own
    modules (live, `ref_outputs`) and once on this repository's shims; only `davisinteractive` (absent
    from the image) is replaced by a stand-in that returns prepared scribble label maps."""
    from oracle import weights as Wt
    _fake_davisinteractive(monkeypatch)
    dp = _load("davis_processor.py", "_ref_caller_davis_processor")
    assert dp.InferenceCore is rt.InferenceCore and dp.S2M is rt.s2m.deeplabv3plus_resnet50
    net = rt.PropagationNetwork(top_k=20, act_dtype=torch.float32)
    net.load_state_dict(prop_sd, strict=True)
    fuse = rt.FusionNet()
    fuse.load_state_dict(fuse_sd, strict=True)
    s2m = rt.S2MNetwork(act_dtype=torch.float32)
    s2m.load_state_dict(Wt.make_s2m_state_dict(), strict=True)
    images, scribbles, want = ref_outputs
    proc = dp.DAVISProcessor(net, fuse, s2m, images, 2, device="cpu")
    for (idx, lab), (w_masks, w_next, w_idx) in zip(scribbles, want):
        masks, nxt, got_idx = proc.interact(_scribble(images.shape[1], idx, lab))
        assert (nxt, got_idx) == (w_next, w_idx) and masks.shape == w_masks.shape == (images.shape[1], 64, 90)
        mism = float((masks != w_masks).mean())
        print(f"davis_processor interaction on frame {idx}: next={nxt} mask mismatch {mism:.4f}")
        # S2M logits of a RANDOM network sit close to the decision boundary, the x1000 "hard" aggregation
        # turns them into one-hot masks and propagation spreads every flipped pixel: low-resolution,
        # random-weight bound as in test_gpu_network.py (<= 5 % for frames that went through fusion / S2M)
        assert mism <= 5e-2


@pytest.fixture()
def ref_outputs(prop_sd, fuse_sd, monkeypatch):
    """The same three interactions on the UNMODIFIED reference stack (reference InferenceCore, networks, S2M)."""
    from oracle import weights as Wt
    _fake_davisinteractive(monkeypatch)
    images, _ = Wt.synthetic_clip(7, 64, 90, 2, seed=88)  # 90 -> padded to 96 by DAVISProcessor
    labs = []
    for i in range(3):
        lab = np.full((64, 90), -1, dtype=np.int64)
        lab[10 + 4 * i:13 + 4 * i, 8:40] = 1
        lab[40:43, 30 + 5 * i:80] = 2
        lab[55:57, 5:30] = 0
        labs.append(lab)
    scribbles = [(3, labs[0]), (3, labs[1]), (3, labs[2])]  # davis_schedule: the third interaction propagates
    r = refshim.load_reference()
    try:
        with refshim.reference_on_path():
            import importlib
            rdp = importlib.import_module("davis_processor")
            from model.s2m.s2m_network import deeplabv3plus_resnet50 as S2M
            sys.modules.pop("davis_processor", None)
            s2m = S2M().eval()
            s2m.load_state_dict(Wt.make_s2m_state_dict(), strict=True)
            proc = rdp.DAVISProcessor(r.build_prop(prop_sd, top_k=20), r.build_fusion(fuse_sd), s2m, images, 2, device="cpu")
            want = [proc.interact(_scribble(7, idx, lab)) for idx, lab in scribbles]
    finally:
        r._restore()
    assert want[0][1] == [3] and want[2][1] is None  # two instant updates, then a propagation
    return images, scribbles, [(m.copy(), n, i) for m, n, i in want]
