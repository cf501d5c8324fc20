"""Heuristic labelers over a batch of scenes: gapro_heuristic_finalize, GaproEngine.run_heuristic on many scenes,
gen_pseudo_labels_heuristic_batch and `gen_ps --label_method`.  The CPU tests check argument validation only; the
GPU tests check the batch against the per-scene oracle, the reference run and the per-scene functions."""
import os

import numpy as np
import pytest
import torch

from gapro_b200 import _lib, synthetic
from gapro_b200.gen_ps import synthetic_inputs, to_scene_inputs

GOLD = os.path.join(os.path.dirname(__file__), "golden")
METHODS = ("box2mask", "volume", "dist", "none")
DATASETS = ("scannetv2", "s3dis")


# ------------------------------------------------------------------------------------------------
# CPU: argument validation
# ------------------------------------------------------------------------------------------------
def _finalize(lib, **kw):
    """gapro_heuristic_finalize on host arrays: every call below must be rejected before touching them."""
    i32 = np.zeros(8, np.int32)
    i64 = np.zeros(8, np.int64)
    rec = np.zeros((4, 4), np.int32)
    a = dict(inst_spp=i32.ctypes.data, inst_pt=i32.ctypes.data, spp_off=i32.ctypes.data, pt_off=i64.ctypes.data,
             box_off=i32.ctypes.data, cls=i64.ctypes.data, instance_classes=18, n_scenes=1, s_total=4, n_points=4,
             spp_align=1, packed=rec.ctypes.data, sem=i32.ctypes.data, inst=i32.ctypes.data)
    a.update(kw)
    return lib.gapro_heuristic_finalize(a["inst_spp"], a["inst_pt"], a["spp_off"], a["pt_off"], a["box_off"], a["cls"],
                                        a["instance_classes"], a["n_scenes"], a["s_total"], a["n_points"],
                                        a["spp_align"], a["packed"], a["sem"], a["inst"], None)


@pytest.mark.parametrize("kw,msg", [
    (dict(box_off=None), b"null pointer"),
    (dict(cls=None), b"null pointer"),
    (dict(inst_spp=None), b"null pointer"),
    (dict(spp_off=None), b"null pointer"),
    (dict(spp_align=0, inst_pt=None), b"null pointer"),
    (dict(spp_align=0, pt_off=None), b"null pointer"),
    (dict(n_scenes=0), b"n_scenes must be positive"),
    (dict(n_scenes=-3, spp_align=0), b"n_scenes must be positive"),
    (dict(packed=None), b"missing output array"),
    (dict(spp_align=0, sem=None), b"missing output array"),
    (dict(spp_align=0, inst=None), b"missing output array"),
    (dict(s_total=0), b"empty batch"),
    (dict(spp_align=0, n_points=0), b"empty batch"),
])
def test_finalize_rejects_bad_arguments(lib, kw, msg):
    assert _finalize(lib, **kw) == -1          # GAPRO_ERR_INVALID
    assert msg in lib.gapro_last_error()
    with pytest.raises(_lib.GaproError, match="gapro_heuristic_finalize"):
        _lib.check(_finalize(lib, **kw), "gapro_heuristic_finalize")


def test_parser_label_method():
    from gapro_b200.gen_ps import parse_args
    assert parse_args([]).label_method == "gp"
    for m in METHODS:
        assert parse_args(["--label_method", m]).label_method == m
    assert parse_args(["--label_method", "gp", "--use_deepfeat"]).use_deepfeat
    with pytest.raises(SystemExit):
        parse_args(["--label_method", "gp_box"])
    for m in METHODS:
        with pytest.raises(SystemExit):
            parse_args(["--label_method", m, "--use_deepfeat"])


def test_batch_api_rejects_unknown_method():
    from gapro_b200.gen_ps_utils import gen_pseudo_labels_heuristic_batch
    with pytest.raises(ValueError, match="unknown heuristic method"):
        gen_pseudo_labels_heuristic_batch([], method="gp")
    with pytest.raises(ValueError):
        gen_pseudo_labels_heuristic_batch([], method="smallest")


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _oracle(inp, method, ds):
    from oracle import heuristic_oracle as H
    args = (inp["xyz"], inp["spp"], inp["instance_cls"].astype(np.int64), inp["instance_box"].astype(np.float32),
            inp["instance_box_volume"].astype(np.float32))
    if method == "box2mask":
        return H.heuristic_labels(*args, dataset_name=ds, box2mask=True)
    return H.heuristic_labels(*args, dataset_name=ds, heuristic_rule=method)


def _batch(dev, inps, method, ds):
    from gapro_b200.gen_ps_utils import gen_pseudo_labels_heuristic_batch
    scenes = [to_scene_inputs(inp, dev) for inp in inps]
    out = gen_pseudo_labels_heuristic_batch(scenes, method=method, instance_classes=18, dataset_name=ds, device=dev)
    assert len(out) == len(inps)
    res = []
    for (sem, inst), inp in zip(out, inps):
        assert sem.dtype == torch.int32 and inst.dtype == torch.int32 and sem.shape == inst.shape == (len(inp["xyz"]),)
        res.append((sem.cpu().numpy(), inst.cpu().numpy()))
    return res


@pytest.fixture(scope="module")
def mixed_batch():
    """Four scenes of different sizes; the third has more than 32 boxes (two mask words for the whole batch)."""
    many = synthetic.SceneConfig(n_points=14_000, n_objects=34, s_target=600, overlap=0.5, n_nested=3)
    mid = synthetic.SceneConfig(n_points=9_000, n_objects=8, s_target=400, overlap=0.5, n_nested=1)
    inps = [synthetic_inputs(synthetic.make_scene(2, "tiny")), synthetic_inputs(synthetic.make_scene(5, "small")),
            synthetic_inputs(synthetic.make_scene(23, many)), synthetic_inputs(synthetic.make_scene(9, mid))]
    n_box = [len(inp["instance_box"]) for inp in inps]
    assert n_box[2] > 32 and max(n_box[:2] + n_box[3:]) <= 32
    assert len({len(inp["xyz"]) for inp in inps}) == 4
    return inps


@pytest.mark.gpu
@pytest.mark.parametrize("ds", DATASETS)
@pytest.mark.parametrize("method", METHODS)
def test_batch_equals_each_scene_alone(dev, lib, mixed_batch, method, ds):
    from oracle import heuristic_oracle as H
    inps = mixed_batch
    if method == "dist":
        # the per-scene source offsets of the dist rule only matter in scenes that hold multi-box points
        multi = [bool((H.point_containment(inp["xyz"], inp["instance_box"]).sum(1) > 1).any()) for inp in inps]
        assert sum(multi[1:]) >= 2, multi
    want = [_oracle(inp, method, ds) for inp in inps]
    got = _batch(dev, inps, method, ds)
    for k, ((s, i), (ws, wi)) in enumerate(zip(got, want)):
        assert np.array_equal(s, ws) and np.array_equal(i, wi), (k, method, ds)
    order = [3, 2, 0, 1]
    got_rev = _batch(dev, [inps[k] for k in order], method, ds)
    for k, (s, i) in zip(order, got_rev):
        assert np.array_equal(s, got[k][0]) and np.array_equal(i, got[k][1]), (k, method, ds)


@pytest.mark.gpu
def test_batch_equals_reference_run(dev, lib):
    ref = np.load(os.path.join(GOLD, "ref_outputs.npz"))
    names = [("tiny", 3), ("small", 4)]
    inps = [synthetic_inputs(synthetic.make_scene(seed, name)) for name, seed in names]
    for ds in DATASETS:
        for method in METHODS:
            got = _batch(dev, inps, method, ds)
            for (name, _), (sem, inst) in zip(names, got):
                key = f"{name}_b2m_{ds}" if method == "box2mask" else f"{name}_heur_{ds}_{method}"
                assert np.array_equal(sem, ref[key + "_sem"]), key
                assert np.array_equal(inst, ref[key + "_inst"]), key


def _former_torch_formulas(b, scene, box_off, cls, instance_classes):
    """The finalisation GaproEngine.run_heuristic did with torch ops before gapro_heuristic_finalize, in numpy:
    sem = -100; sem[b >= 0] = cls_of_scene[b]; sem[b == -1] = instance_classes; inst = where(b >= 0, b, -100)."""
    sem = np.full(len(b), -100, np.int32)
    pos = b >= 0
    sem[pos] = cls[box_off[scene[pos]] + b[pos]].astype(np.int32)
    sem[b == -1] = instance_classes
    return sem, np.where(pos, b, -100).astype(np.int32)


@pytest.mark.gpu
def test_finalize_kernel(dev, lib):
    stream = torch.cuda.current_stream(dev).cuda_stream
    box_off = np.array([0, 2, 5, 6], np.int32)                   # 2, 3 and 1 boxes
    cls = np.array([5, -100, 7, 9, -100, 3], np.int64)
    ic = 18
    # superpoint-aligned: 3 + 4 + 2 superpoints
    spp_off = np.array([0, 3, 7, 9], np.int32)
    inst_spp = np.array([1, -1, 0, 2, 1, -1, 0, 0, -1], np.int32)
    spp_scene = np.repeat(np.arange(3), np.diff(spp_off))
    d = lambda a: torch.from_numpy(a).to(dev)                     # noqa: E731
    packed = torch.full((len(inst_spp), 4), 77, dtype=torch.int32, device=dev)
    keep = [d(inst_spp), d(spp_off), d(box_off), d(cls)]
    assert lib.gapro_heuristic_finalize(keep[0].data_ptr(), None, keep[1].data_ptr(), None, keep[2].data_ptr(),
                                        keep[3].data_ptr(), ic, 3, len(inst_spp), 0, 1, packed.data_ptr(), None, None,
                                        stream) == 0
    p = packed.cpu().numpy()
    sem, inst = _former_torch_formulas(inst_spp, spp_scene, box_off, cls, ic)
    assert np.array_equal(p[:, 0], sem) and np.array_equal(p[:, 1], inst)
    assert (p[:, 2].view(np.float32) == 1.0).all() and (p[:, 3] == 0).all()
    assert sem[3] == -100 and inst[3] == 2 and sem[4] == 9 and sem[7] == 3     # boxes of the 2nd / 3rd scene
    # per point: 4 + 6 + 2 points, -2 = undecided under rule "none"
    pt_off = np.array([0, 4, 10, 12], np.int64)
    inst_pt = np.array([0, -2, -1, 1, 2, -2, 1, 0, -1, 2, 0, -2], np.int32)
    pt_scene = np.repeat(np.arange(3), np.diff(pt_off))
    sem_d = torch.full((12,), 77, dtype=torch.int32, device=dev)
    inst_d = torch.full((12,), 77, dtype=torch.int32, device=dev)
    keep = [d(inst_pt), d(pt_off), d(box_off), d(cls)]
    assert lib.gapro_heuristic_finalize(None, keep[0].data_ptr(), None, keep[1].data_ptr(), keep[2].data_ptr(),
                                        keep[3].data_ptr(), ic, 3, 0, 12, 0, None, sem_d.data_ptr(), inst_d.data_ptr(),
                                        stream) == 0
    sem, inst = _former_torch_formulas(inst_pt, pt_scene, box_off, cls, ic)
    assert np.array_equal(sem_d.cpu().numpy(), sem) and np.array_equal(inst_d.cpu().numpy(), inst)
    assert (sem[inst_pt == -2] == -100).all() and (inst[inst_pt == -2] == -100).all()
    assert sem[4] == -100 and inst[4] == 2 and sem[6] == 9 and sem[10] == 3


def _run_cli(args):
    from gapro_b200 import gen_ps
    gen_ps.main(args)
    torch.cuda.synchronize()


def _files(folder, scans):
    return {scan: torch.load(os.path.join(folder, f"{scan}.pth"), weights_only=False) for scan in scans}


@pytest.mark.gpu
@pytest.mark.parametrize("method", METHODS)
def test_cli_heuristic_labels(dev, lib, tmp_path, monkeypatch, method):
    from gapro_b200.gen_ps import DATA_ROOT, load_scene
    from gapro_b200.gen_ps_utils import gen_pseudo_label, gen_pseudo_label_box2mask
    from tests.golden.hand_cases import CLI_SCANS, write_cli_dataset
    write_cli_dataset(tmp_path)
    monkeypatch.chdir(tmp_path)
    for k, v in (("RANK", "0"), ("WORLD_SIZE", "1"), ("LOCAL_RANK", "0")):
        monkeypatch.setenv(k, v)
    out = tmp_path / "out"
    out.mkdir()
    torch.save(("sentinel",), str(out / f"{CLI_SCANS[1]}.pth"))
    _run_cli(["--save_folder", "out", "--label_method", method, "--eval_pslabel", "--batch_scenes", "2"])
    assert torch.load(str(out / f"{CLI_SCANS[1]}.pth"), weights_only=False) == ("sentinel",)
    scans = [CLI_SCANS[0], CLI_SCANS[2]]
    files = _files(str(out), scans)
    for scan, tup in files.items():
        inp, _, _ = load_scene(os.path.join(DATA_ROOT, "train", f"{scan}_inst_nostuff.pth"), scan)
        sc = to_scene_inputs(inp, dev)
        args = (sc.coords_float, sc.spp, sc.instance_cls, sc.instance_box, sc.instance_box_volume)
        want = (gen_pseudo_label_box2mask(*args) if method == "box2mask" else
                gen_pseudo_label(*args, heuristic_rule=method))
        N, S = len(inp["xyz"]), len(np.unique(inp["spp"]))
        assert len(tup) == 5 and all(isinstance(a, np.ndarray) for a in tup)
        sem, inst, prob, mu, var = tup
        assert [a.dtype for a in tup] == [np.int32, np.int32, np.float32, np.float32, np.float32]
        assert np.array_equal(sem, want[0].cpu().numpy()) and np.array_equal(inst, want[1].cpu().numpy()), scan
        assert prob.shape == (N,) and (prob == 1).all()
        assert mu.shape == var.shape == (S,) and (mu == -100).all() and (var == -100).all()
    # nothing left to do: the files stay as they are
    mtimes = {s: os.path.getmtime(out / f"{s}.pth") for s in scans}
    _run_cli(["--save_folder", "out", "--label_method", method])
    assert mtimes == {s: os.path.getmtime(out / f"{s}.pth") for s in scans}
    # boxes derived on the device: identical files
    _run_cli(["--save_folder", "out_dev", "--label_method", method, "--device_boxes"])
    for scan, tup in _files(str(tmp_path / "out_dev"), CLI_SCANS).items():
        ref = files.get(scan)
        if ref is not None:
            assert all(a.dtype == b.dtype and np.array_equal(a, b) for a, b in zip(tup, ref)), scan
    # mu / var per point
    _run_cli(["--save_folder", "out_pp", "--label_method", method, "--per_point_uncertainty"])
    for scan, tup in _files(str(tmp_path / "out_pp"), scans).items():
        N = len(files[scan][0])
        assert np.array_equal(tup[0], files[scan][0]) and np.array_equal(tup[1], files[scan][1])
        assert tup[3].shape == tup[4].shape == (N,) and (tup[3] == -100).all() and (tup[4] == -100).all()
