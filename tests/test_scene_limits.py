"""The scene stages at the limits of their compiled builds, against the numpy oracle computed here.

* 129-256 boxes per scene: the WORDS = 8 builds of k_occupancy, k_grid_build / k_occ_points / k_occ_finalize and
  k_heuristic, and the 256-wide inter_cnt stride of the host event enumeration, gapro_compact_lists and
  gapro_resolve_spp.  128 boxes (WORDS = 4, the floor on bit 127) is the neighbour below the step.
* gapro_pool_feats at feature widths other than 6 and 32 (the runtime-D kernel, > 48 KB of shared memory from
  D = 49), on superpoints of 1, 31, 32, 33 and thousands of points.
* Point totals that are not a multiple of 4 (the scalar tail of k_broadcast), one-point scenes and a chunk of the
  point-order path spanning 40 scenes, a flat scene (zero extent on z) and box faces on the grid-cell boundaries of
  the point-order path.

Integer and index results and the pooled float32 features are compared bit for bit; the one end-to-end GP check uses
the criteria of the parity suite (labels exact above a posterior margin of 1e-6, mu / var / prob within 1e-5)."""
import numpy as np
import pytest
import torch

from gapro_b200 import _lib, synthetic
from gapro_b200.gen_ps import synthetic_inputs, to_scene_inputs
from tests.conftest import oracle_args, rel_err

EPS = 1e-6
METHODS = ("box2mask", "volume", "dist", "none")
DATASETS = ("scannetv2", "s3dis")
POOL_WIDTHS = (1, 3, 7, 31, 33, 48, 49, 63, 64)


def fake_fit(X, n1, Xt, nz):
    n = len(Xt)
    return dict(conf=np.full(n, 0.75, np.float32), label=np.ones(n, bool), mu=np.zeros(n, np.float32),
                var=np.ones(n, np.float32))


def unpack_bits(bits, B):
    bits = bits.cpu().numpy().view(np.uint32)
    cols = [((bits[:, b // 32] >> (b % 32)) & 1).astype(bool) for b in range(B)]
    return np.stack(cols, 1)


def room_config(n_objects, n_points=80_000):
    """A large room with many small boxes: n_objects instance boxes, 4 walls and the floor slab."""
    return synthetic.SceneConfig(n_points=n_points, n_objects=n_objects, s_target=4000, overlap=0.5, n_nested=10,
                                 room=((22, 26), (16, 20), (2.6, 3.2)), size_range=(0.3, 1.2))


def stage_oracle(inp, noise_seed):
    from oracle import gen_ps_oracle as O
    return O.gen_pseudo_label_oracle(*oracle_args(inp), thresh_spp_occu=0.999, fit_fn=fake_fit, noise_seed=noise_seed,
                                     return_debug=True)


def assert_stages(dbg, i, inp, od, p0):
    """Scene i of a batch (its points start at p0) against the oracle: densified ids, boxes, per-box counts,
    occupancy bits, pooled features, events and each GP region's index lists."""
    s0, s1 = int(dbg.spp_off[i]), int(dbg.spp_off[i + 1])
    b0, b1 = int(dbg.box_off[i]), int(dbg.box_off[i + 1])
    B, n = b1 - b0, len(inp["xyz"])
    assert s1 - s0 == len(od["n_bbs"]) and B == len(od["boxes"])
    assert (dbg.spp_gid.cpu().numpy()[p0:p0 + n] - s0 == od["spp_dense"]).all()
    assert (dbg.boxes[b0:b1] == od["boxes"]).all() and (dbg.boxes_vol[b0:b1] == od["boxes_vol"]).all()
    assert (dbg.cnt_in.cpu().numpy()[s0:s1, :B] == od["cnt_in"]).all()
    assert (dbg.cnt_in.cpu().numpy()[s0:s1, B:] == 0).all()
    assert (unpack_bits(dbg.occ_bits[s0:s1], B) == od["occ_spp"]).all()
    assert (dbg.n_bbs.cpu().numpy()[s0:s1] == od["n_bbs"]).all()
    assert (dbg.feats_spp.cpu().numpy()[s0:s1].view(np.uint32) == od["feats_spp"].view(np.uint32)).all()
    kinds = {0: "nest", 1: "nest", 2: "gp"}
    assert [(kinds[k], a, b) for k, a, b in dbg.events[i]] == [(e[0], e[1], e[2]) for e in od["events"]]
    regs = [r for r in dbg.regions if r["scene"] == i]
    assert len(regs) == len(od["regions"])
    for r, o in zip(regs, od["regions"]):
        assert (r["train_idx"] == np.concatenate([o["b1_inds"], o["b2_inds"]])).all()
        assert (r["test_idx"] == o["inter"]).all() and (r["noise"] == o["noise"]).all()


# ------------------------------------------------------------------------------------------------
# CPU: argument validation
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D,msg", [(0, b"empty input"), (-1, b"empty input"), (65, b"feature dimension 65 > 64")])
def test_pool_feats_rejects_widths_outside_1_to_64(lib, D, msg):
    """Host pointers: the call must be rejected before it reaches the device."""
    buf = np.zeros(64, np.float32)
    idx = np.zeros(2, np.int32)
    assert lib.gapro_pool_feats(buf.ctypes.data, idx.ctypes.data, idx.ctypes.data, 1, D, buf.ctypes.data, None) == -1
    assert msg in lib.gapro_last_error()
    with pytest.raises(_lib.GaproError, match="gapro_pool_feats"):
        _lib.check(lib.gapro_pool_feats(buf.ctypes.data, idx.ctypes.data, idx.ctypes.data, 1, D, buf.ctypes.data,
                                        None), "gapro_pool_feats")


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def engine(dev, lib):
    from gapro_b200.engine import get_engine
    return get_engine(dev)


@pytest.fixture(scope="module")
def room_scene():
    """room_scene(K, n_points): the inputs of the seed-7 room with K instance boxes, built once."""
    cache = {}

    def get(K, n_points=80_000):
        if (K, n_points) not in cache:
            cache[K, n_points] = synthetic_inputs(synthetic.make_scene(7, room_config(K, n_points)))
        return cache[K, n_points]
    return get


@pytest.fixture(scope="module")
def room_stages(room_scene):
    """room_stages(K): (inputs, oracle debug) of the K-box room, noise seed 3, computed once."""
    cache = {}

    def get(K):
        if K not in cache:
            inp = room_scene(K)
            cache[K] = (inp, stage_oracle(inp, 3)[1])
        return cache[K]
    return get


@pytest.fixture(scope="module")
def small_stages():
    """Three small scenes of up to 11 boxes, with their oracle debug (noise seeds 11, 12, 13)."""
    out = []
    for j, (seed, name) in enumerate(((2, "tiny"), (5, "small"), (9, "tiny"))):
        inp = synthetic_inputs(synthetic.make_scene(seed, name))
        out.append((inp, stage_oracle(inp, 11 + j)[1], 11 + j))
    assert max(len(od["boxes"]) for _, od, _ in out) <= 32
    return out


# ----------------------------------------------------------------------- 129 - 256 boxes per scene
@pytest.mark.gpu
@pytest.mark.parametrize("occ_path", ["gather", "points"])
@pytest.mark.parametrize("K,words", [(123, 4), (124, 8), (196, 8), (251, 8)])
def test_stages_bit_exact_up_to_256_boxes(engine, dev, room_stages, K, words, occ_path, monkeypatch):
    """128, 129, 201 and 256 boxes (K instance boxes + 4 walls + the floor): every stage bit-exact on both
    occupancy paths.  At 129 boxes the floor is the first bit of word 4, at 256 it is bit 255."""
    monkeypatch.setattr(engine, "occupancy_path", occ_path)
    inp, od = room_stages(K)
    B = K + 5
    _, dbg = engine.run([to_scene_inputs(inp, dev, noise_seed=3)], thresh_spp_occu=0.999, training_iter=0, debug=True,
                        want_cnt_in=True)
    assert dbg.occ_bits.shape[1] == words and dbg.box_off[1] == B and len(od["boxes"]) == B
    assert_stages(dbg, 0, inp, od, 0)
    gp = [(b1, b2) for kind, b1, b2 in dbg.events[0] if kind == 2]
    assert any(B - 1 in e for e in gp)                          # the floor slab, bit 127 / 128 / 200 / 255
    if words == 8:
        assert (dbg.occ_bits.cpu().numpy()[:, 4:] != 0).any()
    if K > 128:                                                 # instance boxes in words 4..7 take part in GP regions
        assert any(128 <= b < K for e in gp for b in e)


@pytest.mark.gpu
@pytest.mark.parametrize("order", [(0, 1, 2, 3), (1, 2, 0, 3)])
def test_mixed_batch_at_eight_words(engine, dev, room_stages, small_stages, order):
    """The 201-box room with three small scenes: the small scenes run with words = 8 and use word 0 only.  Stages
    per scene against the oracle, and every output equal to the scene run alone."""
    items = [room_stages(196) + (3,)] + small_stages
    items = [items[k] for k in order]
    scenes = [to_scene_inputs(inp, dev, noise_seed=seed) for inp, _, seed in items]
    outs, dbg = engine.run(scenes, thresh_spp_occu=0.999, training_iter=1, debug=True, want_cnt_in=True)
    assert dbg.occ_bits.shape[1] == 8
    p0 = 0
    for i, (inp, od, seed) in enumerate(items):
        assert_stages(dbg, i, inp, od, p0)
        p0 += len(inp["xyz"])
        alone = engine.run([to_scene_inputs(inp, dev, noise_seed=seed)], thresh_spp_occu=0.999, training_iter=1)[0]
        for a, b in zip(alone, outs[i]):
            assert torch.equal(a, b), i


def _compare_scene(out, ref, min_margin):
    sem, inst, prob, mu, var = [t.cpu().numpy() for t in out]
    assert sem.dtype == np.int32 and inst.dtype == np.int32 and prob.dtype == np.float32
    assert mu.dtype == np.float32 and var.dtype == np.float32 and mu.shape == ref[3].shape
    g = ref[3] != -100
    assert ((mu != -100) == g).all()
    assert np.allclose(mu[g], ref[3][g], rtol=1e-4, atol=0) and np.allclose(var[g], ref[4][g], rtol=1e-4, atol=0)
    assert rel_err(mu[g], ref[3][g]) < 1e-5 and rel_err(var[g], ref[4][g]) < 1e-5
    if min_margin > EPS:
        assert (sem == ref[0]).all() and (inst == ref[1]).all()
    else:       # points decided with a posterior margin below EPS are excluded
        agree = (sem == ref[0]) & (inst == ref[1])
        assert agree.mean() > 0.999
    assert np.allclose(prob, ref[2], rtol=1e-5, atol=0)


@pytest.mark.gpu
def test_201_box_scene_end_to_end_against_float64_oracle(engine, dev, room_scene):
    """280 GP regions (M up to 1452), 74 of them with an instance box >= 128; wall and floor boxes (indices 196..200)
    decide superpoints, whose instance label must then be -100.  Three training steps: the smallest posterior margin
    is 8.4e-5, so every label is compared exactly."""
    from oracle import gen_ps_oracle as O
    K = 196
    inp = room_scene(K)
    ref, od = O.gen_pseudo_label_oracle(*oracle_args(inp), thresh_spp_occu=0.999, training_iter=3, noise_seed=3,
                                        return_debug=True)
    margin = min(np.abs(r["res"]["prob64"] - 0.5).min() for r in od["regions"])
    assert margin > EPS
    raw = od["inst_spp_raw"][od["spp_dense"]]
    assert (ref[1] >= 128).any() and ((raw >= K) & (ref[1] == -100) & (ref[0] == 18)).any()
    out = engine.run([to_scene_inputs(inp, dev, noise_seed=3)], thresh_spp_occu=0.999, training_iter=3)[0]
    assert engine.last_stats["n_regions"] == len(od["regions"])
    _compare_scene(out, ref, margin)


def _heuristic_oracle(inp, method, ds):
    from oracle import heuristic_oracle as H
    args = (inp["xyz"], inp["spp"], inp["instance_cls"].astype(np.int64), inp["instance_box"].astype(np.float32),
            inp["instance_box_volume"].astype(np.float32))
    if method == "box2mask":
        return H.heuristic_labels(*args, dataset_name=ds, box2mask=True)
    return H.heuristic_labels(*args, dataset_name=ds, heuristic_rule=method)


def _heuristic_batch(dev, inps, method, ds):
    from gapro_b200.gen_ps_utils import gen_pseudo_labels_heuristic_batch
    out = gen_pseudo_labels_heuristic_batch([to_scene_inputs(inp, dev) for inp in inps], method=method,
                                            instance_classes=18, dataset_name=ds, device=dev)
    assert len(out) == len(inps)
    return [(s.cpu().numpy(), i.cpu().numpy()) for s, i in out]


@pytest.mark.gpu
@pytest.mark.parametrize("ds", DATASETS)
@pytest.mark.parametrize("method", METHODS)
def test_heuristic_labelers_up_to_256_boxes(dev, lib, room_scene, method, ds):
    """196 and 256 instance boxes (the heuristic labelers read no wall or floor box): bit-exact against the oracle.
    In the 256-box room the vote key carries label 256 (box 255)."""
    from oracle import heuristic_oracle as H
    for K, n_points in ((196, 80_000), (256, 40_000)):
        inp = room_scene(K, n_points)
        assert len(inp["instance_box"]) == K
        if method == "dist":          # points in several boxes, some of them >= 128: the rule decides those
            occ = H.point_containment(inp["xyz"], inp["instance_box"])
            assert ((occ.sum(1) > 1) & occ[:, 128:].any(1)).any()
        want = _heuristic_oracle(inp, method, ds)
        assert (want[1] >= 128).any()
        if K == 256 and method in ("box2mask", "volume"):
            assert (want[1] == 255).any()
        (sem, inst), = _heuristic_batch(dev, [inp], method, ds)
        assert np.array_equal(sem, want[0]) and np.array_equal(inst, want[1]), (K, method, ds)


@pytest.mark.gpu
def test_heuristic_mixed_batch_at_eight_words(dev, lib, room_scene, small_stages):
    """A 251-box room between small scenes, one batch per method and dataset: every scene equals its oracle."""
    inps = [small_stages[0][0], room_scene(251, 40_000), small_stages[1][0], small_stages[2][0]]
    for ds in DATASETS:
        for method in METHODS:
            got = _heuristic_batch(dev, inps, method, ds)
            for k, ((s, i), inp) in enumerate(zip(got, inps)):
                ws, wi = _heuristic_oracle(inp, method, ds)
                assert np.array_equal(s, ws) and np.array_equal(i, wi), (k, method, ds)


@pytest.mark.gpu
def test_more_than_256_boxes_are_rejected(engine, dev):
    """257 boxes: 252 instance boxes + 4 walls + the floor on the GP path, 257 instance boxes on the heuristic path."""
    inp = synthetic_inputs(synthetic.make_scene(7, room_config(252, 20_000)))
    sc = to_scene_inputs(inp, dev)
    assert len(inp["instance_box"]) + len(inp["wall_box"]) + 1 == 257
    with pytest.raises(ValueError, match="more than 256 boxes in one scene"):
        engine.run([sc], thresh_spp_occu=0.999)
    inp = synthetic_inputs(synthetic.make_scene(7, room_config(257, 20_000)))
    with pytest.raises(ValueError, match="more than 256 boxes in one scene"):
        engine.run_heuristic([to_scene_inputs(inp, dev)])


# ------------------------------------------------------------------------------- pooling widths
@pytest.fixture(scope="module")
def pool_rows():
    """11 017 points in shuffled order over superpoints of 1, 31, 32, 33, 2000 and 2049 points plus 300 random
    ones (raw ids negative and large); 64 feature columns whose magnitudes span six decades, so that the float32
    sums depend on their order."""
    rng = np.random.default_rng(17)
    sizes = [1, 31, 32, 33, 2000, 2049, 1, 33]
    ids = np.concatenate([np.full(s, k * 7919 - 20_000, np.int64) for k, s in enumerate(sizes)])
    ids = np.concatenate([ids, rng.integers(0, 300, 11_017 - len(ids)) * 1_000_003 + 10**12])
    ids = ids[rng.permutation(len(ids))]
    feats = (rng.normal(size=(len(ids), 64)) * 10.0 ** rng.uniform(-3, 3, (len(ids), 64))).astype(np.float32)
    return ids, feats


def _pool_reference(ids, feats):
    from oracle import gen_ps_oracle as O
    _, dense = np.unique(ids, return_inverse=True)
    S = int(dense.max()) + 1
    fsum, cnt = O.scatter_sum_index_order(feats, dense, S)
    assert {1, 31, 32, 33, 2000, 2049} <= set(cnt.tolist())
    return fsum / np.maximum(cnt, 1).astype(np.float32)[:, None]


def _pool_on(device, ids, feats):
    from gapro_b200.gaussian_process_utils import _pool_by_superpoint
    with torch.cuda.device(device):
        out = _pool_by_superpoint(torch.from_numpy(feats).to(device), torch.from_numpy(ids).to(device))
        return out.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("D", POOL_WIDTHS)
def test_pool_feats_at_runtime_widths(dev, lib, pool_rows, D):
    ids, feats = pool_rows
    f = np.ascontiguousarray(feats[:, :D])
    got = _pool_on(dev, ids, f)
    want = _pool_reference(ids, f)
    assert got.shape == want.shape and (got.view(np.uint32) == want.view(np.uint32)).all()


@pytest.mark.gpu
def test_pool_feats_wide_on_two_devices(lib, pool_rows):
    """D = 64 takes 64 KB of dynamic shared memory, an attribute set per device: pool on cuda:0, on cuda:1, and on
    cuda:0 again in the same process."""
    if torch.cuda.device_count() < 2:
        pytest.skip(f"needs two visible CUDA devices, found {torch.cuda.device_count()}")
    ids, feats = pool_rows
    want = _pool_reference(ids, feats).view(np.uint32)
    for k in (0, 1, 0):
        got = _pool_on(torch.device(f"cuda:{k}"), ids, feats)
        assert (got.view(np.uint32) == want).all(), k


# --------------------------------------------------------------------- ragged and degenerate scenes
def _ragged_scene(rng, n):
    """n points (1..7) in a unit cube above a random origin; one box, or two that are disjoint or nested, all above
    the floor slab: only nest events, so the oracle's labels need no GP fit."""
    org = rng.uniform(-5, 5, 3)
    xyz = org + rng.uniform(0, 1, (n, 3))
    lo = np.array([org[0] + rng.uniform(-0.2, 0.5), org[1] + rng.uniform(-0.2, 0.5), org[2] + 0.15])
    boxes = [np.concatenate([lo, lo + rng.uniform(0.4, 1.0, 3)])]
    kind = rng.integers(3)
    if kind == 1:                          # nested: more than 0.1 inside on every side
        b = boxes[0]
        boxes.append(np.concatenate([b[:3] + 0.12, b[3:] - 0.12]))
    elif kind == 2:                        # disjoint in x
        b = boxes[0].copy()
        b[[0, 3]] += 1.2
        boxes.append(b)
    box = np.array(boxes, np.float32)
    if kind == 1 and n >= 3:               # two points inside the nested box
        xyz[:2] = 0.5 * (box[1, :3] + box[1, 3:]) + rng.uniform(-0.05, 0.05, (2, 3))
    xyz[-1, 2] = org[2]                    # the floor slab is [org_z, org_z + 0.1], below every box
    vol = np.prod(box[:, 3:] - box[:, :3], axis=1).astype(np.float32)
    spp = rng.integers(0, 3, n) * 11 - 5
    return dict(xyz=xyz, mask_feats=rng.normal(size=(n, 6)).astype(np.float32), spp=spp,
                instance_cls=rng.integers(0, 18, len(box)), instance_box=box, instance_box_volume=vol,
                wall_box=[], wall_volume=[])


@pytest.fixture(scope="module")
def ragged_scenes():
    """40 scenes of 1..7 points with their oracle output and debug."""
    rng = np.random.default_rng(23)
    out = []
    for j in range(40):
        inp = _ragged_scene(rng, 1 + (j * 5) % 7)
        ref, od = stage_oracle(inp, j)
        assert not od["regions"]
        out.append((inp, ref, od, j))
    assert sum(1 for _, _, od, _ in out if any(e[0] == "nest" for e in od["events"])) >= 5
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("occ_path", ["gather", "points"])
@pytest.mark.parametrize("tail", [1, 2, 3])
def test_batch_of_one_to_seven_point_scenes(engine, dev, ragged_scenes, occ_path, tail, monkeypatch):
    """About 40 scenes in one batch: one 1024-point chunk of the point-order path spans all of them, and the point
    total leaves 1, 2 or 3 points to the scalar tail of the broadcast.  Stages and final labels against the oracle."""
    monkeypatch.setattr(engine, "occupancy_path", occ_path)
    items = list(ragged_scenes)
    r = (sum(len(inp["xyz"]) for inp, *_ in items) - tail) % 4
    if r:                                  # leave out one scene of r (mod 4) points
        del items[next(k for k, (inp, *_) in enumerate(items) if len(inp["xyz"]) % 4 == r)]
    assert sum(len(inp["xyz"]) for inp, *_ in items) % 4 == tail and len(items) >= 39
    scenes = [to_scene_inputs(inp, dev, noise_seed=seed) for inp, _, _, seed in items]
    outs, dbg = engine.run(scenes, thresh_spp_occu=0.999, debug=True, want_cnt_in=True)
    p0 = 0
    for i, (inp, ref, od, _) in enumerate(items):
        assert_stages(dbg, i, inp, od, p0)
        p0 += len(inp["xyz"])
        got = [t.cpu().numpy() for t in outs[i]]
        assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1]), i
        assert np.array_equal(got[2].view(np.uint32), ref[2].view(np.uint32)), i
        assert np.array_equal(got[3], ref[3]) and np.array_equal(got[4], ref[4]), i


@pytest.mark.gpu
@pytest.mark.parametrize("occ_path", ["gather", "points"])
def test_flat_scene(engine, dev, occ_path, monkeypatch):
    """Every z equal: zero extent on one grid axis.  Every superpoint lies in the floor slab, so none is in one
    instance box alone and no GP region forms: the final labels are compared too."""
    monkeypatch.setattr(engine, "occupancy_path", occ_path)
    inp = synthetic_inputs(synthetic.make_scene(3, "tiny"))
    inp["xyz"] = inp["xyz"].copy()
    inp["xyz"][:, 2] = 0.6
    ref, od = stage_oracle(inp, 5)
    assert od["occ_spp"][:, -1].all() and (od["n_bbs"] > 1).any() and not od["regions"]
    outs, dbg = engine.run([to_scene_inputs(inp, dev, noise_seed=5)], thresh_spp_occu=0.999, debug=True,
                           want_cnt_in=True)
    assert_stages(dbg, 0, inp, od, 0)
    got = [t.cpu().numpy() for t in outs[0]]
    assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1]) and np.array_equal(got[2], ref[2])


STEP = 0.125                     # grid step of every axis below: 32 cells over 4 m in x / y, 8 cells over 1 m in z


def _face_box_value(target, sign):
    """A float32 box coordinate near `target` whose face after the float64 margin, b + sign * 0.005, is a multiple
    of 2**-50: grid lines that differ from it by multiples of STEP are then exact float64 values."""
    b = np.float32(target)
    while True:
        f = np.float64(b) + sign * 0.005
        if f * 2.0 ** 50 == np.floor(f * 2.0 ** 50):
            return b, f
        b = np.nextafter(b, np.float32(10))


def _grid_face_scene():
    """Boxes whose x-min, y-max and z-min faces (after the 0.005 margin) lie exactly on lines lo + i * ext / n of
    the scene's 32 x 32 x 8 grid, with points on and one ulp either side of each such face."""
    rng = np.random.default_rng(31)
    bx, fx = _face_box_value(1.05, -1)          # x-min faces: fx + k * STEP
    by, fy = _face_box_value(2.6, +1)          # y-max faces
    bz, fz = _face_box_value(1.2, -1)          # z-min faces
    lo = np.array([fx - 10 * STEP, fy - 22 * STEP, fz - 2 * STEP])
    hi = lo + np.array([32, 32, 8]) * STEP
    boxes, probes = [], []
    for k in range(8):
        x0, y1, z0 = bx + np.float32(k * STEP), by - np.float32((k % 3) * STEP), bz + np.float32((k % 2) * STEP)
        box = np.array([x0, y1 - np.float32(0.6 + 0.1 * k), z0, x0 + np.float32(0.55), y1, z0 + np.float32(0.45)],
                       np.float32)
        boxes.append(box)
        faces = (np.float64(box[0]) - 0.005, np.float64(box[4]) + 0.005, np.float64(box[2]) - 0.005)
        for ax, f in enumerate(faces):
            assert (f - lo[ax]) / STEP == round((f - lo[ax]) / STEP) and lo[ax] + round((f - lo[ax]) / STEP) * STEP == f
            mid = 0.5 * (box[:3].astype(np.float64) + box[3:].astype(np.float64))
            for v in (np.nextafter(f, -np.inf), f, np.nextafter(f, np.inf)):
                p = mid.copy()
                p[ax] = v
                probes.append(p)
    assert (hi - lo == np.array([32, 32, 8]) * STEP).all()
    box = np.stack(boxes)
    pts = np.concatenate([lo[None], hi[None], np.array(probes), lo + rng.uniform(0, 1, (3000, 3)) * (hi - lo)])
    n_probe = len(probes)
    # each probe point is a superpoint of its own; the rest are grouped at random
    spp = np.concatenate([[0, 1], 10 + np.arange(n_probe), 1000 + rng.integers(0, 150, 3000)])
    return dict(xyz=pts, mask_feats=rng.normal(size=(len(pts), 6)).astype(np.float32), spp=spp,
                instance_cls=rng.integers(0, 18, len(box)), instance_box=box,
                instance_box_volume=np.prod(box[:, 3:] - box[:, :3], axis=1).astype(np.float32),
                wall_box=[], wall_volume=[])


@pytest.mark.gpu
@pytest.mark.parametrize("occ_path", ["gather", "points"])
def test_box_faces_on_grid_cell_boundaries(engine, dev, occ_path, monkeypatch):
    monkeypatch.setattr(engine, "occupancy_path", occ_path)
    inp = _grid_face_scene()
    _, od = stage_oracle(inp, 1)
    # probe j of face ax of box k is superpoint 2 + 9k + 3ax + j: one ulp below, on, one ulp above the face; the
    # x-min and z-min faces hold the two upper probes, the y-max face the two lower ones
    want = np.array([[0, 1, 1], [1, 1, 0], [0, 1, 1]])
    for k in range(8):
        assert (od["cnt_in"][2 + 9 * k:11 + 9 * k, k].reshape(3, 3) == want).all(), k
    _, dbg = engine.run([to_scene_inputs(inp, dev, noise_seed=1)], thresh_spp_occu=0.999, training_iter=1, debug=True,
                        want_cnt_in=True)
    assert_stages(dbg, 0, inp, od, 0)
