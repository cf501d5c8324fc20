"""CPU tests of the host-side mirror: getInstanceInfo, input preparation, the saved-file contract,
the evaluation helpers, wall boxes, sharding, the world_size-2 gather (gloo) and the loud failure
of the product path without a GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from gapro_b200 import eval_ps_labels, gen_ps, gen_ps_utils, scannet_planes, sharding, synthetic
from oracle import gen_ps_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_get_instance_info_equals_oracle_restatement():
    sc = synthetic.make_scene(2, "small")
    pts = np.ones((len(sc.xyz_raw), 4))
    pts[:, :3] = sc.xyz_raw
    xyz = (pts @ sc.axis_align.T)[:, :3]
    a = gen_ps_utils.getInstanceInfo(xyz, sc.inst, sc.sem)
    b = O.get_instance_info(xyz, sc.inst, sc.sem)
    assert a[0] == b[0]
    for x, y in zip(a[1:], b[1:]):
        assert x.shape == y.shape and (x == y).all()
    # ids have a gap (the generator skips one id): fewer boxes than max id + 1
    assert len(a[1]) == a[0] - 1
    assert gen_ps_utils.getInstanceInfo(xyz, np.full(len(xyz), -100.0), sc.sem) is None


def test_prepare_inputs_uses_unaligned_xyz_for_features():
    sc = synthetic.make_scene(1, "tiny")
    inp = gen_ps.synthetic_inputs(sc)
    assert inp["mask_feats"].shape[1] == 6
    assert (inp["mask_feats"][:, :3] == sc.xyz_raw).all()            # Q2: concat happens before alignment
    assert not np.allclose(inp["xyz"], sc.xyz_raw)
    assert inp["xyz"].dtype == np.float64


def test_axis_align_reader(tmp_path):
    A = np.arange(16, dtype=np.float64).reshape(4, 4) / 7
    f = tmp_path / "scene0000_00.txt"
    f.write_text("colorHeight = 968\naxisAlignment = " + " ".join(repr(float(x)) for x in A.ravel()) + " \nnumDepthFrames = 5\n")
    assert (gen_ps.read_axis_align_matrix(str(f)) == A).all()


def test_load_scene_reads_the_reference_layout(tmp_path):
    """dataset/scannetv2/{train,superpoints,scans_transform} as gen_ps.py:27-69 expects them."""
    root = tmp_path / "dataset" / "scannetv2"
    for sub in ("train", "superpoints", "scans_transform/scene0000_00"):
        (root / sub).mkdir(parents=True)
    sc = synthetic.make_scene(9, "tiny")
    fn = str(root / "train" / "scene0000_00_inst_nostuff.pth")
    torch.save((sc.xyz_raw, sc.rgb, sc.sem, sc.inst), fn)
    torch.save(sc.spp, str(root / "superpoints" / "scene0000_00.pth"))
    (root / "scans_transform" / "scene0000_00" / "scene0000_00.txt").write_text(
        "axisAlignment = " + " ".join(repr(float(x)) for x in sc.axis_align.ravel()) + "\n")
    inp, sem, inst = gen_ps.load_scene(fn, "scene0000_00", data_root=str(root))
    ref = gen_ps.prepare_inputs(sc.xyz_raw, sc.rgb, sc.sem, sc.inst, sc.spp, sc.axis_align)
    for k in ("xyz", "mask_feats", "spp", "instance_cls", "instance_box", "instance_box_volume"):
        assert (np.asarray(inp[k]) == np.asarray(ref[k])).all(), k
    assert len(inp["wall_box"]) == 0 and (sem == sc.sem).all() and (inst == sc.inst).all()
    assert os.path.basename(fn)[:12] == "scene0000_00"


def test_saved_file_contract_roundtrip(tmp_path):
    """What ISBNet/isbnet/data/scannetv2.py:46-48 and SPFormer/spformer/dataset/scannetv2.py:275-277 do."""
    N, S = 1000, 40
    res = (torch.randint(-1, 19, (N,), dtype=torch.int32), torch.randint(-1, 5, (N,), dtype=torch.int32),
           torch.rand(N), torch.rand(S), torch.rand(S))
    path = str(tmp_path / "scene0000_00.pth")
    gen_ps.save_pseudo_labels(path, res)
    semantic_label, instance_label, prob_label, mu_label, var_label = torch.load(path, weights_only=False)
    assert semantic_label.dtype == np.int32 and instance_label.dtype == np.int32
    assert prob_label.dtype == mu_label.dtype == var_label.dtype == np.float32
    assert semantic_label.shape == (N,) and mu_label.shape == (S,)
    dense = torch.randint(0, S, (N,))
    gen_ps.save_pseudo_labels(path, res, per_point_uncertainty=True, spp_dense=dense)
    out = torch.load(path, weights_only=False)
    assert out[3].shape == (N,) and (out[3] == res[3][dense].numpy()).all()
    valid = np.random.default_rng(0).random(N) < 0.5          # the loaders' crop indexing
    assert out[3][valid].shape == semantic_label[valid].shape


def test_miou_scene_against_brute_force():
    g = torch.Generator().manual_seed(0)
    N = 3000
    inst = torch.randint(-1, 6, (N,), generator=g)
    inst[inst == 3] = -100                                           # unused id
    sem = torch.randint(0, 4, (N,), generator=g)
    ps_inst = torch.randint(-1, 5, (N,), generator=g)
    ps_sem = torch.randint(0, 4, (N,), generator=g)
    got = eval_ps_labels.get_miou_scene(sem, inst, ps_sem, ps_inst)
    exp = []
    for i in range(int(inst.max()) + 1):
        mi = inst == i
        if not mi.any():
            continue
        ci = sem[torch.nonzero(mi)[0, 0]]
        best = 0.0
        for j in range(int(ps_inst.max()) + 1):
            mj = ps_inst == j
            if not mj.any() or ps_sem[torch.nonzero(mj)[0, 0]] != ci:
                continue
            best = max(best, float((mi & mj).sum()) / (float((mi | mj).sum()) + 1e-4))
        exp.append(best)
    assert np.allclose(got.numpy(), np.array(exp), atol=1e-6)
    conf = eval_ps_labels.get_scene_sem_conf(sem, ps_sem.clone(), num_classes=19)
    assert int(conf.sum()) == N and conf.shape == (19, 19)


def test_wall_boxes_from_planes_json(tmp_path):
    # one vertical wall quad (x = 1 plane, 4 m long, 2.5 m high), one horizontal quad, one triangle
    verts = [[1, 0, 0], [1, 0, -4], [1, 2.5, -4], [1, 2.5, 0], [0, 0, 0], [3, 0, 0], [3, 0, -3], [0, 0, -3]]
    plane = {"verts": verts, "quads": [[0, 1, 2, 3], [4, 5, 6, 7], [0, 1, 2]]}
    cls, boxes, vol = scannet_planes.wall_boxes_from_planes(plane, np.eye(4))
    assert len(boxes) == 1 and cls.tolist() == [18]
    assert np.allclose(boxes[0], [1, 0, 0, 1, 4, 2.5], atol=1e-6) and np.allclose(vol, [0.0])
    assert scannet_planes.get_wall_boxes("scene9999_99", planes_root=str(tmp_path)) == ([], [], [])


def test_cli_flags_match_reference():
    src = open(os.path.join(ROOT, "gapro_b200", "gen_ps.py")).read()
    for flag in ("--save_folder", "--use_deepfeat", "--deepfeat_folder", "--eval_pslabel"):
        assert flag in src
    assert "gaussian_process_kl_pseudo_labels" in src and "pretrain_maskfeats2" in src


def test_sharding_covers_every_scene_once():
    items = [f"scene{i:04d}_00" for i in range(1201)]
    for world in (1, 2, 4, 8):
        parts = [sharding.shard_scenes(items, r, world) for r in range(world)]
        assert sorted(sum(parts, [])) == items
        assert max(map(len, parts)) - min(map(len, parts)) <= 1
    costs = np.random.default_rng(0).pareto(1.5, len(items)) + 1
    parts = [sharding.shard_scenes(items, r, 8, costs) for r in range(8)]
    assert sorted(sum(parts, [])) == items
    loads = [sum(costs[items.index(x)] for x in p) for p in parts]
    assert max(loads) / (sum(loads) / 8) < 1.1        # LPT keeps the ranks balanced
    # the job the bench shards: per-scene cost ~ sum M^3, heavy-tailed over orders of magnitude (SURVEY 8e)
    c = sharding.COST_PER_M3 * np.random.default_rng(1).lognormal(23.0, 1.2, 1201)
    for world in (2, 4, 8):
        assign = sharding.lpt_assignment(c, world)
        assert sorted(sum(assign, [])) == list(range(1201))
        assert sharding.balance_stats(c, assign)["max_over_mean"] <= 1.05
        assert all(list(c[a]) == sorted(c[a], reverse=True) for a in assign)       # heavy scenes first
    assert sharding.scene_cost(1e10, 150_000, 40) > sharding.scene_cost(1e9, 150_000, 40) > 0


WORKER = r"""
import os, sys
sys.path.insert(0, {root!r})
import torch.distributed as dist
from gapro_b200 import sharding
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=2)
items = ["scene%04d_00" % i for i in range(11)]
mine = sharding.shard_scenes(items, dist.get_rank(), 2)
records = sharding.gather_records([(s, len(s), dist.get_rank()) for s in mine], 2)
assert sorted(r[0] for r in records) == items, records
assert {{r[2] for r in records}} == {{0, 1}}
# the cost pass of the CLI / bench: every rank estimates its round-robin share, ONE gather, LPT on every rank
est = {{s: float(int(s[5:9]) % 7 + 1) for s in items[dist.get_rank()::2]}}
merged = {{}}
for d in sharding.gather_records([est], 2):
    merged.update(d)
costs = [merged[s] for s in items]
assign = sharding.lpt_assignment(costs, 2)
both = sharding.gather_records([assign], 2)
assert both[0] == both[1] and sorted(assign[0] + assign[1]) == list(range(11))
assert sharding.balance_stats(costs, assign)["max_over_mean"] < 1.1
dist.barrier()
dist.destroy_process_group()
print("ok")
"""


def test_two_rank_gather_over_gloo(tmp_path):
    port = 29500 + os.getpid() % 2000
    script = tmp_path / "w.py"
    script.write_text(WORKER.format(root=ROOT, port=port))
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                              text=True) for r in range(2)]
    outs = [p.communicate(timeout=180)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    assert all("ok" in o for o in outs)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_product_path_fails_loudly_without_gpu():
    from gapro_b200 import _lib
    from gapro_b200.engine import get_engine
    with pytest.raises(_lib.GaproError):
        get_engine()
    sc = gen_ps.synthetic_inputs(synthetic.make_scene(0, "tiny"))
    t = gen_ps.to_scene_inputs(sc, "cpu")
    with pytest.raises(_lib.GaproError):
        gen_ps_utils.gen_pseudo_label_gaussian_process(t.coords_float, t.mask_feats, t.spp, t.instance_cls, t.instance_box,
                                                       t.instance_box_volume, t.wall_box, t.wall_box_volume)
    from gapro_b200.gaussian_process_utils import fit_gp_spp
    with pytest.raises(_lib.GaproError):
        fit_gp_spp(None, torch.zeros(4, 6), torch.tensor([0]), torch.tensor([1]), torch.tensor([2]))


def test_no_product_module_imports_the_oracle():
    for fn in os.listdir(os.path.join(ROOT, "gapro_b200")):
        if fn.endswith(".py"):
            text = open(os.path.join(ROOT, "gapro_b200", fn)).read()
            assert "import oracle" not in text and "from oracle" not in text, fn


def test_bench_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs next to ours): exactly one JSON line on stdout with
    the keys of the bench contract, kind "port", zero transfer bytes."""
    import json
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "tiny",
                        "--scenes", "1", "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "scenes/s" and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "scenes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["value"] > 0 and "workload" in d["config"]


def test_bench_dump_outputs_is_float32_seeded_and_capped(tmp_path):
    """bench.py --dump-outputs: one float32 file per output field with the scenes in job order; a field over its share
    of the byte cap is cut to the same positions on every call, shared by the per-point fields."""
    import bench
    g = torch.Generator().manual_seed(0)
    outs, off = [], 0
    for n, s in ((3000, 40), (5000, 70)):
        # prob carries the point's position in the job, so the sampled positions can be read back from it
        outs.append((torch.randint(-100, 19, (n,), dtype=torch.int32, generator=g),
                     torch.randint(-100, 30, (n,), dtype=torch.int32, generator=g),
                     torch.arange(off, off + n, dtype=torch.float32), torch.rand(s, generator=g), torch.rand(s, generator=g)))
        off += n
    cap = 5 * (128 + 4 * 1000)                  # 1000 float32 values per file
    for d in ("a", "b"):
        bench.dump_outputs(outs, str(tmp_path / d), max_bytes=cap)
    got = {k: np.load(tmp_path / "a" / f"{k}.npy") for k in bench.OUTPUT_FIELDS}
    for k, a in got.items():
        assert a.dtype == np.float32 and np.array_equal(a, np.load(tmp_path / "b" / f"{k}.npy")), k
    assert sum(os.path.getsize(tmp_path / "a" / f"{k}.npy") for k in got) <= cap
    full = {k: torch.cat([o[i] for o in outs]).numpy() for i, k in enumerate(bench.OUTPUT_FIELDS)}
    for k in ("mu", "var"):
        assert np.array_equal(got[k], full[k])
    pos = got["prob"].astype(np.int64)
    assert len(pos) == 1000 and (np.diff(pos) > 0).all()
    for k in ("sem", "inst"):
        assert np.array_equal(got[k], full[k][pos].astype(np.float32)), k


def test_bench_gpu_arm_refuses_to_run_without_a_gpu():
    import subprocess
    import sys
    if __import__("torch").cuda.is_available():
        pytest.skip("a GPU is present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)
