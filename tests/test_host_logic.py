"""CPU: host-side logic -- drop-in import surface, encoder/state-dict compatibility, slab partition, MC table and
octree oracle properties."""
import json
import os
import numpy as np
import pytest
import torch

from oracle import spec
from helpers import GOLDEN, checksum


def test_dropin_import_surface():
    # the imports RTL/main.py:19-29 performs
    from monoport.lib.common.config import get_cfg_defaults
    from monoport.lib.modeling.MonoPortNet import MonoPortNet, PIFuNetG, PIFuNetC  # noqa: F401
    from monoport.lib.modeling.geometry import orthogonal, perspective  # noqa: F401
    from implicit_seg.functional import Seg3dTopk, Seg3dLossless  # noqa: F401
    from implicit_seg.functional.utils import plot_mask3D  # noqa: F401
    cfg = get_cfg_defaults()
    net = MonoPortNet(cfg.netG)
    keys = set(net.state_dict().keys())
    assert {"surface_classifier.filters.%d.%s" % (l, k) for l in range(5) for k in ("weight", "bias")} <= keys
    assert [tuple(f.weight.shape) for f in net.surface_classifier.filters] == [
        (1024, 257, 1), (512, 1281, 1), (256, 769, 1), (128, 513, 1), (1, 385, 1)]
    c = MonoPortNet(cfg.netC)
    assert [f.weight.shape[1] for f in c.surface_classifier.filters] == [513, 1537, 1025, 769, 641]


def test_encoders_match_reference_if_present():
    """For netG and netC: the reference's state dict loads strictly (same keys and shapes, aliased keys resolve to the same
    values) and the image encoder returns the reference's stage outputs (tests/golden/encoders.npz, written by
    make_golden.py from the reference).  The run is in float64 so that the stored outputs hold on any CPU: the bound is
    summation-order noise, far below any difference in what is computed."""
    g = np.load(os.path.join(GOLDEN, "encoders.npz"))
    for net in ("G", "C"):
        _check_encoder_against_golden(g, net)


def _check_encoder_against_golden(g, net):
    from monoport_b200.modeling import PIFuNetG, PIFuNetC
    layout = json.loads(str(g[net + "_layout"]))
    mine = (PIFuNetG if net == "G" else PIFuNetC)().eval().double()
    mine.load_state_dict(spec.make_encoder_state(layout, int(g["seed"])), strict=True)
    loaded = mine.state_dict()
    np.testing.assert_allclose(np.stack([checksum(loaded[k]) for k, _ in layout]), g[net + "_state_checksum"], rtol=1e-12, atol=0)
    with torch.no_grad():
        outs = [o[0] for o in mine.image_filter(spec.make_image(int(g["image_size"]), int(g["image_seed"])))]
    assert len(outs) == len(g[net + "_out_checksum"])
    idx = torch.from_numpy(g[net + "_out_index"])
    for o, want_sum, want_sample in zip(outs, g[net + "_out_checksum"], g[net + "_out_sample"]):
        assert o.dtype == torch.float64
        np.testing.assert_allclose(o.reshape(-1)[idx].numpy(), want_sample, rtol=1e-11, atol=1e-11)
        np.testing.assert_allclose(checksum(o), want_sum, rtol=1e-11, atol=1e-11)


def test_geometry_helpers_match_oracle():
    from monoport_b200.modeling.geometry import orthogonal, perspective, index
    p = spec.make_points(100, 1)
    cal = spec.scene_calib(20, 33)
    assert torch.allclose(orthogonal(p, cal)[0], spec.project_ref(p[0], cal[0]), atol=1e-6)
    cal2 = cal.clone(); cal2[0, 2, 3] = 3.0
    assert torch.allclose(perspective(p, cal2)[0], spec.project_ref(p[0], cal2[0], "perspective"), atol=1e-6)
    feat = spec.make_feat(8, 16, 16, 2)
    uv = p[:, :2]
    assert torch.allclose(index(feat, uv)[0], spec.bilinear_ref(feat[0], uv[0, 0], uv[0, 1]), atol=1e-6)
    with pytest.raises(NotImplementedError):
        orthogonal(p, cal, transforms=torch.zeros(1, 2, 3))


def test_slab_bounds():
    from monoport_b200.shard import slab_bounds, max_slab
    for R in (17, 257, 513):
        for ws in (1, 2, 4, 8):
            b = slab_bounds(R, ws)
            assert b[0][0] == 0 and sum(nz for _, nz in b) == R
            assert all(b[i][0] + b[i][1] == b[i + 1][0] for i in range(ws - 1))
            assert max(nz for _, nz in b) == max_slab(R, ws)
    assert slab_bounds(257, 8)[0] == (0, 33) and slab_bounds(257, 8)[7] == (225, 32)


@pytest.mark.parametrize("kind", ["sphere", "ellipsoid", "two_blobs"])
def test_mc_oracle_is_watertight_and_outward(kind):
    vol = spec.analytic_volume(33, kind)
    V, F = spec.marching_cubes_ref(vol)
    assert len(F) > 0 and F.min() >= 0 and F.max() == len(V) - 1
    e = np.concatenate([F[:, [0, 1]], F[:, [1, 2]], F[:, [2, 0]]])
    # every directed edge appears once and its reverse appears once: closed, consistently oriented 2-manifold
    fwd = {(a, b) for a, b in e}
    assert len(fwd) == len(e)
    assert all((b, a) in fwd for a, b in e)
    und = np.unique(np.sort(e, 1), axis=0)
    n_comp = 2 if kind == "two_blobs" else 1
    assert len(V) - len(und) + len(F) == 2 * n_comp              # Euler characteristic of n spheres
    a, b, c = V[F[:, 0]], V[F[:, 1]], V[F[:, 2]]
    assert np.einsum("ij,ij->i", a, np.cross(b, c)).sum() > 0      # positive signed volume: normals point outward
    # vertices lie on grid edges
    frac = V - np.floor(V)
    assert ((frac > 0).sum(1) <= 1).all()


def test_mc_table_shape():
    from tools.gen_mc_table import build_table
    ntri, tri, emask = build_table()
    assert ntri.max() == 5 and ntri[0] == 0 and ntri[255] == 0
    assert all(ntri[c] == ntri[255 - c] or True for c in range(256))
    # a case and its complement cut the same edges
    assert all(emask[c] == emask[255 - c] for c in range(256))


def _lookup(field):
    R = field.shape[0]

    def fn(p):
        i = ((p.double() + 1) / 2 * R - 0.5).round().long().clamp(0, R - 1)
        return field[i[:, 2], i[:, 1], i[:, 0]]
    return fn


@pytest.mark.parametrize("kind", ["sphere", "two_blobs"])
def test_octree_oracle_lossless_equals_dense(kind):
    field = torch.from_numpy(spec.analytic_volume(65, kind))
    occ, stats = spec.seg3d_lossless_ref(_lookup(field), [9, 17, 33, 65], faster=False, return_stats=True)
    assert torch.equal(occ > 0.5, field > 0.5)
    evaluated = sum(s["idx"].numel() for s in stats)
    assert evaluated < 0.2 * 65 ** 3
    # evaluated nodes carry exactly the queried values
    idx = stats[-1]["idx"]
    assert torch.equal(occ.reshape(-1)[idx], field.reshape(-1)[idx])


def test_octree_oracle_faster_and_empty():
    field = torch.from_numpy(spec.analytic_volume(65, "sphere"))
    occ, stats = spec.seg3d_lossless_ref(_lookup(field), [9, 17, 33, 65], faster=True, return_stats=True)
    assert stats[-1]["idx"].numel() == 0                       # last level is interpolated only
    assert ((occ > 0.5) != (field > 0.5)).float().mean() < 2e-3
    assert spec.seg3d_lossless_ref(_lookup(torch.zeros(65, 65, 65)), [9, 17, 33, 65]) is None
    occ2, st2 = spec.seg3d_topk_ref(_lookup(field), [9, 17, 33, 65], [0, 3000, 12000, 50000], return_stats=True)
    assert [s["idx"].numel() for s in st2] == [729, 3000, 12000, 50000]
    assert ((occ2 > 0.5) != (field > 0.5)).sum() == 0


def test_level_points_convention():
    # node centres: (c+0.5)/R mapped to [b_min,b_max]; the R (not R-1) divisor mirrors mat_color, RTL/main.py:204-209
    p = spec.level_points(torch.tensor([[0, 0, 0], [256, 256, 256]]), 257, (-1, -1, -1), (1, 1, 1))
    assert torch.allclose(p[0], torch.full((3,), -1 + 1 / 257)) and torch.allclose(p[1], torch.full((3,), 1 - 1 / 257))


def test_obj_writer_matches_reference_format(tmp_path):
    """Same bytes as monoport/lib/mesh_util.py:223-242 writes (tests/golden/obj_writer.npz)."""
    from monoport.lib.mesh_util import save_obj_mesh, save_obj_mesh_with_color
    g = np.load(os.path.join(GOLDEN, "obj_writer.npz"))
    V, Fc, C = g["V"], g["F"], g["C"]
    a, b = tmp_path / "a.obj", tmp_path / "b.obj"
    save_obj_mesh(str(a), V, Fc)
    save_obj_mesh_with_color(str(b), torch.from_numpy(V), torch.from_numpy(Fc), C)
    la, lb = a.read_text().splitlines(), b.read_text().splitlines()
    assert len(la) == 57 + 101 and la[0] == "v %.4f %.4f %.4f" % tuple(V[0]) and la[57] == "f %d %d %d" % tuple(Fc[0] + 1)
    assert lb[0] == "v %.4f %.4f %.4f %.4f %.4f %.4f" % (tuple(V[0]) + tuple(C[0]))
    assert a.read_text() == str(g["obj"]) and b.read_text() == str(g["obj_color"])


def test_bench_reference_arm_contract(tmp_path):
    """`bench.py --impl reference` (the oracle port on the host cores) prints ONE JSON line with the contract's keys, and
    `--dump-outputs` writes the volume its timed step computed."""
    import json
    import os
    import subprocess
    import sys
    from conftest import ROOT
    out = tmp_path / "out"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "occupancy_mpoints_per_s" and d["unit"] == "Mpoints/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["vs_baseline"] is None and "workload" in d["config"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["steps"] == 1 and sorted(os.listdir(out)) == ["volume.npy"]
    import bench
    _, Ws, bs, feats = bench.synthetic()
    S = 48
    pts = spec.level_points(spec._grid_coords(S, 1), S, bench.B_MIN, bench.B_MAX).t().contiguous()
    want = spec.query_ref(feats[0], pts, bench.scene_calib(), Ws, bs, spec.LAST_SIGMOID).reshape(S, S, S)
    vol = np.load(out / "volume.npy")
    assert vol.dtype == np.float32
    np.testing.assert_allclose(vol, want.numpy(), rtol=0, atol=1e-6)      # the bench may run on another thread count


def test_binary_ply_round_trip(tmp_path):
    """SURVEY.md 8f-4: binary PLY dump of reconstruction() output; float32 coordinates and topology round-trip exactly."""
    from monoport_b200.mesh_util import save_ply_mesh, load_ply_mesh
    rng = np.random.default_rng(3)
    V = rng.random((57, 3), dtype=np.float32) * 2 - 1
    Fc = rng.integers(0, 57, size=(101, 3)).astype(np.int32)
    C = rng.random((57, 3), dtype=np.float32)
    p = str(tmp_path / "m.ply")
    save_ply_mesh(p, torch.from_numpy(V), torch.from_numpy(Fc))
    v, f, c = load_ply_mesh(p)
    assert np.array_equal(v, V) and np.array_equal(f, Fc) and c is None
    save_ply_mesh(p, V, Fc, C)
    v, f, c = load_ply_mesh(p)
    assert np.array_equal(v, V) and np.array_equal(f, Fc) and np.array_equal(c, np.rint(C * 255).astype(np.uint8))
    assert open(p, "rb").read(3) == b"ply" and os.path.getsize(p) < 57 * 15 + 101 * 13 + 400
    save_ply_mesh(p, np.zeros((0, 3), np.float32), np.zeros((0, 3), np.int32))        # empty mesh
    v, f, c = load_ply_mesh(p)
    assert v.shape == (0, 3) and f.shape == (0, 3)


def test_modules_with_native_handles_copy_and_pickle():
    """ADVICE r1: nn.Modules that cache ctypes handles must survive copy.deepcopy / pickle (the handles are dropped and
    rebuilt lazily) and copy.copy must not share a handle that two __del__ calls would free twice."""
    import copy
    import pickle
    from monoport_b200.modeling import PIFuNetG
    from monoport_b200.engine import Seg3dLossless, make_query_func
    net = PIFuNetG()
    head = net.surface_classifier
    head._handle, head._handle_key = object(), ("fake",)            # pretend a native handle exists (no GPU here)
    net._feat_handles[("k",)] = object()
    for clone in (copy.deepcopy(net), pickle.loads(pickle.dumps(net))):
        assert clone.surface_classifier._handle is None and clone.surface_classifier._handle_key is None
        assert clone._feat_handles == {}
        assert torch.equal(clone.surface_classifier.filters[0].weight, head.filters[0].weight)
    shallow_head = copy.copy(head)               # a NEW object: it must not carry the pointer the original will free
    assert shallow_head._handle is None and shallow_head.filters is head.filters
    assert copy.copy(net)._feat_handles == {}
    head._handle, head._handle_key = None, None
    net._feat_handles.clear()
    b = np.array([[-1.0, -1.0, -1.0]], dtype=np.float32)
    eng = Seg3dLossless(lambda **kw: None, b, -b, [9, 17], balance_value=0.5)
    eng._handles[("k",)] = object()
    c2 = copy.copy(eng)
    assert c2._handles == {} and c2.resolutions == [9, 17]
    eng._handles.clear()


def test_reconstruction_rejects_even_octree_resolution():
    """ADVICE r1: the coarse-to-fine pyramid needs 2^k+1 nodes per axis; an even resolution gets a clear error up front
    instead of an assertion from inside the engine (the dense branch accepts any resolution)."""
    from monoport_b200.recon import reconstruction
    with pytest.raises(ValueError, match="2\\^k\\+1"):
        reconstruction(object(), "cuda:0", None, 256, (-1, -1, -1), (1, 1, 1), use_octree=True, feats=[[torch.zeros(1, 1, 2, 2)]])
