#!/usr/bin/env python
"""Generate tests/golden/*.npz by running the UNMODIFIED reference (/root/reference) on CPU.

Run in the build container (the reference tree does not exist on the GPU box):
    python tests/golden/make_golden.py

The reference publishes no golden vectors / KATs (SURVEY.md §4), so these are outputs of the reference
itself on seeded synthetic inputs.  Inputs that are large (weights 4.7/6.7 MB, feature maps 16.8/33.5 MB)
are NOT stored: they are regenerated from seeds by oracle.spec.make_weights/make_feat (torch CPU
generator -- bit-reproducible for the pinned torch build); each file stores float64 checksums of the
regenerated tensors so RNG drift is detected instead of silently failing parity.
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))

from oracle import spec  # noqa: E402
from oracle.ref_loader import load_reference  # noqa: E402


def checksum(t):
    t = t.double().reshape(-1)
    w = torch.arange(1, t.numel() + 1, dtype=torch.float64) % 997
    return np.array([t.sum().item(), (t * w).sum().item(), t.abs().max().item()])


def load_head(net, Ws, bs):
    sd = {}
    for l, (W, b) in enumerate(zip(Ws, bs)):
        sd["filters.%d.weight" % l] = W[:, :, None].clone()     # Conv1d weight [Cout,Cin,1]
        sd["filters.%d.bias" % l] = b.clone()
    net.surface_classifier.load_state_dict(sd)


QUERY_CASES = [
    # name, net, wseed, fseed, pseed, N, calib, projection, feat_scale, feat_hw
    dict(name="g_identity", net="G", wseed=11, fseed=12, pseed=13, N=8192, calib="identity", proj="orthogonal", fscale=1.0, hw=128),
    dict(name="g_rot33", net="G", wseed=21, fseed=22, pseed=23, N=8191, calib="rot33", proj="orthogonal", fscale=1.0, hw=128),
    dict(name="g_nocalib", net="G", wseed=31, fseed=32, pseed=33, N=1000, calib="none", proj="orthogonal", fscale=1.0, hw=128),
    dict(name="g_bigfeat", net="G", wseed=41, fseed=42, pseed=43, N=4096, calib="rot33", proj="orthogonal", fscale=4.0, hw=128),
    dict(name="g_persp", net="G", wseed=51, fseed=52, pseed=53, N=2049, calib="persp", proj="perspective", fscale=1.0, hw=128),
    dict(name="g_smallmap", net="G", wseed=61, fseed=62, pseed=63, N=777, calib="rot33", proj="orthogonal", fscale=1.0, hw=32),
    dict(name="c_rot33", net="C", wseed=71, fseed=72, pseed=73, N=4099, calib="rot33", proj="orthogonal", fscale=1.0, hw=128),
    dict(name="c_identity", net="C", wseed=81, fseed=82, pseed=83, N=515, calib="identity", proj="orthogonal", fscale=1.0, hw=128),
]


def make_calib(kind):
    if kind == "identity":
        return torch.eye(4)[None]
    if kind == "rot33":
        return spec.scene_calib(20.0, 33.0)
    if kind == "persp":
        c = spec.scene_calib(10.0, -15.0).clone()
        c[0, 2, 3] = 3.0      # push z away from 0 so x/z, y/z stay finite and mostly in-image
        c[0, :2, :] *= 2.5
        return c
    if kind == "none":
        return None
    raise ValueError(kind)


def border_points(points):
    """Force a few points exactly onto the image border / corners and far outside."""
    p = points.clone()
    n = p.shape[2]
    if n >= 16:
        p[0, :, 0] = torch.tensor([1.0, 0.3, 0.1])
        p[0, :, 1] = torch.tensor([-1.0, -1.0, 0.0])
        p[0, :, 2] = torch.tensor([1.0, 1.0, -0.5])
        p[0, :, 3] = torch.tensor([0.0, 1.0, 0.9])
        p[0, :, 4] = torch.tensor([5.0, 0.0, 0.0])
        p[0, :, 5] = torch.tensor([0.0, 0.0, 0.0])
        p[0, :, 6] = torch.tensor([-1.0, 0.999999, 0.2])
        p[0, :, 7] = torch.tensor([1.0000001, 0.0, 0.2])
    return p


@torch.no_grad()
def gen_query(ns):
    for c in QUERY_CASES:
        chans = spec.G_CHANNELS if c["net"] == "G" else spec.C_CHANNELS
        net = (ns.PIFuNetG() if c["net"] == "G" else ns.PIFuNetC()).eval()
        if c["proj"] == "perspective":
            net.projection = ns.perspective            # what opt.projection='perspective' selects (MonoPortNet.py:27)
        Ws, bs = spec.make_weights(chans, c["wseed"])
        load_head(net, Ws, bs)
        C = chans[0] - 1
        feat = spec.make_feat(C, c["hw"], c["hw"], c["fseed"], c["fscale"])
        pts = border_points(spec.make_points(c["N"], c["pseed"]))
        calib = make_calib(c["calib"])
        # 4 stages like the HG encoder: eval-mode query must only use the LAST one (MonoPortNet.py:63-64)
        decoy = torch.zeros_like(feat)
        out = net.query([[decoy], [decoy], [decoy], [feat]], pts, calibs=calib)
        assert len(out) == 1
        ref = out[0][0].numpy()
        mine = spec.query_ref(feat, pts, calib, Ws, bs,
                              spec.LAST_SIGMOID if c["net"] == "G" else spec.LAST_TANH, c["proj"]).numpy()
        err = np.abs(ref - mine).max()
        print("query %-12s N=%5d  in-img %.2f  |oracle-ref| = %.2e" % (c["name"], c["N"], (ref[0] != 0).mean(), err))
        assert err < 2e-6
        np.savez_compressed(
            os.path.join(HERE, "query_%s.npz" % c["name"]),
            points=pts.numpy(), calib=(calib.numpy() if calib is not None else np.zeros((0,), np.float32)),
            expected=ref, net=c["net"], wseed=c["wseed"], fseed=c["fseed"], fscale=c["fscale"], hw=c["hw"],
            proj=c["proj"], w_checksum=np.stack([checksum(w) for w in Ws]), f_checksum=checksum(feat))


@torch.no_grad()
def gen_forward_vertices(ns):
    for R, kind in ((33, "sphere"), (65, "ellipsoid"), (65, "two_blobs")):
        vol = torch.from_numpy(spec.analytic_volume(R, kind))[None, None]
        rec = dict(R=R, kind=kind, vol_checksum=checksum(vol))
        for d in ("front", "back", "left", "right"):
            X, Y, Z, n = ns.forward_vertices(vol.clone(), d)
            rec["X_" + d], rec["Y_" + d], rec["Z_" + d], rec["N_" + d] = X.numpy(), Y.numpy(), Z.numpy(), n.numpy()
            print("forward_vertices %s R=%d %-5s -> %d verts" % (kind, R, d, X.numel()))
        np.savez_compressed(os.path.join(HERE, "fv_%s_%d.npz" % (kind, R)), **rec)
    assert ns.forward_vertices(None) == (None, None, None, None)


def gen_calib(ns):
    rows = []
    for yaw, pitch in ((20.0, 0.0), (20.0, 33.0), (0.0, -120.0)):
        import math
        E = np.eye(4)
        E[:3, :3] = spec._rot(math.radians(yaw), 0, 0) @ spec._rot(0, math.radians(pitch), 0)
        E[:3, 3] = [0, 0, -2.0]
        K = np.diag([1.0, 1.0, -0.2, 1.0])
        K[2, 3] = -1.0
        rows.append(dict(E=E, K=K, calib=ns.pifu_calib(E, K, device="cpu").numpy()))
    np.savez_compressed(os.path.join(HERE, "calib.npz"),
                        E=np.stack([r["E"] for r in rows]), K=np.stack([r["K"] for r in rows]),
                        calib=np.stack([r["calib"] for r in rows]))


@torch.no_grad()
def gen_query_pitch70(ns):
    """One more netG case at a steep camera pitch (yaw 20, pitch -70) on a 64x64 map, as the reference's query() returns it
    for a single-stage feature list; the inputs are regenerated from their seeds and pinned by checksums."""
    net = ns.PIFuNetG().eval()
    Ws, bs = spec.make_weights(spec.G_CHANNELS, 5)
    load_head(net, Ws, bs)
    feat = spec.make_feat(256, 64, 64, 6)
    pts = spec.make_points(3000, 7)
    ref = net.query([[feat]], pts, calibs=spec.scene_calib(20, -70))[0][0]
    np.savez_compressed(os.path.join(HERE, "reference_query_pitch70.npz"), expected=ref.numpy(),
                        w_checksum=np.stack([checksum(w) for w in Ws]), f_checksum=checksum(feat), p_checksum=checksum(pts))


ENCODER_SEED, ENCODER_IMAGE_SEED, ENCODER_IMAGE_SIZE, ENCODER_SAMPLE = 91, 92, 64, 1024


@torch.no_grad()
def gen_encoders(ns):
    """Image encoders of PIFuNetG (HGFilter) and PIFuNetC (ResnetFilter) in float64 with seeded parameters: the state-dict
    layout, checksums of the parameters as loaded (aliased keys keep the value loaded last), and of every stage's output a
    checksum plus a seeded sample of ENCODER_SAMPLE values (whole outputs would be 1 MB)."""
    rec = dict(seed=ENCODER_SEED, image_seed=ENCODER_IMAGE_SEED, image_size=ENCODER_IMAGE_SIZE)
    for net, factory in (("G", ns.PIFuNetG), ("C", ns.PIFuNetC)):
        ref = factory().eval().double()
        layout = [(k, list(v.shape)) for k, v in ref.state_dict().items()]
        ref.load_state_dict(spec.make_encoder_state(layout, ENCODER_SEED), strict=True)
        outs = [o[0] for o in ref.image_filter(spec.make_image(ENCODER_IMAGE_SIZE, ENCODER_IMAGE_SEED))]
        idx = torch.randint(0, outs[0].numel(), (ENCODER_SAMPLE,), generator=torch.Generator().manual_seed(ENCODER_SEED))
        rec[net + "_layout"] = np.array(json.dumps(layout))
        rec[net + "_state_checksum"] = np.stack([checksum(v) for v in ref.state_dict().values()])
        rec[net + "_out_checksum"] = np.stack([checksum(o) for o in outs])
        rec[net + "_out_index"] = idx.numpy()
        rec[net + "_out_sample"] = np.stack([o.reshape(-1)[idx].numpy() for o in outs])
        print("encoder %s: %d state entries, %d stage outputs of %s" % (net, len(layout), len(outs), tuple(outs[0].shape)))
    np.savez_compressed(os.path.join(HERE, "encoders.npz"), **rec)


def gen_obj_writer():
    """Bytes of the reference's text OBJ writers (monoport/lib/mesh_util.py:223-242) for a small seeded mesh."""
    import importlib.util
    import tempfile
    from oracle.ref_loader import REF_ROOT
    spec_ = importlib.util.spec_from_file_location("_ref_mesh_util", os.path.join(REF_ROOT, "monoport", "lib", "mesh_util.py"))
    ref = importlib.util.module_from_spec(spec_)
    spec_.loader.exec_module(ref)
    rng = np.random.default_rng(0)
    V = rng.normal(size=(57, 3)).astype(np.float32)
    F = rng.integers(0, 57, size=(101, 3)).astype(np.int32)
    C = rng.random((57, 3)).astype(np.float32)
    with tempfile.TemporaryDirectory() as d:
        a, b = os.path.join(d, "a.obj"), os.path.join(d, "b.obj")
        ref.save_obj_mesh(a, V, F)
        ref.save_obj_mesh_with_color(b, V, F, C)
        obj, obj_color = open(a).read(), open(b).read()
    np.savez_compressed(os.path.join(HERE, "obj_writer.npz"), V=V, F=F, C=C, obj=np.array(obj), obj_color=np.array(obj_color))


if __name__ == "__main__":
    torch.set_num_threads(8)
    ns = load_reference()
    gen_query(ns)
    gen_forward_vertices(ns)
    gen_calib(ns)
    gen_query_pitch70(ns)
    gen_encoders(ns)
    gen_obj_writer()
    print("done")
