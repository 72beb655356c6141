"""CPU restatement of the MonoPort occupancy hot path.  TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

Every function cites the reference lines it restates (paths relative to /root/reference).
Pinned pieces are checked against the reference's own outputs in tests/golden/*.npz
(generator: tests/golden/make_golden.py, run in the build container where /root/reference exists).

  query_ref                -- PINNED   (MonoPortNet.query, monoport/lib/modeling/MonoPortNet.py:48-91)
  forward_vertices_ref     -- PINNED   (RTL/recon.py:27-89)
  pifu_calib_ref           -- PINNED   (RTL/recon.py:4-25)
  seg3d_lossless_ref       -- PARITY UNPINNED: `implicit-seg` is an un-vendored, unpinned pip
  seg3d_topk_ref              dependency (requirements.txt:15; call sites RTL/main.py:28-29,188-195,390-395).
                              The algorithm is restated from the call-site contract + SURVEY.md §8c.
  marching_cubes_ref       -- PARITY UNPINNED: there is no marching cubes in the reference.
"""
import math

import numpy as np
import torch
import torch.nn.functional as F

LEAKY_SLOPE = 0.01          # F.leaky_relu default, heads/SurfaceClassifier.py:58
Z_SCALE = 512 // 2 / 200.0  # normalizers/DepthNormalizer.py:40  (= 1.28)

G_CHANNELS = [257, 1024, 512, 256, 128, 1]   # heads/SurfaceClassifier.py:76  (Sigmoid)
C_CHANNELS = [513, 1024, 512, 256, 128, 3]   # heads/SurfaceClassifier.py:84  (Tanh)
LAST_NONE, LAST_SIGMOID, LAST_TANH = 0, 1, 2


# ----------------------------------------------------------------------------------------------
# deterministic synthetic inputs (no checkpoints exist offline: scripts/download_model.sh)
# ----------------------------------------------------------------------------------------------
def make_weights(channels, seed):
    """Skip-MLP weights with nn.Conv1d's default init distribution U(-1/sqrt(fan_in), +1/sqrt(fan_in))
    (the layer input widths follow heads/SurfaceClassifier.py:24-34: layer l>0 sees C_l + C_0)."""
    g = torch.Generator().manual_seed(int(seed))
    Ws, bs = [], []
    for l in range(len(channels) - 1):
        cin = channels[l] + (channels[0] if l > 0 else 0)
        cout = channels[l + 1]
        k = 1.0 / math.sqrt(cin)
        Ws.append(((torch.rand(cout, cin, generator=g) * 2 - 1) * k).contiguous())
        bs.append(((torch.rand(cout, generator=g) * 2 - 1) * k).contiguous())
    return Ws, bs


def make_feat(C, H, W, seed, scale=1.0):
    g = torch.Generator().manual_seed(int(seed))
    return (torch.randn(1, C, H, W, generator=g) * scale).contiguous()


def make_points(N, seed, lo=-1.1, hi=1.1):
    g = torch.Generator().manual_seed(int(seed))
    return (torch.rand(1, 3, N, generator=g) * (hi - lo) + lo).contiguous()


def make_encoder_state(layout, seed):
    """float64 parameters for a state-dict layout [(key, shape), ...], drawn in layout order from one generator: weights
    of rank > 1 U(-1/sqrt(fan_in), +1/sqrt(fan_in)) like the conv default init, norm scales 1 + U(-1/4, 1/4), biases
    U(-1/4, 1/4)."""
    g = torch.Generator().manual_seed(int(seed))
    sd = {}
    for key, shape in layout:
        t = torch.rand(tuple(shape), generator=g, dtype=torch.float64) * 2 - 1
        if len(shape) > 1:
            t = t / math.sqrt(math.prod(shape[1:]))
        elif key.endswith(".weight"):
            t = 1 + 0.25 * t
        else:
            t = 0.25 * t
        sd[key] = t
    return sd


def make_image(size, seed):
    """[1,3,size,size] float64 image in [-1,1) (the encoders' input range)."""
    g = torch.Generator().manual_seed(int(seed))
    return torch.rand(1, 3, size, size, generator=g, dtype=torch.float64) * 2 - 1


def _rot(rx, ry, rz):
    """Rotation R = Rz * Ry * Rx (RTL/scene.py:62-88 make_rotate)."""
    sx, cx, sy, cy, sz, cz = math.sin(rx), math.cos(rx), math.sin(ry), math.cos(ry), math.sin(rz), math.cos(rz)
    Rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]], dtype=np.float64)
    Ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]], dtype=np.float64)
    Rz = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]], dtype=np.float64)
    return Rz @ Ry @ Rx


def pifu_calib_ref(extrinsic, intrinsic):
    """RTL/recon.py:4-25: inv(K' E' diag(1,-1,1,1)) in float64, returned as float32 [1,4,4]."""
    flip = np.diag([1.0, -1.0, 1.0, 1.0])
    K = np.array(intrinsic, dtype=np.float64, copy=True)
    K[2, 2] = K[0, 0]
    K[2, 3] = 0
    E = np.array(extrinsic, dtype=np.float64, copy=True)
    E[2, 3] = 0
    return torch.from_numpy(np.linalg.inv(K @ E @ flip)).unsqueeze(0).float()


def scene_calib(yaw_deg=20.0, pitch_deg=0.0):
    """The demo camera (RTL/scene.py:45-50,108-135): extrinsic = R(yaw about x)*R(pitch about y),
    t=(0,0,-2); intrinsic = orthographic diag(1,1,-0.2,1) with [2,3]=-1.  Fed through pifu_calib."""
    R = _rot(math.radians(yaw_deg), 0, 0) @ _rot(0, math.radians(pitch_deg), 0)
    E = np.eye(4)
    E[:3, :3] = R
    E[:3, 3] = [0, 0, -2.0]
    K = np.diag([1.0, 1.0, -0.2, 1.0])
    K[2, 3] = -1.0
    return pifu_calib_ref(E, K)


# ----------------------------------------------------------------------------------------------
# query()  --  monoport/lib/modeling/MonoPortNet.py:48-91
# ----------------------------------------------------------------------------------------------
def project_ref(points, calib, projection="orthogonal"):
    """geometry.py:19-34 (orthogonal) / :37-55 (perspective).  points [3,N], calib [>=3,4]."""
    if calib is None:
        return points
    R = calib[:3, :3]
    t = calib[:3, 3:4]
    p = t + R @ points
    if projection == "perspective":
        p = torch.cat([p[:2] / p[2:3], p[2:3]], 0)
    return p


def bilinear_ref(feat, u, v):
    """geometry.py:4-16: grid_sample(bilinear, padding zeros, align_corners=True).
    feat [C,H,W]; u,v [N] in [-1,1] -> [C,N].  Restated tap-by-tap (no F.grid_sample)."""
    C, H, W = feat.shape
    ix = (u + 1) / 2 * (W - 1)
    iy = (v + 1) / 2 * (H - 1)
    x0 = torch.floor(ix)
    y0 = torch.floor(iy)
    x1 = x0 + 1
    y1 = y0 + 1
    w_nw = (x1 - ix) * (y1 - iy)
    w_ne = (ix - x0) * (y1 - iy)
    w_sw = (x1 - ix) * (iy - y0)
    w_se = (ix - x0) * (iy - y0)
    flat = feat.reshape(C, H * W)

    def tap(xx, yy, w):
        ok = (xx >= 0) & (xx <= W - 1) & (yy >= 0) & (yy <= H - 1)
        xi = xx.clamp(0, W - 1).long()
        yi = yy.clamp(0, H - 1).long()
        return flat[:, yi * W + xi] * (w * ok.to(w.dtype))[None]

    return tap(x0, y0, w_nw) + tap(x1, y0, w_ne) + tap(x0, y1, w_sw) + tap(x1, y1, w_se)


def mlp_ref(x, Ws, bs, last_op):
    """heads/SurfaceClassifier.py:39-71 with no_residual=False, num_views=1: layer l>0 consumes
    cat([hidden, input]) (hidden FIRST, :55); leaky_relu after every layer but the last (:57-58)."""
    y = x
    for l, (W, b) in enumerate(zip(Ws, bs)):
        inp = y if l == 0 else torch.cat([y, x], 0)
        y = W @ inp + b[:, None]
        if l != len(Ws) - 1:
            y = F.leaky_relu(y, LEAKY_SLOPE)
    if last_op == LAST_SIGMOID:
        y = torch.sigmoid(y)
    elif last_op == LAST_TANH:
        y = torch.tanh(y)
    return y


@torch.no_grad()
def query_ref(feat, points, calib, Ws, bs, last_op, projection="orthogonal", z_scale=Z_SCALE, chunk=65536):
    """MonoPortNet.query in eval mode, B=1, single feature level.
    feat [1,C,H,W] or [C,H,W]; points [1,3,N] or [3,N]; calib [1,4,4]/[4,4]/[3,4]/None -> [Res,N]."""
    feat = feat[0] if feat.dim() == 4 else feat
    points = points[0] if points.dim() == 3 else points
    if calib is not None and calib.dim() == 3:
        calib = calib[0]
    N = points.shape[1]
    res = Ws[-1].shape[0]
    out = torch.empty(res, N, dtype=torch.float32)
    for s in range(0, N, chunk):
        p = points[:, s:s + chunk].float()
        xyz = project_ref(p, calib, projection)
        u, v, z = xyz[0], xyz[1], xyz[2]
        in_img = (u >= -1.0) & (u <= 1.0) & (v >= -1.0) & (v <= 1.0)      # MonoPortNet.py:74
        x = torch.cat([bilinear_ref(feat, u, v), (z * z_scale)[None]], 0)  # :82-83, DepthNormalizer.py:32
        out[:, s:s + chunk] = in_img.float()[None] * mlp_ref(x, Ws, bs, last_op)  # :86-89
    return out


def heightfield_person(Ws, bs, feat, k=40.0, channel=0):
    """Synthetic 'person' (SURVEY.md §8d): random-init weights give a noise surface, so wire a closed,
    body-like field through the *same* dense layers (cost per point unchanged):
      * feature channel `channel` is overwritten with a smooth height map h(u,v) (ellipse-union silhouette);
      * two rows of layer 3 compute lrelu(+z_feat) and lrelu(-z_feat)  (sum = 0.99*|z_feat|);
      * layer 4 reads logit = k*(h - |z_feat|) from its skip access to the input
        (layer-l input order is [hidden, C feat, 1 z], heads/SurfaceClassifier.py:55).
    Occupied where |z_feat| < h(u,v).  Returns (Ws, bs, feat, h)."""
    Ws = [w.clone() for w in Ws]
    bs = [b.clone() for b in bs]
    feat = feat.clone()
    C = feat.shape[1]
    H, W = feat.shape[2:]
    yy, xx = torch.meshgrid(torch.linspace(-1, 1, H), torch.linspace(-1, 1, W), indexing="ij")
    body = 1 - ((xx / 0.28) ** 2 + ((yy - 0.05) / 0.62) ** 2)
    head = 1 - ((xx / 0.16) ** 2 + ((yy + 0.68) / 0.17) ** 2)
    arm = 1 - (((xx.abs() - 0.40) / 0.10) ** 2 + ((yy + 0.05) / 0.40) ** 2)
    h = torch.maximum(torch.maximum(body, head), arm).clamp(min=-1.0) * 0.35
    feat[0, channel] = h
    hid3 = Ws[3].shape[1] - (C + 1)
    Ws[3][0].zero_(); Ws[3][1].zero_()
    Ws[3][0, hid3 + C] = 1.0
    Ws[3][1, hid3 + C] = -1.0
    bs[3][0] = 0.0; bs[3][1] = 0.0
    hid4 = Ws[4].shape[1] - (C + 1)
    Ws[4].zero_()
    Ws[4][0, hid4 + channel] = k
    Ws[4][0, 0] = -k / 0.99
    Ws[4][0, 1] = -k / 0.99
    bs[4].zero_()
    return Ws, bs, feat, h


# ----------------------------------------------------------------------------------------------
# forward_vertices  --  RTL/recon.py:27-89  (restated with explicit index arithmetic)
# ----------------------------------------------------------------------------------------------
@torch.no_grad()
def forward_vertices_ref(sdf, direction="front"):
    if sdf is None:
        return None, None, None, None
    vol = sdf[0, 0]                                   # [D,H,W] = [z,y,x]
    R = vol.shape[2]
    if direction in ("back", "right"):                # :46-51 flip along dim 0
        vol = vol.flip(0)
    if direction in ("left", "right"):                # :44-45, :51 swap dims 0 and 2
        vol = vol.permute(2, 1, 0)
    # :53-55  flip dim 0 again, then view as [x,y,z']  with z' = R-1-z
    A = vol.flip(0).permute(2, 1, 0).contiguous()     # A[x,y,k]
    occ = A > 0.5
    # :57-61  first occupied k along the last axis; ties in max() resolve to the first maximum
    ramp = torch.arange(R, 0, -1, dtype=torch.float32)
    score = occ.float() * ramp
    first = score.argmax(dim=2)                       # 0 when the column is empty
    kk = torch.arange(R).view(1, 1, R)
    keep = occ & ~(kk > first.unsqueeze(2))
    p = keep.nonzero()                                # row-major (x, y, k) order == .nonzero().t() of :62
    X, Y, K = p[:, 0], p[:, 1], p[:, 2]
    K2 = (K - 2).clamp(0, R)
    Y2 = (Y - 2).clamp(0, R)
    X2 = (X - 2).clamp(0, R)
    v1 = A[X, Y, K]
    v2 = A[X, Y, K2]
    v3 = A[X, Y2, K]
    v4 = A[X2, Y, K]
    Z = K2.float() * (0.5 - v1) / (v2 - v1) + K.float() * (v2 - 0.5) / (v2 - v1)     # :77
    Z = Z.clamp(0, R)
    n = torch.stack([v4 - v1, v3 - v1, v2 - v1], 1)
    n = n / torch.norm(n, p=2, dim=1, keepdim=True)
    return X.long(), Y.long(), Z, n


# ----------------------------------------------------------------------------------------------
# Seg3dLossless / Seg3dTopk  --  PARITY UNPINNED restatement (see module docstring)
# ----------------------------------------------------------------------------------------------
def level_points(coords_xyz, res_final, b_min, b_max):
    """Integer node coords (final-resolution index space, columns x,y,z) -> world points [N,3].
    align_corners=False convention: p = (c + 0.5)/R * (b_max-b_min) + b_min.  The divisor R (=257, not 256)
    is corroborated in-tree by mat_color (RTL/main.py:204-209)."""
    c = coords_xyz.to(torch.float32)
    b_min = torch.as_tensor(b_min, dtype=torch.float32).view(1, 3)
    b_max = torch.as_tensor(b_max, dtype=torch.float32).view(1, 3)
    p = c / float(res_final) + 1.0 / (2.0 * res_final)
    return p * (b_max - b_min) + b_min


def _grid_coords(res, stride):
    r = torch.arange(res, dtype=torch.int64) * stride
    z, y, x = torch.meshgrid(r, r, r, indexing="ij")          # z slowest
    return torch.stack([x.reshape(-1), y.reshape(-1), z.reshape(-1)], 1)


def _up2(vol, res):
    return F.interpolate(vol[None, None], size=(res, res, res), mode="trilinear", align_corners=True)[0, 0]


def _dilate(mask, k):
    w = torch.ones(1, 1, k, k, k)
    return F.conv3d(mask.float()[None, None], w, padding=k // 2)[0, 0] > 0


@torch.no_grad()
def seg3d_lossless_ref(query_fn, resolutions, b_min=(-1, -1, -1), b_max=(1, 1, 1), balance=0.5,
                       faster=True, return_stats=False):
    """query_fn(points[N,3] world) -> occupancy [N].  Returns the [R,R,R] (z,y,x) volume or None.

    faster=True (the mode the reference selects, RTL/main.py:195):
      level 0 dense; intermediate levels: 2x trilinear up-sample (align_corners=True), boundary =
      up-sampled binary mask strictly between 0 and 1, box-dilated with k=9 (level 1), 7 (level 2), 3
      (else), already evaluated nodes removed, evaluated in x-major order, scattered; LAST level
      up-sampled only.
    faster=False ("lossless"): k=3 everywhere, last level examined too, and after every level a
      conflict loop re-queries the 27-neighbourhood of nodes whose interpolated and evaluated signs
      disagree until none remain.
    """
    R = int(resolutions[-1])
    stats = []
    res0 = int(resolutions[0])
    stride = (R - 1) // (res0 - 1)
    coords = _grid_coords(res0, stride)
    occ = query_fn(level_points(coords, R, b_min, b_max)).float().reshape(res0, res0, res0)
    stats.append(dict(res=res0, idx=torch.arange(res0 ** 3)))
    if not bool((occ > balance).any()):
        return (None, stats) if return_stats else None
    known = torch.ones(res0, res0, res0, dtype=torch.bool)
    for li, res in enumerate(resolutions[1:], start=1):
        res = int(res)
        stride = (R - 1) // (res - 1)
        last = li == len(resolutions) - 1
        valid = _up2((occ > balance).float(), res)
        occ = _up2(occ, res)
        kn = torch.zeros(res, res, res, dtype=torch.bool)
        kn[::2, ::2, ::2] = known
        known = kn
        if faster and last:
            stats.append(dict(res=res, idx=torch.zeros(0, dtype=torch.int64)))
            break
        boundary = (valid > 0) & (valid < 1)
        k = (9 if li == 1 else 7 if li == 2 else 3) if faster else 3
        boundary = _dilate(boundary, k) & ~known
        # x-major order: sort by (x, y, z)
        idx = _xmajor_indices(boundary)
        stats.append(dict(res=res, idx=idx))
        if idx.numel() == 0:
            continue
        occ, known, extra = _eval_scatter(query_fn, occ, known, idx, res, stride, R, b_min, b_max)
        if not faster:
            # conflict loop
            interp_sign = None
            while True:
                conflicts = extra
                if conflicts is None or conflicts.numel() == 0:
                    break
                nb = _neighbours27(conflicts, res) & ~known
                idx2 = _xmajor_indices(nb)
                if idx2.numel() == 0:
                    break
                stats[-1]["idx"] = torch.cat([stats[-1]["idx"], idx2])
                occ, known, extra = _eval_scatter(query_fn, occ, known, idx2, res, stride, R, b_min, b_max)
    return (occ, stats) if return_stats else occ


def _xmajor_indices(mask):
    """Linear indices (z*H*W + y*W + x) of set nodes ordered by (x, y, z)."""
    p = mask.permute(2, 1, 0).nonzero()       # rows (x, y, z) sorted lexicographically
    res = mask.shape[0]
    return p[:, 2] * res * res + p[:, 1] * res + p[:, 0]


def _eval_scatter(query_fn, occ, known, idx, res, stride, R, b_min, b_max, balance=0.5):
    x = idx % res
    y = (idx // res) % res
    z = idx // (res * res)
    coords = torch.stack([x, y, z], 1) * stride
    vals = query_fn(level_points(coords, R, b_min, b_max)).float()
    flat = occ.reshape(-1)
    conflict = ((flat[idx] - balance) * (vals - balance)) < 0
    flat[idx] = vals
    known.reshape(-1)[idx] = True
    return occ, known, idx[conflict]


def _neighbours27(idx, res):
    m = torch.zeros(res, res, res, dtype=torch.bool)
    m.reshape(-1)[idx] = True
    return _dilate(m, 3)


@torch.no_grad()
def seg3d_topk_ref(query_fn, resolutions, num_points, b_min=(-1, -1, -1), b_max=(1, 1, 1), balance=0.5,
                   return_stats=False):
    """Level 0 dense; every later level: up-sample, pick the num_points[l] nodes with the smallest
    |occ - balance| (ties -> lowest linear index; evaluated in ascending index order), evaluate, scatter."""
    R = int(resolutions[-1])
    res0 = int(resolutions[0])
    stats = []
    coords = _grid_coords(res0, (R - 1) // (res0 - 1))
    occ = query_fn(level_points(coords, R, b_min, b_max)).float().reshape(res0, res0, res0)
    stats.append(dict(res=res0, idx=torch.arange(res0 ** 3)))
    if not bool((occ > balance).any()):
        return (None, stats) if return_stats else None
    for li, res in enumerate(resolutions[1:], start=1):
        res = int(res)
        stride = (R - 1) // (res - 1)
        occ = _up2(occ, res)
        k = min(int(num_points[li]), res ** 3)
        key = (occ.reshape(-1) - balance).abs()
        order = torch.sort(key, stable=True).indices[:k]
        idx = torch.sort(order).values
        stats.append(dict(res=res, idx=idx))
        x = idx % res
        y = (idx // res) % res
        z = idx // (res * res)
        vals = query_fn(level_points(torch.stack([x, y, z], 1) * stride, R, b_min, b_max)).float()
        occ.reshape(-1)[idx] = vals
    return (occ, stats) if return_stats else occ


# ----------------------------------------------------------------------------------------------
# marching cubes  --  PARITY UNPINNED (absent from the reference).  Table: tools/gen_mc_table.py
# ----------------------------------------------------------------------------------------------
def marching_cubes_ref(vol, iso=0.5):
    """vol [D,H,W] (z,y,x) float32 numpy -> (verts [V,3] float32 in index space (x,y,z), faces [F,3] int32).

    Vertex ids: every grid edge is owned by its lower node; node n (linear z*H*W+y*W+x) owns its +x,
    +y, +z edges (axis 0,1,2).  Vertices are numbered in (node, axis) order; faces in (cell, table) order;
    cell linear order is z-slowest over the (D-1,H-1,W-1) cell grid.  Position = a + t*(b-a) with
    t = (iso - va)/(vb - va) computed in float32."""
    from tools.gen_mc_table import build_table, EDGE_CORNERS, EDGE_AXIS, CORNER_OFF
    ntri, tri, _ = build_table()
    vol = np.ascontiguousarray(vol, dtype=np.float32)
    D, H, W = vol.shape
    inside = vol > np.float32(iso)
    # owned-edge activity per node
    act = np.zeros((D, H, W, 3), dtype=bool)
    act[:, :, :-1, 0] = inside[:, :, :-1] != inside[:, :, 1:]
    act[:, :-1, :, 1] = inside[:, :-1, :] != inside[:, 1:, :]
    act[:-1, :, :, 2] = inside[:-1, :, :] != inside[1:, :, :]
    flat = act.reshape(-1)
    vid = np.cumsum(flat, dtype=np.int64) - flat            # exclusive scan in (node, axis) order
    vid = vid.reshape(D, H, W, 3)
    zz, yy, xx, aa = np.nonzero(act)
    a_pos = np.stack([xx, yy, zz], 1).astype(np.float32)
    va = vol[zz, yy, xx]
    vb = vol[zz + (aa == 2), yy + (aa == 1), xx + (aa == 0)]
    t = (np.float32(iso) - va) / (vb - va)
    verts = a_pos.copy()
    verts[np.arange(len(aa)), aa] += t.astype(np.float32)
    # cells
    case = np.zeros((D - 1, H - 1, W - 1), dtype=np.int32)
    for c in range(8):
        dx, dy, dz = CORNER_OFF[c]
        case |= inside[dz:D - 1 + dz, dy:H - 1 + dy, dx:W - 1 + dx].astype(np.int32) << c
    cz, cy, cx = np.nonzero(ntri[case] > 0)
    faces = []
    cc = case[cz, cy, cx]
    for cell in range(len(cc)):
        c = cc[cell]
        for tI in range(ntri[c]):
            f = []
            for e in tri[c, 3 * tI:3 * tI + 3]:
                a, _b = EDGE_CORNERS[e]
                ox, oy, oz = CORNER_OFF[a]
                f.append(vid[cz[cell] + oz, cy[cell] + oy, cx[cell] + ox, EDGE_AXIS[e]])
            faces.append(f)
    faces = np.asarray(faces, dtype=np.int32).reshape(-1, 3)
    return verts.astype(np.float32), faces


def analytic_volume(R, kind="sphere"):
    """Deterministic float32 test volumes built from correctly-rounded IEEE ops only (+,-,*,/,sqrt)."""
    r = (np.arange(R, dtype=np.float32) + np.float32(0.5)) / np.float32(R) * np.float32(2) - np.float32(1)
    z, y, x = np.meshgrid(r, r, r, indexing="ij")
    if kind == "sphere":
        d = np.sqrt(x * x + y * y + z * z)
        f = np.float32(0.6) - d
    elif kind == "ellipsoid":
        d = np.sqrt((x - np.float32(0.1)) ** 2 / np.float32(0.25) + (y + np.float32(0.05)) ** 2 / np.float32(0.49)
                    + (z - np.float32(0.07)) ** 2 / np.float32(0.09))
        f = (np.float32(1) - d) * np.float32(0.4)
    elif kind == "two_blobs":
        d1 = np.sqrt((x - np.float32(0.35)) ** 2 + y * y + z * z)
        d2 = np.sqrt((x + np.float32(0.4)) ** 2 + (y - np.float32(0.2)) ** 2 + z * z)
        f = np.maximum(np.float32(0.3) - d1, np.float32(0.25) - d2)
    else:
        raise ValueError(kind)
    return np.clip(np.float32(0.5) + np.float32(4.0) * f, np.float32(0), np.float32(1)).astype(np.float32)


# ----------------------------------------------------------------------------------------------
# colorization  --  RTL/main.py:212-249 (restated; RTL/main.py itself cannot be imported: flask, cv2, GL ...)
# ----------------------------------------------------------------------------------------------
@torch.no_grad()
def colorization_ref(query_c, X, Y, Z, calib, resolution=257, b_min=(-1, -1, -1), b_max=(1, 1, 1), norm=None):
    """query_c(points[1,3,N], calib) -> [3,N] in [-1,1] (netC).  Returns the [R,R,3] image."""
    image = torch.ones((resolution, resolution, 3), dtype=torch.float32)
    if norm is not None:
        image[X, Y, :] = ((norm + 1) / 2).clamp(0, 1)
        return image
    b_min = torch.tensor(b_min, dtype=torch.float32)
    b_max = torch.tensor(b_max, dtype=torch.float32)
    scale = (b_max - b_min) / resolution
    verts = torch.stack([X.float(), Y.float(), resolution - Z.float()], 1)
    world = verts * scale[None] + b_min[None]
    preds = query_c(world.t().contiguous()[None], calib)
    image[X, Y, :] = (preds * 0.5 + 0.5).t()
    return image
