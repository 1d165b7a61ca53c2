"""Deterministic synthetic workloads for the rasterizer / correlation path (numpy only).

Every constant is anchored in the reference's own data generator and camera glue, so the
shapes, value ranges and matrix conventions are the ones the real pipeline feeds the kernels:
  * camera ring: 16 cams => 22.5 deg between source views, radius 2.0 m, look-at (0,0.85,0),
    pitch -8 deg, fx=fy=0.8*res, cx=res/2, cy=res/2+25*res/1024
    (reference prepare_data/render_data.py:110-114,130,153-160,214-216)
  * novel pose = slerp(R)/lerp(t,K) at `ratio`      (reference lib/utils.py:19-41)
  * world_view_transform = W2V^T, full_proj = W2V^T @ P^T (reference lib/utils.py:36-41)
  * off-centre projection from K                     (reference lib/graphics_utils.py:31-48)
  * pixel-aligned unprojection with +0.5 pixel centres and inverse-depth parameterisation
                                                     (reference lib/utils.py:87-109)
  * value ranges: unit quaternion, scale<=0.01, opacity in (0,1), rgb in [0,1]
                                                     (reference lib/gs_parm_network.py:72-78, lib/GaussianRender.py:30)
Nothing here reads /root/reference.
"""
import math

import numpy as np

ZNEAR, ZFAR = 0.01, 100.0          # reference config/stereo_human_config.py:25-26
SEED = 1314                        # reference train_stage2.py:206-207


def _rot_y(a):
    c, s = math.cos(a), math.sin(a)
    return np.array([[c, 0, s], [0, 1, 0], [-s, 0, c]], np.float64)


def _rot_x(a):
    c, s = math.cos(a), math.sin(a)
    return np.array([[1, 0, 0], [0, c, -s], [0, s, c]], np.float64)


def ring_camera(angle_deg, res, radius=2.0, pitch_deg=-8.0, look_at=(0.0, 0.85, 0.0)):
    """(K[3,3], E[3,4]) of a ring camera: x right, y down, z forward; X_cam = R X_world + t."""
    look_at = np.asarray(look_at, np.float64)
    pos = look_at + _rot_y(math.radians(angle_deg)) @ _rot_x(math.radians(pitch_deg)) @ np.array([0.0, 0.0, radius])
    fwd = look_at - pos
    fwd /= np.linalg.norm(fwd)
    right = np.cross(fwd, np.array([0.0, 1.0, 0.0]))
    right /= np.linalg.norm(right)
    down = np.cross(fwd, right)
    R = np.stack([right, down, fwd])
    t = -R @ pos
    K = np.array([[0.8 * res, 0, res * 0.5], [0, 0.8 * res, res * 0.5 + 25.0 * res / 1024.0], [0, 0, 1]], np.float64)
    return K, np.concatenate([R, t[:, None]], 1)


def _slerp_rot(R0, R1, ratio):
    """Geodesic interpolation R0 * exp(ratio * log(R0^T R1))."""
    Rr = R0.T @ R1
    cosang = min(1.0, max(-1.0, (np.trace(Rr) - 1.0) * 0.5))
    ang = math.acos(cosang)
    if ang < 1e-12:
        return R0.copy()
    axis = np.array([Rr[2, 1] - Rr[1, 2], Rr[0, 2] - Rr[2, 0], Rr[1, 0] - Rr[0, 1]]) / (2.0 * math.sin(ang))
    a = ang * ratio
    Kx = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    return R0 @ (np.eye(3) + math.sin(a) * Kx + (1 - math.cos(a)) * (Kx @ Kx))


def novel_camera(K0, E0, K1, E1, width, height, ratio=0.5, znear=ZNEAR, zfar=ZFAR):
    """The five camera quantities the reference stores in data['novel_view'] (lib/utils.py:8-54),
    as float32 numpy arrays in the reference's (row-vector / transposed) convention."""
    R = _slerp_rot(E0[:, :3], E1[:, :3], ratio)
    t = (1.0 - ratio) * E0[:, 3] + ratio * E1[:, 3]
    K = (1.0 - ratio) * K0 + ratio * K1
    w2v = np.eye(4)
    w2v[:3, :3] = R
    w2v[:3, 3] = t
    Pm = np.zeros((4, 4))
    Pm[0, 0] = 2.0 * K[0, 0] / width
    Pm[1, 1] = 2.0 * K[1, 1] / height
    Pm[0, 2] = (2.0 * K[0, 2] - width) / width
    Pm[1, 2] = (2.0 * K[1, 2] - height) / height
    Pm[3, 2] = 1.0
    Pm[2, 2] = zfar / (zfar - znear)
    Pm[2, 3] = -(zfar * znear) / (zfar - znear)
    wvt = w2v.T.astype(np.float32)
    full = (wvt.astype(np.float64) @ Pm.T).astype(np.float32)
    cam_center = np.linalg.inv(wvt.astype(np.float64))[3, :3].astype(np.float32)
    fovx = 2.0 * math.atan(width / (2.0 * K[0, 0]))
    fovy = 2.0 * math.atan(height / (2.0 * K[1, 1]))
    return dict(FovX=fovx, FovY=fovy, world_view_transform=wvt, full_proj_transform=full, camera_center=cam_center,
                width=int(width), height=int(height), K=K, E=np.concatenate([R, t[:, None]], 1))


_DEPTH_CACHE = {}


def _capsule_depth(K, E, res, radius, y0, y1):
    """Ray-cast a y-axis capsule (segment (0,y0,0)-(0,y1,0), given radius). Returns z-depth [res,res], 0 = miss."""
    key = (K.tobytes(), E.tobytes(), res, radius, y0, y1)
    if key not in _DEPTH_CACHE:
        _DEPTH_CACHE[key] = _capsule_depth_impl(K, E, res, radius, y0, y1)
    return _DEPTH_CACHE[key]


def _capsule_depth_impl(K, E, res, radius, y0, y1):
    R, t = E[:, :3], E[:, 3]
    o = -R.T @ t
    v, u = np.meshgrid(np.arange(res) + 0.5, np.arange(res) + 0.5, indexing="ij")
    dc = np.stack([(u - K[0, 2]) / K[0, 0], (v - K[1, 2]) / K[1, 1], np.ones_like(u)], -1)   # cam-space dir, z=1
    d = dc @ R                                                                                # world dir (R^T dc)
    best = np.full((res, res), np.inf)
    # infinite cylinder x^2+z^2=r^2, clipped to y in [y0,y1]
    a = d[..., 0] ** 2 + d[..., 2] ** 2
    b = 2 * (o[0] * d[..., 0] + o[2] * d[..., 2])
    c = o[0] ** 2 + o[2] ** 2 - radius ** 2
    disc = b * b - 4 * a * c
    ok = disc > 0
    s = np.where(ok, (-b - np.sqrt(np.where(ok, disc, 0))) / (2 * a), np.inf)
    yh = o[1] + s * d[..., 1]
    best = np.where(ok & (s > 0) & (yh >= y0) & (yh <= y1), s, best)
    for yc in (y0, y1):     # end spheres
        oc = o - np.array([0.0, yc, 0.0])
        a2 = (d ** 2).sum(-1)
        b2 = 2 * (d @ oc)
        c2 = oc @ oc - radius ** 2
        disc2 = b2 * b2 - 4 * a2 * c2
        ok2 = disc2 > 0
        s2 = np.where(ok2, (-b2 - np.sqrt(np.where(ok2, disc2, 0))) / (2 * a2), np.inf)
        best = np.where(ok2 & (s2 > 0) & (s2 < best), s2, best)
    return np.where(np.isfinite(best), best, 0.0)    # ray param s with dir z=1 => z-depth


def _attrs(rng, n, z_over_fx):
    rot = rng.standard_normal((n, 4)).astype(np.float32)
    rot /= np.linalg.norm(rot, axis=1, keepdims=True)
    scale = (rng.uniform(0.5, 2.0, (n, 3)) * z_over_fx[:, None]).astype(np.float32)
    scale = np.minimum(scale, np.float32(0.01))
    opacity = rng.uniform(0.2, 1.0, (n, 1)).astype(np.float32)
    rgb = rng.uniform(0.0, 1.0, (n, 3)).astype(np.float32)
    return rot, scale, opacity, rgb


def source_view_maps(res, angle_deg, seed, body_radius=0.425):
    """One source view in the layout lib/network.py writes into data[view]: pixel-aligned maps.
    Returns dict(K, E, depth[res,res], valid[res*res] bool, xyz[res*res,3], img[3,res,res] in [-1,1],
    rot_maps[4,res,res], scale_maps[3,res,res], opacity_maps[1,res,res])  (all float32)."""
    rng = np.random.default_rng(seed)
    K, E = ring_camera(angle_deg, res)
    z = _capsule_depth(K, E, res, body_radius, body_radius, 1.8 - body_radius).astype(np.float32)
    valid = (z > 0).reshape(-1)
    inv = np.where(z > 0, 1.0 / np.maximum(z, 1e-6), 0.0).astype(np.float32)
    # depth2pc arithmetic (reference lib/utils.py:87-109): Z = 1/(inv+1e-8); xy = (uv+0.5-c) * Z / f
    v, u = np.meshgrid(np.arange(res, dtype=np.float32) + 0.5, np.arange(res, dtype=np.float32) + 0.5, indexing="ij")
    Z = (1.0 / (inv + np.float32(1e-8))).astype(np.float32)
    x = ((u - np.float32(K[0, 2])) * Z / np.float32(K[0, 0])).astype(np.float32)
    y = ((v - np.float32(K[1, 2])) * Z / np.float32(K[1, 1])).astype(np.float32)
    pc = np.stack([x, y, Z], -1).reshape(-1, 3).astype(np.float64)
    R, t = E[:, :3], E[:, 3]
    xyz = ((pc - t) @ R).astype(np.float32)          # R^T (p - t)
    xyz[~valid] = 0
    n = res * res
    rot, scale, opacity, rgb = _attrs(rng, n, np.where(valid, Z.reshape(-1), 2.0) / np.float32(K[0, 0]))
    return dict(K=K, E=E, depth=z, valid=valid, xyz=xyz,
                img=(rgb * 2 - 1).reshape(res, res, 3).transpose(2, 0, 1).copy(),
                rot_maps=rot.reshape(res, res, 4).transpose(2, 0, 1).copy(),
                scale_maps=scale.reshape(res, res, 3).transpose(2, 0, 1).copy(),
                opacity_maps=opacity.reshape(res, res, 1).transpose(2, 0, 1).copy())


def gather_valid(views):
    """What lib/GaussianRender.py:14-33 does: boolean-select valid pixels of both views, concat, rgb*0.5+0.5."""
    out = {k: [] for k in ("xyz", "rgb", "rot", "scale", "opacity")}
    for vw in views:
        m = vw["valid"]
        out["xyz"].append(vw["xyz"][m])
        out["rgb"].append(vw["img"].transpose(1, 2, 0).reshape(-1, 3)[m] * np.float32(0.5) + np.float32(0.5))
        out["rot"].append(vw["rot_maps"].transpose(1, 2, 0).reshape(-1, 4)[m])
        out["scale"].append(vw["scale_maps"].transpose(1, 2, 0).reshape(-1, 3)[m])
        out["opacity"].append(vw["opacity_maps"].transpose(1, 2, 0).reshape(-1, 1)[m])
    return {k: np.ascontiguousarray(np.concatenate(v, 0)) for k, v in out.items()}


def stereo_pair_scene(src_res=1024, render_res=None, seed=SEED, ratio=0.5, body_radius=0.425, bg=(0.0, 0.0, 0.0),
                      keep_maps=False):
    """BASELINE C2/C4 unit: two source views at +-11.25 deg -> ~P pixel-aligned Gaussians + the novel camera.
    Returns the flat rasterizer inputs exactly as gaussian_renderer.render() receives them."""
    render_res = render_res or src_res
    views = [source_view_maps(src_res, -11.25, seed * 2 + 0, body_radius),
             source_view_maps(src_res, +11.25, seed * 2 + 1, body_radius)]
    scale = render_res / src_res
    K0, K1 = views[0]["K"].copy(), views[1]["K"].copy()
    K0[:2] *= scale
    K1[:2] *= scale
    cam = novel_camera(K0, views[0]["E"], K1, views[1]["E"], render_res, render_res, ratio)
    g = gather_valid(views)
    sc = dict(means3D=g["xyz"], colors=g["rgb"], opacity=g["opacity"], scales=g["scale"], rots=g["rot"],
              view=cam["world_view_transform"], proj=cam["full_proj_transform"], campos=cam["camera_center"],
              tanfovx=math.tan(cam["FovX"] * 0.5), tanfovy=math.tan(cam["FovY"] * 0.5), W=render_res, H=render_res,
              bg=np.asarray(bg, np.float32), cam=cam)
    if keep_maps:
        sc["views"] = views
    return sc


def random_cube_scene(P=10_000, res=256, seed=SEED, bg=(0.0, 0.0, 0.0), spread=1.0, scale_mul=1.0):
    """BASELINE C1: P Gaussians uniform in a `spread`-m cube centred on the look-at point, novel cam at angle 0."""
    rng = np.random.default_rng(seed)
    K0, E0 = ring_camera(-11.25, res)
    K1, E1 = ring_camera(+11.25, res)
    cam = novel_camera(K0, E0, K1, E1, res, res, 0.5)
    xyz = (rng.uniform(-0.5, 0.5, (P, 3)) * spread + np.array([0.0, 0.85, 0.0])).astype(np.float32)
    zc = (np.concatenate([xyz, np.ones((P, 1), np.float32)], 1) @ cam["world_view_transform"])[:, 2]
    rot, scale, opacity, rgb = _attrs(rng, P, np.maximum(zc, 0.3) / np.float32(K0[0, 0]))
    scale = np.minimum(scale * np.float32(scale_mul), np.float32(0.01 * max(1.0, scale_mul)))
    return dict(means3D=xyz, colors=rgb, opacity=opacity, scales=scale, rots=rot, view=cam["world_view_transform"],
                proj=cam["full_proj_transform"], campos=cam["camera_center"], tanfovx=math.tan(cam["FovX"] * 0.5),
                tanfovy=math.tan(cam["FovY"] * 0.5), W=res, H=res, bg=np.asarray(bg, np.float32), cam=cam)


def corr_inputs(B=2, D=192, H=64, W=64, seed=SEED, dtype=np.float32):
    """fmap1, fmap2 ~ N(0,1) [B,D,H,W]; coords = x-grid + N(0,6^2) (includes out-of-range), [B,2,H,W]."""
    rng = np.random.default_rng(seed)
    f1 = rng.standard_normal((B, D, H, W)).astype(dtype)
    f2 = rng.standard_normal((B, D, H, W)).astype(dtype)
    xs = np.broadcast_to(np.arange(W, dtype=np.float32), (B, H, W))
    ys = np.broadcast_to(np.arange(H, dtype=np.float32)[:, None], (B, H, W))
    coords = np.stack([xs + rng.normal(0, 6.0, (B, H, W)).astype(np.float32), ys], 1).astype(np.float32)
    return f1, f2, np.ascontiguousarray(coords)


def novel_calib_for_show(intr, extr, ratio=0.5):
    """data['novel_view'] intr[B,3,3] / extr[B,3,4] (float32) as reference lib/utils.py:57-84 builds them for the
    stage-1 preview: scipy Slerp of the two source rotations, linear translation and intrinsics."""
    from scipy.spatial.transform import Rotation, Slerp
    K_out, E_out = [], []
    for b in range(intr.shape[1]):
        i0, i1 = intr[0, b], intr[1, b]
        e0, e1 = extr[0, b], extr[1, b]
        rot = Slerp([0, 1], Rotation.from_matrix(np.stack([e0[:3, :3], e1[:3, :3]])))(ratio)
        pose = np.diag([1.0, 1.0, 1.0, 1.0]).astype(np.float32)
        pose[:3, :3] = rot.as_matrix()
        pose[:3, 3] = ((1.0 - ratio) * e0 + ratio * e1)[:3, 3]
        E_out.append(pose[:3, :])
        K_out.append((1.0 - ratio) * i0 + ratio * i1)
    return np.array(K_out, np.float32), np.array(E_out, np.float32)


def stage1_batch(res=256, B=2, seed=SEED, ratio=0.5, flow_noise=0.05):
    """A synthetic stage-1 validation batch as train_stage1.py:96-100 hands it to TaichiRenderBatch.flow2render: per
    source view (lmain, rmain: the ring cameras at -/+11.25 deg) flow_pred[B,1,S,S] (the capsule's inverse depth turned
    into disparity flow, plus seeded noise), mask[B,1,S,S], intr / ref_intr [B,3,3], extr[B,4,4], Tf_x[B], img[B,3,S,S]
    in [-1,1]; and data['novel_view'] intr / extr from novel_calib_for_show.  All float32 numpy."""
    rng = np.random.default_rng(seed)
    names = ("lmain", "rmain")
    out = {n: {k: [] for k in ("flow_pred", "mask", "intr", "extr", "ref_intr", "Tf_x", "img")} for n in names}
    v, u = np.meshgrid(np.arange(res) + 0.5, np.arange(res) + 0.5, indexing="ij")
    for _ in range(B):
        radius = 0.425 * float(rng.uniform(0.9, 1.05))
        phase = float(rng.uniform(0, 6.28))
        tfx = -0.6 * res * float(rng.uniform(0.95, 1.05))              # depth = (flow - offset) / Tf_x
        for name, ang in zip(names, (-11.25, 11.25)):
            K, E = ring_camera(ang, res)
            z = _capsule_depth(K, E, res, radius, radius, 1.8 - radius)
            hit = z > 0
            inv = np.where(hit, 1.0 / np.maximum(z, 1e-6), 0.0)
            Kr = K.copy()
            Kr[0, 2] += 0.1 * res
            offset = Kr[0, 2] - K[0, 2]
            flow = offset + inv * tfx + flow_noise * rng.standard_normal((res, res))
            pc = np.stack([(u - K[0, 2]) * z / K[0, 0], (v - K[1, 2]) * z / K[1, 1], z], -1)
            xyz = (pc - E[:, 3]) @ E[:, :3]
            img = np.where(hit[..., None], 0.8 * np.sin(xyz @ np.array([[9.0, 5.0, 7.0], [4.0, 11.0, 6.0],
                                                                         [7.0, 3.0, 10.0]]).T + phase), -1.0)
            d = out[name]
            d["flow_pred"].append(flow[None]); d["mask"].append(hit[None].astype(np.float64))
            d["intr"].append(K); d["extr"].append(np.vstack([E, [0, 0, 0, 1]])); d["ref_intr"].append(Kr)
            d["Tf_x"].append(tfx); d["img"].append(img.transpose(2, 0, 1))
    data = {n: {k: np.ascontiguousarray(np.array(a, np.float32)) for k, a in out[n].items()} for n in names}
    K_n, E_n = novel_calib_for_show(np.stack([data[n]["intr"] for n in names]),
                                    np.stack([data[n]["extr"] for n in names]), ratio)
    data["novel_view"] = {"intr": K_n, "extr": E_n}
    return data
