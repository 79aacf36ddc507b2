"""Camera images (qs_render, quadruped_springs_b200/render.py, env.render / render_images, BatchedVecEnv.get_images,
VideoRecorder).

An independent fp64 ray caster lives here.  Its geometry comes from the URDF (urdf_numpy_model.Model.fk and the
collision entries of tests/golden/go1_urdf.json), not from the kernel's constants; its look (light, ambient, colours,
sky, checkerboard) restates the table of qs_render.cu.  The CPU tests pin the camera matrices against closed forms and
the caster against analytic hits; the GPU tests (-m gpu) hold the kernel to the caster, to known answers, to batch and
output-subset invariance, and check that rendering changes nothing of the env."""
import math
import os
import types

import numpy as np
import pytest
import torch

from conftest import load_golden
from urdf_numpy_model import LINK_ORDER, Model, rpy_R

CFG3 = dict(enable_springs=True, task_env="JUMPING_FORWARD", motor_control_mode="CARTESIAN_PD",
            action_space_mode="SYMMETRIC", observation_space_mode="ARS_BASIC")   # bench.py configuration 3
FOOT_LINKS = (5, 9, 13, 17)

# the look, as in qs_render.cu
LIGHT = np.array([0.3, -0.4, 0.8660254], dtype=np.float32).astype(np.float64)
AMBIENT = 0.35
SHADOW_OFFSET = 1e-4
ALBEDO = np.array([[80, 88, 104], [214, 132, 44], [66, 128, 196], [150, 156, 164], [40, 40, 44]], dtype=np.float64)
GROUND = np.array([[176, 176, 176], [128, 128, 128]], dtype=np.float64)
SKY = np.array([160, 196, 232], dtype=np.float64)


def seg_code(link):
    return 1 + ((link + 1) << 24)


# ------------------------------------------------------------------ the fp64 reference caster
def primitives(state):
    """[(link, shape, R (local -> world), centre, extents)] of the 18 collision primitives, from the URDF"""
    state = np.asarray(state, dtype=np.float64)
    model = Model()
    poses, _ = model.fk(state[0:3], state[3:7], state[13:25])
    out = []
    for link, name in enumerate(LINK_ORDER[1:]):
        col = model.links[name]["collision"][0]
        Rl, pl = poses[name]
        R = Rl @ rpy_R(col["rpy"])
        c = pl + Rl @ np.asarray(col["xyz"], dtype=np.float64)
        if col["type"] == "box":
            out.append((link, "box", R, c, np.asarray(col["size"], dtype=np.float64) / 2))
        elif col["type"] == "cylinder":
            out.append((link, "cyl", R, c, np.array([col["radius"][0], col["length"][0] / 2, 0.0])))
        else:
            out.append((link, "sphere", R, c, np.array([col["radius"][0], 0.0, 0.0])))
    return out


def intersect(shape, R, c, e, o, d):
    """rays o + t d ([n, 3] each, d unit) against a solid: entry t, exit t (entry > exit: missed), outward world normal
    at the entry"""
    ol, dl = (o - c) @ R, d @ R
    n = o.shape[0]
    nl = np.zeros((n, 3))
    with np.errstate(divide="ignore", invalid="ignore"):
        if shape == "sphere":
            r = e[0]
            b = (ol * dl).sum(1)
            q = ol - b[:, None] * dl
            disc = r * r - (q * q).sum(1)
            s = np.sqrt(np.maximum(disc, 0))
            tn, tf = np.where(disc >= 0, -b - s, 1.0), np.where(disc >= 0, -b + s, 0.0)
            nl = (ol + tn[:, None] * dl) / r
        elif shape == "box":
            t1, t2 = (-e - ol) / dl, (e - ol) / dl
            lo, hi = np.fmin(t1, t2), np.fmax(t1, t2)
            ax = lo.argmax(1)
            tn, tf = lo.max(1), hi.min(1)
            nl[np.arange(n), ax] = np.where(dl[np.arange(n), ax] > 0, -1.0, 1.0)
        else:
            r, hl = e[0], e[1]
            a2 = dl[:, 0] ** 2 + dl[:, 1] ** 2
            b = ol[:, 0] * dl[:, 0] + ol[:, 1] * dl[:, 1]
            cr = ol[:, 0] * dl[:, 1] - ol[:, 1] * dl[:, 0]
            disc = a2 * r * r - cr * cr
            s = np.sqrt(np.maximum(disc, 0))
            par = a2 <= 1e-12
            inside = ol[:, 0] ** 2 + ol[:, 1] ** 2 <= r * r
            s0 = np.where(par, np.where(inside, -np.inf, 1.0), np.where(disc >= 0, (-b - s) / a2, 1.0))
            s1 = np.where(par, np.where(inside, np.inf, 0.0), np.where(disc >= 0, (-b + s) / a2, 0.0))
            z1, z2 = (-hl - ol[:, 2]) / dl[:, 2], (hl - ol[:, 2]) / dl[:, 2]
            z0, zz = np.fmin(z1, z2), np.fmax(z1, z2)
            tn, tf = np.maximum(s0, z0), np.minimum(s1, zz)
            side = s0 >= z0
            p = ol + tn[:, None] * dl
            rn = np.hypot(p[:, 0], p[:, 1])
            nl = np.where(side[:, None], np.stack([p[:, 0] / rn, p[:, 1] / rn, 0 * rn], 1),
                          np.stack([0 * rn, 0 * rn, np.where(dl[:, 2] > 0, -1.0, 1.0)], 1))
    return tn, tf, nl @ R.T


def camera_rays(cam, W, H):
    """per pixel (row-major): ray origin on the near plane, unit direction, eye depth at the origin and per unit t, far"""
    cam = np.asarray(cam, dtype=np.float32).astype(np.float64)
    V, P = cam[:16].reshape(4, 4).T, cam[16:].reshape(4, 4).T
    Minv = np.linalg.inv(P @ V)
    r, c = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    x, y = (2 * (c.ravel() + 0.5) / W - 1), (1 - 2 * (r.ravel() + 0.5) / H)
    one = np.ones_like(x)
    hn = np.stack([x, y, -one, one], 1) @ Minv.T
    hf = np.stack([x, y, one, one], 1) @ Minv.T
    o = hn[:, :3] / hn[:, 3:]
    d = hf[:, :3] / hf[:, 3:] - o
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    z0 = -(o @ V[2, :3] + V[2, 3])
    g = -(d @ V[2, :3])
    far = P[2, 3] / (P[2, 2] + 1)
    return o, d, z0, g, far


def reference_render(state, cam, W, H):
    """seg, depth, rgb (float, unrounded) of one image, plus the shadow flag and the ground-checker parity per pixel and
    the rgb of the other shadow flag / other parity (for pixels on those edges)"""
    o, d, z0, g, far = camera_rays(cam, W, H)
    n = o.shape[0]
    tmax = (far - z0) / g
    with np.errstate(divide="ignore", invalid="ignore"):
        tg = -o[:, 2] / d[:, 2]
    ground = (tg >= 0) & (tg <= tmax)
    tbest = np.where(ground, tg, tmax)
    hit = np.where(ground, -1, -2)
    normal = np.tile([0.0, 0.0, 1.0], (n, 1))
    prims = primitives(state) if np.isfinite(state).all() else []
    for link, shape, R, c, e in prims:
        tn, tf, nw = intersect(shape, R, c, e, o, d)
        better = (tn <= tf) & (tn >= 0) & (tn < tbest)
        tbest = np.where(better, tn, tbest)
        hit = np.where(better, link, hit)
        normal = np.where(better[:, None], nw, normal)
    depth = np.where(hit == -2, far, z0 + tbest * g)
    seg = np.where(hit == -2, -1, np.where(hit == -1, 0, 1 + ((hit + 1) << 24)))
    p = o + tbest[:, None] * d
    ndl = np.maximum(0.0, normal @ LIGHT)
    so = p + SHADOW_OFFSET * normal
    lit = np.ones(n, dtype=bool)
    for link, shape, R, c, e in prims:
        tn, tf, _ = intersect(shape, R, c, e, so, np.tile(LIGHT, (n, 1)))
        lit &= ~((tn <= tf) & (tf >= 0))
    parity = (np.floor(p[:, 0]).astype(np.int64) + np.floor(p[:, 1]).astype(np.int64)) & 1
    kind = np.where(hit < 2, 0, 1 + (hit - 2) % 4)

    def colour(s, par):
        alb = np.where((hit == -1)[:, None], GROUND[par], ALBEDO[np.clip(kind, 0, 4)])
        shade = AMBIENT + (1 - AMBIENT) * ndl * s
        return np.where((hit == -2)[:, None], SKY, alb * shade[:, None])

    s = (lit & (ndl > 0)).astype(np.float64)
    rgb = colour(s, parity)
    rgb_other_shadow = colour(1 - s, parity)
    rgb_other_parity = colour(s, 1 - parity)
    frac = np.minimum(np.abs(p[:, 0] - np.round(p[:, 0])), np.abs(p[:, 1] - np.round(p[:, 1])))
    checker_edge = (hit == -1) & (frac < 1e-4 * (1 + depth))
    sh = lambda a: a.reshape(H, W, *a.shape[1:])
    return dict(seg=sh(seg), depth=sh(depth), rgb=sh(rgb), lit=sh(s > 0), rgb_other_shadow=sh(rgb_other_shadow),
                rgb_other_parity=sh(rgb_other_parity), checker_edge=sh(checker_edge))


def edge_of(lab):
    """pixels with a 4-neighbour of another label"""
    e = np.zeros(lab.shape, dtype=bool)
    e[1:] |= lab[1:] != lab[:-1]
    e[:-1] |= lab[:-1] != lab[1:]
    e[:, 1:] |= lab[:, 1:] != lab[:, :-1]
    e[:, :-1] |= lab[:, :-1] != lab[:, 1:]
    return e


def project(cam, x):
    cam = np.asarray(cam, dtype=np.float64)
    V, P = cam[:16].reshape(4, 4).T, cam[16:].reshape(4, 4).T
    h = P @ V @ np.append(x, 1.0)
    return h[:3] / h[3]


# ------------------------------------------------------------------ CPU: camera matrices
from quadruped_springs_b200.render import (  # noqa: E402
    compute_projection_matrix_fov, compute_view_matrix_from_yaw_pitch_roll, follow_cameras, tile_images)


@pytest.mark.parametrize("yaw,pitch,dist", [(0, -30, 1.0), (45, -10, 2.5), (-120, -70, 0.7), (200, 15, 3.0), (90, -89, 2)])
def test_view_matrix_closed_form(yaw, pitch, dist):
    tgt = np.array([0.3, -1.2, 0.25])
    V = compute_view_matrix_from_yaw_pitch_roll(torch.tensor(tgt)[None], dist, yaw, pitch).numpy()[0]
    M = V.astype(np.float64).reshape(4, 4).T
    R, t = M[:3, :3], M[:3, 3]
    y, p = math.radians(yaw), math.radians(pitch)
    eye = tgt + dist * np.array([math.cos(p) * math.sin(y), -math.cos(p) * math.cos(y), -math.sin(p)])
    up = np.array([math.sin(p) * math.sin(y), -math.sin(p) * math.cos(y), math.cos(p)])
    assert np.allclose(-R.T @ t, eye, atol=2e-6)
    assert np.allclose(R[1], up, atol=1e-6)
    assert np.allclose(R @ R.T, np.eye(3), atol=1e-6)
    if (yaw, pitch) == (0, -30):
        assert np.allclose(eye, tgt + dist * np.array([0, -math.cos(math.pi / 6), 0.5]))
    cam = torch.cat([torch.tensor(V), compute_projection_matrix_fov(60, 4 / 3, 0.1, 100)]).numpy()
    assert np.allclose(project(cam, tgt)[:2], 0, atol=1e-6)


def test_projection_near_far_and_follow_defaults():
    near, far = 0.1, 100.0
    P = compute_projection_matrix_fov(60, 480 / 360, near, far).numpy().astype(np.float64).reshape(4, 4).T
    for z, ndc in ((near, -1.0), (far, 1.0)):
        h = P @ np.array([0.0, 0.0, -z, 1.0])
        assert abs(h[2] / h[3] - ndc) < 1e-5
    assert abs(P[1, 1] - 1 / math.tan(math.radians(30))) < 1e-6 and abs(P[0, 0] - P[1, 1] * 360 / 480) < 1e-6
    cams = follow_cameras(torch.tensor([[1.0, 2.0, 0.3], [0.0, 0.0, 0.1]]))
    assert cams.shape == (2, 32) and cams.dtype == torch.float32
    M = cams[0, :16].double().numpy().reshape(4, 4).T
    assert np.allclose(-M[:3, :3].T @ M[:3, 3], [1.0, 2.0 - math.cos(math.pi / 6), 0.3 + 0.5], atol=2e-6)
    assert np.array_equal(cams[0, 16:].numpy(), compute_projection_matrix_fov(60, 480 / 360, 0.1, 100).numpy())


def test_tile_images_is_sb3s():
    imgs = np.arange(5 * 2 * 3 * 3, dtype=np.uint8).reshape(5, 2, 3, 3)
    t = tile_images(imgs)
    assert t.shape == (3 * 2, 2 * 3, 3)          # ceil(sqrt(5)) = 3 rows, ceil(5 / 3) = 2 columns
    assert np.array_equal(t[0:2, 0:3], imgs[0]) and np.array_equal(t[0:2, 3:6], imgs[1])
    assert np.array_equal(t[4:6, 0:3], imgs[4]) and not t[4:6, 3:6].any()
    four = tile_images(imgs[:4])
    assert four.shape == (4, 6, 3) and np.array_equal(four[2:4, 3:6], imgs[3])


# ------------------------------------------------------------------ CPU: the reference caster against analytic answers
def _rot(axis, th):
    from urdf_numpy_model import rot_axis
    return rot_axis(np.asarray(axis, float) / np.linalg.norm(axis), th)


def test_reference_primitives_hit_at_known_distances():
    R = _rot([1, 2, 3], 0.7)
    c = np.array([0.5, -0.2, 1.0])
    o_loc = np.array([[0.0, 0.0, -5.0], [-10.0, 0.0, 0.0], [-3.0, 0.0, 0.0], [0.0, 0.0, -4.0], [0.3, 0.0, -4.0]])
    d_loc = np.array([[0.0, 0.0, 1.0], [1.0, 0.0, 0.0], [1.0, 0.0, 0.0], [0.0, 0.0, 1.0], [0.0, 0.0, 1.0]])
    o, d = c + o_loc @ R.T, d_loc @ R.T
    cases = [("sphere", np.array([1.0, 0, 0]), 0, 4.0, [0, 0, -1]),
             ("box", np.array([1.0, 2.0, 3.0]), 1, 9.0, [-1, 0, 0]),
             ("cyl", np.array([0.5, 1.0, 0]), 2, 2.5, [-1, 0, 0]),      # side
             ("cyl", np.array([0.5, 1.0, 0]), 3, 3.0, [0, 0, -1]),      # cap
             ("cyl", np.array([0.5, 1.0, 0]), 4, 3.0, [0, 0, -1])]      # cap, off axis
    for shape, e, i, t, nloc in cases:
        tn, tf, nw = intersect(shape, R, c, e, o[i:i + 1], d[i:i + 1])
        assert abs(tn[0] - t) < 1e-12 and tf[0] > tn[0], (shape, i)
        assert np.allclose(nw[0], R @ np.asarray(nloc, float), atol=1e-12), (shape, i)
    # misses: past the sphere, beside the box, past the cylinder's cap rim
    assert not (lambda r: r[0][0] <= r[1][0])(intersect("sphere", R, c, np.array([1.0, 0, 0]), c + np.array([[0, 1.01, -5]]) @ R.T, d[0:1]))
    assert not (lambda r: r[0][0] <= r[1][0])(intersect("box", R, c, np.array([1.0, 2.0, 3.0]), c + np.array([[-10, 2.01, 0]]) @ R.T, d[1:2]))
    assert not (lambda r: r[0][0] <= r[1][0])(intersect("cyl", R, c, np.array([0.5, 1.0, 0]), c + np.array([[0.51, 0, -4]]) @ R.T, d[3:4]))


def test_reference_ground_depth_and_foot_label():
    g = load_golden("rollout_jip_jump.npz")
    state = np.asarray(g["init_state"], dtype=np.float64)
    W, H = 480, 360
    cam = follow_cameras(torch.tensor(state[None, :3], dtype=torch.float32), W, H)[0].numpy()
    ref = reference_render(state, cam, W, H)
    # ground in closed form: pixel ray in eye space (x / P00, y / P11, -1), depth = -eye_z / dir_z
    V = cam[:16].astype(np.float64).reshape(4, 4).T
    P = cam[16:].astype(np.float64).reshape(4, 4).T
    eye = -V[:3, :3].T @ V[:3, 3]
    r, c = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    x, y = 2 * (c + 0.5) / W - 1, 1 - 2 * (r + 0.5) / H
    dz = (V[:3, :3].T @ np.stack([x / P[0, 0], y / P[1, 1], -np.ones_like(x)]).reshape(3, -1))[2].reshape(H, W)
    plane = -eye[2] / dz
    m = ref["seg"] == 0
    assert m.sum() > 0.3 * H * W
    assert np.allclose(ref["depth"][m], plane[m], rtol=1e-12, atol=1e-12)
    # the centre of each visible foot projects to a pixel labelled with that foot
    poses, _ = Model().fk(state[0:3], state[3:7], state[13:25])
    seen = 0
    for leg, link in enumerate(FOOT_LINKS):
        ndc = project(cam, poses[LINK_ORDER[1 + link]][1])
        col, row = int((ndc[0] + 1) / 2 * W), int((1 - ndc[1]) / 2 * H)
        if ref["seg"][row, col] == seg_code(link):
            seen += 1
        else:   # hidden: another robot primitive is in front of it
            assert ref["seg"][row, col] > 0
    assert seen >= 2


def test_save_mp4_round_trip(tmp_path):
    cv2 = pytest.importorskip("cv2")
    from quadruped_springs_b200.render import VideoRecorder
    env = types.SimpleNamespace(device=torch.device("cpu"), num_envs=4, env_time_step=0.01)
    rec = VideoRecorder(env, [0, 1, 2], width=64, height=48, max_frames=7)
    rec._buf.copy_(torch.randint(0, 255, rec._buf.shape, dtype=torch.uint8))
    rec._count = 6
    path = str(tmp_path / "clip.mp4")
    rec.save_mp4(path, fps=25)
    cap = cv2.VideoCapture(path)
    frames = 0
    while True:
        ok, f = cap.read()
        if not ok:
            break
        assert f.shape == (2 * 48, 2 * 64, 3)
        frames += 1
    cap.release()
    assert frames == 6


# ------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def qs():
    import quadruped_springs_b200 as m
    assert torch.cuda.is_available()
    return m


def _settled_state(qs):
    env = qs.BatchedQuadrupedGymEnv(num_envs=1, seed=3, auto_reset=False, enable_noise=False,
                                    enable_springs=True, task_env="JUMPING_IN_PLACE", observation_space_mode="ARS_BASIC")
    env.reset()
    s = env.get_state()[0].cpu().numpy().astype(np.float64)
    env.close()
    return s


def _quat_axis(axis, th):
    a = np.asarray(axis, float) / np.linalg.norm(axis)
    return np.append(a * math.sin(th / 2), math.cos(th / 2))


def _case_states(qs):
    """settled, mid-flight (jump rollout), inverted (backflip rollout), legs at their joint limits, tilted 60 deg,
    out of frame"""
    settled = _settled_state(qs)
    flight = load_golden("rollout_jip_jump.npz")["state"][50].astype(np.float64)
    inverted = load_golden("rollout_backflip.npz")["state"][96].astype(np.float64)
    limits = settled.copy()
    joints = [j for j in Model().joint_of_child.values() if j["type"] == "revolute"]
    lim = {j["name"]: (j["lower"], j["upper"]) for j in joints}
    legs = ("FR", "FL", "RR", "RL")
    for k, leg in enumerate(legs):
        for j, part in enumerate(("hip", "thigh", "calf")):
            lo, hi = lim[f"{leg}_{part}_joint"]
            limits[13 + 3 * k + j] = lo if (k + j) % 2 == 0 else hi
    limits[2] = 0.45
    tilted = settled.copy()
    tilted[3:7] = _quat_axis([1.0, 0.6, 0.0], math.radians(60))
    tilted[2] = 0.35
    away = settled.copy()
    away[0:3] = [0.5, -6.0, 0.3]
    return [settled, flight, inverted, limits, tilted, away]


def _cams(targets, W, H):
    """follow, top-down, low and grazing cameras of each target point"""
    from quadruped_springs_b200.render import compute_projection_matrix_fov, compute_view_matrix_from_yaw_pitch_roll
    t = torch.tensor(np.asarray(targets), dtype=torch.float32)
    P = compute_projection_matrix_fov(60, W / H, 0.1, 100).expand(t.shape[0], 16)
    follow = follow_cameras(t, W, H)
    top = torch.cat([compute_view_matrix_from_yaw_pitch_roll(t, 2.0, 20, -89), P], 1)
    low = t.clone()
    low[:, 2] = 0.05
    graze = torch.cat([compute_view_matrix_from_yaw_pitch_roll(low, 1.3, 35, -7), P], 1)
    return [follow, top, graze]


@pytest.mark.gpu
def test_kernel_matches_reference(qs):
    W, H = 96, 72
    states = _case_states(qs)
    targets = [s[0:3] for s in states[:-1]] + [np.array([0.5, 0.0, 0.3])]
    cams = _cams(targets, W, H)
    st = torch.tensor(np.stack(states * 3), dtype=torch.float32, device="cuda")
    cm = torch.cat(cams).cuda()
    out = qs.render.render_states(st, cm, W, H, rgb=True, depth=True, segmentation=True)
    seg, dep, rgb = (out[k].cpu().numpy() for k in ("segmentation", "depth", "rgb"))
    worst = dict(seg=1.0, depth=0.0, rgb_alt=0)
    robot_px = 0
    for i in range(st.shape[0]):
        ref = reference_render(st[i].double().cpu().numpy(), cm[i].cpu().numpy(), W, H)
        same = seg[i] == ref["seg"]
        frac = same.mean()
        worst["seg"] = min(worst["seg"], frac)
        assert frac >= 0.995, (i, frac)
        assert edge_of(ref["seg"])[~same].all(), (i, np.argwhere(~same & ~edge_of(ref["seg"]))[:5])
        err = np.abs(dep[i] - ref["depth"]) - (1e-4 + 1e-5 * ref["depth"])
        assert (err[same] <= 0).all(), (i, float(err[same].max()))
        worst["depth"] = max(worst["depth"], float((np.abs(dep[i] - ref["depth"]))[same].max()))
        # rgb: within 2 of the reference, or of its other shadow flag / checker parity on those edges
        d0 = np.abs(rgb[i] - ref["rgb"]).max(-1)
        d1 = np.abs(rgb[i] - ref["rgb_other_shadow"]).max(-1)
        d2 = np.abs(rgb[i] - ref["rgb_other_parity"]).max(-1)
        ok0 = d0 <= 2
        alt = (~ok0) & ((edge_of(ref["lit"]) & (d1 <= 2)) | (ref["checker_edge"] & (d2 <= 2)))
        assert (ok0 | alt)[same].all(), (i, np.argwhere(same & ~(ok0 | alt))[:5])
        assert alt.mean() <= 0.005, (i, alt.mean())
        worst["rgb_alt"] = max(worst["rgb_alt"], int(alt.sum()))
        robot_px += int((ref["seg"] > 0).sum())
    # the out-of-frame robot is not in any of its three images; every other case shows the robot
    for j in range(3):
        assert (seg[6 * j + 5] <= 0).all()
        assert all((seg[6 * j + i] > 0).any() for i in range(5))
    print(worst, "robot pixels", robot_px)


@pytest.mark.gpu
def test_known_answers(qs):
    from quadruped_springs_b200.render import compute_projection_matrix_fov, compute_view_matrix_from_yaw_pitch_roll
    W, H = 160, 120
    settled = _settled_state(qs)
    high = settled.copy()
    high[0:3] = [0.0, 0.0, 50.0]
    bad = settled.copy()
    bad[20] = float("nan")
    inf = settled.copy()
    inf[30] = float("inf")
    tgt = torch.tensor([[0.0, 0.0, 0.3]])
    P = compute_projection_matrix_fov(60, W / H, 0.1, 100)[None]
    cams = [torch.cat([compute_view_matrix_from_yaw_pitch_roll(tgt, 1.0, 180, -30), P], 1),
            torch.cat([compute_view_matrix_from_yaw_pitch_roll(tgt, 2.0, 0, -89), P], 1)]
    for cam in cams:
        cam = cam.cuda()
        outs = [qs.render.render_states(torch.tensor(s[None], dtype=torch.float32, device="cuda"), cam, W, H, True, True, True)
                for s in (high, bad, inf)]
        for o in outs[1:]:
            for k in o:
                assert torch.equal(o[k], outs[0][k]), k
        seg, dep = outs[0]["segmentation"][0].cpu().numpy(), outs[0]["depth"][0].cpu().numpy()
        assert set(np.unique(seg)) <= {0, -1} and (seg == 0).mean() > 0.3
        V = cam[0, :16].double().cpu().numpy().reshape(4, 4).T
        Pm = cam[0, 16:].double().cpu().numpy().reshape(4, 4).T
        eye = -V[:3, :3].T @ V[:3, 3]
        r, c = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
        x, y = 2 * (c + 0.5) / W - 1, 1 - 2 * (r + 0.5) / H
        dz = (V[:3, :3].T @ np.stack([x / Pm[0, 0], y / Pm[1, 1], -np.ones_like(x)]).reshape(3, -1))[2].reshape(H, W)
        plane = -eye[2] / dz
        g = seg == 0
        assert np.all(np.abs(dep[g] - plane[g]) <= 1e-4 + 1e-5 * plane[g])
        assert np.allclose(dep[seg == -1], 100.0, rtol=1e-5)
        rgb = outs[0]["rgb"][0].cpu().numpy()
        assert (rgb[seg == -1] == SKY.astype(np.uint8)).all()
    # every visible foot centre lands on its pixel, through the kernel
    W, H = 480, 360
    state = settled
    cam = follow_cameras(torch.tensor(state[None, :3], dtype=torch.float32), W, H)
    seg = qs.render.render_states(torch.tensor(state[None], dtype=torch.float32, device="cuda"), cam.cuda(), W, H,
                                  rgb=False, segmentation=True)["segmentation"][0].cpu().numpy()
    ref = reference_render(state, cam[0].numpy(), W, H)
    poses, _ = Model().fk(state[0:3], state[3:7], state[13:25])
    seen = 0
    for link in FOOT_LINKS:
        ndc = project(cam[0].numpy(), poses[LINK_ORDER[1 + link]][1])
        col, row = int((ndc[0] + 1) / 2 * W), int((1 - ndc[1]) / 2 * H)
        if ref["seg"][row, col] == seg_code(link):
            assert seg[row, col] == seg_code(link), link
            seen += 1
    assert seen >= 2


def _batch_states(qs, n, steps=30):
    env = qs.BatchedQuadrupedGymEnv(num_envs=n, seed=7, auto_reset=True, enable_noise=True, **CFG3)
    env.reset()
    rng = np.random.default_rng(0)
    for _ in range(steps):
        env.step(torch.tensor(rng.uniform(-1, 1, (n, env.action_dim)), dtype=torch.float32, device="cuda"))
    s = env.get_state()
    env.close()
    return s


@pytest.mark.gpu
def test_batch_subset_and_determinism(qs):
    n, W, H = 1024, 64, 48
    st = _batch_states(qs, n)
    cams = follow_cameras(st[:, :3].cpu(), W, H).cuda()
    full = qs.render.render_states(st, cams, W, H, True, True, True)
    again = qs.render.render_states(st, cams, W, H, True, True, True)
    for k in full:
        assert torch.equal(full[k], again[k]), k
    assert (full["segmentation"] > 0).flatten(1).any(1).all()
    for i in (0, 1, 37, 511, 1023):
        one = qs.render.render_states(st[i:i + 1].clone(), cams[i].clone(), W, H, True, True, True)
        for k in full:
            assert torch.equal(one[k][0], full[k][i]), (i, k)
    for rgb, depth, seg in ((True, False, False), (False, True, False), (False, False, True), (False, True, True),
                            (True, False, True)):
        part = qs.render.render_states(st, cams, W, H, rgb, depth, seg)
        assert set(part) == {k for k, f in (("rgb", rgb), ("depth", depth), ("segmentation", seg)) if f}
        for k in part:
            assert torch.equal(part[k], full[k]), k
    # an image size that is not a whole number of 4-byte words takes the byte path of the RGB store
    odd = qs.render.render_states(st[:3], cams[:3], 33, 17)["rgb"]
    for i in range(3):
        assert torch.equal(odd[i], qs.render.render_states(st[i:i + 1], cams[i], 33, 17)["rgb"][0])


@pytest.mark.gpu
@pytest.mark.parametrize("graph", ["1", "0"])
def test_rendering_changes_nothing(qs, graph, monkeypatch):
    monkeypatch.setenv("QS_GRAPH", graph)
    n, steps = 4096, 200
    kw = dict(num_envs=n, seed=21, auto_reset=True, enable_noise=True, **CFG3)
    a, b = qs.BatchedQuadrupedGymEnv(**kw), qs.BatchedQuadrupedGymEnv(**kw)
    a.reset(), b.reset()
    ids = torch.randperm(n, generator=torch.Generator().manual_seed(1))[:64].cuda()
    rng = np.random.default_rng(2)
    drawn = 0
    for step in range(steps):
        act = torch.tensor(rng.uniform(-1, 1, (n, a.action_dim)), dtype=torch.float32, device="cuda")
        oa, ra, da, ia = a.step(act)
        ob, rb, db, ib = b.step(act)
        assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(da, db), step
        assert torch.equal(ia["TimeLimit.truncated"], ib["TimeLimit.truncated"]), step
        img = a.render_images(ids, 64, 64, depth=True, segmentation=True)
        drawn += int((img["segmentation"] > 0).sum())
    assert torch.equal(a.get_state(), b.get_state())
    for key in ("state", "tau_motor", "tau_spring", "foot_force", "contact", "task", "ep_return", "env_steps"):
        assert torch.equal(a._views[key], b._views[key]), key
    assert drawn > 0


@pytest.mark.gpu
def test_interfaces(qs, tmp_path):
    env = qs.BatchedQuadrupedGymEnv(num_envs=8, seed=4, auto_reset=True, enable_noise=False, **CFG3)
    env.reset()
    img = env.render()
    assert isinstance(img, np.ndarray) and img.dtype == np.uint8 and img.shape == (360, 480, 3)
    assert np.array_equal(img, env.render_images([0])["rgb"][0].cpu().numpy())
    assert env.render("human").size == 0
    with pytest.raises(ValueError):
        qs.BatchedQuadrupedGymEnv(num_envs=1, render=True)
    # VecEnv: get_images and the 2 x 2 tiling
    venv = qs.BatchedVecEnv(num_envs=8, render_env_ids=[0, 1, 2, 3], seed=4, enable_noise=False, **CFG3)
    venv.reset()
    venv.step(np.zeros((8, venv.action_space.shape[0]), dtype=np.float32))
    ims = venv.get_images()
    assert len(ims) == 4 and all(i.shape == (360, 480, 3) and i.dtype == np.uint8 for i in ims)
    big = venv.render("rgb_array")
    assert big.shape == (720, 960, 3)
    assert np.array_equal(big[:360, :480], ims[0]) and np.array_equal(big[:360, 480:], ims[1])
    assert np.array_equal(big[360:, :480], ims[2]) and np.array_equal(big[360:, 480:], ims[3])
    with pytest.raises(ValueError):
        qs.BatchedVecEnv(env=venv.env, render_env_ids=[8])
    # VideoRecorder frames are the per-step render_images calls
    rec = qs.VideoRecorder(env, [1, 5], width=96, height=72, max_frames=4)
    rng = np.random.default_rng(3)
    expect = []
    for _ in range(4):
        env.step(torch.tensor(rng.uniform(-1, 1, (8, env.action_dim)), dtype=torch.float32, device="cuda"))
        rec.capture()
        expect.append(env.render_images([1, 5], 96, 72)["rgb"])
    assert torch.equal(rec.frames, torch.stack(expect))
    with pytest.raises(RuntimeError):
        rec.capture()
    pytest.importorskip("cv2")
    rec.save_mp4(str(tmp_path / "v.mp4"))
    assert os.path.getsize(tmp_path / "v.mp4") > 0
    # bad arguments
    st = env.get_state()
    cam = follow_cameras(st[:, :3].cpu()).cuda()
    R = qs.render.render_states
    with pytest.raises(ValueError):
        R(st[:0], cam[:0])
    with pytest.raises(ValueError):
        R(st, cam, width=0)
    with pytest.raises(ValueError):
        R(st[:1], cam[:1], width=5000)
    with pytest.raises(ValueError):
        R(st, cam, rgb=False)
    with pytest.raises(ValueError):
        R(st, cam[:, :16])
    with pytest.raises(ValueError):
        R(st, cam[:3])
    assert torch.equal(R(st[:1], cam[0])["rgb"], R(st[:1], cam[:1])["rgb"])   # one [32] camera serves every row
    env.close()
