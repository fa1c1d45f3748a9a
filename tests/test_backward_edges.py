"""The backward pass at the forward's edge cases, against the float64 torch reference (tests/torch_reference.py,
tests/torch_reference_aux.py): the 0.99 alpha cap and opacity extremes, scale_modifier, long unsaturated tile lists,
far Gaussians past the sort's fourth depth pass, scenes without prepared alpha constants, a context whose workspaces
another frame has grown and overwritten, and windows of full-size frames.

Every case is held to two bars.  A per-Gaussian bar: with e_i = |g_i - r_i| and m_i = |r_i| the row norms of the GPU's
and the reference's gradient of Gaussian i, e_i <= RTOL m_i + ATOL max_j m_j must hold for all but max(3, 1e-4 P) of
the P Gaussians checked.  And the whole-tensor bar of test_backward.py (relative L2 <= 1e-3, cosine >= 0.9999) on the
rows the per-Gaussian bar does not except.  The exceptions are of two kinds.  Saturation ties: the GPU evaluates alpha
with ex2, the reference with exp, so a pixel can stop one entry apart.  And float32 roundoff in the covariance chain of
needle-thin Gaussians: in the C2 corner window one Gaussian with scales (0.015, 1.6, 0.067) gets 9 % error in
grad_rotq, which the float32 build of lcgs_grad.cuh reproduces from the reference's exact 2D gradient and the double
build does not (its conic gradient entries are ~3000 and cancel); in a window of 651 Gaussians that one row would
decide the whole-tensor bar.  A whole-tensor bar alone lets a wrong sub-population through: passing the gradient
straight through the 0.99 cap for every fifth Gaussian moves grad_scale by only 5e-4 relative L2.

Measured on an NVIDIA B200 (1000 W power limit): the median of e_i / m_i per tensor and case is 1e-6 to 1.5e-3 (the
largest in the full-size windows, where dL/dimg covers 9 tiles); the smallest RTOL (with ATOL = RTOL / 10) at which a
tensor passes is at most 1.8e-4 in every case but the 640000x48 window, where it is 3.1e-4 (grad_scale).  RTOL = 1e-3
leaves a margin of 3x there and 5x elsewhere.

Each full-size window takes about 10 s, most of it the oracle's frame and the 5.8 M or 6.1 M-Gaussian scene."""
import ctypes as C
import functools

import numpy as np
import pytest
import torch

from luisacomputegaussiansplatting_b200 import scenes
from oracle import oracle as orc

import torch_reference as tr
from test_backward import NAMES, gpu_backward, metrics, reference, run_backward, scene_arrays
from test_backward_aux import gpu_backward_aux, reference_aux

pytestmark = pytest.mark.gpu

RTOL = 1e-3
ATOL = 1e-4
SPREAD = 1e-5  # run-to-run relative L2 spread of the float atomics (test_backward.py::test_run_to_run_spread)


@pytest.fixture(scope="module")
def lcgs():
    from luisacomputegaussiansplatting_b200 import lcgs as m
    return m


@pytest.fixture(scope="module")
def dev(lcgs):
    d = lcgs.Device(0)
    yield d
    d.close()


def rows(a, n):
    return np.asarray(a, np.float64).reshape(n, -1)


def per_gaussian(got, want):
    """(e, m): the row norms of got - want and of want, one row per Gaussian."""
    n = np.asarray(want).shape[0]
    g, w = rows(got, n), rows(want, n)
    return np.linalg.norm(g - w, axis=1), np.linalg.norm(w, axis=1)


def check_grads(label, got, want):
    """Both bars on every tensor of `want`; prints each tensor's e_i / m_i distribution before asserting."""
    report, failures = [], []
    for n in want:
        e, m = per_gaussian(got[n], want[n])
        P = m.shape[0]
        out = e > RTOL * m + ATOL * m.max()
        bad = int(out.sum())
        allowed = max(3, int(1e-4 * P))
        nz = m > 0
        ratio = e[nz] / m[nz] if nz.any() else np.zeros(1)
        # the smallest RTOL (ATOL scaled with it) at which this tensor would pass the per-Gaussian bar
        q = np.sort(e / (m + ATOL / RTOL * m.max())) if m.max() > 0 else np.zeros(1)
        crit = float(q[-allowed - 1]) if q.size > allowed else 0.0
        # the whole-tensor bar on the rows the per-Gaussian bar does not except (all rows if it fails)
        keep = ~out if bad <= allowed else np.ones_like(out)
        rel, cos = metrics(rows(got[n], P)[keep], rows(want[n], P)[keep])
        rel_all, _ = metrics(got[n], want[n])
        report.append("%s med %.2e p99.9 %.2e max %.2e bad %d/%d crit %.2e rel %.2e (all rows %.2e) cos %.7f" % (
            n, np.median(ratio), np.quantile(ratio, 0.999), ratio.max(), bad, allowed, crit, rel, rel_all, cos))
        if bad > allowed:
            failures.append((n, "per-Gaussian", bad, allowed))
        if not (rel <= 1e-3 and cos >= 0.9999):
            failures.append((n, "whole tensor", rel, cos))
    print("\n%s\n  " % label + "\n  ".join(report))
    assert not failures, (label, failures)


def assert_all_zero(got, ids, what):
    for n, a in got.items():
        assert not np.any(np.asarray(a)[ids]), (what, n)


def uniform(seed, shape):
    return np.random.default_rng(seed).uniform(-1.0, 1.0, shape)


def cap_hits(fr, opacity, dec):
    """Per Gaussian: how many of its blended (pixel, entry) pairs the 0.99 cap clamps (o e^power >= 0.99 in the
    oracle's float32 arithmetic)."""
    opacity = np.ascontiguousarray(opacity, np.float32)
    hits = np.zeros(opacity.shape[0], np.int64)
    for xs, ys, ids, blended in dec:
        if not blended.any():
            continue
        pw = tr._f32_power(fr.means_2d[ids, 0], fr.means_2d[ids, 1], fr.conic[ids], xs.astype(np.float32),
                           ys.astype(np.float32))
        raw = (opacity[ids][None] * np.exp(pw.astype(np.float64)).astype(np.float32)).astype(np.float32)
        hits[ids] += (blended & (raw >= np.float32(0.99))).sum(0)  # a tile lists a Gaussian once
    return hits


def backward_case(lcgs, dev, arrays, pose, W, H, planes, seed, bg=(0.0, 0.0, 0.0), scale_modifier=1.0, deg=3):
    """GPU and reference gradients for L = sum(img R) (+ sum(alpha Ra) + sum(depth Rd) with planes 'both' / 'depth');
    returns (got, want, fr)."""
    R = uniform(seed, (3, H, W))
    if planes is None:
        r, got = gpu_backward(lcgs, dev, arrays, pose, W, H, deg, bg, R, scale_modifier=scale_modifier)
        fr, want, _ = reference(arrays, pose, W, H, deg, bg, R, scale_modifier=scale_modifier)
    else:
        Ra = uniform(seed + 1, (H, W)) if planes == "both" else None
        Rd = uniform(seed + 2, (H, W))
        r, got = gpu_backward_aux(lcgs, dev, arrays, pose, W, H, deg, bg, R, Ra, Rd, scale_modifier=scale_modifier)
        fr, want = reference_aux(arrays, pose, W, H, deg, bg, R, Ra, Rd, scale_modifier=scale_modifier)
    assert np.array_equal(r.tiles_touched.cpu().numpy().view(np.uint32), fr.tiles_touched)
    assert_all_zero(got, fr.tiles_touched == 0, "touches no tile")
    return got, want, fr


# ---- the 0.99 cap and opacity extremes ------------------------------------------------------------------------------

def opacity_extremes_scene(lcgs):
    """test_gpu_parity.py::test_opacity_extremes's mix (opacity 0, 0.0039 < 1/255, exactly 1/255, 1, the scene's own)
    plus one opaque Gaussian, appended last, placed on the view axis and large enough that the cap clamps its alpha on
    hundreds of pixels around its centre."""
    W, H = 640, 400
    arrays, pose = scene_arrays("C3", 8_000)
    op = arrays[4]
    op[0::5] = 0.0
    op[1::5] = 0.0039
    op[2::5] = np.float32(1.0) / np.float32(255.0)
    op[3::5] = 1.0
    front = np.array(list(lcgs.make_camera(*pose, W, H).front), np.float32)
    one = [np.array(scenes.CAM_POS, np.float32) + 3.0 * front, np.full(3, 0.3, np.float32),
           np.array([1.0, 0.0, 0.0, 0.0], np.float32), arrays[3][4], np.ones(1, np.float32)]
    arrays = [np.ascontiguousarray(np.concatenate([a, b.reshape(1, *a.shape[1:])]), np.float32)
              for a, b in zip(arrays, one)]
    return arrays, pose, W, H


@pytest.mark.parametrize("planes", [None, "both"])
def test_cap_and_opacity_extremes(lcgs, dev, planes):
    arrays, pose, W, H = opacity_extremes_scene(lcgs)
    got, want, fr = backward_case(lcgs, dev, arrays, pose, W, H, planes, seed=11, scale_modifier=3.0)
    P = arrays[4].shape[0]
    hits = cap_hits(fr, arrays[4], tr.decisions(fr, arrays[4], W, H))
    print("capped blended entries %d (the opaque Gaussian's %d)" % (hits.sum(), hits[-1]))
    assert hits[:-1].sum() > 200 and hits[-1] > 300
    check_grads("opacity extremes, scale_modifier 3, planes %s" % planes, got, want)
    # opacity 0 and opacity below 1/255 never blend: exactly zero in every output, though they touch tiles
    never = (np.arange(P) % 5 < 2) & (np.arange(P) < P - 1)
    assert (fr.tiles_touched[never] > 0).sum() > 500
    assert_all_zero(got, never, "opacity 0 / 0.0039")
    # the opaque Gaussian: its capped centre pixels give no opacity gradient
    o_got, o_want = float(got["opacity"].reshape(-1)[-1]), float(want["opacity"].reshape(-1)[-1])
    print("opaque Gaussian grad_opacity %.6e, reference %.6e" % (o_got, o_want))
    assert abs(o_want) > 1e-3 and abs(o_got - o_want) <= 1e-4 * abs(o_want)


@pytest.mark.parametrize("prepare_scene", [True, False])
def test_prepared_and_unprepared_alpha_constants(lcgs, dev, prepare_scene):
    """Without lcgs_b200_scene_prepare (alpha_consts NULL) the record rebuild derives the alpha-test constants itself.
    The records, and so every blend decision, are the same either way; only the order of the float atomics differs.
    The blend's own outputs (2D gradients, colour, SH, opacity) agree within the run-to-run spread bar.  pos, scale
    and rotq pass the 2D gradient through the float32 covariance chain, which for the needle-thin Gaussians of this
    scene amplifies the atomics' last-bit noise: they must agree within three times the larger spread of two runs of
    one setting (measured on an NVIDIA B200: rotq 4.4e-6 to 2.4e-5 between the settings, 1.8e-5 between repeats; any
    changed blend decision moves these tensors by orders of magnitude more)."""
    arrays, pose, W, H = opacity_extremes_scene(lcgs)
    R = uniform(12, (3, H, W))

    def run(prep):
        return gpu_backward(lcgs, dev, arrays, pose, W, H, 3, (0.0, 0.0, 0.0), R, scale_modifier=3.0,
                            prepare_scene=prep)[1]

    got, again, other, other_again = run(prepare_scene), run(prepare_scene), run(not prepare_scene), run(not prepare_scene)
    for n in got:
        rel = metrics(got[n], other[n])[0]
        spread = max(metrics(got[n], again[n])[0], metrics(other[n], other_again[n])[0])
        print("%s: between settings %.2e, repeats %.2e" % (n, rel, spread))
        assert rel <= (SPREAD if n in ("sh", "opacity", "means_2d", "conic", "color") else max(SPREAD, 3.0 * spread)), (
            n, rel, spread)
    _, want, _ = reference(arrays, pose, W, H, 3, (0.0, 0.0, 0.0), R, scale_modifier=3.0)
    check_grads("prepare_scene %s" % prepare_scene, got, want)


# ---- scale_modifier ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("scale_modifier", [0.5, 3.0])
@pytest.mark.parametrize("key,P,W,H", [("C1", 3_000, 200, 200), ("C3", 4_000, 320, 180)])
def test_scale_modifier(lcgs, dev, key, P, W, H, scale_modifier):
    """Image and depth-plane loss; scale_modifier scales the covariance in the forward and dL/dscale in the backward."""
    arrays, pose = scene_arrays(key, P)
    got, want, _ = backward_case(lcgs, dev, arrays, pose, W, H, "depth", seed=13, scale_modifier=scale_modifier)
    check_grads("%s P=%d %dx%d scale_modifier %g" % (key, P, W, H, scale_modifier), got, want)


# ---- long unsaturated tile lists --------------------------------------------------------------------------------------

@pytest.mark.parametrize("planes", [None, "both"])
def test_long_unsaturated_lists(lcgs, dev, planes):
    """test_heavy_tailed_tiles_and_huge_splats's geometry (scale_modifier 25, 640x360) at opacity 0.05: lists of more
    than 1000 entries (eight or more rounds of the walk) that the pixels walk almost to the end, so R_i = C - sum w_j c_j
    is a float32 difference of long sums."""
    W, H = 640, 360
    arrays, pose = scene_arrays("C3", 6_000)
    arrays[4][:] = 0.05
    got, want, fr = backward_case(lcgs, dev, arrays, pose, W, H, planes, seed=14, bg=(0.2, 0.4, 0.6),
                                  scale_modifier=25.0)
    lens = fr.ranges[:, 1].astype(np.int64) - fr.ranges[:, 0]
    gx, _ = orc.grids(W, H)
    longest = np.argsort(lens)[-8:]
    examined = [fr.n_examined[t // gx * 16:t // gx * 16 + 16, t % gx * 16:t % gx * 16 + 16].mean() / lens[t]
                for t in longest]
    print("longest lists", lens[longest], "examined share %.3f .. %.3f" % (min(examined), max(examined)))
    assert lens.max() > 1000 and (lens > 1000).sum() >= 8
    assert min(examined) > 0.75
    check_grads("long lists, planes %s" % planes, got, want)


# ---- far Gaussians ----------------------------------------------------------------------------------------------------

def test_far_gaussians_with_a_depth_loss(lcgs, dev):
    """test_far_gaussians_run_the_fourth_depth_pass's scene (a third of the Gaussians pushed 9000x farther and scaled
    up with it) with an image and a depth-plane loss: dL/dz of depths beyond 13107 reaches grad_depth and grad_pos."""
    W, H = 320, 200
    arrays, pose = scene_arrays("C3", 6_000)
    cam = np.asarray(pose[0], np.float32)
    far = np.arange(arrays[0].shape[0]) % 3 == 0
    k = np.float32(9000.0)
    arrays[0][far] = cam + (arrays[0][far] - cam) * k
    arrays[1][far] = arrays[1][far] * k
    got, want, fr = backward_case(lcgs, dev, arrays, pose, W, H, "depth", seed=15)
    touching = fr.tiles_touched > 0
    assert (fr.depth[touching] > 13200.0).sum() > 100 and (fr.depth[touching] < 100.0).sum() > 100
    check_grads("far Gaussians, depth loss", got, want)
    deep = touching & (fr.depth > 13200.0)
    assert np.count_nonzero(got["depth"][deep]) > 100


# ---- a context another frame has grown ------------------------------------------------------------------------------

def test_backward_after_a_larger_frame_on_the_same_device(lcgs, dev):
    """The backward reads the frame's own buffers; its scratch (tile order, records, packed 2D gradients) lives in the
    device context.  Rendering and differentiating a larger frame on another Renderer grows and overwrites that scratch;
    frame A's backward afterwards must still give A's gradients (within the run-to-run spread)."""
    W, H = 320, 180
    arrays, pose = scene_arrays("C3", 4_000)
    R = uniform(16, (3, H, W))
    a = lcgs.Renderer(dev, *arrays, W, H, list_capacity=2_000_000)
    vp = lcgs.view_params(lcgs.make_camera(*pose, W, H))
    a.render_async(vp)
    n_a = dev.num_rendered()
    first = run_backward(lcgs, dev, a, vp, R)

    W2, H2 = 1280, 720
    big, pose2 = scene_arrays("C3", 60_000)
    b = lcgs.Renderer(dev, *big, W2, H2, list_capacity=20_000_000)
    vp2 = lcgs.view_params(lcgs.make_camera(*pose2, W2, H2))
    b.render_async(vp2)
    assert dev.num_rendered() > 10 * n_a
    after_render = run_backward(lcgs, dev, a, vp, R)
    run_backward(lcgs, dev, b, vp2, uniform(17, (3, H2, W2)))
    after_backward = run_backward(lcgs, dev, a, vp, R)
    for again in (after_render, after_backward):
        for n in first:
            rel, _ = metrics(again[n], first[n])
            assert rel <= SPREAD, (n, rel)
    _, want, _ = reference(arrays, pose, W, H, 3, (0.0, 0.0, 0.0), R)
    check_grads("frame A after a larger frame", after_backward, want)


# ---- windows of full-size frames --------------------------------------------------------------------------------------

FULL = {
    "C3": dict(key="C3", P=None, W=1920, H=1080, scale_modifier=1.0),
    "C2": dict(key="C2", P=None, W=1237, H=822, scale_modifier=1.0),
    "wide": dict(key="C3", P=4_000, W=640_000, H=48, scale_modifier=40.0),
}


@functools.lru_cache(maxsize=1)
def full_frame(name):
    c = FULL[name]
    sc, cfg = scenes.make_config_scene(c["key"], P=c["P"]) if c["P"] else scenes.make_config_scene(c["key"])
    W, H = c["W"], c["H"]
    pose = (scenes.CAM_POS, scenes.CAM_TARGET, scenes.world_up(cfg.world))
    arrays = [np.ascontiguousarray(a, np.float32) for a in (sc.pos, sc.scale, sc.rotq, sc.sh, sc.opacity)]
    fr = orc.forward(*arrays, orc.view_params(orc.make_camera(*pose, W, H)), scale_modifier=c["scale_modifier"],
                     capacity=20_000_000 if c["P"] is None else None)
    return arrays, pose, W, H, c["scale_modifier"], fr


def window(fr, W, H, where):
    """3x3 tiles (tile x0, tile y0): around the longest list, or the frame's bottom-right corner."""
    gx, gy = orc.grids(W, H)
    if where == "corner":
        return gx - 3, gy - 3
    t = int(np.argmax(fr.ranges[:, 1].astype(np.int64) - fr.ranges[:, 0]))
    return min(max(t % gx - 1, 0), gx - 3), min(max(t // gx - 1, 0), gy - 3)


@pytest.mark.parametrize("name,where", [("C3", "longest"), ("C2", "longest"), ("C2", "corner"), ("wide", "longest")])
def test_windowed_full_size_frame(lcgs, dev, name, where):
    """dL/dimg random on 3x3 tiles and zero elsewhere: only the Gaussians those tiles list can have a gradient, and
    the reference needs only their decisions and their rows.  C3 (5.8 M Gaussians, 1920x1080) and C2 (6.1 M, 1237x822,
    ragged edge tiles) at the tiles with the longest lists, C2 also at its ragged bottom-right corner, and the
    640000x48 frame (120000 tiles: the tile order is one CTA's).  About 10 s each for C3 and C2."""
    arrays, pose, W, H, sm, fr = full_frame(name)
    gx, gy = orc.grids(W, H)
    tx0, ty0 = window(fr, W, H, where)
    x0, y0 = 16 * tx0, 16 * ty0
    x1, y1 = min(x0 + 48, W), min(y0 + 48, H)
    Rw = np.random.default_rng(18).uniform(-1.0, 1.0, (3, y1 - y0, x1 - x0)).astype(np.float32)

    # GPU: the whole frame, every output kept on the device
    r = lcgs.Renderer(dev, *arrays, W, H, list_capacity=fr.num_rendered + 5, scale_modifier=sm)
    vp = lcgs.view_params(lcgs.make_camera(*pose, W, H))
    r.render_async(vp)
    assert dev.num_rendered() == fr.num_rendered
    P = r.P
    dl = torch.zeros(3, H, W, device="cuda")
    dl[:, y0:y1, x0:x1] = torch.from_numpy(Rw).cuda()
    out = {n: torch.zeros_like(t) for n, t in zip(NAMES, (r.pos, r.scale, r.rotq, r.sh, r.opacity))}
    out.update(means_2d=torch.zeros(P, 2, device="cuda"), conic=torch.zeros(P, 3, device="cuda"),
               color=torch.zeros(P, 3, device="cuda"))
    g = lcgs._capi.Grad()
    g.dl_dimg = dl.data_ptr()
    for n in out:
        setattr(g, "grad_" + n, out[n].data_ptr())
    dev.check(dev.lib.lcgs_b200_render_backward(dev.ctx, C.byref(r.c_scene), C.byref(vp), C.byref(r.c_frame), C.byref(g), None))
    torch.cuda.synchronize()

    # the window's lists and the Gaussians in them
    tiles = [ty * gx + tx for ty in range(ty0, ty0 + 3) for tx in range(tx0, tx0 + 3)]
    dec = tr.decisions(fr, arrays[4], W, H, tiles)
    ids = np.unique(np.concatenate([d[2] for d in dec]))
    lens = [d[2].size for d in dec]
    print("%s %s window tiles (%d, %d): lists %s, %d Gaussians" % (name, where, tx0, ty0, lens, ids.size))
    assert ids.size > 100
    outside = torch.ones(P, dtype=torch.bool, device="cuda")
    outside[torch.from_numpy(ids).cuda()] = False
    for n, t in out.items():
        assert not torch.any(t[outside]), n  # a Gaussian no window tile lists: exactly zero
    got = {n: t[torch.from_numpy(ids).cuda()].cpu().numpy() for n, t in out.items()}

    check_grads("%s %s window" % (name, where), got, window_reference(arrays, pose, W, H, sm, dec, ids, x0, y0, Rw))


def window_reference(arrays, pose, W, H, scale_modifier, dec, ids, x0, y0, Rw):
    """The float64 reference's gradients of L = sum(img[:, y0:, x0:] Rw) for the Gaussians `ids` (ascending) only,
    given the decisions `dec` of the tiles under the window: the float64 preprocess runs on those rows alone."""
    L = [tr.leaf(a[ids]) for a in arrays]
    local = [(xs, ys, np.searchsorted(ids, gi), bl) for xs, ys, gi, bl in dec]
    vp = orc.view_params(orc.make_camera(*pose, W, H))
    means, conic, color, _ = tr.preprocess(*L[:4], vp, 3, scale_modifier)
    for t in (means, conic, color):
        t.retain_grad()
    pixs, cols = tr.blend_pixels(means, conic, color, L[4], local, W)
    Rt = torch.from_numpy(np.asarray(Rw, np.float64))
    loss = sum((c * Rt[:, p // W - y0, p % W - x0].T).sum() for p, c in zip(pixs, cols))
    loss.backward()
    want = {n: x.grad.numpy() for n, x in zip(NAMES, L)}
    want.update(means_2d=means.grad.numpy(), conic=conic.grad.numpy(), color=color.grad.numpy())
    return want
