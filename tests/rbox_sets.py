"""Rotated-box test sets where the IoU, NMS and assignment kernels go wrong, shared by the CPU invariant tests and
the GPU exactness tests, plus the screen for boxes whose device sin/cos may legitimately differ from libm's.

Pure numpy (and the oracle): importable without torch or a GPU."""
import numpy as np

F32 = np.float32


def nested_pairs(n, seed, angle=None, delta=0.0, ratio=(0.1, 0.49), shift=True, img=1024.0):
    """n pairs (outer, inner) that share both long edge lines: same centre line, angle and height, the inner one
    shorter (length ratio in `ratio`) and slid along the axis but still inside.  The true IoU is the length ratio; the
    reference's fp32 clipper can return anything up to 1.0 for them.  delta shrinks the inner height to h * (1 - delta)
    (centred), so the long edges are delta * h / 2 apart.  angle: None = generic, else that angle for every pair."""
    rng = np.random.default_rng(seed)
    c = rng.uniform(64, img - 64, (n, 2))
    w = np.exp(rng.uniform(np.log(20), np.log(400), n))
    h = np.exp(rng.uniform(np.log(2), np.log(40), n))
    th = rng.uniform(-np.pi / 4, 3 * np.pi / 4, n) if angle is None else np.full(n, angle)
    outer = np.stack([c[:, 0], c[:, 1], w, h, th], 1).astype(F32)
    wi = w * rng.uniform(ratio[0], ratio[1], n)
    s = rng.uniform(-1, 1, n) * (w - wi) / 2 if shift else np.zeros(n)
    u = np.stack([np.cos(th), np.sin(th)], 1)
    inner = np.stack([c[:, 0] + s * u[:, 0], c[:, 1] + s * u[:, 1], wi, h * (1 - delta), th], 1).astype(F32)
    if delta == 0.0:
        inner[:, 3] = outer[:, 3]                     # bit-equal heights
    if not shift:
        inner[:, :2] = outer[:, :2]
    inner[:, 4] = outer[:, 4]
    return outer, inner


def interleave(outer, inner):
    """[o0, i0, o1, i1, ...]: pair k is rows (2k, 2k + 1)."""
    out = np.empty((2 * len(outer), 5), F32)
    out[0::2], out[1::2] = outer, inner
    return out


def nested_sets():
    """Shared-edge nested pairs at generic angles, at 0, pi/4 and pi/2, centred and slid, and with the inner height
    shrunk by delta in [0, 1e-2]: named [2n, 5] arrays of interleaved pairs."""
    # (an fp32 centre slid along a generic axis is off the shared line by rounding, so centred pairs are the sharper
    # case: about one in ten of them has a reference IoU above 0.5)
    sets = {"generic": interleave(*nested_pairs(1000, 1, shift=False)),
            "generic_slid": interleave(*nested_pairs(300, 2)),
            "generic_wide": interleave(*nested_pairs(200, 3, ratio=(0.3, 0.95), shift=False))}
    for k, a in enumerate((0.0, np.pi / 4, np.pi / 2)):
        sets["theta_%g" % a] = interleave(*nested_pairs(200, 10 + k, angle=a))
    for k, d in enumerate((1e-7, 1e-6, 1e-5, 1e-4, 1e-3, 1e-2)):
        sets["delta_%g" % d] = interleave(*nested_pairs(200, 20 + k, delta=d, shift=False))
    return sets


def slivers(n, seed):
    """Boxes with one side from 1e-4 to 1 px, laid over fat boxes near them (crossing, nested, parallel)."""
    rng = np.random.default_rng(seed)
    fat = np.stack([rng.uniform(100, 900, n), rng.uniform(100, 900, n), np.exp(rng.uniform(np.log(8), np.log(200), n)),
                    np.exp(rng.uniform(np.log(8), np.log(200), n)), rng.uniform(-np.pi / 4, 3 * np.pi / 4, n)], 1)
    thin = fat.copy()
    thin[:, :2] += rng.normal(0, 0.2, (n, 2)) * fat[:, 2:3]
    thin[:, 2] = fat[:, 2] * np.exp(rng.normal(0, 0.5, n))
    thin[:, 3] = 10 ** rng.uniform(-4, 0, n)
    thin[1::3, 4] = fat[1::3, 4]                       # parallel to its fat box
    thin[2::3, 4] += rng.normal(0, 0.3, len(thin[2::3]))
    return np.concatenate([fat, thin]).astype(F32)


def thin_and_fat():
    """Thin boxes (sides 1e-4 ... 5 px, some at 0 or pi/2) spread over a 2048 px field, and DOTA-like fat ones."""
    from s2anet_b200 import synth
    rng = np.random.default_rng(11)
    n = 400
    thin = np.stack([rng.uniform(0, 2048, n), rng.uniform(0, 2048, n), 10 ** rng.uniform(0.5, 2.7, n),
                     10 ** rng.uniform(-4, 0.7, n), rng.uniform(-np.pi / 4, 3 * np.pi / 4, n)], 1).astype(F32)
    thin[::7, 4] = 0.0
    thin[1::7, 4] = F32(np.pi / 2)
    thin[2::7, 2:4] = thin[2::7, 3:1:-1]
    fat = synth.dota_like_gt(300, 13)
    fat[::5, 4] = 0.0
    return thin, fat


def angle_may_differ(theta):
    """True for a box whose fp32 (cos, sin) may differ between the device and libm: float64 cos or sin of its fp32
    angle lies within 16 double ulps of an fp32 rounding midpoint.  CUDA's double sin/cos are within 2 ulps of the
    exact value and glibc's within 1, so for any other box both round to the same float and every IoU bit agrees."""
    t = np.asarray(theta, np.float32).astype(np.float64)
    flag = np.zeros(t.shape, bool)
    for v in (np.cos(t), np.sin(t)):
        f = v.astype(np.float32)
        for nb in (np.nextafter(f, F32(np.inf)), np.nextafter(f, F32(-np.inf))):
            mid = (f.astype(np.float64) + nb.astype(np.float64)) / 2
            flag |= np.abs(v - mid) <= 16 * np.spacing(np.abs(v))
    return flag


def oracle_iou_image(args):
    """One image's anchor x GT IoU from the oracle (a ctypes call, which releases the GIL: thread pools overlap)."""
    from oracle import oracle
    a, g = args
    return oracle.box_iou_rotated(a, g)
