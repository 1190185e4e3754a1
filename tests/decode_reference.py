"""Op-by-op model of the rotated-box decode (csrc/box_decode.cuh) and of the score sigmoid (sigmoid_t in csrc/decode.cu),
for bit-exact tests of every decode path.

The kernels evaluate the reference's formula (models/boxes.py:82-162, utils/general.py:925-930) with individually
rounded fp32 operations in the reference's order, rounding to the deltas' dtype T where the reference's half tensors
round.  `decode_model` restates that sequence in numpy float32, operation for operation.  Only cosf, sinf and expf are
not correctly rounded, so no float64 reference can be exact: the model takes them as callables.  Given numpy's own
float32 cos / sin / exp it must equal oracle.delta2bbox_rotated bit for bit (CPU tests); given the device's values
(`DeviceMath`, probed through select_decode) it must equal the kernels bit for bit.
"""
import math

import numpy as np
import torch

from tc_reference import round_rne

F32 = np.float32
PI = F32(np.pi)                      # float(np.pi), kPi in box_decode.cuh
QPI = F32(np.pi / 4)                 # float(np.pi / 4) == PI / 4 exactly
DTYPES = (torch.float32, torch.bfloat16, torch.float16)


def to_t(x, dtype):
    """float32 array -> float32 array of the nearest-even `dtype` values (what storing a T element does; NaN and the
    sign of zero pass, overflow goes to inf)."""
    x = np.asarray(x, F32)
    if dtype == torch.float32:
        return x.copy()
    return round_rne(torch.from_numpy(x.astype(np.float64)), dtype).float().numpy()


def t_step(x, dtype, toward):
    """The next `dtype` value after each x (float32 array of dtype values) in the direction of `toward`."""
    x = np.asarray(x, F32)
    if dtype == torch.float32:
        return np.nextafter(x, F32(toward)).astype(F32)
    u = torch.from_numpy(x.reshape(-1)).to(dtype).view(torch.int16).numpy().view(np.uint16).astype(np.int32)
    key = np.where(u & 0x8000, -(u & 0x7FFF), u)                 # values in order; -0 and +0 are both 0
    key = key + np.where(F32(toward) > x.reshape(-1), 1, -1)
    u = np.where(key < 0, 0x8000 | -key, key).astype(np.uint16)
    return torch.from_numpy(u.view(np.int16)).view(dtype).float().numpy().reshape(x.shape)


def clamp_limit(wh_ratio_clip, dtype):
    """The clamp bound of dw / dh: |log(wh_ratio_clip)| (Python float, boxes.py:115) rounded to float, then to T.  This is
    how torch.clamp on a T tensor converts its bound on the GPU (measured: tests/test_gpu_decode_exact.py
    test_clamp_bound_rounds_like_torch), and what clamp_limit in box_decode.cuh does."""
    return to_t(F32(abs(math.log(wh_ratio_clip))), dtype)[()]


def decode_model(anchors_f32, deltas, dtype, wh_ratio_clip, cos, sin, exp):
    """delta2bbox_rotated of box_decode.cuh.  anchors [..., 5] float32; deltas [..., 5] float32 holding `dtype` values;
    cos / sin / exp map float32 arrays to float32 arrays.  Returns [..., 5] float32."""
    a = np.asarray(anchors_f32, F32)
    d = np.asarray(deltas, F32)
    lim = F32(clamp_limit(wh_ratio_clip, dtype))
    with np.errstate(all="ignore"):
        dx, dy, dw, dh, da = (d[..., i] for i in range(5))
        dw = np.where(dw < -lim, -lim, np.where(dw > lim, lim, dw)).astype(F32)     # NaN passes, like torch.clamp
        dh = np.where(dh < -lim, -lim, np.where(dh > lim, lim, dh)).astype(F32)
        ax, ay, aw, ah, at = (a[..., i] for i in range(5))
        cosa, sina = np.asarray(cos(at), F32), np.asarray(sin(at), F32)
        dxw, dyh = dx * aw, dy * ah
        gx = (dxw * cosa - dyh * sina) + ax
        gy = (dxw * sina + dyh * cosa) + ay
        gw = aw * to_t(exp(dw), dtype)
        gh = ah * to_t(exp(dh), dtype)
        ga = to_t(da * PI, dtype) + at
        m = np.fmod(ga + QPI, PI)
        m = np.where(m < 0, m + PI, m).astype(F32)
        gt = m - QPI
    return np.stack([gx, gy, gw, gh, gt], axis=-1).astype(F32)


def exp_args(deltas, dtype, wh_ratio_clip):
    """The arguments decode_model passes to exp: dw and dh after the clamp."""
    d = np.asarray(deltas, F32)
    lim = F32(clamp_limit(wh_ratio_clip, dtype))
    v = d[..., 2:4]
    with np.errstate(invalid="ignore"):
        return np.where(v < -lim, -lim, np.where(v > lim, lim, v)).astype(F32).ravel()


def grid_anchor_model(H, W, stride, scale, angle):
    """fam_grid_anchor of box_decode.cuh -> [H, W, 5] float32."""
    s = F32(stride)
    half = F32(0.5) * (s - F32(1))
    a = np.empty((H, W, 5), F32)
    a[..., 0] = (np.arange(W, dtype=F32) * s + half)[None, :]
    a[..., 1] = (np.arange(H, dtype=F32) * s + half)[:, None]
    a[..., 2] = a[..., 3] = s * F32(scale)
    a[..., 4] = F32(angle)
    return a


def sigmoid_model(x, dtype, exp):
    """sigmoid_t of decode.cu (torch.sigmoid on a T tensor): T(1 / (1 + exp(-x))) with IEEE division."""
    x = np.asarray(x, F32)
    with np.errstate(all="ignore"):
        return to_t(F32(1) / (F32(1) + np.asarray(exp(-x), F32)), dtype)


def numpy_math():
    """numpy's float32 cos / sin / exp: the transcendentals oracle.delta2bbox_rotated uses."""
    def ex(x):
        with np.errstate(over="ignore"):
            return np.exp(np.asarray(x, F32))
    return (lambda x: np.cos(np.asarray(x, F32)), lambda x: np.sin(np.asarray(x, F32)), ex)


def same_bits(a, b):
    """Elementwise: equal float32 bits, or both NaN."""
    a, b = np.asarray(a, F32), np.asarray(b, F32)
    return (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))


def assert_same(got, want, what=""):
    got, want = np.asarray(got, F32), np.asarray(want, F32)
    assert got.shape == want.shape, "%s: shape %s != %s" % (what, got.shape, want.shape)
    ok = same_bits(got, want)
    if not ok.all():
        i = np.argwhere(~ok)[:5]
        raise AssertionError("%s: %d of %d values differ, e.g. at %s: %s != %s" % (
            what, int((~ok).sum()), ok.size, i.tolist(), got[tuple(i.T)].tolist(), want[tuple(i.T)].tolist()))


# ------------------------------------------------------------------------------------------------------------------
# the device's own cosf / sinf / expf
# ------------------------------------------------------------------------------------------------------------------
class DeviceMath:
    """cosf, sinf and expf as the decode kernels evaluate them, probed through select_decode and memoised.

    A probe row is anchor (0, 0, 1, 1, theta) with deltas (1, 0, t, u, 0), in fp32 with topk = 0 and a clip so small
    (1e-300, bound 690.8) that nothing is clamped.  box_decode.cuh then computes
        gx = ((1 * 1) * cosf(theta) - (0 * 1) * sinf(theta)) + 0 = cosf(theta)
        gy = ((1 * 1) * sinf(theta) + (0 * 1) * cosf(theta)) + 0 = sinf(theta)
        gw = 1 * expf(t),  gh = 1 * expf(u)
    exactly: adding a zero and multiplying by one do not round.  The one exception is theta = -0, where
    sinf(-0) + (+0) = +0 loses the sign, so -0 is never probed (cosf(-0) = cosf(+0) and sinf(-0) = -0 exactly)."""

    CLIP = 1e-300

    def __init__(self, device="cuda:0"):
        self.device = device
        self.keys = {"cos": np.empty(0, np.uint32), "sin": np.empty(0, np.uint32), "exp": np.empty(0, np.uint32)}
        self.vals = {k: np.empty(0, F32) for k in self.keys}
        self.probes = 0

    def _missing(self, name, x):
        x = np.asarray(x, F32).ravel()
        x = x[np.isfinite(x) if name != "exp" else ~np.isnan(x)]
        x = np.where(x == 0, F32(0), x).astype(F32)              # -0 -> +0
        u = np.unique(x.view(np.uint32))
        k = self.keys[name]
        if len(k):
            pos = np.clip(np.searchsorted(k, u), 0, len(k) - 1)
            u = u[k[pos] != u]
        return u.view(F32)

    def prefetch(self, angles=(), exps=()):
        """Probe every argument not seen yet, in one select_decode call."""
        ang = self._missing("cos", angles)
        ex = self._missing("exp", exps)
        n = max(len(ang), (len(ex) + 1) // 2)
        if n == 0:
            return
        from s2anet_b200.decode import select_decode
        theta = np.full(n, F32(0.5))
        theta[:len(ang)] = ang
        tu = np.zeros(2 * n, F32)
        tu[:len(ex)] = ex
        anc = np.zeros((1, 1, n, 5), F32)
        anc[..., 2] = anc[..., 3] = 1.0
        anc[0, 0, :, 4] = theta
        reg = np.zeros((1, 5, 1, n), F32)
        reg[0, 0] = 1.0
        reg[0, 2, 0] = tu[0::2]
        reg[0, 3, 0] = tu[1::2]
        cls = torch.zeros(1, 1, 1, n, device=self.device)
        bb, _ = select_decode([cls], [torch.from_numpy(reg).to(self.device)], [torch.from_numpy(anc).to(self.device)],
                              topk=0, wh_ratio_clip=self.CLIP)
        bb = bb[0].cpu().numpy()
        self.probes += 1
        for name, args, vals in (("cos", ang, bb[:len(ang), 0]), ("sin", ang, bb[:len(ang), 1]),
                                 ("exp", ex, bb[:, 2:4].reshape(-1)[:len(ex)])):
            k, new = self.keys[name], args.view(np.uint32)       # (sorted, disjoint from k)
            at = np.searchsorted(k, new)
            self.keys[name] = np.insert(k, at, new)
            self.vals[name] = np.insert(self.vals[name], at, vals.astype(F32))

    def _lookup(self, name, x):
        x = np.asarray(x, F32)
        self.prefetch(**({"exps": x} if name == "exp" else {"angles": x}))
        flat = x.ravel()
        key = np.where(flat == 0, F32(0), flat).astype(F32).view(np.uint32)
        pos = np.clip(np.searchsorted(self.keys[name], key), 0, max(len(self.keys[name]) - 1, 0))
        out = self.vals[name][pos] if len(self.keys[name]) else np.zeros_like(flat)
        probed = self.keys[name][pos] == key if len(self.keys[name]) else np.zeros(flat.shape, bool)
        out = np.where(probed, out, F32(np.nan)).astype(F32)      # NaN arguments (and +-inf angles): NaN
        if name == "sin":
            out = np.where(flat == 0, flat, out).astype(F32)      # sinf(+-0) = +-0
        return out.reshape(x.shape)

    def cos(self, x):
        return self._lookup("cos", x)

    def sin(self, x):
        return self._lookup("sin", x)

    def exp(self, x):
        return self._lookup("exp", x)

    def decode(self, anchors, deltas, dtype, wh_ratio_clip):
        """decode_model with the device's transcendentals (one probe for everything new)."""
        a = np.asarray(anchors, F32)
        self.prefetch(angles=a[..., 4], exps=exp_args(deltas, dtype, wh_ratio_clip))
        return decode_model(a, deltas, dtype, wh_ratio_clip, self.cos, self.sin, self.exp)

    def sigmoid(self, x, dtype):
        x = np.asarray(x, F32)
        self.prefetch(exps=-x)
        return sigmoid_model(x, dtype, self.exp)


# ------------------------------------------------------------------------------------------------------------------
# edge data
# ------------------------------------------------------------------------------------------------------------------
CLIPS = (1e-6, 16 / 1000)            # FAM decode (models/head.py:44) and the final decode (head.py:717)


def all_values(dtype):
    """Every finite value of a 16-bit dtype, as float32."""
    v = torch.arange(-32768, 32768, dtype=torch.int32).to(torch.int16).view(dtype).float().numpy()
    return v[np.isfinite(v)]


def angle_steps(theta, dtype, da):
    """ga + pi/4 as the kernel forms it (before fmod), for delta angles da (float32 dtype values) and anchor angles
    theta (broadcast)."""
    with np.errstate(all="ignore"):
        return (to_t(np.asarray(da, F32) * PI, dtype) + F32(theta)) + QPI


def landing_angles(dtype, theta, rng, per_kind=6):
    """Delta angles da (dtype values) for a fixed anchor angle theta such that ga + pi/4 lands exactly on 0, on a
    nonzero multiple of pi, and one float below 0 or a multiple (where fmod is negative, m + pi rounds to pi and the
    output is 3pi/4 - see box_decode.cuh).  Searches all finite 16-bit values, or fp32 values near the targets."""
    if dtype == torch.float32:
        base = []
        for k in range(-4, 5):
            c = F32((k * np.pi - np.pi / 4 - float(theta)) / np.pi)
            v = c
            for _ in range(40):
                base.append(v)
                v = np.nextafter(v, F32(np.inf))
            v = c
            for _ in range(40):
                v = np.nextafter(v, F32(-np.inf))
                base.append(v)
        cand = np.array(base, F32)
    else:
        cand = all_values(dtype)
        cand = cand[np.abs(cand) <= 4096]
    x = angle_steps(theta, dtype, cand)
    with np.errstate(all="ignore"):
        m = np.fmod(x, PI)
    kinds = {"zero": x == 0, "multiple": (x != 0) & (m == 0),
             "below": (m < 0) & ((m + PI) == PI)}
    out = {}
    for k, sel in kinds.items():
        c = cand[sel]
        out[k] = rng.permutation(c)[:per_kind] if len(c) else c
    return out


def free_landing_rows(dtype, rng, n=4):
    """(da, theta) pairs with theta chosen so that ga + pi/4 lands exactly on 0, on +-pi and 2pi, and one float below 0:
    for select_decode, whose anchors are free."""
    rows = []
    for target in (0.0, np.pi, -np.pi, 2 * np.pi, "below"):
        for _ in range(n):
            da = to_t(F32(rng.normal(0.0, 0.5)), dtype)[()]
            pda = to_t(da * PI, dtype)[()]
            want = F32(-1e-30) if target == "below" else F32(target)
            th = F32(float(want) - float(QPI) - float(pda))
            for _ in range(64):                       # nudge theta until the float sums land exactly
                x = angle_steps(th, dtype, da)[()]
                if (target == "below" and x < 0 and np.fmod(x, PI) + PI == PI) or (target != "below" and x == F32(target)):
                    rows.append((da, th))
                    break
                th = np.nextafter(th, F32(np.inf) if x < want else F32(-np.inf))
    return rows


def edge_deltas(dtype, wh_ratio_clip, theta, rng, n_random=0):
    """[N, 5] float32 deltas holding `dtype` values for anchor angle theta:
      * dw / dh at exactly +-T(lim), the next T values inside and outside, +-inf, NaN, +-0 (every pair of them);
      * da landing ga + pi/4 on 0, on multiples of pi and one float below them (landing_angles);
      * |ga| up to about 1e4, and da * pi beyond the fp16 range;
      * n_random rows of the head's typical magnitudes."""
    lim = F32(clamp_limit(wh_ratio_clip, dtype))
    cl = [lim, -lim, t_step(lim, dtype, 0.0), t_step(-lim, dtype, 0.0), t_step(lim, dtype, np.inf),
          t_step(-lim, dtype, -np.inf), F32(np.inf), F32(-np.inf), F32(np.nan), F32(0.0), F32(-0.0),
          to_t(F32(0.5), dtype)]
    cl = np.array([np.asarray(c, F32)[()] for c in cl], F32)
    rows = []
    T = lambda v: to_t(np.asarray(v, F32), dtype)            # noqa: E731
    for i, w in enumerate(cl):
        for j, h in enumerate(cl):
            rows.append([T(rng.normal(0, 0.5)), T(rng.normal(0, 0.5)), w, h, T(rng.normal(0, 0.4))])
    lands = landing_angles(dtype, theta, rng)
    for k, das in lands.items():
        for da in das:
            rows.append([T(rng.normal(0, 0.5)), T(rng.normal(0, 0.5)), T(rng.normal(0, 0.6)), T(rng.normal(0, 0.6)), da])
    for da in (3000.0, -3183.0, 1234.5, -0.25, 0.75, 1.0, -1.0, 0.5, 20860.0, -65504.0, 1e5, -3e38):
        rows.append([T(1.5), T(-2.25), T(0.125), T(-0.125), T(da)])
    for _ in range(n_random):
        rows.append([T(rng.normal(0, 0.3)), T(rng.normal(0, 0.3)), T(rng.normal(0, 0.6)), T(rng.normal(0, 0.6)),
                     T(rng.normal(0, 0.4))])
    d = np.array([[np.asarray(v, F32)[()] for v in r] for r in rows], F32)
    assert same_bits(d, to_t(d, dtype)).all()
    return d, {k: len(v) for k, v in lands.items()}


def edge_angles(dtype, rng, n_random=64):
    """Anchor angles near the wrap points and near pi/2 (where cosf is tiny and gx cancels), plus random ones."""
    pts = []
    for c in (0.0, np.pi / 4, -np.pi / 4, np.pi / 2, -np.pi / 2, 3 * np.pi / 4, np.pi / 6):
        v = F32(c)
        pts += [v, np.nextafter(v, F32(np.inf)), np.nextafter(v, F32(-np.inf)),
                np.nextafter(np.nextafter(v, F32(np.inf)), F32(np.inf))]
    pts = [p for p in pts if not (p == 0 and np.signbit(p))]
    pts += list(rng.uniform(-np.pi / 4, 3 * np.pi / 4, n_random).astype(F32))
    return np.array(pts, F32)
