"""The scatter step across its material parameters and its geometric edges (CPU: the float and double oracles).

One generator (`space_scene`, `space_inputs`) feeds the explicit-input scatter hooks of both oracles here and of the GPU
in tests/test_gpu_scatter_space.py and tests/test_gpu_f64.py.  It covers lambertian albedos {0, 0.5, 1, 3}, metal fuzz
{-1.5, -0.5, -0.0, 0, 2^-24, 0.3, 1, 1.8} and dielectric indices {0.5, 1/1.5, 1, 1+2^-23, 1.33, 1.5, 2.42, 10}, over
random directions of lengths 1e-6 .. 1e6, normal and grazing incidence, directions within a few ulps of the critical
angle on both sides of it, random words at their extremes, and lambertian normals that cancel the sampled offset.

Checks, each against the double oracle (the same formulas in double) or against the reference's definitions:
  (b) float vs double: equal decisions outside a band of 2^-20 around each threshold, directions within
      K 2^-24 (|d64|inf + 1 + 1/|k|), k the refraction's normal component; attenuations bit for bit;
  (c) anchors: mirror at fuzz 0, index 1 refracts straight through, normal incidence, |d - n| = 1 for lambertian;
  (d) distributions (SURVEY a13-a15): lambertian offsets uniform on the sphere, metal offsets uniform in the ball of
      radius |min(fuzz, 1)|, dielectric reflected fraction = Schlick, refraction obeys Snell.
"""
import numpy as np
import pytest
from scipy import stats

from oracle_lib import Oracle, camera_derive, have_ref
from rrt_b200.types import SceneArrays, material_dtype, sphere_dtype

ULP = 2.0**-24
BAND = 2.0**-20
# The worst direction error of the float oracle against the double oracle, in units of 2^-24 (|d64|inf + 1 + 1/|k|), is
# 5.7 over space_inputs() and 6.3 over the seeds 0-9 (refraction at normal incidence and at the critical angle of index
# 10, where eta = 10 scales the rounding of unit(d) + cos_t n).  The GPU's rsqrtf and __fdividef add up to 4 more.
K_ORACLE = 8.0
K_GPU = K_ORACLE + 4.0

ALBEDO = (0.0, 0.5, 1.0, 3.0)
FUZZ = (-1.5, -0.5, -0.0, 0.0, 2.0**-24, 0.3, 1.0, 1.8)
IR = (0.5, 1 / 1.5, 1.0, 1 + 2.0**-23, 1.33, 1.5, 2.42, 10.0)
LAMB = list(range(len(ALBEDO)))
METAL = [len(ALBEDO) + k for k in range(len(FUZZ))]
DIEL = [len(ALBEDO) + len(FUZZ) + k for k in range(len(IR))]
SPECIAL = np.array([0, 0xFF, 0xFFFFFF00, 0xFFFFFFFF], np.uint32)


def space_scene():
    """One sphere and a material table of every parameter value above (lambertian, then metal, then dielectric)."""
    m = np.zeros(len(ALBEDO) + len(FUZZ) + len(IR), material_dtype)
    m["type"] = [0] * len(ALBEDO) + [1] * len(FUZZ) + [2] * len(IR)
    m["albedo"][LAMB] = np.array(ALBEDO)[:, None] * np.array([1.0, 0.5, 0.25])
    m["albedo"][METAL] = (0.8, 0.6, 0.4)
    m["param"] = [0.0] * len(ALBEDO) + list(FUZZ) + list(IR)
    s = np.zeros(1, sphere_dtype)
    s[0] = ((0, 0, -1), 0.5, 0)
    return SceneArrays(camera_derive((0, 0, 0), (0, 0, -1), (0, 1, 0), 40.0, 1.5, 0.0, 1.0), m, s)


def _unit(v):
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def _tangent(rng, n):
    t = _unit(rng.normal(size=n.shape))
    return _unit(t - np.sum(t * n, axis=-1, keepdims=True) * n)


def _rows(d, n, front, mat, rng):
    """in16 rows (float-representable doubles) for directions d, normals n (rounded to float here); rows whose rounded
    d . n > 0 are turned around, as the render's face test does."""
    d = np.asarray(d, np.float32).astype(np.float64)
    n = np.asarray(n, np.float32).astype(np.float64)
    back = np.sum(d * n, axis=1) > 0
    n[back] *= -1
    k = len(d)
    r = np.zeros((k, 16))
    r[:, 0:3] = rng.uniform(-3, 3, size=(k, 3)).astype(np.float32)
    r[:, 3:6] = d
    r[:, 6] = 0.5
    r[:, 7:10] = rng.uniform(-3, 3, size=(k, 3)).astype(np.float32)
    r[:, 10:13] = n
    r[:, 13] = front
    r[:, 14] = mat
    return r


def _words(rng, k):
    """Random words; a quarter of them replaced by 0, 0xFF, 0xFFFFFF00 or 0xFFFFFFFF, and of word 3 also one half
    set to 0x0000 or 0xFFFF."""
    w = rng.integers(0, 2**32, size=(k, 4), dtype=np.uint64).astype(np.uint32)
    pick = rng.uniform(size=(k, 4)) < 0.25
    w[pick] = rng.choice(SPECIAL, size=int(pick.sum()))
    half = rng.integers(0, 5, size=k)
    w[half == 1, 3] &= 0x0000FFFF
    w[half == 2, 3] |= 0xFFFF0000
    w[half == 3, 3] &= 0xFFFF0000
    w[half == 4, 3] |= 0x0000FFFF
    return w


def _word_cross():
    """Every combination of the special values of words 0-2 and the special values and halves of word 3."""
    w3 = np.concatenate([SPECIAL, np.array([0x0000ABCD, 0xFFFFABCD, 0xABCD0000, 0xABCDFFFF], np.uint32)])
    g = np.meshgrid(SPECIAL, SPECIAL, SPECIAL, w3, indexing="ij")
    return np.stack([x.reshape(-1) for x in g], axis=1).astype(np.uint32)


def space_inputs(seed=0, n_random=600):
    """(in16 [N, 16] float64, every value exact in float; rnd4 [N, 4] uint32; kind [N] str) over the materials of
    space_scene().  kind: random / normal / grazing / critical / words."""
    rng = np.random.default_rng(seed)
    ins, rnds, kinds = [], [], []

    def add(rows, kind, words=None):
        ins.append(rows)
        rnds.append(_words(rng, len(rows)) if words is None else words)
        kinds.extend([kind] * len(rows))

    cross = _word_cross()
    for mat in LAMB + METAL + DIEL:
        # random directions, lengths 1e-6 .. 1e6, on random faces
        k = n_random
        n = _unit(rng.normal(size=(k, 3)))
        d = _unit(rng.normal(size=(k, 3))) * 10.0 ** rng.uniform(-6, 6, size=(k, 1))
        add(_rows(d, n, rng.integers(0, 2, size=k), mat, rng), "random")
        # normal incidence: d = -s n exactly (s a power of two), random and axis-aligned normals
        s = 2.0 ** np.array([-20, -10, -3, 0, 3, 10, 19] * 6)
        n = np.concatenate([_unit(rng.normal(size=(len(s) - 6, 3))), np.eye(3), -np.eye(3)]).astype(np.float32)
        add(_rows(-s[:, None] * n, n, rng.integers(0, 2, size=len(s)), mat, rng), "normal")
        # grazing: d . n = -2^-k |d|
        g = np.repeat([1, 2, 4, 8, 12, 16, 20, 23, 24, 26, 30], 8)
        n = _unit(rng.normal(size=(len(g), 3)))
        eps = 2.0 ** -g[:, None]
        d = (np.sqrt(1 - eps * eps) * _tangent(rng, n) - eps * n) * 10.0 ** rng.uniform(-3, 3, size=(len(g), 1))
        add(_rows(d, n, rng.integers(0, 2, size=len(g)), mat, rng), "grazing")
        # every combination of extreme words on a few random geometries
        k = len(cross)
        n = _unit(rng.normal(size=(k, 3)))
        d = _unit(rng.normal(size=(k, 3)))
        add(_rows(d, n, rng.integers(0, 2, size=k), mat, rng), "words", cross)
        # within a few ulps of the critical angle, on both sides of it: back faces (eta = ir > 1) and front faces
        # (eta = 1 / ir > 1)
        if mat in DIEL:
            ir = float(np.float32(IR[DIEL.index(mat)]))
            front = 1 if ir < 1 else 0
            eta = 1.0 / ir if front else ir
            if eta > 1:  # rounding d and n to float moves eta sin_t by ~eta^2 ulps: keep the 48 closest on each side
                k = 4000
                sin = np.minimum(1.0, (1 + rng.integers(-8, 9, size=k) * 2.0**-23) / eta)[:, None]
                n = _unit(rng.normal(size=(k, 3)))
                d = sin * _tangent(rng, n) - np.sqrt(1 - sin * sin) * n
                rows = _rows(d, n, np.full(k, front), mat, rng)
                c = np.sum(_unit(rows[:, 3:6]) * rows[:, 10:13], axis=1)
                off = eta * np.sqrt(np.maximum(0.0, 1 - c * c)) - 1
                near = np.argsort(np.abs(off))
                add(np.concatenate([rows[near[off[near] < 0][:48]], rows[near[off[near] > 0][:48]]]), "critical")
    return np.concatenate(ins), np.concatenate(rnds), np.array(kinds)


def cancel_inputs(orc, precision):
    """Lambertian rows whose normal is exactly -u(rnd), u the unit-sphere sample that rnd draws in this precision (read
    back from the oracle's own scatter with a zero normal), so that n + u cancels.  -> (in16, rnd4)."""
    rng = np.random.default_rng(17)
    k = 256
    rnd = rng.integers(0, 2**32, size=(k, 4), dtype=np.uint64).astype(np.uint32)
    r = np.zeros((k, 16))
    r[:, 3:6] = _unit(rng.normal(size=(k, 3))).astype(np.float32)
    r[:, 13] = 1
    r[:, 14] = LAMB[2]
    u = orc.scatter(r, rnd)[:, 0:3].astype(np.float64) if precision == "f32" else orc.scatter_f64(r, rnd)[:, 0:3]
    r[:, 10:13] = -u
    return r, rnd


# ---------------------------------------------------------------------------------------------------------------
# the double statement of the formulas (numpy), for the decisions, their bands and the candidates
# ---------------------------------------------------------------------------------------------------------------
def geometry(in16, rnd, materials):
    """Per row: the reflect and refract candidates, the refraction's normal component k, Schlick's reflectance (1 under
    total internal reflection), and the distances of the three decisions from their thresholds."""
    d, n = in16[:, 3:6], in16[:, 10:13]
    mat = in16[:, 14].astype(int)
    typ, par = materials["type"][mat], materials["param"][mat].astype(np.float64)
    ud = d / np.linalg.norm(d, axis=1, keepdims=True)
    dn = np.sum(ud * n, axis=1)
    refl = ud - 2 * dn[:, None] * n
    diel = typ == 2
    ir = np.where(diel, par, 1.0)
    eta = np.where(in16[:, 13] != 0, 1 / ir, ir)
    cos = np.minimum(-dn, 1.0)
    sin = np.sqrt(np.maximum(0.0, 1 - cos * cos))
    tir = eta * sin > 1
    r0 = ((1 - eta) / (1 + eta)) ** 2
    schlick = r0 + (1 - r0) * (1 - cos) ** 5
    u0 = (rnd[:, 0] >> 8).astype(np.float64) * ULP
    perp = eta[:, None] * (ud + cos[:, None] * n)
    k = -np.sqrt(np.abs(1 - np.sum(perp * perp, axis=1)))
    refr = perp + k[:, None] * n
    return dict(ud=ud, n=n, typ=typ, par=par, eta=eta, refl=refl, refr=refr, k=k, tir=tir, diel=diel,
                p_refl=np.where(tir, 1.0, schlick), tir_band=np.abs(eta * sin - 1), draw_band=np.abs(schlick - u0))


def chose_reflection(out, g):
    return np.abs(out[:, 0:3] - g["refl"]).max(axis=1) < np.abs(out[:, 0:3] - g["refr"]).max(axis=1)


def compare(lo, hi, in16, rnd, materials, label):
    """(b): float outputs `lo` against the double outputs `hi` of the same inputs.  Decisions must be equal outside the
    band; directions are compared wherever both sides took the same decision.  Returns the worst direction error in
    units of 2^-24 (|d64|inf + 1 + 1/|k|), the number of rows compared, the ratios and the mask of compared rows."""
    g = geometry(in16, rnd, materials)
    lo = lo.astype(np.float64)
    assert lo[:, 3:6].tobytes() == hi[:, 3:6].tobytes(), label  # attenuations bit for bit
    assert np.isfinite(lo[:, 0:3]).all(), label
    d64 = hi[:, 0:3]
    size = np.abs(d64).max(axis=1)
    diel = g["diel"]
    cont_band = np.abs(np.sum(d64 * g["n"], axis=1)) / np.maximum(np.linalg.norm(d64, axis=1), 1e-300)
    outside = (g["typ"] != 1) | (cont_band > BAND)
    flag = lo[:, 6] != hi[:, 6]
    assert not (flag & outside).any(), (label, "continue flag differs outside the band", np.nonzero(flag & outside)[0][:8])
    # reflect or refract: where the two candidates are apart, both sides picked the same one outside the band
    outside = ~diel | ((g["tir_band"] > BAND) & (g["draw_band"] > BAND))
    apart = np.abs(g["refl"] - g["refr"]).max(axis=1) > 1e-3
    rl, rh = chose_reflection(lo, g), chose_reflection(hi, g)
    bad = diel & outside & apart & (rl != rh)
    assert not bad.any(), (label, "reflect / refract differs outside the band", np.nonzero(bad)[0][:8])
    # directions: outside the band, and inside it where both sides took the same one of two distinct candidates (the
    # lambertian fallback, n + u ~ 0, is an anchor of its own)
    ok = (size > 1e-6) & (~diel | outside | (apart & (rl == rh)))
    inv_k = np.where(diel & ~rh, 1 / np.maximum(np.abs(g["k"]), 1e-300), 0.0)
    ratio = np.abs(lo[:, 0:3] - d64).max(axis=1) / (ULP * (size + 1 + inv_k))
    return float(ratio[ok].max()), int(ok.sum()), ratio, ok


def anchors(out, in16, rnd, kind, materials, tol_ulps, label):
    """(c), to tol_ulps 2^-24: fuzz 0 reflects to the mirror of unit(d); index 1 refracts to unit(d); at normal incidence
    refraction gives unit(d) and reflection -unit(d); the lambertian offset d - n has length 1."""
    g = geometry(in16, rnd, materials)
    out = out.astype(np.float64)
    dirs = out[:, 0:3]
    tol = tol_ulps * ULP
    mirror = (g["typ"] == 1) & (g["par"] == 0)  # 0 and -0
    assert mirror.sum() > 1000
    err = np.abs(dirs - g["refl"]).max(axis=1)
    assert err[mirror].max() <= tol, (label, "mirror", err[mirror].max() / ULP)
    straight = g["diel"] & (g["par"] == 1) & ~chose_reflection(out, g) & (np.abs(g["k"]) > 2.0**-4)
    assert straight.sum() > 500
    err = np.abs(dirs - g["ud"]).max(axis=1) / (1 + 1 / np.maximum(np.abs(g["k"]), 1e-300))
    assert err[straight].max() <= tol, (label, "index 1", err[straight].max() / ULP)
    both = (kind == "normal") & (g["diel"] | mirror)
    assert both.sum() > 100
    refl_d = g["diel"] & (np.abs(dirs + g["ud"]).max(axis=1) < np.abs(dirs - g["ud"]).max(axis=1))
    want = np.where(refl_d[:, None] | (g["typ"] == 1)[:, None], -g["ud"], g["ud"])
    # a refraction scales the rounding of unit(d) + cos_t n (~0 here) by eta
    err = np.abs(dirs - want).max(axis=1) / np.where(g["diel"] & ~refl_d, np.maximum(g["eta"], 1), 1)
    assert err[both].max() <= tol, (label, "normal incidence", err[both].max() / ULP)
    assert refl_d[both].any() and (g["diel"] & both & ~refl_d).any()  # both outcomes occur
    lamb = (g["typ"] == 0) & (np.abs(dirs).max(axis=1) > 1e-6)
    err = np.abs(np.linalg.norm(dirs - g["n"], axis=1) - 1)
    assert err[lamb].max() <= tol, (label, "lambertian", err[lamb].max() / ULP)


def check_cancel(out, in16, label):
    """The cancelling lambertian rows return a finite, nonzero direction: exactly n, or (float hardware that contracts
    n + u into one fma) a residual below the rounding of u.  Returns the number of rows that are exactly n."""
    d = out[:, 0:3].astype(np.float64)
    n = in16[:, 10:13]
    assert np.isfinite(d).all() and (np.abs(d).max(axis=1) > 0).all(), label
    exact = (d == n).all(axis=1)
    assert (exact | (np.abs(d).max(axis=1) <= ULP)).all(), (label, np.abs(d[~exact]).max())
    return int(exact.sum())


# ---------------------------------------------------------------------------------------------------------------
# (d) distributions
# ---------------------------------------------------------------------------------------------------------------
N_DRAWS = 2**18
P_MIN = 1e-3


def draws(mat, seed, front=1, face="random"):
    """N_DRAWS rows of one material with uniform random words; one fixed geometry (lambertian, metal) or a random
    geometry per row (dielectric)."""
    rng = np.random.default_rng(seed)
    k = N_DRAWS
    rnd = rng.integers(0, 2**32, size=(k, 4), dtype=np.uint64).astype(np.uint32)
    if face == "fixed":
        n = np.repeat(_unit(rng.normal(size=(1, 3))), k, axis=0)
        d = np.repeat(_unit(rng.normal(size=(1, 3))) * 2.5, k, axis=0)
    else:
        n = _unit(rng.normal(size=(k, 3)))
        d = _unit(rng.normal(size=(k, 3))) * 10.0 ** rng.uniform(-2, 2, size=(k, 1))
    return _rows(d, n, np.full(k, front), mat, rng), rnd


def check_unit_sphere(w, label):
    """w / |w| uniform on the sphere: z uniform on [-1, 1] and the azimuth uniform."""
    w = w / np.linalg.norm(w, axis=1, keepdims=True)
    p_z = stats.kstest(w[:, 2], "uniform", args=(-1, 2)).pvalue
    p_phi = stats.kstest(np.arctan2(w[:, 1], w[:, 0]), "uniform", args=(-np.pi, 2 * np.pi)).pvalue
    assert p_z > P_MIN and p_phi > P_MIN, (label, p_z, p_phi)


def check_lambertian(out, in16, label):
    check_unit_sphere(out[:, 0:3].astype(np.float64) - in16[:, 10:13], label)


def check_metal(out, in16, rnd, materials, label):
    """w = (d - mirror) / |min(fuzz, 1)|: |w|^3 uniform on [0, 1] and w / |w| uniform (a uniform point of the unit ball)."""
    g = geometry(in16, rnd, materials)
    f = abs(min(float(g["par"][0]), 1.0))
    w = (out[:, 0:3].astype(np.float64) - g["refl"]) / f
    r3 = np.linalg.norm(w, axis=1) ** 3
    p = stats.kstest(r3, "uniform").pvalue
    assert p > P_MIN, (label, "|w|^3", p, float(np.median(r3)))
    check_unit_sphere(w, label)


def check_dielectric(out, in16, rnd, materials, k_budget, label):
    """The reflected fraction is the batch mean of Schlick (1 under total internal reflection) within 5 binomial sigma;
    refracted directions obey Snell, |d_t x n| = eta |unit(d) x n|, and have length 1, within the budget of (b)."""
    g = geometry(in16, rnd, materials)
    out = out.astype(np.float64)
    refl = chose_reflection(out, g)
    p = g["p_refl"]
    sigma = np.sqrt(np.sum(p * (1 - p)))
    assert abs(refl.sum() - p.sum()) <= 5 * sigma + 1, (label, int(refl.sum()), p.sum(), sigma)
    t = ~refl
    assert t.sum() > 1000 or g["tir"].mean() > 0.9, label
    dt = out[t, 0:3]
    budget = k_budget * ULP * (np.abs(dt).max(axis=1) + 1 + 1 / np.abs(g["k"][t]))
    cross_t = np.linalg.norm(np.cross(dt, g["n"][t]), axis=1)
    cross_i = g["eta"][t] * np.linalg.norm(np.cross(g["ud"][t], g["n"][t]), axis=1)
    assert np.all(np.abs(cross_t - cross_i) <= 2 * budget), (label, "Snell", np.max(np.abs(cross_t - cross_i) / budget))
    assert np.all(np.abs(np.linalg.norm(dt, axis=1) - 1) <= 2 * budget), (label, "|d_t|")


DIST_CASES = ([("lambertian", m, 1) for m in LAMB[1:3]]
              + [("metal", METAL[FUZZ.index(f)], 1) for f in (-1.5, -0.5, 0.3, 1.0, 1.8)]
              + [("dielectric", m, front) for m in DIEL for front in (0, 1)])


def dist_id(c):
    kind, mat, front = c
    if kind == "lambertian":
        return "lambertian-%g" % ALBEDO[mat]
    if kind == "metal":
        return "metal-fuzz%g" % FUZZ[METAL.index(mat)]
    return "dielectric-ir%.6g-%s" % (IR[DIEL.index(mat)], "front" if front else "back")


def check_distribution(case, scatter, materials, k_budget, label):
    kind, mat, front = case
    in16, rnd = draws(mat, 1000 + mat + 50 * front, front, "fixed" if kind != "dielectric" else "random")
    out = scatter(in16, rnd)
    if kind == "lambertian":
        check_lambertian(out, in16, label)
    elif kind == "metal":
        check_metal(out, in16, rnd, materials, label)
    else:
        check_dielectric(out, in16, rnd, materials, k_budget, label)


# ---------------------------------------------------------------------------------------------------------------
# the tests: the two oracles
# ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def space():
    scene = space_scene()
    orc = Oracle(scene)
    in16, rnd, kind = space_inputs()
    return scene, orc, in16, rnd, kind


def test_inputs_cover_the_space(space):
    scene, orc, in16, rnd, kind = space
    assert set(in16[:, 14].astype(int)) == set(LAMB + METAL + DIEL)
    assert np.array_equal(in16, in16.astype(np.float32).astype(np.float64))  # the float inputs widen exactly
    d, n = in16[:, 3:6], in16[:, 10:13]
    assert (np.sum(d * n, axis=1) <= 0).all()  # faces as the render computes them
    length = np.linalg.norm(d, axis=1)
    assert length.min() < 2e-6 and length.max() > 5e5
    for w in range(4):
        assert set(SPECIAL) <= set(rnd[:, w])
    assert {0x0000, 0xFFFF} <= set(rnd[:, 3] >> 16) and {0x0000, 0xFFFF} <= set(rnd[:, 3] & 0xFFFF)
    g = geometry(in16, rnd, scene.materials)
    crit = kind == "critical"
    assert (g["tir_band"][crit] < 2.0**-21).mean() > 0.8 and g["tir"][crit].any() and (~g["tir"][crit]).any()
    graze = np.abs(np.sum(g["ud"] * n, axis=1))
    assert graze[kind == "grazing"].min() < 2.0**-28
    assert (np.abs(np.sum(g["ud"] * n, axis=1) + 1)[kind == "normal"] < 2.0**-22).all()  # normal incidence


def test_float_oracle_against_double_oracle(space):
    scene, orc, in16, rnd, kind = space
    lo = orc.scatter(in16.astype(np.float32), rnd)
    hi = orc.scatter_f64(in16, rnd)
    worst, n, ratio, ok = compare(lo, hi, in16, rnd, scene.materials, "float oracle")
    print("float oracle vs double oracle: worst direction error %.3f x 2^-24 (|d64| + 1 + 1/|k|) over %d rows" % (worst, n))
    assert n > 0.98 * len(in16)
    assert worst <= K_ORACLE
    for k in ("random", "normal", "grazing", "critical", "words"):
        assert (ok & (kind == k)).sum() > 100, k


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_anchors_on_the_oracles(space, precision):
    scene, orc, in16, rnd, kind = space
    out = orc.scatter(in16.astype(np.float32), rnd) if precision == "f32" else orc.scatter_f64(in16, rnd)
    # float normals are unit only to 2^-24: a few float ulps in both precisions
    anchors(out, in16, rnd, kind, scene.materials, 8 if precision == "f32" else 4, "oracle " + precision)
    c16, crnd = cancel_inputs(orc, precision)
    cin = c16.astype(np.float32) if precision == "f32" else c16
    out = orc.scatter(cin, crnd) if precision == "f32" else orc.scatter_f64(cin, crnd)
    assert check_cancel(out, c16, "oracle " + precision) == len(c16)  # n + u == 0 exactly: the fallback returns n


@pytest.mark.parametrize("precision", ["f32", "f64"])
@pytest.mark.parametrize("case", DIST_CASES, ids=dist_id)
def test_distributions_on_the_oracles(space, case, precision):
    scene, orc = space[0], space[1]
    if precision == "f32":
        fn = lambda a, r: orc.scatter(a.astype(np.float32), r)
    else:
        fn = orc.scatter_f64
    check_distribution(case, fn, scene.materials, K_ORACLE, "oracle " + precision)


def test_negative_fuzz_blurs_like_positive_fuzz(space):
    """fuzz -0.5 and +0.5 scatter to the same directions, bit for bit: fuzz * u over the points u of the unit ball is
    the same set of offsets, and the samplers here draw it as |fuzz| * u."""
    scene, orc, in16, rnd, kind = space
    m = scene.materials.copy()
    m["param"][METAL[FUZZ.index(-0.5)]] = 0.5
    pos = Oracle(SceneArrays(scene.camera, m, scene.spheres))
    rows = in16[:, 14] == METAL[FUZZ.index(-0.5)]
    a, r = in16[rows], rnd[rows]
    assert pos.scatter(a.astype(np.float32), r).tobytes() == orc.scatter(a.astype(np.float32), r).tobytes()
    assert pos.scatter_f64(a, r).tobytes() == orc.scatter_f64(a, r).tobytes()


# ---------------------------------------------------------------------------------------------------------------
# the executed reference (skipped where oracle/_ref is not built)
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.skipif(not have_ref(), reason="oracle/_ref not built (needs the reference sources)")
def test_varied_materials_mean_radiance_vs_reference():
    """Mean radiance of rays aimed at the metal and glass spheres of final.txt with varied fuzz (negative and above 1
    among them) and indices: the reference's ray_color (its own samplers, double build) against the oracle's estimator,
    equal within Monte-Carlo error, as test_oracle_vs_reference.py::test_estimator_mean_radiance does for the shipped
    scenes.  This pins the |fuzz| radius to the executed reference."""
    import ctypes as C

    from oracle_lib import RefWorld
    from test_path_by_path import varied_scene

    scene = varied_scene()
    orc = Oracle(scene)
    wd = RefWorld(scene, "d")
    m, s = scene.materials, scene.spheres
    cam = scene.camera["origin"][0].astype(np.float64)
    targets = []
    for typ, values in ((1, (-0.7, 1.8, 0.3)), (2, (2.42, 1 / 1.5))):
        for v in values:
            k = np.nonzero((m["type"][s["material"]] == typ) & (m["param"][s["material"]] == np.float32(v)))[0]
            targets.append(k[np.argmin(np.linalg.norm(s["center"][k] - cam, axis=1))])
    n_samp = 4000
    out = np.zeros(3, np.float32)
    for k in targets:
        ray = np.zeros(7, np.float32)
        ray[0:3] = cam
        ray[3:6] = s["center"][k] - cam
        ref_s = np.stack([wd.ray_color_mean(wd.list, ray.astype(np.float64), 50, 1) for _ in range(n_samp)])
        ours = np.zeros((n_samp, 3))
        for j in range(n_samp):
            orc.lib.orc_radiance(C.byref(orc._s), orc.bvh(), C.c_void_p(ray.ctypes.data), int(k), j, 50, C.c_uint64(1234),
                                 C.c_void_p(out.ctypes.data), None)
            ours[j] = out
        se = np.sqrt(ref_s.var(axis=0) / n_samp + ours.var(axis=0) / n_samp)
        assert np.all(np.abs(ours.mean(axis=0) - ref_s.mean(axis=0)) < 5 * se + 2e-3), (int(k), ours.mean(axis=0), ref_s.mean(axis=0), se)
