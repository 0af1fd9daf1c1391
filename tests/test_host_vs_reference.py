"""Host-side mirror (pycwt_b200/{helpers,mothers,wavelet.significance}) and the CPU oracle
against the real reference on seeded random inputs.

Each `*_records` function below makes one family of seeded calls on a module with the
reference's interface and returns `(key, rule, value)` records.  `tests/golden/make_host_golden.py`
runs them on the unmodified reference and stores its records in `host_vs_reference.npz`; the
tests run them on this project and compare record by record.  Arrays of more than `FULL`
elements are stored reduced (see `reduce_record`): a SHA-256 of their bytes where the rule is
bit equality, else a seeded sample of elements with the count of non-finite values and the
sum of squares of the finite ones of the whole array."""
import functools
import hashlib
import warnings
import zlib

import numpy as np
import pytest

from conftest import load_golden

FIXTURE = "host_vs_reference"
FULL = 128          # arrays up to this many elements are stored whole
SAMPLE = 64         # elements stored of a larger array compared within a tolerance

# comparison rules: (name, tolerance)
EQ = ("eq", 0.0)            # a == b on scalars and strings
EXACT = ("exact", 0.0)      # bit-identical arrays (NaN equal to NaN)


def rtol(t):
    return ("rtol", t)      # np.allclose(rtol=t, atol=0, equal_nan=True)


def absdiff(t):
    return ("abs", t)       # max |a - b| < t


def phase(t):
    return ("phase", t)     # max |exp(i a) - exp(i b)| < t


def rel(t):
    return ("rel", t)       # |a - b| <= t |a| (scalars)


def attempt(key, rule, fn, n_out=None):
    """Records of one call: its outputs (`key.i` for each of `n_out` outputs), or the name of
    the exception it raised.  Returns (records, outputs or None)."""
    try:
        r = fn()
    except Exception as e:      # noqa: BLE001  (the reference's own exception types are compared)
        return [(key, ("raises", 0.0), e)], None
    if n_out is None:
        return [(key, rule, r)], r
    return [("%s.%d" % (key, i), rule, r[i]) for i in range(n_out)], r


# ---------------------------------------------------------------------------------------------
# the seeded calls
# ---------------------------------------------------------------------------------------------
def mother_records(mothers):
    f = np.r_[np.linspace(-30, 30, 241), [0.0, 1e-3, 800.0, -800.0]]
    out = []
    for fam, params in (("Morlet", [6, 4.5, 8, 12, 20]), ("Paul", [4, 1, 2, 6, 10]),
                        ("DOG", [2, 1, 3, 6, 9])):
        for p in params:
            w, k = getattr(mothers, fam)(p), "mother.%s(%s)." % (fam, p)
            with np.errstate(all="ignore"):
                out.append((k + "psi_ft", EXACT, w.psi_ft(f)))
                out.append((k + "psi0", rel(4e-16), w.psi(0)))
            out += [(k + "flambda", EQ, w.flambda()), (k + "coi", EQ, w.coi())]
            out += [(k + a, EQ, getattr(w, a)) for a in ("name", "dofmin", "cdelta", "gamma", "deltaj0")]
    out.append(("mother.MexicanHat.name", EQ, mothers.MexicanHat().name))
    return out


def helper_records(helpers):
    out = []
    rs = np.random.RandomState(3)
    for it in range(120):
        n = int(rs.randint(8, 3000))
        x = np.cumsum(rs.randn(n)) * rs.uniform(0.1, 10) if rs.rand() < 0.5 else rs.randn(n)
        out += attempt("ar1.%d" % it, rtol(1e-13), lambda: helpers.ar1(x))[0]
        fr, al = rs.uniform(0, 0.5, size=rs.randint(1, 50)), rs.uniform(-0.95, 0.95)
        out.append(("ar1_spectrum.%d" % it, EXACT, helpers.ar1_spectrum(fr, al)))
        k = int(rs.randint(1, 40))
        out.append(("rect.%d" % it, EXACT, helpers.rect(k, normalize=bool(it % 2))))
        seed, g = int(rs.randint(1e6)), float(rs.uniform(0.01, 0.95) * rs.choice([-1, 1]))
        np.random.seed(seed)
        out.append(("rednoise.%d" % it, EXACT, helpers.rednoise(n, g, 2.0)))  # same draws, same RNG consumption
        c = rs.rand(30) > 0.5
        out.append(("find.%d" % it, EXACT, helpers.find(c)))
    return out


def significance_records(pkg, mothers):
    out = []
    rs = np.random.RandomState(4)
    for it in range(120):
        n, dt = int(rs.randint(32, 2000)), float(10 ** rs.uniform(-1, 1))
        x = rs.randn(n)
        fam = rs.randint(3)
        w = [mothers.Morlet(6), mothers.Paul(4), mothers.DOG(2)][fam]
        S = int(rs.randint(3, 40))
        sj = 2 * dt * 2 ** (np.arange(S) * 0.25)
        st = int(rs.randint(3))
        kw = dict(sigma_test=st, alpha=float(rs.uniform(0, 0.9)),
                  significance_level=float(rs.choice([0.9, 0.95, 0.99])))
        sig = x if rs.rand() < 0.5 else float(x.var())
        if st == 1:
            kw["dof"] = (n - sj).copy()
        if st == 2:
            kw["dof"] = [sj[1], sj[min(S - 1, 5)]]
        out += attempt("significance.%d" % it, rtol(1e-13),
                       lambda: pkg.significance(sig, dt, sj.copy(), wavelet=w, **kw), 2)[0]
    return out


def transform_records(mod):
    """cwt / icwt on random lengths, sampling steps, families, orders and scale steps, then
    xwt and wct on pairs of AR(1) series."""
    from scipy.signal import lfilter
    out = []
    rs = np.random.RandomState(6)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for it in range(60):
            n, dt = int(2 ** rs.uniform(2.2, 11)), float(10 ** rs.uniform(-1, 1))
            x = rs.randn(n)
            fam = rs.randint(3)
            order = [rs.choice([6, 8]), rs.choice([4, 2, 6]), rs.choice([2, 3, 6])][fam]
            w = [mod.Morlet, mod.Paul, mod.DOG][fam](order)
            dj = float(rs.choice([0.5, 0.25, 0.125]))
            with np.errstate(all="ignore"):
                recs, r = attempt("cwt.%d" % it, rtol(1e-12), lambda: mod.cwt(x, dt, dj=dj, wavelet=w), 6)
                out += recs
                if r is not None and w.cdelta != -1 and r[0].size and np.isfinite(r[0]).all():
                    out.append(("icwt.%d" % it, rtol(1e-12), mod.icwt(r[0], r[1], dt, dj, w)))
        m = mod.Morlet(6)
        for it in range(10):
            n, dt = int(2 ** rs.uniform(5, 9)), float(10 ** rs.uniform(-1, 1))
            y1 = lfilter([1], [1, -0.5], rs.randn(n))
            y2 = np.roll(y1, 2) + 0.7 * rs.randn(n)
            dj = float(rs.choice([0.5, 0.25, 1 / 6]))
            out += [("xwt.%d.%d" % (it, i), rtol(1e-11), a)
                    for i, a in enumerate(mod.xwt(y1, y2, dt, dj=dj, wavelet=m))]
            a = mod.wct(y1, y2, dt, dj=dj, sig=False, wavelet=m)
            out += [("wct.%d.WCT" % it, absdiff(1e-10), a[0]), ("wct.%d.aWCT" % it, phase(1e-9), a[1]),
                    ("wct.%d.coi" % it, rtol(1e-14), a[2]), ("wct.%d.freq" % it, EXACT, a[3])]
    return out


# ---------------------------------------------------------------------------------------------
# storing and comparing records
# ---------------------------------------------------------------------------------------------
def _sample_index(key, size):
    rs = np.random.RandomState(zlib.crc32(key.encode()))
    return np.sort(rs.choice(size, SAMPLE, replace=False))


def _sha256(a):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), np.uint8)


def _layout(a):
    return "%s %s" % (a.dtype.str, a.shape)


def _stats(flat):
    fin = np.isfinite(flat)
    return np.array([(~fin).sum(), (np.abs(flat[fin]) ** 2).sum()])


def reduce_record(key, rule, value):
    """The arrays stored for one record, under `key:<field>`."""
    if rule[0] == "raises":
        return {key + ":raises": np.array(type(value).__name__)}
    a = np.asarray(value)
    if rule[0] == "eq" or a.size <= FULL:
        return {key + ":value": a}
    out = {key + ":layout": np.array(_layout(a))}
    if rule[0] == "exact":
        out[key + ":sha256"] = _sha256(a)
        return out
    flat = a.ravel()
    out[key + ":sample"] = flat[_sample_index(key, flat.size)]
    out[key + ":stats"] = _stats(flat)
    return out


def pack(arrays):
    """The stored fields as one flat array per dtype plus an index of `key, array, offset,
    shape` lines: a fixture of a few entries rather than one per field."""
    groups, parts, index = {}, {}, []
    for key, a in arrays.items():
        a = np.asarray(a)
        g = groups.setdefault(a.dtype.str, "g%d" % len(groups))
        chunks = parts.setdefault(g, [])
        off = sum(c.size for c in chunks)
        index.append("%s\t%s\t%d\t%s" % (key, g, off, ",".join(str(d) for d in a.shape)))
        chunks.append(a.ravel())
    out = {g: np.concatenate(c) for g, c in parts.items()}
    out["index"] = np.array(index)
    return out


@functools.lru_cache(maxsize=None)
def stored_fields():
    """The inverse of `pack` on the committed fixture: {key:field: array}."""
    g = load_golden(FIXTURE)
    data = {k: g[k] for k in g.files if k != "index"}
    out = {}
    for line in g["index"]:
        key, grp, off, shape = str(line).split("\t")
        shape = tuple(int(d) for d in shape.split(",") if d)
        n = int(np.prod(shape))
        out[key] = data[grp][int(off):int(off) + n].reshape(shape)
    return out


def _close(rule, a, ref):
    name, tol = rule
    a, ref = np.asarray(a), np.asarray(ref)
    if a.shape != ref.shape:
        return False
    if name == "exact":
        return np.array_equal(a, ref, equal_nan=True)
    if name == "rtol":
        return np.allclose(a, ref, rtol=tol, atol=0, equal_nan=True)
    if name == "abs":
        return a.size == 0 or np.abs(a - ref).max() < tol
    if name == "phase":
        return a.size == 0 or np.abs(np.exp(1j * a) - np.exp(1j * ref)).max() < tol
    if name == "rel":
        return bool(np.all(np.abs(a - ref) <= tol * np.abs(ref)))
    raise ValueError(name)


def check_records(records, prefix):
    """Compares this project's records with the reference's stored ones; every stored record
    under `prefix` must have been produced."""
    g = stored_fields()
    stored = {k.split(":")[0] for k in g if k.startswith(prefix)}
    assert stored, prefix
    seen = set()
    for key, rule, value in records:
        seen.add(key)
        if key + ":raises" in g:
            assert rule[0] == "raises", (key, "the reference raised %s" % g[key + ":raises"])
            assert str(g[key + ":raises"]) in [c.__name__ for c in type(value).__mro__], (key, value)
            continue
        assert rule[0] != "raises", (key, "raised %r where the reference did not" % value)
        if key + ":value" in g:
            ref = g[key + ":value"]
            if rule[0] == "eq":
                assert ref.item() == value, (key, ref, value)
            else:
                assert _close(rule, value, ref), key
            continue
        a = np.asarray(value)
        assert _layout(a) == str(g[key + ":layout"]), (key, _layout(a), g[key + ":layout"])
        if rule[0] == "exact":
            assert np.array_equal(_sha256(a), g[key + ":sha256"]), key
            continue
        flat = a.ravel()
        assert _close(rule, flat[_sample_index(key, flat.size)], g[key + ":sample"]), key
        (nonfinite, s), (nonfinite_ref, s_ref) = _stats(flat), g[key + ":stats"]
        assert nonfinite == nonfinite_ref, (key, nonfinite, nonfinite_ref)
        if rule[0] != "phase":      # an angle's sum of squares depends on its branch
            assert abs(s - s_ref) <= 10 * rule[1] * abs(s_ref), (key, s, s_ref)
    assert seen == stored, sorted(stored ^ seen)[:10]


# ---------------------------------------------------------------------------------------------
# the tests
# ---------------------------------------------------------------------------------------------
def test_mother_wavelets_match():
    from pycwt_b200 import mothers as om
    check_records(mother_records(om), "mother.")


def test_helpers_match():
    from pycwt_b200 import helpers as oh
    check_records(helper_records(oh), ("ar1.", "ar1_spectrum.", "rect.", "rednoise.", "find."))
    assert oh.fft_kwargs(np.zeros(300)) == {"n": 512}


def test_significance_matches():
    import pycwt_b200 as our
    from pycwt_b200 import mothers as om
    check_records(significance_records(our, om), "significance.")


def test_oracle_matches_reference_on_random_inputs():
    """The oracle on random lengths, sampling steps, families, orders and call variants."""
    from oracle import cwt_oracle as orc
    check_records(transform_records(orc), ("cwt.", "icwt.", "xwt.", "wct."))


@pytest.mark.parametrize("rule, a, b, same", [
    (EXACT, [1.0, np.nan], [1.0, np.nan], True), (EXACT, [1.0], [1.0 + 1e-16 * 4], False),
    (rtol(1e-12), [1.0], [1.0 + 1e-13], True), (rtol(1e-12), [1.0], [1.0 + 1e-11], False),
    (absdiff(1e-10), [0.5], [0.5 + 2e-10], False), (phase(1e-9), [np.pi], [-np.pi], True),
    (rel(4e-16), 1.0, 1.0 + 4.4e-16, False)])
def test_comparison_rules(rule, a, b, same):
    assert _close(rule, a, b) == same
