"""GPU: every search kernel against the float64 model of the library's arithmetic (oracle/fp16_model.py).

Where the 1e-3 comparators accept any row near the k-th score, these checks fix the result: each hit's score lies
within the model's bound of the exact score of the stored operands, and no row left out is provably better than the
k-th hit (or than the radius).  On ``fm.exact_inputs`` every accumulation order is exact, so there the kernels must
match the model bit for bit.

How the shapes reach the kernel instantiations (knobs are read per call, set through ``monkeypatch``):
- ``search_mma_kernel<CG, E>``: IVR_MMA_MODE=1, IVR_MMA_CTA_GROUP=CG; k <= 128 gives E = 8, k > 128 E = 0.
- ``search_mma_xres_kernel<E, TN>``: IVR_MMA_MODE=2; TN = 256 up to 512 dims, 224 / 192 at 768 dims (default /
  IVR_XRES_TN_768=192), 160 / 128 at 1024 dims (default / IVR_XRES_TN_1024=128).
- ``search_stream_kernel<NQ, DCH, E>``: path 1; NQ = nq rounded up to 1, 2, 4; DCH = 8 at 512 dims, 12 at 768, 0 at
  any other width; E as above.
- ``search_mma_small_kernel``: IVR_MMA_MODE=3.  List mode (IVR_SMALL_DUMP_MAX_KROWS=0) runs one launch below
  4 * 148 row tiles, two above, three with IVR_MMA_SMALL_RATIO=2; dump mode below 3.5 M rows and 32 queries at
  512 dims.
- ``search_mma_small_range_kernel``: range search, query chunks of 128 / 80 / 64 / 16 at 512 / 768 / 1024 / 4096 dims.

The largest |D - m| / eps per kernel family is printed at the end of the module (``pytest -s``).
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import fp16_model as fm, synth  # noqa: E402

RATIOS = {}


@pytest.fixture(scope="module", autouse=True)
def _report_ratios():
    yield
    for k in sorted(RATIOS):
        print(f"largest |D - m| / eps, {k}: {RATIOS[k]:.4f}")


def make_index(xb):
    import ivr_b200
    idx = ivr_b200.IndexFlatIP(xb.shape[1])
    idx.set_timing(True)
    idx.add(xb)
    return idx


def search(idx, rows16, xq, k, path=0, exact=False, id_offset=0, keys=False, device=False, first=0):
    """One search, checked against the model of the kernel that ran (ids = row of ``rows16`` + first + id_offset,
    ``first`` being the search window's first row); returns (D, I, kernel)."""
    import torch
    if keys:
        K = idx.search_keys_tensor(torch.from_numpy(xq).cuda(), k, id_offset=id_offset, path=path).cpu().numpy()
        D, I = fm.keys_to_DI(K)
    elif device or id_offset:
        D, I = idx.search_tensor(torch.from_numpy(xq).cuda(), k, id_offset=id_offset, path=path)
        D, I = D.cpu().numpy(), I.cpu().numpy()
    else:
        idx.search_path = path
        D, I = idx.search(xq, k)
    kern = idx.last_timing()["kernel"]
    bad = fm.check_topk(D, I, xq, rows16, fm.path_of(kern), id_offset=first + id_offset, exact=exact, ratios=RATIOS, tag=kern)
    assert not bad, "\n".join(bad[:10])
    return D, I, kern


def range_search(idx, rows16, xq, radius, exact=False, id_offset=0, keys=False, first=0):
    import torch
    q = torch.from_numpy(xq).cuda()
    if keys:
        lims, K = idx.range_search_keys_tensor(q, radius, id_offset=id_offset)
        lims, (D, I) = lims.cpu().numpy(), fm.keys_to_DI(K.cpu().numpy())
    elif id_offset:
        lims, D, I = (t.cpu().numpy() for t in idx.range_search_tensor(q, radius, id_offset=id_offset))
    else:
        lims, D, I = idx.range_search(xq, radius)
    bad = fm.check_range(lims, D, I, xq, rows16, "mma", radius, id_offset=first + id_offset, exact=exact, ratios=RATIOS,
                         tag="search_mma_small_range_kernel")
    assert not bad, "\n".join(bad[:10])
    return lims, D, I


def data(kind, n, d, nq, seed):
    if kind == "exact":
        return fm.exact_inputs(n, d, nq, seed)
    return synth.clip_like(n, d, seed, n_centres=256), synth.clip_like(nq, d, seed + 1, n_centres=256)


def set_env(monkeypatch, env):
    for k, v in env.items():
        monkeypatch.setenv(k, str(v))


# (id, dim, rows, queries, k, path, knobs, kernel)
CASES = [
    ("qres_cg1_e8", 512, 20000, 200, 100, 2, {"IVR_MMA_MODE": 1, "IVR_MMA_CTA_GROUP": 1}, "search_mma_kernel"),
    ("qres_cg1_e0", 512, 20000, 200, 200, 2, {"IVR_MMA_MODE": 1, "IVR_MMA_CTA_GROUP": 1}, "search_mma_kernel"),
    ("qres_cg2_e8", 384, 20000, 300, 128, 2, {"IVR_MMA_MODE": 1, "IVR_MMA_CTA_GROUP": 2}, "search_mma_kernel"),
    ("qres_cg2_e0", 384, 20000, 300, 129, 2, {"IVR_MMA_MODE": 1, "IVR_MMA_CTA_GROUP": 2}, "search_mma_kernel"),
    ("xres256_e8", 512, 20000, 300, 100, 2, {"IVR_MMA_MODE": 2}, "search_mma_xres_kernel"),
    ("xres256_e0", 512, 20000, 300, 300, 2, {"IVR_MMA_MODE": 2}, "search_mma_xres_kernel"),
    ("xres224_e8", 768, 20000, 300, 100, 2, {"IVR_MMA_MODE": 2}, "search_mma_xres_kernel"),
    ("xres224_e0", 768, 20000, 300, 200, 2, {"IVR_MMA_MODE": 2}, "search_mma_xres_kernel"),
    ("xres192_e8", 768, 20000, 300, 100, 2, {"IVR_MMA_MODE": 2, "IVR_XRES_TN_768": 192}, "search_mma_xres_kernel"),
    ("xres192_e0", 768, 20000, 300, 200, 2, {"IVR_MMA_MODE": 2, "IVR_XRES_TN_768": 192}, "search_mma_xres_kernel"),
    ("xres160_e8", 1024, 20000, 300, 100, 2, {"IVR_MMA_MODE": 2}, "search_mma_xres_kernel"),
    ("xres160_e0", 1024, 20000, 300, 200, 2, {"IVR_MMA_MODE": 2}, "search_mma_xres_kernel"),
    ("xres128_e8", 1024, 20000, 300, 100, 2, {"IVR_MMA_MODE": 2, "IVR_XRES_TN_1024": 128}, "search_mma_xres_kernel"),
    ("xres128_e0", 1024, 20000, 300, 200, 2, {"IVR_MMA_MODE": 2, "IVR_XRES_TN_1024": 128}, "search_mma_xres_kernel"),
    ("stream_nq1_dch8_e8", 512, 20000, 1, 100, 1, {}, "search_stream_kernel"),
    ("stream_nq1_dch8_e0", 512, 20000, 1, 300, 1, {}, "search_stream_kernel"),
    ("stream_nq2_dch12_e8", 768, 20000, 2, 100, 1, {}, "search_stream_kernel"),
    ("stream_nq2_dch12_e0", 768, 20000, 2, 200, 1, {}, "search_stream_kernel"),
    ("stream_nq4_dch0_e8", 320, 20000, 3, 100, 1, {}, "search_stream_kernel"),
    ("stream_nq4_dch0_e0", 320, 20000, 4, 1025, 1, {}, "search_stream_kernel"),
    ("stream_nq4_dch8_e0", 512, 20000, 4, 129, 1, {}, "search_stream_kernel"),
    ("stream_nq1_dch12_e0", 768, 20000, 1, 1024, 1, {}, "search_stream_kernel"),
    ("small_list_1launch", 512, 30000, 40, 100, 2, {"IVR_MMA_MODE": 3, "IVR_SMALL_DUMP_MAX_KROWS": 0},
     "search_mma_small_kernel"),
    ("small_list_2launch", 256, 100000, 40, 100, 2, {"IVR_MMA_MODE": 3, "IVR_SMALL_DUMP_MAX_KROWS": 0},
     "search_mma_small_kernel"),
    ("small_list_3launch", 256, 100000, 40, 300, 2,
     {"IVR_MMA_MODE": 3, "IVR_SMALL_DUMP_MAX_KROWS": 0, "IVR_MMA_SMALL_RATIO": 2}, "search_mma_small_kernel"),
    ("small_dump", 512, 30000, 20, 100, 2, {"IVR_MMA_MODE": 3}, "search_mma_small_kernel"),
]
LAUNCHES = {"small_list_1launch": 1, "small_list_2launch": 2, "small_list_3launch": 3, "small_dump": 1}


@pytest.mark.parametrize("kind", ["exact", "clip"])
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_instantiations(case, kind, monkeypatch):
    name, d, n, nq, k, path, env, kernel = case
    set_env(monkeypatch, env)
    xb, xq = data(kind, n, d, nq, seed=d + k)
    rows16 = fm.store(xb)
    idx = make_index(xb)
    D, I, kern = search(idx, rows16, xq, k, path, exact=kind == "exact")
    assert kern == kernel
    if name in LAUNCHES:
        assert idx.last_timing()["score_launches"] == LAUNCHES[name]
    if kind == "exact":                                                      # determinism
        D2, I2, _ = search(idx, rows16, xq, k, path, exact=True)
        assert np.array_equal(D, D2) and np.array_equal(I, I2)


@pytest.mark.parametrize("kind", ["exact", "clip"])
@pytest.mark.parametrize("d", [512, 768, 1024, 4096])
def test_range_chunks(d, kind):
    chunk = min(128, 65536 // d // 16 * 16)
    xb, xq = data(kind, 6000 if d == 4096 else 20000, d, chunk + 3, seed=d)
    rows16 = fm.store(xb)
    idx = make_index(xb)
    m, _ = fm.scores(xq, rows16, "mma")
    radius = float(np.float32(np.median(np.sort(m, axis=1)[:, -40])))
    lims, D, I = range_search(idx, rows16, xq, radius, exact=kind == "exact")
    assert lims[-1] > 0
    if kind == "exact":
        lims2, D2, I2 = range_search(idx, rows16, xq, radius, exact=True)
        assert np.array_equal(lims, lims2) and np.array_equal(D, D2) and np.array_equal(I, I2)


@pytest.mark.parametrize("kind", ["exact", "clip"])
@pytest.mark.parametrize("k", [1, 127, 128, 129, 256, 257, 1024, 1025, 2048])
@pytest.mark.parametrize("path", [1, 2], ids=["stream", "mma"])
def test_k_edges(k, path, kind):
    xb, xq = data(kind, 5000, 128, 3 if path == 1 else 24, seed=k)
    rows16 = fm.store(xb)
    search(make_index(xb), rows16, xq, k, path, exact=kind == "exact")


@pytest.mark.parametrize("n", [1, 99, 127, 128, 129, 2047, 2048, 2049])
@pytest.mark.parametrize("mode", ["stream", "qres", "xres", "small"])
def test_n_edges(n, mode, monkeypatch):
    path, nq = (1, 2) if mode == "stream" else (2, 300 if mode in ("qres", "xres") else 24)
    set_env(monkeypatch, {"qres": {"IVR_MMA_MODE": 1}, "xres": {"IVR_MMA_MODE": 2},
                          "small": {"IVR_MMA_MODE": 3, "IVR_SMALL_DUMP_MAX_KROWS": 0}}.get(mode, {}))
    for kind in ("exact", "clip"):
        xb, xq = data(kind, n, 256, nq, seed=n)
        search(make_index(xb), fm.store(xb), xq, 100, path, exact=kind == "exact")


@pytest.mark.parametrize("d", [1, 63, 65, 100, 513, 1280])
def test_odd_dims(d):
    for kind in ("exact", "clip"):
        xb, xq = data(kind, 3000, d, 20, seed=d)
        idx, rows16 = make_index(xb), fm.store(xb)
        for path, q in ((1, xq[:1]), (2, xq)):
            search(idx, rows16, q, 50, path, exact=kind == "exact")
        m, _ = fm.scores(xq, rows16, "mma")
        range_search(idx, rows16, xq, float(np.float32(np.sort(m[0])[-30])), exact=kind == "exact")


@pytest.mark.parametrize("early_qres_krows", [0, 100000])
@pytest.mark.parametrize("mode", [1, 2], ids=["qres", "xres"])
def test_many_seeded_launches(mode, early_qres_krows, monkeypatch):
    xb = synth.clip_like(300_000, 128, seed=3, n_centres=1024)
    xq = synth.clip_like(256, 128, seed=4, n_centres=1024)
    rows16 = fm.store(xb)
    idx = make_index(xb)
    set_env(monkeypatch, {"IVR_MMA_MODE": mode, "IVR_MMA_CTA_GROUP": 2, "IVR_MMA_EARLY_QRES_MAX_KROWS": early_qres_krows})
    for k in (100, 300):
        monkeypatch.setenv("IVR_MMA_TWO_PHASE", "0")
        D0, I0, _ = search(idx, rows16, xq, k, 2)
        monkeypatch.setenv("IVR_MMA_TWO_PHASE", "1")
        monkeypatch.setenv("IVR_MMA_PHASE0_ROWS", "256")
        monkeypatch.setenv("IVR_MMA_PHASE_RATIO", "2")
        D, I, _ = search(idx, rows16, xq, k, 2)
        assert idx.last_timing()["score_launches"] >= 6
        assert np.array_equal(D, D0) and np.array_equal(I, I0)
        monkeypatch.delenv("IVR_MMA_PHASE0_ROWS")
        monkeypatch.delenv("IVR_MMA_PHASE_RATIO")


@pytest.mark.parametrize("path", [1, 2], ids=["stream", "mma"])
def test_boundary_dense_rows(path):
    """Rows whose scores sit on a 2e-5 grid around the k-th score: dozens inside the old 1e-3 band, every one of them
    fixed by the model wherever two neighbours are more than twice the bound apart."""
    d, k, nq = 512, 100, 3 if path == 1 else 16
    rng = np.random.default_rng(7)
    xb = synth.clip_like(20000, d, seed=8, n_centres=64)
    xq = synth.clip_like(nq, d, seed=9, n_centres=64)
    qh = xq / np.linalg.norm(xq, axis=1, keepdims=True)
    kth = np.sort(xb @ xq.T, axis=0)[-k]
    extra = []
    for q in range(nq):
        a = kth[q] + 2e-5 * np.arange(-60, 61)
        u = rng.standard_normal((a.size, d))
        u -= (u @ qh[q])[:, None] * qh[q]
        u /= np.linalg.norm(u, axis=1, keepdims=True)
        extra.append(a[:, None] * qh[q] + np.sqrt(1 - a[:, None] ** 2) * u)
    xb = np.concatenate([xb, np.concatenate(extra)]).astype(np.float32)
    rows16 = fm.store(xb)
    m, _ = fm.scores(xq, rows16, "stream" if path == 1 else "mma")
    kk = np.sort(m, axis=1)[:, -k]
    assert np.all((np.abs(m - kk[:, None]) < 1e-3).sum(axis=1) > 40)
    search(make_index(xb), rows16, xq, k, path)


SCALES = [2.0 ** -140, 1.5 * 2.0 ** -128, 1e-30, 1e30]


@pytest.mark.parametrize("how", ["stream", "small", "qres", "range"])
def test_query_magnitudes(how, monkeypatch):
    """Queries far from unit norm: every path must match its own model (the tcgen05 paths scale the query by a power
    of two clamped to 2^+-127; the streaming kernel multiplies the fp32 query as given)."""
    d = 512
    if how == "qres":
        set_env(monkeypatch, {"IVR_MMA_MODE": 1})
    xb = synth.clip_like(20000, d, seed=21, n_centres=256)
    rows16 = fm.store(xb)
    idx = make_index(xb)
    base = synth.clip_like(6, d, seed=22, n_centres=256)
    sub = base.copy()
    sub[:, 1::2] *= np.float32(2.0 ** -20)                   # components in fp16's subnormal range after scaling
    onehot = np.zeros((1, d), np.float32)
    onehot[0, 5] = np.float32(3.2e38)
    batches = [(base * np.float32(s)).astype(np.float32) for s in SCALES]
    batches += [onehot, np.zeros((1, d), np.float32), sub]
    ex_b, ex_q = fm.exact_inputs(1, d, 4, seed=23, query_exp=-140)
    for xq in batches:
        if how == "range":
            m, _ = fm.scores(xq, rows16, "mma")
            for radius in (0.0, float(np.float32(np.sort(m[0])[-25]))):
                range_search(idx, rows16, xq, radius)
            continue
        nq = {"stream": 1, "small": 8, "qres": 200}[how]
        q = np.resize(xq, (nq, d)).astype(np.float32)
        search(idx, rows16, q, 100, 1 if how == "stream" else 2)
    # exact inputs with queries near 2^-140: the rescaled scores are fp32 subnormals, still exact
    xb2, xq2 = fm.exact_inputs(5000, d, 8, seed=24, query_exp=-140)
    idx2, rows2 = make_index(xb2), fm.store(xb2)
    if how == "range":
        range_search(idx2, rows2, xq2, 0.0, exact=True)
    else:
        q = np.resize(xq2, ({"stream": 1, "small": 8, "qres": 200}[how], d)).astype(np.float32)
        search(idx2, rows2, q, 100, 1 if how == "stream" else 2, exact=True)


NAN_AT = [0, 127, 128, 129, 2047, 2048, 4095]


@pytest.mark.parametrize("how", ["stream", "list", "dump", "keys", "range", "range_keys"])
def test_nan_rows(how, monkeypatch):
    """Rows holding a NaN score NaN against every query and are never returned."""
    d, n = 256, 5000
    if how in ("list", "keys"):
        set_env(monkeypatch, {"IVR_MMA_MODE": 3, "IVR_SMALL_DUMP_MAX_KROWS": 0})
    elif how == "dump":
        set_env(monkeypatch, {"IVR_MMA_MODE": 3})
    xb, xq = data("clip", n, d, 8, seed=31)
    xb[NAN_AT, 3] = np.nan
    rows16 = fm.store(xb)
    idx = make_index(xb)
    if how.startswith("range"):
        range_search(idx, rows16, xq, -1.0, keys=how == "range_keys")          # every finite row is a hit
        return
    q = xq[:1] if how == "stream" else xq
    for k in (100, 1000):
        search(idx, rows16, q, k, 1 if how == "stream" else 2, keys=how == "keys")
    # more rows than finite ones: k' = the finite rows, then padding
    small = xb[:300].copy()
    small[::3, 0] = np.nan
    idx2, rows2 = make_index(small), fm.store(small)
    D, I, _ = search(idx2, rows2, q, 250, 1 if how == "stream" else 2, keys=how == "keys")
    assert np.all(I[:, 200:] == -1)


def test_inf_component_through_normalize_l2():
    import ivr_b200
    xb, xq = data("clip", 2000, 128, 4, seed=41)
    xb[[5, 1000], 7] = np.inf
    ivr_b200.normalize_L2(xb)
    assert np.isnan(xb[5]).any() and np.isnan(xb[1000]).any()
    idx, rows16 = make_index(xb), fm.store(xb)
    for path, q in ((1, xq[:1]), (2, xq)):
        D, I, _ = search(idx, rows16, q, 2048, path)
        assert not np.isin(I, [5, 1000]).any() and np.all(I[:, 1998:] == -1)
    range_search(idx, rows16, xq, -2.0)


def test_one_handle_many_calls(monkeypatch):
    """A seeded sequence of calls on one handle, each checked: state that outlives a call (select-merge tickets and
    pool counters, dump-mode memsets, per-launch keys, cached row descriptors) must not leak into the next one."""
    import torch
    rng = np.random.default_rng(2024)
    d = 256
    xb = synth.clip_like(90000, d, seed=51, n_centres=512)
    idx = make_index(xb[:60000])
    stored = xb[:60000]
    knobs = ["IVR_MMA_MODE", "IVR_SMALL_DUMP_MAX_KROWS", "IVR_MMA_CTA_GROUP", "IVR_MMA_TWO_PHASE", "IVR_MMA_PHASE0_ROWS"]
    for step in range(48):
        if step == 24:                                           # regrow mid-sequence
            idx.add(torch.from_numpy(xb[60000:]).cuda())
            stored = xb
        for kn in knobs:
            monkeypatch.delenv(kn, raising=False)
        mode = int(rng.integers(0, 4))
        if mode:
            monkeypatch.setenv("IVR_MMA_MODE", str(mode))
        if rng.random() < 0.5:
            monkeypatch.setenv("IVR_SMALL_DUMP_MAX_KROWS", "0")
        if rng.random() < 0.3:
            monkeypatch.setenv("IVR_MMA_PHASE0_ROWS", "512")
        if rng.random() < 0.2:
            monkeypatch.setenv("IVR_MMA_TWO_PHASE", "0")
        monkeypatch.setenv("IVR_MMA_CTA_GROUP", str(int(rng.integers(0, 3))))
        nq = int(rng.choice([1, 2, 3, 5, 16, 33, 64] + ([] if mode == 3 else [200])))
        k = int(rng.choice([1, 10, 100, 128, 129, 300, 1024, 1025]))
        n = len(stored)
        first, count = 0, n
        if rng.random() < 0.3:
            first = int(rng.integers(0, n // 2))
            count = int(rng.integers(1, n - first))
            idx.set_window(first, count)
        rows16 = fm.store(stored[first:first + count])
        off = int(rng.choice([0, 0, 7, 1 << 20]))
        xq = synth.clip_like(nq, d, seed=1000 + step, n_centres=512)
        kind = rng.choice(["host", "device", "keys", "range"])
        if kind == "range":
            m, _ = fm.scores(xq[:1], rows16, "mma")
            r = float(np.float32(np.sort(m[0])[-min(50, count)]))
            range_search(idx, rows16, xq, r, id_offset=off, keys=bool(rng.random() < 0.5), first=first)
        else:
            path = int(rng.choice([0, 1, 2]))
            search(idx, rows16, xq, k, path, id_offset=0 if kind == "host" else off, keys=kind == "keys",
                   device=kind == "device", first=first)
        idx.set_window()
