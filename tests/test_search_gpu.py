"""GPU: exact top-k search parity -- CUDA path (through the C ABI) vs. the oracle.

Tolerance (north_star): identical ids except ties within 1e-3 of the k-th score; scores
within 1e-3 (rows are stored as fp16, accumulation is fp32).
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import comparator, flat_ip, synth  # noqa: E402

TOL = 1e-3


def build(xb, chunk=None):
    import ivr_b200
    idx = ivr_b200.IndexFlatIP(xb.shape[1])
    ref = flat_ip.IndexFlatIP(xb.shape[1])
    if chunk is None:
        idx.add(xb)
    else:                                          # ragged multi-chunk add (regrowth path)
        for s in range(0, len(xb), chunk):
            idx.add(xb[s:s + chunk])
    ref.add(xb)
    assert idx.ntotal == ref.ntotal == len(xb)
    return idx, ref


def check(idx, ref, xq, k, path=0, tol=TOL):
    idx.search_path = path
    D, I = idx.search(xq, k)
    Dr, Ir = ref.search(xq, k)
    bad = comparator.compare_topk(D, I, Dr, Ir, lambda ids: ref.scores_of(xq, ids), tol)
    assert not bad, "\n".join(bad[:10])
    return D, I


@pytest.mark.parametrize("d", [512, 768, 384, 100, 64, 1024])
@pytest.mark.parametrize("nq", [1, 2, 3, 4, 7])
def test_stream_path_dims_and_batches(d, nq):
    xb = synth.clip_like(20000, d, seed=31, n_centres=256)
    xq = synth.clip_like(nq, d, seed=32, n_centres=256)
    idx, ref = build(xb)
    check(idx, ref, xq, 100, path=1)
    assert idx.last_timing()["path"] == "stream"


@pytest.mark.parametrize("k", [1, 5, 50, 100, 128, 129, 300, 1000, 2048])
def test_stream_path_k_values(k):
    xb = synth.clip_like(30000, 128, seed=33, n_centres=64)
    xq = synth.clip_like(3, 128, seed=34, n_centres=64)
    idx, ref = build(xb, chunk=7001)
    check(idx, ref, xq, k, path=1)


@pytest.fixture(params=[(1, 1), (2, 1), (2, 2)], ids=["qres_cta_group1", "qres_cta_group2", "xres_cta_group2"])
def cta_group(request, monkeypatch):
    """Kernel variants of the tcgen05 path: query-tile-resident (1 CTA / CTA pair), row-tile-resident."""
    cg, mode = request.param
    monkeypatch.setenv("IVR_MMA_CTA_GROUP", str(cg))
    monkeypatch.setenv("IVR_MMA_MODE", str(mode))
    return request.param


@pytest.mark.parametrize("d", [512, 384, 64, 100, 768, 1024])
@pytest.mark.parametrize("nq", [5, 128, 300])
def test_mma_path_dims_and_batches(d, nq, cta_group):
    xb = synth.clip_like(30000, d, seed=61, n_centres=256)
    xq = synth.clip_like(nq, d, seed=62, n_centres=256)
    idx, ref = build(xb)
    check(idx, ref, xq, 100, path=2)
    assert idx.last_timing()["path"] == "mma"


@pytest.mark.parametrize("n", [1, 100, 255, 256, 257, 1000, 5000])
def test_mma_path_small_indexes(n, cta_group):
    xb = synth.gaussian_unit(n, 128, seed=63 + n)
    xq = synth.gaussian_unit(37, 128, seed=64)
    idx, ref = build(xb)
    D, I = check(idx, ref, xq, 100, path=2)
    if n < 100:
        assert (I[:, n:] == -1).all()


@pytest.mark.parametrize("k", [1, 10, 128, 129, 300, 1000, 2048])
def test_mma_path_k_values(k, cta_group):
    xb = synth.clip_like(40000, 128, seed=65, n_centres=64)
    xq = synth.clip_like(200, 128, seed=66, n_centres=64)
    idx, ref = build(xb)
    check(idx, ref, xq, k, path=2)


def test_config_a_100k_x512_1k_queries_k100(cta_group):
    """BASELINE config A in full: 100k x 512, 1000 queries, k=100 (batched tcgen05 path)."""
    xb = synth.clip_like(100_000, 512, seed=1234 + 1)
    xq = synth.clip_like(1000, 512, seed=4321)
    idx, ref = build(xb)
    check(idx, ref, xq, 100, path=0)
    assert idx.last_timing()["path"] == "mma"


def test_mma_adversarial_ties_and_duplicates(cta_group):
    xb = synth.gaussian_unit(60_000, 512, seed=0)
    xq = synth.gaussian_unit(150, 512, seed=1)
    idx, ref = build(xb)
    check(idx, ref, xq, 100, path=2)
    base = synth.gaussian_unit(50, 64, seed=9)
    xb = np.concatenate([base] * 40)
    idx, ref = build(xb)
    check(idx, ref, base[:20], 100, path=2)


def test_mma_more_query_tiles_than_cta_groups(cta_group):
    """nq beyond one launch's capacity (#CTA groups x tile) runs as several launches."""
    xb = synth.clip_like(3000, 64, seed=71, n_centres=32)
    xq = synth.clip_like(19500, 64, seed=72, n_centres=32)
    idx, ref = build(xb)
    check(idx, ref, xq, 10, path=2)


@pytest.mark.parametrize("mode", [1, 2], ids=["query_tile_resident", "row_tile_resident"])
def test_mma_two_phase_large_shard(mode, monkeypatch):
    """A shard big enough (>= 4 x 256k rows) for the two-phase search: the prefix phase seeds the
    admission thresholds of the bulk phase; results must stay exact."""
    monkeypatch.setenv("IVR_MMA_MODE", str(mode))
    xb = synth.clip_like(1_200_000, 64, seed=73, n_centres=512)
    xq = synth.clip_like(300, 64, seed=74, n_centres=512)
    idx, ref = build(xb)
    D2, I2 = check(idx, ref, xq, 100, path=2)
    monkeypatch.setenv("IVR_MMA_TWO_PHASE", "0")                 # single phase must give the same ids/scores
    D1, I1 = check(idx, ref, xq, 100, path=2)
    assert np.array_equal(I1, I2) and np.array_equal(D1, D2)


@pytest.fixture(params=["lists", "dump"])
def small_kernel(request, monkeypatch):
    """Force the small-batch (operand-swapped, row-streaming) tcgen05 kernel, in both of its result modes:
    seeded candidate lists (large shards) and materialised scores + tile maxima (small shards)."""
    monkeypatch.setenv("IVR_MMA_MODE", "3")
    monkeypatch.setenv("IVR_SMALL_DUMP_MAX_KROWS", "0" if request.param == "lists" else "100000")
    return request.param


@pytest.mark.parametrize("d", [512, 768, 1024, 384, 100, 64])
@pytest.mark.parametrize("nq", [1, 2, 5, 16, 17, 33, 64])
def test_small_kernel_dims_and_batches(d, nq, small_kernel):
    xb = synth.clip_like(30000, d, seed=81, n_centres=256)
    xq = synth.clip_like(nq, d, seed=82, n_centres=256)
    idx, ref = build(xb)
    check(idx, ref, xq, 100, path=2)
    t = idx.last_timing()
    assert t["path"] == "mma" and t["kernel"] == "search_mma_small_kernel"


@pytest.mark.parametrize("d,nq", [(512, 128), (512, 100), (768, 80), (256, 128), (64, 97)])
def test_small_kernel_widest_batches(d, nq, small_kernel):
    xb = synth.clip_like(25000, d, seed=83, n_centres=128)
    xq = synth.clip_like(nq, d, seed=84, n_centres=128)
    idx, ref = build(xb)
    check(idx, ref, xq, 100, path=2)
    assert idx.last_timing()["kernel"] == "search_mma_small_kernel"


@pytest.mark.parametrize("n", [1, 100, 127, 128, 129, 1000, 5000, 19001])
def test_small_kernel_small_indexes(n, small_kernel):
    xb = synth.gaussian_unit(n, 128, seed=85 + n)
    xq = synth.gaussian_unit(37, 128, seed=86)
    idx, ref = build(xb)
    D, I = check(idx, ref, xq, 100, path=2)
    if n < 100:
        assert (I[:, n:] == -1).all()


@pytest.mark.parametrize("k", [1, 10, 100, 128, 129, 300, 1000, 2048])
def test_small_kernel_k_values(k, small_kernel):
    xb = synth.clip_like(40000, 128, seed=87, n_centres=64)
    xq = synth.clip_like(48, 128, seed=88, n_centres=64)
    idx, ref = build(xb)
    check(idx, ref, xq, k, path=2)


def test_small_kernel_unsupported_shapes_fall_back_in_auto_mode_and_fail_loudly_when_forced(monkeypatch):
    import ivr_b200
    xb = synth.clip_like(20000, 1024, seed=89, n_centres=64)
    xq = synth.clip_like(100, 1024, seed=90, n_centres=64)
    idx, ref = build(xb)
    check(idx, ref, xq, 50, path=2)                               # 112 queries x 1024 dims do not fit beside the row ring
    assert idx.last_timing()["kernel"] == "search_mma_xres_kernel"
    monkeypatch.setenv("IVR_MMA_MODE", "3")
    with pytest.raises(ivr_b200._native.NativeError):
        idx.search(xq, 50)


@pytest.mark.parametrize("ratio", [0, 2], ids=["two_launches", "three_launches"])
def test_small_kernel_seeded_launches_match_single_launch(ratio, small_kernel, monkeypatch):
    """Shards of >= 4 tiles per SM are searched in 2-3 launches, each seeding the next one's thresholds."""
    if small_kernel == "dump":
        pytest.skip("seeding launches belong to the candidate-list mode")
    if ratio:
        monkeypatch.setenv("IVR_MMA_SMALL_RATIO", str(ratio))
    xb = synth.clip_like(300_000, 64, seed=91, n_centres=512)
    xq = synth.clip_like(24, 64, seed=92, n_centres=512)
    idx, ref = build(xb)
    D2, I2 = check(idx, ref, xq, 100, path=2)
    n_launches = idx.last_timing()["score_launches"]
    assert n_launches == (3 if ratio else 2)
    monkeypatch.setenv("IVR_MMA_TWO_PHASE", "0")
    D1, I1 = check(idx, ref, xq, 100, path=2)
    assert idx.last_timing()["score_launches"] == 1
    assert np.array_equal(I1, I2) and np.array_equal(D1, D2)


def test_small_kernel_rising_scores_force_list_compaction(small_kernel, monkeypatch):
    """Rows sorted by ASCENDING similarity to the queries: every row beats the current threshold, so the
    candidate lists fill and compact over and over -- the worst case of the fused top-k."""
    monkeypatch.setenv("IVR_MMA_TWO_PHASE", "0")
    rng = np.random.default_rng(93)
    d, n = 64, 120_000
    q = synth.gaussian_unit(4, d, seed=94)
    alpha = np.linspace(0.0, 3.0, n, dtype=np.float32)[:, None]
    xb = rng.standard_normal((n, d), dtype=np.float32) * 0.3 + alpha * q.mean(axis=0, keepdims=True) * np.sqrt(d)
    xb /= np.linalg.norm(xb, axis=1, keepdims=True)
    idx, ref = build(np.ascontiguousarray(xb, dtype=np.float32))
    check(idx, ref, q, 100, path=2)
    check(idx, ref, q[:1], 128, path=2)
    check(idx, ref, q[:2], 200, path=2)                           # k > 128: in-memory compaction of 512-entry lists


def test_small_kernel_ties_and_duplicates(small_kernel):
    base = synth.gaussian_unit(50, 64, seed=95)
    xb = np.concatenate([base] * 40)
    idx, ref = build(xb)
    check(idx, ref, base[:20], 100, path=2)
    xb = synth.gaussian_unit(60_000, 512, seed=0)
    xq = synth.gaussian_unit(60, 512, seed=1)
    idx, ref = build(xb)
    check(idx, ref, xq, 100, path=2)


def test_auto_mode_uses_the_small_kernel_for_small_batches():
    xb = synth.clip_like(50_000, 512, seed=96, n_centres=128)
    idx, ref = build(xb)
    for nq, kern in [(1, "search_stream_kernel"), (2, "search_mma_small_kernel"), (3, "search_mma_small_kernel"),
                     (16, "search_mma_small_kernel"), (64, "search_mma_small_kernel"), (300, "search_mma_kernel")]:
        xq = synth.clip_like(nq, 512, seed=97 + nq, n_centres=128)
        check(idx, ref, xq, 100, path=0)
        assert idx.last_timing()["kernel"] == kern, (nq, idx.last_timing())


def test_mma_vit_l14_768d_batch():
    """768-d (CLIP ViT-L/14, the reference's configured model) on the batched path: 128-row tiles."""
    xb = synth.clip_like(60_000, 768, seed=75, n_centres=128)
    xq = synth.clip_like(700, 768, seed=76, n_centres=128)
    idx, ref = build(xb)
    check(idx, ref, xq, 100, path=0)
    t = idx.last_timing()
    assert t["path"] == "mma" and t["kernel"] == "search_mma_xres_kernel"


def test_mma_and_stream_paths_agree():
    xb = synth.clip_like(50_000, 512, seed=67, n_centres=128)
    xq = synth.clip_like(8, 512, seed=68, n_centres=128)
    idx, ref = build(xb)
    D1, I1 = check(idx, ref, xq, 50, path=1)
    D2, I2 = check(idx, ref, xq, 50, path=2)
    assert np.abs(D1 - D2).max() < 1e-3


def test_config_a_100k_x512_k100_stream():
    """BASELINE config A shape (100k x 512, k=100), a slice of the 1k queries on the K3 path."""
    xb = synth.clip_like(100_000, 512, seed=1234 + 1)
    xq = synth.clip_like(16, 512, seed=4321)
    idx, ref = build(xb)
    check(idx, ref, xq, 100, path=1)


def test_adversarial_ties_gaussian():
    xb = synth.gaussian_unit(50_000, 512, seed=0)
    xq = synth.gaussian_unit(4, 512, seed=1)
    idx, ref = build(xb)
    check(idx, ref, xq, 100, path=1)


def test_small_and_empty_indexes():
    import ivr_b200
    idx = ivr_b200.IndexFlatIP(64)
    xq = synth.gaussian_unit(3, 64, seed=2)
    D, I = idx.search(xq, 5)                                   # empty index: all padding
    assert (I == -1).all() and (D == flat_ip.NEG_PAD).all()
    for n in (1, 3, 99, 100, 101, 257):
        xb = synth.gaussian_unit(n, 64, seed=3 + n)
        idx, ref = build(xb)
        D, I = check(idx, ref, xq, 100, path=1)
        if n < 100:
            assert (I[:, n:] == -1).all() and (D[:, n:] == flat_ip.NEG_PAD).all()
    D0, I0 = idx.search(np.zeros((0, 64), np.float32), 5)
    assert D0.shape == (0, 5) and I0.shape == (0, 5)


def test_duplicates_and_exact_ties():
    base = synth.gaussian_unit(50, 64, seed=9)
    xb = np.concatenate([base] * 40)                           # every row appears 40x -> massive exact ties
    xq = base[:3]
    idx, ref = build(xb)
    D, I = check(idx, ref, xq, 100, path=1)
    assert np.all(np.abs(D[:, :40] - 1.0) < 5e-3)


def test_reset_and_readd():
    xb = synth.clip_like(5000, 64, seed=40, n_centres=32)
    xq = synth.clip_like(2, 64, seed=41, n_centres=32)
    idx, ref = build(xb)
    idx.reset()
    assert idx.ntotal == 0
    idx.add(xb[:1234])
    ref2 = flat_ip.IndexFlatIP(64)
    ref2.add(xb[:1234])
    check(idx, ref2, xq, 10, path=1)


def test_errors():
    import ivr_b200
    from ivr_b200 import _native as nat
    idx = ivr_b200.IndexFlatIP(32)
    idx.add(synth.gaussian_unit(10, 32, seed=1))
    with pytest.raises(ValueError):
        idx.search(np.ones((1, 31), np.float32), 5)            # dimension mismatch
    with pytest.raises(ValueError):
        idx.add(np.ones((4, 33), np.float32))
    with pytest.raises(ValueError):
        idx.search(np.ones((1, 32), np.float32), 0)
    with pytest.raises(nat.NativeError) as e:
        idx.search(np.ones((1, 32), np.float32), nat.IVR_MAX_K + 1)
    assert e.value.code == nat.IVR_EUNSUPPORTED


def test_normalize_l2_matches_oracle():
    import ivr_b200
    x = (synth.gaussian_unit(1000, 100, seed=5) * 3.7).astype(np.float32)
    x[17] = 0
    want = x.copy()
    flat_ip.normalize_L2(want)
    ivr_b200.normalize_L2(x)
    assert np.allclose(x, want, atol=1e-6) and not x[17].any()


def test_device_tensor_search_and_id_offset():
    import torch
    import ivr_b200
    xb = synth.clip_like(8000, 512, seed=50, n_centres=64)
    xq = synth.clip_like(3, 512, seed=51, n_centres=64)
    idx = ivr_b200.IndexFlatIP(512)
    idx.add(torch.from_numpy(xb).cuda())                       # device-side add
    ref = flat_ip.IndexFlatIP(512)
    ref.add(xb)
    D, I = idx.search_tensor(torch.from_numpy(xq).cuda(), 20, id_offset=1_000_000_000_000)
    torch.cuda.synchronize()
    Dr, Ir = ref.search(xq, 20)
    bad = comparator.compare_topk(D.cpu().numpy(), I.cpu().numpy() - 1_000_000_000_000, Dr, Ir,
                                  lambda ids: ref.scores_of(xq, ids), TOL)
    assert not bad, bad


def test_topk_merge_kernel_matches_oracle():
    import ctypes
    import torch
    from ivr_b200 import _native as nat
    rng = np.random.default_rng(0)
    for n_parts, nq, k in ((8, 33, 100), (2, 5, 7), (130, 3, 20), (3, 4, 1000)):
        D = np.sort(rng.standard_normal((n_parts, nq, k)).astype(np.float32), axis=2)[:, :, ::-1].copy()
        I = np.stack([np.stack([rng.permutation(10 * k)[:k] for _ in range(nq)]) + p * 10_000_000
                      for p in range(n_parts)]).astype(np.int64)
        I[0, 0, k // 2:] = -1                                   # a short (padded) shard list
        D[0, 0, k // 2:] = flat_ip.NEG_PAD
        D[1 % n_parts, 1 % nq, 0] = D[0, 1 % nq, 0]             # an exact cross-shard tie
        Dm, Im = flat_ip.merge_shard_results(list(D), list(I), k)
        Dd, Id = torch.from_numpy(D).cuda(), torch.from_numpy(I).cuda()
        Do = torch.empty((nq, k), dtype=torch.float32, device="cuda")
        Io = torch.empty((nq, k), dtype=torch.int64, device="cuda")
        nat.check(nat.lib.ivr_topk_merge_device(0, Dd.data_ptr(), Id.data_ptr(), n_parts, nq, k,
                                                Do.data_ptr(), Io.data_ptr(),
                                                torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        assert np.array_equal(Io.cpu().numpy(), Im), (n_parts, nq, k)   # integer/bit exact
        assert np.array_equal(Do.cpu().numpy(), Dm)


def test_packed_key_search_and_key_merge_match_the_unpacked_path():
    """The cross-shard exchange format: search_keys_tensor == pack(search_tensor) bit for bit on every kernel family,
    and ivr_topk_merge_keys_device == the (D, I) merge == the oracle merge."""
    import torch
    import ivr_b200
    from ivr_b200 import _native as nat
    xb = synth.clip_like(50_000, 512, seed=91, n_centres=64)
    idx = ivr_b200.IndexFlatIP(512)
    idx.add(xb)
    for nq, k, off in ((1, 100, 0), (16, 100, 123_456), (300, 100, 4_000_000_000), (5, 7, 17), (3, 300, 0)):
        q = torch.from_numpy(synth.clip_like(nq, 512, seed=92 + nq, n_centres=64)).cuda()
        D, I = idx.search_tensor(q, k, id_offset=off)
        keys = idx.search_keys_tensor(q, k, id_offset=off)
        torch.cuda.synchronize()
        want = flat_ip.pack_keys(D.cpu().numpy(), I.cpu().numpy())
        assert np.array_equal(keys.cpu().numpy().view(np.uint64), want), (nq, k, off)
    with pytest.raises(nat.NativeError):                            # global ids must stay below 2^32
        idx.search_keys_tensor(q, 10, id_offset=(1 << 32) - 10)
    # k > ntotal: padding keys are 0
    small = ivr_b200.IndexFlatIP(64)
    small.add(synth.gaussian_unit(5, 64, seed=1))
    keys = small.search_keys_tensor(torch.from_numpy(synth.gaussian_unit(2, 64, seed=2)).cuda(), 8)
    assert (keys[:, 5:] == 0).all() and (keys[:, :5] != 0).all()
    empty = ivr_b200.IndexFlatIP(64)
    assert (empty.search_keys_tensor(torch.zeros(2, 64, device="cuda"), 4) == 0).all()
    # merge of gathered keys
    rng = np.random.default_rng(3)
    for n_parts, nq, k in ((8, 33, 100), (2, 5, 7), (64, 3, 20), (3, 4, 1000), (64, 2, 300), (40, 2, 100), (8, 1100, 100)):
        D = np.sort(rng.standard_normal((n_parts, nq, k)).astype(np.float32), axis=2)[:, :, ::-1].copy()
        I = np.stack([np.stack([rng.permutation(10 * k)[:k] for _ in range(nq)]) + p * 10_000_000
                      for p in range(n_parts)]).astype(np.int64)
        I[0, 0, k // 2:] = -1
        D[0, 0, k // 2:] = flat_ip.NEG_PAD
        D[1 % n_parts, 1 % nq, 0] = D[0, 1 % nq, 0]
        Dm, Im = flat_ip.merge_shard_results(list(D), list(I), k)
        kd = torch.from_numpy(flat_ip.pack_keys(D, I).view(np.int64)).cuda()
        Do = torch.empty((nq, k), dtype=torch.float32, device="cuda")
        Io = torch.empty((nq, k), dtype=torch.int64, device="cuda")
        nat.check(nat.lib.ivr_topk_merge_keys_device(0, kd.data_ptr(), n_parts, nq, k, Do.data_ptr(), Io.data_ptr(),
                                                     torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        assert np.array_equal(Io.cpu().numpy(), Im) and np.array_equal(Do.cpu().numpy(), Dm), (n_parts, nq, k)
    with pytest.raises(nat.NativeError):                            # more than one merge level would need scratch
        nat.check(nat.lib.ivr_topk_merge_keys_device(0, kd.data_ptr(), 65, 1, 1, Do.data_ptr(), Io.data_ptr(), None))


@pytest.mark.parametrize("d", [1280, 2048])
@pytest.mark.parametrize("nq", [1, 2, 3, 16, 100])
def test_dims_beyond_1024_pick_a_kernel_that_fits(d, nq):
    """Only the small-batch tcgen05 kernel and the streaming kernel exist beyond 1024 dims: the automatic choice must
    land on one of them (nq=2..~50 at 1280 dims: small-batch; larger batches: streaming), never on 'unsupported'."""
    import ivr_b200
    xb = synth.clip_like(6000, d, seed=93, n_centres=32)
    xq = synth.clip_like(nq, d, seed=94, n_centres=32)
    idx, ref = build(xb)
    check(idx, ref, xq, 20, path=0)
    tile_fits = ((nq + 15) // 16 * 16) * ((d + 63) // 64 * 64) * 2 <= 128 * 1024     # resident query tile <= 128 KB
    small_fits = 2 <= nq and tile_fits                               # one query streams on the SIMT kernel
    t = idx.last_timing()
    assert t["kernel"] == ("search_mma_small_kernel" if small_fits else "search_stream_kernel"), t
    if tile_fits:
        check(idx, ref, xq, 20, path=2)                              # forcing the tcgen05 path works too
        assert idx.last_timing()["kernel"] == "search_mma_small_kernel"
    else:
        idx.search_path = 2
        with pytest.raises(ivr_b200._native.NativeError):
            idx.search(xq, 20)


def test_device_add_then_host_add_that_regrows_keeps_every_row():
    """A device-side add queues its fp32->fp16 conversion on the caller's stream; a following host add that regrows the
    row block must copy AFTER that conversion has run (it runs on the handle's own stream)."""
    import torch
    import ivr_b200
    d = 256
    xa = synth.clip_like(200_000, d, seed=95, n_centres=64)
    xb2 = synth.clip_like(150_000, d, seed=96, n_centres=64)
    side = torch.cuda.Stream()
    idx = ivr_b200.IndexFlatIP(d)
    idx.reserve(len(xa))                                            # exact: the next add must regrow
    xa_dev = torch.from_numpy(xa).cuda()
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)                              # ~0.1 s: the conversion is still pending at the host add
        idx.add(xa_dev)
    idx.add(xb2)
    ref = flat_ip.IndexFlatIP(d)
    ref.add(np.concatenate([xa, xb2]))
    xq = np.concatenate([xa[:3], xb2[-3:]])
    check(idx, ref, xq, 10, path=0)


def test_wrappers_against_reference_golden(search_golden):
    """The reference's own wrapper outputs (golden) vs. our wrappers on the CUDA index."""
    import ivr_b200
    sg = search_golden
    u = ivr_b200.UnifiedIndex()
    u.build_from_embeddings(sg["xb"], sg["meta"])
    ref = flat_ip.IndexFlatIP(sg["xb"].shape[1])
    ref.add(sg["xb"])
    for key, want in sg["results"]["search_vectors"].items():
        if key == "k20_q0_even":
            got = u.search_vectors(sg["xq"][0], k=20, filter_func=lambda m: m["frame_id"] % 2 == 0)
            assert all(g["metadata"]["frame_id"] % 2 == 0 for g in got) and abs(len(got) - len(want)) <= 1
            continue
        k, q = key.split("_")
        k, qi = int(k[1:]), int(q[1:])
        got = u.search_vectors(sg["xq"][qi], k=k)
        assert len(got) == len(want)
        assert [g["rank"] for g in got] == [w[0] for w in want]           # 0-based, dense
        D = np.array([[1.0 - g["similarity_score"] for g in got]], np.float32)
        I = np.array([[g["index"] for g in got]], np.int64)
        Dr = np.array([[1.0 - w[1] for w in want]], np.float32)
        Ir = np.array([[w[2] for w in want]], np.int64)
        bad = comparator.compare_topk(D, I, Dr, Ir, lambda ids: ref.scores_of(sg["xq"][qi:qi + 1], ids), TOL)
        assert not bad, (key, bad)
        for g in got:
            assert g["metadata"] is sg["meta"][g["index"]]
    assert u.faiss_index.last_timing()["path"] in ("stream", "mma")    # it really ran on the device
    b = ivr_b200.UnifiedBuilderIntegration(system=None)
    b.unified_index = u
    for key, want in sg["results"]["search_unified_fast"].items():
        got = b.search_unified_fast(sg["xq"][1], k=30, similarity_threshold=float(key[3:]))
        assert abs(len(got) - len(want)) <= 1                               # threshold on 1-ip, 1e-3 band
        for g, w in zip(got, want):
            assert abs(g["similarity_score"] - w[1]) < 2 * TOL
        for g in got:
            assert g["similarity_score"] >= float(key[3:]) and g["temporal_context"] == []
            assert type(g["metadata"]).__name__ == "KeyframeMetadata"
    ids, scores, meta = ivr_b200.RAGBuilder().build_index(sg["xb"], sg["meta"]).search(sg["xq"], top_k=5)
    assert ids.shape == (len(sg["xq"]), 5) and np.all(np.diff(scores, axis=1) <= 0)


def test_batched_front_end_on_gpu(search_golden):
    """search_vectors_batch on the CUDA index: every query's hit list against the oracle (the batch runs on a
    tcgen05 kernel with fp16 queries, the single-query wrapper on the streaming kernel: ties may differ)."""
    import ivr_b200
    sg = search_golden
    u = ivr_b200.UnifiedIndex()
    u.build_from_embeddings(sg["xb"], sg["meta"])
    xbn = sg["xb"].copy()
    flat_ip.normalize_L2(xbn)                          # build_from_embeddings normalises (unified_index.py:1776)
    ref = flat_ip.IndexFlatIP(xbn.shape[1])
    ref.add(xbn)
    k = 25
    batch = u.search_vectors_batch(sg["xq"], k=k)
    assert len(batch) == len(sg["xq"])
    Dr, Ir = ref.search(sg["xq"], k)
    D = np.array([[1.0 - g["similarity_score"] for g in got] for got in batch], np.float32)
    I = np.array([[g["index"] for g in got] for got in batch], np.int64)
    bad = comparator.compare_topk(D, I, Dr, Ir, lambda ids: ref.scores_of(sg["xq"], ids), TOL)
    assert not bad, bad[:5]
    for got in batch:
        assert [g["rank"] for g in got] == list(range(k))
        assert all(g["metadata"] is sg["meta"][g["index"]] for g in got)
    b = ivr_b200.UnifiedBuilderIntegration(system=None)
    b.unified_index = u
    out = b.search_unified_fast_batch(sg["xq"], k=k, similarity_threshold=0.0)
    assert [len(o) for o in out] == [sum(g["similarity_score"] >= 0.0 for g in got) for got in batch]


def test_faiss_retriever_on_gpu(search_golden):
    import ivr_b200
    sg = search_golden
    raw = (sg["xb"] * np.float32(2.5)).astype(np.float32)
    kms = [ivr_b200.KeyframeMetadata(folder_name=m["folder_name"], image_name=m["image_name"],
                                     frame_id=m["frame_id"], file_path=m["file_path"],
                                     clip_features=(raw[i] if i % 7 else None))
           for i, m in enumerate(sg["meta"])]
    fr = ivr_b200.FAISSRetriever()
    fr.build_index(raw, kms, validate_consistency=False)
    assert fr.index.ntotal == sg["results"]["ntotal"]
    out = fr.search(sg["xq"][:3] * np.float32(1.7), k=12)
    want = sg["results"]["faiss_retriever_search"]
    assert len(out) == len(want) == 36
    assert [r.rank for r in out] == [w[3] for w in want]
    # same hit SETS per query (order inside a 1e-3 band may differ), identical re-scored cosines
    for q in range(3):
        g = {(r.metadata.folder_name, r.metadata.image_name): r.similarity_score for r in out[q * 12:(q + 1) * 12]}
        w = {(x[0], x[1]): x[2] for x in want[q * 12:(q + 1) * 12]}
        common = set(g) & set(w)
        assert len(common) >= 11
        for key in common:
            assert abs(g[key] - w[key]) < 1e-6
    one = fr.search(sg["xq"][4], k=5)
    assert [(r.metadata.folder_name, r.metadata.image_name, r.rank) for r in one] == \
        [(w[0], w[1], w[3]) for w in sg["results"]["faiss_retriever_search_1d"]]
    by_id = sg["results"]["faiss_retriever_search_by_id"]
    hits = fr.search_by_id(by_id["key"], k=7)
    assert [(r.metadata.folder_name, r.metadata.image_name) for r in hits][:1] == [tuple(by_id["hits"][0][:2])]
    assert len(hits) == len(by_id["hits"])


def test_similarity_relationships_vs_oracle():
    """MetadataManager._build_similarity_relationships (core.py:3493-3531): per-folder top-10 > 0.7."""
    import ivr_b200
    rng = np.random.default_rng(5)
    all_meta, all_feat = {}, {}
    for f, n in enumerate((1, 2, 37, 400)):
        folder = f"L{f:02d}_V001"
        x = synth.clip_like(n, 128, seed=80 + f, n_centres=6) * np.float32(rng.uniform(0.5, 3.0))
        metas = [ivr_b200.KeyframeMetadata(folder_name=folder, image_name=f"{i:04d}", frame_id=i,
                                           file_path=f"{folder}/{i:04d}.jpg",
                                           clip_features=(x[i] if (i % 11) != 5 else None)) for i in range(n)]
        all_meta[folder] = metas
        keep = [i for i in range(n) if (i % 11) != 5]
        all_feat[folder] = ([metas[i].get_unique_key() for i in keep], x[keep])
    got = ivr_b200.build_similarity_relationships(all_meta)
    want, sims = flat_ip.similarity_relationships(all_feat)
    assert set(got) == set(want)
    for key, wl in want.items():
        gl = got[key]
        s = sims[key]
        assert len(gl) <= 10 and len(set(gl)) == len(gl)
        ranked = sorted((v for o, v in s.items()), reverse=True)
        cut = max(0.7, ranked[min(10, len(ranked) - 1)])          # admission level: threshold or the 11th best
        for o in gl:                                                # nothing clearly below the admission level
            assert s[o] > cut - 1e-3, (key, o, s[o], cut)
        for o in wl:                                                # nothing clearly above it is missing
            if s[o] > cut + 1e-3:
                assert o in gl or o == key, (key, o, s[o], cut)


def test_similarity_relationships_vs_reference_golden(relationships_golden):
    """The reference's own graph (golden) vs. the CUDA path: the GPU supplies candidates (fp16 rows), the decision
    is taken on float32 cosines like the reference's -> IDENTICAL neighbour lists, order included."""
    import ivr_b200
    rg = relationships_golden
    all_meta = {}
    for folder, x in rg["features"].items():
        all_meta[folder] = [ivr_b200.KeyframeMetadata(folder_name=folder, image_name=f"{i:04d}", frame_id=i,
                                                     file_path=f"keyframes/{folder}/{i:04d}.jpg",
                                                     clip_features=(x[i] if (i % 11) != 5 else None))
                            for i in range(len(x))]
    got = ivr_b200.build_similarity_relationships(all_meta)
    want = rg["graph"]
    assert set(got) == set(want)
    diff = [key for key in want if got[key] != want[key]]
    assert not diff, (len(diff), diff[:5], [(got[k], want[k]) for k in diff[:2]])
    assert all(key not in got[key] for key in got)               # self is dropped by id, never listed


def test_randomised_shapes_auto_path():
    """Seeded random sweep over (rows, dim, queries, k) through the AUTO path: whichever kernel the
    dispatcher picks (streaming, small-batch, query-/row-tile-resident) must match the oracle."""
    rng = np.random.default_rng(2026)
    seen = set()
    for case in range(36):
        n = int(rng.choice([1, 7, 129, 1000, 5000, 20011, 60000]))
        d = int(rng.choice([1, 3, 64, 65, 100, 128, 257, 384, 512, 513, 768, 1000, 1024]))
        nq = int(rng.choice([1, 2, 3, 15, 16, 17, 63, 64, 65, 127, 128, 129, 255, 257, 600]))
        k = int(rng.choice([1, 2, 10, 100, 128, 129, 200]))
        xb = synth.clip_like(n, d, seed=1000 + case, n_centres=min(64, max(1, n)))
        xq = synth.clip_like(nq, d, seed=2000 + case, n_centres=min(64, max(1, n)))
        idx, ref = build(xb)
        check(idx, ref, xq, k, path=0)
        seen.add(idx.last_timing()["kernel"])
        idx.close()
    assert {"search_stream_kernel", "search_mma_small_kernel", "search_mma_kernel"} <= seen, seen


def _device_clip_like(n, d, seed, chunk=500_000):
    """Seeded CLIP-like rows generated on the device in chunks (SURVEY.md 8d), yielded as float32 CUDA tensors."""
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    cen = torch.nn.functional.normalize(torch.randn(1024, d, generator=g, device="cuda"), dim=1)
    for s in range(0, n, chunk):
        m = min(chunk, n - s)
        z = torch.randint(0, 1024, (m,), generator=g, device="cuda")
        yield torch.nn.functional.normalize(cen[z] + (0.5 / d ** 0.5) * torch.randn(m, d, generator=g, device="cuda"), dim=1)


@pytest.mark.parametrize("n,d,nqs", [(10_000_000, 768, (1, 16)), (12_500_000, 512, (4096,)), (100_000_000, 512, (4096,))],
                         ids=["config_c_10Mx768", "config_d_shard_12M5x512", "config_d_one_gpu_100Mx512"])
def test_full_size_configs_against_exact_scan(n, d, nqs):
    """BASELINE configs C and D (per-GPU shard) at FULL size: the oracle cannot run here in seconds, so up to 64
    queries are checked against an exact fp32 scan (torch, on the device) of the same rows -- every kernel's
    answer must contain exactly the rows above the k-th exact score, up to the 1e-3 tie band."""
    import torch
    import ivr_b200
    k, n_chk = 100, min(64, max(nqs))
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.cuda.empty_cache()
    if torch.cuda.mem_get_info()[0] < n * d * 2 + (16 << 30):
        pytest.skip("not enough free HBM for this configuration")
    idx = ivr_b200.IndexFlatIP(d)
    idx.reserve(n)
    q_all = next(_device_clip_like(max(nqs), d, seed=4321))
    best_s = torch.full((n_chk, k), -2.0, device="cuda")
    best_i = torch.full((n_chk, k), -1, dtype=torch.int64, device="cuda")
    off = 0
    for x in _device_clip_like(n, d, seed=99):
        idx.add(x)
        s = q_all[:n_chk] @ x.T                                             # exact fp32 scores of the check queries
        ts, ti = torch.topk(s, k, dim=1)
        cat_s, cat_i = torch.cat([best_s, ts], 1), torch.cat([best_i, ti + off], 1)
        best_s, sel = torch.topk(cat_s, k, dim=1)
        best_i = torch.gather(cat_i, 1, sel)
        off += x.shape[0]
    Dr, Ir = best_s.cpu().numpy(), best_i.cpu().numpy()
    for nq in nqs:
        D, I = idx.search_tensor(q_all[:nq].contiguous(), k)
        Dn, In = D[:n_chk].cpu().numpy(), I[:n_chk].cpu().numpy()
        for q in range(min(n_chk, nq)):
            s_k = Dr[q, -1]
            must = Ir[q][Dr[q] > s_k + TOL]
            assert np.isin(must, In[q]).all(), (nq, q, "misses rows above the k-th exact score + tol")
            exact = dict(zip(Ir[q].tolist(), Dr[q].tolist()))
            for i_, d_ in zip(In[q].tolist(), Dn[q].tolist()):
                if i_ in exact:
                    assert abs(exact[i_] - d_) <= TOL
                else:
                    assert s_k - TOL <= d_ <= s_k + 2 * TOL, (nq, q, i_, d_, s_k)     # only near-k ties may differ
            assert np.all(np.diff(Dn[q]) <= 0) and len(set(In[q].tolist())) == k
    idx.close()


def test_row_tile_resident_large_k_runs_in_several_query_batches(monkeypatch):
    """k = 2048 makes every candidate list 4096 entries: the row-tile-resident kernel then takes at most 1536
    queries per launch (8 GiB list budget), so 1700 queries run as two batches."""
    monkeypatch.setenv("IVR_MMA_MODE", "2")
    xb = synth.clip_like(6000, 64, seed=111, n_centres=32)
    xq = synth.clip_like(1700, 64, seed=112, n_centres=32)
    idx, ref = build(xb)
    check(idx, ref, xq, 2048, path=2)
    assert idx.last_timing()["kernel"] == "search_mma_xres_kernel"


def test_faiss_layout_serialisation_round_trip_through_the_device(tmp_path):
    """faiss_compat.serialize_index / deserialize_index / write_index / read_index in the FAISS IndexFlatIP layout
    ('IxFI' header + float32 payload): a hand-built buffer loads and searches like the rows it holds, and a round trip
    through the device reproduces the fp16-rounded rows bit for bit."""
    import struct
    import ivr_b200
    fc = ivr_b200.faiss_compat
    n, d = 70_000, 96                                             # d not a multiple of 64: padded columns are dropped again
    xb = synth.clip_like(n, d, seed=97, n_centres=64)
    xq = synth.clip_like(5, d, seed=98, n_centres=64)
    buf = (b"IxFI" + struct.pack("<iqqq?i", d, n, 1 << 20, 1 << 20, True, 0) + struct.pack("<Q", n * d) + xb.tobytes())
    idx = fc.deserialize_index(np.frombuffer(buf, np.uint8))      # what unified_index.py:1182 passes
    ref = flat_ip.IndexFlatIP(d)
    ref.add(xb)
    assert idx.ntotal == n and idx.d == d
    check(idx, ref, xq, 50)
    rows16 = xb.astype(np.float16).astype(np.float32)
    assert np.array_equal(idx.reconstruct_n(0, n), rows16)
    assert np.array_equal(idx.reconstruct_n(n - 7, 7), rows16[-7:])
    out = fc.serialize_index(idx)
    assert out.dtype == np.uint8 and bytes(out[:45]) == buf[:45]
    assert np.array_equal(out[45:].view(np.float32).reshape(n, d), rows16)
    again = fc.deserialize_index(out)
    assert np.array_equal(fc.serialize_index(again), out)         # idempotent after the first rounding
    path = tmp_path / "index.faiss"
    fc.write_index(idx, str(path))
    assert path.read_bytes() == out.tobytes()
    back = fc.read_index(str(path), fc.IO_FLAG_MMAP)
    assert back.ntotal == n
    D1, I1 = idx.search(xq, 20)
    D2, I2 = back.search(xq, 20)
    assert np.array_equal(I1, I2) and np.array_equal(D1, D2)
    empty = fc.deserialize_index(fc.serialize_index(fc.IndexFlatIP(d)))
    assert empty.ntotal == 0 and empty.d == d
    with pytest.raises(NotImplementedError):
        fc.deserialize_index(np.frombuffer(b"IxF2" + buf[4:], np.uint8))
    with pytest.raises(ValueError):
        fc.deserialize_index(np.frombuffer(buf[:-8], np.uint8))
    with pytest.raises(ivr_b200._native.NativeError):
        idx.reconstruct_n(n - 1, 5)


@pytest.mark.parametrize("layout", ["faiss_index dataset", "index/faiss (old, LZ4-framed)", "embeddings only"])
def test_load_unified_index_from_an_rvdb_container(tmp_path, layout):
    """UnifiedIndex.load_unified_index on a .rvdb-shaped file (tests/hdf5_fixture.py builds it from the published HDF5 /
    LZF / LZ4 formats; metadata framed by pyarrow's real LZ4 codec): the index arrives through deserialize_index
    (unified_index.py:1182 / 1185-1188) or is built from the embedding chunks (1755-1793), and searches like an index
    built from the same arrays in memory."""
    pytest.importorskip("pyarrow")
    import os
    import struct
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from test_host_logic import _rvdb_fixture
    import ivr_b200
    n, d = 3000, 96
    emb = (synth.clip_like(n, d, seed=99, n_centres=32) * np.float32(1.7)).astype(np.float32)     # raw, un-normalised
    meta = [{"file_path": f"keyframes/L01_V001/{i:04d}.jpg", "folder_name": "L01_V001", "image_name": f"{i:04d}.jpg",
             "frame_id": i, "file_hash": f"{i:016x}", "file_size": 1000 + i} for i in range(n)]
    unit = emb.copy()
    flat_ip.normalize_L2(unit)
    faiss_bytes = (b"IxFI" + struct.pack("<iqqq?i", d, n, 1 << 20, 1 << 20, True, 0) + struct.pack("<Q", n * d) + unit.tobytes())
    path = str(tmp_path / "unified.rvdb")
    _rvdb_fixture(path, emb, meta, with_faiss_bytes=None if layout == "embeddings only" else faiss_bytes,
                  old_layout=layout.startswith("index/faiss"))
    u = ivr_b200.UnifiedIndex()
    info = u.load_unified_index(path)
    assert u.is_loaded and u.faiss_index.ntotal == n and info["index_info"]["processed_files"] == n
    assert u.metadata_list == meta and u.vectors is None
    mem = ivr_b200.UnifiedIndex()
    mem.build_from_embeddings(emb, meta)
    xq = synth.clip_like(4, d, seed=100, n_centres=32)
    for q in xq:
        a, b = u.search_vectors(q, k=20), mem.search_vectors(q, k=20)
        assert [h["index"] for h in a] == [h["index"] for h in b]
        np.testing.assert_allclose([h["similarity_score"] for h in a], [h["similarity_score"] for h in b], atol=1e-6)
        assert all(h["metadata"] is u.metadata_list[h["index"]] for h in a)
    v = ivr_b200.load_optimized_index(path)
    assert v.faiss_index.ntotal == n
    w = ivr_b200.UnifiedIndex()
    w.load_unified_index(path, load_vectors=True)
    assert np.array_equal(w.vectors, emb)


def test_small_kernel_dump_mode_clustered_rows_overflow_the_pool_and_stay_exact(monkeypatch):
    """Dump mode bounds the k-th best by the k-th largest TILE maximum.  5000 near-identical rows packed into ~40
    consecutive tiles make that bound useless (every one of them passes it): the candidate pool overflows and the
    kernel falls back to the exact radix select -- slow, but the result must still be exact."""
    monkeypatch.setenv("IVR_MMA_MODE", "3")
    rng = np.random.default_rng(7)
    d, n = 512, 40_000                                             # 3 queries x 512 dims: the dump-mode shape rule holds
    xb = synth.gaussian_unit(n, d, seed=70)
    q = synth.gaussian_unit(3, d, seed=71)
    hot = q[0] + 0.02 * rng.standard_normal((5000, d)).astype(np.float32)      # a burst of near-duplicates of query 0
    xb[10_000:15_000] = hot / np.linalg.norm(hot, axis=1, keepdims=True)
    idx, ref = build(np.ascontiguousarray(xb, dtype=np.float32))
    check(idx, ref, q, 100, path=2)
    check(idx, ref, q, 1000, path=2)
    assert idx.last_timing()["kernel"] == "search_mma_small_kernel"


@pytest.mark.parametrize("nq,path", [(1, 1), (3, 0), (16, 0), (100, 0), (300, 2)])
def test_search_window_scores_only_its_rows_and_keeps_stored_row_ids(nq, path):
    """ivr_index_set_window (elastic shard boundaries): a windowed search equals the oracle over that row range,
    ids are stored rows + id_offset, and two adjacent windows merged equal the whole index -- on every kernel path."""
    import torch
    n, d, k = 30000, 128, 50
    xb = synth.clip_like(n, d, seed=61, n_centres=64)
    xq = synth.clip_like(nq, d, seed=62, n_centres=64)
    idx, ref = build(xb)
    idx.search_path = path
    cut = 12345
    parts = []
    for first, count in ((0, cut), (cut, n - cut)):
        sub = flat_ip.IndexFlatIP(d)
        sub.add(xb[first:first + count])
        idx.set_window(first, count)
        D, I = idx.search(xq, k)
        Dr, Ir = sub.search(xq, k)
        bad = comparator.compare_topk(D, I - first, Dr, Ir, lambda ids: sub.scores_of(xq, ids), TOL)
        assert not bad, "\n".join(bad[:5])
        assert I.min() >= first and I.max() < first + count
        Dt, It = idx.search_tensor(torch.from_numpy(xq).cuda(), k, id_offset=1000)
        assert np.array_equal(It.cpu().numpy(), I + 1000)
        parts.append((D, I))
    Dm, Im = flat_ip.merge_shard_results([p[0] for p in parts], [p[1] for p in parts], k)
    Dr, Ir = ref.search(xq, k)
    bad = comparator.compare_topk(Dm, Im, Dr, Ir, lambda ids: ref.scores_of(xq, ids), TOL)
    assert not bad, "\n".join(bad[:5])
    idx.set_window(5, 7)                              # fewer rows than k: padded like a 7-row index
    D, I = idx.search(xq, k)
    assert np.all(I[:, 7:] == -1) and np.all((I[:, :7] >= 5) & (I[:, :7] < 12))
    idx.set_window(0, 0)                              # empty window: all padding
    D, I = idx.search(xq, k)
    assert np.all(I == -1)
    idx.set_window(n - 10, 11)                        # reaches beyond the index
    with pytest.raises(Exception, match="window"):
        idx.search(xq, k)
    idx.set_window()                                  # cleared: the whole index again
    check(idx, ref, xq, k, path=path)
