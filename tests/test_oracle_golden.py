"""CPU: the oracle restatements against the golden vectors produced by the reference."""
import numpy as np
import pytest

from oracle import comparator, dedup as od, flat_ip, synth

CFG = dict(enable_similarity_filtering=True, similarity_threshold=0.95, min_frame_distance=1,
           similarity_window_size=5, use_advanced_similarity_filtering=False)
VARIANTS = {
    "adv_w8_t095": dict(use_advanced_similarity_filtering=True, similarity_window_size=8),
    "adv_w5_t095": dict(use_advanced_similarity_filtering=True, similarity_window_size=5),
    "adv_w3_t090": dict(use_advanced_similarity_filtering=True, similarity_window_size=3,
                        similarity_threshold=0.90),
    "adv_w1_t095": dict(use_advanced_similarity_filtering=True, similarity_window_size=1),
    "basic_m1_t095": dict(),
    "basic_m2_t095": dict(min_frame_distance=2),
    "basic_m1_t098": dict(similarity_threshold=0.98),
    "disabled": dict(enable_similarity_filtering=False),
}


def cfg(**kw):
    c = dict(CFG)
    c.update(kw)
    return c


@pytest.mark.parametrize("name", ["dedup_d64", "dedup_d512"])
def test_dedup_oracle_matches_reference(dedup_golden, name):
    g = dedup_golden[name]
    x = g["x"]
    emb = [r for r in x]
    n = len(emb)
    sims = od.calculate_similarities(emb)
    assert np.array_equal(np.asarray(sims, np.float32), g["sims"])          # bit-exact
    for thr, tag in ((0.75, "t075"), (0.3, "t030")):
        tp = od.detect_scene_transitions(sims, thr)
        assert np.array_equal(np.asarray(tp, np.int64), g[f"transitions_{tag}"])
        for ml in (1, 2, 5):
            sc = od.group_into_scenes(tp, n, ml)
            assert np.array_equal(np.asarray(sc, np.int64).reshape(-1, 2), g[f"scenes_{tag}_m{ml}"])
    scenes = od.group_into_scenes(od.detect_scene_transitions(sims, 0.75), n, 2)
    for tag, kw in VARIANTS.items():
        _, rows, stats = od.apply_similarity_filtering_to_scenes(emb, list(range(n)), scenes, cfg(**kw))
        assert np.array_equal(np.asarray(rows, np.int64), g[f"kept_{tag}"]), tag
        assert [stats["original"], stats["filtered"], stats["removed"]] == g[f"stats_{tag}"].tolist()
    whole = list(range(n))
    assert od.filter_similar_frames_advanced(emb, whole, cfg(**VARIANTS["adv_w8_t095"])) == g["kept_whole_adv_w8"].tolist()
    assert od.filter_similar_frames_in_scene(emb, whole, cfg()) == g["kept_whole_basic"].tolist()
    emb_none = list(emb[:40])
    for i in (0, 7, 8, 39):
        emb_none[i] = None
    assert np.array_equal(np.asarray(od.calculate_similarities(emb_none), np.float32), g["sims_none40"])


@pytest.mark.parametrize("name", ["dedup_d64", "dedup_d512"])
def test_dedup_vectorised_oracle_matches_reference(dedup_golden, name):
    """The fast (vectorised) oracle used at large sizes agrees with the reference outputs."""
    g = dedup_golden[name]
    x = g["x"]
    n = len(x)
    cosv = od.consecutive_cosines_fast(x)
    assert np.allclose(cosv, g["sims"], atol=2e-6)
    scenes = od.scenes_from_cosines(cosv, n, 0.75, 2)
    assert np.array_equal(np.asarray(scenes, np.int64).reshape(-1, 2), g["scenes_t075_m2"])
    for tag, w, thr in (("adv_w8_t095", 8, 0.95), ("adv_w5_t095", 5, 0.95), ("adv_w3_t090", 3, 0.90),
                        ("adv_w1_t095", 1, 0.95)):
        keep = od.window_keep_mask(x, scenes, w, thr)
        assert np.array_equal(np.nonzero(keep)[0], g[f"kept_{tag}"]), tag
    assert od.guard_band_ok(x, 8, (0.95, 0.75, 0.98, 0.9, 0.3))


def test_flat_ip_against_torch_topk():
    import torch
    xb = synth.clip_like(5000, 64, seed=1, n_centres=64)
    xq = synth.clip_like(17, 64, seed=2, n_centres=64)
    idx = flat_ip.IndexFlatIP(64)
    idx.add(xb[:3000])
    idx.add(xb[3000:])
    assert idx.ntotal == 5000
    D, I = idx.search(xq, 100, db_block=1024)                       # exercises the running merge
    tv, ti = torch.topk(torch.from_numpy(xq) @ torch.from_numpy(xb).T, 100, dim=1)
    assert not comparator.compare_topk(D, I, tv.numpy(), ti.numpy(), lambda ids: idx.scores_of(xq, ids), tol=1e-5)
    assert np.all(np.diff(D, axis=1) <= 0)


def test_flat_ip_padding_and_ties():
    idx = flat_ip.IndexFlatIP(8)
    D, I = idx.search(np.ones((2, 8), np.float32), 3)
    assert (I == -1).all() and (D == flat_ip.NEG_PAD).all()
    x = np.zeros((5, 8), np.float32)
    x[:, 0] = [1, 2, 2, 2, 0]
    idx.add(x)
    D, I = idx.search(np.eye(1, 8, dtype=np.float32), 7)
    assert I[0].tolist() == [1, 2, 3, 0, 4, -1, -1]                  # ties -> lower id first
    assert D[0, 5] == flat_ip.NEG_PAD
    D2, I2 = idx.search(np.eye(1, 8, dtype=np.float32), 2)
    assert I2[0].tolist() == [1, 2]


def test_normalize_l2_contract():
    x = np.array([[3, 4, 0], [0, 0, 0], [1, 1, 1]], np.float32)
    flat_ip.normalize_L2(x)
    assert np.allclose(x[0], [0.6, 0.8, 0]) and not x[1].any()
    assert np.allclose(np.linalg.norm(x[2]), 1, atol=1e-6)
    with pytest.raises(ValueError):
        flat_ip.normalize_and_validate(np.array([np.nan, 1.0]))


def test_merge_shard_results_oracle():
    xb = synth.gaussian_unit(3000, 32, seed=3)
    xq = synth.gaussian_unit(5, 32, seed=4)
    full = flat_ip.IndexFlatIP(32)
    full.add(xb)
    D, I = full.search(xq, 50)
    Ds, Is = [], []
    for a, b in ((0, 700), (700, 2900), (2900, 3000)):
        s = flat_ip.IndexFlatIP(32)
        s.add(xb[a:b])
        d, i = s.search(xq, 50)
        Ds.append(d)
        Is.append(np.where(i >= 0, i + a, -1))
    Dm, Im = flat_ip.merge_shard_results(Ds, Is, 50)
    # BLAS blocks differently for different shard shapes -> last-ulp score differences are expected
    assert np.array_equal(Im, I) and np.allclose(Dm, D, atol=1e-6)


def test_comparator_flags_real_errors():
    xb = synth.clip_like(2000, 32, seed=5, n_centres=16)
    xq = synth.clip_like(3, 32, seed=6, n_centres=16)
    idx = flat_ip.IndexFlatIP(32)
    idx.add(xb)
    D, I = idx.search(xq, 20)
    so = lambda ids: idx.scores_of(xq, ids)
    assert comparator.compare_topk(D, I, D, I, so) == []
    Ibad = I.copy()
    Ibad[0, 0] = int(np.argmin(xb @ xq[0]))                          # clearly not a top hit
    assert comparator.compare_topk(D, Ibad, D, I, so)
    Dbad = D.copy()
    Dbad[1, 3] += 0.01
    assert comparator.compare_topk(Dbad, I, D, I, so)


# ---------------------------------------------------------------------------
# O4: similar-sequence search, pinned to the reference's TemporalAnalyzer
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["a", "b", "c"])
def test_sequence_oracle_matches_reference(temporal_golden, name):
    from oracle import temporal as ot
    tg = temporal_golden
    case, db, target = tg["cases"][name], tg["arrays"][f"{name}_db"], tg["arrays"][f"{name}_target"]
    L, thr = case["sequence_length"], case["threshold"]
    got = ot.find_similar_sequences(target, db, L, thr)
    assert [[int(j), float(s)] for j, s in got] == case["hits"]          # bit-for-bit, including the order
    # the vectorised oracle: same hit set, similarities within float32 rounding of the BLAS/sklearn order
    sims = ot.window_similarities(target, db, L)
    want = sorted((j, s) for j, s in case["hits"])
    t_idx, j_idx = np.nonzero(sims >= np.float32(thr))
    fast = sorted((int(j), float(sims[t, j])) for t, j in zip(t_idx, j_idx))
    assert [j for j, _ in fast] == [j for j, _ in want]
    np.testing.assert_allclose([s for _, s in fast], [s for _, s in want], rtol=0, atol=2e-6)
    # guard band the GPU test relies on: no window within 1e-4 of the threshold
    assert not (np.abs(sims - np.float32(thr)) < 1e-4).any()
    # scene boundaries of the same analyzer (core.py:3584-3642)
    from oracle import dedup as od
    assert [list(b) for b in od.detect_scene_boundaries(db, 0.3, 5)] == case["scene_boundaries"]


def test_scene_boundaries_short_clip_with_and_without_validation(temporal_golden):
    """core.py:3601-3608: the 'too few features -> single scene' shortcut is part of validate_inputs.  120 nine-frame
    slices run through the unmodified reference both ways (33 of them answer differently)."""
    from oracle import dedup as od
    sc, db = temporal_golden["cases"]["short_clip"], temporal_golden["arrays"]["a_db"]
    differ = 0
    for c in sc["slices"]:
        sl = db[c["start"]:c["start"] + sc["length"]]
        for flag, key in ((True, "validated"), (False, "unvalidated")):
            got = od.detect_scene_boundaries(sl, sc["threshold"], sc["min_scene_length"], validate_inputs=flag)
            assert [list(b) for b in got] == c[key], (c["start"], key)
        differ += c["validated"] != c["unvalidated"]
    assert differ >= 20


def test_sequence_oracle_short_inputs_and_mean_order(temporal_golden):
    from oracle import temporal as ot
    tg = temporal_golden
    assert tg["cases"]["short"]["hits"] == []
    assert ot.find_similar_sequences(tg["arrays"]["a_target"][:3], tg["arrays"]["a_db"], 5) == []
    assert ot.compute_sequence_similarity(np.zeros((3, 4), np.float32), np.zeros((2, 4), np.float32)) == 0.0
    # the summation order the CUDA kernel implements IS NumPy's float32 np.mean for every length it accepts
    rng = np.random.default_rng(5)
    for n in range(1, 129):
        for _ in range(20):
            a = (rng.random(n) * 0.3 + 0.7).astype(np.float32)
            assert np.float32(np.mean([np.float32(v) for v in a])) == ot.numpy_mean_f32(a)


# ---------------------------------------------------------------------------
# O5: DBSCAN phase + scene changes of filter_research_update.py, pinned to the reference (real scikit-learn)
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["s384", "s64", "s512"])
def test_cluster_oracle_matches_reference(research_golden, name):
    from oracle import cluster as oc, dedup as od
    rg = research_golden
    case, x = rg["cases"][name], rg["arrays"][name]
    assert od.detect_scene_changes(list(x), case["scene_threshold"]) == case["scene_changes"]
    pinned = 0
    for span, want in case["clusters"].items():
        a, b = (int(v) for v in span.split(":"))
        got = oc.cluster_similar_frames(list(x[a:b]), case["eps"], case["min_samples"])
        if want == "ValueError":                  # reference + recent scikit-learn: negative 1 - cos from rounding
            assert (1 - oc.cosine_matrix(x[a:b])).min() < 0
            continue
        assert got == want, span
        assert [oc.select_representative_frame(g, list(x[a:b])) for g in got] == case["representatives"][span], span
        pinned += 1
    assert pinned >= 5


def test_cluster_oracle_edges_and_dbscan_rule(research_golden):
    from oracle import cluster as oc
    assert research_golden["cases"]["edge"] == {"empty": [], "one": [[0]]}
    assert oc.cluster_similar_frames([]) == [] and oc.cluster_similar_frames([np.ones(4, np.float32)]) == [[0]]
    # chain 0-1-2 (core 1), border 3 reached from core 2?, isolated 4: labels follow the index-order / LIFO rule
    nb = [np.array([0, 1]), np.array([0, 1, 2]), np.array([1, 2, 3]), np.array([2, 3]), np.array([4])]
    assert oc.dbscan_labels(nb, 2).tolist() == [0, 0, 0, 0, -1]
    assert oc.dbscan_labels(nb, 3).tolist() == [0, 0, 0, 0, -1]      # 0 and 3 are border points of cores 1 and 2
    assert oc.groups_from_labels([1, -1, 1, 0]) == [[0, 2], [1], [3]]


def test_similarity_relationships_oracle_matches_reference(relationships_golden):
    """core.py:3493-3531 -- the oracle reproduces the reference's graph exactly (same sklearn-order cosines,
    same argsort tie behaviour)."""
    rg = relationships_golden
    all_feat = {}
    for folder, x in rg["features"].items():
        keep = [i for i in range(len(x)) if (i % 11) != 5]
        all_feat[folder] = ([f"{folder}_{i:04d}" for i in keep], x[keep])
    graph, _ = flat_ip.similarity_relationships(all_feat)
    assert graph == rg["graph"]


def test_multithreaded_cpu_baseline_matches_the_numpy_oracle():
    """oracle/flat_ip_mt (the TIMED CPU baseline: torch sgemm + topk on every host thread) returns exactly what the
    NumPy oracle returns -- ids, order (ties -> lower id), scores, -1 / -FLT_MAX padding."""
    from oracle import flat_ip, flat_ip_mt, synth
    for n, d, nq, k, blk in ((30_000, 64, 33, 100, 1 << 13), (5, 16, 3, 8, 4), (12_345, 128, 7, 50, 1 << 12)):
        xb = synth.clip_like(n, d, seed=n, n_centres=32)
        xq = synth.clip_like(nq, d, seed=n + 1, n_centres=32)
        a = flat_ip.IndexFlatIP(d)
        a.add(xb)
        b = flat_ip_mt.IndexFlatIP(d, db_block=blk)
        b.add(xb[:n // 2])
        b.add(xb[n // 2:])
        D, I = a.search(xq, k)
        D2, I2 = b.search(xq, k)
        assert np.array_equal(I, I2)
        np.testing.assert_allclose(D2, D, rtol=0, atol=2e-6)
    dup = np.tile(synth.gaussian_unit(10, 32, seed=5), (30, 1))      # exact ties across the k-th boundary: like FAISS,
    a, b = flat_ip.IndexFlatIP(32), flat_ip_mt.IndexFlatIP(32, db_block=64)   # no promise WHICH tied row is returned
    a.add(dup); b.add(dup)
    (D, I), (D2, I2) = a.search(dup[:4], 40), b.search(dup[:4], 40)
    np.testing.assert_allclose(D2, D, rtol=0, atol=2e-6)
    np.testing.assert_allclose(a.scores_of(dup[:4], I2), D2, rtol=0, atol=2e-6)
    assert all(len(set(r.tolist())) == 40 for r in I2) and np.array_equal(I[:, :30], I2[:, :30])


def test_key_packing_round_trip_and_order():
    """oracle/flat_ip.pack_keys restates csrc/common.cuh make_key: unsigned descending key order == score descending,
    then lower id; id < 0 -> key 0."""
    from oracle import flat_ip
    rng = np.random.default_rng(0)
    D = rng.standard_normal((50, 40)).astype(np.float32)
    D[0, :5] = [0.0, -0.0, 1e-38, -1e-38, np.float32(3.0)]
    I = rng.integers(0, 2 ** 32 - 1, size=(50, 40), dtype=np.int64)
    I[1, 3:9] = -1
    keys = flat_ip.pack_keys(D, I)
    D2, I2 = flat_ip.unpack_keys(keys)
    ok = I >= 0
    assert np.array_equal(I2[ok], I[ok]) and np.array_equal(D2[ok].view(np.uint32), D[ok].view(np.uint32))
    assert (I2[~ok] == -1).all() and (keys[~ok] == 0).all()
    for r in range(50):
        order = np.argsort(keys[r])[::-1]
        want = np.lexsort((np.where(I[r] < 0, 2 ** 40, I[r]), -D[r].astype(np.float64) + 0.0, I[r] < 0))
        assert np.array_equal(D[r][order][ok[r][order]], D[r][want][ok[r][want]])


def test_inline_keep_chain_rules_match_the_reference(chain_golden):
    """The last-kept rule of video_frame_filter.extract_unique_frames (run as it is, decoder / model stubbed) and
    Phase 4 of filter_research_update (its statements executed from the parsed source): the restatements reproduce the
    reference's kept frames exactly."""
    from oracle import dedup as od
    for name, case in chain_golden["cases"].items():
        x = list(chain_golden["arrays"][name])
        if name.startswith("vff"):
            got = od.extract_unique_rule(x, case["threshold"])
        else:
            got = od.temporal_window_filter(x, case["threshold"], case["temporal_window"])
        assert got == case["kept"], name
        assert 0.1 * len(x) < len(got) < 0.95 * len(x)              # the rule really dropped and really kept frames
