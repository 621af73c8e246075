"""The results of one omni_ctx must not depend on the calls made on it before.

A context keeps state from one call to the next: grow-only workspace slots, two caches of the candidate-centre tables in
workspace slot 5 (keyed by the centres, the label map, K and the stream), the helper context of the banded host call, the
resize tables and the device flags.  The other GPU modules make one engine per module and issue their calls in one fixed
order, while the stage scripts and library users keep one engine per device for the whole process and mix the entry points
freely.  Here each test starts from a fresh context and varies the order; every label, mask and edge output is compared
bit for bit with the C oracle, and k-means and tracing (which the oracle does not cover cheaply) with the same call on a
fresh context."""
import hashlib
import itertools

import numpy as np
import pytest

from helpers import synth, uniform_img

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

# Engine.set_fast_path: label-domain pipeline, dense first generation, dense edges + Lab cells, generic kernels
FAMILIES = (1, 3, 2, 0)


def _omni():
    import omni_b200
    return omni_b200


def _cm():
    from oracle import cmodel
    return cmodel


@pytest.fixture
def fresh():
    e = _omni().Engine(0)
    yield e
    e.close()


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.cpu().numpy()


def image(h, w, seed):
    return synth(h, w, seed, cell=16) if min(h, w) >= 16 else uniform_img(h, w, seed)


def ec_of(ksize=3, low=50, high=150, morph_k=3, oi=1, ci=1):
    return _omni().EdgeConfig(low=low, high=high, ksize=ksize, morph_k=morph_k, open_iters=oi, close_iters=ci)


def centres(img, K, seed):
    """K Lab centres near colours of the image (so that the layers are populated), with fractional parts."""
    lab = _cm().bgr2lab(img).reshape(-1, 3).astype(np.float32)
    rng = np.random.default_rng(seed)
    return (lab[rng.integers(0, lab.shape[0], K)] + rng.uniform(-4, 4, (K, 3))).astype(np.float32)


def make_lut(kind, K, seed=0):
    """identity, a permutation, or a permutation with one label >= K (no plane of its own; the RGB-cell tables hold labels in
    4 bits and cannot take it, so the assignment uses the Lab-cell tables)."""
    if kind == "identity":
        return np.arange(K, dtype=np.uint8)
    lut = np.random.default_rng(seed).permutation(K).astype(np.uint8)
    if kind == "high":
        lut[K // 2] = (K + 32) // 2
    return lut


def uses_rgb_cells(K, lut):
    return K <= 16 and int(np.max(lut)) < K


_MEMO = {}


def oracle(img, ctr, lut, ec):
    """(labels, masks, edges) of the fused call by the C oracle; ec None: no edges."""
    K = len(ctr)
    lut = np.arange(K, dtype=np.uint8) if lut is None else np.asarray(lut, np.uint8)
    img = np.ascontiguousarray(img)
    key = (img.shape, hashlib.blake2b(img).digest(), np.asarray(ctr, np.float32).tobytes(), lut.tobytes(),
           None if ec is None else (ec.ksize, ec.low, ec.high, ec.morph_k, ec.open_iters, ec.close_iters))
    if key not in _MEMO:
        cm = _cm()
        raw = cm.assign_f32(cm.bgr2lab(img), ctr)
        masks = cm.layer_masks(raw, K, lut)
        edges = None if ec is None else \
            np.stack([cm.edge_chain(m, ec.morph_k, ec.open_iters, ec.close_iters, ec.ksize, ec.low, ec.high) for m in masks])
        if len(_MEMO) >= 12:
            _MEMO.pop(next(iter(_MEMO)))
        _MEMO[key] = (lut[raw], masks, edges)
    return _MEMO[key]


def check_fused(eng, img, ctr, lut, ec, what="", **out):
    labels, masks, edges = eng.color_edge(dev(img), ctr, lut, ec, want_labels=True, **out)
    wl, wm, we = oracle(img, ctr, lut, ec)
    assert np.array_equal(host(labels), wl), f"labels {what}"
    assert np.array_equal(host(masks), wm), f"masks {what}"
    assert np.array_equal(host(edges), we), f"edges {what}"
    return labels, masks, edges


def table_builds(eng, call):
    """Runs call() with profiling on: {kernel name: launches} of the three table-building kernels."""
    eng.profile(True)
    try:
        call()
        s = eng.profile_summary()
    finally:
        eng.profile(False)
    return {k: s[k][0] for k in ("build_cells", "build_rgbcells", "build_tables") if k in s}


def label_domain_call(eng, img):
    """A fused blur-3 call with K <= 16 and every label < K: the label-domain pipeline, whose tables take the larger slot 5."""
    check_fused(eng, img, centres(img, 8, 99), None, ec_of(3), "label-domain call")


# ---- 2a. the sequences that reallocate slot 5 between two identical first-generation assignments ----------------------------
KBIG = {4: 17, 16: 24, 20: 20}          # K > 16 of the fused sequence (first generation at blur 3)


@pytest.mark.parametrize("lut_kind", ["identity", "perm", "high"])
@pytest.mark.parametrize("K", [4, 16, 20])
@pytest.mark.parametrize("seq", ["blur_sweep", "assign_label_assign", "kbig_label_kbig", "reserve"])
def test_tables_rebuilt_after_slot5_grows(fresh, seq, K, lut_kind):
    """A first-generation assignment, then a call that reallocates workspace slot 5 (where the first generation keeps its
    tables), then the first assignment again with the same centres, label map, K and stream.  The last call must rebuild its
    tables: the new allocation holds nothing, whatever address it has."""
    eng = fresh
    eng.set_fast_path(1)
    img = image(300, 420, 7 + K)
    if seq == "kbig_label_kbig":
        K = KBIG[K]
    ctr, lut = centres(img, K, K), make_lut(lut_kind, K, K)
    if seq == "assign_label_assign":
        def first():
            assert np.array_equal(host(eng.assign_lab(dev(img), ctr, lut)), oracle(img, ctr, lut, None)[0])
    else:
        ec = ec_of({"blur_sweep": 5, "kbig_label_kbig": 3, "reserve": 7}[seq])

        def first():
            check_fused(eng, img, ctr, lut, ec, seq)
    assert "build_cells" in table_builds(eng, first)
    if seq == "reserve":
        eng.reserve(img.shape[0], img.shape[1], K)
    else:
        grew = False
        if seq == "blur_sweep":                   # the same image and centres at blur 3
            grew = "build_tables" in table_builds(eng, lambda: check_fused(eng, img, ctr, lut, ec_of(3), "blur 3"))
            assert grew == uses_rgb_cells(K, lut)
        if not grew:
            assert "build_tables" in table_builds(eng, lambda: label_domain_call(eng, img))
    b = table_builds(eng, first)
    assert "build_cells" in b, b
    assert ("build_rgbcells" in b) == uses_rgb_cells(K, lut), b


# ---- 2b. kernel families in every order on one context ---------------------------------------------------------------------------
@pytest.mark.parametrize("order", list(itertools.permutations(FAMILIES)), ids=lambda o: "-".join(map(str, o)))
def test_family_order(fresh, order):
    img = image(257, 389, 5)
    ctr, lut = centres(img, 12, 5), make_lut("perm", 12, 5)
    for mode in order:
        fresh.set_fast_path(mode)
        for ks in (3, 7):
            check_fused(fresh, img, ctr, lut, ec_of(ks), f"family {mode}, blur {ks}")


# ---- 2c. small changes of the cache key ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("tables", ["label_pipeline", "first_generation"])
def test_small_key_changes_rebuild(fresh, tables):
    ksize, build = (3, "build_tables") if tables == "label_pipeline" else (5, "build_cells")
    K = 8
    img = image(240, 352, 11)
    ctr, ident, perm = centres(img, K, 11), make_lut("identity", K), make_lut("perm", K, 3)
    ulp = ctr.copy()
    ulp[3, 1] = np.nextafter(ctr[3, 1], np.float32(np.inf))
    side = torch.cuda.Stream()
    steps = [("first call", ctr, perm, None), ("lut only", ctr, ident, None), ("one ULP", ulp, ident, None),
             ("K - 1, same first centres", ulp[:K - 1], ident[:K - 1], None), ("K + 1", ulp, ident, None),
             ("second stream", ulp, ident, side)]
    for name, c, lut, stream in steps:
        torch.cuda.synchronize()                  # one stream at a time on a context
        if stream is None:
            b = table_builds(fresh, lambda: check_fused(fresh, img, c, lut, ec_of(ksize), name))
        else:
            with torch.cuda.stream(stream):
                b = table_builds(fresh, lambda: check_fused(fresh, img, c, lut, ec_of(ksize), name))
            stream.synchronize()
        assert b.get(build) == 1, (name, b)
    with torch.cuda.stream(side):                 # the same call again: served from the cache
        assert build not in table_builds(fresh, lambda: check_fused(fresh, img, ulp, ident, ec_of(ksize), "repeat"))
    side.synchronize()


# ---- 2d. cache on = cache off ----------------------------------------------------------------------------------------------------
ENTRY_POINTS = ["assign_lab", "color_edge_blur3", "color_edge_blur5", "color_edge_batch", "color_edge_packed", "host_color_edge",
                "host_color_edge_packed_banded"]


def _bits(planes):
    return np.packbits(planes > 0, axis=-1)


def _run_entry(entry, eng, frames, ctr, lut):
    """(outputs of the call, the same outputs by the oracle) as lists of host arrays."""
    ec = ec_of(5 if entry == "color_edge_blur5" else 3)
    f0 = frames[0]
    if entry == "assign_lab":
        return [host(eng.assign_lab(dev(f0), ctr, lut))], [oracle(f0, ctr, lut, None)[0]]
    if entry.startswith("color_edge_blur"):
        return [host(t) for t in eng.color_edge(dev(f0), ctr, lut, ec, want_labels=True)], list(oracle(f0, ctr, lut, ec))
    if entry == "color_edge_batch":
        m, e = eng.color_edge_batch(dev(frames), ctr, lut, ec)
        _l, wm, we = oracle(frames[-1], ctr, lut, ec)
        return [host(m[-1]), host(e[-1]), host(m), host(e)], [wm, we]
    if entry == "color_edge_packed":
        mb, eb, counts = eng.color_edge_packed(dev(frames), ctr, lut, ec, want_counts=True)
        want = [np.concatenate([_bits(oracle(f, ctr, lut, ec)[i]) for f in frames]) for i in (1, 2)]
        return [host(mb), host(eb), counts], want
    if entry == "host_color_edge":
        r = eng.host_color_edge(f0, ctr, lut, ec)
        return [r["labels"], r["masks"], r["edges"], r["counts"]], list(oracle(f0, ctr, lut, ec))
    r = eng.host_color_edge_packed(f0, ctr, lut, ec)
    assert eng.last_band_resends() >= 0                  # the banded path ran (helper context, tables held over the bands)
    _l, wm, we = oracle(f0, ctr, lut, ec)
    return [r["mask_bits"], r["edge_bits"], r["counts"]], [_bits(wm), _bits(we)]


@pytest.mark.parametrize("entry", ENTRY_POINTS)
def test_table_cache_on_equals_off(entry):
    omni = _omni()
    h, w, K, n = {"color_edge_batch": (96, 160, 12, 3), "color_edge_packed": (130, 250, 8, 2),
                  "host_color_edge_packed_banded": (1100, 1920, 8, 1)}.get(entry, (240, 352, 8, 1))
    frames = np.stack([image(h, w, 20 + f) for f in range(n)])
    A, B = centres(frames[0], K, 1), centres(frames[0], K, 2)
    lut = make_lut("perm", K, 4)
    e_on, e_off = omni.Engine(0), omni.Engine(0)
    try:
        e_off.set_table_cache(False)
        for i, ctr in enumerate((A, B, A, A)):
            got_on, want = _run_entry(entry, e_on, frames, ctr, lut)
            got_off, _w = _run_entry(entry, e_off, frames, ctr, lut)
            for j, (a, b) in enumerate(zip(got_on, got_off)):
                assert np.array_equal(a, b), (i, j)
            for j, (a, b) in enumerate(zip(got_on, want)):
                assert np.array_equal(a, b), (i, j)
    finally:
        e_on.close()
        e_off.close()


# ---- 2e. the cache still caches ------------------------------------------------------------------------------------------------
def test_table_cache_hits(fresh):
    K = 8
    img = image(240, 352, 3)
    frames = np.stack([img, image(240, 352, 4)])
    ctr, lut = centres(img, K, 3), make_lut("perm", K, 1)

    def first():
        check_fused(fresh, img, ctr, lut, ec_of(5), "first generation")

    def label():
        check_fused(fresh, img, ctr, lut, ec_of(3), "label pipeline")

    def batch():
        m, e = fresh.color_edge_batch(dev(frames), ctr, lut, ec_of(3))
        _l, wm, we = oracle(frames[1], ctr, lut, ec_of(3))
        assert np.array_equal(host(m[1]), wm) and np.array_equal(host(e[1]), we)

    both = {"build_cells": 1, "build_rgbcells": 1}
    assert table_builds(fresh, first) == both
    assert table_builds(fresh, first) == {}
    assert table_builds(fresh, label) == {"build_tables": 1}           # grows slot 5 once
    assert table_builds(fresh, label) == {}
    assert table_builds(fresh, batch) == {}                            # frame batches share the tables (bench.py config 4)
    assert table_builds(fresh, first) == both                          # slot 5 was reallocated since the first call
    assert table_builds(fresh, first) == {}
    assert table_builds(fresh, label) == {}
    fresh.set_table_cache(False)
    for _ in range(2):
        assert table_builds(fresh, first) == both
        assert table_builds(fresh, label) == {"build_tables": 1}
        assert table_builds(fresh, batch) == {"build_tables": 1}


# ---- 2f. workspaces that grow and shrink -----------------------------------------------------------------------------------------
GROW_SHRINK = [((1500, 2100), 16, 3), ((37, 45), 3, 3), ((700, 33), 32, 3), ((1, 1), 2, 3), ((1500, 2100), 8, 7),
               ((257, 389), 16, 3)]


@pytest.mark.parametrize("mode", FAMILIES)
def test_workspaces_grow_and_shrink(fresh, mode):
    """Large, tiny, many planes, 1x1, large again, then a mid-size geometry into outputs pre-filled with 7s: stale bytes of
    larger workspaces, run-list counters and the zero fill must not leak into a smaller geometry.  Then Engine.reserve for a
    larger geometry, and the whole sequence again."""
    fresh.set_fast_path(mode)

    def sequence():
        for i, ((h, w), K, ks) in enumerate(GROW_SHRINK):
            img = image(h, w, 40 + i)
            ctr, lut = centres(img, K, i), make_lut("perm", K, i)
            what = f"family {mode}, step {i}: {h}x{w}, K={K}, blur {ks}"
            if i == len(GROW_SHRINK) - 1:
                out = {"labels": torch.full((h, w), 7, dtype=torch.uint8, device="cuda"),
                       "masks": torch.full((K, h, w), 7, dtype=torch.uint8, device="cuda"),
                       "edges": torch.full((K, h, w), 7, dtype=torch.uint8, device="cuda")}
                check_fused(fresh, img, ctr, lut, ec_of(ks), what, **out)
            else:
                check_fused(fresh, img, ctr, lut, ec_of(ks), what)

    sequence()
    fresh.reserve(2000, 2400, 16, ksize=7)
    sequence()


# ---- 2g. seeded mixed sequences of every entry point -----------------------------------------------------------------------------
GEOMS = [(1, 1), (37, 45), (129, 257), (300, 420), (700, 33), (480, 640)]
MIXED = ["fused", "batch", "packed", "host_color_edge", "host_color_edge_packed", "edges", "layer_masks", "assign_lab",
         "resize_area", "thin", "skeleton_degree", "kmeans_lab", "trace", "swatch"]


def _same_trace(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert x.total_fg == y.total_fg and np.array_equal(x.stats, y.stats) and np.array_equal(x.polylines, y.polylines)
        assert len(x.paths) == len(y.paths) and all(np.array_equal(p, q) for p, q in zip(x.paths, y.paths))


def _on_fresh_engine(mode, call):
    ref = _omni().Engine(0)
    try:
        ref.set_fast_path(mode)
        return call(ref)
    finally:
        ref.close()


def _mixed_step(eng, rng, pool):
    """Draws one step and runs it against its reference; returns its description (drawn before anything runs)."""
    cm = _cm()
    entry = MIXED[int(rng.integers(len(MIXED)))]
    h, w = GEOMS[int(rng.integers(len(GEOMS)))]
    K = int(rng.integers(2, 33))
    mode = FAMILIES[int(rng.integers(len(FAMILIES)))]
    p = int(rng.integers(len(pool)))
    img_seed = int(rng.integers(3))
    lut_kind = ("identity", "perm", "high")[int(rng.integers(3))] if K <= 30 else "perm"
    ks = (3, 5, 7)[int(rng.integers(3))]
    low, high = float(rng.choice([20, 50, 75.5])), float(rng.choice([100, 150, 210]))
    extra = int(rng.integers(1 << 30))
    desc = f"{entry} {h}x{w} K={K} family={mode} centres={p} image={img_seed} lut={lut_kind} blur={ks} low={low} high={high} x={extra}"
    yield desc
    eng.set_fast_path(mode)
    img = image(h, w, 100 + img_seed)
    ctr = pool[p][:K]
    lut = make_lut(lut_kind, K, extra)
    ec = ec_of(ks, low, high)
    sub = np.random.default_rng(extra)
    if entry == "fused":
        check_fused(eng, img, ctr, lut, ec)
    elif entry == "batch":
        n = int(sub.integers(2, 4))
        frames = np.stack([image(h, w, 100 + img_seed + f) for f in range(n)])
        m, e = eng.color_edge_batch(dev(frames), ctr, lut, ec)
        _l, wm, we = oracle(frames[-1], ctr, lut, ec)
        assert np.array_equal(host(m[-1]), wm) and np.array_equal(host(e[-1]), we)
    elif entry == "packed":
        n = max(1, min(2, 32 // K))
        frames = np.stack([image(h, w, 100 + img_seed + f) for f in range(n)])
        with_edges = bool(sub.integers(2))
        mb, eb = eng.color_edge_packed(dev(frames), ctr, lut, ec if with_edges else None)
        assert np.array_equal(host(mb), np.concatenate([_bits(oracle(f, ctr, lut, None)[1]) for f in frames]))
        if with_edges:
            assert np.array_equal(host(eb), np.concatenate([_bits(oracle(f, ctr, lut, ec)[2]) for f in frames]))
    elif entry == "host_color_edge":
        r = eng.host_color_edge(img, ctr, lut, ec)
        wl, wm, we = oracle(img, ctr, lut, ec)
        assert np.array_equal(r["labels"], wl) and np.array_equal(r["masks"], wm) and np.array_equal(r["edges"], we)
        assert np.array_equal(r["counts"][:, 1], (wm > 0).reshape(K, -1).sum(1))
    elif entry == "host_color_edge_packed":
        n = int(sub.integers(1, 3))
        frames = np.stack([image(h, w, 100 + img_seed + f) for f in range(n)])
        r = eng.host_color_edge_packed(frames, ctr, lut, ec)
        assert np.array_equal(r["mask_bits"], np.concatenate([_bits(oracle(f, ctr, lut, ec)[1]) for f in frames]))
        assert np.array_equal(r["edge_bits"], np.concatenate([_bits(oracle(f, ctr, lut, ec)[2]) for f in frames]))
    elif entry == "edges":
        masks = oracle(img, ctr, None, None)[1]
        mk, oi, ci = int(sub.choice([1, 2, 3, 5, 9, 15])), int(sub.integers(3)), int(sub.integers(3))
        eks = int(sub.choice([3, 5, 7, 9]))
        got = host(eng.edges(dev(masks), ec_of(eks, low, high, mk, oi, ci)))
        want = np.stack([cm.edge_chain(m, mk, oi, ci, eks, low, high) for m in masks])
        assert np.array_equal(got, want), (mk, oi, ci, eks)
    elif entry == "layer_masks":
        labels = oracle(img, ctr, None, None)[0]
        oi, ci = [(1, 1), (0, 0), (2, 1), (0, 3)][int(sub.integers(4))]
        assert np.array_equal(host(eng.layer_masks(dev(labels), K, oi, ci)), cm.layer_masks(labels, K, None, oi, ci)), (oi, ci)
    elif entry == "assign_lab":
        assert np.array_equal(host(eng.assign_lab(dev(img), ctr, lut)), oracle(img, ctr, lut, None)[0])
    elif entry == "resize_area":
        nh, nw = max(1, h // int(sub.integers(1, 4))), max(1, int(w * sub.uniform(0.3, 1.0)))
        got = host(eng.resize_area(dev(img), nw, nh))
        d = np.abs(got.astype(np.int16) - cm.resize_area(img, nw, nh).astype(np.int16))
        if h % nh == 0 and w % nw == 0:
            assert d.max() == 0, (nh, nw)
        else:
            assert d.max() <= 1 and (d != 0).mean() < 1e-3, (nh, nw)
    elif entry in ("thin", "skeleton_degree", "trace"):
        edges = oracle(img, ctr, None, ec_of(3))[2]
        skel = np.stack([cm.thin_zhangsuen(e) for e in edges])
        if entry == "thin":
            assert np.array_equal(host(eng.thin_zhangsuen(dev(edges))), skel)
        elif entry == "skeleton_degree":
            from oracle import refport
            deg, nodes = (host(t) for t in eng.skeleton_degree(dev(skel)))
            for k in range(K):
                wd, ep, jn = refport.skeleton_degree(skel[k])
                assert np.array_equal(deg[k], wd) and np.array_equal(nodes[k] == 1, ep) and np.array_equal(nodes[k] == 2, jn), k
        else:
            _same_trace(eng.trace_centerlines(dev(skel)), _on_fresh_engine(mode, lambda r: r.trace_centerlines(dev(skel))))
    elif entry == "kmeans_lab":
        kk = min(K, h * w)

        def km(e):
            return e.kmeans_lab(dev(img), kk, attempts=2, max_iter=10, seed=extra)
        c1, comp1 = km(eng)
        c2, comp2 = _on_fresh_engine(mode, km)
        assert np.array_equal(c1, c2) and comp1 == comp2
    else:                                          # swatch
        px = img.reshape(-1, 3)
        cols = px[sub.integers(0, px.shape[0], K)].astype(np.int32)
        tol = int(sub.integers(0, 80))
        got, gc = eng.swatch_masks(dev(img), cols, tol, with_choice=True)
        want, wc = cm.swatch_masks(img, cols, tol, with_choice=True)
        assert np.array_equal(host(got), want) and np.array_equal(gc, wc), tol


@pytest.mark.parametrize("seed", range(6))
def test_mixed_sequences(fresh, seed):
    rng = np.random.default_rng(seed)
    pool = [centres(image(256, 256, 900 + i), 32, i) for i in range(3)]     # three centre sets that recur
    log = []
    for i in range(25):
        step = _mixed_step(fresh, rng, pool)
        log.append(next(step))
        try:
            for _ in step:
                pass
        except Exception as e:
            steps = "\n".join(f"  {j}: {s}" for j, s in enumerate(log))
            pytest.fail(f"seed {seed}, step {i} failed: {type(e).__name__}: {e}\nsteps so far:\n{steps}")


# ---- 2h. two contexts on one device ------------------------------------------------------------------------------------------------
def test_two_contexts_interleaved():
    omni = _omni()
    img1, img2 = image(240, 352, 31), image(300, 200, 32)
    c1, c2 = centres(img1, 8, 1), centres(img2, 20, 2)
    l1, l2 = make_lut("perm", 8, 1), make_lut("identity", 20)
    e1, e2 = omni.Engine(0), omni.Engine(0)
    e3 = None
    try:
        e2.set_fast_path(3)
        first = None
        for rnd in range(2):
            for eng, img, c, lut, ks in ((e1, img1, c1, l1, 3), (e2, img2, c2, l2, 5), (e1, img1, c1, l1, 5), (e2, img2, c2, l2, 3),
                                         (e1, img2, c2, l2, 3), (e2, img1, c1, l1, 3)):
                out = [host(t) for t in check_fused(eng, img, c, lut, ec_of(ks), f"round {rnd}, blur {ks}")]
                if first is None:
                    first = out
            assert np.array_equal(host(e2.assign_lab(dev(img1), c1, l1)), oracle(img1, c1, l1, None)[0])
        e1.close()
        e3 = omni.Engine(0)                       # re-created: the same bytes as the first context's first call
        out = [host(t) for t in check_fused(e3, img1, c1, l1, ec_of(3), "re-created context")]
        assert all(np.array_equal(a, b) for a, b in zip(out, first))
    finally:
        for e in (e1, e2, e3):
            if e is not None:
                e.close()
