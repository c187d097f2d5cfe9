"""Full-size parity of BASELINE configs[3] (cfg4: + & - -> and user:*, ~95 M relationships -- the HBM regime the
roofline target is quoted on) and of the machinery that only engages at that size: warp stacks spilling to HBM,
sub-query buffer overflow answered in halves, the path memo. Checker = the CPU oracle (a port: "parity unpinned"
against SpiceDB for these operators, DESIGN.md 2), on >= 50 000 sampled checks of the very batch bench.py times,
spanning both `view` and `restricted_view`.

ZGPU_FULLSIZE_SCALE picks the store size: 1.0 = the full 95 M relationships (what scripts/gpu_ci.sh runs: the oracle's
index build alone is 30 s per store then, 12 minutes for this file); the default 0.25 (24 M relationships, a 0.5 GB
store: still four times the L2) keeps the -m gpu suite within a few minutes. bench.py compares the whole 1 M-check batch
of cfg4 at scale 1.0 with the oracle on every run."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SCALE = float(os.environ.get("ZGPU_FULLSIZE_SCALE", "0.25"))
SAMPLE = 60_000


@pytest.fixture(scope="module")
def zg():
    import zgpu

    return zgpu


@pytest.fixture(scope="module")
def big(zg):
    """The cfg4 workload, the oracle's answers on the sample, and the sample's indices."""
    from oracle.pyoracle import Oracle
    from spicedb_kubeapi_proxy_b200 import workloads

    w = workloads.cfg4(scale=SCALE)
    o = Oracle(w.schema)
    w.load_into(o)
    items = w.check_items(o, zg.CHECK_DTYPE)
    n = min(SAMPLE, items.size)
    want = o.check_bulk(items[:n], nthreads=os.cpu_count() or 8)
    del o
    return w, items, want


def _engine(zg, w, **kw):
    e = zg.Engine(w.schema, **kw)
    w.load_into(e)
    e.publish()
    return e


def test_cfg4_full_size_sample_is_bit_exact(zg, big):
    w, items, want = big
    e = _engine(zg, w)
    assert e.stats()["tuples"] > 90_000_000 * SCALE
    got = e.check_bulk(items)
    n = want.size
    mism = np.flatnonzero(got[:n] != want)
    assert mism.size == 0, f"{mism.size} of {n} differ, first at {mism[:5]}: {items[mism[:5]]}"
    # both permissions are in the sample, with both answers
    view, rview = e.slot_id("document", "view"), e.slot_id("document", "restricted_view")
    for perm in (view, rview):
        sel = items["perm"][:n] == perm
        assert sel.sum() > n // 10 and (want[sel] == 2).any() and (want[sel] == 1).any()
    assert 0.2 < (want == 2).mean() < 0.8
    assert not (got == 255).any()
    # properties that do not need the oracle, over the whole batch: restricted_view = view & org->member can only
    # remove grants; re-asking gives the same answers; the device entry point agrees
    as_view = items.copy()
    as_view["perm"] = view
    gv = e.check_bulk(as_view)
    r = items["perm"] == rview
    assert not ((got[r] == 2) & (gv[r] != 2)).any()
    assert np.array_equal(e.check_bulk(items), got)
    st = e.stats()
    assert st["passes"] == 0  # folder#view is a pure union: one launch answers the batch
    e.close()


def test_cfg4_full_size_with_the_path_memo_forced_on(zg, big, monkeypatch):
    """Every batch remembers its child visits from the first expansion round on: skipping a repeated
    (check, slot, object, depth) visit must not change an answer on the large store either."""
    w, items, want = big
    monkeypatch.setenv("ZGPU_MEMO_AFTER", "0")
    e = _engine(zg, w)
    monkeypatch.delenv("ZGPU_MEMO_AFTER")
    n = want.size
    got = e.check_bulk(items[: 4 * n])
    assert np.array_equal(got[:n], want)
    assert e.stats()["memo_batches"] > 0
    e.close()


def test_forward_only_engine_agrees_at_full_size(zg, big):
    """No reverse-row probes at all (ZG_FLAG_FORWARD_ONLY): the plain frontier expansion, same answers."""
    w, items, want = big
    e = _engine(zg, w, forward_only=True)
    n = want.size
    assert np.array_equal(e.check_bulk(items[:n]), want)
    e.close()


def test_subquery_passes_and_overflow_split_on_a_large_store(zg):
    """cfg4 with a NON-PURE folder#view (`- banned`): every document -> folder edge raises a sub-query, level after
    level up the folder chain. With a pass buffer far smaller than one batch's sub-queries the batch is answered in
    halves, recursively; answers equal the oracle's and those of an engine with the default buffer."""
    from oracle.pyoracle import Oracle
    from spicedb_kubeapi_proxy_b200 import workloads

    w = workloads.cfg4(scale=min(SCALE, 0.2), nonpure_folders=True)
    o = Oracle(w.schema)
    w.load_into(o)
    items = w.check_items(o, zg.CHECK_DTYPE)
    n = min(SAMPLE, items.size)
    want = o.check_bulk(items[:n], nthreads=os.cpu_count() or 8)
    del o
    big_buf = _engine(zg, w)
    small_buf = _engine(zg, w, subquery_capacity=20_000)
    got = big_buf.check_bulk(items)
    assert np.array_equal(got[:n], want)
    assert big_buf.stats()["passes"] >= 2, "the folder chain must take several sub-query passes"
    assert np.array_equal(small_buf.check_bulk(items), got)
    assert small_buf.stats()["split_batches"] > 0
    big_buf.close(), small_buf.close()


def test_thousand_update_write_on_the_large_store_is_a_merge(zg, big):
    """pkg/authz/distributedtx/activity.go:47-77 writes <= 1000 updates per call (spicedb.go:34); on the 95 M store
    such a write must not cost a rebuild (0.65 s): the journal is merged into the resident CSR in one streaming
    pass. Timed here (device ms of the publish), answers checked on a probe set that includes every touched
    document, against the oracle with the same updates."""
    import json
    import time

    from oracle.pyoracle import Oracle
    from test_gpu_parity import _random_updates

    w, items, want = big
    e = _engine(zg, w)
    rng = np.random.default_rng(11)
    t_full = e.stats()["last_publish_ms"]
    times = []
    all_ups = []
    for _ in range(5):
        ups = _random_updates(zg, e, w, rng, 1000, new_objects=False)
        t0 = time.perf_counter()
        e.apply_updates(ups)
        e.publish()
        times.append((time.perf_counter() - t0) * 1e3)
        all_ups.append(ups)
    st = e.stats()
    assert st["delta_publishes"] == 5 and st["full_publishes"] == 1, st
    rec = {"store_tuples": int(st["tuples"]), "updates_per_write": 1000, "wall_ms": times,
           "device_ms_last": st["last_publish_ms"], "full_rebuild_device_ms": t_full, "scale": SCALE}
    print("write merge:", json.dumps(rec))  # shown with -s, and with the failure report
    assert min(times) < 50.0, rec  # target: < 5 ms; the bound leaves room for a noisy box
    # parity after the writes: the oracle replays them (one re-index), probes = touched documents x their checks
    o = Oracle(w.schema)
    w.load_into(o)
    for ups in all_ups:
        o.apply_updates(ups)
    doc_rels = {e.slot_id("document", r) for r in ("parent", "org", "owner", "editor", "viewer", "banned")}
    touched = np.concatenate([u["res"][np.isin(u["rel"], list(doc_rels))] for u in all_ups])
    probe = items[:20000].copy()
    probe["res"][: touched.size] = touched[: probe.size]
    got, exp = e.check_bulk(probe), o.check_bulk(probe, nthreads=os.cpu_count() or 8)
    bad = np.flatnonzero(got != exp)
    assert bad.size == 0, f"{bad.size} of {probe.size} differ; first {bad[:8]} (touched probes: < {touched.size}): " \
                          f"{probe[bad[:8]]} gpu {got[bad[:8]]} oracle {exp[bad[:8]]}"
    e.close()
