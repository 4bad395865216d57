"""fp16 stores and fp16 queries on the B200 (B2_F16): the tcgen05 filter on kind::f16 with fp16 operands, the exact finalize,
the dense path, k-means and the all-pairs kernel over fp16 rows — bit-exact ids AND score bits against the oracle run on the
fp16-widened rows. Queries of every element type against every store; fp32 / bf16 queries rounded to fp16 for the filter
(including the subnormal range and values beyond fp16's range, which must take the exact path)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle
from helpers import bits, gauss, grid

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FMAX = np.finfo(np.float32).max


def f16(x):
    return np.asarray(x, dtype=np.float32).astype(np.float16).astype(np.float32)


def store(nv, x, dtype, metric):
    if dtype == "f16":
        return nv.Index(nv.f32_to_f16_bits(x), nv.F16, metric), f16(x)
    if dtype == "bf16":
        xb = nv.f32_to_bf16_bits(x)
        return nv.Index(xb, nv.BF16, metric), nv.bf16_bits_to_f32(xb)
    return nv.Index(x, nv.F32, metric), x


def queries(nv, q, qt):
    if qt == "f16":
        return nv.f32_to_f16_bits(q), nv.F16, f16(q)
    if qt == "bf16":
        qb = nv.f32_to_bf16_bits(q)
        return qb, nv.BF16, nv.bf16_bits_to_f32(qb)
    return q, nv.F32, q


def check(nv, x, q, k, metric, qt, dtype="f16", ids=None):
    idx, xf = store(nv, x, dtype, metric)
    qa, code, qf = queries(nv, q, qt)
    nv.stats_reset()
    D, I = idx.search(qa, k, code, ids=ids)
    st = nv.stats()
    Do, Io = oracle.knn(xf, qf, k, metric) if ids is None else oracle.knn_subset(xf, qf, k, ids, metric)
    idx.close()
    assert np.array_equal(I, Io), f"top-k indices differ in {(I != Io).any(axis=1).sum()} of {len(I)} rows"
    assert np.array_equal(bits(D), bits(Do)), "scores are not bit-identical to the canonical oracle score"
    return st


@pytest.mark.parametrize("d", [768, 384, 100, 30])
@pytest.mark.parametrize("qt", ["f32", "bf16", "f16"])
@pytest.mark.parametrize("k", [1, 10, 32, 64, 200, 1000])
@pytest.mark.parametrize("metric", [0, 1])
def test_f16_store_matrix(gpu, metric, k, qt, d):
    st = check(gpu, gauss(8192, d, 1 + d), gauss(300, d, 2 + d), k, metric, qt)
    assert st["filter_launches"] >= 1, "the tcgen05 filter did not run"
    # the certificate covers continuous data; at k = 1000 the k + 32 survivors of an 8k-row corpus leave too little room and many
    # queries take the dense path (still exact, as for bf16 / fp32 in test_gpu_search.py::test_large_k_goes_through_the_filter)
    if k <= 200:
        assert st["fallback_queries"] <= 6, st


@pytest.mark.parametrize("metric", [0, 1])
def test_ties_subsets_and_padding(gpu, metric):
    check(gpu, grid(300, 16, 3), grid(40, 16, 4), 17, metric, "f16")                      # dense path, grid ties (j/64 exact in fp16)
    check(gpu, grid(5000, 8, 6), grid(64, 8, 7), 10, metric, "f16")                       # tie-heavy: certified fallback
    rng = np.random.default_rng(5)
    x, q = gauss(6000, 64, 8), gauss(120, 64, 9)
    check(gpu, x, q, 8, metric, "f32", ids=rng.permutation(6000)[:2500])                  # permuted subset through the filter
    check(gpu, x, q, 8, metric, "f16", ids=np.array([5, 7, 7, 100, 2999]))                # K > len(ids): -1 padding
    idx, _ = store(gpu, x, "f16", metric)
    D, I = idx.search(q, 9000, gpu.F32)                                                   # K > n
    Do, Io = oracle.knn(f16(x), q, 9000, metric)
    assert np.array_equal(I, Io) and np.array_equal(bits(D), bits(Do))
    assert (I[:, 6000:] == -1).all() and (D[:, 6000:] == (FMAX if metric else -FMAX)).all()
    idx.close()


@pytest.mark.parametrize("qt", ["f32", "bf16"])
@pytest.mark.parametrize("metric", [0, 1])
def test_queries_beyond_fp16_range_take_the_exact_path(gpu, metric, qt):
    x, q = gauss(8192, 128, 10), gauss(200, 128, 11)
    q[::7, 5] = 1e5
    n_bad = len(q[::7])
    st = check(gpu, x, q, 10, metric, qt)
    assert st["filter_launches"] >= 1 and st["fallback_queries"] >= n_bad


@pytest.mark.parametrize("qt", ["f32", "bf16"])
@pytest.mark.parametrize("metric", [0, 1])
def test_small_norm_queries_in_the_subnormal_range(gpu, metric, qt):
    """Query elements around 1e-6 are fp16 subnormals (spacing 2^-24): rounding them moves every filter score by up to ~1 %,
    far more than the 2^-11 relative bound, so the filter's order near rank k is wrong for many queries. Only the absolute
    2^-25 sqrt(d) term of the certificate keeps the answer exact."""
    x = gauss(8192, 256, 12)
    q = gauss(300, 256, 13, normalize=False) * np.float32(2e-6)
    qf = queries(gpu, q, qt)[2]
    # the rounding does change the order near rank k on this data
    Dr, Ir = oracle.knn(f16(x), f16(qf), 10, metric)
    Do, Io = oracle.knn(f16(x), qf, 10, metric)
    assert (Ir != Io).any(axis=1).sum() > 10
    check(gpu, x, q, 10, metric, qt)


@pytest.mark.parametrize("metric", [0, 1])
@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_other_stores_with_f16_queries(gpu, metric, dtype):
    for n, k in ((8192, 10), (8192, 200), (3000, 5)):
        st = check(gpu, gauss(n, 96, 14), gauss(300, 96, 15), k, metric, "f16", dtype=dtype)
        assert st["filter_launches"] >= 1 and st["fallback_queries"] <= 6, st


def _mixture(n, d, k_true, seed, spread=1.0):
    rng = np.random.default_rng(seed)
    centers = gauss(k_true, d, seed + 1) * 4
    return (centers[rng.integers(0, k_true, n)] + spread * gauss(n, d, seed + 2, normalize=False)).astype(np.float32)


@pytest.mark.parametrize("n,d,k,full", [
    (30_000, 48, 640, False),
    (9_000, 64, 8, False),
    (20_000, 100, 1030, True),     # d % 8 != 0: padded filter copy
    (6_000, 30, 17, True),         # rows of 60 bytes: generic accumulate
    (5_000, 768, 300, True),
])
def test_kmeans_on_an_f16_store(gpu, n, d, k, full):
    x = f16(_mixture(n, d, min(k, 50), 100 + n % 97 + d))
    idx = gpu.Index(gpu.f32_to_f16_bits(x), gpu.F16, 1)
    a, c, obj = idx.kmeans(k, niter=5, full_lloyd=full)
    ao, co, oo = oracle.kmeans(x, k, niter=5, full_lloyd=full)
    assert np.array_equal(a, ao), f"{(a != ao).sum()} of {n} assignments differ"
    assert np.array_equal(bits(c), bits(co))
    assert np.allclose(obj, oo, rtol=1e-5)
    idx.close()


def test_kmeans_f16_empty_clusters_and_ties(gpu):
    rng = np.random.default_rng(21)
    x = f16(gauss(1500, 16, 22, normalize=False))
    x[rng.random(1500) < 0.7] = x[0]
    idx = gpu.Index(gpu.f32_to_f16_bits(x), gpu.F16, 1)
    a, c, obj = idx.kmeans(24, niter=6, full_lloyd=True)
    ao, co, oo = oracle.kmeans(x, 24, niter=6, full_lloyd=True)
    assert np.array_equal(a, ao) and np.array_equal(bits(c), bits(co))
    idx.close()
    g = grid(4000, 6, 11)
    idx = gpu.Index(gpu.f32_to_f16_bits(g), gpu.F16, 1)
    a, c, obj = idx.kmeans(40, niter=4, full_lloyd=True)
    ao, co, oo = oracle.kmeans(g, 40, niter=4, full_lloyd=True)
    assert np.array_equal(a, ao) and np.array_equal(bits(c), bits(co))
    idx.close()


PAIRS = r"""
import json, sys
import numpy as np
sys.path.insert(0, %r); sys.path.insert(0, %r + "/tests")
import oracle
from helpers import gauss
from lotus_b200 import _native as nv
out = {}
for n, d in ((3000, 96), (1500, 200), (257, 64)):
    x = gauss(n, d, 30 + n)
    rng = np.random.default_rng(n)
    src, dst = rng.choice(n, n // 20, replace=False), rng.choice(n, n // 20, replace=False)
    x[dst] = x[src] + 0.15 * gauss(len(src), d, 31 + n, normalize=False) / np.sqrt(d)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    xb = nv.f32_to_f16_bits(x)
    idx = nv.Index(xb, nv.F16, 0)
    oi, oj, cnt = oracle.threshold_pairs(nv.f16_bits_to_f32(xb), 0.9)
    pi, pj = idx.threshold_pairs(0.9)
    out[f"{n}x{d}"] = {"pairs": int(cnt), "same": bool(np.array_equal(pi, oi) and np.array_equal(pj, oj))}
    idx.close()
print(json.dumps(out))
""" % (ROOT, ROOT)


@pytest.mark.parametrize("two_cta", ["1", "0"])
def test_threshold_pairs_on_an_f16_store(two_cta):
    r = subprocess.run([sys.executable, "-c", PAIRS], capture_output=True, text=True, timeout=300,
                       env=dict(os.environ, B2_PAIR_2CTA=two_cta))
    assert r.returncode == 0, r.stderr[-3000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    for name, v in res.items():
        assert v["pairs"] > 5 and v["same"], (name, v)


def test_device_hand_off_of_fp16_tensors(gpu, tmp_path):
    import torch

    from lotus_b200.vs import B200VS
    dev = torch.device("cuda", 0)
    x, q = gauss(6000, 128, 40), gauss(200, 128, 41)
    xt, qt = torch.from_numpy(x).to(dev).half(), torch.from_numpy(q).to(dev).half()
    for fs, metric in (("Flat", 0), ("SQfp16", 1)):
        vs = B200VS(factory_string=fs, dtype="f16" if fs == "Flat" else "auto", metric=metric)
        vs.index(None, xt, str(tmp_path / fs))
        assert vs.b2_index.dtype == gpu.F16
        gpu.stats_reset()
        out = vs(qt, 10)
        Do, Io = oracle.knn(f16(x), f16(q), 10, metric)
        assert np.array_equal(out.indices, Io) and np.array_equal(bits(out.distances), bits(Do))
        assert gpu.stats()["filter_launches"] >= 1
        out = vs(q, 10)                                      # host fp32 queries
        Do, Io = oracle.knn(f16(x), q, 10, metric)
        assert np.array_equal(out.indices, Io) and np.array_equal(bits(out.distances), bits(Do))
        vs.close()
    bad = xt.clone()
    bad[3, 3] = float("inf")
    with pytest.raises(ValueError, match="fp16"):
        B200VS(dtype="f16").index(None, bad, str(tmp_path / "bad"))


@pytest.mark.parametrize("metric", [0, 1])
@pytest.mark.parametrize("qt", ["f16", "f32"])
def test_staged_sharded_search_on_an_f16_store(gpu, metric, qt):
    import torch
    dev = torch.device("cuda", 0)
    x, q = gauss(24_000, 96, 200 + metric), gauss(6000, 96, 201)
    k, G = 32, 3
    xb = gpu.f32_to_f16_bits(x)
    qa, code, qf = queries(gpu, q, qt)
    q_dev = torch.from_numpy(qa.view(np.int16) if qa.dtype == np.uint16 else qa).to(dev)
    shards = [gpu.Index(np.ascontiguousarray(xb[g * 8000:(g + 1) * 8000]), gpu.F16, metric) for g in range(G)]
    st = torch.cuda.current_stream().cuda_stream
    lowers = [torch.empty(len(q), dtype=torch.float32, device=dev) for _ in range(G)]
    j = -(-k // G)
    for s, lo in zip(shards, lowers):
        s.search_stage1_dev(q_dev.data_ptr(), len(q), k, code, j, lo.data_ptr(), stream=st)
    hint = torch.stack(lowers).min(dim=0).values.contiguous()
    assert bool(torch.isfinite(hint).any().item())
    packed = torch.empty((G, len(q), k), dtype=torch.int64, device=dev)
    for g, s in enumerate(shards):
        s.search_stage2_packed_dev(hint.data_ptr(), packed[g].data_ptr(), stream=st)
    out_s = torch.empty((len(q), k), dtype=torch.float32, device=dev)
    out_i = torch.empty((len(q), k), dtype=torch.int64, device=dev)
    gpu.merge_topk_packed_dev(packed.data_ptr(), np.arange(G) * 8000, G, len(q), k, metric, 0, out_s.data_ptr(), out_i.data_ptr(), stream=st)
    Do, Io = oracle.knn(f16(x), qf, k, metric)
    assert np.array_equal(out_i.cpu().numpy(), Io)
    assert np.array_equal(bits(out_s.cpu().numpy()), bits(Do))
    for s in shards:
        s.close()


def test_reference_sq_operator_replay(gpu, tmp_path):
    from lotus_b200.vs import B200VS
    from sq_replay import replay_reference_sq_calls
    vs = B200VS(factory_string="SQfp16")
    assert replay_reference_sq_calls(vs, str(tmp_path)) > 0
    vs.close()
