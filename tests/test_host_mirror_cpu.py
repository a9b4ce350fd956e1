"""CPU-only tests of the host-side mirror's pure-NumPy pieces (no device calls): the TToperator algebra used by the time
steppers, `ttv_to_diag_tto`, `bubble_sort_swaps`, the `QTTvector` wrapper, batch sharding helpers — each against the oracle's
restatement of the same reference function."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import ttn_b200 as t      # noqa: E402  (importing does not need a GPU; device calls would raise)
import ttn_oracle as o    # noqa: E402


def _mirror_tto(A):
    return t.TToperator(A.N, [c.copy() for c in A.tto_vec], A.tto_dims, list(A.tto_rks))


def _dense(A):
    return o.tto_to_matrix(o.TToperator(A.N, list(A.tto_vec), tuple(A.tto_dims), list(A.tto_rks)))


def test_operator_algebra_of_the_steppers_vs_oracle():
    # tt_operators.jl:524-532 (id_tto), tt_operations.jl:71-96 (+), 268-278 (scalar *): I - h A as built by euler.jl:99-143
    d, h = 5, 0.01
    A = _mirror_tto(o.laplace_dd(d))
    M = t.tto_add(t.id_tto(d), t.tto_scale(-h, A))
    assert np.allclose(_dense(M), np.eye(2 ** d) - h * o.tto_to_matrix(o.laplace_dd(d)), atol=1e-14)
    Mo = o.tto_add(o.id_tto(d), o.tto_scale(-h, o.laplace_dd(d)))
    assert list(M.tto_rks) == list(Mo.tto_rks)
    for a, b in zip(M.tto_vec, Mo.tto_vec):
        assert np.array_equal(a, b)
    Mc = t.tto_scale(1j, A)
    assert Mc.tto_vec[0].dtype == np.complex128 and np.allclose(_dense(Mc), 1j * o.tto_to_matrix(o.laplace_dd(d)))
    with pytest.raises(AssertionError):
        t.tto_add(t.id_tto(4), t.id_tto(5))


def test_ttv_to_diag_tto_vs_dense():
    # tt_operations.jl:318-338; test_tt_operations.jl:4-37
    rng = np.random.default_rng(2)
    x = o.rand_tt((3, 2, 2), 2, rng=rng)
    D = t.ttv_to_diag_tto(x)
    assert tuple(D.tto_dims) == tuple(x.ttv_dims) and list(D.tto_rks) == list(x.ttv_rks)
    assert np.allclose(_dense(D), np.diag(o.ttv_to_tensor(x).reshape(-1)), atol=1e-14)


def test_bubble_sort_swaps_and_qttvector_wrapper():
    # qtt_tools.jl:704-718, 370-379
    rng = np.random.default_rng(3)
    for _ in range(10):
        perm = [int(v) for v in rng.permutation(9)]
        assert t.bubble_sort_swaps(perm) == o.bubble_sort_swaps(perm)
    x = o.rand_tt((2,) * 6, 2, rng=rng)
    q = t.QTTvector(x, 3, 2, "interleaved")
    assert (q.n_dims, q.bits_per_dim, q.ordering, q.N) == (3, 2, "interleaved", 6) and q.ttv_rks == list(x.ttv_rks)
    with pytest.raises(AssertionError):
        t.QTTvector(x, 4, 2, "serial")


def test_increase_ranks_zero_padding_and_noise_branches():
    """increase_ranks (src/tt_tools.jl:443-489) in the host mirror: noise = 0 equals the oracle's zero padding bit for bit and
    leaves the represented tensor unchanged; noise != 0 fills exactly the new blocks of the three branches of
    increase_ranks_noise with `noise` x (orthonormal columns or rows), the old block untouched (tt_tools.jl:446-458)."""
    rng = np.random.default_rng(5)
    dims = (2, 3, 2, 2)
    x = o.rand_tt(dims, 2, rng=rng)
    xm = t.TTvector(x.N, x.ttv_vec, x.ttv_dims, x.ttv_rks, x.ttv_ot)
    z = t.increase_ranks(xm, 4)
    zo = o.increase_ranks(x, 4)
    assert z.ttv_rks == zo.ttv_rks == o.r_and_d_to_rks([1, 4, 4, 4, 1], dims, rmax=4)
    for a, b in zip(z.ttv_vec, zo.ttv_vec):
        assert np.array_equal(a, b)
    with pytest.raises(AssertionError):
        t.increase_ranks(xm, 2)                               # "New bond dimension too low", tt_tools.jl:483
    eps = 1e-3
    y = t.increase_ranks(xm, 4, noise=eps, rng=np.random.default_rng(7))
    assert y.ttv_rks == z.ttv_rks and y.ttv_ot == [0] * x.N
    for i, (c, c0) in enumerate(zip(y.ttv_vec, x.ttv_vec)):
        n, a, b = c0.shape
        _, rkm, rk = c.shape
        assert np.array_equal(c[:, :a, :b], c0)
        if rkm == a and rk > b:                               # new right block: orthonormal columns of an (n rkm) x (rk - b) matrix
            Q = c[:, :, b:].reshape((n * rkm, rk - b), order="F") / eps
            assert np.allclose(Q.T @ Q, np.eye(rk - b), atol=1e-12)
        elif rk == b and rkm > a:                             # new left block: orthonormal rows
            Q = np.reshape(np.asfortranarray(c[:, a:, :]), (rkm - a, n * rk), order="F") / eps      # undoes Julia's column-major reshape
            assert np.allclose(Q @ Q.T, np.eye(rkm - a), atol=1e-12)
        elif rk > b and rkm > a:                              # corner block only; the off-diagonal new blocks stay zero
            assert np.all(c[:, :a, b:] == 0) and np.all(c[:, a:, :b] == 0)
            Q = c[:, a:, b:].reshape(((rkm - a) * n, rk - b), order="F") / eps
            assert np.allclose(Q.T @ Q, np.eye(rk - b), atol=1e-12)
    dz = o.ttv_to_tensor(o.TTvector(x.N, y.ttv_vec, dims, y.ttv_rks, [0] * x.N)) - o.ttv_to_tensor(x)
    assert 0 < np.linalg.norm(dz) < 50 * eps * np.linalg.norm(o.ttv_to_tensor(x))
    qz = t.rand_orthogonal(5, 3, np.random.default_rng(1), np.complex128)
    assert qz.shape == (5, 3) and np.allclose(qz.conj().T @ qz, np.eye(3), atol=1e-12)


def test_batch_sharding_helpers():
    # SURVEY.md section 8(e): vectors split evenly over the ranks, no data-path collective
    for n, world in ((4096, 8), (10, 3), (5, 8), (0, 2)):
        parts = [t.shard_batch(n, r, world) for r in range(world)]
        idx = [i for first, count in parts for i in range(first, first + count)]
        assert idx == list(range(n))
        sizes = [count for _, count in parts]
        assert max(sizes) - min(sizes) <= 1


def test_device_calls_fail_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    rng = np.random.default_rng(4)
    x = o.rand_tt((2, 2, 2), 2, rng=rng)
    with pytest.raises(Exception):
        t.tt_compress_(x, 1)
    with pytest.raises(Exception):
        t.hadamard_ttm(x, x)


def test_committed_bench_line_follows_the_contract():
    """`profiles/bench_end_of_round_r01.json` is the line `python bench.py` printed on a B200 at the end of the round: it must
    carry every key of the bench contract (metric/config of BASELINE.json, e2e with host<->device bytes, roofline against the
    measured peak, CPU baseline with its sample, clocks sampled under load, launch count)."""
    import json
    d = json.load(open(os.path.join(ROOT, "profiles", "bench_end_of_round_r01.json")))
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "e2e", "roofline", "cpu_baseline", "clocks", "gpu_launches"):
        assert k in d, k
    assert d["n_gpus"] == 1 and d["warmup"] >= 3 and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["dtype"] == "f64" and d["data"] == "synthetic" and "cfg2" in d["config"]["workload"] and "model" not in d["config"]
    assert abs(d["value"] - 1000.0 / d["ms_per_step"]) < 1e-6 * d["value"]
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] > 9e7 and e["d2h_bytes_per_step"] > 0 and 0 < e["value"] <= d["value"] * 1.02
    r = d["roofline"]
    assert r["bound"] in ("hbm", "tensor") and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and r["unit"] in ("GB/s", "TFLOP/s")
    c = d["cpu_baseline"]
    assert c["kind"] in ("port", "reference") and c["cores"] >= 1 and c["sample"] and c["value"] > 0
    assert d["gpu_launches"] > 0
    assert d["clocks"]["samples"] >= 1 and not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}


def test_committed_round2_bench_line_follows_the_contract():
    """`profiles/bench_end_of_round_r02.json`: the line `python bench.py --steps 20 --warmup 5` printed on one B200 at the end of
    round 2.  Headline = cfg5 (4096 ComplexF64 QTT vectors, apply + tt_compress!), strong scaling over the ranks; value and
    ms_per_step must agree, the end-to-end leg must move every step's inputs and results over PCIe, the roofline must name its
    dominant kernel family with achieved / peak, and no Gram-path fallback may hide inside the timed region."""
    import json
    d = json.load(open(os.path.join(ROOT, "profiles", "bench_end_of_round_r02.json")))
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "e2e", "roofline", "cpu_baseline", "clocks", "gpu_launches", "extras"):
        assert k in d, k
    assert d["metric"] == "tt_rounding sweeps/s" and d["unit"] == "sweeps/s"
    assert d["n_gpus"] == 1 and d["warmup"] >= 3 and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["dtype"] == "c128" and d["data"] == "synthetic" and d["scaling"] == "strong"
    c = d["config"]
    assert "cfg5" in c["workload"] and "model" not in c and c["total_vectors"] == 4096 and c["d"] == 30 and c["rank"] == 64
    assert c["gram_path_fallbacks_in_timed_region"] == 0 and c["out_max_rank"] == 64
    assert abs(d["value"] - 4096 / (d["ms_per_step"] * 1e-3)) < 1e-6 * d["value"]
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] > 1e10 and e["d2h_bytes_per_step"] > 1e10 and 0 < e["value"] <= d["value"] * 1.02
    assert abs(e["value"] - 4096 / (e["ms_per_step"] * 1e-3)) < 1e-6 * e["value"]
    r = d["roofline"]
    assert r["bound"] == "tensor" and r["unit"] == "TFLOP/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert set(r["families"]) == {"gemm", "jacobi"} and all(0 < f["frac"] < 1 for f in r["families"].values())
    assert 0 < r["whole_step"]["executed"]["frac"] < 1
    b = d["cpu_baseline"]
    assert b["kind"] == "port" and b["cores"] >= 1 and b["sample"] and 0 < b["reference_faithful_value"] < b["value"] < d["value"]
    assert d["gpu_launches"] > 1000
    assert d["clocks"]["samples"] >= 1 and not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    x = d["extras"]
    for k in ("cfg2_sweeps_per_s", "matvec_cfg4_tflops", "dmrg_sweep_s", "mals_cfg3_heat_s", "mals_cfg3_heat_max_rank"):
        assert k in x, k
    assert x["mals_cfg3_heat_max_rank"] == 128


def test_bench_helpers_without_a_gpu():
    """Pieces of bench.py that do not need a device: the committed ncu capture feeds roofline.traffic, the NUMA binding is a no-op
    without NVML, the cfg5 config names the workload and carries no model keys, and both arms describe the same config."""
    sys.path.insert(0, ROOT)
    import bench
    tr = bench.captured_traffic()
    assert tr is not None and 3e7 < tr < 2e8            # 296 lower triangles of 128 x 128 ComplexF64 = 39 MB + what L2 lets through
    assert bench.bind_to_gpu_numa(0) is None or isinstance(bench.bind_to_gpu_numa(0), int)
    c1, c8 = bench.cfg5_config(1, 296), bench.cfg5_config(8, 296)
    assert "cfg5" in c1["workload"] and "model" not in c1 and c1["total_vectors"] == bench.TOTAL5 == 4096
    assert {k for k in c1} == {k for k in c8}
    rks, Rk = bench.cfg5_ranks()
    assert max(rks) == 64 and max(Rk) == 4 and len(rks) == bench.D5 + 1 == 31
    m = bench.cfg5_flop_model()
    assert 1.3e10 < m["total"] < 1.5e10                 # SURVEY.md section 8(d)-5: ~13-14 GFLOP per vector
    # --dump-outputs: each sampled vector is found exactly once over the ranks, worker threads and chunks, and the sample stays
    # under 64 MB as float64 (rounded ranks <= 64, 16 bytes per complex entry)
    for world, chunk, nw in ((1, 296, 3), (8, 100, 2), (3, 7, 4)):
        found = []
        for r in range(world):
            first, nvec = t.shard_batch(bench.TOTAL5, r, world)
            ids, plan = bench.dump_plan(first, nvec, chunk, nw)
            found += [g for wi, pos in plan.items() for j, cols in pos.items() for b, g in cols
                      if first + (j * nw + wi) * chunk + b == g and b < chunk]
        assert sorted(found) == list(ids) and len(set(ids)) == bench.DUMP_SAMPLE
    per_vector = sum(2 * min(rks[k], 64) * min(rks[k + 1], 64) * 16 for k in range(bench.D5))
    assert bench.DUMP_SAMPLE * per_vector < 64e6
