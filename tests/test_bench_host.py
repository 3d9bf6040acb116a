"""Host-side pieces of bench.py that do not need a GPU: the committed ncu traffic lookup, the algorithmic byte counts
(DESIGN.md section 4), the clock sampler's behaviour on a box without NVML and the --dump-outputs writer; one GPU test
runs bench.py end to end with --dump-outputs."""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench


def test_traffic_lookup_reads_the_committed_capture():
    t = bench.measured_traffic("srfrd_gemm_tn")
    assert isinstance(t, int) and 1e6 < t < 200e6           # DRAM bytes per launch of the dominant kernel at C2 (packed rows: ~7 MB)
    assert bench.measured_traffic("srfrd_catalogue_topk") > 1e9
    assert bench.measured_traffic("no_such_kernel") is None
    for k in ("srfrd_score_loss_fused@C3", "srfrd_embed_bwd@C3", "srfrd_adam_step@C3", "srfrd_embed_ln_fwd@C3"):
        assert bench.measured_traffic(k) > 1e9              # catalogue-scale captures of K4 / K5 / K7 / K1


def test_algorithmic_bytes_of_the_gemm_variants():
    from srfrd_b200._lib import GemmEpilogue
    M, N, K = 204800, 80, 80

    def args(**kw):
        ep = GemmEpilogue()
        for k, v in kw.items():
            setattr(ep, k, v)
        return [None, 0, None, 0, M, N, K, ctypes.byref(ep), None]
    base = M * K * 2 + N * K * 2 + M * N * 2
    b, f = bench.algorithmic_bytes("srfrd_gemm_tn", args(out_bf16=1), 0.1)
    assert b == base and f == 2.0 * M * N * K
    b, _ = bench.algorithmic_bytes("srfrd_gemm_tn", args(out_bf16=1, residual=1, row_ids=1), 0.1)
    assert b == base + M * N * 2 + M * 8
    b, _ = bench.algorithmic_bytes("srfrd_gemm_tn", args(out_bf16=1, residual=1, ln_out_bf16=1, ln_stats=1), 0.1)
    assert b == base + M * N * 2 + M * N * 2 + M * 8          # + LayerNorm output and (mean, rstd)
    b, _ = bench.algorithmic_bytes("srfrd_gemm_wgrad", [None, 0, None, 0, M, 80, 80], 0.1)
    assert b == M * 160 * 2 + 80 * 80 * 4


def test_clock_sampler_degrades_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    s = bench.ClockSampler(0)
    s.start()
    out = s.stop()
    assert set(out) >= {"sm_mhz", "sm_max_mhz", "reasons", "samples"} and out["samples"] == 0


def test_write_outputs_saves_float_arrays_within_the_limit(tmp_path):
    d = tmp_path / "out"
    n = bench.write_outputs(str(d), {"loss": torch.tensor([0.25]), "ids": torch.tensor([[3, 2 ** 40 + 1]]),
                                     "h": torch.ones(4, dtype=torch.bfloat16), "x": np.arange(3.0)})
    got = {f[:-4]: np.load(d / f) for f in os.listdir(d)}
    assert set(got) == {"loss", "ids", "h", "x"} and n == sum(a.nbytes for a in got.values())
    assert got["loss"].dtype == np.float32 and got["h"].dtype == np.float32 and got["x"].dtype == np.float64
    assert got["ids"].dtype == np.float64 and got["ids"].tolist() == [[3.0, float(2 ** 40 + 1)]]
    with pytest.raises(ValueError, match="limit"):
        bench.write_outputs(str(tmp_path / "big"), {"a": np.zeros(4, np.float32),
                                                    "b": np.zeros(bench.DUMP_LIMIT // 8, np.float64)})
    assert not (tmp_path / "big").exists()


@pytest.mark.gpu
def test_bench_dump_outputs_are_the_same_every_run(tmp_path):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    runs = []
    for i in range(2):
        d = tmp_path / f"dump{i}"
        r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", "50", "--warmup", "2",
                            "--no-extras", "--no-cpu", "--dump-outputs", str(d)], cwd=tmp_path, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-3000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 50
        runs.append({f[:-4]: np.load(d / f) for f in os.listdir(d)})
    got = runs[0]
    assert set(got) == {"train_loss", "catalogue_scores", "catalogue_ids", "catalogue_encode_scores", "catalogue_encode_ids"}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= bench.DUMP_LIMIT
    assert got["train_loss"].shape == (1,) and np.isfinite(got["train_loss"]).all() and got["train_loss"][0] > 0
    for pre in ("catalogue", "catalogue_encode"):
        s, ids = got[pre + "_scores"], got[pre + "_ids"]
        assert s.shape == ids.shape == (16384, 10)
        assert (np.diff(s, axis=1) <= 0).all() and ids.min() >= 0 and ids.max() <= 1_000_000
    # same arguments, same inputs: the catalogue passes are exact, the loss (float-atomic gradient sums) agrees to rounding
    for k, a in got.items():
        if k == "train_loss":
            np.testing.assert_allclose(runs[1][k], a, rtol=1e-5)
        else:
            assert np.array_equal(runs[1][k], a), k
