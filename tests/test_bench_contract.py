"""bench.py's JSON-line contract, as far as it can be checked without a GPU: the reference arm (`--impl reference`, the CPU
restatement of DeepFM/deepfm.py:178-235) really runs here, and the GPU arm's `config` comes from the same builder."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
             "dtype", "data", "config", "e2e", "gpu_launches"}


def _reference_line(extra=(), env=None):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "deepfm_small",
                          "--steps", "2", "--warmup", "1", *extra], capture_output=True, text=True, timeout=600,
                         env={**os.environ, **(env or {})})
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    return lines


def test_reference_arm_line_has_the_contract_keys_and_the_gpu_arms_config():
    import bench
    lines = _reference_line()
    assert len(lines) == 1                                          # ONE JSON line
    d = json.loads(lines[0])
    assert BASE_KEYS | {"impl", "cpu_baseline"} <= set(d)
    assert d["impl"] == "reference" and d["metric"] == "ctr_fwd_bwd_samples_per_sec" and d["unit"] == "samples/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["gpu_launches"] == 0
    assert d["steps"] == 2 and d["warmup"] >= 3                     # the timing rules ask for W >= 3
    assert d["value"] > 0 and abs(d["value"] - d["config"]["global_batch"] / (d["ms_per_step"] * 1e-3)) <= 1e-6 * d["value"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # the config the GPU arm prints for the same workload at N = 1 (bench.run_deepfm builds it with the same function)
    cfg = bench.DEEPFM["deepfm_small"]
    assert cb["same_config_as_gpu_arm"] is True
    assert d["config"] == bench.deepfm_config("deepfm_small", cfg["model"], cfg["B"], 1, cfg["F"], cfg["D"], cfg["rows_per_field"],
                                              "uniform int64", cfg["id_batches"])


def test_reference_arm_under_torchrun_env_prints_on_rank_0_only():
    assert _reference_line(("--gpus", "2"), env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}) == []
    (line,) = _reference_line(("--gpus", "2"), env={"RANK": "0", "WORLD_SIZE": "2", "LOCAL_RANK": "0"})
    d = json.loads(line)
    assert d["n_gpus"] == 2 and "single-process" in d["config"]["note"]


def test_dump_outputs_writes_float32_whole_and_one_seeded_row_sample(tmp_path):
    import numpy as np
    import torch
    import bench
    g = torch.Generator().manual_seed(0)
    B, F, D = 8192, 40, 32                                             # 2 x 42 MB of tile / row_grads: must be sampled
    fm2, tile = torch.randn((B, 1), generator=g), torch.randn((B, F, D), generator=g)
    tile[:, 0, 0] = torch.arange(B)                                    # each row says which it is
    grads = tile * 2
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), whole={"fm2": fm2}, per_sample={"tile": tile, "row_grads": grads})
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["fm2.npy", "row_grads.npy", "tile.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 * 10 ** 6
    a = {f: np.load(tmp_path / "a" / f) for f in files}
    for f in files:
        assert a[f].dtype == np.float32 and np.array_equal(a[f], np.load(tmp_path / "b" / f))
    assert np.array_equal(a["fm2.npy"], fm2.numpy())
    n = a["tile.npy"].shape[0]
    assert 0 < n < B and a["tile.npy"].shape == a["row_grads.npy"].shape == (n, F, D)
    rows = a["tile.npy"][:, 0, 0].astype(np.int64)
    assert (np.diff(rows) > 0).all() and np.array_equal(a["tile.npy"], tile.numpy()[rows])
    assert np.array_equal(a["row_grads.npy"], grads.numpy()[rows])   # the same rows of every sampled output


def test_bench_rejects_zero_steps_and_dumps_it_cannot_make():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"], ["--workload", "dcn_cfg2", "--dump-outputs", "x"],
                  ["--workload", "deepfm_small_sharded", "--dump-outputs", "x"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=300)
        assert out.returncode == 2 and "error:" in out.stderr and not out.stdout, extra


@pytest.mark.gpu
def test_bench_dump_outputs_are_the_last_timed_step_and_repeat(tmp_path):
    """Same arguments -> the same dumped outputs; one more timed step -> the last step ran on the next id batch."""
    import numpy as np

    def run(steps, d):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "deepfm_small", "--steps", str(steps),
                              "--warmup", "3", "--no-extra", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / d)],
                             capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-2000:]
        (line,) = [l for l in out.stdout.splitlines() if l.startswith("{")]
        assert json.loads(line)["steps"] == steps
        return {f: np.load(tmp_path / d / f) for f in ("fm2.npy", "tile.npy", "row_grads.npy")}

    a, b, c = run(5, "a"), run(5, "b"), run(6, "c")
    for f in a:
        assert a[f].dtype == np.float32 and np.isfinite(a[f]).all() and np.array_equal(a[f], b[f]), f
    assert a["fm2.npy"].shape == (8192, 1) and not np.array_equal(a["fm2.npy"], c["fm2.npy"])


def test_algorithmic_bytes_match_survey_8d():
    import bench
    fwd, bwd = bench.bytes_per_sample(40, 32)
    assert fwd + bwd == 40 * (8 + 20 * 32) + 8 == 25928             # SURVEY 8(d): F*(8 + 20*D) + 8 per sample at config 5
    assert fwd == 40 * (8 + 2 * 32 * 4) + 4 and bwd == 40 * 3 * 32 * 4 + 4


def test_cpu_baseline_model_computes_the_same_function_as_the_gpu_arm():
    """oracle/torch_cpu_model.py (what `--impl reference` and cpu_baseline time) against the NumPy oracle: the FM2 logit, the
    dense(1) head over the concatenated embeddings, the loss, and the sparse table gradients of one step."""
    import numpy as np
    import torch
    from oracle import layers_np as O, torch_cpu_model as M
    F, D, rows, B = 5, 8, 50, 64
    m = M.DeepFMLookupFM2CPU(F, D, rows, seed=3)
    g = torch.Generator().manual_seed(0)
    ids = torch.randint(0, rows, (B, F), generator=g)
    labels = (torch.rand((B, 1), generator=g) < 0.3).float()
    logit, fm2 = m.forward(ids)
    table = np.concatenate([t.detach().numpy() for t in m.tables])
    off = np.arange(F + 1, dtype=np.int64) * rows
    e = O.embedding_lookup(table, ids.numpy(), off).astype(np.float64)
    ref_fm2 = O.fm2_fwd(e)
    assert np.abs(fm2.detach().numpy() - ref_fm2).max() <= 1e-5 * np.abs(ref_fm2).max()
    ref_logit = ref_fm2 + e.reshape(B, F * D) @ m.w_deep.detach().numpy().astype(np.float64)
    assert np.abs(logit.detach().numpy() - ref_logit).max() <= 1e-5 * np.abs(ref_logit).max()
    loss = m.step(ids, labels)
    y = labels.numpy().astype(np.float64)
    want_loss = np.mean(np.maximum(ref_logit, 0) - ref_logit * y + np.log1p(np.exp(-np.abs(ref_logit))))   # TF's stable form
    assert abs(loss - want_loss) <= 1e-5 * abs(want_loss)
    d_logit = (1 / (1 + np.exp(-ref_logit)) - y) / B
    want = O.fm2_bwd(e, d_logit[:, 0]) + d_logit[:, :, None] * m.w_deep.detach().numpy().astype(np.float64).reshape(1, F, D)
    dense = O.embedding_lookup_bwd_dense(F * rows, ids.numpy(), off, want)
    got = np.concatenate([t.grad.to_dense().numpy() for t in m.tables])
    assert m.tables[0].grad.is_sparse                                  # IndexedSlices-like gradients, as in the reference
    assert np.abs(got - dense).max() <= 1e-5 * np.abs(dense).max()


def test_cpu_layer_baselines_compute_the_references_chains():
    """oracle/torch_cpu_layers.py (the CPU baselines of configs 2-4) against the NumPy oracle, which itself is pinned by the
    fixtures executed from the reference's layer files."""
    import numpy as np
    import torch
    from oracle import layers_np as O, torch_cpu_layers as C
    g = torch.Generator().manual_seed(5)
    rel = lambda a, b: np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)          # noqa: E731

    dcn = C.DCNCrossCPU(F=4, D=8, L=3, rows=30, seed=1)
    ids, gout = dcn.make_batch(17, g)
    table = np.concatenate([t.detach().numpy() for t in dcn.tables]); off = np.arange(5, dtype=np.int64) * 30
    x0 = O.embedding_lookup(table, ids.numpy(), off).reshape(17, 32).astype(np.float64)
    ws = np.stack([w.detach().numpy()[:, 0] for w in dcn.wl]).astype(np.float64); bs = np.stack([b.detach().numpy()[:, 0] for b in dcn.bl]).astype(np.float64)
    assert rel(dcn.forward(ids).detach().numpy(), O.cross_stack_fwd(x0, ws, bs)[-1]) <= 1e-5
    dcn.step(ids, gout)
    dx0, dws, dbs = O.cross_stack_bwd(x0, ws, bs, gout.numpy().astype(np.float64))[:3]
    assert rel(np.stack([w.grad.numpy()[:, 0] for w in dcn.wl]), dws) <= 1e-5 and dcn.tables[0].grad.is_sparse

    xd = C.XDeepFMCinCPU(F=5, D=4, maps=(6, 3), rows=20, seed=2)
    ids, gp = xd.make_batch(9, g)
    table = np.concatenate([t.detach().numpy() for t in xd.tables]); off = np.arange(6, dtype=np.int64) * 20
    x0 = O.embedding_lookup(table, ids.numpy(), off).astype(np.float64)
    filts = [f.detach().numpy()[0].astype(np.float64) for f in xd.filters]
    xs, pooled = O.cin_stack_fwd(x0, filts)
    got_pooled, got_last = xd.forward(ids)
    assert rel(got_pooled.detach().numpy(), pooled) <= 1e-5 and rel(got_last.detach().numpy(), xs[-1]) <= 1e-5
    xd.step(ids, gp)
    assert all(f.grad is not None and float(f.grad.abs().max()) > 0 for f in xd.filters)

    for soft in (False, True):
        din = C.DINAttentionCPU(T=7, H=8, rows=25, seed=3, is_softmax=soft)
        hist, tgt, lens, go = din.make_batch(11, g)
        lens[0] = 0; hist[0] = -1                                                 # an empty history (din_attention.py:52's case)
        tab = din.table.detach().numpy().astype(np.float64)
        keys = tab[np.where(hist.numpy() >= 0, hist.numpy(), 25)]
        assert np.all(keys[0] == 0)
        ref = O.din_attention_fwd(tab[tgt.numpy()[:, 0]], keys, lens.numpy(), *[p.detach().numpy().astype(np.float64) for p in din.params()[1:]],
                                  is_softmax=soft)
        assert rel(din.forward(hist, tgt, lens).detach().numpy(), ref) <= 1e-5
        din.step(hist, tgt, lens, go)
        assert din.table.grad.is_sparse and din.w1.grad is not None


def test_reference_arm_for_a_layer_workload_and_the_guard_around_the_cpu_baselines():
    import bench
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "din_cfg4", "--steps", "2",
                          "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    (line,) = [l for l in out.stdout.splitlines() if l.startswith("{")]
    d = json.loads(line)
    assert BASE_KEYS | {"impl", "cpu_baseline"} <= set(d) and d["impl"] == "reference"
    assert d["config"]["workload"] == "din_cfg4" and d["config"]["B"] == 4096 and d["cpu_baseline"]["same_config_as_gpu_arm"] is True
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] == "port" and d["steps"] == 2
    # inside the GPU arm a failing CPU baseline must not cost the line: it is reported in place of the number
    assert "unavailable" in bench.safe_cpu_layer_baseline("no_such_config", 1.0)
    assert set(bench.CPU_LAYER_SAMPLE_B) <= set(bench.LAYER_WORKLOADS) == set(bench.LAYER_MODELS)
