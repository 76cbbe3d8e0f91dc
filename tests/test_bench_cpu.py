"""CPU checks of bench.py's host-side pieces: the synthetic workload is the one SURVEY.md 8d prescribes and is reproducible,
the roofline work model follows BASELINE.md 4, every tool script at least compiles."""
import glob
import os
import py_compile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_workload_is_the_survey_config_and_reproducible():
    b = _bench()
    t1, n1 = b.make_workload(256, b.SEED, 0)
    t2, n2 = b.make_workload(256, b.SEED, 0)
    assert n1 == n2 and all(torch.equal(a, c) for a, c in zip(t1, t2))
    assert len(t1) == 256 and all(16 <= int(t.numel()) < 160 for t in t1) and all(75 <= n < 1000 for n in n1)
    assert all(int(t.min()) >= 1 and int(t.max()) < 255 for t in t1)
    t3, n3 = b.make_workload(256, b.SEED, 1)                 # another rank owns other utterances (weak scaling)
    assert n3 != n1


def test_stage_work_model_matches_the_baseline_formulas():
    b = _bench()
    texts = [torch.zeros(100, dtype=torch.long)]
    w = b.stage_work(texts, [500])
    n, s0 = 500.0, 138.0
    kv = 122880.0
    assert np.isclose(w["t3_bytes"], n * 1.0234e9 + 2 * (s0 * n + n * (n + 1) / 2) * kv + 2 * n * kv)
    T = 2.0 * (500 + 250)
    assert np.isclose(w["flow_flops"], 113.2e6 * 750 + 90.1e3 * 750 * 750 + 10 * 2 * T * (132161536.0 + 114688.0 * T))
    assert np.isclose(w["hift_flops"], 612.3e6 * 1000) and np.isclose(w["hift_bytes"], 0.30e6 * 1000)


def test_dump_outputs_sample_is_fixed_and_bounded(tmp_path):
    """--dump-outputs: the same utterances every run, whole waveforms within 64 MB even when every utterance reaches its
    budget, float32 waveforms + float64 lengths of the whole batch."""
    b = _bench()
    for budget_max in (1000, 75, 20000):
        idx = b.dump_sample(256, budget_max)
        assert idx == b.dump_sample(256, budget_max) and idx == sorted(set(idx)) and 0 <= idx[0] and idx[-1] < 256
        assert len(idx) == 1 or len(idx) * budget_max * 960 * 4 + 256 * 8 <= b.DUMP_BYTES
    assert len(b.dump_sample(256, 1000)) == 16 and b.dump_sample(3, 10) == [0, 1, 2]
    wavs = [torch.full((960 * n,), float(n)) for n in (5, 0, 7, 3)]
    b.dump_outputs(str(tmp_path), wavs, 10)
    assert np.load(tmp_path / "wav_lengths.npy").tolist() == [4800.0, 0.0, 6720.0, 2880.0]
    for i in b.dump_sample(4, 10):
        w = np.load(tmp_path / f"wav_{i:03d}.npy")
        assert w.dtype == np.float32 and np.array_equal(w, wavs[i].numpy())
    assert sum(f.stat().st_size for f in tmp_path.iterdir()) <= b.DUMP_BYTES


def test_tool_scripts_compile():
    for f in glob.glob(os.path.join(ROOT, "tools", "*.py")) + [os.path.join(ROOT, "bench.py"), os.path.join(ROOT, "__graft_entry__.py")]:
        py_compile.compile(f, doraise=True)
