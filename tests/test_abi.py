"""The C-ABI library loads, exports every symbol include/b200audio.h declares, its host-only entry points
agree with the oracle, and every device entry point fails LOUDLY without a GPU.  CPU only."""
import ctypes as C
import re
from pathlib import Path

import numpy as np
import pytest

from oracle import dsp, llama

ROOT = Path(__file__).resolve().parent.parent


def test_exports_every_declared_symbol(b2a):
    # the boundary (b200audio.h) and the test / benchmark hooks (b200audio_internal.h, not bound by a Swift host)
    public = set(re.findall(r"\b(b2a_[a-z0-9_]+)\s*\(", (ROOT / "include" / "b200audio.h").read_text()))
    internal = set(re.findall(r"\b(b2a_[a-z0-9_]+)\s*\(", (ROOT / "include" / "b200audio_internal.h").read_text()))
    assert len(public) >= 30 and not (public & internal)
    assert not any(n.endswith(("_test", "_debug_trace", "_debug_layout", "_create_random", "_bench_flags")) for n in public)
    declared = public | internal
    lib = C.CDLL(str(b2a._ffi.LIB_PATH))
    for name in declared:
        assert hasattr(lib, name), name
    assert declared == set(b2a._ffi.SIGNATURES), declared ^ set(b2a._ffi.SIGNATURES)


def test_host_tables_match_oracle(b2a):
    assert np.abs(b2a.hanning_window(400) - dsp.hanning_window(400)).max() < 2e-7
    assert np.abs(b2a.hanning_window(400, periodic=True) - dsp.periodic_hann_window(400)).max() < 2e-7
    for scale, nm in (("htk", 80), ("htk", 128), ("slaney", 80), ("slaney", 128)):
        a, o = b2a.mel_filters(16000, 400, nm, mel_scale=scale), dsp.mel_filters(16000, 400, nm, mel_scale=scale)
        assert a.shape == o.shape and np.abs(a - o).max() < 1e-6 * max(1.0, o.max())
        assert np.array_equal(a != 0, o != 0) or np.abs(a - o)[(a != 0) != (o != 0)].max() < 1e-7


def test_reference_known_answers_for_hamming_and_power_to_db(b2a):
    """Tests/MLXAudioCodecsTests.swift:117-140 (SharedDSPTests), on the oracle and on the library's host helpers."""
    for hw, pdb in ((dsp.hamming_window, dsp.power_to_db), (b2a.hamming_window, b2a.power_to_db)):
        periodic, symmetric = hw(4), hw(4, periodic=False)
        assert len(periodic) == 4 and len(symmetric) == 4
        assert abs(periodic[0] - 0.08) < 1e-3 and abs(periodic[1] - 0.54) < 1e-3 and abs(periodic[3] - 0.54) < 1e-3
        assert abs(symmetric[0] - 0.08) < 1e-3 and abs(symmetric[3] - 0.08) < 1e-3 and abs(symmetric[1] - symmetric[2]) < 1e-3
        clipped = pdb(np.array([1e-10, 1e-5, 1.0], np.float32), top_db=80)
        assert abs(clipped[0] + 80) < 1e-2 and abs(clipped[1] + 50) < 1e-2 and abs(clipped[2]) < 1e-3
        assert len(hw(0)) == 0 and list(hw(1)) == [1.0]                             # the guard branches (:26-27)
    for n, per in ((400, True), (400, False), (7, True)):
        assert np.abs(b2a.hamming_window(n, per) - dsp.hamming_window(n, per)).max() < 5e-7          # float32 phase, as the reference computes it
    x = np.random.default_rng(0).random(1000).astype(np.float32) ** 8
    assert np.abs(b2a.power_to_db(x, top_db=30) - dsp.power_to_db(x, top_db=30)).max() < 1e-4
    assert np.abs(b2a.power_to_db(x) - dsp.power_to_db(x)).max() < 1e-4


def test_token_plumbing_matches_oracle(b2a):
    M = b2a.LlamaTTSModel
    prompts = [[1, 2, 3], [9], [4, 5, 6, 7, 8]]
    ids, mask = M.prepare_input_ids(prompts)
    oids, omask = llama.prepare_input_ids(prompts)
    assert np.array_equal(ids, oids) and np.array_equal(mask, omask)
    rng = np.random.default_rng(0)
    S, E, O = llama.START_OF_SPEECH, llama.END_OF_SPEECH, llama.AUDIO_TOKEN_OFFSET
    rows = rng.integers(O, O + 7 * 4096, size=(3, 40)).astype(np.int32)
    rows[0, 3] = S; rows[1, 10] = S; rows[2, 25] = E; rows[1, 30] = E
    assert M.parse_output(rows) == llama.parse_output(rows)
    rows2 = rng.integers(O, O + 7 * 4096, size=(2, 21)).astype(np.int32)          # no start-of-speech: whole rows
    assert M.parse_output(rows2) == llama.parse_output(rows2)
    codes = [rng.integers(0, 4096, (1, 6 * k), dtype=np.int32) for k in (1, 2, 4)]
    cl = M.code_list_from_codes(codes)
    assert cl == llama.code_list_from_codes(codes)
    back = M.codes_from_code_list(cl)
    assert all(np.array_equal(a, b) for a, b in zip(back, llama.codes_from_code_list(cl)))
    assert all(np.array_equal(a, b) for a, b in zip(back, codes))
    assert [c.shape for c in M.codes_from_code_list([])] == [(1, 0)] * 3            # empty input edge case


def test_error_mapping_and_no_cpu_fallback(b2a):
    E = b2a.AudioGenerationError
    with pytest.raises(E) as ei:
        b2a.hanning_window(1)
    assert ei.value.case == "invalidInput"
    if b2a.device_count() == 0:
        for make in (lambda: b2a.IncrementalMelSpectrogram(), lambda: b2a.LogMel("whisper")):
            with pytest.raises(E) as ei:
                make()
            assert ei.value.case == "cudaError" and "no CPU fallback" in ei.value.message


def test_product_path_never_imports_oracle():
    pkg = ROOT / "mlx-audio-swift_b200"
    for f in list(pkg.rglob("*.py")) + list(pkg.rglob("*.cu")) + list(pkg.rglob("*.cuh")):
        txt = f.read_text()
        assert "import oracle" not in txt and "from oracle" not in txt, f


def test_bench_cpu_arm_thread_budget():
    """bench.py's CPU legs size their thread pool from what the process may really use, not from the host's CPU count."""
    import os
    import sys
    sys.path.insert(0, str(ROOT))
    import bench
    n = bench.usable_cpus()
    assert 1 <= n <= (os.cpu_count() or 1) and n <= len(os.sched_getaffinity(0))


def test_bench_workload_accounting():
    """The numbers bench.py's line is built from: BASELINE.md's audio per utterance, SURVEY.md 8(d)'s bytes per decode step, the
    prompt that makes parseOutput crop like a real checkpoint, and the sharding of the two scaling modes."""
    import sys
    from pathlib import Path
    sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
    import bench
    from oracle import llama
    assert bench.frames_per_utterance() == 73 and abs(bench.audio_seconds_per_utterance() - 73 * 2048 / 24000.0) < 1e-12     # 6.229 s
    ids = bench.make_prompts(0)
    assert ids.shape == (8, 64) and (ids[:, 0] == 128259).all() and (ids[:, -1] == 128257).all()
    # parseOutput on prompt + 512 generated code tokens keeps exactly the 73 whole frames after the last START_OF_SPEECH
    gen = [128266 + (i % 7) * 4096 + 5 for i in range(512)]
    rows = llama.parse_output(np.asarray([ids[0].tolist() + gen]))
    assert len(rows) == 1 and len(rows[0]) == 73 * 7
    layers = llama.codes_from_code_list(rows[0])
    assert [int(c.shape[1]) for c in layers] == [73, 146, 292]
    cfg = bench.ORPHEUS
    H, I, V, L = 3072, 8192, 156940, 28
    per_layer = (24 + 16) * 128 * H + H * 24 * 128 + 3 * I * H
    assert bench.weight_bytes(cfg) == 2 * (L * per_layer + V * H)                       # every matrix once + the tied head, bf16
    assert bench.kv_bytes(cfg, 8, 320, 2) == 2 * 8 * 8 * 320 * 128 * 2 * 28             # bf16 K and V at the loop's mean context
    assert bench.kv_bytes(cfg, 8, 320, 4) == 2 * bench.kv_bytes(cfg, 8, 320, 2)
    assert abs((bench.weight_bytes(cfg) + bench.kv_bytes(cfg, 8, 320, 2)) / 1e9 - 6.895) < 1e-3
    assert bench.bench_config(cfg, 4, "weak")["global_batch"] == 32 and bench.bench_config(cfg, 4, "strong")["global_batch"] == 8
    assert bench.bench_config(cfg, 8, "strong")["rows_per_gpu"] == 1


def test_bench_output_dump(tmp_path, monkeypatch):
    """--dump-outputs: one float32 / float64 .npy per output (integers exactly as float64), a bounded total, and a step count that
    is really used (no zero-step run)."""
    import sys
    sys.path.insert(0, str(ROOT))
    import bench
    wave = np.random.default_rng(0).standard_normal((2, 5)).astype(np.float32)
    lens = np.array([5, 2**40 + 1], dtype=np.int64)
    bench.write_outputs(tmp_path / "d", {"wave": wave, "lens": lens, "half": wave.astype(np.float16)})
    got = {p.stem: np.load(p) for p in (tmp_path / "d").glob("*.npy")}
    assert set(got) == {"wave", "lens", "half"}
    assert got["wave"].dtype == np.float32 and np.array_equal(got["wave"], wave)
    assert got["lens"].dtype == np.float64 and got["lens"].astype(np.int64).tolist() == lens.tolist()
    assert got["half"].dtype == np.float32
    with pytest.raises(ValueError):
        bench.write_outputs(tmp_path / "big", {"x": np.zeros(bench.DUMP_BYTES_MAX // 4 + 1, np.float32)})
    assert not (tmp_path / "big").exists()
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "0"])
    with pytest.raises(SystemExit):
        bench.main()
