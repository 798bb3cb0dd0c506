"""CPU: the benchmark drivers run end to end through the C-ABI test double (tools/dryrun_bench.py) and print ONE JSON line that
carries every key of the measurement contract.  Guards the driver logic of scripts that otherwise only run on the GPU box; the
numbers are meaningless here and are not looked at."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CONTRACT = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
            "config", "clocks", "e2e", "gpu_launches", "roofline")


def _run(which, *flags):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "dryrun_bench.py"), which, *flags], capture_output=True, text=True, timeout=600,
                       cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [ln for ln in r.stdout.strip().split("\n") if ln.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    return json.loads(lines[0])


@pytest.mark.parametrize("which", ["decode", "lora"])
def test_bench_driver_prints_the_contract_line(which):
    d = _run(which)
    for k in CONTRACT:
        assert k in d, k
    assert set(d["e2e"]) >= {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"}
    assert set(d["roofline"]) >= {"bound", "achieved", "peak", "unit", "frac", "traffic"}
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    assert "workload" in d["config"]
    if which == "decode":
        assert d["metric"] == "decode_tokens_per_s" and d["scaling"] == "strong"
        assert set(d["attention"]) >= {"decode", "prefill"} and "error" not in d["attention"]
        assert d["ts_encoder"]["patch_rows"] > 0
        assert d["config"]["variants"] == {"decode_fused": 0, "peer_ll": 1, "native_step": 0, "decode_chain": 0}      # peer_ll: default since round 2 (only acts under TP)
        # side blocks: BASELINE configs[3] (second model instance, 30 series x 512 points) and the GPTQ-Int4 decode (third instance, 4-bit projections)
        c4, w4 = d["config4"], d["w4a16"]
        assert "error" not in c4 and c4["batch"] == 8 and c4["context"] == 30 * (46 + 2 + 32) + 64 and c4["tokens_per_s"] > 0
        assert c4["identical_tokens_on_all_ranks"] and set(c4["e2e"]) >= {"value", "unit", "seconds"}
        assert "error" not in w4 and w4["kernel"] == "mma" and set(w4["by_batch"]) >= {"1", "2"}
        for b in w4["by_batch"].values():
            assert b["w4_ms_per_step"] > 0 and b["bf16_ms_per_step"] > 0 and min(v for k, v in b.items() if k.startswith("min_greedy_agreement")) >= 1
    else:
        assert d["metric"] == "lora_finetune_positions_per_s" and d["scaling"] == "weak"
        assert 11.0 < d["loss"] < 13.0          # ln(vocab) at initialisation (LoRA B = 0)


def test_decode_variant_probe_selects_only_on_equal_tokens_and_a_gain(monkeypatch):
    """bench.py's guarded probe: the cluster-fused decode GEMMs are used for the measured run only if a child run shows identical greedy
    tokens AND a shorter step; every other outcome keeps the default path."""
    import argparse
    sys.path.insert(0, ROOT)
    import bench
    args = argparse.Namespace(batch=32)

    def fake(outcomes):
        return lambda level, a, timeout=360: dict(outcomes[level])

    cases = [
        ({0: {"ms_per_step": 1.00, "tokens_sha1": "ab"}, 1: {"ms_per_step": 0.90, "tokens_sha1": "ab"}}, 1),      # same tokens, faster
        ({0: {"ms_per_step": 1.00, "tokens_sha1": "ab"}, 1: {"ms_per_step": 0.90, "tokens_sha1": "cd"}}, 0),      # different tokens
        ({0: {"ms_per_step": 1.00, "tokens_sha1": "ab"}, 1: {"ms_per_step": 0.995, "tokens_sha1": "ab"}}, 0),     # no real gain
        ({0: {"ms_per_step": 1.00, "tokens_sha1": "ab"}, 1: {"error": "rc=-6: trap"}}, 0),                         # the variant faulted
        ({0: {"error": "timeout"}, 1: {"ms_per_step": 0.5, "tokens_sha1": "ab"}}, 0),                              # no baseline
        ({0: {"ms_per_step": 1.00, "tokens_sha1": None}, 1: {"ms_per_step": 0.5, "tokens_sha1": None}}, 0),        # nothing to compare
        ({0: {"ms_per_step": 1.00, "tokens_sha1": "ab", "ms_by_batch": {"1": 0.5, "32": 1.0}},
          1: {"ms_per_step": 0.90, "tokens_sha1": "ab", "ms_by_batch": {"1": 0.6, "32": 0.9}}}, 0),                # a side batch got slower
        ({0: {"ms_per_step": 1.00, "tokens_sha1": "ab", "ms_by_batch": {"1": 0.5, "32": 1.0}},
          1: {"ms_per_step": 0.90, "tokens_sha1": "ab", "ms_by_batch": {"1": 0.45, "32": 0.9}}}, 1),
    ]
    monkeypatch.setattr(bench, "_probe_compare", lambda level, a, timeout=420: {"error": "not probed in this case"})
    for outcomes, want in cases:
        monkeypatch.setattr(bench, "_probe_run", fake(outcomes))
        rec = bench.probe_decode_variant(args)
        assert rec["selected"] == want, (outcomes, rec)
    # level 2: only after level 1 was adopted, only within the numeric bound, only if faster again
    lvl = {0: {"ms_per_step": 1.00, "tokens_sha1": "ab"}, 1: {"ms_per_step": 0.90, "tokens_sha1": "ab"}, 2: {"ms_per_step": 0.80, "tokens_sha1": "zz"}}
    for cmp, want in (({"max_rel": 3e-3, "finite": True}, 2), ({"max_rel": 5e-2, "finite": True}, 1), ({"max_rel": 1e-3, "finite": False}, 1),
                      ({"error": "rc=1"}, 1)):
        monkeypatch.setattr(bench, "_probe_run", fake(lvl))
        monkeypatch.setattr(bench, "_probe_compare", lambda level, a, timeout=420, c=cmp: dict(c))
        assert bench.probe_decode_variant(args)["selected"] == want, cmp
    slow2 = dict(lvl)
    slow2[2] = {"ms_per_step": 0.89, "tokens_sha1": "zz"}
    monkeypatch.setattr(bench, "_probe_run", fake(slow2))
    monkeypatch.setattr(bench, "_probe_compare", lambda level, a, timeout=420: {"max_rel": 1e-3, "finite": True})
    assert bench.probe_decode_variant(args)["selected"] == 1
    monkeypatch.setattr(bench, "_probe_run", lambda *a, **k: (_ for _ in ()).throw(RuntimeError("boom")))
    assert bench.probe_decode_variant(args)["selected"] == 0                # the probe itself failing is not fatal either


def test_probe_child_run_parses_the_json_line_and_survives_failures(tmp_path, monkeypatch):
    import argparse
    sys.path.insert(0, ROOT)
    import bench
    good = tmp_path / "good.py"
    good.write_text("import os, sys\nprint('NCCL noise')\nprint('{\"ms_per_step\": 0.5, \"by_batch\": {\"1\": {\"tokens_sha1\": \"a' + os.environ['CTS_DECODE_FUSED'] + '\"}, \"32\": {\"tokens_sha1\": \"b\"}}, \"launches_per_step\": 7}')\n")
    bad = tmp_path / "bad.py"
    bad.write_text("import sys\nprint('about to die', file=sys.stderr)\nsys.exit(134)\n")
    slow = tmp_path / "slow.py"
    slow.write_text("import time\ntime.sleep(30)\n")
    args = argparse.Namespace(batch=4)
    monkeypatch.setattr(bench, "__file__", str(good))
    assert bench._probe_run(1, args) == {"ms_per_step": 0.5, "tokens_sha1": "1:a1/32:b", "launches_per_step": 7, "ms_by_batch": {"1": None, "32": None}}
    monkeypatch.setattr(bench, "__file__", str(bad))
    assert "error" in bench._probe_run(1, args) and "rc=134" in bench._probe_run(1, args)["error"]
    monkeypatch.setattr(bench, "__file__", str(slow))
    assert "error" in bench._probe_run(1, args, timeout=1)


def test_dump_outputs_writes_the_last_timed_step(tmp_path):
    """--dump-outputs: the measured batch's last-step logits (float32) and its greedy tokens (float64) land in DIR; --steps sets how many
    timed steps ran (three more steps = three more tokens), and the inputs are the same from run to run (the shorter run's tokens are a
    prefix of the longer run's)."""
    runs = {}
    for steps in (2, 5):
        out = tmp_path / f"steps{steps}"
        d = _run("decode", "--dump-outputs", str(out), "--steps", str(steps), "--no-w4", "--no-config4")
        assert d["steps"] == steps and d["dumped_outputs"]["names"] == ["logits", "tokens"]
        lg, tok = np.load(out / "logits.npy"), np.load(out / "tokens.npy")
        assert lg.dtype == np.float32 and tok.dtype == np.float64 and np.isfinite(lg).all()
        assert lg.shape[0] == tok.shape[0] == d["config"]["batch"] and lg.shape[1] == 152064
        assert sum(f.stat().st_size for f in out.iterdir()) <= 64 << 20
        runs[steps] = tok
    assert runs[5].shape[1] - runs[2].shape[1] == 3
    assert np.array_equal(runs[5][:, : runs[2].shape[1]], runs[2])


def test_dump_outputs_keeps_a_fixed_sample_of_columns_within_the_budget(tmp_path, monkeypatch):
    import torch
    sys.path.insert(0, ROOT)
    import bench
    lg, tok = torch.randn(3, 5000, dtype=torch.bfloat16), torch.randint(0, 5000, (3, 7), dtype=torch.int32)
    monkeypatch.setattr(bench, "DUMP_BYTES", 20000)
    for sub in ("a", "b"):
        assert bench.dump_outputs(str(tmp_path / sub), lg, tok) == ["logits", "logits_columns", "tokens"]
    got = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in ("logits", "logits_columns", "tokens")}
    assert sum(a.nbytes for a in got.values()) <= 20000
    cols = got["logits_columns"].astype(np.int64)
    assert np.all(np.diff(cols) > 0) and got["logits"].shape == (3, cols.size)
    assert np.array_equal(got["logits"], lg.float().numpy()[:, cols]) and np.array_equal(got["tokens"], tok.numpy())
    for n, a in got.items():
        assert np.array_equal(np.load(tmp_path / "b" / f"{n}.npy"), a), n


def test_the_kv_cache_makes_room_for_every_requested_step():
    sys.path.insert(0, ROOT)
    import bench
    assert bench.seq_capacity(20 + 5 + 8) == 1024                      # the size every recorded run used
    for steps in (430, 500, 2000):
        cap = bench.seq_capacity(steps + 3 + 8)
        assert cap % 64 == 0 and cap >= bench.PROMPT_POSITIONS + steps + 3 + 8
