"""`bench.py` end to end on the CPU: the real script, the real `HaloStencil` / `BlockTimer` / `Comm` classes, the
emulated native module of tests/test_halo_python_emulated.py (host memory, launches execute at once) and fake CUDA
events.  Numbers mean nothing here; what is checked is the driver contract — ONE JSON line from rank 0 with every key the
driver reads, internally consistent, verification words zero because the emulated kernels really compute the stencil —
and that every branch of the script (extras, stock arms, rows = 1, end-to-end path, roofline block) executes."""
import importlib.util
import json
import os
import sys

import pytest
import torch

from tests.emu_device import TickingEvent
from tests.test_halo_python_emulated import emu  # noqa: F401  (the fixture)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load_bench():
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.parametrize("extras", [False, True])
def test_bench_line_has_the_contract_keys(emu, monkeypatch, capsys, extras):  # noqa: F811
    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    monkeypatch.setattr(torch.cuda, "Event", TickingEvent)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "HPCP_DEVICE"):
        monkeypatch.delenv(k, raising=False)
    msg, steps = 8192, 4
    argv = ["bench.py", "--gpus", "1", "--steps", str(steps), "--warmup", "3", "--bytes", str(msg), "--tile-kb", "1",
            "--preheat-ms", "1", "--blocks", "3", "--e2e-steps", "2"] + ([] if extras else ["--no-extras"])
    monkeypatch.setattr(sys, "argv", argv)
    bench = _load_bench()
    monkeypatch.setattr(bench, "cpu_concurency", lambda impl: {"impl": impl, "stub": True})
    rc = bench.main()
    lines = [l for l in capsys.readouterr().out.splitlines() if l.startswith("{")]
    assert rc == 0 and len(lines) == 1, "exactly one JSON line"
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches"):
        assert key in d, key
    assert d["impl"] == "ours" and d["n_gpus"] == 1 and d["steps"] == steps and d["warmup"] == 3
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["dtype"] == "fp32" and d["data"] == "synthetic"
    assert d["unit"] == "GB/s" and d["vs_baseline"] is None
    # 2 ms per block of `steps` steps -> value = N x 2 messages / time
    assert d["ms_per_step"] == pytest.approx(2.0 / steps)
    assert d["value"] == pytest.approx(2 * msg / (d["ms_per_step"] * 1e-3) / 1e9, abs=0.006)    # rounded to 0.01 GB/s
    assert len(d["blocks_ms_per_step"]) == 3 and d["wrong_words"] == 0
    cfg = d["config"]
    assert cfg["rows"] == 8 and cfg["message_bytes"] == msg and cfg["steps_per_launch"] == steps
    assert cfg["parallelism"] == "ring1" and "l2" in cfg and "timing" in cfg
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    e2e = d["e2e"]
    assert e2e["h2d_bytes_per_step"] == e2e["d2h_bytes_per_step"] == cfg["rows"] * msg
    assert e2e["value"] > 0 and e2e["wrong_words"] == 0 and e2e["value"] != d["value"]
    assert d["gpu_launches"] == 1 and d["gpu_launches_all_blocks"] >= 3
    roof = d["roofline"]
    assert roof["hbm_gbs"] > 0 and roof["bound_ms"] == roof["hbm_ms"] and roof["nvlink_ms"] == 0   # N=1: no link
    if extras:
        for key in ("overlap_pct", "unfused_compute_ms", "unfused_exchange_ms", "one_launch_per_step_ms", "stock",
                    "speedup_vs_stock_memcpy", "rows_1", "cpu_concurency"):
            assert key in d, key
        assert d["stock"]["wrong_words"] == 0 and d["stock"]["nccl_sendrecv_ms"] is None      # NCCL arm needs N > 1
        assert d["rows_1"]["wrong_words"] == 0
        assert "legacy_triad_ring_put" in d or "legacy_error" in d
    else:
        assert "stock" not in d and "cpu_concurency" not in d
    assert not emu.live, "bench.py returned every allocation"


def test_bench_dump_outputs_is_the_timed_call(emu, monkeypatch, capsys, tmp_path):  # noqa: F811
    """--dump-outputs: the slab after one timed call (K steps from the initial field), the same whatever the pre-heat
    and block count ran before it, equal to the PyTorch reference; a field larger than DUMP_ELEMS keeps its seeded
    columns."""
    import numpy as np

    from hpc_patterns_b200.models.halo import initial_field, reference_steps

    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    monkeypatch.setattr(torch.cuda, "Event", TickingEvent)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "HPCP_DEVICE"):
        monkeypatch.delenv(k, raising=False)
    msg, steps = 8192, 5
    want = reference_steps(initial_field(1, 8, msg // 4), steps).numpy()
    dumps = []
    for blocks, dump_elems in ((3, None), (2, None), (2, 8 * 300)):
        out = tmp_path / f"dump{len(dumps)}"
        monkeypatch.setattr(sys, "argv", ["bench.py", "--gpus", "1", "--steps", str(steps), "--warmup", "3", "--bytes",
                                          str(msg), "--tile-kb", "1", "--preheat-ms", "1", "--blocks", str(blocks),
                                          "--e2e-steps", "1", "--no-extras", "--dump-outputs", str(out)])
        bench = _load_bench()
        if dump_elems:
            monkeypatch.setattr(bench, "DUMP_ELEMS", dump_elems)
        assert bench.main() == 0
        assert [p.name for p in out.iterdir()] == ["field_rank0.npy"]
        dumps.append(np.load(out / "field_rank0.npy"))
    capsys.readouterr()
    assert dumps[0].dtype == np.float32 and dumps[0].shape == (8, msg // 4)
    assert np.array_equal(dumps[0], want) and np.array_equal(dumps[1], want)
    cols = bench.dump_columns(msg // 4, 300)
    assert len(cols) == 300 and np.array_equal(dumps[2], want[:, cols])
    assert not emu.live


def test_reference_arm_line(monkeypatch, capsys):
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--gpus", "4", "--steps", "20", "--warmup", "5"])
    monkeypatch.delenv("RANK", raising=False)
    bench = _load_bench()
    monkeypatch.setattr(bench, "cpu_concurency", lambda impl: {"impl": impl, "stub": True})
    assert bench.main() == 0
    d = json.loads(capsys.readouterr().out.strip())
    assert d["impl"] == "reference" and "unavailable" in d and "\n" not in d["unavailable"]
    assert d["cpu_concurency"] == {"impl": "reference", "stub": True}
    # ranks other than 0 of a torchrun launch print nothing and exit 0
    monkeypatch.setenv("RANK", "3")
    assert bench.main() == 0 and capsys.readouterr().out == ""


@pytest.mark.parametrize("flags,what", [([], "pull/persistent"), (["--mode", "push"], "push/persistent"),
                                        (["--per-step"], "pull/per-step"), (["--stock", "memcpy"], "stock-memcpy"),
                                        (["--mode", "push", "--l2-hint", "--ctas", "2"], "push/persistent")])
def test_python_halo_program_report_lines(emu, monkeypatch, capsys, tmp_path, flags, what):  # noqa: F811
    """`python -m hpc_patterns_b200 halo` (process-per-GPU twin of bin/halo) on the emulated device: the reference-style
    report — `Passed <rank>`, the elapsed line, the JSON row — for every way of stepping."""
    from hpc_patterns_b200.models import halo as halo_mod

    monkeypatch.setattr(torch.cuda, "Event", TickingEvent)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "HPCP_DEVICE"):
        monkeypatch.delenv(k, raising=False)
    row = tmp_path / "rows.jsonl"
    rc = halo_mod.main(["--rows", "3", "--bytes", "6144", "--steps", "4", "--iters", "2", "--tile-kb", "1", "--json",
                        str(row)] + flags)
    out = capsys.readouterr().out
    assert rc == 0 and "Passed 0" in out
    assert f"Elapsed (max over ranks, min of 2): 2.0000 ms for 4 steps = 0.50000 ms/step | halo {what} P=1 rows=3" in out
    d = json.loads(row.read_text())
    assert d["pattern"] == "halo" and d["variant"] == what and d["mismatches"] == 0 and d["ranks"] == 1
    assert d["bus_GBps"] == pytest.approx(2 * 6144 / (0.5 * 1e6))
    if "--ctas" in flags:
        assert d["ctas"] == 2
    assert not emu.live
