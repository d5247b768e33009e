"""The C-ABI library loads on a CPU-only box and exports every symbol include/strolle_b200.h declares;
without a GPU it fails loudly instead of falling back."""
import os
import re

import pytest

import strolle_b200
from strolle_b200 import build as st_build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(strolle_b200.lib_path()):
        st_build.build()
    return strolle_b200.load_library()


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "strolle_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(st_[a-z0-9_]+)\s*\(", src)))


def test_every_declared_symbol_is_exported(lib):
    names = declared_symbols()
    assert len(names) >= 30
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/strolle_b200.h but not exported"


def test_pass_names(lib):
    names = list(strolle_b200.PASS_NAMES)
    assert names[0] == "prim_gbuffer" and "frame_denoising_wavelet" in names and len(names) == 27


def test_no_cpu_fallback(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(strolle_b200.StrolleError, match="no CPU fallback"):
        strolle_b200.Engine()


def test_product_does_not_touch_the_oracle():
    """Only tests/, __graft_entry__.smoke() and bench.py may import, link or execute anything under oracle/."""
    pkg = os.path.join(ROOT, "strolle_b200")
    banned = [r"\bimport\s+oracle", r"\bfrom\s+oracle", r"pyoracle", r"liboracle", r"oracle/", r"orc_[a-z_]+\(", r"#include\s+\"orc_"]
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                for pat in banned:
                    assert not re.search(pat, text), f"{f} references the oracle ({pat})"


def test_rust_sys_crate_matches_the_header():
    """rust/strolle-b200-sys/src/lib.rs is generated from include/strolle_b200.h (tools/gen_rust_sys.py): the committed file must be
    what the generator produces now, and must declare every C entry point exactly once."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("gen_rust_sys", os.path.join(ROOT, "tools", "gen_rust_sys.py"))
    gen = importlib.util.module_from_spec(spec); spec.loader.exec_module(gen)
    text, names = gen.generate()
    assert open(gen.OUT).read() == text, "run python tools/gen_rust_sys.py"
    assert sorted(names) == declared_symbols()


def test_rust_engine_forwards_every_reference_method():
    """The safe crate has every public method of strolle::Engine (strolle/src/lib.rs:132-301) and each one calls into the C ABI."""
    src = open(os.path.join(ROOT, "rust", "strolle-b200", "src", "lib.rs")).read()
    src = src[src.index("impl<P: Params> Engine<P> {"):]
    for method, ffi in [("new", "st_multi_create"), ("insert_mesh", "st_multi_insert_mesh"), ("remove_mesh", "st_multi_remove_mesh"), ("insert_material", "st_multi_insert_material"),
                        ("has_material", "st_multi_has_material"), ("remove_material", "st_multi_remove_material"), ("insert_image", "st_multi_insert_image"),
                        ("remove_image", "st_multi_remove_image"), ("insert_instance", "st_multi_insert_instance"), ("remove_instance", "st_multi_remove_instance"),
                        ("insert_light", "st_multi_insert_light"), ("remove_light", "st_multi_remove_light"), ("update_sun", "st_multi_update_sun"),
                        ("create_camera", "st_multi_create_camera"), ("update_camera", "st_multi_update_camera"), ("render_camera", "st_multi_render_camera"),
                        ("delete_camera", "st_multi_delete_camera"), ("tick", "st_multi_tick")]:
        m = re.search(r"pub fn %s\b.*?\n    }\n" % method, src, flags=re.S)
        assert m, f"Engine::{method} missing"
        assert ffi in m.group(0), f"Engine::{method} does not call {ffi}"
    sys_src = open(os.path.join(ROOT, "rust", "strolle-b200-sys", "src", "lib.rs")).read()
    for ffi in set(re.findall(r"sys::(st_\w+)\(", src)):
        assert f"pub fn {ffi}(" in sys_src, f"{ffi} used by the safe crate but not declared by the sys crate"


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU restatement timed on the host cores; no GPU involved) prints ONE JSON line with the keys the
    bench contract names, its own cpu_baseline and an e2e block that repeats the line's value with zero copy bytes."""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1", "--width", "160", "--height", "90"],
                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=300, cwd=ROOT).stdout
    lines = [l for l in out.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "Mrays/s" and d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1
    for key in ("metric", "value", "ms_per_step", "scaling", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["value"] > 0 and "160x90" in d["config"]["workload"]


def run_bench_dump(args, out_dir):
    """Runs bench.py with --dump-outputs out_dir; returns its JSON line and the arrays it wrote."""
    import json
    import subprocess
    import sys
    import numpy as np
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args + ["--dump-outputs", str(out_dir)],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-3000:]
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0]), {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


def test_bench_reference_arm_dumps_identical_outputs(tmp_path):
    """`--dump-outputs DIR` writes the frame of the last timed step; the same arguments give the same inputs, so two runs write the same bits."""
    import numpy as np
    args = ["--impl", "reference", "--steps", "3", "--warmup", "1", "--width", "96", "--height", "54"]
    d, a = run_bench_dump(args, tmp_path / "a")
    _, b = run_bench_dump(args, tmp_path / "b")
    assert d["steps"] == 3 and list(a) == ["output"] and list(b) == ["output"]
    assert a["output"].shape == (54, 96, 4) and a["output"].dtype == np.float32
    assert np.isfinite(a["output"]).all() and a["output"][..., :3].mean() > 0.01
    assert (a["output"].view(np.uint32) == b["output"].view(np.uint32)).all()


def test_bench_dump_samples_large_frames(monkeypatch):
    """A frame larger than the dump budget is written as a fixed seeded sample of pixels with their indices; row strips (one per
    rank, gathered in rank order) give the same sample as the whole frame."""
    import numpy as np
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 32 * 500)
    h, w = 40, 30
    frame = np.random.RandomState(1).rand(h, w, 4).astype(np.float32)
    whole = bench.dump_frame(frame, 0, w, h)
    idx = whole["output_pixels"]
    assert idx.dtype == np.float64 and len(idx) == 500 and (np.diff(idx) > 0).all()
    assert (whole["output"] == frame.reshape(-1, 4)[idx.astype(np.int64)]).all()
    strips = [bench.dump_frame(frame[y0:y1], y0, w, h) for y0, y1 in [(0, 7), (7, 25), (25, 40)]]
    assert (np.concatenate([s["output"] for s in strips]) == whole["output"]).all()
    assert all((s["output_pixels"] == idx).all() for s in strips)
    monkeypatch.setattr(bench, "DUMP_BYTES", h * w * 16)
    assert list(bench.dump_frame(frame, 0, w, h)) == ["output"]


@pytest.mark.gpu
def test_bench_cuda_arm_dumps_identical_outputs(tmp_path):
    """The CUDA arm: the dumped frame is deterministic across runs with the same arguments and close to the strict CPU oracle's frame of
    the same frame id (the product default shades with FMA / SFU approximations)."""
    import numpy as np
    args = ["--steps", "4", "--warmup", "3", "--width", "96", "--height", "54", "--no-extras", "--no-cpu-baseline"]
    d, a = run_bench_dump(args, tmp_path / "a")
    _, b = run_bench_dump(args, tmp_path / "b")
    _, ref = run_bench_dump(["--impl", "reference"] + args[:8], tmp_path / "ref")
    assert d["steps"] == 4 and a["output"].shape == (54, 96, 4)
    assert (a["output"].view(np.uint32) == b["output"].view(np.uint32)).all()
    x, y = a["output"][..., :3].astype(np.float64), ref["output"][..., :3].astype(np.float64)
    assert np.sqrt(((x - y) ** 2).sum() / (y ** 2).sum()) <= 1e-2
