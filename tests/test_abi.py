"""The drop-in boundary: the shared libraries load and export every symbol the headers declare."""
import ctypes as C
import os
import re

import numpy as np

import pytest


def _declared(header: str) -> list[str]:
    text = open(header).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(ctts_(?:gpu|front|b200)_[a-z0-9_]+)\s*\(", text)))


def test_gpu_library_exports_header_symbols(H):
    gpu = H.importlib.import_module("2026-simple-c-tts_b200.gpu")
    L = gpu.lib()
    names = _declared(os.path.join(H.ROOT, "include", "ctts_gpu.h"))
    assert "ctts_gpu_synth_batch" in names and "ctts_gpu_init" in names and len(names) >= 14
    for n in names:
        assert hasattr(L, n), n


def test_front_library_exports_header_symbols(H):
    L = H.front.lib()
    names = _declared(os.path.join(H.ROOT, "include", "ctts_front.h"))
    assert len(names) >= 12
    for n in names:
        assert hasattr(L, n), n


def test_pipeline_library_exports_header_symbols(H):
    """libctts_b200.so (texts -> PCM over the two libraries): loads without a device, exports ctts_b200.h."""
    pipe = H.importlib.import_module("2026-simple-c-tts_b200.pipeline")
    L = pipe.lib()
    names = _declared(os.path.join(H.ROOT, "include", "ctts_b200.h"))
    assert names == ["ctts_b200_capacity_hint", "ctts_b200_plan_cache_create", "ctts_b200_plan_cache_destroy",
                     "ctts_b200_plan_cache_stats", "ctts_b200_synth_texts"]
    for n in names:
        assert hasattr(L, n), n
    assert C.sizeof(pipe.Timing) == 6 * 8 and C.sizeof(pipe.Options) == 32
    cache = pipe.PlanCache(1 << 20)
    assert cache.stats() == {"hits": 0, "misses": 0, "entries": 0, "bytes": 0}
    cache.close()


def test_capacity_hint_covers_the_bounds(H, small_db, front_small):
    """ctts_b200_capacity_hint (no planning) must not be smaller than the slot space the planned batch needs."""
    pipe = H.importlib.import_module("2026-simple-c-tts_b200.pipeline")
    texts = H.corpus.batch(40, seed=5, target_chars=150) + ["", "1234567 e 89", "a"]
    speeds = [1.0, 0.5, 2.0, 0.7] * 10 + [1.0, 0.5, 0.5]
    plan = front_small.plan(texts, speeds)
    _, out, _ = front_small.bounds(plan)
    need = int(sum((int(b) + 7) // 8 * 8 + 8 for b in out))
    assert pipe.capacity_hint(front_small, pipe.TextBatch(texts, speeds)) >= need


def test_ctypes_mirrors_match_the_headers(H, tmp_path):
    """Every struct that crosses the C-ABI: sizeof and the offset of the last member as gcc sees them in include/*.h
    against the ctypes mirrors the Python host side (and these tests) use."""
    import subprocess
    gpu = H.importlib.import_module("2026-simple-c-tts_b200.gpu")
    pipe = H.importlib.import_module("2026-simple-c-tts_b200.pipeline")
    pairs = [
        ("ctts_gpu_run_info", "reuse_bound_samples", gpu.RunInfo),
        ("ctts_gpu_wsola_stats", "walked_frames", gpu.WsolaStats),
        ("ctts_b200_options", "cache", pipe.Options),
        ("ctts_b200_timing", "reserved", pipe.Timing),
        ("ctts_front_config", None, H.front.Config),
        ("ctts_assembly_params", None, H.front.AssemblyParams),
        ("ctts_batch_plan", "ops", H.front.CBatchPlan),
        ("ctts_plan_op", "e1", None),
    ]
    lines = ["#include <stdio.h>", "#include <stddef.h>", '#include "ctts_plan.h"', '#include "ctts_front.h"',
             '#include "ctts_gpu.h"', '#include "ctts_b200.h"', "int main(void) {"]
    for name, last, _ in pairs:
        off = f"offsetof({name}, {last})" if last else "0"
        lines.append(f'  printf("{name} %zu %zu\\n", sizeof({name}), (size_t){off});')
    lines += ["  return 0;", "}"]
    src = tmp_path / "sizes.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "sizes"
    subprocess.run(["gcc", "-std=c99", "-I", os.path.join(H.ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = dict((l.split()[0], (int(l.split()[1]), int(l.split()[2]))) for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    for name, last, mirror in pairs:
        size, off = out[name]
        if mirror is None:
            assert size == H.front.OP_DTYPE.itemsize and off == H.front.OP_DTYPE.fields[last][1], name
            continue
        assert C.sizeof(mirror) == size, (name, C.sizeof(mirror), size)
        if last:
            assert getattr(mirror, last).offset == off, (name, last)


def test_plan_op_abi_is_32_bytes(H):
    assert H.front.OP_DTYPE.itemsize == 32
    assert C.sizeof(H.front.AssemblyParams) == 32
    assert C.sizeof(H.front.Config) == 21 * 4


def test_no_cpu_fallback_without_device(H, small_db):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    gpu = H.importlib.import_module("2026-simple-c-tts_b200.gpu")
    with pytest.raises(gpu.GpuError):
        gpu.GpuSynth(small_db, 0)


def test_product_does_not_import_the_oracle(H):
    # only tests/, smoke() and bench.py's baseline legs may touch oracle/
    pkg_dir = os.path.join(H.ROOT, "2026-simple-c-tts_b200")
    for root, _, files in os.walk(pkg_dir):
        for f in files:
            if f.endswith((".py", ".c", ".cu", ".cuh", ".h")):
                src = open(os.path.join(root, f), errors="replace").read()
                for needle in ("libctts_oracle", "libctts_ref", "ctts_oracle", "oracle/", "ctts_ref_bench"):
                    assert needle not in src, (f, needle)


def test_c_command_line_has_no_cpu_fallback(H, small_db, tmp_path):
    """The plain-C `ctts synth` driver (csrc/cli/ctts_b200.c) is built by build(); without a CUDA device
    it must fail like the library does instead of synthesising anything on the CPU."""
    import subprocess
    import torch
    b = H.importlib.import_module("2026-simple-c-tts_b200._build")
    exe = b.build_cli()
    assert os.path.exists(exe)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 1 and "synth-batch" in r.stderr
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    (tmp_path / "voice.db").write_bytes(small_db)
    r = subprocess.run([exe, "synth", "voice.db", "olá mundo", "o.wav", "1.0"], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 1 and "no CPU fallback" in r.stderr and not (tmp_path / "o.wav").exists()


def test_a_plan_is_never_destroyed_after_its_context(H, monkeypatch):
    """ctts_gpu_plan_destroy reads the plan's context: closing the context first (explicitly, or the garbage
    collector finalizing both in any order) must not lead to a destroy after ctts_gpu_free."""
    gpu = H.importlib.import_module("2026-simple-c-tts_b200.gpu")
    calls = []

    class FakeLib:
        def ctts_gpu_init(self, out, *_):
            out._obj.value = 1
            return 0

        def ctts_gpu_plan_create(self, ctx, plan, prm, off, out):
            out._obj.value = 100 + len(calls)
            calls.append(("create", out._obj.value))
            return 0

        def ctts_gpu_plan_destroy(self, h):
            calls.append(("destroy", h.value))

        def ctts_gpu_free(self, h):
            calls.append(("free", h.value))

    monkeypatch.setattr(gpu, "_lib", FakeLib())
    plan = H.front.BatchPlan(np.zeros(1, np.uint32), np.zeros(0, np.float32), np.zeros(0, H.front.OP_DTYPE))
    g = gpu.GpuSynth(b"", 0)
    a = g.create_plan(plan, H.front.AssemblyParams())
    b = g.create_plan(plan, H.front.AssemblyParams())
    b.close()
    g.close()
    a.close()
    g.close()
    assert [c[0] for c in calls].count("free") == 1
    assert all(k != "destroy" for k, _ in calls[calls.index(("free", 1)):]), calls
    assert sorted(h for k, h in calls if k == "destroy") == [100, 101]
