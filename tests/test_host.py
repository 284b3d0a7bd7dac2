"""CPU tests of the host-side logic: C-ABI exports, planning queries, sharder, workloads, and that
the product path fails loudly (no CPU fallback) without a GPU."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import pytorch_end2end_speech_recognition_b200 as b200
from pytorch_end2end_speech_recognition_b200 import _lib, build, workloads

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    header = open(os.path.join(ROOT, "include", "b200ctc.h")).read()
    declared = set(re.findall(r"B200CTC_API\s+[\w\s\*]+?\b(b200ctc_\w+)\s*\(", header))
    assert declared == set(_lib.EXPORTED_SYMBOLS)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.b200ctc_version() == 200
    assert lib.b200ctc_status_string(0) == b"success"
    assert lib.b200ctc_status_string(1) == b"invalid value"


def test_library_is_in_tree_and_sm100a():
    assert os.path.dirname(build.LIB_PATH).startswith(ROOT)
    assert any("compute_100a" in f for f in build.NVCC_FLAGS)


def test_workspace_query_and_validation():
    n = b200.workspace_bytes([400] * 128, [800] * 128, 800, 30)
    assert n >= 128 * 800 * 201 * 32
    lib = _lib.load()
    out = ctypes.c_size_t()
    ll = (ctypes.c_int * 2)(3, 4)
    al = (ctypes.c_int * 2)(10, 99)      # act_len > T
    assert lib.b200ctc_get_workspace_size(ll, al, 20, 5, 2, ctypes.byref(out)) == 1
    al = (ctypes.c_int * 2)(10, 20)
    assert lib.b200ctc_get_workspace_size(ll, al, 20, 5, 2, ctypes.byref(out)) == 0
    assert lib.b200ctc_get_workspace_size(ll, al, 20, 0, 2, ctypes.byref(out)) == 1   # V < 1


def test_product_has_no_cpu_fallback():
    acts = torch.randn(5, 2, 4)
    with pytest.raises(RuntimeError):
        b200.ctc_loss_and_grad(acts, [1, 2], [5, 5], [1, 1])
    with pytest.raises(RuntimeError):
        b200.cpu_ctc(acts, None, None, None, None, 2, None)
    with pytest.raises(RuntimeError):
        b200.CTCLoss()(acts, torch.tensor([1, 2], dtype=torch.int32), torch.tensor([5, 5], dtype=torch.int32),
                       torch.tensor([1, 1], dtype=torch.int32))
    with pytest.raises(RuntimeError):
        b200.GreedyDecoder(0)(torch.randn(2, 5, 4), [5, 5], device="cpu")
    if not torch.cuda.is_available():
        lib = _lib.load()
        h = ctypes.c_void_p()
        assert lib.b200ctc_create(ctypes.byref(h), 0) == 2   # execution failed: no device


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "pytorch_end2end_speech_recognition_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), f
                assert "liboracle" not in src, f


def test_balance_shards_is_a_partition_and_balanced():
    wl = workloads.make_lengths_and_labels("C5")
    for n in (1, 2, 4, 8):
        shards = b200.balance_shards(wl.act_lens, wl.label_lens, wl.V, n)
        allidx = np.sort(np.concatenate(shards))
        assert np.array_equal(allidx, np.arange(wl.B))
        work = b200.shard.lattice_work(wl.act_lens, wl.label_lens, wl.V)
        loads = np.array([work[s].sum() for s in shards])
        assert loads.max() <= loads.mean() * 1.02 + work.max()
        for s in shards:
            assert np.all(np.diff(wl.act_lens[s]) <= 0)       # longest first inside a shard


def test_shard_batch_slices_labels():
    labels = np.arange(10, dtype=np.int32)
    flat, ll, al = b200.shard_batch(labels, [3, 2, 5], [9, 8, 7], np.array([2, 0]))
    assert flat.tolist() == [5, 6, 7, 8, 9, 0, 1, 2] and ll.tolist() == [5, 3] and al.tolist() == [7, 9]


@pytest.mark.parametrize("key", ["C1", "C2", "C3", "C4", "C5"])
def test_workloads_are_feasible_and_seeded(key):
    wl = workloads.make_lengths_and_labels(key)
    wl2 = workloads.make_lengths_and_labels(key)
    assert np.array_equal(wl.labels, wl2.labels) and np.array_equal(wl.act_lens, wl2.act_lens)
    cfg = workloads.CONFIGS[key]
    assert wl.B == cfg.B and wl.act_lens.max() <= cfg.T and wl.label_lens.max() <= cfg.Lmax
    assert wl.labels.min() >= 1 and wl.labels.max() < cfg.V
    off = 0
    for b in range(wl.B):
        lab = wl.labels[off:off + wl.label_lens[b]]
        assert len(lab) + int(np.sum(lab[1:] == lab[:-1])) <= wl.act_lens[b]
        off += wl.label_lens[b]
    total, strict, frames = workloads.algorithmic_bytes(wl)
    assert total > strict > 0 and frames == int(wl.act_lens.sum())
    assert np.all(np.diff(wl.act_lens) <= 0)


def test_concatenate_labels_matches_the_reference_loop():
    """Same result as the python loop of models/pytorch_v3/ctc/ctc.py:544-547 (restated inline)."""
    import pytorch_end2end_speech_recognition_b200 as b200
    rng = np.random.RandomState(3)
    ys = rng.randint(0, 50, size=(7, 12))
    y_lens = np.array([12, 0, 5, 1, 12, 7, 3], dtype=np.int32)
    expect = []
    for b in range(7):
        expect.extend(ys[b][:y_lens[b]])
    out = b200.concatenate_labels(ys, y_lens)
    assert out.dtype == np.int32 and out.tolist() == expect
    import torch
    assert b200.concatenate_labels(torch.tensor(ys), torch.tensor(y_lens)).tolist() == expect
    with pytest.raises(b200.B200CTCError):
        b200.concatenate_labels(ys, np.array([13, 0, 0, 0, 0, 0, 0]))


def test_bench_roofline_inputs_are_readable():
    """bench.py's roofline object reads the committed ncu traffic (profiles/r01_traffic.json) and the measured
    peak; a format slip there would silently turn `roofline.traffic` into null."""
    import importlib.util
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    traffic = bench.measured_traffic("C3")
    assert isinstance(traffic, int) and 3e8 < traffic < 6e8        # DRAM bytes of one C3 lattice launch
    assert bench.measured_traffic("C1") is None
    peak, kind = bench.peaks()
    assert 3000.0 < peak < 9000.0 and kind in ("measured", "fallback")
    from pytorch_end2end_speech_recognition_b200 import workloads
    wl = workloads.make_lengths_and_labels("C3")
    total, strict, frames = workloads.algorithmic_bytes(wl)
    assert frames == 102400 and strict < total < 7e8


def test_workspace_bound_covers_every_length_combination():
    rng = np.random.RandomState(3)
    for _ in range(20):
        B, T, V, Lmax = rng.randint(1, 40), rng.randint(1, 300), int(rng.choice([5, 30, 62, 200, 3386])), rng.randint(0, 120)
        ll = rng.randint(0, Lmax + 1, size=B).astype(np.int32)
        al = rng.randint(0, T + 1, size=B).astype(np.int32)
        assert b200.workspace_bytes(ll, al, T, V) <= b200.ctc.workspace_bound(T, V, B, Lmax)


def test_evaluation_entry_points_have_no_cpu_path():
    with pytest.raises(RuntimeError):
        b200.beam_search_decode(torch.randn(2, 5, 4), [5, 5], 3)
    with pytest.raises(RuntimeError):
        b200.edit_distance(torch.zeros(2, 3, dtype=torch.int32), [3, 3], torch.zeros(2, 3, dtype=torch.int32), [3, 3])
    with pytest.raises(RuntimeError):
        b200.posteriors(torch.randn(2, 5, 4))
    with pytest.raises(RuntimeError):
        b200.ctc_loss_from_padded(torch.randn(2, 5, 4), np.zeros((2, 2), np.int64), [5, 5], [1, 1])
    lib = _lib.load()
    n = ctypes.c_size_t()
    assert lib.b200ctc_beam_search_workspace(4, 100, 30, 10, ctypes.byref(n)) == 0 and n.value > 0
    assert lib.b200ctc_beam_search_workspace(4, 100, 30, 65, ctypes.byref(n)) == 1          # beam_width > 64
    assert lib.b200ctc_edit_distance_workspace(4, 50, 60, ctypes.byref(n)) == 0 and n.value >= 4 * 51 * 61
    assert lib.b200ctc_get_workspace_bound(100, 30, 4, 20, ctypes.byref(n)) == 0 and n.value > 0


def test_torch_extension_builds_in_tree_and_is_the_loss_binding():
    """The thin PyTorch C++ extension over the C ABI: built next to the library (not into site-packages), so
    that it travels with the repository snapshot and shows up as loaded native code; the loss calls go through
    that very module."""
    path = build.build_extension()
    assert path.startswith(ROOT) and os.path.exists(path)
    from pytorch_end2end_speech_recognition_b200 import ctc
    assert os.path.samefile(ctc._ext().__file__, path)
    with pytest.raises(RuntimeError):
        ctc._ext().loss_and_grad_host(torch.zeros(2, 1, 3), torch.zeros(1), torch.zeros(1), torch.zeros(1))


def test_library_variant_is_the_only_copy_in_the_process(tmp_path):
    """B200CTC_LIB redirects the whole process: the extension's dependency on libb200ctc.so resolves, by SONAME,
    to the variant the package loaded, so the loss and the ctypes diagnostics run one copy of the library."""
    import shutil
    import subprocess
    import sys
    build.build_extension()
    variant = os.path.realpath(str(tmp_path / "libb200ctc_variant.so"))     # /proc/self/maps shows real paths
    shutil.copy(build.LIB_DEFAULT, variant)
    code = ("import sys; sys.path.insert(0, %r)\n"
            "from pytorch_end2end_speech_recognition_b200 import ctc\n"
            "ctc._ext()\n"
            "print(sorted({l.split()[-1] for l in open('/proc/self/maps') if 'libb200ctc' in l}))\n" % ROOT)
    env = dict(os.environ, B200CTC_LIB=variant)
    out = subprocess.run([sys.executable, "-c", code], env=env, cwd=ROOT, check=True, capture_output=True, text=True)
    assert out.stdout.strip().splitlines()[-1] == repr([variant])


def test_extension_that_cannot_be_built_raises(monkeypatch, tmp_path):
    """No fallback: when the extension can be neither built nor imported, the loss raises."""
    from pytorch_end2end_speech_recognition_b200 import ctc

    def fail(*args, **kwargs):
        raise OSError("no host compiler")
    monkeypatch.setattr(build, "build_extension", fail)
    monkeypatch.setattr(build, "extension_path", lambda: str(tmp_path / "missing.so"))
    monkeypatch.setattr(ctc, "_EXT", None)
    with pytest.raises(b200.B200CTCError):
        ctc._ext()


def test_both_bench_arms_describe_the_same_config():
    import bench
    wl = workloads.make_lengths_and_labels("C3")
    total, _, frames = workloads.algorithmic_bytes(wl)
    a = bench.config_dict(wl, frames, total, 1)
    assert set(a) == {"workload", "per_gpu_batch", "frames_per_step_per_gpu", "algorithmic_bytes_per_step_per_gpu",
                      "n_gpus", "parallelism"}
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert src.count('"config": config_dict(') == 2                   # the b200 arm and the reference arm
