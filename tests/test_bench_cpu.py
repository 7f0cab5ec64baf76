"""bench.py control flow without a GPU: every device call is replaced by a stub, so that the step accounting of both
arms (passes per step, images counted, identical `config` objects, bytes per step) is checked on the CPU."""
import contextlib
import ctypes
import importlib.util
import io
import json
import os
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _FakeFn:
    def __init__(self, name, lib):
        self.name, self.lib, self.restype, self.argtypes = name, lib, None, None

    def __call__(self, *a):
        self.lib.calls[self.name] = self.lib.calls.get(self.name, 0) + 1
        if "ExtractSift" in self.name:
            a[0]._obj.numPts = 1710
        if "MatchSiftData" in self.name:
            return 0.2
        if "AllocSiftTempMemory" in self.name:
            return 1234
        return 0


class _FakeLib:
    def __init__(self):
        self.calls, self.fns = {}, {}

    def __getattr__(self, n):
        if n.startswith("_Z") or n.startswith("cuda"):
            return self.__dict__["fns"].setdefault(n, _FakeFn(n, self))
        raise AttributeError(n)


def _load_bench(monkeypatch):
    monkeypatch.setattr(sys, "argv", ["bench.py"])
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    small = np.zeros((bench.H, bench.W), np.float32)
    monkeypatch.setattr(bench, "bind_numa", lambda i: {"bound": False})
    monkeypatch.setattr(bench, "make_images", lambda rank, distinct, standalone=False: [small] * distinct)
    return bench


def _args(impl):
    return types.SimpleNamespace(gpus=1, steps=20, warmup=5, impl=impl, batch=32, rounds=0, streams=2, distinct=8, no_cpu=True,
                                 dump_outputs=None)


def test_both_arms_count_the_same_work(monkeypatch):
    bench = _load_bench(monkeypatch)
    # ---- reference arm: the library handle is a stub
    fake = _FakeLib()
    monkeypatch.setattr(bench.ctypes, "CDLL", lambda *a, **k: fake)
    monkeypatch.setattr(bench, "load_cudart", lambda: _FakeLib())

    class SM:
        @staticmethod
        def synth_descriptors(n, seed):
            return np.zeros(n, np.dtype([("x", "f4", 144)]))
    monkeypatch.setattr(bench, "synth_module", lambda standalone=False: SM)
    monkeypatch.setattr(bench.os.path, "exists", lambda p: True)
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        bench.run_reference(_args("reference"))
    ref = json.loads(buf.getvalue().strip().splitlines()[-1])
    extracts = [v for k, v in fake.calls.items() if "ExtractSift" in k][0]
    assert ref["config"]["images_per_step_per_gpu"] == 384                  # 12 passes over 32 images
    assert extracts == (5 + 20 + 10) * 384                                  # warm-up + timed + e2e steps
    assert ref["impl"] == "reference" and ref["e2e"]["h2d_bytes_per_step"] == 384 * bench.W * bench.H * 4

    # ---- product arm: the package is a stub
    class L:
        n = 0
        buf = (ctypes.c_float * (bench.W * bench.H))()
        def cs_device_sync(self): pass
        def cs_max_batch(self): return 32
        def cs_event_create(self): return 1
        def cs_event_record(self, e, h): pass
        def cs_event_elapsed_ms(self, a, b): return 320.0
        def cs_launch_count(self): return L.n
        def cs_extractor_host_image_at(self, h, i): return ctypes.addressof(L.buf)
    lib = L()

    class Img:
        d_data = 1
        def Allocate(self, *a): return self
        def Download(self): return 0.0

    class Ex:
        submitted = 0
        def __init__(self, *a, **k): self.handle = 1
        def submit_device_batch(self, ptrs, *a):
            L.n += 6
            Ex.submitted += len(ptrs)
        def submit_host_batch(self, ptrs, *a): pass
        def wait_batch(self, b): return [1710] * b
    cs = types.SimpleNamespace(InitCuda=lambda d: None, lib=lambda: lib, CudaImage=Img, Extractor=Ex,
                               iAlignUp=lambda a, b: a if a % b == 0 else a - a % b + b)
    monkeypatch.setitem(sys.modules, "cudasift_b200", cs)
    for f in ("bench_dropin", "bench_roofline", "bench_match"):
        monkeypatch.setattr(bench, f, lambda *a, **k: {})
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        bench.run_product(_args("b200"))
    prod = json.loads(buf.getvalue().strip().splitlines()[-1])
    assert Ex.submitted == (5 + 20) * 384
    assert abs(prod["value"] - 20 * 384 / 0.320) < 1.0                       # images of the timed steps / device time
    assert prod["config"] == ref["config"]                                   # what the driver compares (same_config)
    assert prod["e2e"]["images"] >= 512 and prod["e2e"]["h2d_bytes_per_step"] == 384 * bench.W * bench.H * 4
    assert prod["gpu_launches"] == 20 * 12 * 2 * 6


def test_dump_outputs_layout_and_cap(monkeypatch, tmp_path):
    """--dump-outputs: float arrays only, images in order, each image's keypoints in canonical order whatever order the
    device wrote them in, and a fixed seeded sample of rows (named in rows.npy) when the whole would exceed the cap."""
    bench = _load_bench(monkeypatch)
    from cudasift_b200.records import SIFT_DTYPE
    rng = np.random.default_rng(1)
    imgs = []
    for n in (5, 0, 7):
        p = np.zeros(n, SIFT_DTYPE)
        for f in bench.DUMP_FIELDS:
            p[f] = rng.random(n)
        p["data"] = rng.random((n, 128))
        imgs.append(p)

    def load(d):
        return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}
    bench.dump_outputs(str(tmp_path / "a"), imgs)
    bench.dump_outputs(str(tmp_path / "b"), [p[::-1] for p in imgs])          # another arrival order
    a, b = load(tmp_path / "a"), load(tmp_path / "b")
    assert sorted(a) == ["counts", "descriptors", "keypoints"]
    for k in a:
        assert a[k].dtype in (np.float32, np.float64) and np.array_equal(a[k], b[k]), k
    assert a["counts"].tolist() == [5, 0, 7] and a["keypoints"].shape == (12, 7) and a["descriptors"].shape == (12, 128)
    first = np.sort(imgs[0], order=["subsampling", "ypos", "xpos", "scale", "orientation"])
    assert np.array_equal(a["keypoints"][:5, 0], first["xpos"]) and np.array_equal(a["descriptors"][:5], first["data"])
    row_bytes = 4 * (7 + 128)
    cap = 3 * 8 + 4 * 128 + 6 * (row_bytes + 8)                                # room for 6 of the 12 rows
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", cap)
    bench.dump_outputs(str(tmp_path / "c"), imgs)
    bench.dump_outputs(str(tmp_path / "d"), imgs)
    c, d = load(tmp_path / "c"), load(tmp_path / "d")
    rows = c["rows"].astype(int)
    assert len(rows) == 6 and np.all(np.diff(rows) > 0) and np.array_equal(c["rows"], d["rows"])
    assert np.array_equal(c["keypoints"], a["keypoints"][rows]) and np.array_equal(c["descriptors"], a["descriptors"][rows])
    assert sum(v.nbytes for v in c.values()) <= cap
