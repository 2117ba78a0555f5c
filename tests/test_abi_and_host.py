"""CPU-side checks: the C-ABI library builds/loads and exports every symbol the header declares (no
compute calls), the host-side kwargs logic mirrors the reference, and the product package has no CPU
fallback and never touches the oracle."""
import os
import re

import numpy as np
import pytest
import torch

import cases
from oracle import specinv_oracle as O
from spectrogram_inversion_b200 import engine

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from spectrogram_inversion_b200.build import build_library
    build_library()
    from spectrogram_inversion_b200 import _lib
    return _lib


def header_symbols():
    text = open(os.path.join(ROOT, "include", "specinv_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(specinv_[a-z_0-9]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(lib):
    handle = lib.lib()
    syms = header_symbols()
    assert len(syms) >= 15
    for s in syms:
        assert hasattr(handle, s), s
    assert sorted(lib.EXPORTS) == syms
    assert handle.specinv_abi_version() == 1
    assert handle.specinv_error_string(-2).decode().startswith("configuration not supported")


def test_binding_signatures_match_the_header():
    """Every prototype of include/specinv_b200.h against the restype / argtypes that _lib._declare gives it, type by
    type: ctypes passes a wrongly declared argument without complaint, so only this check catches one."""
    import ctypes as C
    from types import SimpleNamespace
    from spectrogram_inversion_b200 import _lib

    class Stub:
        def __getattr__(self, name):
            fn = SimpleNamespace()
            setattr(self, name, fn)
            return fn

    stub = Stub()
    _lib._declare(stub)
    types = {"int": C.c_int, "int64_t": C.c_int64, "size_t": C.c_size_t, "uint32_t": C.c_uint32, "double": C.c_double,
             "const char*": C.c_char_p, "const specinv_desc*": C.POINTER(_lib.Desc), "void**": C.POINTER(C.c_void_p),
             "int64_t*": C.POINTER(C.c_int64), "size_t*": C.POINTER(C.c_size_t), "uint32_t*": C.POINTER(C.c_uint32)}

    def ctype(decl):
        t = re.sub(r"\s*\*\s*", "*", " ".join(decl.split()))
        return types[t] if t in types else C.c_void_p if t.endswith("*") else t

    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "specinv_b200.h")).read(), flags=re.S)
    protos = re.findall(r"([\w\s*]+?)\b(specinv_\w+)\s*\(([^)]*)\)\s*;", text)
    assert sorted(name for _, name, _ in protos) == header_symbols()
    for ret, name, params in protos:
        fn = stub.__dict__.get(name)
        assert fn is not None, f"{name} is not declared"
        params = [p for p in (p.strip() for p in params.split(",")) if p and p != "void"]
        want = [ctype(re.sub(r"\s*\b\w+$", "", p)) for p in params]
        assert fn.restype is ctype(ret), (name, fn.restype, ret)
        assert len(fn.argtypes) == len(want), (name, fn.argtypes, params)
        for i, (got, w) in enumerate(zip(fn.argtypes, want)):
            assert got is w, (name, i, params[i], got, w)


def test_host_only_entry_points(lib):
    """specinv_signal_length / specinv_plan_bytes are pure host arithmetic: callable without a GPU."""
    import ctypes as C
    handle = lib.lib()
    for case in cases.ITER_CASES:
        inp = cases.make_case_inputs(case)
        mag = inp["mag"] if inp["mag"].ndim == 3 else inp["mag"][None]
        a = O.args_helper(mag.shape[1], mag.dtype, **inp["kwargs"])
        d = lib.make_desc(a.n_fft, a.hop_length, mag.shape[2], mag.shape[0], a.center,
                          lib.PAD_MODES[a.pad_mode], a.normalized, a.onesided,
                          lib.F32 if mag.dtype == np.float32 else lib.F64)
        L = C.c_int64()
        assert handle.specinv_signal_length(C.byref(d), C.byref(L)) == 0
        assert L.value == a.signal_length(mag.shape[2])
        nbytes = C.c_size_t()
        assert handle.specinv_plan_bytes(C.byref(d), C.byref(nbytes)) == 0
        assert nbytes.value > 2 * L.value * mag.dtype.itemsize
    ok = lib.make_desc(1000, 250, 10, 1, True, 0, False, True, lib.F32)       # not a power of two: direct-DFT kernels
    assert handle.specinv_signal_length(C.byref(ok), C.byref(L)) == 0 and L.value == 9 * 250
    odd = lib.make_desc(1001, 250, 10, 1, True, 0, False, False, lib.F32)     # odd n_fft: two-sided only, direct DFT
    assert handle.specinv_signal_length(C.byref(odd), C.byref(L)) == 0 and L.value == 9 * 250 + 1
    bad = lib.make_desc(1001, 250, 10, 1, True, 0, False, True, lib.F32)      # an odd n_fft has no onesided spectrum
    assert handle.specinv_signal_length(C.byref(bad), C.byref(L)) == -1
    bad = lib.make_desc(1024, 0, 10, 1, True, 0, False, True, lib.F32)
    assert handle.specinv_signal_length(C.byref(bad), C.byref(L)) == -1


@pytest.mark.parametrize("case", cases.ITER_CASES, ids=lambda c: c["name"])
def test_args_helper_mirrors_reference_rules(case):
    from spectrogram_inversion_b200.stft_args import args_helper
    inp = cases.make_case_inputs(case)
    mag = inp["mag"] if inp["mag"].ndim == 3 else inp["mag"][None]
    kw = {k: (torch.from_numpy(v) if isinstance(v, np.ndarray) else v) for k, v in inp["kwargs"].items()}
    kw["not_an_stft_kwarg"] = 123            # unknown keys are ignored (methods.py:42-46)
    got = args_helper(torch.from_numpy(mag), **kw)
    want = O.args_helper(mag.shape[1], mag.dtype, **inp["kwargs"])
    assert (got.n_fft, got.hop_length, got.win_length) == (want.n_fft, want.hop_length, want.win_length)
    assert (got.center, got.pad_mode, got.normalized, got.onesided) == (want.center, want.pad_mode, want.normalized, want.onesided)
    assert got.window.shape == (want.n_fft,) and np.array_equal(got.window.numpy(), want.window)
    assert got.signal_length(mag.shape[2]) == want.signal_length(mag.shape[2])


def test_assertions_fire_before_any_gpu_work():
    import spectrogram_inversion_b200 as S
    spec = torch.rand(65, 20)
    with pytest.raises(AssertionError):
        S.griffin_lim(spec, alpha=-0.1)
    with pytest.raises(AssertionError):
        S.griffin_lim(spec, max_iter=0)
    with pytest.raises(AssertionError):
        S.griffin_lim(spec, eva_iter=0)
    with pytest.raises(AssertionError):
        S.griffin_lim(spec, tol=-1.0)
    with pytest.raises(AssertionError):
        S.griffin_lim(spec, metric="xx")
    with pytest.raises(AssertionError):
        S.ADMM(spec, metric="xx")
    with pytest.raises(AssertionError):
        S.RTISI_LA(spec.to(torch.complex64))


def test_rtisi_unknown_kwargs_raise_like_the_reference():
    """methods.py:308-310, :385: on the non-asymmetric path the caller's kwargs reach torch.stft, so an unknown key
    is a TypeError (before any device work); the asymmetric path ignores it like griffin_lim / ADMM (:42-46)."""
    import spectrogram_inversion_b200 as S
    spec = torch.rand(65, 20)
    with pytest.raises(TypeError, match="unexpected keyword argument 'foo'"):
        S.RTISI_LA(spec, max_iter=1, verbose=0, foo=1)


@pytest.mark.skipif(torch.cuda.is_available(), reason="only meaningful on a box without a GPU")
def test_no_cpu_fallback():
    import spectrogram_inversion_b200 as S
    spec = torch.rand(65, 20)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        S.griffin_lim(spec, max_iter=2, verbose=False)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        S.sc(spec, spec)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "spectrogram_inversion_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "specinv_oracle" not in text and "import oracle" not in text and "from oracle" not in text, f
                assert "/root/reference" not in text, f


def test_metric_value_formulas():
    from spectrogram_inversion_b200.engine import metric_value
    rs = np.random.RandomState(0)
    a, b = np.abs(rs.randn(5, 9, 7)), np.abs(rs.randn(5, 9, 7))
    d, e, g = O.metric_sums(a, b)
    assert abs(metric_value("SC", d, e, g) - O.sc(a, b)) < 1e-9
    assert abs(metric_value("SNR", d, e, g) - O.snr(a, b)) < 1e-9
    assert abs(metric_value("SER", d, e, g) - O.ser(a, b)) < 1e-9


def test_package_exports_the_reference_names_and_lbfgs_runs():
    """torch_specinv/__init__.py:6 re-exports griffin_lim, RTISI_LA, ADMM, L_BFGS, phase_init; L_BFGS is generic
    autograd on a user transform (out of scope for the kernels) and runs on plain PyTorch."""
    import spectrogram_inversion_b200 as S
    for name in ("griffin_lim", "RTISI_LA", "ADMM", "L_BFGS", "phase_init", "sc", "snr", "ser", "spectral_convergence"):
        assert callable(getattr(S, name)), name
    assert S.methods.griffin_lim is S.griffin_lim and S.metrics.sc is S.sc
    x = torch.randn(400)
    f = lambda v: torch.stft(v, 64, return_complex=True, window=torch.hann_window(64)).abs()
    spec = f(x)
    y = S.L_BFGS(spec, f, samples=(400,), outer_max_iter=2, verbose=0, eva_iter=1, max_iter=5)
    assert y.shape == (400,) and not y.requires_grad


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the unmodified reference from baseline/_ref on the host cores, or the oracle port
    when it is not installed) prints one JSON line with the contract keys."""
    import json
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "cfg1",
                        "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    installed = os.path.exists(os.path.join(ROOT, "baseline", "_ref", "torch_specinv", "methods.py"))
    assert line["impl"] == "reference" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == ("reference" if installed else "port")
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and "workload" in line["config"]


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--warmup", "-1"],
                                  ["--impl", "reference", "--dump-outputs", "unused"]])
def test_bench_rejects_bad_arguments(argv, tmp_path):
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *argv], capture_output=True, text=True,
                       timeout=120, cwd=tmp_path)
    assert r.returncode == 2 and "error:" in r.stderr, r.stderr[-2000:]
    assert not (tmp_path / "unused").exists()


@pytest.mark.gpu
def test_bench_dumps_the_same_outputs_on_every_run(tmp_path):
    """`bench.py --dump-outputs DIR`: the last timed step's signal, a seeded row sample once the batch exceeds
    32 MiB (40 signals of 239872 samples: 34 rows), identical from run to run; --steps sets the timed steps."""
    import json
    import subprocess
    import sys
    got = []
    for run in ("a", "b"):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--batch",
                            "40", "--configs", "none", "--no-cpu", "--dump-outputs", str(tmp_path / run)],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert line["steps"] == 2 and len(line["e2e"]["ms_per_step_all"]) == 2
        assert sorted(os.listdir(tmp_path / run)) == ["signal.npy"]
        got.append(np.load(tmp_path / run / "signal.npy"))
    assert got[0].dtype == np.float32 and got[0].shape == (34, 937 * 256)
    assert np.isfinite(got[0]).all() and np.abs(got[0]).max() > 0
    assert np.array_equal(got[0], got[1])


def test_every_custom_op_has_a_fake_kernel():
    """SURVEY.md section 8b: each specinv_b200:: op carries a register_fake implementation, so FakeTensorMode /
    torch.compile can trace through callers without a device (the ops mutate caller-owned buffers, return nothing)."""
    from torch._subclasses.fake_tensor import FakeTensorMode
    from spectrogram_inversion_b200 import _ops
    assert len(_ops.ALL_OPS) == 16
    with FakeTensorMode():
        f = lambda *shape, dt=torch.float32: torch.empty(*shape, dtype=dt, device="cuda")
        B, T, M, L = 2, 9, 64, 8 * 32
        plan = torch.empty(4096, dtype=torch.uint8, device="cuda")
        x0, x1 = f(B, L), f(B, L)
        qm, qn = f(B, T, M, dt=torch.complex64), f(B, T, dt=torch.complex64)
        mm, mn = f(B, T, M), f(B, T)
        sums = f(2, dt=torch.float64)
        k = (128, 32, True, 0, False, True)
        assert _ops.plan_init(plan, f(128), 128, 32, T, B, True, 0, False, True) is None
        assert _ops.stft(plan, x0, qm, qn, *k) is None and _ops.istft(plan, qm, qn, x0, *k) is None
        assert _ops.gl_iter(plan, x0, x1, qm, qn, qm.clone(), qn.clone(), mm, mn, sums, 0.5, *k) is None
        assert _ops.admm_iter(plan, x0, x1, qm, qn, qm, qn, qm.clone(), qn.clone(), qm.clone(), qn.clone(), mm, mn, sums,
                              0.1, *k) is None
        with pytest.raises(RuntimeError):
            _ops.gl_iter(plan, x0, f(B, L + 1), qm, qn, qm.clone(), qn.clone(), mm, mn, sums, 0.5, *k)
        assert _ops.pack(f(B, M + 1, T), mm, mn, 128, True) is None
        assert _ops.unpack(qm, qn, f(B, M + 1, T, dt=torch.complex64), 128, True) is None
        assert _ops.metric_sums(mm, mm, f(3, dt=torch.float64)) is None
        assert _ops.phase_init(mm, mn, qm, qn, 128, 32, True) is None and _ops.spec_abs(qm, qn, mm, mn, 128, True) is None
        assert _ops.rtisi_la(plan, f(128), mm, mn, x0, f(256), 3, False, 4, 0.99, 0.1, *k) is None
        assert _ops.plan_init_ranged(plan, f(128), 128, 32, T, B, False, True, 0, 20) is None
        assert _ops.phase_init_ex(mm, mn, qm, qn, f(0, dt=torch.float64), f(B, M + 1, dt=torch.float64), 128, 32, True) is None
        assert _ops.halo_sum(f(B, 96), f(B, 96), f(B, 96)) is None and _ops.fill_padding(x0, 0, 64, L, 0) is None


class _FakeSolver(engine._Solver):
    """The real step / run_many over a launch that records whether it evaluates (no GPU): loss decreases
    geometrically."""

    def __init__(self):
        self.g, self.n_bins_total, self.calls, self.loss = 1.0, 10, [], 1.0
        self.cur, self.iterations = 0, 0
        self.sums, self._nosums = torch.zeros(2, dtype=torch.float64), torch.empty(0, dtype=torch.float64)

    def _launch(self, sums):
        self.calls.append(sums.numel() > 0)
        self.loss *= 0.9
        if sums.numel():
            sums[0], sums[1] = self.loss, 1.0


@pytest.mark.parametrize("max_iter,eva_iter", [(23, 4), (10, 10), (7, 10), (30, 1), (1, 1)])
def test_training_loop_keeps_the_reference_cadence_with_and_without_host_reads(max_iter, eva_iter):
    """methods.py:153-190: iteration i is evaluated iff i % eva_iter == eva_iter - 1.  With tol == 0, no progress bar and
    no history the loop does not read the sums back, but must evaluate on exactly the same iterations."""
    from spectrogram_inversion_b200.engine import training_loop
    want = [i % eva_iter == eva_iter - 1 for i in range(max_iter)]
    blind, watched = _FakeSolver(), _FakeSolver()
    assert training_loop(blind, max_iter, 0.0, False, eva_iter, "sc") == max_iter
    hist = []
    assert training_loop(watched, max_iter, 0.0, False, eva_iter, "sc", history=hist) == max_iter
    assert blind.calls == want and watched.calls == want
    assert [h[0] for h in hist] == [i for i in range(max_iter) if want[i]]


def test_training_loop_stops_early_like_the_reference():
    """methods.py:186-190: stop when (previous - loss) / init < tol and previous > loss (checked from the second
    evaluation on); the returned count is the number of iterations done."""
    from spectrogram_inversion_b200.engine import training_loop
    s = _FakeSolver()
    # losses at evaluations: 0.9^2, 0.9^4, ... ; relative improvement (l_{k-1} - l_k) / l_0 falls below 0.1 at k = 2
    n = training_loop(s, 100, 0.1, False, 2, "snr")
    l = [0.9 ** (2 * (k + 1)) / 10 for k in range(50)]
    k_stop = next(k for k in range(1, 50) if (l[k - 1] - l[k]) / l[0] < 0.1 and l[k - 1] > l[k])
    assert n == 2 * (k_stop + 1) and len(s.calls) == n
