"""CPU tests of the host-side logic: the C-ABI library loads and exports every declared symbol, the
drop-in module keeps the reference's checkpoint ABI and argument checks, the generated FFT codelets
are correct when compiled for the host, the device GELU polynomial is accurate, and the
data-parallel helpers work over gloo with world_size 2.  No GPU compute is issued here."""
import ctypes
import os
import re
import subprocess
import sys
import tempfile

import numpy as np
import pytest
import torch

from cfdbench_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="session")
def built_lib():
    from cfdbench_b200 import build
    return build.build()


def test_library_exports_every_declared_symbol(built_lib):
    hdr = open(os.path.join(ROOT, "include", "cfdbench_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(fno_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 18
    lib = ctypes.CDLL(built_lib)
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} is declared in include/cfdbench_b200.h but not exported"
    from cfdbench_b200 import _lib
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    assert _lib.load().fno_version() == _lib.ABI_VERSION == 3


def test_struct_layouts_match_header():
    from cfdbench_b200 import _lib
    P = ctypes.sizeof(ctypes.c_void_p)
    assert ctypes.sizeof(_lib.FnoWeights) == 8 + P * (2 + 3 * 8 + 4 + 2)
    assert ctypes.sizeof(_lib.FnoWorkspace) == 6 * P
    assert ctypes.sizeof(_lib.FnoTrainSaved) == P * (9 + 8 + 8)
    assert ctypes.sizeof(_lib.FnoGrads) == P * (2 + 4 * 8 + 4)
    assert ctypes.sizeof(_lib.FnoBwdScratch) == 6 * P
    assert ctypes.sizeof(_lib.FnoWeightsBwd) == 16 * P
    assert ctypes.sizeof(_lib.FnoAdamTensors) == 8 + 32 * (4 * P + 8)


def test_size_helpers(built_lib):
    from cfdbench_b200 import _lib
    lib = _lib.load()
    assert lib.fno_act_bytes(256, _lib.ACT_F32) == 256 * 32 * 4096 * 4
    assert lib.fno_act_bytes(256, _lib.ACT_BF16) == 256 * 32 * 4096 * 2
    assert lib.fno_modes_bytes(2) == 2 * 288 * 32 * 8
    assert lib.fno_rollout_host_scratch_bytes(4, 5, 3) >= (4 * 2 + 4 + 3 * 4 * 2) * 4096 * 4 + 4 * 5 * 4


def _model(p=5, **kw):
    from cfdbench_b200 import Fno2d, loss_name_to_fn
    return Fno2d(in_chan=2, out_chan=2, n_case_params=p, loss_fn=loss_name_to_fn("nmse"), num_layers=4,
                 hidden_dim=32, modes1=12, modes2=12, device="cpu", **kw)


def test_state_dict_is_the_reference_checkpoint_abi():
    """SURVEY.md 8b: keys, shapes, dtypes must equal the reference's so checkpoints interchange."""
    m = _model(8)
    sd = m.state_dict()
    expect = synth.make_state_dict(0, n_params=8)
    assert list(sd.keys()) == list(expect.keys())
    for k, v in expect.items():
        assert tuple(sd[k].shape) == v.shape, k
        assert sd[k].dtype == (torch.complex64 if np.iscomplexobj(v) else torch.float32), k
    assert sum(p.numel() for p in m.parameters()) == 1188706 + 32 * 3  # cavity count + 3 extra lift columns
    m.load_state_dict({k: torch.from_numpy(v) for k, v in expect.items()})
    for k, v in expect.items():
        np.testing.assert_array_equal(m.state_dict()[k].numpy(), v)
    assert _model(5).state_dict()["fc0.weight"].shape == (32, 10, 1, 1)


def test_default_init_distribution_matches_reference_initialisers():
    torch.manual_seed(0)
    m = _model()
    w = m.blocks[0].conv0.weights1.detach()
    assert 0 <= float(w.real.min()) and float(w.real.max()) < 1 / 1024 and float(w.imag.max()) < 1 / 1024
    assert abs(float(w.real.mean()) - 0.5 / 1024) < 2e-5
    assert float(m.fc1.weight.abs().max()) <= 1 / np.sqrt(32) + 1e-7


def test_unsupported_configurations_raise():
    from cfdbench_b200 import Fno2d, loss_name_to_fn
    lf = loss_name_to_fn("nmse")
    with pytest.raises(ValueError):
        Fno2d(2, 2, 5, lf, 4, hidden_dim=20, device="cpu")
    with pytest.raises(ValueError):
        Fno2d(2, 2, 5, lf, 4, modes1=16, modes2=16, hidden_dim=32, device="cpu")
    with pytest.raises(ValueError):
        Fno2d(3, 2, 5, lf, 4, hidden_dim=32, device="cpu")
    with pytest.raises(ValueError):
        Fno2d(2, 2, 5, lf, 4, hidden_dim=32, padding=8, device="cpu")
    with pytest.raises(ValueError):
        Fno2d(2, 2, 5, lf, 4, hidden_dim=32, act_dtype="float16", device="cpu")


def test_no_cpu_fallback():
    from cfdbench_b200 import _lib
    m = _model()
    with pytest.raises(_lib.FnoNativeError):
        m(torch.zeros(1, 2, 64, 64), torch.zeros(1, 5))
    with pytest.raises(_lib.FnoNativeError):
        m.generate_many(torch.zeros(2, 64, 64), torch.zeros(5), torch.ones(64, 64), 2)


def test_loss_mirror_matches_reference_definition():
    from cfdbench_b200 import loss_name_to_fn
    from oracle import fno_numpy as onp
    rng = np.random.default_rng(0)
    a, b = rng.standard_normal((2, 2, 64, 64)).astype(np.float32), rng.standard_normal((2, 2, 64, 64)).astype(np.float32)
    out = loss_name_to_fn("nmse")(preds=torch.from_numpy(a), labels=torch.from_numpy(b))
    ref = onp.mse_loss(a.astype(np.float64), b.astype(np.float64), True)
    assert loss_name_to_fn("nmse").get_score_names() == ["mse", "rmse", "mae", "nmse"]
    assert loss_name_to_fn("mse").get_score_names() == ["mse", "rmse", "mae"]
    for k, v in ref.items():
        assert abs(out[k].item() - v) < 1e-5 * abs(v)
    with pytest.raises(NotImplementedError):
        loss_name_to_fn("l1")


# ------------------------------------------------------------------------------- generated codelets

HOST_SHIM = r'''
#include "fft_codelets.cuh"
using namespace fno_codelets;
extern "C" {
void h_rfft64_lo13(const float* x, float* re, float* im) { rfft64_lo13<float>(x, re, im); }
void h_c2r64_in12(const float* zre, const float* zim, float* y) { c2r64_in12<float>(zre, zim, y); }
#define CF(J) void h_cfft64_r##J(const float* a, const float* b, float* c, float* d) { cfft64_r##J<float>(a, b, c, d); }
CF(0) CF(1) CF(2) CF(3)
#define IC(R) void h_icfft64_in24_r##R(const float* a, const float* b, float* c, float* d) { icfft64_in24_r##R<float>(a, b, c, d); }
IC(0) IC(1) IC(2) IC(3) IC(4) IC(5) IC(6) IC(7)
}
'''


@pytest.fixture(scope="session")
def host_codelets():
    from cfdbench_b200 import build
    build.ensure_codelets()
    d = tempfile.mkdtemp(prefix="fno_codelets_")
    src = os.path.join(d, "shim.cpp")
    with open(src, "w") as f:
        f.write(HOST_SHIM)
    so = os.path.join(d, "shim.so")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off",
                           "-I", os.path.join(ROOT, "cfdbench_b200", "csrc"), src, "-o", so])
    return ctypes.CDLL(so)


def _fp(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))


def test_codelets_in_float32_against_numpy_fft(host_codelets):
    rng = np.random.default_rng(0)
    lib = host_codelets
    for _ in range(5):
        x = rng.standard_normal(64).astype(np.float32)
        re, im = np.zeros(13, np.float32), np.zeros(13, np.float32)
        lib.h_rfft64_lo13(_fp(x), _fp(re), _fp(im))
        ref = np.fft.fft(x.astype(np.float64))[:13]
        assert np.abs((re + 1j * im) - ref).max() < 2e-5
        z = (rng.standard_normal(64) + 1j * rng.standard_normal(64)).astype(np.complex64)
        zr, zi = np.ascontiguousarray(z.real), np.ascontiguousarray(z.imag)
        ref = np.fft.fft(z.astype(np.complex128))
        keep = list(range(12)) + list(range(53, 64))
        for j in range(4):
            bins = [k for k in keep if k % 4 == j]
            ore, oim = np.zeros(6, np.float32), np.zeros(6, np.float32)
            getattr(lib, f"h_cfft64_r{j}")(_fp(zr), _fp(zi), _fp(ore), _fp(oim))
            assert np.abs((ore + 1j * oim)[:len(bins)] - ref[bins]).max() < 3e-5
        y = (rng.standard_normal(24) + 1j * rng.standard_normal(24)).astype(np.complex64)
        full = np.zeros(64, np.complex128)
        full[list(range(12)) + list(range(52, 64))] = y
        ref = np.fft.ifft(full) * 64
        yr, yi = np.ascontiguousarray(y.real), np.ascontiguousarray(y.imag)
        for r in range(8):
            ore, oim = np.zeros(8, np.float32), np.zeros(8, np.float32)
            getattr(lib, f"h_icfft64_in24_r{r}")(_fp(yr), _fp(yi), _fp(ore), _fp(oim))
            assert np.abs((ore + 1j * oim) - ref[r::8]).max() < 2e-5
        zz = (rng.standard_normal(12) + 1j * rng.standard_normal(12)).astype(np.complex64)
        zr, zi = np.ascontiguousarray(zz.real), np.ascontiguousarray(zz.imag)
        out = np.zeros(64, np.float32)
        lib.h_c2r64_in12(_fp(zr), _fp(zi), _fp(out))
        z0 = zz.astype(np.complex128)
        z0[0] = z0[0].real  # Im of the DC bin is dropped (irfft2 semantics)
        w = np.arange(64)
        ref = np.real(sum(z0[k] * np.exp(2j * np.pi * k * w / 64) for k in range(12)))
        assert np.abs(out - ref).max() < 2e-5


def test_codelet_generator_selftest():
    subprocess.check_call([sys.executable, os.path.join(ROOT, "cfdbench_b200", "csrc", "gen_codelets.py"), "--selftest"],
                          stdout=subprocess.DEVNULL)


def test_device_gelu_polynomial_in_float32():
    """Emulate fno_common.cuh's gelu_erf in numpy float32 (coefficients parsed from the header)."""
    from math import erf
    src = open(os.path.join(ROOT, "cfdbench_b200", "csrc", "fno_common.cuh")).read()
    coef = [np.float32(float(re.search(rf"#define FNO_GELU_C{i} (\S+)f", src).group(1))) for i in range(9)]
    x = np.linspace(-8, 8, 400001).astype(np.float32)
    ax = np.abs(x)
    z = ax * np.float32(0.70710678118654752)  # no clamp: p(z) keeps decreasing beyond the fit range
    p = np.full_like(z, coef[8])
    for c in coef[7::-1]:
        p = (p * z + c).astype(np.float32)
    e = np.exp2(p.astype(np.float64)).astype(np.float32)
    g = np.maximum(x, np.float32(0)) + (z * np.float32(-0.70710678118654752)) * e
    ref = np.array([0.5 * v * (1 + erf(v / np.sqrt(2))) for v in x.astype(np.float64)])
    assert np.abs(g - ref).max() < 6e-7
    assert np.sqrt(np.mean((g - ref) ** 2)) < 1.5e-7
    # packed form used by the tensor-core epilogues: polynomial in |x| with the 1/2 folded into the exponent
    dco = [np.float32(float(re.search(rf"#define FNO_GELU_D{i} (\S+)f", src).group(1))) for i in range(9)]
    for k in range(9):  # D_k = C_k 2^{-k/2}, D_0 = C_0 - 1
        want = float(coef[k]) * 2.0 ** (-k / 2) - (1.0 if k == 0 else 0.0)
        assert abs(float(dco[k]) - want) <= 2e-7 * max(abs(want), 1e-3), (k, dco[k], want)
    q = np.full_like(ax, dco[8])
    for c in dco[7::-1]:
        q = (q * ax + c).astype(np.float32)
    assert np.all(np.diff(q[x >= 0]) < 0)  # monotone: no clamp needed
    h = np.exp2(q.astype(np.float64)).astype(np.float32)
    g2 = (np.maximum(x, np.float32(0)).astype(np.float64) - ax.astype(np.float64) * h).astype(np.float32)
    assert np.abs(g2 - ref).max() < 6e-7
    assert np.sqrt(np.mean((g2 - ref) ** 2)) < 1.5e-7


def test_device_gelu_degree5_variant_in_float32():
    """gelu_erf2_deg5_batch (project kernel, bf16 storage): degree-5 fit, max abs error below torch's own fp32 GELU."""
    from math import erf
    src = open(os.path.join(ROOT, "cfdbench_b200", "csrc", "fno_common.cuh")).read()
    eco = [np.float32(float(re.search(rf"#define FNO_GELU_E{i} (\S+)f", src).group(1))) for i in range(6)]
    xw = np.linspace(-40, 40, 800001).astype(np.float32)   # well beyond the fit range [0, 8]: the tail must underflow
    aw = np.abs(xw)
    q = np.full_like(aw, eco[5])
    for c in eco[4::-1]:
        q = (q * aw + c).astype(np.float32)
    assert np.all(np.diff(q[xw >= 0]) < 0)  # monotone decreasing: 2^q underflows, no clamp needed
    h = np.exp2(q.astype(np.float64)).astype(np.float32)
    g = (np.maximum(xw, np.float32(0)).astype(np.float64) - aw.astype(np.float64) * h).astype(np.float32)
    ref = np.array([0.5 * v * (1 + erf(v / np.sqrt(2))) for v in xw.astype(np.float64)])
    assert np.abs(g - ref).max() < 8e-7
    t = torch.nn.functional.gelu(torch.from_numpy(xw)).numpy()
    assert np.abs(g - ref).max() < np.abs(t - ref).max()   # more accurate than torch's fp32 nn.GELU() (1.3e-6)
    sel = np.abs(xw) <= 8
    assert np.sqrt(np.mean((g[sel] - ref[sel]) ** 2)) < 2.5e-7


# ----------------------------------------------------------------------------- data-parallel (gloo)

def _dp_worker(rank, world, port, tmp):
    import torch.distributed as dist
    from cfdbench_b200 import dp
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    r, l, w = dp.init_from_env("gloo")
    assert (r, w) == (rank, world)
    # shard ranges tile the batch
    spans = [dp.shard_range(2048, i, world) for i in range(world)]
    assert spans[0][0] == 0 and spans[-1][1] == 2048 and all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
    # flat gradient buffer with an interleaved complex segment
    g = torch.Generator().manual_seed(rank)
    flat = torch.randn(1000, generator=g)
    cview = torch.view_as_complex(flat[100:300].view(100, 2))
    expect = sum(torch.randn(1000, generator=torch.Generator().manual_seed(i)) for i in range(world)) / world
    dp.allreduce_mean_(flat)
    assert torch.allclose(flat, expect, atol=1e-6)
    assert torch.allclose(torch.view_as_real(cview).reshape(-1), expect[100:300], atol=1e-6)
    with pytest.raises(TypeError):
        dp.allreduce_mean_(cview)
    assert dp.max_over_ranks(float(rank)) == float(world - 1)
    dist.barrier()
    dist.destroy_process_group()
    open(os.path.join(tmp, f"ok{rank}"), "w").write("ok")


def test_data_parallel_helpers_gloo_world2(tmp_path):
    import torch.multiprocessing as mp
    port = 29500 + os.getpid() % 2000
    mp.spawn(_dp_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert os.path.exists(tmp_path / "ok0") and os.path.exists(tmp_path / "ok1")


def test_shard_range_ragged():
    from cfdbench_b200 import dp
    assert [dp.shard_range(10, r, 4) for r in range(4)] == [(0, 3), (3, 6), (6, 8), (8, 10)]
    assert dp.shard_range(1, 0, 1) == (0, 1)


# ----------------------------------------------------------------------------- bench.py contract (reference arm, CPU)

def test_bench_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` (the reference's CPU path, timed on the host) must print exactly one JSON line
    with the driver's keys and the same metric / unit / workload naming as the GPU arm."""
    import json
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--batch", "2"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in d, key
    assert d["impl"] == "reference" and d["metric"] == "fno_rollout_steps_per_sec" and d["unit"] == "steps/s"
    assert d["higher_is_better"] is True and d["gpu_launches"] == 0 and d["value"] > 0
    ref_built = os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "src", "models", "fno"))
    assert d["cpu_baseline"]["kind"] == ("reference" if ref_built else "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["cpu_model"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    import bench
    assert d["config"]["workload"] == bench.workload_name(2)


def test_bench_dump_outputs_writes_float32_within_the_limit(tmp_path):
    """bench.py --dump-outputs: one float32 .npy per array; over the byte limit, the same seeded batch rows every time."""
    import bench
    a = torch.arange(8 * 2 * 4 * 4, dtype=torch.float32).reshape(8, 2, 4, 4)
    bench.dump_outputs(str(tmp_path / "full"), {"x": a})
    np.testing.assert_array_equal(np.load(tmp_path / "full" / "x.npy"), a.numpy())
    limit = 2 * 3 * a[0].numel() * 4   # two arrays, three rows each
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), {"x": a, "y": a.double()}, limit=limit)
    x1, y1, x2 = (np.load(tmp_path / d / f"{n}.npy") for d, n in (("s1", "x"), ("s1", "y"), ("s2", "x")))
    assert x1.dtype == y1.dtype == np.float32 and x1.shape == (3, 2, 4, 4) and x1.nbytes + y1.nbytes <= limit
    np.testing.assert_array_equal(x1, x2)
    rows = x1[:, 0, 0, 0].astype(int) // a[0].numel()
    np.testing.assert_array_equal(x1, a.numpy()[rows])
    assert list(rows) == sorted(set(rows))


def test_bench_train_line_names_the_allreduce_mode():
    """bench.py: the train-step line states the all-reduce mode actually used (Fno2d.dp_segments), only when world > 1."""
    import bench
    one = bench._train_result(2.0, 64, 1, "cavity", True, "f32", "one")
    assert one["value"] == 500.0 and one["global_batch"] == 64 and "all-reduce" not in one["what"]
    two = bench._train_result(2.0, 64, 2, "cylinder", True, "bf16", "one")
    assert two["global_batch"] == 128 and "ONE NCCL AVG all-reduce" in two["what"] and "bf16 storage" in two["what"]
    assert "per gradient segment" in bench._train_result(2.0, 64, 2, "cavity", False, "f32", "all")["what"]
