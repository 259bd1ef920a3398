"""CPU: C-ABI library loads and exports every symbol the header declares; constant-table header in
sync; host-side helpers; two-process gloo test of the only collective on the path."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def built_lib():
    from starry_process_b200 import build

    return build.build()


def test_header_symbols_exported(built_lib):
    import ctypes

    hdr = open(os.path.join(ROOT, "include", "spb200.h")).read()
    names = sorted(set(re.findall(r"\b(spb_[a-z0-9_A-Z]+)\s*\(", hdr)))
    assert len(names) >= 25
    lib = ctypes.CDLL(built_lib)
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing
    from starry_process_b200 import _lib

    assert sorted(_lib.PROTOTYPES) == names
    _lib.load()
    assert _lib.load().spb_version() >= 100


def test_sass_is_sm100a_with_fp64_tensor_ops(built_lib):
    out = subprocess.run(["cuobjdump", "-lelf", built_lib], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    sass = subprocess.run(["cuobjdump", "-sass", built_lib], capture_output=True, text=True).stdout
    assert "DMMA.8x8x4" in sass      # FP64 tensor-core MMA (mma.sync.m8n8k4.f64)
    assert "LDGSTS" in sass          # cp.async staging


def test_tables_header_in_sync():
    from starry_process_b200 import _tables as T

    off = T.offsets()
    hdr = open(os.path.join(ROOT, "starry_process_b200", "csrc", "spb_tables.h")).read()
    for name, cnt in T.LAYOUT:
        assert "#define SPB_TAB_%s %dull" % (name, off[name]) in hdr
        assert "#define SPB_TAB_%s_COUNT %dull" % (name, cnt) in hdr
    assert "#define SPB_TAB_TOTAL %dull" % off["_TOTAL"] in hdr


def test_tables_match_oracle_constants(oracle):
    """The product's own host tables against the oracle's restatement of the reference constants."""
    from starry_process_b200 import _tables as T

    blob, off = T.build_tables()
    nat = oracle.get_native("port")
    assert np.array_equal(blob[off["RX90"]:off["RX90"] + 5456], nat.Rx(15, 2, 0.5 * np.pi))
    for th in (-1.0471975511965976, 0.3):
        assert np.array_equal(T.rx_numeric(th), nat.Rx(15, 2, th))
    R1 = T.wigner_poly(15, 0, 1, 0, -1)
    R2 = oracle.wigner_poly_R(15, 0, 1, 0, -1)
    assert all(np.array_equal(a, b) for a, b in zip(R1, R2))
    wnp, Wnp = oracle.flux_precompute(15)
    assert np.array_equal(blob[off["FLUX_W"]:off["FLUX_W"] + 65536].reshape(256, 256), Wnp)
    theta, Bp, _ = oracle.spot_Bp(15)
    assert np.array_equal(blob[off["BP"]:off["BP"] + 16000].reshape(16, 1000), Bp)
    # the pinned longitude eigenvector table reproduces what this host's LAPACK gives, or at least
    # the same projector onto the significant modes
    U, t_lon, T_lon = oracle.longitude_tensors(15)
    Upin = np.load(os.path.join(ROOT, "starry_process_b200", "data", "longitude_U_ydeg15.npy"))
    assert np.abs(Upin @ Upin.T - U @ U.T).max() <= 1e-9


def test_gauss2beta_and_bounds_helpers(oracle):
    import starry_process_b200 as spb

    a, b = spb.gauss2beta(30.0, 5.0)
    ao, bo = oracle.gauss2beta(30.0, 5.0)
    assert abs(a - ao) <= 1e-15 and abs(b - bo) <= 1e-15
    mu, sg = spb.beta2gauss(a, b)
    muo, sgo = oracle.beta2gauss(ao, bo)
    assert abs(mu - muo) <= 1e-12 and abs(sg - sgo) <= 1e-12
    mus = np.array([0.0, 20.0, 85.0])
    av, bv = spb.gauss2beta(mus, np.array([5.0, 10.0, 40.0]))
    aov, bov = oracle.gauss2beta(mus, np.array([5.0, 10.0, 40.0]))
    assert np.allclose(av, aov, rtol=0, atol=1e-14) and np.allclose(bv, bov, rtol=0, atol=1e-14)
    from starry_process_b200.sp import _check_bounds

    with pytest.raises(ValueError, match="r out of bounds"):
        _check_bounds("r", 2.0, 0, 0.5 * np.pi)
    _check_bounds("r", 0.5 * np.pi + 5e-7, 0, 0.5 * np.pi)  # inside the 1e-6 tolerance


def test_no_cpu_fallback():
    """Without a CUDA device the product refuses to run instead of falling back."""
    import torch

    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    import starry_process_b200 as spb

    with pytest.raises(RuntimeError, match="CUDA"):
        spb.StarryProcess(r=10, mu=30, sigma=5, c=0.1, n=10)


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "starry_process_b200")
    for dirpath, _, files in os.walk(pkg):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, fn)).read()
                assert "import oracle" not in txt and "from oracle" not in txt
                assert "/root/reference" not in txt


def test_shard_range():
    from starry_process_b200 import shard_range

    for n, w in ((4096, 8), (10, 3), (2, 4), (0, 2)):
        spans = [shard_range(n, r, w) for r in range(w)]
        assert spans[0][0] == 0 and spans[-1][1] == n
        assert all(spans[k][1] == spans[k + 1][0] for k in range(w - 1))
        sizes = [e - b for b, e in spans]
        assert max(sizes) - min(sizes) <= 1


_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, %r)
from starry_process_b200.distributed import shard_range, gather_lnlike
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%%s" %% sys.argv[2], rank=int(sys.argv[1]), world_size=2)
n = 11
b, e = shard_range(n)
full = torch.arange(n, dtype=torch.float64) * 1.5 - 3.0
out = gather_lnlike(full[b:e].clone(), n)
assert torch.equal(out, full), (out, full)
# equal shards (weak scaling): one collective, no host sync
mine = torch.arange(4, dtype=torch.float64) + 10.0 * dist.get_rank()
out2 = gather_lnlike(mine, 8, equal_shards=True)
assert torch.equal(out2, torch.cat([torch.arange(4, dtype=torch.float64), torch.arange(4, dtype=torch.float64) + 10.0])), out2
dist.barrier()
dist.destroy_process_group()
print("ok", sys.argv[1])
"""


def test_gather_lnlike_two_ranks_gloo(tmp_path):
    import socket

    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    script = tmp_path / "worker.py"
    script.write_text(_WORKER % ROOT)
    procs = [subprocess.Popen([sys.executable, str(script), str(r), str(port)],
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT) for r in range(2)]
    outs = [p.communicate(timeout=180)[0].decode() for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    assert all("ok" in o for o in outs)


def test_design_unrolled_body_in_sync():
    """csrc/design_gen.inc (committed) is what csrc/gen_design.py generates from the product's own
    Rx(pi/2) table, and the sparsity it bakes in is the 1372-entry pattern of that table."""
    import importlib.util

    from starry_process_b200 import _tables as T

    path = os.path.join(ROOT, "starry_process_b200", "csrc", "gen_design.py")
    spec = importlib.util.spec_from_file_location("gen_design", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    inc = open(os.path.join(ROOT, "starry_process_b200", "csrc", "design_gen.inc")).read()
    assert inc == mod.generate()
    rx90 = T.rx_numeric(0.5 * np.pi)
    vals, idx = T.rx90_nonzeros(rx90)
    assert len(vals) == 1372 == dict(T.LAYOUT)["RX90_NZ"]
    dropped = np.abs(rx90).copy()
    for (l, mp, j) in idx:
        dropped[T.nwig(l - 1) + mp * (2 * l + 1) + j] = 0.0
    assert dropped.max() < 1e-15 and np.abs(vals).min() > 1e-5


def test_temporal_kernels_host_module(oracle):
    """starry_process_b200.temporal mirrors temporal.py:8-16 (callable form, torch tensors) and
    carries the kernel codes the CUDA assembly switches on."""
    import torch

    from starry_process_b200 import temporal

    t1 = np.linspace(0, 3, 17)
    t2 = np.linspace(0.5, 2, 9)
    for fn, ofn, kind in ((temporal.Matern32Kernel, oracle.Matern32Kernel, 1),
                          (temporal.ExpSquaredKernel, oracle.ExpSquaredKernel, 2)):
        K = fn(torch.tensor(t1), torch.tensor(t2), 0.7).numpy()
        assert K.shape == (17, 9)
        assert np.abs(K - ofn(t1, t2, 0.7)).max() <= 1e-15
        assert fn.spb_kind == kind


def test_sass_uses_clusters_and_tma(built_lib):
    """The small-batch Cholesky is a thread-block-cluster kernel (cluster barriers, distributed
    shared memory) and the design-matrix kernel stores through TMA: both must be in the SASS."""
    import subprocess

    sass = subprocess.run(["cuobjdump", "-sass", built_lib], capture_output=True, text=True).stdout
    assert "UCGABAR_ARV" in sass or "BAR.CLUSTER" in sass or "CGABAR" in sass  # barrier.cluster
    assert "UTMASTG" in sass                                                  # cp.async.bulk.tensor store
    assert "UTMALDG" in sass            # TMA-fed operand ring of the Cholesky kernel
    assert "DMMA" in sass


def test_sass_cholesky_orders_generic_writes_before_tma_reads(built_lib):
    """ADVICE r1 (high): the batched Cholesky writes its factor with st.global (generic proxy) and
    re-reads it through TMA (async proxy) in later panels: the kernel must carry the
    fence.proxy.async.global that orders the two (SASS: FENCE.VIEW.ASYNC.G)."""
    import subprocess

    sass = subprocess.run(["cuobjdump", "-sass", built_lib], capture_output=True, text=True).stdout
    beg = sass.index("potrf_lnlike_kernel")
    end = sass.find("Function :", beg)
    body = sass[beg:end if end > 0 else None]
    assert "UTMALDG" in body and "FENCE.VIEW.ASYNC.G" in body


def test_longitude_basis_tables():
    """The pinned longitude eigenvector table is what scripts/gen_longitude_U.py regenerates in the
    build container (SHA-256 recorded next to it), the "host" basis is this host's own eigh, both span
    the same 31-dimensional space, and only the LON_T block of the constant blob depends on it."""
    import hashlib
    import json

    from starry_process_b200 import _tables as T

    Up, Uh = T.longitude_U("pinned"), T.longitude_U("host")
    meta = json.load(open(T.PINNED_LONGITUDE[:-4] + ".json"))
    assert hashlib.sha256(np.ascontiguousarray(Up).tobytes()).hexdigest() == meta["sha256"]
    assert Up.shape == Uh.shape == (256, 31)
    assert np.abs(Up @ Up.T - Uh @ Uh.T).max() <= 1e-14
    bp, off = T.build_tables("pinned")
    bh, _ = T.build_tables("host")
    diff = np.nonzero(bp != bh)[0]
    if diff.size:   # (identical on the host that generated the pinned table)
        assert diff.min() >= off["LON_T"] and diff.max() < off["LON_T"] + 31 * T.NWIG
    with pytest.raises(ValueError):
        T.build_tables("nonsense")


def test_sass_int8_cholesky_uses_tcgen05_tmem_and_tma(built_lib):
    """potrf_i8.cuh: the panel updates of the INT8 path must be tcgen05.mma.kind::i8 (SASS UTCIMMA) with
    accumulators read back from tensor memory (LDTM), operands fetched by 4-D TMA loads (UTMALDG.4D),
    tcgen05.commit (UTCBAR) hand-offs and the generic -> async proxy fence before the planes are re-read."""
    sass = subprocess.run(["cuobjdump", "-sass", built_lib], capture_output=True, text=True).stdout
    beg = sass.index("potrf_i8_kernel")
    end = sass.find("Function :", beg)
    body = sass[beg:end if end > 0 else None]
    for mnemonic in ("UTCIMMA", "LDTM", "UTMALDG.4D", "UTCBAR", "FENCE.VIEW.ASYNC.G", "DMMA.8x8x4"):
        assert mnemonic in body, mnemonic
    # the second-moment SYRK of the Ylm moments and the lower-triangle (A Sigma) A^T (syrk_i8.cu) run on the
    # same machinery
    for kernel in ("syrk_i8_kernel", "gemm_i8_lower_kernel"):
        beg = sass.index(kernel)
        end = sass.find("Function :", beg)
        body = sass[beg:end if end > 0 else None]
        for mnemonic in ("UTCIMMA", "LDTM", "UTMALDG.4D", "UTCBAR"):
            assert mnemonic in body, (kernel, mnemonic)


def test_uniform_time_stamp_detection():
    """Host logic of spb_noise_model.uniform_dt: linspace / arange grids are recognised, anything else is not."""
    from starry_process_b200.sp import StarryProcess

    f = StarryProcess._uniform_dt
    assert f(None, np.linspace(0, 4, 1000)) == pytest.approx(4 / 999, rel=1e-14)
    assert f(None, 0.02 * np.arange(5000)) == pytest.approx(0.02, rel=1e-12)
    # a large offset rounds the stamps themselves off the grid (ulp(1e5) = 7e-10 of a step): the reference
    # sees those roundings, so this is NOT treated as uniform
    assert f(None, 1e5 + 0.02 * np.arange(5000)) == 0.0
    assert f(None, [0.0, 1.0]) == 0.0                                  # too short
    assert f(None, np.sort(np.random.default_rng(0).uniform(0, 4, 100))) == 0.0
    t = np.linspace(0, 4, 1000)
    t[500] += 1e-9
    assert f(None, t) == 0.0                                            # one displaced stamp
    assert f(None, t[::-1]) == 0.0                                      # decreasing
