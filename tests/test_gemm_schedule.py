"""The persistent GEMMs' work deal on the CPU, exhaustively.

`gemm_3xtf32_persistent_kernel` (csrc/gemm_tc.cu) and `gemm_planes_kernel` (csrc/gemm_tma.cu) deal their work out on
the device from the live sizes: `pg::make_sched` gives each CTA (pair) its store tiles and its range of split-K
k-blocks, `pg::next_item` cuts that range into items.  Both are `__host__ __device__`, so `tests/native/
gemm_sched_probe.cu` runs the very same functions on the CPU for every CTA (pair) of a launch and checks that each
(problem, tile, k-block) is dealt exactly once, that no split-K item is longer than `kMaxKbPerItem` or crosses a
tile, and that store items cover the whole live K - over every G, both pair widths, four output widths, the store
and split-K problems alone and together, and the live sizes around every tile and k-block edge.

The probe is compiled with nvcc for the CPU (the test is skipped where nvcc is missing); test_gpu_live_sizes uses it
to show that its live sizes reach every branch of make_sched."""
import json
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "computational-chemistry-ai_b200", "csrc")
PROBE_SRC = os.path.join(ROOT, "tests", "native", "gemm_sched_probe.cu")
GENCODE = ["-gencode", "arch=compute_100a,code=sm_100a"]   # as build.py


def nvcc_path():
    p = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    return p if os.path.exists(p) else shutil.which("nvcc")


def build_probe(out_dir):
    nvcc = nvcc_path()
    if not nvcc:
        pytest.skip("nvcc not found")
    exe = os.path.join(str(out_dir), "gemm_sched_probe")
    r = subprocess.run([nvcc] + GENCODE + ["-O2", "-std=c++17", "--expt-relaxed-constexpr", "-o", exe, PROBE_SRC],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout
    return exe


def probe_flags(exe, cases):
    """Correctness and branch flags of make_sched for each case (PAIR, G, nprob, ovh, red0, N0, M0, K0, red1, N1, M1, K1)."""
    text = "".join(" ".join(str(int(x)) for x in c) + "\n" for c in cases)
    r = subprocess.run([exe, "flags"], input=text, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, check=True)
    out = [json.loads(line) for line in r.stdout.splitlines()]
    assert len(out) == len(cases)
    return out


def source_constants():
    """Tile sizes and the per-item k-block limit, read from gemm_persist.cuh."""
    src = open(os.path.join(CSRC, "gemm_persist.cuh")).read()
    m = re.search(r"constexpr int BM = (\d+), BN = (\d+), BK = (\d+);", src)
    assert m, "tile constants moved"
    kmax = re.search(r"constexpr int kMaxKbPerItem = (\d+);", src)
    assert kmax, "kMaxKbPerItem moved"
    return dict(BM=int(m.group(1)), BN=int(m.group(2)), BK=int(m.group(3)), kMaxKbPerItem=int(kmax.group(1)))


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    return build_probe(tmp_path_factory.mktemp("sched_probe"))


def test_schedule_constants_are_what_the_probe_checks():
    c = source_constants()
    assert (c["BM"], c["BN"], c["BK"], c["kMaxKbPerItem"]) == (128, 256, 32, 16), c


def test_every_tile_and_k_block_dealt_exactly_once(probe, tmp_path):
    r = subprocess.run([probe, "sweep"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, check=True, timeout=600)
    rep = json.loads(r.stdout)
    with open(tmp_path / "gemm_schedule_sweep.json", "w") as fh:
        json.dump(rep, fh, indent=1)
    assert rep["failures"] == 0, (rep["first_failure"], rep["first_failing_case"])
    # PAIR 1 and 2 x every G x 4 widths x (store alone, split-K alone, both in either order) x the edge sizes
    assert rep["cases"] > 2_000_000, rep["cases"]
    # the flags are recomputed by the probe; they must describe what make_sched really did
    assert rep["recompute_mismatch"] == 0
    # every branch of the balancing is exercised
    for k in ("r_zero", "r_pos", "xhi_clamped", "u_lt_g", "multi_item"):
        assert rep[k] > 0, k
    # `if (r * x_hi > U) x_hi = U / r` can never fire: T <= (U + r(t+1)cost + (G-r)t cost) / G gives
    # x_hi = T - (t+1)cost <= (U - (G-r)cost) / G <= U / G, so r * x_hi <= r * U / G <= U.  It stays in the kernel as
    # a guard; a change of the levelling that makes it reachable would show here.
    assert rep["clamp_u"] == 0


def test_flags_of_single_cases(probe):
    """The flags mode on hand-picked cases whose branches are known."""
    G = 74
    cases = [
        # split-K alone over 2 k-blocks: 2 units < 74 pairs
        (2, G, 1, 4, 1, 256, 256, 64, 0, 256, 0, 0),
        # grouped at 74 * 256 rows: the store tiles divide evenly (r = 0)
        (2, G, 2, 4, 0, 256, 74 * 256, 256, 1, 256, 256, 74 * 256),
        # one more row: r = 1
        (2, G, 2, 4, 0, 256, 74 * 256 + 1, 256, 1, 256, 256, 74 * 256 + 1),
        # 10 store tiles of cost 12 against 1 split-K unit: x_hi < 0
        (2, G, 2, 4, 0, 256, 10 * 256, 256, 1, 256, 256, 1),
        # split-K alone, 1 pair, 100 k-blocks: cut into items of <= 16
        (2, 1, 1, 4, 1, 256, 256, 3200, 0, 256, 0, 0),
    ]
    out = probe_flags(probe, cases)
    assert all(o["error"] == "" and o["recompute_ok"] for o in out), out
    assert out[0]["u_lt_g"] and not out[0]["multi_item"]
    assert out[1]["r_zero"] and not out[1]["r_pos"]
    assert out[2]["r_pos"]
    assert out[3]["xhi_clamped"]
    assert out[4]["multi_item"]
    assert not any(o["clamp_u"] for o in out)
