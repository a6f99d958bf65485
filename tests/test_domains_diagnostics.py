"""On-demand diagnostics under the Morton-domain decomposition (params.decomposition = 1): `sph_conserved`,
`simulate(drift=...)` and `sph_column_density` on N ranks, one process per rank, against the single-rank run.

`sph_conserved` is collective there: every rank walks its own particles over [top | local | LET] (the same nodes in the
same order as the single-rank walk, so each particle's term has the same bits), the ranks' totals are all-gathered and
folded in rank order, and every rank returns the same sums; only the grouping of the sum over particles differs from
one rank.  `sph_column_density` scatters every rank's own rows and sums the images over the ranks.

The ranks share cuda:0 through the host-segment communicator (runs on the 1-GPU box); the NCCL case needs 2 GPUs.
Scales of test_widen_conserved.assert_same_sums: |value| for energies and mass, sqrt(2 E_kin M) for momentum, |L| for
angular momentum."""
import json
import os
import subprocess
import sys
import uuid

import numpy as np
import pytest

from summersph_b200 import MODE_FIXED_H, MODE_VARIABLE_H, FLAG_SOFT_USES_HI
from summersph_b200._abi import CONSERVED, conserved_dict

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
WORKER = os.path.join(HERE, "_dd_diag_rank.py")
MODES = {"fixed": MODE_FIXED_H, "variable": MODE_VARIABLE_H, "variable_soft_hi": MODE_VARIABLE_H | FLAG_SOFT_USES_HI}


def _ngpu():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def run_diag(tmp_path, tag, world, spec, comm="host"):
    """Launch `world` worker processes on one scenario; returns one result dict per rank."""
    token = "-"
    if world > 1:
        if comm == "nccl":
            import ctypes as C
            from summersph_b200.engine import load_library
            buf = (C.c_char * 128)()
            assert load_library().sph_comm_unique_id(buf) == 0
            token = bytes(buf).hex()
        else:
            token = "/sphdiag_" + uuid.uuid4().hex[:16]
    procs, outs = [], []
    for r in range(world):
        out = str(tmp_path / f"{tag}_r{r}.npz")
        outs.append(out)
        dev = r if comm == "nccl" else 0
        procs.append(subprocess.Popen([sys.executable, WORKER, str(r), str(world), comm, str(dev), token, out, json.dumps(spec)],
                                      stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    logs = []
    for p in procs:
        try:
            o, _ = p.communicate(timeout=float(os.environ.get("SPH_TEST_RANK_TIMEOUT", "900")))
        except subprocess.TimeoutExpired:
            for q in procs:
                q.kill()
            raise
        logs.append(o)
    for r, p in enumerate(procs):
        assert p.returncode == 0, f"rank {r} failed:\n{logs[r][-4000:]}"
    return [dict(np.load(o)) for o in outs]


@pytest.fixture(autouse=True)
def _library(built_engine):
    """The workers load the engine library: build it first whichever test runs alone."""
    return built_engine


def assert_sums_close(got, ref, tol, what):
    """got, ref: the 12 sph_conserved slots; scales as in test_widen_conserved.assert_same_sums."""
    g, o = conserved_dict(got), conserved_dict(ref)
    for k in ("e_kin", "e_int", "e_pot", "e_pot_gas", "e_pot_sink", "mass"):
        sc = max(abs(o[k]), 1e-300)
        assert abs(g[k] - o[k]) <= tol * sc, (what, k, g[k], o[k])
    p_scale = np.sqrt(2 * abs(o["e_kin"]) * o["mass"]) or 1.0
    l_scale = max(np.sqrt(o["lx"] ** 2 + o["ly"] ** 2 + o["lz"] ** 2), 1e-300)
    for k in ("px", "py", "pz"):
        assert abs(g[k] - o[k]) <= tol * p_scale, (what, k, g[k], o[k])
    for k in ("lx", "ly", "lz"):
        assert abs(g[k] - o[k]) <= tol * l_scale, (what, k, g[k], o[k])


def assert_ranks_identical(res, key):
    for r in range(1, len(res)):
        assert np.array_equal(res[r][key], res[0][key]), (key, r)


@pytest.fixture(scope="module")
def upload_ref(tmp_path_factory, built_engine):
    """Single-rank sums straight after the upload, and the oracle's, per mode."""
    from summersph_b200 import default_params, ics
    from oracle.oracle import Oracle
    d = tmp_path_factory.mktemp("diag_ref")
    out = {}
    b, s = ics.keplerian_disc(60_000, seed=12)
    for name, mode in MODES.items():
        one = run_diag(d, f"one_{name}", 1, {"scenario": "upload", "mode": mode})[0]["cons"]
        o = Oracle(default_params(mode)); o.upload(b, s)
        out[name] = (one, np.array([o.conserved()[k] for k in CONSERVED]))
    return out


@pytest.mark.parametrize("name", list(MODES))
@pytest.mark.parametrize("world", [2, 3, 4])
def test_conserved_after_upload(world, name, upload_ref, tmp_path):
    """The tree (migration, halo, LET) is built inside the call; every rank returns the same bits, equal to one rank up
    to the grouping of the sum over particles."""
    res = run_diag(tmp_path, f"up{world}_{name}", world, {"scenario": "upload", "mode": MODES[name]})
    assert_ranks_identical(res, "cons")
    one, orc = upload_ref[name]
    assert_sums_close(res[0]["cons"], one, 1e-12, f"world {world} {name} vs one rank")
    assert_sums_close(res[0]["cons"], orc, 1e-10, f"world {world} {name} vs oracle")


@pytest.mark.parametrize("sinks", [1, 2])
def test_conserved_after_accretion_and_removals(sinks, tmp_path):
    """Three loop bodies of the accretion + bounds set-up: particles left, so the call rebuilds the tree."""
    spec = {"scenario": "removals", "mode": MODE_VARIABLE_H, "steps": 3, "sinks": sinks}
    one = run_diag(tmp_path, f"rm1_{sinks}", 1, spec)[0]
    assert one["meta"][2] < 60_000, "the set-up is meant to remove particles"
    for world in (2, 3):
        res = run_diag(tmp_path, f"rm{world}_{sinks}", world, spec)
        assert_ranks_identical(res, "cons")
        assert np.array_equal(res[0]["meta"], one["meta"]), (world, res[0]["meta"], one["meta"])
        assert_sums_close(res[0]["cons"], one["cons"], 1e-10, f"world {world} sinks {sinks}")


@pytest.mark.parametrize("world", [2, 3])
def test_conserved_quiet_run_reuses_the_tree(world, tmp_path):
    """Nothing is removed in four loop bodies: the call walks evaluation B's tree and LET."""
    spec = {"scenario": "quiet", "mode": MODE_VARIABLE_H, "steps": 4}
    one = run_diag(tmp_path, f"q1_{world}", 1, spec)[0]
    assert one["meta"][2] == 60_000
    res = run_diag(tmp_path, f"q{world}", world, spec)
    assert_ranks_identical(res, "cons")
    assert_sums_close(res[0]["cons"], one["cons"], 1e-10, f"quiet world {world}")


def test_conserved_does_not_change_the_run(tmp_path):
    """A domain run that asks for the sums before and between its steps ends where the same run without them ends."""
    res = run_diag(tmp_path, "ask", 2, {"scenario": "ask", "mode": MODE_VARIABLE_H, "steps": 3})
    for r in range(2):
        assert np.array_equal(res[r]["run1"], res[r]["run0"]), (r, res[r]["run0"], res[r]["run1"])


def test_simulate_drift_on_every_rank(tmp_path):
    """simulate(drift={}) on every rank of a 2-rank domain engine: one report, equal to the single-rank one."""
    spec = {"scenario": "simulate", "mode": MODE_VARIABLE_H, "steps": 3}
    one = run_diag(tmp_path, "sim1", 1, spec)[0]
    res = run_diag(tmp_path, "sim2", 2, spec)
    for k in ("first", "last", "report", "meta"):
        assert_ranks_identical(res, k)
    assert np.array_equal(res[0]["meta"][:2], one["meta"][:2]) and res[0]["meta"][0] == 3
    assert_sums_close(res[0]["first"], one["first"], 1e-10, "simulate first")
    assert_sums_close(res[0]["last"], one["last"], 1e-10, "simulate last")


@pytest.mark.parametrize("world", [2, 3])
def test_column_density_sums_the_domains(world, tmp_path):
    """Every rank returns the image of all resident gas (own rows only: the halo copies are not counted twice), equal to
    the single-rank image; the 1024 x 1024 frame is reduced in several host-communicator chunks."""
    spec = {"scenario": "image", "mode": MODE_FIXED_H}
    one = run_diag(tmp_path, f"img1_{world}", 1, spec)[0]
    res = run_diag(tmp_path, f"img{world}", world, spec)
    assert sum(int(r["halo"][0]) for r in res) > 0, "the build inside sph_conserved fills a halo"
    for k in ("img_z", "img_x", "img_big"):
        assert_ranks_identical(res, k)
        ref = one[k]
        assert np.max(np.abs(res[0][k] - ref)) <= 1e-13 * ref.max(), (world, k)
    px = (240.0 / 1024) ** 2
    assert res[0]["img_big"].sum() * px == pytest.approx(float(one["mass"][0]), rel=2e-3)
    assert res[0]["img_big"].min() >= 0.0


@pytest.mark.skipif(_ngpu() < 2, reason="needs 2 GPUs")
def test_conserved_nccl_two_gpus(upload_ref, tmp_path):
    res = run_diag(tmp_path, "nccl2", 2, {"scenario": "upload", "mode": MODE_VARIABLE_H}, comm="nccl")
    assert_ranks_identical(res, "cons")
    one, orc = upload_ref["variable"]
    assert_sums_close(res[0]["cons"], one, 1e-12, "nccl vs one rank")
    assert_sums_close(res[0]["cons"], orc, 1e-10, "nccl vs oracle")
