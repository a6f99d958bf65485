"""The host-facing downloads (sph_download, _diag, _tree, _neighbours) in the multi-rank forms that the other suites do
not reach: the replicated form's tree and neighbour sets, the neighbour list form under domains, and a domain that owns
no rows.  One process per rank on cuda:0 (host-segment collectives), as in test_multi_gpu.py."""
import numpy as np
import pytest

from summersph_b200 import MODE_VARIABLE_H, MODE_FIXED_H
from test_multi_gpu import run_ranks, assert_identical

pytestmark = pytest.mark.gpu

SPH_ERR_STATE = -5
STATE = ("x", "y", "z", "vx", "vy", "vz", "u", "m", "alpha", "h", "s_x", "s_y", "s_z", "s_vx", "s_vy", "s_vz", "s_m", "meta")


@pytest.mark.parametrize("mode", [MODE_VARIABLE_H, MODE_FIXED_H])
def test_replicated_tree_and_neighbours_bit_identical(mode, built_engine, tmp_path):
    """Replicated form: keys, order, levels, cells, sizes, neighbour counts and hashes - and everything else the worker
    downloads - are bit-identical to one rank."""
    ref = run_ranks(tmp_path, "one", 1, "host", mode, extra="tree")[0]
    for world in (2, 3):
        res = run_ranks(tmp_path, f"rep{world}", world, "host", mode, extra="tree")
        for r in range(world):
            assert_identical(res[r], ref, f"replicated world {world} rank {r}")


def test_domains_refuse_neighbour_list_on_every_rank(built_engine, tmp_path):
    """Under domains the CSR list form is refused with SPH_ERR_STATE on every rank, before any collective (no rank waits)."""
    res = run_ranks(tmp_path, "nbl", 3, "host", MODE_VARIABLE_H, steps=0, n=30_000, domains=1, extra="nblist")
    for r in range(3):
        assert int(res[r]["nblist_code"][0]) == SPH_ERR_STATE, (r, res[r]["nblist_code"])
        assert "the list form is not available under the domain decomposition" in str(res[r]["nblist_msg"][0]), r


def test_replicated_neighbour_list_works(built_engine, tmp_path):
    res = run_ranks(tmp_path, "nbr", 2, "host", MODE_VARIABLE_H, n=30_000, extra="nblist")
    for r in range(2):
        assert int(res[r]["nblist_code"][0]) == 0, (r, res[r].get("nblist_msg"))


@pytest.mark.parametrize("world", [2, 3])
def test_domain_without_rows_downloads(world, built_engine, tmp_path):
    """Rank 0 owns every row, the other domains none: the downloads decide "no particles" from the global count, so
    every rank takes part in the gathers and receives all rows (a rank that refused alone would leave its peers waiting)."""
    ref = run_ranks(tmp_path, "one0", 1, "host", MODE_VARIABLE_H, steps=0, n=30_000)[0]
    res = run_ranks(tmp_path, f"empty{world}", world, "host", MODE_VARIABLE_H, steps=0, n=30_000, domains=1, ics="rank0")
    for r in range(world):
        for k in STATE:
            assert np.array_equal(res[r][k], ref[k], equal_nan=True), (world, r, k)
        for k in res[0]:
            if k.startswith("d_"):      # no evaluation ran: whatever rank 0 holds, every rank receives the same values
                assert np.array_equal(res[r][k], res[0][k], equal_nan=True), (world, r, k)
