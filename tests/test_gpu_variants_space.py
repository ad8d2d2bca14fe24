"""Variant records of open archives (sccg_archive_variants) over the whole of their contract on the B200 through the product
library: the batteries of test_emu_variants_space.py, with long gaps of more than 4 Mbp whose first differences from the
start and from the end lie thousands of CTAs apart, and a call with more gap tiles than the B200's grid of 148 x 8 CTAs."""
import pytest

import sccg_b200
from test_emu_variants_space import (check_global_n_runs, check_long_gaps, check_many_archives, check_nrun_cache, check_odd_bytes,
                                     check_output_paths, check_scan_sizes, check_thread_tile_edges, check_token_forms)

pytestmark = pytest.mark.gpu

B200_GRID = 148 * 8                                                           # sm_count x 8 CTAs on the gap-byte kernels


@pytest.fixture(scope="module")
def ctx():
    c = sccg_b200.Context(0)
    yield c
    c.close()


def test_thread_tile_edges(ctx):
    check_thread_tile_edges(ctx)


def test_long_gaps(ctx):
    check_long_gaps(ctx, big=4_300_000, grid=B200_GRID)


def test_scan_sizes(ctx):
    check_scan_sizes(ctx)


def test_global_n_runs(ctx):
    check_global_n_runs(ctx)


def test_nrun_cache(ctx):
    check_nrun_cache(ctx)


def test_many_archives(ctx):
    check_many_archives(ctx)


def test_odd_bytes(ctx):
    check_odd_bytes(ctx)


def test_token_forms(ctx):
    check_token_forms(ctx)


def test_output_paths(ctx):
    check_output_paths(ctx)
