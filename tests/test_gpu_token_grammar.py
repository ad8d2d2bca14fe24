"""Record-body tokens outside the canonical "(d,l)" text on the B200 (`-m gpu`) against the oracle: the checks of
token_grammar_cases.py (also run on the CPU by test_emu_token_grammar.py)."""
import pytest

import sccg_b200
import token_grammar_cases as tg

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = sccg_b200.Context(0)
    yield c
    c.close()


def test_body_table(ctx):
    tg.check_table(ctx)


def test_phase_and_length_sweep(ctx):
    tg.check_sweep(ctx)


@pytest.mark.parametrize("seeds", [range(0, 4), range(4, 8), range(8, 12)], ids=["0-3", "4-7", "8-11"])
def test_fuzzed_bodies(ctx, seeds):
    tg.check_fuzz(ctx, seeds)


def test_every_entry_point(ctx):
    tg.check_entry_corpus(ctx)


def test_own_round_trip(ctx):
    tg.check_roundtrips(ctx)
