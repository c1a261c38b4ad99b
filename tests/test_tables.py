"""Rule DATA tables: product header == oracle copy == compiled reference == a fresh parse of
the reference header (when CORINTHO_AI_REFERENCE names a checkout of the original project)."""
import os
import re
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from util import NO_REFERENCE, reference_file  # noqa: E402

UTIL_H = reference_file("corintho_ai/cpp/include/util.h")


def parse_generated(path, prefix):
    src = open(path).read()

    def arr(name):
        blk = src[src.index(prefix + name):]
        blk = blk[blk.index("= {") + 2:blk.index("};")]
        return [int(t, 0) for t in re.findall(r"0x[0-9a-fA-F]+|\d+", blk.replace("u,", ",").replace("u}", "}"))]

    return (np.array(arr("LineBreakers[102][3]"), np.uint32).reshape(102, 3),
            np.array(arr("GammaBits[1024]"), np.uint32),
            np.array(arr("SpaceSym[8][16]"), np.int32).reshape(8, 16),
            np.array(arr("MoveSym[8][96]"), np.int32).reshape(8, 96))


PRODUCT = os.path.join(ROOT, "corintho_ai_b200", "csrc", "corintho_tables.h")
ORACLE = os.path.join(ROOT, "oracle", "oracle_tables.inc")


def test_product_tables_equal_oracle_tables():
    a, b = parse_generated(PRODUCT, "kC"), parse_generated(ORACLE, "kO")
    for x, y in zip(a, b):
        assert (x == y).all()


def test_tables_against_compiled_reference(ref, oracle):
    lb, gam, ssym, msym = parse_generated(PRODUCT, "kC")
    for i in range(102):
        assert (ref.line_breaker(i) == lb[i]).all()
        assert (oracle.line_breaker(i) == lb[i]).all()
    for i in range(1024):
        assert ref.gamma_sample(i).view(np.uint32) == gam[i]
        assert oracle.gamma_sample(i).view(np.uint32) == gam[i]
    for k in range(8):
        assert [ref.space_symmetry(k, j) for j in range(16)] == list(ssym[k])
        assert [ref.move_symmetry(k, j) for j in range(96)] == list(msym[k])


@pytest.mark.skipif(UTIL_H is None, reason=NO_REFERENCE)
def test_tables_against_reference_header():
    import gen_tables
    masks, gam_bits, space, move = gen_tables.parse_util_h(UTIL_H)
    lb, gam, ssym, msym = parse_generated(PRODUCT, "kC")
    assert (np.array(masks, np.uint32) == lb).all()
    assert (np.array(gam_bits, np.uint32) == gam).all()
    assert (np.array(space) == ssym).all() and (np.array(move) == msym).all()


def test_survey_q1b_table_slips_are_preserved():
    """SURVEY.md Q1b: mask 84 contains b4D (id 13), mask 78 contains c4D (id 14)."""
    lb = parse_generated(PRODUCT, "kC")[0]
    assert (lb[84][0] >> 13) & 1 and not (lb[84][0] >> 17) & 1
    assert (lb[78][0] >> 14) & 1 and not (lb[78][0] >> 18) & 1


def test_symmetries_are_permutations():
    _, _, ssym, msym = parse_generated(PRODUCT, "kC")
    for k in range(8):
        assert sorted(ssym[k]) == list(range(16)) and sorted(msym[k]) == list(range(96))
