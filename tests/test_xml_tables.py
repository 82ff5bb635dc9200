"""The 128-bit power-of-five table of the device number parser (diasss_b200/csrc/pow5_128.inc), recomputed from its
definition with Python integers: entry q is 5^q scaled into [2^127, 2^128), truncated for q >= 0 and rounded up from the
truncated reciprocal for q < 0 (Lemire, "Number Parsing at a Gigabyte per Second", 2021)."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _committed():
    text = open(os.path.join(ROOT, "diasss_b200", "csrc", "pow5_128.inc")).read()
    return [(int(h, 16) << 64) | int(lo, 16) for h, lo in re.findall(r"0x([0-9a-f]{16})ull, 0x([0-9a-f]{16})ull", text)]


def test_pow5_table_matches_its_definition():
    got = _committed()
    assert len(got) == 308 + 342 + 1
    for q, v in zip(range(-342, 309), got):
        assert (1 << 127) <= v < (1 << 128), q
        if q >= 0:
            p = 5 ** q                                     # the leading 128 bits of 5^q
            want = p << (128 - p.bit_length()) if p.bit_length() <= 128 else p >> (p.bit_length() - 128)
        else:
            p = 5 ** -q
            z = p.bit_length()
            want = (1 << (z + 127)) // p + 1 if q >= -27 else (1 << (2 * z + 128)) // p + 1
            want >>= max(0, want.bit_length() - 128)
        assert v == want, q
    # spot values: 5^0 = 2^127, 5^1 = 0b101 << 125, 5^-1 = 0xcc..cd
    assert got[342] == 1 << 127 and got[343] == 5 << 125 and got[341] == int("cc" * 15 + "cd", 16)


def test_generator_reproduces_the_committed_file():
    import importlib.util
    spec = importlib.util.spec_from_file_location("gen_pow5", os.path.join(ROOT, "tools", "gen_pow5.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    assert gen.render() == open(os.path.join(ROOT, "diasss_b200", "csrc", "pow5_128.inc")).read()
