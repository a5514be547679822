"""minstd_jump's table (battle_kernels.cuh): 16807^(2^b) mod (2^31 - 1) for every bit of the largest jump a step can
ask for -- one draw per attack, at most 2 * 8191 attacks (the 14-bit slot field caps a group at 8191 agents)."""
import os
import re

from conftest import PKG

M = 2 ** 31 - 1


def table():
    src = open(os.path.join(PKG, "csrc", "battle_kernels.cuh")).read()
    m = re.search(r"minstd_jump\(uint32_t s, uint32_t n\) \{\s*const uint32_t pw\[(\d+)\] = \{([^}]*)\};.*?b < (\d+); b\+\+",
                  src, re.S)
    assert m, "minstd_jump table not found"
    values = [int(v.strip().rstrip("u")) for v in m.group(2).split(",")]
    assert int(m.group(1)) == len(values) == int(m.group(3))
    return values


def test_table_holds_the_powers_for_every_bit_of_the_largest_jump():
    pw = table()
    assert (2 * 8191).bit_length() <= len(pw)
    assert pw == [pow(16807, 2 ** b, M) for b in range(len(pw))]


def test_square_and_multiply_over_the_table_is_the_sequential_chain():
    pw = table()
    s0 = 12345
    state = s0
    for n in range(1, 2 * 8191 + 1):
        state = state * 16807 % M
        if n in (1, 4095, 4096, 4097, 8191, 8192, 12000, 16382):
            acc = s0
            for b in range(len(pw)):
                if (n >> b) & 1:
                    acc = acc * pw[b] % M
            assert acc == state, n
