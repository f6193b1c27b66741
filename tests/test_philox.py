"""The host Philox4x32-10 that replays mb_sample_paths' draws, against Random123's known-answer vectors (no device needed)."""
from sample_replay import philox4x32_10, uniform


def test_philox4x32_10_known_answers():
    assert philox4x32_10((0, 0, 0, 0), (0, 0)) == (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)
    ones = 0xFFFFFFFF
    assert philox4x32_10((ones,) * 4, (ones, ones)) == (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)
    assert philox4x32_10((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0)) == \
        (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)


def test_uniform_takes_53_bits_of_the_first_two_words():
    r = philox4x32_10((3, 5, 7, 0), (11, 0))
    assert uniform(11, 7, 5, 3) == ((r[0] << 21) | (r[1] >> 11)) / 2.0 ** 53
    us = [uniform(2 ** 40 + 9, k, j, t) for k in range(4) for j in range(4) for t in range(8)]
    assert all(0.0 <= u < 1.0 for u in us) and len(set(us)) == len(us)
