"""CPU: the candidates capacity_batch resolves (batch.capacity_candidates) are exactly the payloads hide_message gives every prefix
of a message: the MSB-first bits of head + body[:body_len] equal str_to_binary_str(f"{n}#{message[:n]}") for every n."""
import pytest

from mp3stego_b200.batch import capacity_candidates
from mp3stego_b200.steganography import str_to_binary_str

MESSAGES = {
    "ascii": "The quick brown fox jumps over the lazy dog 0123456789 #%&" * 3,
    "utf8": "aéb€c\U0001F600d üß中文 \U0001F3B5x#y" * 4,   # 2-, 3- and 4-byte characters
}


def _bits(head, body, body_len):
    return "".join(format(b, "08b") for b in head + body[:body_len])


@pytest.mark.parametrize("name", sorted(MESSAGES))
def test_every_prefix_is_the_framed_message(name):
    m = MESSAGES[name]
    body, cands = capacity_candidates(m)
    assert body == m.encode("utf-8")
    assert len(cands) == len(m) + 1
    if name == "utf8":
        assert {len(ch.encode("utf-8")) for ch in m} == {1, 2, 3, 4}
    for n, (head, bl) in enumerate(cands):
        assert len(head) <= 32
        assert _bits(head, body, bl) == str_to_binary_str(f"{n}#{m[:n]}"), n


@pytest.mark.parametrize("name", sorted(MESSAGES))
def test_bit_limit_drops_only_prefixes_that_cannot_fit(name):
    m = MESSAGES[name]
    full = capacity_candidates(m)[1]
    for limit in (0, 15, 16, 17, 100, 8 * len(m.encode("utf-8"))):
        body, cands = capacity_candidates(m, limit)
        assert cands == full[:len(cands)]
        assert all(8 * (len(h) + bl) <= limit for h, bl in cands)
        if len(cands) < len(full):
            h, bl = full[len(cands)]
            assert 8 * (len(h) + bl) > limit
