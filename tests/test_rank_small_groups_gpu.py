"""Tie groups of 2..32 words ranked by LCP walks along the group's most frequent word, one warp per
window of 32 group starts (rank_small_lcp_k), against the oracle and against the warp chunk-pass
kernels it replaced (PFPB200_RANK_WARP_PASSES=1).  Bit-exact: every byte of the five streams."""
import os

import numpy as np
import pytest

from conftest import assert_same_files
from oracle import pfp_oracle as orc

pytestmark = pytest.mark.gpu

DNA = b"ACGT"
PROTEIN = b"ACDEFGHIKLMNPQRSTVWY"     # 20 letters: too many for the compacted first key


@pytest.fixture(scope="module")
def scanners(pkg):
    """{"walks": default context, "passes": context with PFPB200_RANK_WARP_PASSES=1}"""
    out = {"walks": pkg.pfp.Scanner(0)}
    os.environ["PFPB200_RANK_WARP_PASSES"] = "1"
    try:
        out["passes"] = pkg.pfp.Scanner(0)
    finally:
        os.environ.pop("PFPB200_RANK_WARP_PASSES", None)
    yield out
    for s in out.values():
        s.close()


def check_both(scanners, text, w, p, what):
    want = orc.parse(text, w, p)
    for arm, s in scanners.items():
        assert_same_files(s.parse_host(text, w, p, sai=True), want, f"{what} ({arm})")
    return want


def family_offsets(wlen, w):
    """Substitution offsets inside a word of wlen bytes (its first and last w bytes are the triggers):
    both sides of every 8-byte chunk border, then the last byte in front of the closing trigger."""
    offs = []
    for k in range(2, wlen // 8 + 1):
        offs += [8 * k - 1, 8 * k, 8 * k + 1]
    offs.append(wlen - w - 1)
    return [o for o in offs if w <= o <= wlen - w - 1]


def family_text(seed, sizes, alphabet=DNA, w=10, p=100, base_len=1200, filler=300, truncated_tail=True):
    """For each size H: a random base copied H times, copy j > 0 with one substitution in the same
    word of the base (a different offset or letter per copy), so that the word forms a family of
    exactly H distinct words.  Substitutions that would add or remove a trigger are skipped.
    Random filler between families; the text ends in a copy cut inside the family's word, so the
    last word is a family member's prefix followed by the w bytes 0x02 that close the text."""
    rng = np.random.default_rng(seed)
    letters = np.frombuffer(alphabet, np.uint8)
    parts = []
    last_cut = None
    for H in sizes:
        while True:
            base = rng.choice(letters, base_len)
            t = orc.triggers(base.tobytes(), w, p).astype(np.int64)
            spans = [(int(t[i]) - w + 1, int(t[i + 1]) + 1) for i in range(len(t) - 1)]
            spans = [sp for sp in spans if sp[1] - sp[0] >= 3 * w + 24]
            if spans:
                break
        s, e = spans[int(rng.integers(len(spans)))]
        variants = [(o, c) for o in family_offsets(e - s, w) for c in letters]
        rng.shuffle(variants)
        copies = [base]
        for o, c in variants:
            if len(copies) == H:
                break
            if base[s + o] == c:
                continue
            v = base.copy()
            v[s + o] = c
            if np.array_equal(orc.triggers(v.tobytes(), w, p), t):
                copies.append(v)
        assert len(copies) == H, f"family of {H}: only {len(copies)} variants keep the triggers"
        parts += copies
        parts.append(rng.choice(letters, filler))
        last_cut = base[:s + (e - s) // 2]
    if truncated_tail:
        parts.append(last_cut)
    return np.concatenate(parts).tobytes()


def tie_groups(dict_bytes, prefix):
    """Sizes and first ranks of the runs of .dict words sharing their first `prefix` bytes."""
    words = dict_bytes[:-1].split(b"\x01")[:-1]
    groups, start = [], 0
    for i in range(1, len(words) + 1):
        if i == len(words) or words[i][:prefix] != words[start][:prefix]:
            groups.append((start, i - start))
            start = i
    return groups


@pytest.mark.parametrize("H", [8, 20, 30])
@pytest.mark.parametrize("w,p", [(10, 100), (6, 50), (16, 500), (32, 1000)])
def test_pangenome_vs_oracle(pkg, scanners, H, w, p):
    """Dictionaries made mostly of 2..32-word families (H haplotypes of one base)."""
    text = pkg.synth.pangenome_text(200_000, H, 150 + H).numpy().tobytes()
    check_both(scanners, text, w, p, f"pangenome H={H} w{w} p{p}")


@pytest.mark.parametrize("alphabet", [DNA, PROTEIN], ids=["dna", "raw_bytes"])
def test_crafted_families(scanners, alphabet):
    """Families of exactly 2, 31, 32 and 33 words (and sizes between) whose members differ at both
    sides of chunk borders and at the last byte before the closing trigger; groups crossing a
    32-position window border; a last word that is a family member's prefix up to the 0x02 bytes
    closing the text; the first word (0x02 ...).  With 20 letters the first key holds 8 raw bytes
    instead of 21 DNA symbols."""
    sizes = [2, 31, 32, 33, 2, 3, 5, 9, 17, 31, 32, 33, 2, 7, 13, 32, 2, 31, 4, 33, 2, 32, 11, 6] * 2
    seed = 151 if alphabet == DNA else 152
    text = family_text(seed, sizes, alphabet)
    want = check_both(scanners, text, 10, 100, f"crafted {alphabet[:4]!r}")
    # the text has what the test is about: groups of those sizes, some crossing a window border
    groups = tie_groups(want.dict, 16)
    small = [(s, m) for s, m in groups if 2 <= m <= 32]
    assert {2, 31, 32, 33} <= {m for _, m in groups}
    assert any(s // 32 != (s + m - 1) // 32 for s, m in small)
    words = want.dict[:-1].split(b"\x01")[:-1]
    tail = [wd.rstrip(b"\x02") for wd in words if wd.endswith(b"\x02" * 10)]
    assert any(wd.startswith(tw) and wd != tw for tw in tail for wd in words), "no prefix of a family member"
    assert words[0][0] == 2


def big_family_text(seed, H, w=10, p=100, base_len=1200):
    """One family of H words: copies of a random base, each with two substitutions (at offsets past
    the 16 bytes the first key can hold) in the same word of the base."""
    rng = np.random.default_rng(seed)
    letters = np.frombuffer(DNA, np.uint8)
    while True:
        base = rng.choice(letters, base_len)
        t = orc.triggers(base.tobytes(), w, p).astype(np.int64)
        spans = [(int(t[i]) - w + 1, int(t[i + 1]) + 1) for i in range(len(t) - 1)]
        spans = [sp for sp in spans if sp[1] - sp[0] >= 80]
        if spans:
            break
    s, e = spans[0]
    copies, seen = [base], set()
    while len(copies) < H:
        o = rng.integers(16, e - s - w, 2)
        c = rng.choice(letters, 2)
        v = base.copy()
        v[s + o] = c
        key = v[s:e].tobytes()
        if key in seen or np.array_equal(v, base) or not np.array_equal(orc.triggers(v.tobytes(), w, p), t):
            continue
        seen.add(key)
        copies.append(v)
    return np.concatenate(copies + [rng.choice(letters, 5000)]).tobytes()


def test_family_larger_than_local_max(scanners):
    """A tie group of 3000 words goes through global radix-sort rounds until its parts fit a CTA
    (2048 words); the groups already finished on chip in a round stay as they are."""
    text = big_family_text(154, 3000)
    want = check_both(scanners, text, 10, 100, "family of 3000")
    assert max(m for _, m in tie_groups(want.dict, 16)) == 3000


def test_walks_equal_passes_64mb(pkg, scanners):
    """A/B at a size the oracle is too slow for: 16 haplotypes x 4 Mbp."""
    t = pkg.synth.pangenome_text(4_000_000, 16, 153).cuda()
    got = {arm: s.fetch(s.parse_device(t, 10, 100, sai=True)) for arm, s in scanners.items()}
    assert_same_files(got["walks"], got["passes"], "64 MB: LCP walks vs warp chunk passes")
