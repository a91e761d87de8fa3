"""Linear-time check of a suffix array and BWT against their text, in torch on the device of the inputs.

TEST INFRASTRUCTURE ONLY: used by tests/ and tools/ as the checker of outputs too large for the oracle's
suffix sort (a 4 GB text and more); nothing under big-bwt_b200/ may import this.  The suffix array has
n + 1 rows over T$ ($ = the end of the text, smaller than every char); row 0 is the $ suffix, the row .sa
leaves out.  Four checks, together a complete check of a suffix array:
  * the suffix array is a permutation of [0, n];
  * bwt[i] == T[sa[i] - 1] at every row with sa[i] > 0;
  * the EOF char 0 sits at the row of the suffix at position 0;
  * adjacent rows: T[sa[i]] < T[sa[i+1]], or they are equal and ISA[sa[i]+1] < ISA[sa[i+1]+1]
    (Burkhardt-Kaerkkaeinen), the end of the text smaller than every char.
This checks the arrays; it is not a second suffix sort.  Every pass works on `chunk` rows at a time, so
that the temporaries stay small next to the int64 suffix and inverse suffix arrays.
"""
from __future__ import annotations

import torch

CHUNK = 1 << 28
SABYTES = 5


def decode5(b: torch.Tensor) -> torch.Tensor:
    """uint8 tensor of k little-endian 5-byte values (k * 5 bytes, any shape) -> int64 tensor of k values"""
    b = b.reshape(-1, SABYTES).to(torch.int64)
    return b[:, 0] | (b[:, 1] << 8) | (b[:, 2] << 16) | (b[:, 3] << 24) | (b[:, 4] << 32)


def encode5(v: torch.Tensor) -> torch.Tensor:
    """int64 tensor of values below 2^40 -> uint8 tensor of their little-endian 5-byte forms (k * 5 bytes)"""
    return torch.stack([(v >> (8 * j)) & 255 for j in range(SABYTES)], dim=1).to(torch.uint8).reshape(-1)


def load_sa(path, n, device="cuda", chunk=CHUNK):
    """.sa (n values of 5 bytes, rows 1..n) -> int64 suffix array of rows 0..n on `device`"""
    sa = torch.empty(n + 1, dtype=torch.int64, device=device)
    sa[0] = n
    with open(path, "rb") as f:
        i = 1
        while i <= n:
            k = min(chunk, n + 1 - i)
            b = f.read(SABYTES * k)
            if len(b) != SABYTES * k:
                raise ValueError(f"{path}: {(i - 1 + len(b) // SABYTES)} values, {n} expected")
            sa[i:i + k] = decode5(torch.frombuffer(bytearray(b), dtype=torch.uint8).to(device))
            i += k
    return sa


def linear_checks(T, sa, bwt, chunk=CHUNK):
    """T: text (uint8, n), sa: int64 (n + 1 rows), bwt: uint8 (n + 1), all on one device.  Returns the
    list of failed checks (empty: the suffix array and the BWT are those of T)."""
    dev = T.device
    n = T.numel()
    if bwt.numel() != n + 1 or sa.numel() != n + 1:
        return [f"sizes: bwt {bwt.numel()}, sa {sa.numel()}, text {n}"]
    if int(sa.min()) < 0 or int(sa.max()) > n:
        return ["suffix array values outside [0, n]"]
    isa = torch.full((n + 2,), -1, dtype=torch.int64, device=dev)
    for a in range(0, n + 1, chunk):
        b = min(n + 1, a + chunk)
        isa[sa[a:b]] = torch.arange(a, b, dtype=torch.int64, device=dev)
    if bool((isa[:n + 1] < 0).any()):                             # n + 1 values in [0, n]: a repeat leaves a hole
        return ["the suffix array is not a permutation of [0, n]"]
    fails = []
    if int(bwt[int(isa[0])]) != 0:
        fails.append(f"the EOF char is not at row {int(isa[0])}, the row of the suffix at position 0")
    Tx = torch.empty(n + 1, dtype=torch.int16, device=dev)
    Tx[:n] = T.to(torch.int16)
    Tx[n] = -1                                                    # the end of the text: smaller than every char
    bad_bwt = bad_order = 0
    for a in range(0, n + 1, chunk):
        b = min(n + 1, a + chunk)
        s = sa[a:b]
        prev = torch.where(s > 0, Tx[(s - 1).clamp(min=0)], torch.zeros_like(s, dtype=torch.int16))
        bad_bwt += int((prev != bwt[a:b].to(torch.int16)).sum())
        e = min(b, n)                                             # rows a..e-1 against rows a+1..e
        if e > a:
            s0, s1 = sa[a:e], sa[a + 1:e + 1]
            c0, c1 = Tx[s0], Tx[s1]
            r0 = isa[(s0 + 1).clamp(max=n + 1)]
            r1 = isa[(s1 + 1).clamp(max=n + 1)]
            ok = (c0 < c1) | ((c0 == c1) & (r0 < r1))
            bad_order += int((~ok).sum())
    if bad_bwt:
        fails.append(f"bwt[i] != T[sa[i]-1] at {bad_bwt} rows")
    if bad_order:
        fails.append(f"adjacent rows out of order at {bad_order} places")
    return fails
