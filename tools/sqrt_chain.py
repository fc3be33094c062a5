#!/usr/bin/env python
"""Addition chain for the BLS12-381 square-root exponent (p+1)/4, emitted as C++ code.

fp_sqrt computes a^((p+1)/4) (p = 3 mod 4).  The exponent is public, so the power is a fixed sequence of
squarings and products.  The chain is a sliding-window decomposition e = sum d_j 2^(s_j) over a small set D of
odd digits: a^d for every d in D is built first (a short chain from a^2), then the windows run from the top
one down, each a run of squarings followed by one product with a^(d_j).  The number of windows for a given D
is minimal (dynamic programming over the bit positions); D itself comes from a seeded local search that
weighs the products of the windows and of the digit chain, the squarings of the digit chain, and one register
set (12 words) per digit that stays live through the windows.

Writes go-curdleproofs_b200/csrc/fp_sqrt_chain.cuh (straight-line code: every temporary a named Fp local,
squaring runs as loops of FpM::sqr, nothing indexed at run time) and prints the chain's squaring and product
counts.  --check compares the header with what the script would write."""
import argparse
import functools
import os
import random
import sys

P = 0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffaaab
E = (P + 1) // 4
NBITS = E.bit_length()
W = 9                # longest window
SQR = 234 / 300      # a dedicated squaring in products (DESIGN §5)
PER_DIGIT = 0.25     # register pressure of one more live digit, in products
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                   "go-curdleproofs_b200", "csrc", "fp_sqrt_chain.cuh")


def windows(D):
    """minimal list of (low bit, digit) covering E with digits in D, most significant first"""
    INF = 1 << 30
    f = [INF] * (NBITS + 1)
    back = [None] * (NBITS + 1)
    f[0] = 0
    for i in range(NBITS):
        if f[i] == INF:
            continue
        if not (E >> i) & 1:
            if f[i] < f[i + 1]:
                f[i + 1], back[i + 1] = f[i], (i, 0)
            continue
        for L in range(1, W + 1):
            if i + L > NBITS:
                break
            v = (E >> i) & ((1 << L) - 1)
            if (v >> (L - 1)) & 1 and v in D and f[i] + 1 < f[i + L]:
                f[i + L], back[i + L] = f[i] + 1, (i, v)
    out, j = [], NBITS
    while j:
        i, v = back[j]
        if v:
            out.append((i, v))
        j = i
    return out


def digit_chain(D):
    """steps (value, x, y) building every d in D from 1: value = x + y (a squaring when x == y)"""
    have, steps = {1}, []

    def add(v, x, y):
        have.add(v)
        steps.append((v, x, y))

    add(2, 1, 1)
    for d in sorted(D):
        if d in have:
            continue
        x = next((x for x in sorted(have, reverse=True) if d - x in have), None)
        if x is not None:
            add(d, x, d - x)
            continue
        pair = next(((x, y) for x in sorted(have, reverse=True) for y in sorted(have, reverse=True)
                     if 0 < d - x - y and d - x - y in have), None)
        if pair:
            x, y = pair
            add(x + y, x, y)
            add(d, x + y, d - x - y)
            continue
        x = max(c for c in have if c < d and c % 2)
        while x < d:
            add(x + 2, x, 2)
            x += 2
    return steps


@functools.lru_cache(maxsize=None)
def cost(D):
    steps = digit_chain(D)
    s = sum(1 for v, x, y in steps if x == y)
    return len(windows(D)) - 1 + len(steps) - s + SQR * s + PER_DIGIT * len(D)


def search(seed=1, restarts=4, iters=1500):
    rnd = random.Random(seed)
    cands = list(range(3, 1 << W, 2))
    best = None
    for _ in range(restarts):
        D = frozenset({1} | set(rnd.sample(range(3, 64, 2), 8)))
        for _ in range(iters):
            S = set(D)
            r = rnd.random()
            if r < 0.8 and len(S) > 1:
                S.discard(rnd.choice(sorted(S - {1})))
            if r >= 0.4:
                S.add(rnd.choice(cands))
            S = frozenset(S)
            if cost(S) <= cost(D):
                D = S
        if best is None or cost(D) < cost(best):
            best = D
    return best


def emit(D):
    steps = digit_chain(D)
    wins = windows(D)
    used = {v for _, v in wins}
    # drop digit-chain steps nothing needs (digits the windows never use, and what only they needed)
    need = set(used)
    for v, x, y in reversed(steps):
        if v in need:
            need |= {x, y}
    steps = [s for s in steps if s[0] in need]
    name = lambda v: "a" if v == 1 else f"x{v}"  # noqa: E731
    nsqr = sum(1 for v, x, y in steps if x == y)
    nmul = len(steps) - nsqr
    body = [f"  Fp {', '.join(name(v) for v, _, _ in steps)};"]
    for v, x, y in steps:
        body.append(f"  FpM::sqr({name(v)}, {name(x)});" if x == y else f"  FpM::mul({name(v)}, {name(x)}, {name(y)});")
    s0, d0 = wins[0]
    body.append(f"  r = {name(d0)};")
    prev = s0
    for s, d in wins[1:]:
        body.append(f"  fp_sqr_n(r, {prev - s});")
        body.append(f"  FpM::mul(r, r, {name(d)});")
        nsqr += prev - s
        nmul += 1
        prev = s
    if prev:
        body.append(f"  fp_sqr_n(r, {prev});")
        nsqr += prev
    head = [
        "// Generated by tools/sqrt_chain.py; do not edit.",
        f"// r = a^((p+1)/4): {nsqr} squarings and {nmul} products; digits (a^d, d odd) {sorted(used)}.",
        "// Included by fields.cuh inside namespace cdl, after Fp and fp_sqr_n.",
        "#pragma once",
        "",
        "CDL_FN void fp_pow_sqrt_exp(Fp& r, const Fp& a) {",
    ]
    return "\n".join(head + body + ["}", ""]), nsqr, nmul


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--check", action="store_true", help="exit 1 if the header differs from a fresh emission")
    ap.add_argument("--seed", type=int, default=1)
    args = ap.parse_args()
    D = search(args.seed)
    text, nsqr, nmul = emit(D)
    print(f"(p+1)/4: {NBITS} bits, {bin(E).count('1')} set; chain: {nsqr} squarings, {nmul} products "
          f"(the 4-bit fixed window it replaces: 384 squarings, 110 products with its table)")
    if args.check:
        with open(OUT) as f:
            sys.exit(0 if f.read() == text else 1)
    with open(OUT, "w") as f:
        f.write(text)
    print("wrote", OUT)


if __name__ == "__main__":
    main()
