"""Lane-accurate Python emulation of the segmented scan of csrc/seqsum2.cuh (seq2_warp_segscan, the scan over
the warp tails and the carry composition), checked against a sequential composition from each run's first thread.
Pair composition is not commutative, so a wrong operand order or a wrong segment flag shows up immediately.
usage: python tools/seqsum2/emulate_scan.py [cases]"""
import random
import sys

SAT = 1 << 26


def compose(L, R):  # apply L, then R  (seq_compose)
    a0 = L[0] + (R[1] if (L[0] & 1) else R[0])
    a1 = L[1] + (R[1] if ((1 + L[1]) & 1) else R[0])
    return (min(a0, SAT), min(a1, SAT))


def warp_segscan(p, f):
    """p[32], f[32] -> in place, exactly the loop of seq2_warp_segscan (all lanes read the pre-step values)."""
    d = 1
    while d < 32:
        up = [p[l - d] if l >= d else p[l] for l in range(32)]
        fu = [f[l - d] if l >= d else f[l] for l in range(32)]
        for l in range(32):
            if l >= d and not f[l]:
                p[l] = compose(up[l], p[l])
                f[l] = fu[l]
        d <<= 1


def block_scan(cls, pr, T):
    NW = T // 32
    LIT = None
    out = list(pr)
    flags = [0] * T
    wtail, wtail_f = [None] * 32, [1] * 32
    for w in range(NW):
        p = [out[w * 32 + l] for l in range(32)]
        f = []
        for l in range(32):
            t = w * 32 + l
            prev = cls[t - 1] if t > 0 else LIT
            f.append(0 if (cls[t] is not LIT and prev == cls[t]) else 1)
        warp_segscan(p, f)
        for l in range(32):
            out[w * 32 + l] = p[l]
            flags[w * 32 + l] = f[l]
        wtail[w], wtail_f[w] = p[31], f[31]
    t = [wtail[l] if l < NW else (0, 0) for l in range(32)]
    tf = [wtail_f[l] if l < NW else 1 for l in range(32)]
    warp_segscan(t, tf)
    for w in range(1, NW):
        for l in range(32):
            i = w * 32 + l
            if not flags[i]:
                out[i] = compose(t[w - 1], out[i])
    return out


def reference(cls, pr, T):
    out = [None] * T
    for i in range(T):
        if cls[i] is None or i == 0 or cls[i - 1] != cls[i]:
            out[i] = pr[i]
        else:
            out[i] = compose(out[i - 1], pr[i])
    return out


def main():
    cases = int(sys.argv[1]) if len(sys.argv) > 1 else 300
    rng = random.Random(1)
    for c in range(cases):
        T = rng.choice([256, 512, 1024])
        cls, e = [], 0
        run_p = rng.choice([0.02, 0.1, 0.5])
        for i in range(T):
            if rng.random() < run_p:
                e += rng.choice([0, 1])
                cls.append(None if rng.random() < 0.5 else e)
            else:
                cls.append(e if (cls and cls[-1] is not None) or rng.random() < 0.7 else None)
        pr = [(0, 0) if cls[i] is None else (rng.randrange(0, 50), rng.randrange(0, 50)) for i in range(T)]
        got, want = block_scan(cls, pr, T), reference(cls, pr, T)
        for i in range(T):
            if cls[i] is not None and got[i] != want[i]:
                print("MISMATCH case", c, "T", T, "thread", i, got[i], want[i])
                return 1
    print(f"{cases} cases ok (T in 256/512/1024, runs crossing warp boundaries, literal threads interleaved)")
    return 0


if __name__ == "__main__":
    sys.exit(main())
