"""Model of the grid-wide phase synchronisation of k_decode_persistent (csrc/decode_persistent.cuh): monotone epoch
counters with the kernel's exact target expressions, several CTAs, several layers, several launches (decode launches with
lm_head and prefill launches without), random interleavings.  Checks: no deadlock; a phase never starts before every
producer of its input finished (all QKV rows before attention, all heads before Wo, all rows of x before a norm, the whole
hidden activation before W2); the lm_head counter survives prefill launches in between.
usage: python tools/sim/decode_persistent_epochs.py [runs]"""
import random
import sys

QKV, ATT, WO, GU, W2, LM, TICK, LMTICK = 0, 1, 2, 3, 4, 5, 8, 9


def launch(sync, nC, nL, n_heads, with_logits, rng, done):
    tick, lmtick = sync[TICK], sync[LMTICK]
    finished = {"ctas": 0}

    def cta(c):
        def arrive(k):
            sync[k] += 1

        def wait(k, target):
            while sync[k] - target < 0:
                yield

        for l in range(nL):
            e = tick * nL + l + 1
            done[("qkv", tick, l)] = done.get(("qkv", tick, l), 0) + 1
            arrive(QKV)
            yield
            if c < n_heads:
                yield from wait(QKV, e * nC)
                assert done[("qkv", tick, l)] == nC, "attention before all QKV rows"
                done[("att", tick, l)] = done.get(("att", tick, l), 0) + 1
                arrive(ATT)
                yield
            yield from wait(ATT, e * n_heads)
            assert done[("att", tick, l)] == n_heads, "Wo before all heads"
            done[("wo", tick, l)] = done.get(("wo", tick, l), 0) + 1
            arrive(WO)
            yield
            yield from wait(WO, e * nC)
            assert done[("wo", tick, l)] == nC, "norm2 before x is complete"
            done[("gu", tick, l)] = done.get(("gu", tick, l), 0) + 1
            arrive(GU)
            yield
            yield from wait(GU, e * nC)
            assert done[("gu", tick, l)] == nC, "W2 before the hidden activation is complete"
            done[("w2", tick, l)] = done.get(("w2", tick, l), 0) + 1
            arrive(W2)
            yield
            yield from wait(W2, e * nC)
            assert done[("w2", tick, l)] == nC, "next layer before x is complete"
        if with_logits:
            done[("lm", tick)] = done.get(("lm", tick), 0) + 1
            arrive(LM)
            yield
            if c != 0:
                finished["ctas"] += 1
                return
            yield from wait(LM, (lmtick + 1) * nC)
            assert done[("lm", tick)] == nC, "argmax merge before all partials"
        elif c != 0:
            finished["ctas"] += 1
            return
        sync[TICK] = tick + 1
        if with_logits:
            sync[LMTICK] = lmtick + 1
        finished["ctas"] += 1

    procs = {c: cta(c) for c in range(nC)}
    stalled = 0
    while procs:
        c = rng.choice(list(procs))
        snap = tuple(sync)
        try:
            next(procs[c])
        except StopIteration:
            del procs[c]
            stalled = 0
            continue
        stalled = 0 if tuple(sync) != snap else stalled + 1
        assert stalled < 50000, f"deadlock with CTAs {sorted(procs)} (tick {tick})"
    assert finished["ctas"] == nC


def main():
    runs = int(sys.argv[1]) if len(sys.argv) > 1 else 100
    rng = random.Random(3)
    for _ in range(runs):
        nC, nL = rng.choice([3, 5, 8]), rng.choice([1, 2, 4])
        n_heads = rng.randrange(1, nC + 1)
        sync, done = [0] * 16, {}
        for _launch in range(rng.choice([1, 3, 6])):
            launch(sync, nC, nL, n_heads, rng.random() < 0.6, rng, done)
    print(f"{runs} runs ok: epochs consistent across decode and prefill launches, no deadlock, no early phase start")
    return 0


if __name__ == "__main__":
    sys.exit(main())
