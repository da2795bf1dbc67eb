"""Model check of the persistent kernel's flagged exchange (q3_mega.cuh, ll_store; DESIGN.md section 4).

The o_proj / down rows travel as (value, epoch) words with NO barrier between writer and reader, pushed into every rank's
landing zone; the zones are reused one layer later.  This is a discrete-event model of exactly the dependency structure the
kernel has (per layer: poll down -> qkv -> grid barrier -> attention -> grid barrier -> o_proj rows out -> poll o -> gate/up
-> grid barrier -> down rows out), with the weakest delivery the hardware allows: every 8-byte store is delivered
individually at an arbitrary later time (only stores of one thread to the SAME word stay in order), barriers do not
flush them, and CTAs run in any interleaving.  Checked over many random schedules:
  I1  a poll only ever completes on words whose epoch AND value are the expected ones;
  I2  no store lands on a word while some CTA of that rank has not yet finished polling the word's previous contents
      (the reuse-safety argument written next to ll_store);
  I3  the schedule always runs to completion (no deadlock)."""
import random

import pytest


def _simulate(ranks, ctas, layers, seed, break_dependency=False):
    rnd = random.Random(seed)
    O, DOWN = 0, 1
    epoch = lambda l, kind: 1 + 2 * l + kind
    value = lambda l, kind, r, c: (l * 7 + kind * 3 + r * 101 + c * 13) & 0xFFFF
    # zone[kind][dest_rank][(writer_rank, writer_cta)] = (value, epoch)
    zone = [[{(r, c): (0, 0) for r in range(ranks) for c in range(ctas)} for _ in range(ranks)] for _ in range(2)]
    inflight = []            # (kind, dest, key, value, epoch); delivered in random order, FIFO per (kind, dest, key)
    polled = {}              # (rank, cta, kind) -> last epoch whose poll completed
    barrier_count = [dict() for _ in range(ranks)]   # rank -> barrier id -> arrivals

    def program(r, c):
        for l in range(layers):
            if l > 0:
                yield ("poll", DOWN, epoch(l - 1, DOWN), l - 1)
            yield ("barrier", (l, "qkv"))
            yield ("barrier", (l, "att"))
            yield ("store", O, l)
            if not break_dependency:
                yield ("poll", O, epoch(l, O), l)
            yield ("barrier", (l, "gu"))
            yield ("store", DOWN, l)
        yield ("poll", DOWN, epoch(layers - 1, DOWN), layers - 1)

    progs = {(r, c): program(r, c) for r in range(ranks) for c in range(ctas)}
    cur = {k: next(p) for k, p in progs.items()}
    steps = 0
    while cur or inflight:
        steps += 1
        assert steps < 200000, "I3: no progress"
        choices = []
        if inflight:
            choices.append(("deliver", None))
        for (r, c), act in cur.items():
            if act[0] == "store":
                choices.append(("run", (r, c)))
            elif act[0] == "poll":
                _, kind, ep, l = act
                if all(zone[kind][r][k][1] == ep for k in zone[kind][r]):
                    choices.append(("run", (r, c)))
            else:  # barrier: arrive once, then wait for the whole rank
                bid = act[1]
                arrived = barrier_count[r].setdefault(bid, set())
                if (r, c) not in arrived or len(arrived) == ctas:
                    choices.append(("run", (r, c)))
        assert choices, "I3: deadlock"
        what, who = rnd.choice(choices)
        if what == "deliver":
            # any in-flight store whose predecessors to the same word have been delivered
            firsts = {}
            for i, m in enumerate(inflight):
                firsts.setdefault(m[:3], i)
            i = rnd.choice(list(firsts.values()))
            kind, dest, key, val, ep = inflight.pop(i)
            old_ep = zone[kind][dest][key][1]
            if old_ep:  # I2: everybody on `dest` must be done with the previous contents of this word
                for c in range(ctas):
                    assert polled.get((dest, c, kind), 0) >= old_ep, f"I2: store of epoch {ep} lands on epoch {old_ep} still needed by CTA {c} of rank {dest}"
            zone[kind][dest][key] = (val, ep)
            continue
        r, c = who
        act = cur[who]
        if act[0] == "store":
            _, kind, l = act
            for dest in range(ranks):  # the same word into every rank's zone, each store on its own
                inflight.append((kind, dest, (r, c), value(l, kind, r, c), epoch(l, kind)))
        elif act[0] == "poll":
            _, kind, ep, l = act
            for (wr, wc), (val, e) in zone[kind][r].items():
                assert e == ep and val == value(l, kind, wr, wc), "I1"
            polled[(r, c, kind)] = ep
        else:
            arrived = barrier_count[r][act[1]]
            if (r, c) not in arrived:
                arrived.add((r, c))
                continue  # arrived; stays at the barrier until everybody has
        try:
            cur[who] = next(progs[who])
        except StopIteration:
            del cur[who]
    return steps


@pytest.mark.parametrize("ranks,ctas,layers", [(1, 5, 4), (2, 4, 4), (4, 3, 3)])
def test_flagged_exchange_is_safe_under_any_schedule_and_delivery_order(ranks, ctas, layers):
    for seed in range(150):
        _simulate(ranks, ctas, layers, seed)


def test_the_model_detects_a_missing_dependency():
    """Negative control: if the gate/up prologue did NOT wait for the o_proj words (so nothing orders a CTA's reads before the
    next layer's writes), the checker finds the reuse hazard (or the stale read) within a few schedules."""
    failures = 0
    for seed in range(60):
        try:
            _simulate(2, 4, 4, seed, break_dependency=True)
        except AssertionError:
            failures += 1
    assert failures > 0
