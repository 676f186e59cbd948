"""Model check of the cut-face exchange protocol (DESIGN.md section 5) - host logic only, no GPU.

Every GPU owns a staging buffer with S slots; exchange number n lives in slot n % S and every word carries n as its tag.
Three kinds of launches touch it (all ranks issue the same sequence, each at its own pace):

  H  k_halo: copies, SENDS exchange E+1 into the peers' slot and WAITS until its own slot holds E+1 (round 1's path, used
     after something other than a sweep changed the field);
  W  a sweep whose producer warps SEND exchange E+1 while it runs and whose last CTA advances E (it never waits);
  U  the unpack launch before the next sweep: WAITS until its own slot holds E, unpacks it.

The shipped order is W U W U ...: the values of exchange E are out of the slot before the sweep that sends E+1 starts.  The
variant measured and rejected in round 2 consumed exchange E INSIDE the sweep that sends E+1 (no launch between two sweeps).
The model explores every interleaving of two ranks and checks (a) no rank overwrites a slot whose exchange its peer still
has to read, (b) nobody waits for ever.  It pins the claims of the design notes: with FOUR slots the shipped order is safe and
live for every launch sequence the host logic can issue; two slots would do for a plain W U W U ... but not once a sending
sweep is followed by a prolongation and a fresh halo exchange (nobody unpacks that send, so a rank gets two exchanges ahead);
the in-sweep variant also needs four."""
import itertools
from collections import deque

import pytest


def expand(program, in_sweep):
    """program: string over H (halo exchange), W (sending sweep), U (unpack), X (field changed outside a sweep: no launch),
    the strip-state transitions halo_exchanged, sweep_done, unpacked and field_changed of pamg_api.cu.  Returns the list of atomic steps of one rank: ('send', n) / ('wait', n) with the exchange numbers resolved."""
    steps, e = [], 0
    for op in program:
        if op == "H":
            steps += [("send", e + 1), ("wait", e + 1)]
            e += 1
        elif op == "W":
            if in_sweep:
                # the sweep reads exchange e (anywhere during its run) and sends e + 1: both orders are possible
                steps += [("par", ("wait", e), ("send", e + 1))]
            else:
                steps += [("send", e + 1)]
            e += 1
        elif op == "U":
            steps += [("wait", e)]
        elif op == "X":
            pass
        else:
            raise ValueError(op)
    return steps


def flatten_choices(steps):
    """('par', a, b) -> both orders; yields every fully ordered step list"""
    options = [[(s,)] if s[0] != "par" else [(s[1], s[2]), (s[2], s[1])] for s in steps]
    for pick in itertools.product(*options):
        yield [x for grp in pick for x in grp]


def check(program, slots, in_sweep=False):
    """Returns None when every interleaving of two ranks is safe and terminates, else a short description of the failure."""
    for sa in flatten_choices(expand(program, in_sweep)):
        for sb in flatten_choices(expand(program, in_sweep)):
            prog = (sa, sb)
            waits = [sorted({n for k, n in p if k == "wait"}) for p in prog]      # what each rank will read, ever
            start = (0, 0, (0,) * slots, (0,) * slots, 0, 0)   # pcs, slot tags at rank 0 / rank 1, last exchange read per rank
            seen, todo = {start}, deque([start])
            while todo:
                pc0, pc1, s0, s1, r0, r1 = todo.popleft()
                pcs, stage, read = [pc0, pc1], [list(s0), list(s1)], [r0, r1]
                moved = False
                for me in (0, 1):
                    if pcs[me] >= len(prog[me]):
                        continue
                    kind, n = prog[me][pcs[me]]
                    peer = 1 - me
                    npcs, nstage, nread = list(pcs), [list(stage[0]), list(stage[1])], list(read)
                    if kind == "send":
                        old = stage[peer][n % slots]
                        if old > read[peer] and old in waits[peer]:
                            return f"{program} S={slots}: rank {me} writes exchange {n} over unread exchange {old}"
                        nstage[peer][n % slots] = n
                    else:
                        if stage[me][n % slots] != n:
                            if stage[me][n % slots] > n:
                                return f"{program} S={slots}: rank {me} waits for {n}, slot already holds {stage[me][n % slots]}"
                            continue                      # not there yet: this rank cannot move
                        nread[me] = max(nread[me], n)
                    npcs[me] += 1
                    moved = True
                    st = (npcs[0], npcs[1], tuple(nstage[0]), tuple(nstage[1]), nread[0], nread[1])
                    if st not in seen:
                        seen.add(st); todo.append(st)
                if not moved and not (pcs[0] >= len(prog[0]) and pcs[1] >= len(prog[1])):
                    return f"{program} S={slots}: deadlock at steps {pcs}"
    return None


def shipped_programs(max_len):
    """what the host logic can issue on one level: a halo exchange first; then sweeps, each followed by an unpack before
    anything reads the strips again - or by a field change (X) and a new halo exchange"""
    out = []
    def grow(p, pending):
        if len(p) >= max_len:
            out.append(p); return
        # "XHH": told changed (or update_overlaps as written was called): the told values of the cut faces are exchanged by a
        # k_halo launch of their own, which leaves nothing to unpack, and a second one exchanges the tnew values
        # (exchange_told + ensure_strips, theta != 1; launch_halo with HALO_ALL)
        if pending:                       # a sweep has sent: unpack, or the field changes and k_halo exchanges afresh
            grow(p + "U", False)
            grow(p + "XH", False)
            grow(p + "XHH", False)
        else:
            grow(p + "W", True)
            grow(p + "XH", False)
            grow(p + "XHH", False)
    grow("H", False)
    return sorted(set(out))


def test_shipped_order_is_safe_and_live_with_four_slots():
    for prog in shipped_programs(9):
        assert check(prog, 4) is None


def test_sends_nobody_unpacks_need_more_than_two_slots():
    # post-smoothing on a coarse level ends with a sending sweep that nobody unpacks; the next visit starts with a halo exchange.
    # A rank that skips that wait gets two exchanges ahead of a peer that still has to unpack: four slots absorb it, two do not
    for prog in ("HWUWUWXHWUW", "HWXHWXHWXHWXHWU", "HWUWUWUWXHWUWUWUWXH"):
        assert check(prog, 4) is None
    assert check("HWUWUWUWU", 2) is None                       # plain W U W U ...: two slots would do
    bad = check("HWUWUWXHWUW", 2)
    assert bad is not None and "over unread exchange" in bad


def test_unpacking_inside_the_sweep_needs_four_slots():
    for prog in ("H" + "W" * 8, "HWWWXHWWWW", "HWXHWWXHWW"):
        assert check(prog, 4, in_sweep=True) is None
    bad = check("H" + "W" * 8, 2, in_sweep=True)
    assert bad is not None and "over unread exchange" in bad
