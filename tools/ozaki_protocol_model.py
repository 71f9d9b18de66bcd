#!/usr/bin/env python
"""Explicit-state model of the barrier protocol of `ozaki_update_kernel` (csrc/ozaki.cu): one producer thread, two MMA-issuing
threads on alternate stages, the epilogue, and the asynchronous agents behind them (TMA copies completing on `full`, tcgen05.commit
arriving on `empty` / `acc_full` when an issuer's MMAs have executed).  Every interleaving of a small instance is explored; checked:

  * no deadlock: every thread runs to completion;
  * an issuer only ever consumes a stage that holds the K quarter it is about to multiply (no parity wait passing a phase early);
  * the producer never overwrites a stage whose MMAs have not executed, nor one with a copy still in flight;
  * in every pass the quarter-0 MMAs (which initialise the accumulators) are issued before any other quarter's;
  * the epilogue of a pass starts only after ALL MMAs of that pass (both issuers) have executed, and the MMAs of pass B only after
    the epilogue of pass A has drained the accumulators.

mbarrier semantics as in PTX: a barrier has a phase bit and a pending count; the last expected arrival flips the phase;
`try_wait.parity p` succeeds once the phase with parity p has completed, i.e. as soon as the current phase bit differs from p.
With an ODD number of stages the two-issuer variant fails exactly as the GPU did (the odd issuer's second quarter lives in the even
issuer's first stage, and its parity wait passes before that stage has ever been filled); the kernel therefore uses two issuers only
with an even stage count (`dual`) -- `explore(..., force_dual=True)` reproduces the failure.

Digit-plane filter: each pass walks its own MEMBER k-tiles (4 K quarters each; quarter kq is quarter kq % 4 of the kq // 4-th
member), so `members_a` / `members_b` may be any increasing lists, with gaps, a single member, or -- pass A only -- none.  A pass
without members issues nothing: both issuers arrive on acc_full directly (the odd one does not wait for init_done, which nobody would
arrive on), and the epilogue skips its TMEM read (`skip`); converting accumulators no MMA of the pass has written is a violation.
`empty_pass_fix=False` models the issuers without that rule (a plain init_done wait and commit), which deadlocks.  Test
infrastructure, CPU only."""
from collections import deque


class Violation(Exception):
    pass


def build_threads(members, nst_a, nst_b, force_dual=False, empty_pass_fix=True):
    """Programs as lists of (op, args): wait(bar, parity) | arrive(bar) | load(stage, pass, tag) | consume(stage, pass, kq, tag, who) |
    commit(bar, who) | epi(pass) | skip(pass).  tag = (member k-tile, quarter within it)."""
    P, E = [], []
    issuers = [[], []]
    for pas, nst in ((0, nst_a), (1, nst_b)):
        mem = members[pas]
        nq = 4 * len(mem)
        tag = lambda kq, mem=mem: (mem[kq // 4], kq % 4)
        full = lambda s, p=pas: ("full", p, s)
        empty = lambda s, p=pas: ("empty", p, s)
        dual = force_dual or nst % 2 == 0
        if pas:
            P.append(("wait", ("acc_full",), 0))
        for kq in range(nq):
            s = kq % nst
            P.append(("wait", empty(s), ((kq // nst) & 1) ^ 1))
            P.append(("load", s, pas, tag(kq)))
        for who in (0, 1):
            T = issuers[who]
            if who == 1 and not dual:
                if pas:
                    T.append(("wait", ("acc_full",), 0))
                T.append(("arrive", ("acc_full",)))
                continue
            if pas:
                T.append(("wait", ("acc_empty",), 0))
            if nq == 0 and empty_pass_fix:
                T.append(("arrive", ("acc_full",)))
                continue
            if who == 1:
                T.append(("wait", ("init_done", pas), 0))
            for kq in range(who, nq, 2 if dual else 1):
                s = kq % nst
                T.append(("wait", full(s), (kq // nst) & 1))
                T.append(("consume", s, pas, kq, tag(kq), who))
                T.append(("commit", empty(s), who, s, pas))
                if kq == 0:
                    T.append(("arrive", ("init_done", pas)))
            T.append(("commit", ("acc_full",), who, None, pas))
        E.append(("wait", ("acc_full",), pas))
        E.append(("epi", pas) if nq or not empty_pass_fix else ("skip", pas))
        if pas == 0:
            E.append(("arrive", ("acc_empty",)))
    return [P, issuers[0], issuers[1], E]


def explore(nq=8, nst_a=6, nst_b=4, force_dual=False, max_states=2_000_000, members_a=None, members_b=None, empty_pass_fix=True):
    """nq: K quarters per pass when the member lists are not given (every k-tile 0 .. nq/4 - 1 is a member)."""
    dense = list(range(nq // 4))
    members = (dense if members_a is None else list(members_a), dense if members_b is None else list(members_b))
    nqs = (4 * len(members[0]), 4 * len(members[1]))
    threads = build_threads(members, nst_a, nst_b, force_dual, empty_pass_fix)
    counts = {("acc_full",): 2, ("acc_empty",): 1}
    bars0 = {}
    for T in threads:
        for ins in T:
            if ins[0] in ("wait", "arrive"):
                bars0.setdefault(ins[1], None)
            if ins[0] == "commit":
                bars0.setdefault(ins[1], None)
    names = sorted(bars0, key=repr)
    bidx = {n: i for i, n in enumerate(names)}
    cnt = [counts.get(n, 1) for n in names]
    nstages = max(nst_a, nst_b)
    # state: pcs, barrier (phase, pending) tuples, stage content, stage in-flight load, stage busy (MMAs issued, not executed),
    # per-issuer FIFO of outstanding commits, pass progress flags
    init = (
        (0, 0, 0, 0),
        tuple((0, c) for c in cnt),
        tuple([None] * nstages),       # content (pass, kq)
        tuple([None] * nstages),       # in-flight load (pass, kq, barrier index)
        tuple([0] * nstages),          # busy: number of issued, not yet executed consumers
        ((), ()),                      # outstanding commits per issuer: tuples (barrier index, stage or -1)
        (0, 0),                        # MMAs issued per pass (quarters)
        (0, 0),                        # MMAs executed per pass (quarters)
        0,                             # epilogues done
        ((), ()),                      # per issuer: quarters issued and not yet covered by a fired commit (pass tags)
    )

    def arrive(bars, i):
        ph, pend = bars[i]
        pend -= 1
        if pend < 0:
            raise Violation(f"arrival overflow on {names[i]}")
        if pend == 0:
            ph, pend = ph ^ 1, cnt[i]
        b = list(bars)
        b[i] = (ph, pend)
        return tuple(b)

    seen = {init}
    todo = deque([init])
    finals = 0
    while todo:
        st = todo.pop()
        pcs, bars, content, flight, busy, fifo, issued, executed, epis, uncommitted = st
        succ = []
        # thread steps
        for ti, T in enumerate(threads):
            pc = pcs[ti]
            if pc >= len(T):
                continue
            ins = T[pc]
            npcs = pcs[:ti] + (pc + 1,) + pcs[ti + 1:]
            if ins[0] == "wait":
                ph, _ = bars[bidx[ins[1]]]
                if ph != ins[2]:
                    succ.append((npcs, bars, content, flight, busy, fifo, issued, executed, epis, uncommitted))
            elif ins[0] == "arrive":
                succ.append((npcs, arrive(bars, bidx[ins[1]]), content, flight, busy, fifo, issued, executed, epis, uncommitted))
            elif ins[0] == "load":
                _, s, pas, kq = ins  # kq: the tag (member k-tile, quarter)
                if busy[s]:
                    raise Violation(f"producer overwrites stage {s} (pass {pas}, quarter {kq}) while its MMAs have not executed")
                if flight[s] is not None:
                    raise Violation(f"two copies in flight into stage {s}")
                fl = list(flight)
                fl[s] = (pas, kq, bidx[("full", pas, s)])
                succ.append((npcs, bars, content, tuple(fl), busy, fifo, issued, executed, epis, uncommitted))
            elif ins[0] == "consume":
                _, s, pas, kq, tg, who = ins
                if content[s] != (pas, tg) or flight[s] is not None:
                    raise Violation(f"issuer {who} consumes stage {s} for pass {pas} quarter {kq} {tg} but it holds {content[s]} (in flight: {flight[s]})")
                if kq != 0 and issued[pas] == 0:
                    raise Violation(f"pass {pas}: quarter {kq} issued before quarter 0 (accumulators not initialised)")
                if pas == 1 and epis < 1:
                    raise Violation("pass B MMA issued before the epilogue of pass A drained the accumulators")
                bz = list(busy)
                bz[s] += 1
                iss = list(issued)
                iss[pas] += 1
                un = list(uncommitted)
                un[who] = un[who] + (pas,)
                succ.append((npcs, bars, content, flight, tuple(bz), fifo, tuple(iss), executed, epis, tuple(un)))
            elif ins[0] == "commit":
                _, bar, who, s, pas = ins
                ff = list(fifo)
                # the commit covers every MMA this issuer has issued so far
                ff[who] = ff[who] + ((bidx[bar], -1 if s is None else s, len(uncommitted[who])),)
                un = list(uncommitted)
                succ.append((npcs, bars, content, flight, busy, tuple(ff), issued, executed, epis, tuple(un)))
            elif ins[0] == "epi":
                pas = ins[1]
                if executed[pas] != nqs[pas]:
                    raise Violation(f"epilogue of pass {pas} starts with {executed[pas]} of {nqs[pas]} quarters executed")
                if issued[pas] == 0:
                    raise Violation(f"epilogue of pass {pas} reads accumulators that no MMA has initialised")
                succ.append((npcs, bars, content, flight, busy, fifo, issued, executed, epis + 1, uncommitted))
            elif ins[0] == "skip":
                succ.append((npcs, bars, content, flight, busy, fifo, issued, executed, epis + 1, uncommitted))
        # asynchronous agents: a copy lands; the oldest outstanding commit of an issuer fires (its MMAs have executed)
        for s in range(nstages):
            if flight[s] is not None:
                pas, kq, bi = flight[s]
                ct = list(content)
                ct[s] = (pas, kq)
                fl = list(flight)
                fl[s] = None
                succ.append((pcs, arrive(bars, bi), tuple(ct), tuple(fl), busy, fifo, issued, executed, epis, uncommitted))
        for who in (0, 1):
            if fifo[who]:
                bi, s, ncov = fifo[who][0]
                ff = list(fifo)
                rest = tuple((b2, s2, n2 - ncov) for (b2, s2, n2) in fifo[who][1:])
                ff[who] = rest
                un = list(uncommitted)
                done = un[who][:ncov]
                un[who] = un[who][ncov:]
                ex = list(executed)
                for pas in done:
                    ex[pas] += 1
                bz = list(busy)
                if s >= 0:
                    bz[s] -= 1
                succ.append((pcs, arrive(bars, bi), content, flight, tuple(bz), tuple(ff), issued, tuple(ex), epis, tuple(un)))
        if not succ:
            if all(pcs[i] >= len(threads[i]) for i in range(4)):
                finals += 1
                continue
            raise Violation(f"deadlock at pcs {pcs}: " + ", ".join(str(threads[i][pcs[i]]) if pcs[i] < len(threads[i]) else "done" for i in range(4)))
        for nx in succ:
            if nx not in seen:
                seen.add(nx)
                if len(seen) > max_states:
                    raise RuntimeError("state space larger than expected")
                todo.append(nx)
    return {"states": len(seen), "final_states": finals}


if __name__ == "__main__":
    print("dual, 6 / 4 stages:", explore(8, 6, 4))
    print("single issuer in pass B, 6 / 3 stages:", explore(8, 6, 3))
    try:
        explore(8, 6, 3, force_dual=True)
    except Violation as v:
        print("two issuers on 3 stages:", v)
    print("empty pass A, members 1, 4 in pass B:", explore(members_a=[], members_b=[1, 4]))
    print("single member in both passes:", explore(members_a=[3], members_b=[3]))
    try:
        explore(members_a=[], members_b=[0, 2], empty_pass_fix=False)
    except Violation as v:
        print("empty pass A without its rule:", v)
