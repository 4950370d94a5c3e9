#!/usr/bin/env python
"""
Discrete-event replay of the persistent factorisation kernel's task queue (no GPU): 148 workers draw tickets in queue
order, each waits for the counters its task names, runs for the task's duration and signals.  Task durations are the
measured ones (DESIGN.md 3.3, profiles/r01s3_ncu_summary.md): DIAG 35 us + 10 us per fused update panel, PANEL 25 us (8 us per row strip of the tile below the diagonal block),
narrow update 31 us, wide update 17 W + 12 us, TRANSPOSE 5 us.  Prints the makespan, the critical chain
(sum over panels of DIAG + PANEL) and the work bound (sum of durations / workers) of the library's own queue.

    python tools/factor_sim.py [nb ...]        e.g.  python tools/factor_sim.py 32 64
"""
import ctypes
import heapq
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

DIAG, PANEL, UPD, TRANSPOSE, XT, Y = range(6)


def duration_us(t):
    op, s = int(t[0]), int(t[4])
    if op == DIAG:
        return 35.0 + 10.0 * s
    if op == PANEL:
        return 8.0 if s > 0 else 25.0  # s > 0: one of the four row strips of the tile below the diagonal block
    if op == UPD:
        return 31.0 if s == 1 else 17.0 * s + 12.0
    if op == TRANSPOSE:
        return 5.0
    return 20.0 * max(1, s)  # inverse tasks (only below N = 512 since the int8 engine took them over)


def task_list(nb, nsm):
    from pygpso_b200 import backend

    lib = backend.load_library()
    nt, nc = ctypes.c_int(0), ctypes.c_int(0)
    assert lib.gpso_debug_factor_tasks(nb, nsm, None, 0, ctypes.byref(nt), ctypes.byref(nc)) == 0
    buf = np.zeros(nt.value * 16, dtype=np.int32)
    assert lib.gpso_debug_factor_tasks(nb, nsm, buf.ctypes.data_as(ctypes.POINTER(ctypes.c_int)), buf.size, ctypes.byref(nt),
                                       ctypes.byref(nc)) == 0
    return buf.reshape(-1, 16), nc.value


def simulate(nb, nsm=148, with_inverse=False):
    tasks, ncounters = task_list(nb, nsm)
    if not with_inverse:
        tasks = tasks[tasks[:, 0] <= TRANSPOSE]
    # time at which each counter reaches each value: counters only grow, so keep the list of increment times
    reach = [[] for _ in range(ncounters)]   # reach[c][v-1] = time the counter became >= v
    free = [(0.0, w) for w in range(nsm)]
    heapq.heapify(free)
    busy = 0.0
    end = 0.0
    wait_total = 0.0
    for t in tasks:
        t_free, w = heapq.heappop(free)
        ready = t_free
        for k in range(3):
            c, v = int(t[6 + k]), int(t[9 + k])
            if c >= 0 and v > 0:
                assert len(reach[c]) >= v, "queue is not a topological order"
                ready = max(ready, reach[c][v - 1])
        d = duration_us(t)
        wait_total += ready - t_free
        done = ready + d
        busy += d
        c, v = int(t[12]), int(t[13])
        if v > 0:
            while len(reach[c]) < v:
                reach[c].append(done)
        else:
            reach[c].append(done)
            reach[c].sort()
        heapq.heappush(free, (done, w))
        end = max(end, done)
    chain = sum(duration_us(t) for t in tasks if t[0] == DIAG) + 8.0 * (nb - 1)
    # the other chain of dependent tasks: PANEL(i, p) -> narrow UPDATE of tile (i, p+1) -> PANEL(i, p+1) ... on the rows just below
    # the diagonal (25 + 31 us per step with unblocked updates)
    update_chain = (25.0 + 31.0) * (nb - 1)
    return {"nb": nb, "tasks": len(tasks), "makespan_us": end, "work_bound_us": busy / nsm, "chain_us": chain, "update_chain_us": update_chain,
            "idle_waiting_us_per_worker": wait_total / nsm}


def main():
    for nb in [int(a) for a in sys.argv[1:]] or [32, 64]:
        r = simulate(nb)
        print(f"nb = {nb} (N = {nb * 128}): makespan {r['makespan_us']:.0f} us, work bound {r['work_bound_us']:.0f} us, "
              f"DIAG+PANEL chain {r['chain_us']:.0f} us, mean wait per worker {r['idle_waiting_us_per_worker']:.0f} us, "
              f"{r['tasks']} tasks")


if __name__ == "__main__":
    main()
