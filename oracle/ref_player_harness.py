"""Drive the REAL reference CChessPlayer (agent/player.py, unmodified) with a deterministic fake network
over a real multiprocessing.Pipe (SURVEY.md Appendix B).  Build-container only (needs /root/reference)."""
import threading
from multiprocessing import Pipe

import numpy as np

from . import ref_import
from .player import fake_eval_from_planes


class FakeNetServer:
    def __init__(self):
        self.me, self.you = Pipe()
        self.stop = False
        self.positions = 0
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def _run(self):
        while not self.stop:
            if self.me.poll(0.001):
                try:
                    planes = self.me.recv()
                except EOFError:
                    return
                self.positions += len(planes)
                self.me.send([fake_eval_from_planes(p) for p in planes])

    def close(self):
        self.stop = True


class FairLock:
    """A first-come-first-served lock.  The real player's sender thread sleeps while holding its queue lock and takes it
    again right after releasing it (player.py:113-123); with the runtime's unfair locks a search thread waiting for that
    lock can starve for as long as the host's thread wake-up latency keeps losing the race.  Served in arrival order, every
    waiter gets the lock after at most one more sender turn; the search's results do not depend on it."""

    def __init__(self):
        self._cond = threading.Condition(threading.Lock())
        self._next = 0
        self._serving = 0

    def acquire(self, blocking=True, timeout=-1):
        with self._cond:
            ticket = self._next
            self._next += 1
            while ticket != self._serving:
                self._cond.wait()
        return True

    def release(self):
        with self._cond:
            self._serving += 1
            self._cond.notify_all()

    def __enter__(self):
        return self.acquire()

    def __exit__(self, *exc):
        self.release()


def make_config(sims, search_threads=1, **over):
    cfg = ref_import.config("mini")
    pc = cfg.play
    pc.simulation_num_per_move = sims
    pc.search_threads = search_threads
    for k, v in over.items():
        setattr(pc, k, v)
    return cfg


def real_player_moves(states_and_opts, sims, seed, search_threads=1, use_history=False, **over):
    """Run action() of ONE real player object over a list of (state, turns, no_act, increase_temp[, hist]);
    returns per call: (action, {move: (n, w, q, p)}, sum_n)."""
    pm = ref_import.player_module()
    cfg = make_config(sims, search_threads, **over)
    srv = FakeNetServer()
    np.random.seed(seed)
    player = pm.CChessPlayer(cfg, pipes=srv.you, enable_resign=False, use_history=use_history)
    player.q_lock = FairLock()          # before any search runs; the sender and receiver pick it up on their next turn
    out = []
    try:
        for call in states_and_opts:
            state, turns, no_act, inc = call[:4]
            hist = list(call[4]) if len(call) > 4 and call[4] is not None else None
            action, policy = player.action(state, turns, no_act, increase_temp=inc, hist=hist)
            node = player.tree[state]
            edges = {m: (int(a.n), float(a.w), float(a.q), float(a.p)) for m, a in node.a.items()}
            out.append((action, edges, int(node.sum_n)))
    finally:
        player.close(wait=False)
        srv.close()
    return out
