"""Self-play output contract of the reference (SURVEY 8f-1): per finished game the arrays ``selfplay_worker`` hands to
``DataManager.add_selfplay_data`` (azchess/selfplay/internal.py:447-466, 612-651):

    s          float32[T, 19, 8, 8]   encode_board of the position before every searched move       (internal.py:447)
    pi         float32[T, 4672]       MCTS visit distribution returned by MCTS.run                   (internal.py:408, mcts.py:828-849);
                                      the improved policy softmax(logits + sigma) in Gumbel mode (DESIGN.md §9)
    z          float32[T]             game result (White's view) x (+1 White / -1 Black to move)     (internal.py:612-616)
    legal_mask uint8[T, 4672]         MoveEncoder.get_legal_actions                                  (internal.py:454)
    meta_moves int32[1], meta_result float32[1], meta_resigned int8[1], meta_draw int8[1],
    meta_avg_policy_entropy float32[1], meta_avg_sims float32[1]                                    (internal.py:632-637)

The games run on the GPU (selfplay.SelfPlayEngine) and so does the assembly of their records: per ply the packed root positions (72 B),
the root children's policy indices and visit counts stay in HBM, in a ring of ``max_game_len`` plies.  When games end, the rows of all
of them are gathered on the device, go back through the encode kernel in one batch (planes + legal masks), ``pi`` is scattered on the
device as ``n / total`` (float64 divide, float32 store -- mcts.py:846), and each array crosses to the host ONCE per group of finished
games; the per-game arrays are views of it.  ``ssl_{task}`` arrays (internal.py:460-466, 644-648) come from the SSL target kernel
(``m0_ssl_targets``) for the tasks in ``ssl_tasks``.
"""
from __future__ import annotations

import os
import time
from typing import Any, Dict, List, Optional

import numpy as np

from . import _native

GROUP_ROWS = 32000      # positions assembled per encode launch / host transfer: 32,588 B each with all SSL maps = one 1 GiB pinned block


class GameRecorder:
    """Collects the training records of the games a SelfPlayEngine plays.

        rec = GameRecorder(sp)
        sp.start()
        while ...:
            sp.begin_move(); [sp.search_step() ...]
            rec.after_search()          # root positions + visit counts of this ply -> the device ring (no host round trip)
            sp.end_move()
            for game in rec.iter_after_move(defer=True):   # finished games as the reference's game_data dictionaries
                np.savez_compressed(path, **game)
        for game in rec.flush(): ...

    With ``defer=True`` the records of the games that ended on a ply are assembled and copied to the host on a side stream WHILE the
    next ply is searched, and are handed out by the next call (or by ``flush()``); ``after_move()`` / ``defer=False`` hand them out at once.
    """

    MAX_INFLIGHT = 2     # groups whose device-to-host copies may be in flight before the oldest is handed out (pinned host memory bound)

    def __init__(self, sp, keep_plies: Optional[int] = None, ssl_tasks=()):
        import collections
        import torch
        self.sp = sp
        self.G = sp.G
        self._torch = torch
        dev = sp.device
        # a game's searched plies are consecutive engine plies and there are at most max_game_len of them; the ring keeps as many plies
        # again, so a finished game's rows stay readable for max_game_len more plies (iter_after_move(max_games=...))
        self.max_game_plies = L = int(sp.sp.get("max_game_len", 200))
        self.keep_plies = K = max(int(keep_plies), L + 3) if keep_plies else 2 * L + 3
        self._pos = torch.zeros((K, self.G, 9), dtype=torch.int64, device=dev)
        self._idx = torch.zeros((K, self.G, 256), dtype=torch.int16, device=dev)
        self._vis = torch.zeros((K, self.G, 256), dtype=torch.int32, device=dev)
        self._cnt = torch.zeros((K, self.G), dtype=torch.int32, device=dev)
        # Gumbel search: the recorded pi is the improved policy of the root children (float32, child order), not n / total
        self._gpi = torch.zeros((K, self.G, 256), dtype=torch.float32, device=dev) if getattr(sp, "gumbel", None) else None
        self._mvcnt = torch.zeros((self.G,), dtype=torch.int32, device=dev)
        self._now = 0                                       # engine plies recorded so far
        self._start = np.zeros((self.G,), dtype=np.int64)   # engine ply at which the current game of a slot started
        self.ssl_tasks = tuple(t for t in ssl_tasks if t in ("piece", "threat", "pin", "fork", "control"))   # model.ssl_tasks (internal.py:251-256)
        self._side = torch.cuda.Stream(device=dev)          # gathers, encode / SSL / scatter launches and the D2H copies of finished games
        self._inflight = collections.deque()                # groups launched on the side stream, oldest first
        self._backlog = collections.deque()                 # finished games (slot, first ply, plies, engine record) not launched yet
        self._ring_read = None                              # event: the side stream has read the ring rows of every launched group
        self.timing = collections.Counter()                 # host seconds by phase (tools/worker_throughput.py reports them)

    def after_search(self) -> None:
        """Call after the last search step of a ply and before SelfPlayEngine.end_move()."""
        torch = self._torch
        eng = self.sp.engine
        lib = _native.lib()
        if self._ring_read is not None:      # the ring slot written below may only be reused once the pending gathers have read the ring
            torch.cuda.current_stream(self.sp.device).wait_event(self._ring_read)
            self._ring_read = None
        st = _native.current_stream()
        k = self._now % self.keep_plies
        if self._gpi is not None:
            self.sp.gumbel_result()
            self._gpi[k].copy_(eng.gb_pi_children)
        else:
            eng.result(with_pi=False)
        _native.check(lib.m0_games_get_positions(eng._h, self._pos[k].data_ptr(), st), "m0_games_get_positions")
        # policy index of every root child (child order = legal-move order = m0_legal_moves order)
        _native.check(lib.m0_legal_moves(self._pos[k].data_ptr(), self.G, None, self._idx[k].data_ptr(), self._mvcnt.data_ptr(), st), "m0_legal_moves")
        self._vis[k].copy_(eng.res_visits)
        self._cnt[k].copy_(eng.res_count)
        self._now += 1

    def after_move(self) -> List[Dict[str, np.ndarray]]:
        """Call after SelfPlayEngine.end_move(); returns the game_data dictionaries of the games that just ended."""
        return list(self.iter_after_move())

    def iter_after_move(self, defer: bool = False, max_games: Optional[int] = None):
        """after_move() as a generator.  The finished games are assembled in groups of <= 32,000 positions, so a ply on which thousands
        of games end (all slots reaching max_game_len together) never holds more than a few groups' arrays (~1 GB of planes / masks /
        pi each) on the host.  ``defer``: see the class docstring.  ``max_games``: start the assembly of at most this many games now;
        the others wait on the DEVICE (their rows stay valid in the ring for another max_game_len plies) and are started by later
        calls, oldest first -- a caller whose shard writers are busy keeps the GPU searching instead of blocking on them.
        Exhaust the generator before the next after_search()."""
        now = self._now                              # one past the ply just played
        t0 = time.perf_counter()
        finished = self.sp.finished_games()
        self.timing["finished_games"] += time.perf_counter() - t0
        for fin in finished:
            slot = fin["slot"]
            first = int(self._start[slot])
            self._start[slot] = now
            # the engine's own count of searched plies: 0 for a game that was over after its opening plies (the reference saves nothing
            # for it, internal.py:627 / :654)
            T = min(now - first, int(fin["moves"]))
            if T <= 0 or now - first > self.max_game_plies:
                continue  # (a ring shorter than the game: skipped, never truncated)
            self._backlog.append((slot, first, T, fin))
        yield from self._deliver_all()               # groups launched on earlier plies: their copies ran under this ply's search
        # deferred: never wait for a copy here -- at most MAX_INFLIGHT groups are started per call (a ply on which every slot ends is
        # spread over the following plies), except for games whose ring rows are about to be overwritten
        yield from self._launch_backlog(float("inf") if max_games is None else int(max_games), wait=not defer)
        if not defer:
            yield from self._deliver_all()

    def flush(self):
        """Assemble and hand out everything that is still waiting (the end of the run, or a caller that wants all games now)."""
        yield from self._deliver_all()
        yield from self._launch_backlog(float("inf"))
        yield from self._deliver_all()

    def pending_games(self) -> int:
        """Games whose host arrays are in flight (page-locked memory is held for them)."""
        return sum(len(g["todo"]) for g in self._inflight)

    def backlog_games(self) -> int:
        """Finished games still waiting in the device ring."""
        return len(self._backlog)

    def _deliver_all(self):
        while self._inflight:
            yield from self._deliver(self._inflight.popleft())

    def _launch_backlog(self, budget, wait: bool = True):
        """Start the assembly of backlog games, oldest first, in groups of <= GROUP_ROWS positions: ``budget`` games, plus every game whose
        oldest ring row is about to be overwritten.  When MAX_INFLIGHT groups are in flight: ``wait`` hands out the oldest to make
        room, otherwise the rest of the backlog stays for the next call."""
        now, K = self._now, self.keep_plies
        # the ring row of ply `first` is rewritten by the after_search of ply first + K: everything up to the last backlog entry that
        # close to it is started now, whatever the budget says (the backlog is ordered by the END of the games, not by their start)
        force = 0
        for i, item in enumerate(self._backlog):
            if item[1] + K - now <= 2:
                force = i + 1
        synced = False
        while self._backlog:
            group, rows = [], 0
            full = not wait and len(self._inflight) >= self.MAX_INFLIGHT
            while self._backlog and (not group or rows + self._backlog[0][2] <= GROUP_ROWS):
                if (budget <= 0 or full) and force <= 0:
                    break
                item = self._backlog.popleft()
                group.append(item)
                rows += item[2]
                budget -= 1
                force -= 1
            if not group:
                return
            if not synced:
                torch = self._torch
                ready = torch.cuda.Event()
                ready.record(torch.cuda.current_stream(self.sp.device))     # the ring holds everything up to the ply just played
                self._side.wait_event(ready)
                synced = True
            while len(self._inflight) >= self.MAX_INFLIGHT:
                yield from self._deliver(self._inflight.popleft())
            t0 = time.perf_counter()
            self._inflight.append(self._launch(group))
            self.timing["launch"] += time.perf_counter() - t0

    def _launch(self, todo) -> Dict[str, Any]:
        """Queue the assembly of a group of finished games on the side stream: their rows gathered from the ring, ONE encode launch
        (planes + legal masks), one SSL launch and one scatter of the visit distribution over the concatenated positions, one D2H copy
        per array into page-locked memory.  Nothing here waits for the device."""
        torch = self._torch
        lib = _native.lib()
        dev = self.sp.device
        K = self.keep_plies
        lens = np.array([T for _, _, T, _ in todo], dtype=np.int64)
        offs = np.concatenate([[0], np.cumsum(lens)])
        N = int(offs[-1])
        within = np.arange(N, dtype=np.int64) - np.repeat(offs[:-1], lens)
        ply = (np.repeat(np.array([first for _, first, _, _ in todo], dtype=np.int64), lens) + within) % K
        slot = np.repeat(np.array([s for s, _, _, _ in todo], dtype=np.int64), lens)
        # (page-locked staging: a pageable host-to-device copy would block this thread until the side stream has finished the groups
        # queued before this one)
        h_index = torch.empty((2, N), dtype=torch.int64, pin_memory=True)
        h_index[0].copy_(torch.from_numpy(ply))
        h_index[1].copy_(torch.from_numpy(slot))
        with torch.cuda.stream(self._side):
            d_index = h_index.to(dev, non_blocking=True)
            d_ply, d_slot = d_index[0], d_index[1]
            dpos = self._pos[d_ply, d_slot].contiguous()                        # [N, 9]
            idx = (self._idx[d_ply, d_slot].to(torch.int64) & 0xFFFF)            # [N, 256] policy indices (uint16 stored as int16)
            vis = self._vis[d_ply, d_slot]
            cnt = self._cnt[d_ply, d_slot]
            self._ring_read = torch.cuda.Event()
            self._ring_read.record(self._side)
            live = torch.arange(256, device=dev)[None, :] < cnt[:, None]
            n = torch.where(live, vis, 0).to(torch.float64)
            tot = n.sum(1)
            # pi[child.move_idx] = child.n / total: float64 divide, float32 store (mcts.py:840-847); the padding entries add 0.0 at index 0
            vals = torch.where(live & (tot[:, None] > 0), n / tot.clamp(min=1.0)[:, None], 0.0).to(torch.float32)
            if self._gpi is not None:
                vals = torch.where(live, self._gpi[d_ply, d_slot], 0.0)
            pi = torch.zeros((N, 4672), dtype=torch.float32, device=dev)
            pi.scatter_add_(1, torch.where(live, idx, 0), vals)
            planes = torch.empty((N, 19, 8, 8), dtype=torch.float32, device=dev)
            mask = torch.empty((N, 4672), dtype=torch.uint8, device=dev)
            _native.check(lib.m0_encode_positions(dpos.data_ptr(), N, planes.data_ptr(), mask.data_ptr(), None, None, None, _native.current_stream()),
                          "m0_encode_positions")
            turns = torch.where((dpos[:, 8] & 1) != 0, 1.0, -1.0).to(torch.float32)               # packed state word: bit 0 = side to move
            maps = {}
            if self.ssl_tasks:
                from .encoding import ssl_targets_device
                maps = ssl_targets_device(dpos)

            # ONE page-locked block per group from torch's caching host allocator, the arrays carved out of it: the copies run at PCIe
            # speed (57 GB/s measured against 13 GB/s into pageable memory), the per-game arrays handed out are views of the block (no
            # copy on the host), and the block returns to the cache when the last view is dropped.  A fresh page-locked allocation
            # costs ~0.45 s per GB on the box, a cached one microseconds: GROUP_ROWS keeps a full group just under a 1 GiB block.
            srcs = [planes, mask, pi, turns, tot] + [maps[t] for t in self.ssl_tasks]
            offsets, total = [], 0
            for t in srcs:
                offsets.append(total)
                total += (t.numel() * t.element_size() + 255) & ~255
            t0 = time.perf_counter()
            block = torch.empty((total,), dtype=torch.uint8, pin_memory=True)
            self.timing["launch_pinned_block"] += time.perf_counter() - t0
            views = []
            for t, off in zip(srcs, offsets):
                h = block[off:off + t.numel() * t.element_size()].view(t.dtype).view(t.shape)
                h.copy_(t, non_blocking=True)
                views.append(h)
            hosts, ssl_hosts = views[:5], dict(zip(self.ssl_tasks, views[5:]))
            done = torch.cuda.Event()
            done.record(self._side)
        return {"todo": todo, "offs": offs, "hosts": hosts, "ssl": ssl_hosts, "done": done}

    def _deliver(self, grp) -> List[Dict[str, np.ndarray]]:
        """The game_data dictionaries of a launched group; the per-game arrays are views of the group's host arrays."""
        t0 = time.perf_counter()
        grp["done"].synchronize()
        self.timing["deliver_wait_for_copy"] += time.perf_counter() - t0
        t0 = time.perf_counter()
        planes_h, mask_h, pi_h, turns_h, tot_h = [h.numpy() for h in grp["hosts"]]
        ssl_h = {t: h.numpy() for t, h in grp["ssl"].items()}
        offs = grp["offs"]
        out = []
        for i, (_, _, T, fin) in enumerate(grp["todo"]):
            a, b = int(offs[i]), int(offs[i + 1])
            z = float(fin["result"])
            out.append({
                **{f"ssl_{t}": ssl_h[t][a:b] for t in ssl_h},
                "s": planes_h[a:b], "pi": pi_h[a:b], "z": (np.float32(z) * turns_h[a:b]).astype(np.float32), "legal_mask": mask_h[a:b],
                "meta_moves": np.array([T], dtype=np.int32), "meta_result": np.array([z], dtype=np.float32),
                "meta_resigned": np.array([1 if fin["resigned"] else 0], dtype=np.int8), "meta_draw": np.array([1 if z == 0.0 else 0], dtype=np.int8),
                "meta_avg_policy_entropy": np.array([fin["avg_policy_entropy"]], dtype=np.float32),
                "meta_avg_sims": np.array([float(tot_h[a:b].mean()) if T else 0.0], dtype=np.float32),
            })
        self.timing["deliver_build_dicts"] += time.perf_counter() - t0
        return out


def write_game_npz(directory: str, game: Dict[str, np.ndarray], worker_id: int, game_id: int, compresslevel: Optional[int] = None) -> str:
    """The shard writer used when no DataManager is passed to ``selfplay_worker``: np.savez_compressed of the game_data dictionary,
    written to a temporary name and renamed (as DataManager._save_npz_shard does, data_manager.py:198-228).  The reference names its
    shards ``selfplay_{timestamp}_{uuid8}.npz`` and records them in SQLite (data_manager.py:230-243) -- that bookkeeping is the
    caller's (out of scope here); this writer names them ``selfplay_w{worker}_g{game}_{ms}.npz``.  ``compresslevel`` 1..9 writes the
    same .npz container (np.load reads it unchanged) with that deflate level instead of zipfile's default 6: level 1 takes a third of
    the time per 200-ply game for a 1.6 times larger file."""
    import time
    os.makedirs(directory, exist_ok=True)
    path = os.path.join(directory, f"selfplay_w{worker_id}_g{game_id}_{int(time.time() * 1000)}.npz")
    tmp = path + ".tmp"
    if compresslevel is None:
        with open(tmp, "wb") as f:
            np.savez_compressed(f, **game)
    else:
        import zipfile
        with zipfile.ZipFile(tmp, "w", compression=zipfile.ZIP_DEFLATED, compresslevel=int(compresslevel), allowZip64=True) as zf:
            for k, v in game.items():
                with zf.open(k + ".npy", "w", force_zip64=True) as f:
                    np.lib.format.write_array(f, np.asanyarray(v), allow_pickle=False)
    os.replace(tmp, path)
    return path
