"""Recorder-compatible export (postprocessing/recorder.py:18-56 of the reference) for selected envs
of a ``BatchedBoatEnv``: the same ``;``-separated CSVs -- per-step rows with the nine columns of
``BoatEnv.return_all_data`` (boat_env.py:128-140), one ``info.csv`` row per finished episode, the
wind table once -- so the reference's ``Replayer`` / renderer can consume GPU runs unchanged.
``BatchedRecorder`` reads the fields from the host around every step; ``DeviceRecorder`` records into a
device ring and writes the same files at each flush.

The single-env drop-in ``sac_agent_b200.BoatEnv`` needs none of this: the reference's own
``Recorder(env)`` works on it as is (it only touches ``experiment_dir``, ``return_all_data()``,
``info`` and ``boat.wind``).
"""
from __future__ import annotations

import csv
import os

import numpy as np

from . import _lib

DATA_COLUMNS = ("boat_position_x", "boat_position_y", "boat_velocity_x", "boat_velocity_y", "boat_angle",
                "action_rudder", "reward", "rudder_angle", "n")
INFO_COLUMNS = ("termination", "reached_goal", "out_of_bounds", "out_of_fuel", "rudder_broken", "timeout",
                "episode_reward")
_FIELDS = ("s_x", "s_y", "v_x", "v_y", "s_r", "rudder_angle")
TERM_NAMES = ("", "reached_goal", "out_of_bounds", "out_of_fuel", "timeout", "rudder_broken")


def _append_rows(path, header, rows):
    """Appends ``rows`` to one ``;``-separated file, opened once; the header goes first when the file is new."""
    new = not os.path.exists(path)
    with open(path, "a", newline="") as f:
        w = csv.writer(f, delimiter=";")
        if new:
            w.writerow(header)
        w.writerows(rows)


class EpisodeBook:
    """Per-env bookkeeping and CSV rows of the reference's recorder, shared by both recorders: the last action /
    reward columns, episode numbering, the cumulative ``info`` counters (boat_env.py:24-32) and the file naming
    (no prefix when the only recorded id is 0, ``env<id>_`` otherwise).  Values are written as given, so the
    callers hand over numpy float64 scalars (or the int 0 of a row no step led to), like ``csv.writer`` saw them
    in the single-env reference."""

    def __init__(self, ids, experiment_dir):
        self.ids = [int(i) for i in ids]
        self.dir = os.path.join(experiment_dir, "episodes")
        os.makedirs(self.dir, exist_ok=True)
        self.episode = {i: 0 for i in self.ids}
        self.info = {i: dict.fromkeys(INFO_COLUMNS[1:], 0) | {"termination": ""} for i in self.ids}
        self.last_action = {i: 0 for i in self.ids}
        self.last_reward = {i: 0 for i in self.ids}

    def name(self, i, what):
        prefix = "" if self.ids == [0] else f"env{i}_"
        return os.path.join(self.dir, prefix + what)

    def data_row(self, i, s_x, s_y, v_x, v_y, s_r, rudder_angle):
        """(path, row) of env i's current state in its current episode's data file."""
        return (self.name(i, f"episode_{self.episode[i]}_data.csv"),
                [s_x, s_y, v_x, v_y, s_r, self.last_action[i], self.last_reward[i], rudder_angle, 20])

    def after_step(self, i, action, reward, term):
        """Book-keeping of one step of env i.  On termination the finished episode's ``info.csv`` (path, row) is
        returned and the next episode starts with zero action / reward columns; otherwise None."""
        self.last_action[i], self.last_reward[i] = action, reward
        self.info[i]["episode_reward"] += reward   # sequential float64 sum in step order
        if not term:
            return None
        name = TERM_NAMES[int(term)]
        self.info[i]["termination"] = name
        self.info[i][name] += 1
        out = self.name(i, "info.csv"), [self.info[i][k] for k in INFO_COLUMNS]
        self.info[i]["episode_reward"] = 0
        self.episode[i] += 1
        self.last_action[i] = self.last_reward[i] = 0
        return out

    def write_wind(self, i, wind_velocity, wind_angle):
        """wind.csv of env i (recorder.py:45-56), written once per file."""
        path = self.name(i, "wind.csv")
        if os.path.exists(path):
            return
        with open(path, "w", newline="") as f:
            w = csv.writer(f, delimiter=";")
            w.writerow(["wind_velocity", "wind_angle"])
            w.writerows(np.column_stack((wind_velocity, wind_angle)))


class BatchedRecorder:
    """Call ``write_data_to_csv()`` BEFORE every ``env.step`` (like main.py:79-81: row k is the state
    after k steps, the terminal step is never written) and ``after_step(actions)`` after it.
    ``env_ids`` are the env's own (local) indices.  Every call copies whole-population fields to the host:
    at scale, ``DeviceRecorder`` records the same files without that traffic."""

    def __init__(self, env, env_ids, experiment_dir):
        self.env = env
        self.book = EpisodeBook(env_ids, experiment_dir)
        self.ids, self.dir = self.book.ids, self.book.dir
        self.episode, self.info = self.book.episode, self.book.info
        self.last_action, self.last_reward = self.book.last_action, self.book.last_reward

    def write_data_to_csv(self):
        cols = {f: self.env.get_field(f).double().cpu().numpy() for f in _FIELDS}
        for i in self.ids:
            path, row = self.book.data_row(i, *(cols[f][i] for f in _FIELDS))
            _append_rows(path, DATA_COLUMNS, [row])

    def after_step(self, actions):
        """Book-keeping of one ``env.step(actions)``: last action / reward columns, and on termination the
        ``info.csv`` row of the finished episode (cumulative counters, boat_env.py:24-32)."""
        a = np.asarray(actions.detach().cpu() if hasattr(actions, "detach") else actions, dtype=np.float64).reshape(-1)
        r = self.env.reward.double().cpu().numpy()
        term = self.env.term.cpu().numpy()
        for i in self.ids:
            done = self.book.after_step(i, a[i], r[i], term[i])
            if done:
                path, row = done
                _append_rows(path, INFO_COLUMNS, [row])
        return None

    def write_winds_to_csv(self):
        """wind.csv of each recorded env's CURRENT episode (recorder.py:45-56), written once per file."""
        for i in self.ids:
            if not os.path.exists(self.book.name(i, "wind.csv")):
                self.book.write_wind(i, *self.env.wind_table(i))


# ring columns in the env's precision, in boatenv_record_ring order
_RING_T = ("s_x", "s_y", "v_x", "v_y", "s_r", "rudder_angle", "action", "reward")


class DeviceRecorder:
    """The recorder of postprocessing/recorder.py:18-56 for a fixed set of envs of a ``BatchedBoatEnv``, recorded
    on the device.  After each step one small kernel copies the recorded envs' state, action, reward and
    termination code into a device ring; nothing goes to the host until ``flush()``, which makes one copy of the
    ring and appends to the same CSVs ``BatchedRecorder`` writes, byte for byte (each file opened once per flush).

        env.reset(); rec = DeviceRecorder(env, ids, experiment_dir); rec.start()
        for t in ...: env.step(a)  (or memory.step_store(env, a));  rec.capture(a)
        rec.close()

    The fused collection kernel records inside itself: ``agent.collect(env, T, recorder=rec)`` (or
    ``TensorCorePolicy.collect(env, memory, T, recorder=rec)``) writes the T rows that T rounds of act +
    ``step_store`` + ``capture()`` would, in the same launch, so collection keeps one launch per T steps.  T may
    not exceed ``capacity``; rows that would not fit beside the pending ones are preceded by a flush.  Collect calls
    and ``capture()`` steps may be mixed on one recorder.

    ``env_ids`` are GLOBAL env ids (``env.env_id_offset`` + local index) inside the env's shard; files are named
    by them.  Rows: ``start()`` takes the state after reset, each ``capture()`` the state after the step (under
    auto-reset the next episode's first state) with that step's action / reward.  The result equals
    ``BatchedRecorder`` called before every step, after every step, and once more after the last.  A full ring is
    flushed by ``capture()`` itself, so no row is lost.  ``step_k`` / ``step_k_host`` windows (one observation
    per K sub-steps) and ``step_host`` steps (outputs in host buffers) cannot be recorded."""

    def __init__(self, env, env_ids, experiment_dir, capacity=1024):
        import torch
        ids = [int(i) for i in env_ids]
        lo, hi = env.env_id_offset, env.env_id_offset + env.n_envs
        if not ids:
            raise ValueError("env_ids is empty")
        if len(set(ids)) != len(ids):
            raise ValueError("env_ids has duplicates")
        outside = [i for i in ids if not lo <= i < hi]
        if outside:
            raise ValueError(f"env ids {outside[:8]} are outside this env's shard [{lo}, {hi})")
        if int(capacity) < 1:
            raise ValueError("capacity must be positive")
        self.env, self.ids, self.capacity = env, ids, int(capacity)
        self.book = EpisodeBook(ids, experiment_dir)
        self._local = torch.tensor([i - lo for i in ids], dtype=torch.int64, device=env.device)
        cap, m = self.capacity, len(ids)
        es = torch.empty(0, dtype=env.dtype).element_size()
        # one device buffer: 8 columns of T, episode (uint32), term (uint8) -- a flush is one copy
        self._nbytes = cap * m * (len(_RING_T) * es + 4 + 1)
        self._buf = torch.zeros(self._nbytes, dtype=torch.uint8, device=env.device)
        self._cols, off = {}, 0
        for name, dt, size in [(n, env.dtype, es) for n in _RING_T] + [("episode", torch.int32, 4),
                                                                        ("term", torch.uint8, 1)]:
            self._cols[name] = self._buf[off:off + cap * m * size].view(dt).view(cap, m)
            off += cap * m * size
        self._ring = _lib.RecordRing(**{k: v.data_ptr() for k, v in self._cols.items()}, capacity=cap)
        self._rows = self._flushed = 0        # rows captured / flushed so far
        self._stepped = []                    # per pending row: taken after a step (True) or after reset (False)
        self._ev = torch.cuda.Event()

    @property
    def pending(self):
        """Rows captured and not flushed yet."""
        return self._rows - self._flushed

    @property
    def episodes_finished(self):
        """Episodes of the recorded envs that ended in the flushed rows (one info.csv row each)."""
        return sum(self.book.episode.values())

    def _record(self, n, stepped, launch):
        """Reserves the next ``n`` rows (flushing first if they do not fit beside the pending ones), calls
        ``launch(row)``, which queues the writes of rows ``row .. row + n - 1`` on the current stream, and books
        them: the event marks their end, each is taken after a step (``stepped``) or after reset."""
        import torch
        if self.pending + n > self.capacity:
            self.flush()
        launch(self._rows)
        self._ev.record(torch.cuda.current_stream(self.env.device))
        self._rows += n
        self._stepped.extend([stepped] * n)

    def _take(self, stepped, actions=None):
        env = self.env
        if stepped:
            self._record(1, True, lambda row: env.record_rows(self._local, self._ring, row, env._actions(actions),
                                                              env.reward, env.term))
        else:
            self._record(1, False, lambda row: env.record_rows(self._local, self._ring, row))

    def start(self):
        """Captures the current state (call it after ``env.reset()``) and writes each env's wind.csv."""
        self._take(False)
        for i, j in zip(self.ids, self._local.tolist()):
            self.book.write_wind(i, *self.env.wind_table(j))

    def capture(self, actions):
        """Captures the step ``env.step(actions)`` / ``memory.step_store(env, actions)`` just made: one launch on
        the current stream reading ``env.reward`` and ``env.term``, no synchronisation."""
        self._take(True, actions)

    def flush(self):
        """Waits for the captures (an event on the stream they were queued on), copies the ring to the host once
        and appends the rows captured since the last flush to the CSVs."""
        n = self.pending
        if n == 0:
            return
        self._ev.synchronize()
        host = self._buf.cpu().numpy()
        cap, m = self.capacity, len(self.ids)
        cols, off = {}, 0
        ft = np.float32 if self.env.dtype.itemsize == 4 else np.float64
        for name, dt in [(k, ft) for k in _RING_T] + [("episode", np.uint32), ("term", np.uint8)]:
            size = cap * m * np.dtype(dt).itemsize
            cols[name] = host[off:off + size].view(dt).reshape(cap, m).astype(np.float64 if dt is ft else dt)
            off += size
        state = [cols[f] for f in _FIELDS]
        files = {}
        for r in range(n):
            slot = (self._flushed + r) % cap
            for j, i in enumerate(self.ids):
                if self._stepped[r]:
                    done = self.book.after_step(i, cols["action"][slot, j], cols["reward"][slot, j],
                                                cols["term"][slot, j])
                    if done:
                        files.setdefault(done[0], (INFO_COLUMNS, []))[1].append(done[1])
                path, row = self.book.data_row(i, *(c[slot, j] for c in state))
                files.setdefault(path, (DATA_COLUMNS, []))[1].append(row)
        for path, (header, rows) in files.items():
            _append_rows(path, header, rows)
        self._flushed += n
        del self._stepped[:n]

    def close(self):
        """Flushes what is left and releases the ring."""
        if getattr(self, "_buf", None) is not None:
            self.flush()
            self._buf = self._cols = None
