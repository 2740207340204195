"""numpy restatement of the frame-deduplicated replay storage (csrc/dz_frames.cu, include/dqn_zoo_b200.h
dz_frame_store): the frame hash, the insert rule (zero frame, window of the last W adds, candidate order, ring
allocation and reclaim, pool overflow) and the closed-form synthetic fill.  The device's frame slots, metadata and
counters are compared with this bit for bit."""

import numpy as np

WINDOW = 16
_M = (1 << 64) - 1
K0, K1 = 0xA0761D6478BD642F, 0x9E3779B97F4A7C15


def mix64(x):
  """splitmix64 finalizer on uint64 arrays (wrapping arithmetic)."""
  x = np.asarray(x, dtype=np.uint64)
  with np.errstate(over='ignore'):
    x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
  return x ^ (x >> np.uint64(31))


def frame_hash(data) -> int:
  """mix64(n ^ K0) + sum_k mix64(w_k ^ k * K1) mod 2^64, w_k the little-endian 8-byte words of the zero-padded bytes."""
  b = np.ascontiguousarray(data, dtype=np.uint8).reshape(-1)
  n = b.size
  padded = np.zeros((n + 7) // 8 * 8, dtype=np.uint8)
  padded[:n] = b
  w = padded.view('<u8').astype(np.uint64)
  with np.errstate(over='ignore'):
    k = np.arange(w.size, dtype=np.uint64) * np.uint64(K1)
  terms = [int(x) for x in mix64(w ^ k)]
  return (int(mix64(np.uint64(n ^ K0))) + sum(terms)) & _M


def planes(stack):
  """(H, W, S) stack -> S frames (H*W bytes each), channel order."""
  s = np.asarray(stack, dtype=np.uint8)
  return [np.ascontiguousarray(s[:, :, c]).reshape(-1) for c in range(s.shape[2])]


class FrameStore:
  """The device store's state after the same sequence of adds (frames in slots 1..F, slot 0 the zero frame)."""

  def __init__(self, capacity, frame_capacity, obs_shape):
    h, w, self.stack = obs_shape
    self.obs_shape = tuple(obs_shape)
    self.capacity, self.F, self.frame_bytes = capacity, frame_capacity, h * w
    P = 2 * self.stack
    self.frames = np.zeros((frame_capacity + 1, self.frame_bytes), dtype=np.uint8)
    self.row_frames = np.zeros((capacity, P), dtype=np.int32)
    self.hash = np.zeros(frame_capacity + 1, dtype=np.uint64)
    self.born = np.full(frame_capacity + 1, -1, dtype=np.int64)
    self.last_ref = np.full(frame_capacity + 1, -1, dtype=np.int64)
    self.appends = 0
    self.window = np.full((WINDOW, 1 + P), -1, dtype=np.int64)   # per add (id % W): id, appended slots
    self.pool_full = False
    self.full_ids = []

  def add(self, item_id, oldest_live, s_tm1, s_t):
    """One insert (dz_replay_add with a frame store); returns the row's 2S slots."""
    P = 2 * self.stack
    ps = planes(s_tm1) + planes(s_t)
    hs = [frame_hash(p) for p in ps]
    appended = []
    row = []
    full = False
    for p in range(P):
      choice = -1
      if not ps[p].any():
        choice = 0
      else:
        cands = [s for s in reversed(appended) if int(self.hash[s]) == hs[p]]
        for j in range(item_id - 1, max(item_id - WINDOW, 0) - 1, -1):
          ent = self.window[j % WINDOW]
          if ent[0] != j:
            continue
          for s in ent[1:][::-1]:
            if s > 0 and self.born[s] == j and int(self.hash[s]) == hs[p]:
              cands.append(int(s))
        for s in cands:
          if np.array_equal(self.frames[s], ps[p]):
            choice = s
            break
      if choice < 0:
        slot = 1 + self.appends % self.F
        if self.appends >= self.F and self.last_ref[slot] >= oldest_live:
          full = True
          break
        self.frames[slot] = ps[p]
        self.hash[slot] = np.uint64(hs[p])
        self.born[slot] = item_id
        appended.append(slot)
        self.appends += 1
        choice = slot
      if choice > 0:
        self.last_ref[choice] = item_id
      row.append(choice)
    r = item_id % self.capacity
    self.row_frames[r] = -1 if full else row
    if full:
      self.pool_full = True
      self.full_ids.append(item_id)
    ent = np.full(1 + P, -1, dtype=np.int64)
    ent[0] = item_id
    ent[1:1 + len(appended)] = appended
    self.window[item_id % WINDOW] = ent
    return self.row_frames[r].copy()

  def stack_of(self, slots):
    """Re-assembles an (H, W, S) stack from S frame slots (-1 reads as zeros)."""
    h, w, S = self.obs_shape
    out = np.zeros((h * w, S), dtype=np.uint8)
    for c, s in enumerate(slots):
      if s >= 0:
        out[:, c] = self.frames[s]
    return out.reshape(h, w, S)

  def get(self, item_id):
    row = self.row_frames[item_id % self.capacity]
    return self.stack_of(row[:self.stack]), self.stack_of(row[self.stack:])

  def state_vector(self):
    """The device's d_state: appends, reserved 0, then the window entries."""
    return np.concatenate([[self.appends, 0], self.window.reshape(-1)]).astype(np.int64)


def min_frame_capacity(capacity, obs_shape, transitions):
  """Smallest F with which `transitions` (a list of (s_tm1, s_t)) fit without overflow (linear search)."""
  F = 1
  while True:
    st = FrameStore(capacity, F, obs_shape)
    live = []
    for i, (a, b) in enumerate(transitions):
      live.append(i)
      if len(live) > capacity:
        live.pop(0)
      st.add(i, live[0], a, b)
      if st.pool_full:
        break
    if not st.pool_full:
      return F
    F += 1


# ---- closed-form synthetic fill (dz_replay_fill_synthetic_frames) ------------------------------------------------


def synthetic_frame(seed, a, frame_bytes):
  """Bytes of the frame with append index `a`: splitmix64 words of a counter keyed by seed."""
  words = frame_bytes // 8
  with np.errstate(over='ignore'):
    base = np.uint64(seed) * np.uint64(0x9E3779B97F4A7C15) + np.uint64(0x5851F42D4C957F2D) + \
        np.uint64(a) * np.uint64(words)
    ctr = base + np.arange(words, dtype=np.uint64)
  return mix64(ctr).astype('<u8').view(np.uint8)


def synthetic_transitions(n, episode_length, seed, obs_shape):
  """The stacks (s_tm1, s_t) of transitions 0..n-1 of the synthetic episode stream: a new frame per timestep, stacks
  padded with trailing zero planes at episode start (processors.py:497-504), 1-step transitions."""
  h, w, S = obs_shape
  L = episode_length
  out = []
  for i in range(n):
    e, t = divmod(i, L)
    a0 = e * (L + 1)

    def stack(T):
      st = np.zeros((h * w, S), dtype=np.uint8)
      js = list(range(0, T + 1)) if T < S else list(range(T - S + 1, T + 1))
      for c, j in enumerate(js):
        st[:, c] = synthetic_frame(seed, a0 + j, h * w)
      return st.reshape(h, w, S)
    out.append((stack(t), stack(t + 1)))
  return out


def synthetic_fill(capacity, frame_capacity, obs_shape, n, episode_length, seed, rows=None):
  """Closed-form FrameStore state after n sequential adds of `synthetic_transitions` (no eviction: n <= capacity).
  Returns a FrameStore; frame bytes are generated only for the slots named in `rows`' stacks when `rows` is given
  (the full 1M-row store is too large to restate), else for every appended frame."""
  h, w, S = obs_shape
  L = episode_length
  st = FrameStore(1, 1, obs_shape)
  st.capacity, st.F = capacity, frame_capacity
  P = 2 * S
  appends = n + -(-n // L)
  assert appends <= frame_capacity
  st.appends = appends
  i = np.arange(n, dtype=np.int64)
  e, t = i // L, i % L

  def slots(which, c):
    T = t + which
    j = np.where(T < S, c, T - S + 1 + c)
    valid = (T >= S) | (c <= T)
    return np.where(valid, 1 + e * (L + 1) + j, 0).astype(np.int32)
  row_frames = np.stack([slots(p // S, p % S) for p in range(P)], axis=1)
  a = np.arange(appends, dtype=np.int64)
  fe, fj = a // (L + 1), a % (L + 1)
  te = np.minimum(L, n - fe * L)
  born = np.full(frame_capacity + 1, -1, dtype=np.int64)
  last_ref = np.full(frame_capacity + 1, -1, dtype=np.int64)
  born[1 + a] = fe * L + np.maximum(fj - 1, 0)
  last_ref[1 + a] = fe * L + np.minimum(fj + S - 1, te - 1)
  st.born, st.last_ref = born, last_ref
  st.row_frames = row_frames
  window = np.full((WINDOW, 1 + P), -1, dtype=np.int64)
  for k in range(max(0, n - WINDOW), n):
    ee, tt = divmod(k, L)
    a0 = ee * (L + 1)
    window[k % WINDOW, 0] = k
    if tt == 0:
      window[k % WINDOW, 1:3] = (1 + a0, 2 + a0)
    else:
      window[k % WINDOW, 1] = 1 + a0 + tt + 1
  st.window = window
  want = np.arange(appends) if rows is None else np.unique(row_frames[np.asarray(rows)].reshape(-1) - 1)
  want = want[want >= 0]
  st.frames = {int(x) + 1: synthetic_frame(seed, int(x), h * w) for x in want}
  st.frames[0] = np.zeros(h * w, dtype=np.uint8)
  st.hash = {s: frame_hash(f) for s, f in st.frames.items()}
  return st
