"""numpy restatement of the device `spaces` env (oracle/SPEC_spaces.md).  TEST INFRASTRUCTURE: independent of
pufferlib_b200/csrc/env_spaces.cu, which the GPU tests check against it bit for bit.

The reference env (ocean.py:356-404) behind EpisodeStats, GymnasiumPufferEnv and Serial: every step is terminal, the
next send() resets (action ignored), a step row repeats the observation of the reset row before it.  Observation record
(np.dtype(align=True) of the Dict, keys sorted): flat int8[5] at byte 0, 3 zero bytes, image float32[5][5] at byte 8,
108 bytes.  Actions [N, 2]: column 0 = flat, column 1 = image.  Only the RNG is builder-defined (counter-based rand32).
"""
import numpy as np

RECORD_BYTES = 108
NVEC = (2, 2)
DRAWS_PER_RESET = 30          # 25 image values (row-major), then 5 flat values


def mix32(x):
    """splitmix64 finaliser, upper 32 bits (uint64 numpy arrays, wrapping arithmetic)."""
    with np.errstate(over='ignore'):
        x = x + np.uint64(0x9E3779B97F4A7C15)
        x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        x = x ^ (x >> np.uint64(31))
    return (x >> np.uint64(32)).astype(np.uint32)


def rand32(seed_e, ctr):
    with np.errstate(over='ignore'):
        return mix32(np.asarray(seed_e, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15)
                     + np.asarray(ctr, dtype=np.uint64) * np.uint64(0xD1B54A32D192ED03))


def draw_observation(seed_e, k):
    """Observation of reset number k (0 = async_reset) of the envs with per-env seeds seed_e: (flat int8 [n, 5],
    image float32 [n, 5, 5]).  Image value = (b0 + b1 + b2 + b3 - 510) / 128 over the four bytes of one draw (exact in
    fp32, so the sign of the 25-value sum does not depend on summation order); flat value = draw % 3 - 1."""
    seed_e = np.asarray(seed_e, dtype=np.uint64).reshape(-1, 1)
    ctr = np.asarray(k, dtype=np.uint64).reshape(-1, 1) * np.uint64(DRAWS_PER_RESET) + \
        np.arange(DRAWS_PER_RESET, dtype=np.uint64)[None]
    r = rand32(seed_e, ctr).astype(np.int64)
    byte_sum = (r & 255) + ((r >> 8) & 255) + ((r >> 16) & 255) + ((r >> 24) & 255)
    image = ((byte_sum[:, :25] - 510).astype(np.float32) / np.float32(128)).reshape(-1, 5, 5)
    flat = (r[:, 25:] % 3 - 1).astype(np.int8)
    return flat, image


def pack(flat, image):
    """[n, 5] int8 + [n, 5, 5] float32 -> [n, 108] uint8 records (padding bytes zero)."""
    n = flat.shape[0]
    rec = np.zeros((n, RECORD_BYTES), dtype=np.uint8)
    rec[:, 0:5] = np.ascontiguousarray(flat, dtype=np.int8).view(np.uint8)
    rec[:, 8:] = np.ascontiguousarray(image, dtype=np.float32).reshape(n, 25).view(np.uint8)
    return rec


def reward(flat, image, actions):
    """0.5 * [sum(flat) > 0 == a_flat] + 0.5 * [sum(image) > 0 == a_image]; actions clamped into [0, 2) per column."""
    a = np.clip(np.asarray(actions, dtype=np.int64).reshape(-1, 2), 0, 1)
    flat_sign = flat.astype(np.int64).sum(1) > 0
    image_sign = np.asarray([np.sum(im) > 0 for im in image])      # np.sum over one (5, 5) array, as ocean.py:388
    return (0.5 * (flat_sign == a[:, 0]) + 0.5 * (image_sign == a[:, 1])).astype(np.float32)


class SpacesSerial:
    """Serial-like vectoriser (async_reset / send / recv).  obs_source(env_ids, k) -> (flat, image) replaces the
    counter-based draws, e.g. with the observations a reference run recorded."""

    def __init__(self, num_envs, env_index_offset=0, obs_source=None):
        self.n = num_envs
        self.offset = int(env_index_offset)
        self.obs_source = obs_source
        self.observations = np.zeros((num_envs, RECORD_BYTES), dtype=np.uint8)
        self.rewards = np.zeros(num_envs, dtype=np.float32)
        self.terminals = np.zeros(num_envs, dtype=bool)
        self.truncations = np.zeros(num_envs, dtype=bool)
        self.masks = np.ones(num_envs, dtype=bool)
        self.agent_ids = np.arange(num_envs)
        self.infos = []

    def _draw(self, ids):
        if self.obs_source is not None:
            return self.obs_source(ids, self.k[ids])
        seed_e = (np.uint64(self.seed) + np.uint64(self.offset) + ids.astype(np.uint64))
        return draw_observation(seed_e, self.k[ids])

    def async_reset(self, seed=42):
        self.seed = seed % (1 << 64)
        ids = np.arange(self.n)
        self.k = np.zeros(self.n, dtype=np.int64)
        self.done = np.zeros(self.n, dtype=bool)
        self.flat, self.image = self._draw(ids)
        self.observations[:] = pack(self.flat, self.image)
        self.rewards[:] = 0
        self.terminals[:] = False
        self.infos = []

    def send(self, actions):
        a = np.asarray(actions, dtype=np.int64).reshape(self.n, 2)
        resetting = self.done.copy()
        stepping = ~resetting
        self.rewards[:] = 0
        if resetting.any():
            ids = np.nonzero(resetting)[0]
            self.k[ids] += 1
            f, im = self._draw(ids)
            self.flat[ids], self.image[ids] = f, im
        if stepping.any():
            ids = np.nonzero(stepping)[0]
            self.rewards[ids] = reward(self.flat[ids], self.image[ids], a[ids])
        self.terminals[:] = stepping
        self.done = stepping.copy()
        self.observations[:] = pack(self.flat, self.image)
        self.infos = [{'episode_return': float(self.rewards[i]), 'episode_length': 1, 'score': float(self.rewards[i])}
                      for i in np.nonzero(self.terminals)[0]]

    def recv(self):
        return (self.observations, self.rewards, self.terminals, self.truncations, self.infos, self.agent_ids,
                self.masks)
