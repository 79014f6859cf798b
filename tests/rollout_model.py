"""Host model of the per-agent frame history of closed-loop serving (bc_stage_history, trainer.RolloutActStep): which frame
every ring slot of every agent holds after each tick, and which ring planes form each agent's window. Shared by
tests/test_rollout_host.py (against a per-agent deque) and tests/test_gpu_rollout_serving.py (against the device)."""
import numpy as np


class RingModel:
    """n_agents x 8 tick slots of frame ids (-1 = never written). Tick t uses slot s = t mod 4: the new frame goes to slots
    s and s + 4, or to all 8 for an agent that is reset (and for every agent on a reset_all tick)."""

    def __init__(self, n_agents: int, cams: int):
        self.n, self.cams = n_agents, cams
        self.slots = np.full((n_agents, 8), -1, np.int64)
        self.t = 0

    def tick(self, frame_ids, reset, reset_all: bool = False) -> int:
        """frame_ids (n,) ids of this tick's frames, reset (n,) bool. Returns the slot of this tick."""
        s = self.t % 4
        for a in range(self.n):
            if reset_all or reset[a]:
                self.slots[a, :] = frame_ids[a]
            else:
                self.slots[a, s] = self.slots[a, s + 4] = frame_ids[a]
        self.t += 1
        return s

    def window(self, s: int) -> np.ndarray:
        """(n, 4) frame ids of every agent's window after the tick of slot s, oldest first."""
        return self.slots[:, s + 1:s + 5].copy()

    def plane(self, a: int, j: int, k: int) -> int:
        """Ring plane of agent a, tick slot j, camera k."""
        return (a * 8 + j) * self.cams + k

    def window_planes(self, s: int, a: int) -> list:
        """Ring planes of agent a's window, in conv1's channel order (channel = cams * frame + camera): the contiguous planes
        [(s+1)*cams, (s+5)*cams) of its ring, which is what RolloutActStep points conv1 at."""
        base = a * 8 * self.cams + (s + 1) * self.cams
        return [base + ch for ch in range(4 * self.cams)]
