"""Reference for amira_gmg_linear_walks: a plain loop that restates GeneMerGraph._walk over a step table, and the
oracle-backed test double with DeviceGraph.linear_walks built on it.  TEST INFRASTRUCTURE ONLY."""
import numpy as np

from tests.fake_device import OracleBackedDevice


def walk_loop(st, s0, want_branched=False):
    """GeneMerGraph._walk restated on one walk state s0 = 2 * node + side (0 = fw, 1 = bw) of the step table `st`
    (linear_steps, as lists): the nodes after the start node, in walk order.  A walk that never ends raises, as the
    library does (AMIRA_E_STATE)."""
    from amira_b200._lib import AmiraLibraryError
    n0, s, out = s0 >> 1, s0, []
    for _ in range(2 * len(st["degree"]) + 1):
        side = "bw" if s & 1 else "fw"
        ext, nx, d = st[side + "_ext"][s >> 1], st[side + "_next"][s >> 1], st[side + "_dir"][s >> 1]
        if not ext or nx == n0:
            if want_branched and nx >= 0:
                out.append(nx)
            return out
        out.append(nx)
        s = 2 * nx + (0 if d == 1 else 1)
    raise AmiraLibraryError("the walk from state %d never ends" % s0)


class WalkingDevice(OracleBackedDevice):
    """the test double with linear_walks: walk_loop from every state -> (offsets, nodes), as DeviceGraph.linear_walks"""

    def linear_walks(self, states, want_branched=False):
        masks = self._masks                   # the library's walks leave the filter masks alone
        st = {f: v.tolist() for f, v in self.linear_steps().items()}
        self._masks = masks
        states = np.asarray(states, np.int64).ravel()
        if len(states) and (states.min() < 0 or states.max() >= 2 * len(st["degree"])):
            raise ValueError("linear_walks: state out of range")
        off, out = [0], []
        for s0 in states.tolist():
            out.extend(walk_loop(st, s0, want_branched))
            off.append(len(out))
        return np.asarray(off, np.int64), np.asarray(out, np.int32)
