"""Loader for the UNMODIFIED reference -- test infrastructure.

Imports ``ofighters.lib.battleground`` & friends from the original Ofighters
source tree named by the environment variable OFB_REFERENCE_ROOT after
injecting ``sys.modules`` shims for the third-party packages that are absent
here (matplotlib, keras, tensorflow, tkinter, pandas = mocks; skimage.draw.disk
= the restatement in oracle/disk.py).  Nothing of the reference is copied or
edited; see SURVEY.md Appendix C.

The reference is not part of this repository: only ``oracle/gen_golden.py``
and the tests marked ``reference`` (skipped when OFB_REFERENCE_ROOT is unset)
use this.
"""
import contextlib
import io
import os
import sys
import types
from unittest.mock import MagicMock

REFERENCE_ROOT = os.environ.get("OFB_REFERENCE_ROOT", "")

_MOCKED = [
    "matplotlib", "matplotlib.pyplot", "matplotlib.cm", "matplotlib.figure",
    "matplotlib.backends", "matplotlib.backends.backend_tkagg", "matplotlib.animation",
    "tensorflow", "keras", "keras.models", "keras.layers", "keras.layers.core",
    "keras.optimizers", "keras.layers.advanced_activations", "keras.backend",
    "tkinter", "tkinter.ttk", "tkinter.filedialog", "tkinter.messagebox", "pandas",
]

_loaded = None


def available():
    return bool(REFERENCE_ROOT) and os.path.isdir(os.path.join(REFERENCE_ROOT, "ofighters", "lib"))


def load():
    """Return a namespace with the reference's hot-path classes."""
    global _loaded
    if _loaded is not None:
        return _loaded
    if not available():
        raise RuntimeError("reference tree not present: set OFB_REFERENCE_ROOT to the original Ofighters source tree")
    from oracle.disk import disk
    for m in _MOCKED:
        if m not in sys.modules:
            sys.modules[m] = MagicMock(name=m)
    if "skimage" not in sys.modules:
        skd = types.ModuleType("skimage.draw")
        skd.disk = disk
        sk = types.ModuleType("skimage")
        sk.draw = skd
        sys.modules["skimage"] = sk
        sys.modules["skimage.draw"] = skd
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    with contextlib.redirect_stdout(io.StringIO()):
        from ofighters.lib import battleground as m_bg
        from ofighters.lib import ship as m_ship
        from ofighters.lib import laser as m_laser
        from ofighters.lib import observation as m_obs
        from ofighters.lib import action as m_action
        from ofighters.lib import couple as m_couple
        from ofighters.lib import form as m_form
        from ofighters.agents import agent as m_agent
    ns = types.SimpleNamespace(
        battleground=m_bg, ship=m_ship, laser=m_laser, observation=m_obs,
        action=m_action, couple=m_couple, form=m_form, agent=m_agent,
        Battleground=m_bg.Battleground, Ship=m_ship.Ship, Laser=m_laser.Laser,
        Observation=m_obs.Observation, Action=m_action.Action,
        Point=m_couple.Point, Couple=m_couple.Couple, Circle=m_form.Circle,
        Agent=m_agent.Agent,
    )
    _loaded = ns
    return ns


class ScriptedBot:
    """``bot.play(obs) -> Action`` object replaying a pre-generated action tape.

    Plugged in through the reference's own bot seam ``Agent(behavior, bot=...)``
    (agents/agent.py:19-37).  ``tape[t] = (shoot, thrust, px, py)``.  When
    ``as_vector`` is set the Action is built from a float (4,1) vector exactly
    like ``QlearnIA.play`` does (agents/qlearnIA_V2.py:447-454), which makes
    the pointing coordinates ``np.float64``.
    Records the 8-value head of every observation it is shown plus ``obs.done``.
    """

    def __init__(self, ref, tape, as_vector=False):
        self.ref = ref
        self.tape = tape
        self.t = 0
        self.as_vector = as_vector
        self.seen = []

    def play(self, obs):
        import numpy as np
        self.seen.append((np.asarray(obs.vector[:8, 0], dtype=np.float64).copy(), bool(obs.done)))
        s, th, px, py = (int(v) for v in self.tape[self.t])
        self.t += 1
        if self.as_vector:
            v = np.zeros((4, 1))
            v[0] = s
            v[1] = th
            v[2] = px
            v[3] = py
            return self.ref.Action(vector=v)
        return self.ref.Action(shoot=bool(s), thrust=bool(th), pointing=self.ref.Point(px, py))


class ReferenceArena:
    """One reference ``Battleground`` driven by scripted actions and injected spawns.

    Mirrors what the Tk controller does around it (lib/ofighters.py:656-707):
    destroyed lasers are pruned before the next frame; after ``max_time``
    frames ``restart()`` is called instead of ``frame()``.
    """

    def __init__(self, n_ships, spawn_xy, tapes, vector_ships=(), width=400, height=400):
        ref = load()
        self.ref = ref
        with contextlib.redirect_stdout(io.StringIO()):
            bg = ref.Battleground(ships={"idle": n_ships}, largeur=width, hauteur=height)
        self.bg = bg
        self.bots = []
        for i, ship in enumerate(bg.ships):
            x, y = int(spawn_xy[i][0]), int(spawn_xy[i][1])
            ship.body.x, ship.body.y = x, y
            ship.pointing = ref.Point(x, y)
            bot = ScriptedBot(ref, tapes[i], as_vector=(i in vector_ships))
            ship.agent = ref.Agent("scripted", bot=bot)
            self.bots.append(bot)
        with contextlib.redirect_stdout(io.StringIO()):
            bg.absolute_state = ref.Observation(battleground=bg)

    def prune(self):
        self.bg.lasers = [l for l in self.bg.lasers if l.state != "destroyed"]

    def frame(self):
        with contextlib.redirect_stdout(io.StringIO()):
            self.prune()
            self.bg.frame()

    def restart(self, spawn_xy):
        """``Battleground.restart`` with its ``randint`` draws replaced by ``spawn_xy``."""
        vals = []
        for x, y in spawn_xy:
            vals += [int(x), int(y)]
        it = iter(vals)
        m_bg = self.ref.battleground
        saved = m_bg.randint
        m_bg.randint = lambda a, b: next(it)
        try:
            with contextlib.redirect_stdout(io.StringIO()):
                self.bg.restart()
        finally:
            m_bg.randint = saved
