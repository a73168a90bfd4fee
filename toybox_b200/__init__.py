"""toybox_b200: a B200-native batched simulator for the hot path of toybox-rs/Toybox -- the per-frame
step/transition and frame render of Breakout, Amidar and Space Invaders that the reference drives one
environment at a time through `ctoybox`.  See DESIGN.md / INTEGRATION.md.

    from toybox_b200 import BatchedToybox          # N envs on one GPU
    from toybox_b200.ctoybox import Toybox, Input  # the reference's ctoybox surface at batch size 1
"""
from ._lib import ToyboxError, build, lib  # noqa: F401
from .pool import BatchedToybox, GAMES, schema_for_config, schema_for_state  # noqa: F401
from .snapshot import StateSnapshot  # noqa: F401

__all__ = ["BatchedToybox", "GAMES", "ToyboxError", "build", "lib", "schema_for_state", "schema_for_config", "StateSnapshot"]
