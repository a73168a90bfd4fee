"""Device-resident state snapshots (include/toybox_b200.h, tbx_state_save / tbx_state_load; DESIGN.md 4.7): the saved state of
k envs as one int32[rows, k] device tensor plus the geometry tables its records refer to.  Saving, restoring and forking envs
this way never leaves the GPU; JSON (to_state_json / write_state_json) stays the validated, editable form."""
import ctypes as C
import struct

import numpy as np
import torch

from . import _lib

_GAME_NAMES = ("breakout", "amidar", "space_invaders")   # the game field of the tables blob header
_HEADER = struct.Struct("<6I")                            # tbx_state_blob_header
TBL_WORD = 14                                             # TbxHdr.tbl: the record word that indexes the tables (tbx_records.h)


class StateSnapshot:
    """The state of k envs: `data` int32[rows, k] (column j = one env's record, plus its wrapper words when `wrapped`: 5, or 7
    with sticky actions), `tables` the blob of geometry tables the records index, and for a wrapped env `obs`
    uint8[k, stack, out_h, out_w], the
    envs' observation rings, whose newest frame is in ring slot `slot`.  `game`, `rows`, `format` and `table_count` come from
    the blob's header.  Picklable (torch.save / torch.load); `.to(device)` moves it to another GPU."""

    def __init__(self, data, tables, wrapped=False, obs=None, slot=0):
        tables = bytes(tables)
        if len(tables) < _HEADER.size:
            raise ValueError("state snapshot: the tables blob is truncated")
        magic, fmt, game, rows, _, count = _HEADER.unpack_from(tables)
        if magic != 0x53584254 or game >= len(_GAME_NAMES):
            raise ValueError("state snapshot: not a tables blob")
        if data.dtype != torch.int32 or data.dim() != 2 or data.shape[0] != rows:
            raise ValueError("state snapshot: data must be int32[%d, k]" % rows)
        if bool(wrapped) != (obs is not None) or (obs is not None and obs.shape[0] != data.shape[1]):
            raise ValueError("state snapshot: a wrapped snapshot carries one observation ring per env")
        self.data, self.tables, self.wrapped, self.obs, self.slot = data, tables, bool(wrapped), obs, int(slot)
        self.game, self.rows, self.format, self.table_count = _GAME_NAMES[game], rows, fmt, count

    @property
    def k(self):
        return self.data.shape[1]

    @property
    def device(self):
        return self.data.device

    def to(self, device):
        return StateSnapshot(self.data.to(device), self.tables, self.wrapped, None if self.obs is None else self.obs.to(device), self.slot)

    def __repr__(self):
        return "StateSnapshot(%s, k=%d, rows=%d, format=%d%s, %s)" % (self.game, self.k, self.rows, self.format,
                                                                     ", wrapped" if self.wrapped else "", self.device)


if hasattr(torch.serialization, "add_safe_globals"):     # torch.load(weights_only=True), the default, may rebuild snapshots
    torch.serialization.add_safe_globals([StateSnapshot])


def tables_blob(fn, handle):
    """tbx_state_tables / tbx_wrap_state_tables as bytes"""
    size = C.c_size_t()
    _lib.check(fn(handle, None, 0, C.byref(size)))
    buf = C.create_string_buffer(size.value)
    _lib.check(fn(handle, buf, size.value, C.byref(size)))
    return buf.raw


def id_tensor(ids, limit, device, what):
    """None, or `ids` as a contiguous int32 tensor on `device`.  Host sequences are range-checked here (IndexError); device
    tensors keep their values and are checked by the kernel (skipped entries are reported by check())."""
    if ids is None:
        return None
    if torch.is_tensor(ids) and ids.is_cuda:
        return ids.reshape(-1).to(device=device, dtype=torch.int32).contiguous()
    a = np.asarray(ids.cpu() if torch.is_tensor(ids) else ids, dtype=np.int64).reshape(-1)
    if a.size and (a.min() < 0 or a.max() >= limit):
        raise IndexError("%s out of range 0..%d" % (what, limit - 1))
    return torch.as_tensor(a.astype(np.int32), device=device)


def load_args(snap, device, n_envs, env_ids, columns):
    """(data on `device`, env id tensor or None, column tensor or None, entry count) of a load"""
    if not isinstance(snap, StateSnapshot):
        raise TypeError("expected a StateSnapshot")
    data = snap.data if snap.data.device == device else snap.data.to(device)
    ids = id_tensor(env_ids, n_envs, device, "env id")
    cols = id_tensor(columns, snap.k, device, "column")
    if ids is not None and cols is not None and ids.numel() != cols.numel():
        raise ValueError("env_ids and columns must have the same length")
    n = ids.numel() if ids is not None else cols.numel() if cols is not None else snap.k
    if ids is None and n > n_envs:
        raise ValueError("%d entries for %d envs: pass env_ids" % (n, n_envs))
    if cols is None and n > snap.k:
        raise ValueError("%d entries for a snapshot of %d envs: pass columns" % (n, snap.k))
    return data.contiguous(), ids, cols, n


def fork_columns(k, n, device):
    """columns of a fork of k saved sources into n destinations: pairwise, or one source into every destination"""
    if k == n:
        return None
    if k == 1:
        return torch.zeros(n, dtype=torch.int32, device=device)
    raise ValueError("fork: %d sources for %d destinations (give one source, or one per destination)" % (k, n))
