"""Seed / call-counter bookkeeping for the fused Philox noise.

Every fused forward consumes one ``offset`` (the Philox call counter); the backward
of that call regenerates the same noise from the saved (seed, offset).  This plays
the role torch's global CUDA generator plays for the reference
(``expand([E,K]).rsample()``, stag/layers.py:117-127):

* the state is PROCESS-GLOBAL (one stream for all threads, like torch's default generator);
* by default the seed follows torch's: it is ``torch.initial_seed()`` (non-deterministic unless
  ``torch.manual_seed`` was called), and a later ``torch.manual_seed(k)`` restarts the stream at
  (k, 0) -- so ``torch.manual_seed`` makes a run reproducible, as it does for the reference;
* ``manual_seed(seed)`` sets the seed explicitly; ``fold_rank(rank)`` derives a per-rank stream
  from the current seed (data-parallel ranks working on DIFFERENT minibatches; ranks sharding
  the Monte-Carlo samples of ONE forward keep a common seed and differ in ``sample_base``);
* ``get_state()`` / ``set_state()`` return / restore (seed, offset) for checkpoint / resume (the
  state is deliberately not part of ``state_dict``: the reference's keys are kept, SURVEY 8(b));
* CUDA graphs: a captured step bakes its host-side offsets into the kernel parameters, so every replay would redraw
  the SAME noise.  ``enable_device_counter(device)`` adds a device-side word to the call counter of every launch
  (``StagNoise::counter``); ``advance_device_counter()`` -- called at the end of the step, inside the capture --
  bumps it by the number of offsets the step reserved, so replay i draws what the i-th eager step would have drawn.
"""
import threading

import torch

_lock = threading.Lock()
_state = {"seed": None, "offset": 0, "torch_seed": None, "explicit": False}
_MASK = 0xFFFFFFFFFFFFFFFF
_dev_counters = {}            # device -> int32 tensor [1] (the kernels read it as uint32)
_dev_mark = {"offset": 0}     # host offset at the last advance_device_counter()


def _sync_with_torch():
    """Called with the lock held: adopt torch's seed at first use and whenever torch is re-seeded."""
    ts = int(torch.initial_seed()) & _MASK
    if _state["seed"] is None or ts != _state["torch_seed"]:
        _state["seed"], _state["offset"], _state["explicit"] = ts, 0, False
        _dev_mark["offset"] = 0
    _state["torch_seed"] = ts


def manual_seed(seed):
    with _lock:
        _state["seed"] = int(seed) & _MASK
        _state["offset"] = 0
        _dev_mark["offset"] = 0
        _state["explicit"] = True
        _state["torch_seed"] = int(torch.initial_seed()) & _MASK


def fold_rank(rank):
    """Derive this rank's stream from the current seed (splitmix-style odd multiplier)."""
    with _lock:
        _sync_with_torch()
        _state["seed"] = (_state["seed"] ^ ((int(rank) + 1) * 0x9E3779B97F4A7C15)) & _MASK
        _state["offset"] = 0
        _dev_mark["offset"] = 0
        _state["explicit"] = True


def get_state():
    with _lock:
        _sync_with_torch()
        return _state["seed"], _state["offset"]


def set_state(seed, offset):
    with _lock:
        _state["seed"], _state["offset"] = int(seed) & _MASK, int(offset)
        _dev_mark["offset"] = int(offset)
        _state["explicit"] = True
        _state["torch_seed"] = int(torch.initial_seed()) & _MASK


def _rewind(seed, offset):
    """Return the stream to a (seed, offset) that ``get_state()`` gave, without moving the device-counter mark as
    ``set_state`` does: code that replays its own draws (the chunks of ``StagModel.predictive``) stays transparent to
    ``advance_device_counter``."""
    with _lock:
        _state["seed"], _state["offset"] = int(seed) & _MASK, int(offset)


def enable_device_counter(device):
    """Create (or return) the device-side call counter of `device`; from now on every launch on that device adds it
    to its Philox counter.  Starts at 0."""
    device = torch.device(device)
    if device.type == "cuda" and device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    with _lock:
        if device not in _dev_counters:
            _dev_counters[device] = torch.zeros(1, dtype=torch.int32, device=device)
            _sync_with_torch()
            _dev_mark["offset"] = _state["offset"]
        return _dev_counters[device]


def disable_device_counter(device=None):
    with _lock:
        if device is None:
            _dev_counters.clear()
        else:
            _dev_counters.pop(torch.device(device), None)


def device_counter(device):
    """The counter tensor of `device`, or None when ``enable_device_counter`` was not called for it."""
    if not _dev_counters or device is None:
        return None
    device = torch.device(device)
    if device.type == "cuda" and device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    return _dev_counters.get(device)


def advance_device_counter():
    """Add the number of offsets reserved since the last call (or since ``enable_device_counter``) to every device
    counter -- a torch op on the current stream, so inside a CUDA-graph capture it becomes part of the graph -- and
    rewind the host-side offset by the same amount: replays and eager steps then draw identical streams."""
    with _lock:
        n = _state["offset"] - _dev_mark["offset"]
        _state["offset"] = _dev_mark["offset"]
    for t in _dev_counters.values():
        t.add_(int(n))
    return n


def next_offset():
    """Reserve one Philox call counter and return (seed, offset)."""
    with _lock:
        _sync_with_torch()
        off = _state["offset"]
        _state["offset"] = off + 1
        return _state["seed"], off
