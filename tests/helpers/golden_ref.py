"""Stored reference-side values for the drop-in comparisons of tests/test_reference_dropin.py.

Each tests/helpers/reference_*.py compares the product or the oracle with the original instant-nsr-pl code.  Every value it takes from
the original code goes through ``Tape.ref(key, fn)``:

    python tests/helpers/reference_forward.py --record /path/to/instant-nsr-pl   # runs the original code, writes tests/golden/<name>.npz
    python tests/helpers/reference_forward.py                                     # reads the stored values back (how the tests run)

so the comparison needs nothing outside the repository.  Tensors of more than SMALL entries are stored as a fixed sample: UNIFORM
positions drawn from a generator seeded with the tensor's size (not stored) plus the TOP largest magnitudes (the non-zeros of a sparse
gradient), with shape, dtype and the largest magnitude; ``pick`` compares a full tensor with such a sample at those positions."""
import json
import os
import sys

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'golden')
SMALL = 128
UNIFORM, TOP = 64, 16


class Sample:
    def __init__(self, shape, dtype, idx, values, absmax):
        self.shape, self.dtype, self.idx, self.values, self.absmax = tuple(shape), dtype, idx, values, absmax


def is_array(v):
    return torch.is_tensor(v) or isinstance(v, Sample)


def pick(ours, ref):
    """(ours, ref) as flat tensors of equal length: the whole tensors, or ours at the positions of the stored sample"""
    ours = torch.as_tensor(ours).detach()
    if isinstance(ref, Sample):
        assert tuple(ours.shape) == ref.shape or ours.numel() == int(np.prod(ref.shape)), (tuple(ours.shape), ref.shape)
        return ours.reshape(-1)[ref.idx], ref.values
    return ours.reshape(-1), torch.as_tensor(ref).detach().reshape(-1)


def amax(t):
    return t.absmax if isinstance(t, Sample) else float(torch.as_tensor(t).detach().abs().max())


def _positions(n, top):
    return torch.cat([torch.randint(0, n, (UNIFORM,), generator=torch.Generator().manual_seed(n)), top])


_DTYPES = {str(d): d for d in (torch.float16, torch.bfloat16, torch.float32, torch.float64, torch.int8, torch.int16, torch.int32,
                               torch.int64, torch.uint8, torch.bool)}


class Tape:
    def __init__(self, name):
        self.path = os.path.join(GOLDEN, f'{name}.npz')
        self.recording = '--record' in sys.argv
        self.reference = sys.argv[sys.argv.index('--record') + 1] if self.recording else None
        self.arrays, self.index = {}, {}
        if not self.recording:   # one JSON index + every array's bytes in one blob (one zip member instead of hundreds)
            with np.load(self.path) as z:
                self.index, layout, blob = json.loads(str(z['index'])), json.loads(str(z['layout'])), z['blob'].tobytes()
            self.arrays = {k: np.frombuffer(blob, dtype=dt, count=int(np.prod(shape)), offset=off).reshape(shape)
                           for k, (off, dt, shape) in layout.items()}

    def ref(self, key, fn, whole=False):
        """fn() when recording (the value is stored under ``key``; ``whole``: tensors are stored whole, not sampled), else the stored value"""
        if self.recording:
            assert key not in self.index, key
            v = fn()
            self.index[key] = self._encode(v, key, whole)
            return self._decode(self.index[key])
        return self._decode(self.index[key])

    def check_state(self, module, key):
        """asserts that ``module`` (built from seeds; its weights are loaded into the original model when recording) holds the state it
        held when the values were recorded: both sides of a comparison start from the same weights"""
        sd = self.ref(key, lambda: {k: v.detach().clone() for k, v in module.state_dict().items()})
        own = module.state_dict()
        assert sorted(own) == sorted(sd), sorted(set(own) ^ set(sd))
        for k, v in sd.items():
            a, b = pick(own[k], v)
            assert torch.equal(a, b.to(a.dtype)), f'{key}: {k} differs from the recorded state'

    def save(self):
        assert self.recording
        layout, parts, off = {}, [], 0
        for k, a in self.arrays.items():
            a = np.ascontiguousarray(a)
            layout[k] = (off, a.dtype.str, list(a.shape))
            parts.append(a.tobytes())
            off += len(parts[-1])
        np.savez_compressed(self.path, index=np.array(json.dumps(self.index)), layout=np.array(json.dumps(layout)),
                            blob=np.frombuffer(b''.join(parts), dtype=np.uint8))
        print(f'wrote {self.path}: {len(self.arrays)} arrays, {os.path.getsize(self.path)} bytes', file=sys.stderr)

    # ---- (de)serialisation of tensors, arrays, scalars, strings, None, lists / tuples and dicts of them
    def _encode(self, v, path, whole=False):
        if torch.is_tensor(v) or isinstance(v, np.ndarray):
            t = torch.as_tensor(v).detach().cpu()
            if whole or t.numel() <= SMALL:
                self.arrays[path] = t.numpy()
                return {'t': path, 'dtype': str(t.dtype)}
            flat = t.reshape(-1)
            mag = flat.double().abs()
            top = torch.topk(mag, TOP).indices
            self.arrays[path + '#top'] = top.numpy().astype(np.int32)
            self.arrays[path] = flat[_positions(t.numel(), top)].numpy()
            return {'s': path, 'shape': list(t.shape), 'dtype': str(t.dtype), 'absmax': float(mag.max())}
        if isinstance(v, dict):
            return {'d': {str(k): self._encode(x, f'{path}/{k}', whole) for k, x in v.items()}}
        if isinstance(v, (list, tuple)):
            return {'l': [self._encode(x, f'{path}/{i}', whole) for i, x in enumerate(v)], 'tuple': isinstance(v, tuple)}
        if isinstance(v, (np.floating, np.integer, np.bool_)):
            v = v.item()
        assert v is None or isinstance(v, (bool, int, float, str)), (path, type(v))
        return {'v': v}

    def _decode(self, e):
        if 't' in e:
            return torch.from_numpy(np.array(self.arrays[e['t']])).to(_DTYPES[e['dtype']])
        if 's' in e:
            idx = _positions(int(np.prod(e['shape'])), torch.from_numpy(self.arrays[e['s'] + '#top']).long())
            return Sample(e['shape'], _DTYPES[e['dtype']], idx,
                          torch.from_numpy(np.array(self.arrays[e['s']])).to(_DTYPES[e['dtype']]), e['absmax'])
        if 'd' in e:
            return {k: self._decode(x) for k, x in e['d'].items()}
        if 'l' in e:
            items = [self._decode(x) for x in e['l']]
            return tuple(items) if e['tuple'] else items
        return e['v']
