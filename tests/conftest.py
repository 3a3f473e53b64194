import os
import sys
import zlib

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (a B200)")


def pytest_collection_modifyitems(config, items):
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def load_golden(name):
    """tests/golden/<name>.npz -> dict of torch tensors (fixtures written by oracle/make_golden.py)."""
    with np.load(os.path.join(GOLDEN, name + ".npz")) as data:
        return {k: torch.from_numpy(data[k]) for k in data.files}


# GG_RECORD_GOLDEN=1 (with the original project importable, and its kernels built into oracle/_ref/ for the GPU tests)
# recomputes what the tests pinned with Pinned compare against and rewrites their tests/golden/ files
RECORD = os.environ.get("GG_RECORD_GOLDEN") == "1"


class Pinned:
    """Values of the original project that a test compares against, stored in tests/golden/<name>.npz.

    pin(key, got, reference) -> (got, want), both flattened to the elements kept for `key`: all of them up to KEEP, else a
    seeded sample of KEEP plus the reference's largest-magnitude element (so that a tolerance relative to the kept `want`'s
    magnitude is relative to the whole tensor's).  The shape of `got` must be the reference's.  With a tuple `got`,
    `reference` returns a tuple of as many tensors and the result is a list of pairs; `keep` overrides KEEP.  pin.value(key, reference) keeps a
    small array (scalars, key lists) whole.  `reference` computes the value with the original project; it runs only when
    recording, and save() then writes the file."""
    KEEP = 64

    def __init__(self, name):
        self.path = os.path.join(GOLDEN, name + ".npz")
        self.data = {}
        if not RECORD:
            with np.load(self.path) as blob:
                self.data = {k: blob[k] for k in blob.files if not k.startswith("pinned.")}
                offset = 0
                for entry in blob["pinned.index"]:    # "<key>|<top>|<d0>,<d1>,...|<count>": one per pinned tensor
                    key, top, dims, count = str(entry).split("|")
                    self.data[key + ".top"] = int(top)
                    self.data[key + ".shape"] = [int(d) for d in dims.split(",") if d]
                    self.data[key] = blob["pinned.values"][offset:offset + int(count)]
                    offset += int(count)

    def value(self, key, reference):
        if RECORD:
            self.data[key] = np.asarray(reference())
        return self.data[key]

    def __call__(self, key, got, reference, keep=None):
        many = isinstance(got, (tuple, list))
        gots = list(got) if many else [got]
        wants = [None] * len(gots)
        if RECORD:
            wants = list(reference()) if many else [reference()]
            assert len(wants) == len(gots), key
        keep = self.KEEP if keep is None else keep
        pairs = [self._one("%s.%d" % (key, i) if many else key, g, w, keep) for i, (g, w) in enumerate(zip(gots, wants))]
        return pairs if many else pairs[0]

    def _one(self, key, got, want, keep):
        if want is not None:
            want = want.detach().cpu() if torch.is_tensor(want) else torch.as_tensor(np.asarray(want))
            self.data[key + ".shape"] = np.array(want.shape, dtype=np.int64)
            want = want.reshape(-1)
            self.data[key + ".top"] = np.array(int(want.abs().nan_to_num(0.0).argmax()) if want.numel() else 0, dtype=np.int64)
        shape = tuple(int(s) for s in self.data[key + ".shape"])
        assert tuple(got.shape) == shape, "%s: shape %s vs %s" % (key, tuple(got.shape), shape)
        numel = int(np.prod(shape))
        idx = None
        if numel > keep:
            g = torch.Generator().manual_seed(zlib.crc32(key.encode()))
            idx = torch.cat([torch.randint(numel, (keep,), generator=g), torch.tensor([int(self.data[key + ".top"])])]).unique()
        if want is not None:
            self.data[key] = (want if idx is None else want[idx]).numpy()
        got = got.detach().cpu().reshape(-1)
        return (got if idx is None else got[idx]), torch.from_numpy(self.data[key])

    def save(self):
        """Packed: the pinned tensors' kept elements in one float32 array, one index string each (few, small zip members)."""
        if not RECORD:
            return
        pinned = [k for k in self.data if k + ".shape" in self.data]
        rest = {k: v for k, v in self.data.items() if k not in pinned and not k.endswith((".shape", ".top"))}
        index = ["%s|%d|%s|%d" % (k, self.data[k + ".top"], ",".join(str(d) for d in self.data[k + ".shape"]), self.data[k].size)
                 for k in pinned]
        values = np.concatenate([self.data[k].astype(np.float32).reshape(-1) for k in pinned]) if pinned else np.zeros(0, np.float32)
        np.savez_compressed(self.path, **rest, **{"pinned.index": np.array(index), "pinned.values": values})


def state_dict_layout(module):
    """["<key>:<d0>,<d1>,...", ...]: the keys and shapes of a module's state dict (what load_state_dict checks)."""
    return ["%s:%s" % (k, ",".join(str(d) for d in v.shape)) for k, v in module.state_dict().items()]


def zeros_state_dict(layout):
    """A state dict of zeros laid out as `layout` (state_dict_layout's strings)."""
    entries = (str(e).rsplit(":", 1) for e in layout)
    return {k: torch.zeros([int(d) for d in dims.split(",") if d]) for k, dims in entries}


def golden_cases(blob):
    names = []
    for k in blob:
        n = k.rsplit(".", 1)[0]
        if n not in names:
            names.append(n)
    return names


def assert_close(actual, expected, rtol=1e-3, atol=None, what=""):
    """The north-star tolerance: 1e-3 relative (to the tensor's magnitude) in fp32."""
    actual = actual.detach().float().cpu()
    expected = expected.detach().float().cpu()
    assert actual.shape == expected.shape, "%s: shape %s vs %s" % (what, tuple(actual.shape), tuple(expected.shape))
    scale = expected.abs().max().item()
    tol = rtol * max(scale, 1e-6) if atol is None else atol
    err = (actual - expected).abs().max().item() if actual.numel() else 0.0
    assert err <= tol, "%s: max abs err %.3e > %.3e (ref magnitude %.3e)" % (what, err, tol, scale)
