"""TEST INFRASTRUCTURE - storage of the fixtures under tests/golden/.

A fixture is one nested dict, written with torch.save.  One that would exceed MAX_BYTES is written as parts instead,
<name>.0.pt, <name>.1.pt, ..., each a list of (key path, value) leaves in the dict's order; load() puts the dict back
together, so a test sees the same keys, order and values either way.
"""
import glob
import io
import os

import torch

GOLD = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
MAX_BYTES = 1_000_000
_PART_BUDGET = 900_000          # serialised leaves per part; the rest of MAX_BYTES covers the part file's own overhead


def _serialised_size(obj):
    buf = io.BytesIO()
    torch.save(obj, buf)
    return buf.tell()


def _leaves(obj, path=()):
    if isinstance(obj, dict) and obj:
        for k, v in obj.items():
            yield from _leaves(v, path + (k,))
    else:
        yield path, obj


def _paths(name, root):
    single = os.path.join(root, name + ".pt")
    parts = sorted(glob.glob(os.path.join(root, glob.escape(name) + ".[0-9]*.pt")),
                   key=lambda p: int(p[:-len(".pt")].rsplit(".", 1)[1]))
    return single, parts


def save(name, obj, root=GOLD):
    """writes `obj` as <root>/<name>.pt, or in parts when it is larger than MAX_BYTES; returns the paths written"""
    os.makedirs(root, exist_ok=True)
    single, parts = _paths(name, root)
    for p in [single] + parts:
        if os.path.exists(p):
            os.remove(p)
    if _serialised_size(obj) <= MAX_BYTES:
        torch.save(obj, single)
        return [single]
    groups, cur, cur_bytes = [], [], 0
    for leaf in _leaves(obj):
        n = _serialised_size([leaf])
        if n > _PART_BUDGET:
            raise ValueError("%s: the entry %s alone is %d bytes" % (name, "/".join(map(str, leaf[0])), n))
        if cur and cur_bytes + n > _PART_BUDGET:
            groups.append(cur)
            cur, cur_bytes = [], 0
        cur.append(leaf)
        cur_bytes += n
    groups.append(cur)
    written = []
    for i, group in enumerate(groups):
        path = os.path.join(root, "%s.%d.pt" % (name, i))
        torch.save(group, path)
        assert os.path.getsize(path) <= MAX_BYTES, path
        written.append(path)
    return written


def load(name, root=GOLD):
    """the dict save() was given"""
    single, parts = _paths(name, root)
    if os.path.exists(single):
        return torch.load(single, weights_only=False)
    if not parts:
        raise FileNotFoundError("no fixture %r under %s" % (name, root))
    out = {}
    for path in parts:
        for keys, value in torch.load(path, weights_only=False):
            node = out
            for k in keys[:-1]:
                node = node.setdefault(k, {})
            node[keys[-1]] = value
    return out
