"""Bit-identity A/B of the PairSynthesizer entry points on the seeded inputs of tests/test_gpu_pipeline_calls.py.

    python profiles/pipetail/ab_results.py dump ROOT OUT.pt    every scenario with the package of the tree at ROOT:
                                                              each result's fields and the hsr_* calls it made
    python profiles/pipetail/ab_results.py compare A.pt B.pt   tensor fields bit for bit (torch.equal on the bits),
                                                              the other fields by value, and the call sequences
"""
import dataclasses
import os
import sys

import torch

TESTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "..", "tests")


def _bits(t):
    return t.view({torch.float32: torch.int32, torch.float64: torch.int64}.get(t.dtype, t.dtype))


def _fields(res):
    out = {}
    for i, r in enumerate(res if isinstance(res, list) else [res]):
        for f in dataclasses.fields(r):
            v = getattr(r, f.name)
            if isinstance(v, torch.Tensor):
                out[f"{i}.{f.name}"] = v.detach().cpu().clone()
            elif f.name != "grid":                       # an S2Target object: the inputs' own
                out[f"{i}.{f.name}"] = repr(v)
    return out


def dump(root, path):
    sys.path[:0] = [os.path.abspath(root), TESTS]
    import test_gpu_pipeline_calls as t

    out = {}
    for name in sorted(t.SCENARIOS):
        res, calls = t.run_recorded(name)
        out[name] = {"calls": calls, "fields": _fields(res)}
    torch.save(out, path)
    print(f"{len(out)} scenarios -> {os.path.basename(path)}")


def compare(a_path, b_path):
    a, b = torch.load(a_path), torch.load(b_path)
    bad = 0
    for name in sorted(set(a) | set(b)):
        if name not in a or name not in b:
            print(f"{name}: only in one dump")
            bad += 1
            continue
        fa, fb = a[name]["fields"], b[name]["fields"]
        diff = sorted(k for k in set(fa) | set(fb) if k not in fa or k not in fb or not (
            torch.equal(_bits(fa[k]), _bits(fb[k])) if isinstance(fa[k], torch.Tensor) else fa[k] == fb[k]))
        n_t = sum(isinstance(v, torch.Tensor) for v in fa.values())
        same_calls = a[name]["calls"] == b[name]["calls"]
        print(f"{name}: {n_t} tensor fields, {len(fa) - n_t} other; differing: {diff or 'none'}; "
              f"calls {'same' if same_calls else 'DIFFER'} ({len(a[name]['calls'].split())} / "
              f"{len(b[name]['calls'].split())})")
        if not same_calls:
            print(f"  A: {a[name]['calls']}\n  B: {b[name]['calls']}")
        bad += bool(diff)
    print(f"scenarios with differing fields: {bad}")
    return bad


if __name__ == "__main__":
    if sys.argv[1] == "dump":
        dump(sys.argv[2], sys.argv[3])
    else:
        sys.exit(1 if compare(sys.argv[2], sys.argv[3]) else 0)
