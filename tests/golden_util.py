"""Helpers shared by the parity tests: load the reference's recorded outputs."""
import os

import numpy as np
import torch

import cases  # tests/golden/cases.py (on sys.path via conftest)

_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference_outputs.npz')
_BLOB = None


def blob():
    global _BLOB
    if _BLOB is None:
        _BLOB = dict(np.load(_PATH))
    return _BLOB


def ref(case, key, prec='f32'):
    return torch.from_numpy(blob()[f'{case}|{key}|{prec}'])


def has(case, key, prec='f32'):
    return f'{case}|{key}|{prec}' in blob()


def rows(case, key):
    """Indices of the rows recorded for (case, key) when a large output is stored as a fixed sample of its rows
    (make_golden.sample_large), else None."""
    return torch.from_numpy(blob()[f'{case}|{key}|rows']) if has(case, key, 'rows') else None


def pick(case, key, got):
    """`got` restricted to the rows recorded for (case, key)"""
    r = rows(case, key)
    return got if r is None else got[r.to(got.device)]


def case_names(prefixes=None, ops=None):
    out = []
    for n in cases.CASES:
        if prefixes is not None and not any(n.startswith(p) for p in prefixes):
            continue
        out.append(n)
    return out


def close_or_arbitrated(new, ref32, ref64, rtol=1e-5, atol=1e-5):
    """Row passes if |new-ref32| <= atol+rtol|ref| OR |new-ref64| <= |ref32-ref64| + atol+rtol|ref|
    (SURVEY.md section 8c).  Returns (fraction_failing, fraction_using_second_clause, max_abs_err)."""
    new = new.detach().cpu().double()
    r32 = ref32.double()
    r64 = ref64.double()
    tol = atol + rtol * r64.abs()
    c1 = (new - r32).abs() <= tol
    c2 = (new - r64).abs() <= (r32 - r64).abs() + tol
    ok = c1 | c2
    return (1.0 - ok.double().mean().item(), ((~c1) & c2).double().mean().item(),
            (new - r32).abs().max().item() if new.numel() else 0.0)
