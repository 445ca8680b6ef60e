"""Token rows -> document ids, on the GPU (lstur_intern_rows / lstur_intern_table, csrc/intern.cu).

Cook's .npz files (task/cook.py:14-28) carry every history and candidate slot as its own title token row with a
vertical and a subvertical id, where the paper handlers' device paths address documents by id.  `intern` gives every
distinct (tokens, vertical, subvertical) key one id — 0 for the all-zero key, then 1, 2, ... in the order of first
occurrence — and builds the document table those ids index, so that the slots become the `hist_doc` / `cand_doc` id
arrays of lstur_forward and lstur_score_impressions.  Equal ids mean equal keys in every column: no hashing.
"""
import ctypes

import numpy as np
import torch

from . import _lib


def _ptr(t):
    return ctypes.c_void_p(None if t is None else t.data_ptr())


def _stream(device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _upload(a, device):
    """int32 on the device, converted as LsturEngine.to_device_batch converts host token arrays"""
    t = a if torch.is_tensor(a) else torch.from_numpy(np.ascontiguousarray(a))
    t = t.to(device)
    return (t if t.dtype == torch.int32 else t.to(torch.int32)).contiguous()


def intern(parts, L, device=None):
    """parts: list of (tokens (..., L), vert (...) or None, subvert (...) or None), host or device arrays; a part's leading
    dimensions are its slots.  The parts are interned together, in order, into ONE table; a column that is None in every
    part is not part of the key (and its table is None).
    -> (ids, table): ids = one int32 device tensor per part, shaped like its leading dimensions; table =
    dict(doc_tokens (n_unique, L), doc_vert (n_unique,) or None, doc_subvert (n_unique,) or None) int32 device tensors,
    with doc_tokens[ids] equal to the parts' token rows."""
    if not torch.cuda.is_available():
        raise _lib.LsturError('intern needs a CUDA device (no CPU fallback)')
    lib = _lib.load()
    dev = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
    shapes = [tuple(np.shape(tok))[:-1] for tok, _, _ in parts]
    for (tok, v, s), sh in zip(parts, shapes):
        assert np.shape(tok)[-1] == L, (np.shape(tok), L)
        assert v is None or tuple(np.shape(v)) == sh, (np.shape(v), sh)
        assert s is None or tuple(np.shape(s)) == sh, (np.shape(s), sh)
    counts = [int(np.prod(sh, dtype=np.int64)) for sh in shapes]
    n = int(sum(counts))
    assert n < 2 ** 31 - 1, 'more than 2^31 - 2 rows'
    has_v = any(v is not None for _, v, _ in parts)
    has_s = any(s is not None for _, _, s in parts)
    tokens = torch.zeros((n, L), dtype=torch.int32, device=dev)
    vert = torch.zeros(n, dtype=torch.int32, device=dev) if has_v else None
    subvert = torch.zeros(n, dtype=torch.int32, device=dev) if has_s else None
    r0 = 0
    for (tok, v, s), k in zip(parts, counts):       # each part uploaded into its rows; the raw uploads go when we return
        tokens[r0:r0 + k] = _upload(tok, dev).reshape(k, L)
        if v is not None:
            vert[r0:r0 + k] = _upload(v, dev).reshape(k)
        if s is not None:
            subvert[r0:r0 + k] = _upload(s, dev).reshape(k)
        r0 += k
    p, st = _ptr, _stream(dev)
    ids = torch.empty(n, dtype=torch.int32, device=dev)
    first_row = torch.empty(n + 1, dtype=torch.int32, device=dev)
    ws = torch.empty(int(lib.lstur_intern_workspace_bytes(n, L)), dtype=torch.uint8, device=dev)
    n_unique = ctypes.c_int()
    _lib.check(lib.lstur_intern_rows(n, L, p(tokens), p(vert), p(subvert), p(ids), p(first_row), ctypes.byref(n_unique),
                                     p(ws), ws.numel(), st))
    u = n_unique.value
    table = dict(doc_tokens=torch.empty((u, L), dtype=torch.int32, device=dev),
                 doc_vert=torch.empty(u, dtype=torch.int32, device=dev) if has_v else None,
                 doc_subvert=torch.empty(u, dtype=torch.int32, device=dev) if has_s else None)
    _lib.check(lib.lstur_intern_table(u, L, p(tokens), p(vert), p(subvert), p(first_row), p(table['doc_tokens']),
                                      p(table['doc_vert']), p(table['doc_subvert']), st))
    out, r0 = [], 0
    for sh, k in zip(shapes, counts):
        out.append(ids[r0:r0 + k].reshape(sh).clone())
        r0 += k
    return out, table


def group_rows(user, scale, hist_doc):
    """Consecutive rows with the same user, scale and history row (lstur_group_rows): user (n,) int32, scale (n,)
    float32 or None, hist_doc (n, W) int32 device tensors -> host int64 array of the first row of every group."""
    lib = _lib.load()
    n = int(user.numel())
    W = int(hist_doc.shape[1]) if hist_doc.dim() == 2 else 0
    dev = user.device
    starts = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    ws = torch.empty(int(lib.lstur_intern_workspace_bytes(n, 0)), dtype=torch.uint8, device=dev)
    n_groups = ctypes.c_int()
    p = _ptr
    _lib.check(lib.lstur_group_rows(n, W, p(user), p(scale), p(hist_doc), p(starts), ctypes.byref(n_groups), p(ws),
                                    ws.numel(), _stream(dev)))
    return starts[:n_groups.value].cpu().numpy().astype(np.int64)


def gather_samples(pos, m, src, out):
    """lstur_gather_samples: row b < m of each B-row device buffer in `out` <- sample pos[b] (int32 device tensor) of the
    same-named table in `src` (user, scale, hist_doc, cand_doc, label; 'user' and 'hist_doc' required, the others read
    only when `out` has them); rows b >= m (a ragged last batch) repeat pos[0] with an all-zero label row."""
    B, W = out['hist_doc'].shape
    C = out['cand_doc'].shape[1] if 'cand_doc' in out else 0
    names = ('user', 'scale', 'hist_doc', 'cand_doc', 'label')
    tables = [_ptr(src[k] if k in out else None) for k in names]
    bufs = [_ptr(out.get(k)) for k in names]
    _lib.check(_lib.load().lstur_gather_samples(B, m, W, C, _ptr(pos), *tables, *bufs, _stream(pos.device)))
