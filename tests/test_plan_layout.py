"""Plan layout over a matrix of configurations (every user-encoder arch x precision x training / inference x scorer, and
the optional parts on top): every workspace region lies inside the workspace, 256-byte aligned and disjoint from the
others; every dense tensor lies inside the arena, disjoint from the others, and the title-encoder bucket ends the
arena's head; an unknown name is an error.  Plan creation is host-only: no GPU needed."""
import ctypes
import itertools
import os
import re

from mnexp_b200 import _lib

ENGINE_SRC = os.path.join(os.path.dirname(os.path.abspath(_lib.__file__)), 'csrc', 'engine.cu')
LSTUR_ERR_ARG = -1


def _listed(macro):
    """Names of the X-macro list `macro` in engine.cu (the one list the plan's fields and name tables come from)."""
    src = open(ENGINE_SRC).read()
    body = re.search(r'#define %s\(X\)((?:[^\n]*\\\n)*[^\n]*)' % macro, src).group(1)
    return re.findall(r'X\((?:\w+,\s*)?(\w+)\)', body)


WS_NAMES = _listed('LSTUR_WS_REGIONS')
DENSE_NAMES = _listed('LSTUR_DENSE_TENSORS')

# (G, Ue, U) of each arch for document vectors of width D (include/lstur_b200.h, LSTUR_ARCH_*)
ARCH_DIMS = {
    0: lambda D, G: (G, G, G), 1: lambda D, G: (G, G, D), 2: lambda D, G: (G, G, 2 * G), 3: lambda D, G: (G, G, G),
    4: lambda D, G: (G, G, G), 5: lambda D, G: (G, D, D), 6: lambda D, G: (G, G, D), 7: lambda D, G: (G, G + 8, D),
    8: lambda D, G: (G, G + 8, G + 8), 9: lambda D, G: (G, G, D + G), 10: lambda D, G: (G, G, D),
    11: lambda D, G: (G, G, D + G), 12: lambda D, G: (G, 2 * G, G), 13: lambda D, G: (G, G, 1), 14: lambda D, G: (G, G, G),
    15: lambda D, G: (G, G, 2 * G),
}

# optional parts, each on top of the whole arch x precision x mode x scorer matrix
EXTRAS = [
    {},
    dict(dv=4, ds=4, n_vert=16, n_subvert=30),
    dict(aux_nv=5, aux_hidden=8, aux_gain=0.3),
    dict(cls_nv=6),
    dict(trainable_word_emb=1),
    dict(loss_model=1, C=1, bce_neg=4, gain=2.0),
    dict(L=50),
    dict(B=2048),
    dict(dropout=0.2),
    dict(use_dense=0),
]


def configs():
    """-> [(key, lstur_config kwargs)] of the matrix."""
    out = []
    for extra, arch, prec, bw, score in itertools.product(range(len(EXTRAS)), range(16), (0, 2), (1, 0), (0, 1, 2)):
        cfg = dict(B=8, W=5, C=3, L=7, E=12, F=16, KS=3, use_dense=1, Dd=16, dv=0, ds=0, G=16, arch=arch,
                   score_model=score, rec_act=0, precision=prec, V=120, n_users=50, n_docs=81, dropout=0.0,
                   save_for_backward=bw, n_vert=0, n_subvert=0, Hs=0 if score == 0 else 8, loss_model=0, bce_neg=0,
                   gain=0.0, trainable_word_emb=0, aux_nv=0, aux_hidden=0, aux_gain=0.0, cls_nv=0)
        cfg.update(EXTRAS[extra])
        if cfg['trainable_word_emb'] and not bw:
            continue
        if not cfg['use_dense']:
            cfg['Dd'] = cfg['F']
        D = cfg['Dd'] + cfg['dv'] + cfg['ds']
        cfg['G'], cfg['Ue'], cfg['U'] = ARCH_DIMS[arch](D, cfg['G'])
        out.append(((extra, arch, prec, bw, score), cfg))
    return out


def plan_layout(lib, cfg):
    """-> None if the plan is refused, else (workspace_bytes, dense_count, dense_head_count, {ws name: (offset, count)},
    {dense name: (offset, count)}); a region's offset is its byte offset (view of a workspace at address 0)."""
    c = _lib.lstur_config(**cfg)
    plan = ctypes.c_void_p()
    if lib.lstur_plan_create(ctypes.byref(c), ctypes.byref(plan)) != 0:
        return None
    try:
        ptr, off, cnt = ctypes.c_void_p(), ctypes.c_longlong(), ctypes.c_longlong()
        ws = {}
        for name in WS_NAMES:
            if lib.lstur_plan_view(plan, None, name.encode(), ctypes.byref(ptr), ctypes.byref(cnt)) == 0:
                ws[name] = (ptr.value or 0, cnt.value)
        dense = {}
        for name in DENSE_NAMES:
            if lib.lstur_plan_dense_offset(plan, name.encode(), ctypes.byref(off), ctypes.byref(cnt)) == 0:
                dense[name] = (off.value, cnt.value)
        return (lib.lstur_plan_workspace_bytes(plan), lib.lstur_plan_dense_count(plan),
                lib.lstur_plan_dense_head_count(plan), ws, dense)
    finally:
        lib.lstur_plan_destroy(plan)


def _disjoint(spans):
    spans = sorted(spans)
    return all(a[0] + a[1] <= b[0] for a, b in zip(spans, spans[1:]))


def test_names_listed_once():
    assert len(WS_NAMES) == len(set(WS_NAMES)) and len(WS_NAMES) > 100
    assert len(DENSE_NAMES) == len(set(DENSE_NAMES)) and len(DENSE_NAMES) > 30


def test_layout_over_config_matrix(lib):
    n_valid = 0
    for key, cfg in configs():
        lay = plan_layout(lib, cfg)
        D = cfg['Dd'] + cfg['dv'] + cfg['ds']
        # the matrix's only refused plans: a 'dot' scorer whose user vector is not as wide as the document vector
        assert (lay is None) == (cfg['score_model'] == 0 and cfg['U'] != D), (key, lib.lstur_last_error())
        if lay is None:
            continue
        n_valid += 1
        ws_bytes, dense_count, dense_head, ws, dense = lay
        for name in ('tokens', 'doc_vec', 'user_vec', 'logits', 'probs', 'loss', 'gemm_ws', 'colsum_ws'):
            assert name in ws, (key, name)
        for name, (off, cnt) in ws.items():
            assert off % 256 == 0 and cnt >= 0 and off + 4 * cnt <= ws_bytes, (key, name, off, cnt, ws_bytes)
        assert _disjoint([(off, 4 * cnt) for off, cnt in ws.values()]), key
        for name, (off, cnt) in dense.items():
            assert off % 4 == 0 and cnt > 0 and off + cnt <= dense_count, (key, name, off, cnt, dense_count)
        assert _disjoint(list(dense.values())), key
        att_b_end = dense['att_b'][0] + dense['att_b'][1]
        assert dense_head == (att_b_end + 3) // 4 * 4, key
        assert all(off >= dense_head for name, (off, _) in dense.items() if name not in ('conv_w', 'conv_b', 'att_w', 'att_b'))
    assert n_valid > 1500


def test_unknown_names(lib):
    cfg = configs()[0][1]
    c = _lib.lstur_config(**cfg)
    plan = ctypes.c_void_p()
    assert lib.lstur_plan_create(ctypes.byref(c), ctypes.byref(plan)) == 0
    try:
        ptr, off, cnt = ctypes.c_void_p(), ctypes.c_longlong(), ctypes.c_longlong()
        for name in (b'no_such_region', b'doc_ve', b'', b'conv_w'):
            assert lib.lstur_plan_view(plan, None, name, ctypes.byref(ptr), ctypes.byref(cnt)) == LSTUR_ERR_ARG, name
        for name in (b'no_such_tensor', b'conv', b'', b'doc_vec', b'con_w'):
            assert lib.lstur_plan_dense_offset(plan, name, ctypes.byref(off), ctypes.byref(cnt)) == LSTUR_ERR_ARG, name
    finally:
        lib.lstur_plan_destroy(plan)
