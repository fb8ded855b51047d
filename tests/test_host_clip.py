"""C ABI of the gradient-clipping entry points (gradnorm.cu, rowwise.cu) without a GPU: the symbols are declared and exported,
and bad arguments are rejected before anything is launched."""
import ctypes

import pytest

import ac_tsr_b200 as A

FAKE = 256          # a non-NULL device address: every call below fails its argument checks before touching it


def test_clip_symbols_are_declared_and_exported():
    import __graft_entry__ as g
    g.build()
    protos = A._lib.parse_header()
    dll = ctypes.CDLL(A._lib.LIB_PATH)
    for name in ('acsr_grad_norm_max_blocks', 'acsr_grad_norm_partial', 'acsr_adam_step_clipped'):
        assert name in protos and hasattr(dll, name), name
    assert A.LIB.query('acsr_grad_norm_max_blocks') >= A.LIB.query('acsr_num_sms')
    assert [t for _, t in protos['acsr_grad_norm_partial'][1]][4] is ctypes.c_double          # norm_type keeps its double precision


def _ranges(*r):
    return (ctypes.c_int64 * (2 * len(r)))(*[x for p in r for x in p])


@pytest.mark.parametrize('args,match', [
    ((None, 10, _ranges((0, 10)), 1, 2.0, FAKE, FAKE, FAKE), 'NULL'),
    ((FAKE, 10, None, 1, 2.0, FAKE, FAKE, FAKE), 'NULL'),
    ((FAKE, 10, _ranges((0, 10)), 1, 2.0, None, FAKE, FAKE), 'NULL'),
    ((FAKE, 10, _ranges((0, 10)), 1, 2.0, FAKE, None, FAKE), 'NULL'),
    ((FAKE, 10, _ranges((0, 10)), 1, 2.0, FAKE, FAKE, None), 'NULL'),
    ((FAKE, -1, _ranges((0, 10)), 1, 2.0, FAKE, FAKE, FAKE), 'n=-1'),
    ((FAKE, 10, _ranges((0, 10)), 0, 2.0, FAKE, FAKE, FAKE), 'n_ranges'),
    ((FAKE, 10, _ranges(*[(0, 1)] * 9), 9, 2.0, FAKE, FAKE, FAKE), 'n_ranges'),
    ((FAKE, 10, _ranges((0, 10)), 1, 0.0, FAKE, FAKE, FAKE), 'norm_type'),
    ((FAKE, 10, _ranges((0, 10)), 1, -2.0, FAKE, FAKE, FAKE), 'norm_type'),
    ((FAKE, 10, _ranges((0, 10)), 1, float('nan'), FAKE, FAKE, FAKE), 'norm_type'),
    ((FAKE, 10, _ranges((0, 11)), 1, 2.0, FAKE, FAKE, FAKE), 'range 0'),
    ((FAKE, 10, _ranges((0, 4), (6, 5)), 2, 2.0, FAKE, FAKE, FAKE), 'range 1'),
    ((FAKE, 10, _ranges((-1, 4)), 1, 2.0, FAKE, FAKE, FAKE), 'range 0'),
])
def test_grad_norm_partial_rejects_bad_arguments_without_a_gpu(args, match):
    A.LIB.load()
    with pytest.raises(A.AcsrError, match=match):
        A.LIB.call('acsr_grad_norm_partial', *args, None)


def _adam(**kw):
    a = dict(param=FAKE, grad=FAKE, exp_avg=FAKE, exp_avg_sq=FAKE, n=10, lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=0.0,
             step_count=FAKE, partials=FAKE, n_partials=1, norm_type=2.0, max_norm=1.0, total_out=FAKE, stream=None)
    a.update(kw)
    return [a[n] for n, _ in A._lib.parse_header()['acsr_adam_step_clipped'][1]]


@pytest.mark.parametrize('kw,match', [
    (dict(param=None), 'NULL'), (dict(grad=None), 'NULL'), (dict(partials=None), 'NULL'), (dict(total_out=None), 'NULL'),
    (dict(step_count=None), 'NULL'), (dict(n=-5), 'n=-5'), (dict(n_partials=0), 'n_partials'), (dict(n_partials=1025), 'n_partials'),
    (dict(norm_type=0.0), 'norm_type'), (dict(norm_type=float('nan')), 'norm_type'), (dict(max_norm=0.0), 'max_norm'),
    (dict(max_norm=-1.0), 'max_norm'), (dict(max_norm=float('nan')), 'max_norm'),
])
def test_adam_step_clipped_rejects_bad_arguments_without_a_gpu(kw, match):
    A.LIB.load()
    with pytest.raises(A.AcsrError, match=match):
        A.LIB.call('acsr_adam_step_clipped', *_adam(**kw))
