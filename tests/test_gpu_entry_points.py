"""Every batched C entry point exists as a uint64 host call, a device call (`*_device`, torch CUDA tensors on the
caller's stream) and a uint32 host call (`hecuda_u32_*`).  The three must compute the same residues, launch the same
kernels in the same chunks and refuse bad arguments with the same code and message.

The context is made with HECUDA_CHUNK=3 and driven at batch 10, so ops with scratch run in chunks of 3+3+3+1 (and of 1
for multiply+relinearize and the ct x ct inner product of 2 pairs).  The batch is below 64, so the host pipeline's stage
clamp does not engage and the host and device calls chunk alike.  It is a Bfv<UInt32> context, so that the uint32 calls
can be compared with the uint64 calls on the same context."""
import os

import numpy as np
import pytest

import hecuda
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

N, T, B, PAIRS, TERMS, ELEMENT = 64, 641, 10, 2, 3, 3


class Setup:
    pass


@pytest.fixture(scope="module")
def s():
    hecuda.set_device(0)
    old = os.environ.get("HECUDA_CHUNK")
    os.environ["HECUDA_CHUNK"] = "3"
    try:
        moduli = orc.generate_primes([28, 28, 29], False, N)
        d = Setup()
        d.g = hecuda.Context(N, moduli, T, scalar=np.uint32)
        d.other = hecuda.Context(N, moduli, T, scalar=np.uint32)
        d.g64 = hecuda.Context(N, orc.generate_primes([50, 50, 51], False, N), T)
    finally:
        if old is None:
            del os.environ["HECUDA_CHUNK"]
        else:
            os.environ["HECUDA_CHUNK"] = old
    o = orc.Context(N, moduli, T, word_bits=32)
    L = d.L = d.g.L
    sk, rk = o.keygen(5)
    gk = o.galois_keygen(77, sk, ELEMENT)
    d.key, d.other_key = hecuda.EvaluationKey(d.g, rk), hecuda.EvaluationKey(d.other, rk)
    for k in (d.key, d.other_key):
        k.setGaloisKey(ELEMENT, gk)
    q = moduli[:L]

    def uniform(seed, base, *shape):
        return orc.fill_uniform(seed, base, N, int(np.prod(shape[:-1]))).reshape(shape)

    d.ct2a, d.ct2b = uniform(1, q, B, 2, L, N), uniform(2, q, B, 2, L, N)
    d.ct3 = uniform(3, q, B, 3, L, N)
    d.poly_q = uniform(4, q, B, L, N)
    d.poly_qbsk = uniform(5, q + d.g.bskModuli, B, 2 * L + 1, N)
    d.ipa = uniform(6, q, B, PAIRS, 2, L, N)
    d.ipb = uniform(7, q, B, PAIRS, 2, L, N)
    d.query = uniform(8, q, TERMS, 2, L, N)
    d.pts = uniform(9, q, B, TERMS, L, N)
    rng = np.random.default_rng(10)
    d.present = rng.integers(0, 2, (B, TERMS), dtype=np.uint8)
    d.plain = rng.integers(0, T, (B, N), dtype=np.uint64)
    yield d
    for k in (d.key, d.other_key):
        k.close()
    for g in (d.g, d.other, d.g64):
        g.close()


class Op:
    """One batched operation: its symbol (without the hecuda_ / hecuda_u32_ prefix and the _device suffix), inputs,
    output shape and argument list.  `args(a)` lays out the arguments from a.h, a.key, a.l, a.batch, a.ins (input
    pointers) and a.out.  `host_chunk` is the host pipeline's items per chunk (None: one chunk at this size)."""

    def __init__(self, stem, inputs, out, args, host_chunk=None, device=True, u32=True, inplace=False, key=None, level=False):
        self.stem, self.inputs, self.out, self.args = stem, inputs, out, args
        self.host_chunk, self.device, self.u32, self.inplace, self.key, self.level = (host_chunk, device, u32, inplace, key,
                                                                                     level)


def ntt(stem):
    return Op(stem, lambda d: [d.poly_q], lambda d, b: (b, d.L, N), lambda a: (a.h, hecuda.BASE_Q, a.ins[0], a.l, a.batch),
              inplace=True)


def mul_relin(ms):
    return Op("bfv_multiply_relinearize", lambda d: [d.ct2a, d.ct2b], lambda d, b: (b, 2, d.L - ms, N),
              lambda a: (a.h, a.key, a.ins[0], a.ins[1], ms, a.out, a.batch), host_chunk=1, key="relin")


OPS = {
    "ntt_forward": ntt("ntt_forward"),
    "ntt_inverse": ntt("ntt_inverse"),
    "multiply": Op("bfv_multiply", lambda d: [d.ct2a, d.ct2b], lambda d, b: (b, 3, d.L, N),
                   lambda a: (a.h, a.ins[0], a.ins[1], a.out, a.batch), host_chunk=3),
    "relinearize": Op("bfv_relinearize", lambda d: [d.ct3], lambda d, b: (b, 2, d.L, N),
                      lambda a: (a.h, a.key, a.ins[0], a.l, a.out, a.batch), host_chunk=3, key="relin", level=True),
    "mod_switch_down": Op("bfv_mod_switch_down", lambda d: [d.ct3], lambda d, b: (b, 3, d.L - 1, N),
                          lambda a: (a.h, a.ins[0], 3, a.l, a.out, a.batch), level=True),
    "multiply_relinearize": mul_relin(0),
    "multiply_relinearize_mod_switch_down": mul_relin(1),
    "relinearize_mod_switch_down": Op("bfv_relinearize_mod_switch_down", lambda d: [d.ct3], lambda d, b: (b, 2, d.L - 1, N),
                                      lambda a: (a.h, a.key, a.ins[0], a.l, a.out, a.batch), host_chunk=3, device=False,
                                      key="relin", level=True),
    "apply_galois": Op("bfv_apply_galois", lambda d: [d.ct2a], lambda d, b: (b, 2, d.L, N),
                       lambda a: (a.h, a.key, a.ins[0], a.l, ELEMENT, a.out, a.batch), host_chunk=3, key="galois",
                       level=True),
    "inner_product": Op("bfv_inner_product", lambda d: [d.ipa, d.ipb], lambda d, b: (b, 3, d.L, N),
                        lambda a: (a.h, a.ins[0], a.ins[1], a.out, PAIRS, a.batch), host_chunk=1),
    "inner_product_plaintexts": Op("bfv_inner_product_plaintexts", lambda d: [d.query, d.pts, d.present],
                                   lambda d, b: (b, 2, d.L, N),
                                   lambda a: (a.h, a.ins[0], 2, a.l, TERMS, a.ins[1], a.ins[2], a.out, a.batch), u32=False,
                                   level=True),
    "plaintext_to_eval": Op("plaintext_to_eval", lambda d: [d.plain], lambda d, b: (b, d.L, N),
                            lambda a: (a.h, a.ins[0], a.l, a.out, a.batch), u32=False, level=True),
    "lift_q_to_qbsk": Op("rnstool_lift_q_to_qbsk", lambda d: [d.poly_q], lambda d, b: (b, 2 * d.L + 1, N),
                         lambda a: (a.h, a.ins[0], a.out, a.batch), device=False),
    "floor_qbsk_to_q": Op("rnstool_floor_qbsk_to_q", lambda d: [d.poly_qbsk], lambda d, b: (b, d.L, N),
                          lambda a: (a.h, a.ins[0], a.out, a.batch), device=False),
}


def variants(op):
    return ["host"] + (["device"] if op.device else []) + (["u32"] if op.u32 else [])


class Args:
    pass


def run(d, op, io, batch=B, h="ctx", key="key", l=None):
    """Calls one variant; returns (rc, last error, output as uint64, kernel launches)."""
    lib = hecuda.load_library()
    a = Args()
    a.h = {"ctx": d.g._h, "null": None, "g64": d.g64._h}[h]
    a.key = {"key": d.key._h, "none": None, "other": d.other_key._h}[key]
    a.l, a.batch = d.L if l is None else l, batch
    inputs = [x[:batch] if x.shape[0] == B else x for x in op.inputs(d)]
    shape = op.out(d, batch)
    if io == "device":
        ins = [torch.from_numpy(x.view(np.int64) if x.dtype == np.uint64 else x).cuda() for x in inputs]
        out = ins[0] if op.inplace else torch.zeros(shape, dtype=torch.int64, device="cuda")
        a.ins, a.out = [t.data_ptr() for t in ins], out.data_ptr()
        fn = getattr(lib, "hecuda_" + op.stem + "_device")
        extra = (torch.cuda.current_stream().cuda_stream,)
    else:
        wide = np.uint32 if io == "u32" else np.uint64
        ins = [np.ascontiguousarray(x.astype(wide) if x.dtype == np.uint64 else x) for x in inputs]
        out = ins[0] if op.inplace else np.zeros(shape, dtype=wide)
        a.ins, a.out = [x.ctypes.data for x in ins], out.ctypes.data
        fn = getattr(lib, ("hecuda_u32_" if io == "u32" else "hecuda_") + op.stem)
        extra = ()
    torch.cuda.synchronize()
    before = lib.hecuda_kernel_launch_count()
    rc = fn(*op.args(a), *extra)
    launches = lib.hecuda_kernel_launch_count() - before
    message = (lib.hecuda_last_error() or b"").decode() if rc else ""
    torch.cuda.synchronize()
    if io == "device":
        result = out.cpu().numpy().view(np.uint64)
    else:
        result = out.astype(np.uint64)
    return rc, message, result, launches


@pytest.mark.parametrize("name", sorted(OPS))
def test_variants_match_the_uint64_host_call(s, name):
    op = OPS[name]
    rc, _, want, launches = run(s, op, "host")
    assert rc == 0 and launches > 0
    assert want.any()
    host_chunk = op.host_chunk or B
    chunks = -(-B // host_chunk)
    for io in variants(op)[1:]:
        rc, msg, got, n = run(s, op, io)
        assert rc == 0, msg
        assert np.array_equal(got, want), io
        if io == "device":
            assert n == launches
        else:  # a widen after each input's H2D copy and a narrow before the D2H copy, per chunk
            assert n == launches + chunks * (len(op.inputs(s)) + 1)


@pytest.mark.parametrize("name", sorted(OPS))
def test_empty_batch(s, name):
    op = OPS[name]
    for io in variants(op):
        rc, msg, _, launches = run(s, op, io, batch=0)
        assert (rc, msg, launches) == (0, "", 0), io


def same_error(s, op, **kw):
    results = {io: run(s, op, io, **kw)[:2] for io in variants(op)}
    assert len(set(results.values())) == 1, results
    rc, msg = results["host"]
    assert rc != 0 and msg
    return rc


@pytest.mark.parametrize("name", sorted(OPS))
def test_same_errors_everywhere(s, name):
    op = OPS[name]
    assert same_error(s, op, h="null") == -1
    if op.key:
        assert same_error(s, op, key="none") == -5
        assert same_error(s, op, key="other") == -1
    if op.level:
        assert same_error(s, op, l=s.L + 1) == -1


def test_u32_calls_need_a_32_bit_context(s):
    seen = set()
    for name, op in OPS.items():
        if op.u32:
            rc, msg, _, launches = run(s, op, "u32", h="g64")
            assert rc == -1 and launches == 0, name
            seen.add(msg)
    assert seen == {"invalidContext: not a Bfv<UInt32> context (hecuda_context_create_u32)"}
