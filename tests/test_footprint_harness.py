"""The arena helper of tests/test_gpu_footprint.py on CPU tensors: it must report every kind of stray or missing store at
the right (argument, index), or the GPU footprint tests would pass vacuously."""
import pytest
import torch

from test_gpu_footprint import GUARD, SENTINEL, Arg, padded_strides, same_bits, verify

DT = [torch.bfloat16, torch.float16, torch.float32]


def _fails(*args, match):
    with pytest.raises(AssertionError, match=match):
        verify(*args)


def test_padded_strides():
    assert padded_strides((2, 3, 4, 5), [7, 1, 2, 0]) == [3 * (4 * 7 + 1) + 7, 4 * 7 + 1, 7, 1]
    assert padded_strides((2, 3, 4, 5), [0, 8, 0, 0], order=(0, 2, 1, 3)) == [4 * 3 * 13, 13, 3 * 13, 1]


@pytest.mark.parametrize("dtype", DT)
def test_clean_write_passes(dtype):
    o = Arg("o", (2, 3, 5, 8), dtype, "out", device="cpu", pad=[3, 1, 2, 0], order=(0, 2, 1, 3)).arm()
    x = Arg.of("x", torch.randn(2, 3, 5, 8).to(dtype), pad=[1, 0, 3, 0]).arm()
    assert (o.ptr - o.buf.data_ptr()) % 256 == 0 and (x.ptr - x.buf.data_ptr()) % 256 == 0
    o.t.copy_(x.t * 2)
    verify(o, x)
    same_bits(o.t, x.t * 2)


def test_sentinels_are_nans():
    for dt, s in SENTINEL.items():
        bits = torch.tensor([s - (1 << 16) if dt != torch.float32 and s >= 1 << 15 else s],
                            dtype=torch.int16 if dt != torch.float32 else torch.int64)
        v = bits.to(torch.int32 if dt == torch.float32 else torch.int16).view(dt)
        assert torch.isnan(v).all(), dt


@pytest.mark.parametrize("dtype", DT)
def test_stray_stores_are_located(dtype):
    def armed():
        o = Arg("o", (2, 3, 8), dtype, "out", device="cpu", pad=[4, 2, 0]).arm()
        o.t.fill_(1.0)
        return o
    o = armed()
    o.buf[GUARD - 3] = 0
    _fails(o, match=r"o: front guard, byte -3: store outside")
    o = armed()
    o.buf[GUARD + o.region + 100] = 0
    _fails(o, match=r"o: back guard, byte 100: store outside")
    o = armed()
    esz = o.esz
    gap = o.strides[1] - 1                                  # first padding element after row (0, 0)
    o.buf[GUARD + gap * esz] = 0
    _fails(o, match=rf"o: gap, region byte {gap * esz}: store outside")
    o = armed()
    o.buf[GUARD + o.region - 1] = 0                          # tail of the region after the last element
    _fails(o, match=r"o: gap, region byte")


def test_store_outside_a_partial_write_set_is_located():
    p = Arg("pool", (4, 2, 6), torch.float16, "inout", device="cpu")
    p.t.copy_(torch.randn(4, 2, 6))
    w = torch.zeros(4, 2, 6, dtype=torch.bool)
    w[1, 0] = True
    p.arm(w)
    p.t[1, 0] = 3.0
    verify(p)
    p.t[2, 1, 4] = 7.0
    _fails(p, match=r"pool: element \(2, 1, 4\): store outside the write set")


@pytest.mark.parametrize("dtype", DT)
def test_missed_element_is_reported(dtype):
    o = Arg("lse", (3, 5), dtype, "out", device="cpu", pad=[2, 0]).arm()
    o.t.fill_(0.5)
    o.t[2, 4] = float("nan")
    verify(o)                                                # a NaN a kernel writes is not the sentinel
    o.arm()
    o.t.fill_(0.5)
    o.bits()[2, 4] = o.snap.view(o.dtype).as_strided(o.shape, o.strides, GUARD // o.esz).view(o.bits().dtype)[2, 4]
    _fails(o, match=r"lse: element \(2, 4\) of the write set was never written \(1 elements")


def test_input_mutation_is_reported():
    x = Arg.of("seq_lens", torch.tensor([5, 0, 17], dtype=torch.int32)).arm()
    x.t[1] = 1
    _fails(x, match=r"seq_lens: element \(1,\): input modified")
    q = Arg.of("q", torch.randn(2, 4, 8), pad=[0, 3, 0]).arm()
    q.buf[GUARD + 4 * 8 * 4] = 0                             # a gap byte of an input
    _fails(q, match=r"q: gap, region byte 128: input modified")


def test_workspace_may_change_but_not_its_guards():
    w = Arg("workspace", (1000,), torch.uint8, "ws", device="cpu").arm()
    w.t.fill_(7)
    verify(w)
    w.buf[GUARD + 1000] = 0                                  # past the declared bytes, inside the 256-byte granule
    _fails(w, match=r"workspace: gap, region byte 1000")


def test_value_mismatch_is_reported():
    a, b = torch.zeros(3, 4), torch.zeros(3, 4)
    b[1, 2] = -0.0
    with pytest.raises(AssertionError, match=r"1 elements differ .* first at \(1, 2\)"):
        same_bits(a, b)
