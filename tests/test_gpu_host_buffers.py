"""GPU tests (``-m gpu``) of the host side's device buffers and result replication: a buffer that would have to grow
inside a CUDA-graph capture is refused, and fp32 mode refuses every result replication it cannot honour."""
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.fail("gpu-marked tests need a CUDA device (there is no CPU fallback to test)")
    return torch.device("cuda:0")


def test_first_topk_inside_a_graph_capture_is_refused(dev):
    """A fresh engine has no top-k table yet: preparing one inside a capture returns PBG_ERR_INVALID naming the table,
    instead of a device synchronisation that would break the caller's capture.  Outside the capture the same engine
    then returns what a second fresh engine returns."""
    from pbg import cabi
    from pbg.engine import Engine
    g = torch.Generator().manual_seed(31)
    q, table = torch.randn(64, 128, generator=g).to(dev), torch.randn(5000, 128, generator=g).to(dev)
    eng = Engine(128, 8, 8, 16, dev)
    cs = torch.cuda.Stream(dev)
    with torch.cuda.stream(cs):
        with pytest.raises(cabi.PbgError) as err:
            with torch.cuda.graph(torch.cuda.CUDAGraph(), stream=cs):
                eng.cosine_topk(q, table, 10)
    assert err.value.status == cabi.PBG_ERR_INVALID
    assert "top-k table" in str(err.value)
    torch.cuda.synchronize()
    scores, idx = eng.cosine_topk(q, table, 10)
    ref_scores, ref_idx = Engine(128, 8, 8, 16, dev).cosine_topk(q, table, 10)
    torch.cuda.synchronize()
    assert torch.equal(scores, ref_scores) and torch.equal(idx, ref_idx)


def test_fp32_pass_refuses_a_probs_multicast_alone(dev, synth):
    """Result multicast is a bf16-mode feature: in fp32 mode a probs multicast address alone is refused with
    PBG_ERR_UNSUPPORTED (the address is never dereferenced: the call fails before any launch), and clearing it
    restores the normal result."""
    import modular_prot_b_gan as m
    from pbg import cabi
    G, D = synth.make_models(m.ModularGenerator, m.ModularDiscriminator)
    eng = m.make_fused_engine(G.to(dev).eval(), D.to(dev).eval())
    g = torch.Generator().manual_seed(32)
    h, r, t = (torch.randn(256, 128, generator=g).to(dev) for _ in range(3))
    ref_logits, ref_probs = eng.discriminator_forward(h, r, t, precision="fp32")
    eng.set_result_multicast(probs=0x10000)
    with pytest.raises(cabi.PbgError) as err:
        eng.discriminator_forward(h, r, t, precision="fp32")
    assert err.value.status == cabi.PBG_ERR_UNSUPPORTED
    eng.set_result_multicast()
    logits, probs = eng.discriminator_forward(h, r, t, precision="fp32")
    torch.cuda.synchronize()
    assert torch.equal(logits, ref_logits) and torch.equal(probs, ref_probs)
