"""Kernel-level parity tests: every C-ABI entry point against the CPU oracle / the committed
reference outputs.  Run on the B200 box (``pytest -m gpu``)."""
import numpy as np
import pytest
import torch

from helpers import load_golden
from oracle import lanczos_oracle as orc
from oracle import segment_oracle

pytestmark = pytest.mark.gpu


def dev():
  return torch.device('cuda:0')


def ops():
  from lanczosnetwork_b200 import ops as _ops
  return _ops


# ------------------------------------------------------------------------------------------
# operators/segment_reduction
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize('shape,S', [((3, 7, 5), 4), ((2, 16, 8), 16), ((1, 1, 1), 1),
                                     ((4, 33, 12), 9), ((0, 5, 4), 3)])
def test_segment_sum_matches_oracle(shape, S):
  rng = np.random.RandomState(sum(shape) + S)
  data = rng.randn(*shape).astype(np.float32)
  seg = rng.randint(0, S, size=shape[:2]).astype(np.int64)
  out = ops().segment_sum_forward(torch.from_numpy(data).to(dev()), torch.from_numpy(seg).to(dev()), S)
  ref = segment_oracle.segment_sum_forward(data, seg, S)
  np.testing.assert_allclose(out.cpu().numpy(), ref, rtol=1e-6, atol=1e-6)   # fp32 atomics: order
  gout = rng.randn(shape[0], S, shape[2]).astype(np.float32)
  gd = ops().segment_sum_backward(torch.from_numpy(gout).to(dev()), torch.from_numpy(seg).to(dev()), shape)
  assert np.array_equal(gd.cpu().numpy(), segment_oracle.segment_sum_backward(gout, seg, shape))


def test_segment_sum_reference_flavours_agree_where_consistent():
  """S == dim1 and ids shared across the batch: the reference CPU loop, its CUDA kernel and the
  intended semantics coincide -- and so does ours."""
  rng = np.random.RandomState(0)
  B, C, X = 3, 6, 4
  data = rng.randn(B, C, X).astype(np.float32)
  seg = np.tile(rng.randint(0, C, size=(1, C)), (B, 1)).astype(np.int64)
  a = segment_oracle.segment_sum_forward(data, seg, C, 'intended')
  b = segment_oracle.segment_sum_forward(data, seg, C, 'ref_cuda')
  c = segment_oracle.segment_sum_forward(data, seg, C, 'ref_cpu')
  np.testing.assert_allclose(a, b, atol=1e-6)
  np.testing.assert_allclose(a, c, atol=1e-6)
  out = ops().segment_sum_forward(torch.from_numpy(data).to(dev()), torch.from_numpy(seg).to(dev()), C)
  np.testing.assert_allclose(out.cpu().numpy(), a, atol=1e-6)


def test_segment_sum_matches_compiled_reference_kernel():
  """The reference's OWN CUDA kernels (operators/src/cuda/segment_reduction.cu:39-95) as a second
  checker on the domain where the reference is self-consistent (num_segments == dim1, its hard-coded
  output batch stride dim1*dim2, segment_reduction.cu:48); also pins the oracle's ``ref_cuda``
  flavour.  Their inputs and outputs are stored in tests/golden/segment_reduction_ref.npz (written by
  tests/golden/make_segment_golden.py); integer-valued data make fp32 atomic sums exact in any
  order -> bit-exact comparison."""
  g = load_golden('segment_reduction_ref.npz')
  for i, (B, C, X) in enumerate(g['shapes'].tolist()):
    data, seg, out_ref = g['c%d_data' % i], g['c%d_seg' % i], g['c%d_out' % i]
    d_seg = torch.from_numpy(seg).to(dev())
    ours = ops().segment_sum_forward(torch.from_numpy(data).to(dev()), d_seg, C)
    assert np.array_equal(ours.cpu().numpy(), out_ref)
    assert np.array_equal(out_ref, segment_oracle.segment_sum_forward(data, seg, C, 'ref_cuda'))
    assert np.array_equal(out_ref, segment_oracle.segment_sum_forward(data, seg, C, 'intended'))
    gout = torch.from_numpy(g['c%d_gout' % i]).to(dev())
    g_ours = ops().segment_sum_backward(gout, d_seg, (B, C, X))
    assert np.array_equal(g_ours.cpu().numpy(), g['c%d_grad' % i])


def test_segment_sum_autograd_and_module():
  from lanczosnetwork_b200.operators.modules import UnsortedSegmentSum
  rng = np.random.RandomState(3)
  data = torch.from_numpy(rng.randn(2, 9, 8).astype(np.float32)).to(dev()).requires_grad_(True)
  seg = torch.from_numpy(rng.randint(0, 5, size=(2, 9))).to(dev())
  out = UnsortedSegmentSum(5)(data, seg)
  ref = torch.zeros(2, 5, 8, device=dev()).index_put_(
      (torch.arange(2, device=dev())[:, None].expand(2, 9), seg), data.detach(), accumulate=True)
  torch.testing.assert_close(out, ref, rtol=1e-6, atol=1e-6)
  w = torch.from_numpy(rng.randn(2, 5, 8).astype(np.float32)).to(dev())
  (out * w).sum().backward()
  gref = w[torch.arange(2, device=dev())[:, None].expand(2, 9), seg]
  assert torch.equal(data.grad, gref)


def test_native_module_exports_reference_names():
  from lanczosnetwork_b200.operators._ext import segment_reduction as sr
  for name in ('unsorted_segment_sum_forward', 'unsorted_segment_sum_forward_gpu',
               'unsorted_segment_sum_backward', 'unsorted_segment_sum_backward_gpu'):
    assert callable(getattr(sr, name))
  with pytest.raises(RuntimeError):
    sr.unsorted_segment_sum_forward(torch.zeros(1, 2, 3), torch.zeros(1, 2, dtype=torch.long),
                                    (1, 2, 3), torch.zeros(1, 2, 3))


# ------------------------------------------------------------------------------------------
# generic strided batched GEMM
# ------------------------------------------------------------------------------------------
def test_bgemm_strided_channel_innermost_and_transposed():
  rng = np.random.RandomState(1)
  B, N, E1, D, K = 5, 26, 7, 40, 20
  L = torch.from_numpy(rng.randn(B, N, N, E1).astype(np.float32)).to(dev())
  X = torch.from_numpy(rng.randn(B, N, D).astype(np.float32)).to(dev())
  C = E1
  msg = torch.zeros(B, N, C * D, device=dev())
  ops().bgemm(L, (N * N * E1, 1, N * E1, E1), X, (N * D, 0, D, 1), msg, (N * C * D, D, C * D, 1),
              B, E1, N, D, N)
  ref = torch.cat([torch.bmm(L[..., e].double(), X.double()) for e in range(E1)], dim=2)
  torch.testing.assert_close(msg.double(), ref, rtol=1e-5, atol=1e-5)
  Q = torch.from_numpy(rng.randn(B, N, K).astype(np.float32)).to(dev())
  U = torch.empty(B, K, D, device=dev())
  ops().bgemm(Q, (N * K, 0, 1, K), X, (N * D, 0, D, 1), U, (K * D, 0, D, 1), B, 1, K, D, N)
  torch.testing.assert_close(U.double(), torch.bmm(Q.transpose(1, 2).double(), X.double()),
                             rtol=1e-5, atol=1e-5)
  f = torch.from_numpy(rng.randn(B, K, 3).astype(np.float32)).to(dev())
  out = torch.empty(B, 3, N, D, device=dev())
  ops().bgemm(Q, (N * K, 0, K, 1), U, (K * D, 0, D, 1), out, (3 * N * D, N * D, D, 1), B, 3, N, D,
              K, kscale=f, s_str=(K * 3, 1, 3))
  ref = torch.einsum('bnk,bks,bkd->bsnd', Q.double(), f.double(), U.double())
  torch.testing.assert_close(out.double(), ref, rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize('M,N,K', [(1, 1, 1), (65, 63, 17), (130, 2, 100), (64, 64, 16)])
def test_bgemm_bias_relu_edges(M, N, K):
  rng = np.random.RandomState(M + N + K)
  A = torch.from_numpy(rng.randn(M, K).astype(np.float32)).to(dev())
  W = torch.from_numpy(rng.randn(N, K).astype(np.float32)).to(dev())
  b = torch.from_numpy(rng.randn(N).astype(np.float32)).to(dev())
  out = torch.empty(M, N, device=dev())
  ops().bgemm(A, (0, 0, K, 1), W, (0, 0, 1, K), out, (0, 0, N, 1), 1, 1, M, N, K, bias=b, relu=True)
  ref = torch.relu(A.double() @ W.double().t() + b.double())
  torch.testing.assert_close(out.double(), ref, rtol=1e-5, atol=1e-5)


# ------------------------------------------------------------------------------------------
# tcgen05 3xTF32 dense layer
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize('M,N,K,relu', [(128, 128, 32, False), (300, 128, 1920, True),
                                        (26624, 128, 960, True), (1000, 2000, 512, False),
                                        (77, 8, 128, False), (2048, 128, 8, True),
                                        (64, 4096, 2000, True), (5, 40, 100, False),
                                        (256, 4096, 4096, True), (130, 520, 3204, False)])
def test_linear_tf32x3_fp32_grade(M, N, K, relu):
  g = torch.Generator(device='cpu').manual_seed(M * 7 + N * 3 + K)
  x = torch.randn(M, K, generator=g).to(dev())
  w = (torch.randn(N, K, generator=g) / np.sqrt(K)).to(dev())
  b = torch.randn(N, generator=g).to(dev())
  w_hi, w_lo = ops().split_tf32(w)
  # the split is exact to ~2^-22 relative and hi is representable in tf32
  assert torch.equal(w_hi.view(torch.int32) & 0x1FFF, torch.zeros_like(w_hi, dtype=torch.int32))
  assert (w - (w_hi + w_lo)).abs().max() <= 2.0 ** -21 * w.abs().max()
  out = ops().linear_tf32x3(x, w_hi, w_lo, b, relu)
  # deep K with few output tiles runs split-K: a second call must find its counters at zero
  assert torch.equal(out, ops().linear_tf32x3(x, w_hi, w_lo, b, relu))
  ref = x.double() @ w.double().t() + b.double()
  if relu:
    ref = torch.relu(ref)
  torch.backends.cuda.matmul.allow_tf32 = False
  f32 = x @ w.t() + b
  if relu:
    f32 = torch.relu(f32)
  err = (out.double() - ref).abs().max().item()
  err32 = (f32.double() - ref).abs().max().item()
  scale = ref.abs().max().item()
  # stated tolerance: within 8x the error of a true fp32 GEMM or 6e-6 of the output scale
  # (tensor-core accumulation truncates: ~K/8 truncation steps on the main accumulator)
  print('linear_tf32x3 M=%d N=%d K=%d: max err %.3g (fp32 cuBLAS %.3g) at scale %.3g' % (M, N, K, err, err32, scale))
  assert err <= max(8 * err32, 6e-6 * scale), (err, err32, scale)


def test_linear_tf32x3_rejects_bad_k():
  x = torch.randn(4, 10, device=dev())
  w = torch.randn(8, 10, device=dev())
  with pytest.raises(RuntimeError):
    ops().linear_tf32x3(x, w, w, None, False)


# ------------------------------------------------------------------------------------------
# small graph ops
# ------------------------------------------------------------------------------------------
def test_embedding_power_table_readout():
  rng = np.random.RandomState(2)
  table = torch.from_numpy(rng.randn(70, 64).astype(np.float32))
  idx = torch.from_numpy(rng.randint(0, 70, size=(9, 26)))
  out = ops().embedding_rows(idx.to(dev()), table.to(dev()))
  assert torch.equal(out.cpu(), table[idx])

  D = torch.from_numpy(rng.uniform(-1, 1, size=(9, 20)).astype(np.float32))
  D[0, -3:] = 0.0
  powers = [1, 2, 3, 5, 7, 10, 20, 30]
  tab = ops().ritz_power_table(D.to(dev()), powers).cpu()
  ref = orc.ritz_power_table(D.double(), powers)
  np.testing.assert_allclose(tab.numpy(), ref.numpy(), rtol=1.2e-7, atol=1e-45)
  ref32 = orc.ritz_power_table(D, powers)
  np.testing.assert_allclose(tab.numpy(), ref32.numpy(), rtol=4e-7, atol=1e-44)

  B, N, H, P = 6, 26, 128, 16
  state = torch.from_numpy(rng.randn(B, N, H).astype(np.float32))
  params = {'filter.0.weight': torch.from_numpy(rng.randn(P, H).astype(np.float32) * 0.1),
            'filter.0.bias': torch.from_numpy(rng.randn(P).astype(np.float32)),
            'att_func.0.weight': torch.from_numpy(rng.randn(1, H).astype(np.float32) * 0.1),
            'att_func.0.bias': torch.from_numpy(rng.randn(1).astype(np.float32))}
  mask = torch.zeros(B, N, dtype=torch.uint8)
  for b, n in enumerate([26, 1, 7, 13, 20, 25]):
    mask[b, :n] = 1
  spec = {'num_layer': 0}
  for m in (mask, None):
    ref = orc.readout({k: v.double() for k, v in params.items()}, spec, state.double(), m)
    out = ops().readout(state.to(dev()), params['filter.0.weight'].to(dev()),
                        params['filter.0.bias'].to(dev()),
                        params['att_func.0.weight'].reshape(-1).to(dev()),
                        params['att_func.0.bias'].to(dev()), None if m is None else m.to(dev()))
    np.testing.assert_allclose(out.cpu().numpy(), ref.numpy(), rtol=1e-5, atol=2e-6)


def test_gaussian_laplacian_matches_reference_output():
  g = load_golden('ada_forward_small.npz')
  from helpers import deterministic_state_dict
  from lanczosnetwork_b200 import configs
  from lanczosnetwork_b200.model import AdaLanczosNet
  cfg = configs.qm8_ada_lanczos_net(num_layer=2, hidden_dim=[32, 32], num_eig_vec=8,
                                    long_diffusion_dist=[2, 5], short_diffusion_dist=[1, 3])
  emb = deterministic_state_dict(AdaLanczosNet(cfg), int(g['weight_seed']))['embedding.weight']
  x = emb[torch.from_numpy(g['node_feat'])]
  out = ops().gaussian_laplacian(x.to(dev()), torch.from_numpy(g['L']).to(dev())).cpu().numpy()
  assert np.array_equal(out != 0, g['Le'] != 0)        # adjacency structure: exact
  np.testing.assert_allclose(out, g['Le'], rtol=2e-5, atol=1e-6)


# ------------------------------------------------------------------------------------------
# Lanczos tridiagonalisation / Ritz pairs / powers
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize('case', ['qm8', 'small', 'nomask', 'cta64', 'cta100'])
def test_lanczos_matches_reference_outputs(case):
  g = load_golden('ada_lanczos_layer.npz')
  A = torch.from_numpy(g[case + '_A'])
  mask = None if case == 'nomask' else torch.from_numpy(g[case + '_mask'])
  q1 = torch.from_numpy(g[case + '_q1'])
  K = int(g[case + '_K'])
  out = ops().lanczos_tridiag(A.to(dev()), None if mask is None else mask.to(dev()), q1.to(dev()), K)
  T_ref, Q_ref = g[case + '_T'], g[case + '_Q']
  T, Q = out['T'].cpu().numpy(), out['Q'].cpu().numpy()
  o64 = orc.lanczos_tridiagonalise(A.double(), mask, q1.double(), K)
  # integer / index logic: bit-exact (retained Krylov directions and node rows)
  assert np.array_equal(out['idx'].cpu().numpy(), o64['idx'].numpy())
  assert np.array_equal(T != 0, T_ref != 0)
  assert np.array_equal(Q != 0, Q_ref != 0)
  # floating point: no further from the fp64 oracle than 4x the reference's own fp32 error,
  # with an absolute floor (near-breakdown steps amplify rounding by 1/beta)
  eT_ref = np.abs(T_ref - o64['T'].numpy()).max()
  eQ_ref = np.abs(Q_ref - o64['Q'].numpy()).max()
  assert np.abs(T - o64['T'].numpy()).max() <= max(4 * eT_ref, 2e-5)
  assert np.abs(Q - o64['Q'].numpy()).max() <= max(4 * eQ_ref, 2e-4)
  np.testing.assert_allclose(out['alpha'].cpu().numpy(), np.diagonal(T, axis1=1, axis2=2))


@pytest.mark.parametrize('case', ['qm8', 'small', 'cta64', 'cta100'])
def test_tridiag_ritz_against_lapack(case):
  g = load_golden('ada_lanczos_layer.npz')
  T, Q = g[case + '_T'], g[case + '_Q']
  alpha = np.ascontiguousarray(np.diagonal(T, axis1=1, axis2=2))
  K = alpha.shape[1]
  beta = np.zeros_like(alpha)
  beta[:, :K - 1] = np.diagonal(T, offset=1, axis1=1, axis2=2)
  theta, V, status = ops().tridiag_ritz(torch.from_numpy(alpha).to(dev()),
                                        torch.from_numpy(beta).to(dev()),
                                        torch.from_numpy(Q).to(dev()))
  assert int(status.abs().sum()) == 0
  th_o, S_o, V_o = orc.tridiag_ritz(alpha, beta[:, :K - 1], Q)
  theta, V = theta.cpu().numpy().astype(np.float64), V.cpu().numpy().astype(np.float64)
  # Ritz values: ordered by descending magnitude, equal to LAPACK's as a multiset and in order
  assert np.all(np.diff(np.abs(theta), axis=1) <= 1e-7)
  np.testing.assert_allclose(np.sort(theta, axis=1), np.sort(th_o, axis=1), atol=3e-6)
  # sign / rotation invariant filters V g(theta) V^T for g = id, square, |.|^1/2
  for fn in (lambda t: t, lambda t: t * t, lambda t: np.sqrt(np.abs(t))):
    ours = np.einsum('bnk,bk,bmk->bnm', V, fn(theta), V)
    ref = np.einsum('bnk,bk,bmk->bnm', V_o, fn(th_o), V_o)
    np.testing.assert_allclose(ours, ref, atol=2e-5)
  # and V diag(theta) V^T reproduces Q T Q^T
  qtq = np.einsum('bnk,bkj,bmj->bnm', Q.astype(np.float64), T.astype(np.float64), Q.astype(np.float64))
  np.testing.assert_allclose(np.einsum('bnk,bk,bmk->bnm', V, theta, V), qtq, atol=2e-5)


def _check_ritz(theta, V, alpha, beta, Q, T):
  """(theta, V) of a fused launch against LAPACK on the launch's own tridiagonal."""
  K = alpha.shape[1]
  th_o, S_o, V_o = orc.tridiag_ritz(alpha, beta[:, :K - 1], Q)
  theta, V = theta.astype(np.float64), V.astype(np.float64)
  assert np.all(np.diff(np.abs(theta), axis=1) <= 1e-7)
  np.testing.assert_allclose(np.sort(theta, axis=1), np.sort(th_o, axis=1), atol=3e-6)
  for fn in (lambda t: t, lambda t: t * t, lambda t: np.sqrt(np.abs(t))):
    ours = np.einsum('bnk,bk,bmk->bnm', V, fn(theta), V)
    ref = np.einsum('bnk,bk,bmk->bnm', V_o, fn(th_o), V_o)
    np.testing.assert_allclose(ours, ref, atol=2e-5)
  qtq = np.einsum('bnk,bkj,bmj->bnm', Q.astype(np.float64), T.astype(np.float64), Q.astype(np.float64))
  np.testing.assert_allclose(np.einsum('bnk,bk,bmk->bnm', V, theta, V), qtq, atol=2e-5)


@pytest.mark.parametrize('case', ['qm8', 'small', 'nomask', 'cta64', 'cta100'])
def test_fused_lanczos_ritz_matches_reference_outputs(case):
  """lnb_lanczos_ritz (one launch: compress -> Lanczos -> QL -> V = Q S) against the EXECUTED
  reference's T, Q on the five regimes of the golden file, same yardsticks as the two-kernel path;
  its Ritz pairs against LAPACK on its own tridiagonal; and against the two-kernel path."""
  g = load_golden('ada_lanczos_layer.npz')
  A = torch.from_numpy(g[case + '_A'])
  mask = None if case == 'nomask' else torch.from_numpy(g[case + '_mask'])
  q1 = torch.from_numpy(g[case + '_q1'])
  K = int(g[case + '_K'])
  dm = None if mask is None else mask.to(dev())
  out = ops().lanczos_ritz(A.to(dev()), dm, q1.to(dev()), K)
  T_ref, Q_ref = g[case + '_T'], g[case + '_Q']
  T, Q = out['T'].cpu().numpy(), out['Q'].cpu().numpy()
  o64 = orc.lanczos_tridiagonalise(A.double(), mask, q1.double(), K)
  assert np.array_equal(out['idx'].cpu().numpy(), o64['idx'].numpy())
  assert np.array_equal(T != 0, T_ref != 0)
  assert np.array_equal(Q != 0, Q_ref != 0)
  eT_ref = np.abs(T_ref - o64['T'].numpy()).max()
  eQ_ref = np.abs(Q_ref - o64['Q'].numpy()).max()
  assert np.abs(T - o64['T'].numpy()).max() <= max(4 * eT_ref, 2e-5)
  assert np.abs(Q - o64['Q'].numpy()).max() <= max(4 * eQ_ref, 2e-4)
  alpha, beta = out['alpha'].cpu().numpy(), out['beta'].cpu().numpy()
  np.testing.assert_array_equal(alpha, np.diagonal(T, axis1=1, axis2=2))
  np.testing.assert_array_equal(beta[:, :K - 1], np.diagonal(T, offset=1, axis1=1, axis2=2))
  assert int((out['status'] & 1).sum()) == 0
  assert int((out['status'] & 2).sum()) == 0          # these operators are sparse: packed on chip
  _check_ritz(out['theta'].cpu().numpy(), out['V'].cpu().numpy(), alpha, beta, Q, T)
  # the tridiagonalisation-only call (AdaLanczosNet) returns the same T, Q bit for bit
  only = ops().lanczos_ritz(A.to(dev()), dm, q1.to(dev()), K, want_ritz=False)
  assert torch.equal(only['T'], out['T']) and torch.equal(only['Q'], out['Q'])
  assert 'theta' not in only


@pytest.mark.parametrize('N,K,B', [(26, 20, 64), (64, 40, 9), (200, 40, 5), (256, 40, 4),
                                   (500, 24, 3), (1024, 40, 3)])
def test_fused_lanczos_ritz_sweep_sizes_vs_fp64(N, K, B):
  """Every thread-group configuration of the fused kernel (32 ... 512 threads per graph) on
  G(n, min(0.5, 8/n)) operators with ragged sizes: idx exact, T / Q within 4x the fp32 oracle's own
  distance from the fp64 oracle, Ritz pairs against LAPACK."""
  import bench
  rng = np.random.RandomState(N + K)
  A = np.zeros((B, N, N), np.float32)
  mask = np.zeros((B, N), np.uint8)
  for b in range(B):
    n = N if b == 0 else int(rng.randint(N // 2, N + 1))
    A[b, :n, :n] = bench.gnp_operator(rng, n, min(0.5, 8.0 / n))
    mask[b, :n] = 1
  q1 = rng.randn(B, N).astype(np.float32)
  out = ops().lanczos_ritz(torch.from_numpy(A).to(dev()), torch.from_numpy(mask).to(dev()),
                           torch.from_numpy(q1).to(dev()), K)
  o64 = orc.lanczos_tridiagonalise(torch.from_numpy(A).double(), torch.from_numpy(mask),
                                   torch.from_numpy(q1).double(), K)
  o32 = orc.lanczos_tridiagonalise(torch.from_numpy(A), torch.from_numpy(mask),
                                   torch.from_numpy(q1), K)
  assert np.array_equal(out['idx'].cpu().numpy(), o64['idx'].numpy())
  eT = np.abs(o32['T'].numpy() - o64['T'].numpy()).max()
  eQ = np.abs(o32['Q'].numpy() - o64['Q'].numpy()).max()
  T, Q = out['T'].cpu().numpy(), out['Q'].cpu().numpy()
  assert np.abs(T - o64['T'].numpy()).max() <= max(4 * eT, 2e-5)
  assert np.abs(Q - o64['Q'].numpy()).max() <= max(4 * eQ, 2e-4)
  assert int(out['status'].sum()) == 0
  _check_ritz(out['theta'].cpu().numpy(), out['V'].cpu().numpy(), out['alpha'].cpu().numpy(),
              out['beta'].cpu().numpy(), Q, T)


def test_fused_lanczos_ritz_dense_operator_streams_and_agrees():
  """A dense operator does not fit the on-chip pool: the kernel streams its rows per iteration
  (status bit 1) and must agree with the packed path's arithmetic on the same matrix -- here
  checked against the fp64 oracle like every other case -- and with the two-kernel path."""
  rng = np.random.RandomState(5)
  for N, K, B in ((26, 20, 7), (96, 24, 3), (300, 16, 2)):
    M = rng.randn(B, N, N).astype(np.float32) / np.sqrt(N)
    A = ((M + M.transpose(0, 2, 1)) * 0.5).astype(np.float32)
    q1 = rng.randn(B, N).astype(np.float32)
    dA, dq = torch.from_numpy(A).to(dev()), torch.from_numpy(q1).to(dev())
    out = ops().lanczos_ritz(dA, None, dq, K)
    if N * N > 65535 or N > 26:
      assert int((out['status'] & 2).min()) == 2
    o64 = orc.lanczos_tridiagonalise(torch.from_numpy(A).double(), None, torch.from_numpy(q1).double(), K)
    o32 = orc.lanczos_tridiagonalise(torch.from_numpy(A), None, torch.from_numpy(q1), K)
    assert np.array_equal(out['idx'].cpu().numpy(), o64['idx'].numpy())
    eT = np.abs(o32['T'].numpy() - o64['T'].numpy()).max()
    T, Q = out['T'].cpu().numpy(), out['Q'].cpu().numpy()
    assert np.abs(T - o64['T'].numpy()).max() <= max(4 * eT, 2e-5)
    assert int((out['status'] & 1).sum()) == 0
    _check_ritz(out['theta'].cpu().numpy(), out['V'].cpu().numpy(), out['alpha'].cpu().numpy(),
                out['beta'].cpu().numpy(), Q, T)


def test_fused_lanczos_proper_mode_is_a_krylov_factorisation():
  """LNB_LANCZOS_PROPER (the online (D, V) provider's mode): Q has m = idx orthonormal columns,
  Q^T A Q = T_m (so the Ritz values are Rayleigh-Ritz values of A), exhausted Krylov spaces
  (n_b <= K, simple spectrum) reproduce the operator, and columns / entries past m are zero."""
  import bench
  rng = np.random.RandomState(31)
  B, N, K = 24, 30, 20
  A = np.zeros((B, N, N), np.float32)
  mask = np.zeros((B, N), np.uint8)
  sizes = rng.randint(3, N + 1, size=B)
  for b, n in enumerate(sizes):
    A[b, :n, :n] = bench.gnp_operator(rng, int(n), 0.3)
    mask[b, :n] = 1
  q1 = rng.randn(B, N).astype(np.float32)
  out = ops().lanczos_ritz(torch.from_numpy(A).to(dev()), torch.from_numpy(mask).to(dev()),
                           torch.from_numpy(q1).to(dev()), K, proper=True)
  idx = out['idx'].cpu().numpy()
  Q = out['Q'].cpu().numpy().astype(np.float64)
  T = out['T'].cpu().numpy().astype(np.float64)
  th = out['theta'].cpu().numpy().astype(np.float64)
  V = out['V'].cpu().numpy().astype(np.float64)
  assert np.all(idx >= 1) and np.all(idx <= np.minimum(sizes, K))
  beta = out['beta'].cpu().numpy().astype(np.float64)
  for b in range(B):
    m = idx[b]
    # fp32 Lanczos loses orthogonality like eps / beta_min at a near-breakdown step (betas down to the
    # 1e-4 acceptance threshold are kept): the stated tolerance scales accordingly
    bmin = beta[b, :m - 1].min() if m > 1 else 1.0
    tol = 2e-5 + 4e-6 / bmin
    np.testing.assert_allclose(Q[b].T @ Q[b], np.diag((np.arange(K) < m).astype(np.float64)), atol=tol)
    np.testing.assert_allclose(Q[b].T @ A[b].astype(np.float64) @ Q[b], T[b], atol=tol)
    assert np.all(T[b, m:, :] == 0) and np.all(Q[b][:, m:] == 0)
    lam = np.linalg.eigvalsh(A[b, :sizes[b], :sizes[b]].astype(np.float64))
    if m == sizes[b]:                    # Krylov space exhausted the graph: exact decomposition
      np.testing.assert_allclose((V[b] * th[b]) @ V[b].T, A[b], atol=2 * tol)
      np.testing.assert_allclose(np.sort(th[b, :m]), lam, atol=tol)
    elif m < K:                          # breakdown before K: invariant subspace -> exact eigenvalues
      for v in th[b, :m]:
        assert np.abs(lam - v).min() < 2 * tol
  assert (idx == np.minimum(sizes, K)).mean() > 0.5
  assert int((out['status'] & 1).sum()) == 0


def test_fused_lanczos_ritz_edges():
  """Empty batch, N = 1, N < K (zero padding), all-masked graph next to a full one, unsupported
  sizes refused loudly."""
  o = ops()
  z = o.lanczos_ritz(torch.zeros(0, 5, 5, device=dev()), None, torch.zeros(0, 5, device=dev()), 4)
  assert z['theta'].shape == (0, 4) and z['V'].shape == (0, 5, 4)
  one = o.lanczos_ritz(torch.full((2, 1, 1), 0.5, device=dev()), None, torch.ones(2, 1, device=dev()), 3)
  assert one['idx'].tolist() == [0, 0] or one['idx'].tolist() == [1, 1]
  ref = orc.lanczos_tridiagonalise(torch.full((2, 1, 1), 0.5), None, torch.ones(2, 1), 3)
  assert one['idx'].cpu().tolist() == ref['idx'].tolist()
  np.testing.assert_allclose(one['T'].cpu().numpy(), ref['T'].numpy(), atol=1e-6)
  rng = np.random.RandomState(8)
  N, K = 6, 10
  import bench
  A = np.stack([bench.gnp_operator(rng, N, 0.5) for _ in range(3)])
  mask = np.ones((3, N), np.uint8); mask[1, 4:] = 0
  A[1, 4:, :] = 0; A[1, :, 4:] = 0
  q1 = rng.randn(3, N).astype(np.float32)
  out = o.lanczos_ritz(torch.from_numpy(A).to(dev()), torch.from_numpy(mask).to(dev()),
                       torch.from_numpy(q1).to(dev()), K)
  r64 = orc.lanczos_tridiagonalise(torch.from_numpy(A).double(), torch.from_numpy(mask),
                                   torch.from_numpy(q1).double(), K)
  assert np.array_equal(out['idx'].cpu().numpy(), r64['idx'].numpy())
  np.testing.assert_allclose(out['T'].cpu().numpy(), r64['T'].numpy(), atol=2e-5)
  assert out['T'].shape == (3, K, K) and float(out['T'][:, N:, :].abs().sum()) == 0.0
  with pytest.raises(RuntimeError):
    o.lanczos_ritz(torch.zeros(1, 1100, 1100, device=dev()), None, torch.ones(1, 1100, device=dev()), 8)
  with pytest.raises(RuntimeError):
    o.lanczos_ritz(torch.zeros(1, 8, 8), None, torch.ones(1, 8), 4)          # CPU tensors: loud


@pytest.mark.parametrize('dense_filter', [True, False])
def test_graph_messages_one_launch_matches_bmm_composition(dense_filter):
  """lnb_graph_messages (whole message matrix of a general-shape layer in one launch) against the
  reference formulation in fp64: [L_0^k X] ++ [Q G_s Q^T X] ++ [L_e X] (model/lanczos_net.py:157-180,
  ada_lanczos_net.py:321-345), dense symmetric and diagonal filters, ragged feature widths."""
  rng = np.random.RandomState(3 + int(dense_filter))
  for B, N, E1, D, K, S, short in ((5, 26, 7, 128, 20, 5, [1, 2, 3]), (3, 32, 2, 70, 32, 8, []),
                                   (4, 9, 16, 10, 8, 1, [2, 5]), (2, 17, 3, 33, 4, 0, [1])):
    L = (rng.randn(B, N, N, E1) * (rng.rand(B, N, N, E1) < 0.3) / 3).astype(np.float32)
    X = rng.randn(B, N, D).astype(np.float32)
    Q = rng.randn(B, N, K).astype(np.float32) / np.sqrt(N)
    if dense_filter:
      G = rng.randn(B, S, K, K).astype(np.float32)
      filt = ((G + G.transpose(0, 1, 3, 2)) * 0.5).astype(np.float32)
    else:
      filt = rng.randn(B, K, S).astype(np.float32)
    C = len(short) + S + E1
    out = torch.full((B, N, C * D + 3), 7.0, device=dev())[:, :, :C * D].contiguous()   # any row stride
    o = ops()
    o.graph_messages(torch.from_numpy(L).to(dev()), torch.from_numpy(X).to(dev()),
                     torch.from_numpy(Q).to(dev()) if S else None,
                     torch.from_numpy(filt).to(dev()) if S else None, dense_filter, short, out)
    L64, X64, Q64 = L.astype(np.float64), X.astype(np.float64), Q.astype(np.float64)
    blocks, walk = [], X64
    for step in range(1, (max(short) if short else 0) + 1):
      walk = np.einsum('bnm,bmd->bnd', L64[..., 0], walk)
      if step in short:
        blocks.append(walk)
    U = np.einsum('bnk,bnd->bkd', Q64, X64)
    for s_ in range(S):
      Wk = np.einsum('bkj,bjd->bkd', filt[:, s_].astype(np.float64), U) if dense_filter else \
          filt[:, :, s_].astype(np.float64)[:, :, None] * U
      blocks.append(np.einsum('bnk,bkd->bnd', Q64, Wk))
    for e in range(E1):
      blocks.append(np.einsum('bnm,bmd->bnd', L64[..., e], X64))
    ref = np.concatenate(blocks, axis=2)
    np.testing.assert_allclose(out.cpu().numpy(), ref, rtol=2e-5, atol=2e-5 * max(1.0, np.abs(ref).max()))
  with pytest.raises(RuntimeError):
    ops().graph_messages(torch.zeros(1, 40, 40, 2, device=dev()), torch.zeros(1, 40, 8, device=dev()),
                         None, None, False, [], torch.zeros(1, 40, 16, device=dev()))


def test_tridiag_powers_and_symmetrize():
  g = load_golden('ada_lanczos_layer.npz')
  T = torch.from_numpy(g['qm8_T'])
  powers = [5, 7, 10, 20, 30]
  out = ops().tridiag_powers(T.to(dev()), powers).cpu()          # [B,K,S,K]
  ref = torch.stack(orc.tridiag_power_stack(T.double(), powers), dim=2)   # [B,K,S,K]
  np.testing.assert_allclose(out.numpy(), ref.numpy(), rtol=2e-5, atol=1e-7)
  B, K, S = 3, 8, 5
  Y = torch.randn(B, K * K * S)
  G = ops().symmetrize_filters(Y.to(dev()), K, S).cpu()
  Y4 = Y.reshape(B, K, K, S)
  ref = ((Y4 + Y4.transpose(1, 2)) * 0.5).permute(0, 3, 1, 2)
  assert torch.equal(G, ref.contiguous())


# ------------------------------------------------------------------------------------------
# fused spectral convolution layer (tcgen05, messages produced on-chip)
# ------------------------------------------------------------------------------------------
def _conv_case(B, N, Din, H, K, S, E1, seed, molecular=True):
  rng = np.random.RandomState(seed)
  L = np.zeros((B, N, N, E1), np.float32)
  V = np.zeros((B, N, K), np.float32)
  sizes = rng.randint(max(2, N // 4), N + 1, size=B)
  sizes[0] = N
  for b, n in enumerate(sizes):
    if molecular:
      from lanczosnetwork_b200 import data
      _, adjs = data.synthetic_molecule(rng, n, num_bond_type=E1 - 1)
      L[b, :n, :n, 0] = data.get_laplacian(adjs.sum(axis=2))
      for e in range(E1 - 1):
        L[b, :n, :n, 1 + e] = data.get_laplacian(adjs[:, :, e])
    else:
      L[b, :n, :n] = rng.randn(n, n, E1) * (rng.rand(n, n, E1) < 0.5)
    kk = min(K, n)
    V[b, :n, :kk] = np.linalg.qr(rng.randn(n, n))[0][:, :kk]
  X = rng.randn(B, N, Din).astype(np.float32)
  coeff = rng.randn(B, K, S).astype(np.float32)
  W = (rng.randn(H, (S + E1) * Din) / np.sqrt((S + E1) * Din)).astype(np.float32)
  bias = rng.randn(H).astype(np.float32)
  return [torch.from_numpy(a) for a in (X, L, V, coeff, W, bias)]


@pytest.mark.parametrize('B,N,Din,H,molecular', [
    (10, 26, 64, 128, True), (9, 26, 128, 128, True), (4, 32, 128, 128, True),
    (1, 5, 32, 128, True), (7, 40, 128, 128, True), (3, 100, 128, 128, False),
    (5, 26, 128, 64, True), (300, 26, 128, 128, True)])
def test_spectral_conv_fused_matches_fp64_and_unfused(B, N, Din, H, molecular):
  from lanczosnetwork_b200 import spectral_conv as sc
  K, S, E1 = 20, 8, 7
  X, L, V, coeff, W, bias = _conv_case(B, N, Din, H, K, S, E1, B * 1000 + N + Din, molecular)
  # fp64 reference of one layer: msgs = [V diag(f_s) V^T X] ++ [L_e X]; relu(cat W^T + b)
  Xd, Ld, Vd, fd = X.double(), L.double(), V.double(), coeff.double()
  msgs = [torch.bmm(torch.bmm(Vd * fd[:, :, s].unsqueeze(1), Vd.transpose(1, 2)), Xd) for s in range(S)]
  msgs += [torch.bmm(Ld[..., e], Xd) for e in range(E1)]
  ref = torch.relu(torch.cat(msgs, dim=2) @ W.double().t() + bias.double())
  d = dev()
  Xg, Lg, Vg, cg, Wg, bg = [t.to(d) for t in (X, L, V, coeff, W, bias)]
  assert ops().fused_conv_supported(N, Din, K, H, 0, False, S, E1)
  prep = ops().graph_prepare(Lg, Vg)
  # the compression is exact: rebuilding dense rows from the ELL lists returns L bit-for-bit
  ell_val, ell_idx, ell_max, gext, tiles = [t.cpu() for t in prep]
  for b in range(min(B, 3)):
    for e in range(E1):
      dense = torch.zeros(N, N)
      for t in range(int(ell_max[b, e])):
        dense[torch.arange(N), ell_idx[b, e, t].long()] += ell_val[b, e, t]
      assert torch.equal(dense, L[b, :, :, e])
  # packed tiles: consecutive graph ranges covering [0, B) within the row / Ritz-row budgets
  T = int(tiles[0])
  starts = tiles[1:T + 2].tolist()
  assert starts[0] == 0 and starts[-1] == B and all(a < b for a, b in zip(starts, starts[1:]))
  # next-fit: a tile is closed only because the next graph would not fit
  for a, b in zip(starts[:-1], starts[1:-1]):
    assert (b - a == 32 or int(gext[a:b + 1, 0].sum()) > 128 or
            int(((gext[a:b + 1, 1] + 3) // 4 * 4).sum()) > 128)
  for a, b in zip(starts, starts[1:]):
    assert b - a <= 32 and int(gext[a:b, 0].sum()) <= 128
    assert int(((gext[a:b, 1] + 3) // 4 * 4).sum()) <= 128
  w_hi, w_lo = ops().split_tf32(Wg)
  out = ops().spectral_conv_fused(Xg, Vg, cg, prep, w_hi, w_lo, bg, True)
  cache = sc.WeightCache()
  unf = sc.graph_conv_layer_unfused(Xg, Lg, Vg, cg, False, [], S, Wg, bg, cache, 'w')
  scale = ref.abs().max().item()
  e_f = (out.double().cpu() - ref).abs().max().item()
  e_u = (unf.double().cpu() - ref).abs().max().item()
  assert e_f <= 8e-6 * scale + 1e-6, (e_f, e_u, scale)   # ~K/8 truncating accumulation steps
  assert e_u <= 8e-6 * scale + 1e-6, (e_f, e_u, scale)


def test_linear_grouped_block_diagonal():
  g = torch.Generator().manual_seed(5)
  M, G, N, K = 700, 7, 128, 128
  x = torch.randn(M, G * K, generator=g).to(dev())
  w = (torch.randn(G * N, K, generator=g) / np.sqrt(K)).to(dev())
  b = torch.randn(G * N, generator=g).to(dev())
  w_hi, w_lo = ops().split_tf32(w)
  out = ops().linear_tf32x3_grouped(x, w_hi, w_lo, b, G, True)
  ref = torch.cat([torch.relu(x[:, i * K:(i + 1) * K].double() @ w[i * N:(i + 1) * N].double().t()
                              + b[i * N:(i + 1) * N].double()) for i in range(G)], dim=1)
  assert (out.double() - ref).abs().max().item() <= 6e-6 * ref.abs().max().item()
  # narrow groups (the last MLP stage: 8 outputs per layer)
  N2 = 8
  w2 = (torch.randn(G * N2, K, generator=g) / np.sqrt(K)).to(dev())
  b2 = torch.randn(G * N2, generator=g).to(dev())
  h2, l2 = ops().split_tf32(w2)
  out2 = ops().linear_tf32x3_grouped(x, h2, l2, b2, G, False)
  ref2 = torch.cat([x[:, i * K:(i + 1) * K].double() @ w2[i * N2:(i + 1) * N2].double().t()
                    + b2[i * N2:(i + 1) * N2].double() for i in range(G)], dim=1)
  assert out2.shape == (M, G * N2)
  assert (out2.double() - ref2).abs().max().item() <= 6e-6 * ref2.abs().max().item()


def test_filter_mlp_chain_matches_fp64():
  """All layers' Ritz-filter MLPs in one kernel vs an fp64 evaluation, with and without the
  compact row list."""
  from lanczosnetwork_b200 import spectral_conv as sc
  g = torch.Generator().manual_seed(11)
  B, K, S, Hd, L = 37, 20, 8, 128, 3
  D = (torch.rand(B, K, generator=g) * 2 - 1)
  keff = torch.randint(0, K + 1, (B,), generator=g)
  for b in range(B):
    D[b, keff[b]:] = 0
  layers, ref_w = [], []
  for l in range(L):
    dims = [(Hd, S), (Hd, Hd), (Hd, Hd), (S, Hd)]
    ps = []
    for i, (o, k) in enumerate(dims):
      w = (torch.randn(o, k, generator=g) / np.sqrt(k)).to(dev())
      b_ = (torch.randn(o, generator=g) * 0.1).to(dev())
      ps.append(('l%d.%d' % (l, i), w, b_))
    layers.append(ps)
  powers = [1, 2, 3, 5, 7, 10, 20, 30]
  table = ops().ritz_power_table(D.to(dev()), powers)
  ref = []
  for ps in layers:
    h = table.reshape(B * K, S).double()
    for i, (_, w, b_) in enumerate(ps):
      h = h @ w.double().t() + b_.double()
      if i < 3:
        h = torch.relu(h)
    ref.append(h.reshape(B, K, S))
  cache = sc.WeightCache()
  out, _ = sc.ritz_filter_coefficients(D.to(dev()), powers, layers, cache)
  for l in range(L):
    err = (out[l].double() - ref[l]).abs().max().item()
    assert err <= 5e-6 * ref[l].abs().max().item() + 1e-6, (l, err)
  gext = torch.stack([torch.full((B,), 5), keff], dim=1).int().to(dev())
  rowmap, nrows = ops().ritz_rowmap(gext, K)
  assert int(nrows) == int(keff.sum())
  want = torch.cat([torch.arange(int(keff[b])) + b * K for b in range(B)]).int()
  assert torch.equal(rowmap[:int(nrows)].cpu(), want)
  out2, _ = sc.ritz_filter_coefficients(D.to(dev()), powers, layers, cache, gext)
  for l in range(L):
    for b in range(B):
      kk = int(keff[b])
      assert torch.equal(out2[l][b, :kk], out[l][b, :kk])


@pytest.mark.parametrize('N,K,B', [(200, 40, 5), (256, 40, 3), (129, 20, 4), (33, 40, 9), (100, 70, 3)])
def test_lanczos_tridiag_mid_sizes_and_fallback_vs_oracle(N, K, B):
  """lnb_lanczos_tridiag above the QM8 size (the fused kernel without its QL stage; K = 70 > 64 takes
  the CTA-per-graph fallback) against the fp64 oracle with the fp32 oracle's own error as the
  yardstick (no reference output exists at these sizes in the goldens)."""
  import networkx as nx
  from lanczosnetwork_b200 import data
  rng = np.random.RandomState(N + K)
  A = np.zeros((B, N, N), np.float32)
  mask = np.zeros((B, N), np.uint8)
  for b in range(B):
    n = N if b == 0 else int(rng.randint(N // 2, N + 1))
    g = nx.fast_gnp_random_graph(n, min(0.5, 8.0 / n), seed=int(rng.randint(10 ** 6)))
    A[b, :n, :n] = data.get_laplacian(np.asarray(nx.to_numpy_array(g)))
    mask[b, :n] = 1
  q1 = rng.randn(B, N).astype(np.float32)
  out = ops().lanczos_tridiag(torch.from_numpy(A).to(dev()), torch.from_numpy(mask).to(dev()),
                              torch.from_numpy(q1).to(dev()), K)
  o64 = orc.lanczos_tridiagonalise(torch.from_numpy(A).double(), torch.from_numpy(mask),
                                   torch.from_numpy(q1).double(), K)
  o32 = orc.lanczos_tridiagonalise(torch.from_numpy(A), torch.from_numpy(mask),
                                   torch.from_numpy(q1), K)
  assert np.array_equal(out['idx'].cpu().numpy(), o64['idx'].numpy())
  eT = np.abs(o32['T'].numpy() - o64['T'].numpy()).max()
  eQ = np.abs(o32['Q'].numpy() - o64['Q'].numpy()).max()
  assert np.abs(out['T'].cpu().numpy() - o64['T'].numpy()).max() <= max(4 * eT, 2e-5)
  assert np.abs(out['Q'].cpu().numpy() - o64['Q'].numpy()).max() <= max(4 * eQ, 2e-4)


def test_spectral_stack_equals_layer_by_layer():
  """The one-kernel stack (state kept in shared memory across layers, embedding gather in front,
  readout behind) reproduces the per-layer fused kernel bit-for-bit and the readout kernel to
  rounding."""
  from lanczosnetwork_b200 import spectral_conv as sc
  B, N, K, S, E1, H, L = 37, 26, 20, 8, 7, 128, 3
  X, Lop, V, coeff, W, bias = _conv_case(B, N, 64, H, K, S, E1, 4242, True)
  d = dev()
  g = torch.Generator().manual_seed(3)
  ids = torch.randint(0, 70, (B, N), generator=g)
  emb = torch.randn(70, 64, generator=g)
  dins = [64, H, H]
  Ws = [(torch.randn(H, (S + E1) * dd, generator=g) / np.sqrt((S + E1) * dd)).to(d) for dd in dins]
  bs = [torch.randn(H, generator=g).to(d) for _ in dins]
  coeffs = torch.randn(L, B, K, S, generator=g).to(d)
  Lg, Vg = Lop.to(d), V.to(d)
  prep = ops().graph_prepare(Lg, Vg)
  # layer by layer through the single-layer entry point
  state = emb.to(d)[ids.to(d)]
  for l in range(L):
    hi, lo = ops().split_tf32(Ws[l])
    state = ops().spectral_conv_fused(state, Vg, coeffs[l], prep, hi, lo, bs[l], True, write_pad=True)
  cache = sc.WeightCache()
  kw = (S + E1) * H
  w_hi, w_lo, ball = cache.split_conv_stack('t', Ws, bs, kw)
  mask = (torch.arange(N)[None, :] < torch.randint(1, N + 1, (B, 1), generator=g)).to(torch.uint8).to(d)
  W_out, b_out = torch.randn(16, H, generator=g).to(d) * 0.1, torch.randn(16, generator=g).to(d)
  w_att, b_att = torch.randn(H, generator=g).to(d) * 0.1, torch.randn(1, generator=g).to(d)
  st, score = ops().spectral_stack_forward(prep, Vg, w_hi, w_lo, ball, dins, H, S, coeff=coeffs,
                                           coeff_stride=coeffs.stride(0), node_ids=ids.to(d),
                                           emb=emb.to(d), want_state=True,
                                           readout=(W_out, b_out, w_att, b_att), mask=mask)
  assert torch.equal(st, state)
  ref = ops().readout(state, W_out, b_out, w_att, b_att, mask)
  torch.testing.assert_close(score, ref, rtol=1e-5, atol=1e-6)
  # no mask: mean over all N nodes, padded ones included
  _, score2 = ops().spectral_stack_forward(prep, Vg, w_hi, w_lo, ball, dins, H, S, coeff=coeffs,
                                           coeff_stride=coeffs.stride(0), X=emb.to(d)[ids.to(d)],
                                           readout=(W_out, b_out, w_att, b_att), mask=None)
  torch.testing.assert_close(score2, ops().readout(state, W_out, b_out, w_att, b_att, None),
                             rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize('cheby', [False, True])
def test_operator_chain_matches_step_by_step(cheby):
  """lnb_operator_chain (power chain of model/dcnn.py:88-92, Chebyshev chain of
  model/cheby_net.py:88-93) against the step-by-step fp64 recurrence."""
  B, N, D, E1, steps = 9, 26, 160, 3, 12
  g = torch.Generator().manual_seed(77 + int(cheby))
  L = torch.randn(B, N, N, E1, generator=g) * (torch.rand(B, N, N, E1, generator=g) < 0.2) / 3
  X = torch.randn(B, N, D, generator=g)
  sel = [-1 if s % 3 == 1 else s for s in range(steps)]       # some steps are not stored
  out = torch.full((B, N, (2 + steps) * D), 7.0).to(dev())
  ops().operator_chain(L.to(dev()), X.to(dev()), steps, sel, out, 2, chebyshev=cheby)
  L0 = L[..., 0].double()
  prev2, cur, ref = X.double(), X.double(), []
  for s in range(steps):
    nxt = torch.bmm(L0, cur)
    if cheby and s > 0:
      nxt = 2.0 * nxt - prev2
    prev2, cur = cur, nxt
    ref.append(nxt)
  got = out.cpu().double()
  assert torch.all(got[:, :, :2 * D] == 7.0)                   # blocks in front untouched
  for s in range(steps):
    blk = got[:, :, (2 + s) * D:(3 + s) * D]
    if sel[s] < 0:
      assert torch.all(blk == 7.0)
    else:
      scale = ref[s].abs().max().item()
      assert (blk - ref[s]).abs().max().item() <= 2e-6 * max(1.0, scale) * (s + 1), s
