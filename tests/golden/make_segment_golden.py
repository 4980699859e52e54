"""Record outputs of the reference's OWN segment-reduction CUDA kernels
(operators/src/cuda/segment_reduction.cu:39-95), compiled by oracle/build_ref.py into oracle/_ref/.

    python oracle/build_ref.py                          # where the reference checkout is present
    python tests/golden/make_segment_golden.py          # on a CUDA device; writes segment_reduction_ref.npz

Cases lie on the domain where the reference is self-consistent (num_segments == dim1, its hard-coded
output batch stride dim1*dim2, segment_reduction.cu:48).  Data are integer-valued, so fp32 atomic sums
are exact in any order and the stored outputs are bit-exact.  tests/test_gpu_kernels.py compares the
product's kernels and the oracle's ``ref_cuda`` flavour with them.
"""
import ctypes
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
LIB = os.path.join(ROOT, 'oracle', '_ref', 'libsegment_reduction_ref.so')
SHAPES = ((3, 6, 4), (5, 33, 16), (1, 1, 1), (2, 70, 7))


def main(out_path):
  ref = ctypes.CDLL(LIB)
  fwd = ref.unsorted_segment_sum_forward_gpu_kernel_launcher
  bwd = ref.unsorted_segment_sum_backward_gpu_kernel_launcher
  for f in (fwd, bwd):
    f.restype = None
    f.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.POINTER(ctypes.c_int),
                  ctypes.c_void_p]
  dev = torch.device('cuda:0')
  stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
  rng = np.random.RandomState(11)
  arrays = {'shapes': np.array(SHAPES, dtype=np.int64)}
  for i, (B, C, X) in enumerate(SHAPES):
    data = rng.randint(-8, 9, size=(B, C, X)).astype(np.float32)
    seg = rng.randint(0, C, size=(B, C)).astype(np.int64)
    gout = rng.randn(B, C, X).astype(np.float32)
    d_data, d_seg, d_gout = (torch.from_numpy(a).to(dev) for a in (data, seg, gout))
    shape = (ctypes.c_int * 3)(B, C, X)
    out = torch.zeros(B, C, X, device=dev)
    fwd(stream, d_data.data_ptr(), d_seg.data_ptr(), shape, out.data_ptr())
    grad = torch.zeros(B, C, X, device=dev)
    bwd(stream, d_gout.data_ptr(), d_seg.data_ptr(), shape, grad.data_ptr())
    torch.cuda.synchronize()
    arrays.update({'c%d_data' % i: data, 'c%d_seg' % i: seg, 'c%d_out' % i: out.cpu().numpy(),
                   'c%d_gout' % i: gout, 'c%d_grad' % i: grad.cpu().numpy()})
  np.savez_compressed(out_path, **arrays)
  print('%s %.1f KB' % (out_path, os.path.getsize(out_path) / 1024.0))


if __name__ == '__main__':
  main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, 'segment_reduction_ref.npz'))
