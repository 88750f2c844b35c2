import ctypes as C, os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from recommender_tensorflow_b200 import _lib
lib = _lib.load()
for (M, N, K) in [(65536, 256, 384), (65536, 128, 256), (65536, 256, 128), (65536, 384, 256)]:
    A = torch.randn(M, K, device="cuda"); B = torch.randn(N, K, device="cuda"); Cc = torch.empty(M, N, device="cuda")
    rc = lib.dfm_test_tc_gemm(2, C.c_void_p(A.data_ptr()), C.c_void_p(B.data_ptr()), C.c_void_p(Cc.data_ptr()), M, N, K, 1)
    assert rc == 0, rc
