import sys, time, ctypes; sys.path.insert(0, __import__('os').path.dirname(__import__('os').path.dirname(__import__('os').path.abspath(__file__))))
import torch, tneq_b200
from tneq_b200 import _lib
lib = _lib.load()
dev = torch.device('cuda:0')
def gemm_time(M,N,K,nb=1,iters=5):
    A = torch.randn(nb,M,K,device=dev); B = torch.randn(nb,N,K,device=dev); C = torch.empty(nb,M,N,device=dev)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    def run():
        _lib.check(lib.tnq_gemm_tf32x3(ctypes.c_void_p(A.data_ptr()), ctypes.c_void_p(B.data_ptr()), ctypes.c_void_p(C.data_ptr()), M,N,K,K,K,N,nb,M*K,N*K,M*N,0,st))
    for _ in range(2): run()
    torch.cuda.synchronize()
    e0,e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters): run()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)/iters
    print(f"gemm M={M} N={N} K={K} nb={nb}: {ms:.3f} ms  {2*M*N*K*nb/ms/1e9:.1f} TFLOP/s fp32-equivalent ({3*2*M*N*K*nb/ms/1e9:.1f} issued TF32)")
gemm_time(16384,8192,128); gemm_time(8192,8192,8192); gemm_time(16384,128,8192); gemm_time(8192,128,128,nb=256)
torch.backends.cuda.matmul.allow_tf32=False
a=torch.randn(8192,8192,device=dev); b=torch.randn(8192,8192,device=dev)
for tf in (False, True):
    torch.backends.cuda.matmul.allow_tf32=tf
    for _ in range(2): a@b
    torch.cuda.synchronize(); e0,e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); 
    for _ in range(5): a@b
    e1.record(); torch.cuda.synchronize(); print('cublas 8192^3 tf32' if tf else 'cublas 8192^3 fp32', 2*8192**3*5/e0.elapsed_time(e1)/1e9, 'TFLOP/s')
del a,b
# cfg4 probe: python tools/cfg4_probe.py [chi] [B] [dtype: complex64 | complex128]
chi = int(sys.argv[1]) if len(sys.argv)>1 else 64
n, B = 16, int(sys.argv[2]) if len(sys.argv)>2 else 256
dtype = sys.argv[3] if len(sys.argv)>3 else 'complex64'
cdt = getattr(torch, dtype)
print('cfg4 probe:', torch.cuda.get_device_name(dev), 'n', n, 'chi', chi, 'B', B, dtype)
be = tneq_b200.BackendFactory.create_backend('b200', device='cuda:0', dtype=dtype)
eng = tneq_b200.EngineSiamese(backend=be, strategy_mode='balanced', mx_K=chi)
g = tneq_b200.QCTNHelper.generate_example_graph(n=n, graph_type='mps', dim_char=str(chi))
torch.manual_seed(0)
t=time.time(); q = tneq_b200.QCTN(g, backend=be); torch.cuda.synchronize(); print('qctn init', time.time()-t)
for c in q.cores: q.cores_weights[c].requires_grad_(True)
st = [torch.zeros(chi, device=dev, dtype=cdt) for _ in range(n)]
for s in st: s[-1]=1
eye = torch.eye(chi, dtype=cdt, device=dev).expand(B,chi,chi)
out = eng.contract_with_compiled_strategy(q, st, [eye]*n); torch.cuda.synchronize()
print('KAT-1 identity measurement -> ', out[:4], 'max dev from 1:', (out-1).abs().max().item())
x = torch.randn(B,n, device=dev)*0.3
mx,_ = eng.generate_data(x, K=chi, ret_type='TNTensor')
for it in range(4):
    torch.cuda.synchronize(); t=time.time()
    l0 = _lib.launch_count()
    loss, grads = eng.contract_with_compiled_strategy_for_gradient(q, st, mx)
    torch.cuda.synchronize(); dt=time.time()-t
    fn = eng._compiled(q, st, mx, True, 'symmetric'); r = next(iter(fn.plans.values())).gemm_runner('bwd')
    print(f'train step {it}: {dt*1e3:.1f} ms  loss {loss.item():.4f}  launches {_lib.launch_count()-l0}  gemm flops so far {r.flops:.3e}  mem {torch.cuda.max_memory_allocated()/2**30:.1f} GiB', flush=True)
print('grad norms', [round(g_.abs().max().item(),6) for g_ in grads[:3]])
