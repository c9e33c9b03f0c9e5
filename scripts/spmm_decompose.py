"""Times the packed page kernel at config-2 conv size (DEG, PAGES and F from the environment)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from gnn_tableextraction_b200 import _lib, ops
DEV = "cuda"
PAGE, deg, pages, f = 300, int(os.environ.get("DEG", "10")), int(os.environ.get("PAGES", "1666")), int(os.environ.get("F", "218"))
n, e = PAGE * pages, PAGE * pages * deg
gen = torch.Generator(device=DEV).manual_seed(0)
indptr = (torch.arange(n + 1, device=DEV, dtype=torch.int64) * deg).to(torch.int32)
base = (torch.arange(n, device=DEV, dtype=torch.int32) // PAGE * PAGE).repeat_interleave(deg)
idx = (torch.randint(0, PAGE, (e,), device=DEV, generator=gen, dtype=torch.int32) + base).contiguous()
w = torch.rand(e, device=DEV, generator=gen)
norm = ops.degree_norm(indptr)
page_off = torch.arange(pages + 1, device=DEV, dtype=torch.int32) * PAGE
pg = (page_off, pages, PAGE, PAGE * deg)
x = ops.empty_padded(n, f, DEV); x.normal_(generator=gen)
add = ops.empty_padded(n, f, DEV); add.normal_(generator=gen)
y = ops.empty_padded(n, f, DEV)
pk = ops.paged_pack_edges(indptr, idx, w, pg)
def t(fn, it=20):
    for _ in range(3): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(it): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / it
a = t(lambda: ops.spmm_packed(indptr, pk, x, pg, mode=_lib.GTE_AGG_SUM_NORM, row_norm=norm, out=y))
b = t(lambda: ops.spmm_packed(indptr, pk, x, pg, mode=_lib.GTE_AGG_SUM, addend=add, out=y))
c = t(lambda: y.copy_(x))
print(f"pages={pages} deg={deg} f={f}: fwd {a*1e3:.1f} us, with addend {b*1e3:.1f} us, torch copy x->y {c*1e3:.1f} us")
