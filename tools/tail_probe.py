import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vqa_b200.model import VQAModel
from vqa_b200.synth import synth_batch
torch.manual_seed(0)
for kw in (dict(), dict(use_se_attention=False, use_spatial_attention=False)):
    m = VQAModel(**kw).eval().cuda()
    _, img, ids, mask = synth_batch(256, 1, full_length=True)
    img, ids, mask = img.cuda(), ids.cuda(), mask.cuda()
    eng = m.engine()
    with torch.no_grad():
        for _ in range(2): m(img, ids, mask)
    prog, plan = eng.plan_for(256, 20, "nchw_f32", 1, False, 0)
    logits = torch.empty(256, 1000, device="cuda")
    ext = [img.data_ptr(), ids.data_ptr(), mask.data_ptr(), logits.data_ptr(), 0, 0]
    st = torch.cuda.current_stream().cuda_stream
    for k, op in enumerate(prog.ops):
        if op.kind != "stage_tail": continue
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(3): plan.run(ext, st, k, k + 1)
        torch.cuda.synchronize(); a.record()
        for _ in range(10): plan.run(ext, st, k, k + 1)
        b.record(); torch.cuda.synchronize()
        print(kw, op.name, "CS", op.i["CS"], f"{a.elapsed_time(b) / 10 * 1000:.1f} us")
