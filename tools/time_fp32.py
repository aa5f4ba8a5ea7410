"""CP pass in precision="fp32": linear layers on the tensor cores (bf16 hi / lo split).
Usage: python tools/time_fp32.py [batch]"""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
dev = torch.device("cuda", 0)
B = int(sys.argv[1]) if len(sys.argv) > 1 else 8192
model, _ = bench.make_model(dev, precision="fp32")
img, txt, mask, text, cand, _ = bench.make_cp_inputs(B, dev, 1000)
enc = {"image_embeddings": img, "text_embeddings": txt}
for _ in range(2):
    p = model.score_cp(outfit_mask=mask, encoder_input_dict=enc)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(3):
    p = model.score_cp(outfit_mask=mask, encoder_input_dict=enc)
e1.record(); torch.cuda.synchronize()
print(f"fp32 cp pass ms {e0.elapsed_time(e1) / 3:.3f}  ({B / (e0.elapsed_time(e1) / 3) * 1e3:,.0f} outfits/s)  probs[:4] {p[:4].tolist()}")
