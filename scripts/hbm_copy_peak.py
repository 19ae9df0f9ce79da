"""HBM copy bandwidth of one GPU, the roofline peak bench.py divides by (HBM_PEAK_GBS):

    python scripts/hbm_copy_peak.py > profiles/hbm_copy_peak_b200.txt

torch copy_ of 1 Gi bf16 elements (2 GiB, far larger than the 126 MB L2) into a second buffer, CUDA-event
timed over 50 copies after 5 warm-up copies, three times; bytes counted = read + write.  The card's name and
power limit are printed with the numbers because the rate depends on them."""
import subprocess

import torch

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                      str(torch.cuda.current_device())], capture_output=True, text=True)
print("gpu:", smi.stdout.strip() or torch.cuda.get_device_name())
x = torch.empty(1 << 30, dtype=torch.bfloat16, device="cuda")
y = torch.empty_like(x)
for _ in range(5):
    y.copy_(x)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
for _ in range(3):
    e0.record()
    for _ in range(50):
        y.copy_(x)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 50
    print(f"copy 2 GiB bf16: {ms:.3f} ms -> {2 * x.numel() * x.element_size() / ms / 1e6:.1f} GB/s (read + write)")
