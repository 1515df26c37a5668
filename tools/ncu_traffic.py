"""profiles/r02_traffic.json + a text summary from one `ncu --set full` capture of a block forward
(tools/profile_block.py): per stage of dn_block_fwd the DRAM bytes (read + write) of its kernel, duration, tensor-pipe
activity and cache hit rates.  bench.py reads the json for `roofline.traffic`.

    python tools/ncu_traffic.py gpurun_out/r02_block.ncu-rep profiles/r02_traffic.json > profiles/r02_ncu_full_summary.txt
"""
import csv, json, subprocess, sys
rep, out_json = sys.argv[1], sys.argv[2]
raw = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
rows = list(csv.reader(raw.splitlines()))
hdr, units = rows[0], rows[1]
ix = {h: i for i, h in enumerate(hdr)}
# launch sequence of dn_block_fwd at C = 128 with the tensor-core gradient features; for a capture of the commuted
# route (C_width != 128, no rotations, the bf16 engine, patched operators) pass "commuted" as third argument
STAGE = [("to_basis_kernel", "to_basis"), ("pack_weights_kernel", "pack_weights"), ("rows_chain", "from_basis_pq"),
         ("spmm_gxy", "grad_gather_x"), ("rows_chain", "grad_dots_gemm"), ("rows_chain", "grad_dots_gemm_2"), ("rows_chain", "mlp")]
if len(sys.argv) > 3 and sys.argv[3] == "commuted":
    STAGE = [("to_basis_kernel", "to_basis"), ("pack_weights_kernel", "pack_weights"), ("rows_chain", "from_basis_pq"),
             ("spmm_features", "grad_features_gather"), ("rows_chain", "mlp")]
def val(r, name, scale=None):
    v = float(r[ix[name]].replace(",", ""))
    u = units[ix[name]]
    if scale == "bytes":
        v *= {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}[u]
    if scale == "us":
        v *= {"ns": 1e-3, "us": 1, "ms": 1e3, "s": 1e6}.get(u, 1)   # ncu's "us" column may print as "us" or "usecond"
    return v
traffic, k = {}, 0
for r in rows[2:]:
    name = r[ix["Kernel Name"]]
    if k >= len(STAGE) or STAGE[k][0] not in name:
        continue
    stage = STAGE[k][1]; k += 1
    rd, wr = val(r, "dram__bytes_read.sum", "bytes"), val(r, "dram__bytes_write.sum", "bytes")
    us = val(r, "gpu__time_duration.sum", "us")
    tens = val(r, "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active")
    traffic[stage] = rd + wr
    traffic[stage + "_detail"] = {"kernel": name.split("(")[0].split("::")[-1], "dram_read_mb": rd / 1e6, "dram_write_mb": wr / 1e6,
                                  "us_under_ncu": us, "tensor_pipe_active_pct": tens,
                                  "dram_throughput_pct": val(r, "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed"),
                                  "l1_hit_pct": val(r, "l1tex__t_sector_hit_rate.pct"), "l2_hit_pct": val(r, "lts__t_sector_hit_rate.pct"),
                                  "issue_active_pct": val(r, "smsp__issue_active.avg.pct_of_peak_sustained_active"),
                                  "registers": val(r, "launch__registers_per_thread")}
    d = traffic[stage + "_detail"]
    print("{:22s} {:28s} {:7.1f} us  DRAM {:6.1f}+{:6.1f} MB ({:4.1f} % of peak)  tensor pipe {:4.1f} %  L1 hit {:4.1f} %  L2 hit {:4.1f} %  issue {:4.1f} %  regs {}".format(
        stage, d["kernel"], us, d["dram_read_mb"], d["dram_write_mb"], d["dram_throughput_pct"], tens, d["l1_hit_pct"], d["l2_hit_pct"],
        d["issue_active_pct"], int(d["registers"])))
json.dump(traffic, open(out_json, "w"), indent=1)
