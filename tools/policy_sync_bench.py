"""Cost of the squashed head's weight sync (SquashedGaussianPolicy.sync_weights) on the routes a SAC / TQC learner can take,
per call and inside a collect / learn loop.

    python tools/policy_sync_bench.py [--out profiles/<name>.json]

6DoF shapes (obs 9, act 6), bf16 and fp32 handles.  The learner's parameters are fp32 CUDA tensors.

* Per call, three routes, alternating round by round after a warm-up:
  - "state_dict": load_state_dict(actor.state_dict()) from the CUDA tensors, the route before the device path existed:
    host copies of the ten tensors, the host entry (staging copy, packing kernel, synchronise);
  - "host_entry": sync_weights() of a policy that holds CPU tensors (the host entry alone);
  - "device": sync_weights() of a policy that shares the CUDA tensors (load_state_dict(share=True)): host wall time per
    call (the enqueue; the call does not wait for the device), and the packing kernel's device time from CUDA events
    around the replay of a CUDA graph of 100 calls.
  Host wall times end in a device synchronise for the two synchronising routes.
* SAC-shaped collection loop at 131 072 environments on the 6DoF set-point env, T = 128 steps of (act, env.step_async,
  an in-place parameter update standing in for optimizer.step(), sync): env-steps/s for "state_dict" (eager), "device"
  (eager) and "device_graph" (the whole T-step loop captured as one CUDA graph), next to the rate without any update or
  sync ("no_sync", eager and as a graph: the ceiling).  The variants alternate round by round; medians of the rounds.

Prints one JSON line (with the device name, power limit and max SM clock, read with a read-only nvidia-smi query) and
writes it to --out when given."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info(index):
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, clock = [s.strip() for s in q.split(",")]
        return {"nvidia_smi_name": name, "power_limit": power, "sm_max_clock": clock}
    except Exception as e:   # the timing does not depend on it; say why it is missing
        return {"nvidia_smi_error": str(e)}


def learner_params(torch, obs_dim, act_dim, dev, seed=0):
    from marinevehiclereinforcementlearning_b200.policy import squashed_param_shapes
    g = torch.Generator().manual_seed(seed)
    return {k: (torch.randn(s, generator=g) * 0.1).to(dev) for k, s in squashed_param_shapes(obs_dim, act_dim).items()}


def per_call(torch, precision, dev, rounds, calls):
    from marinevehiclereinforcementlearning_b200 import SquashedGaussianPolicy
    params = learner_params(torch, 9, 6, dev)
    mk = lambda: SquashedGaussianPolicy(9, 6, device=dev, seed=1, action_noise_std=0.1, precision=precision)
    via_sd, via_host, via_dev = mk(), mk(), mk()
    via_host.load_state_dict({k: v.cpu() for k, v in params.items()})
    via_dev.load_state_dict(params, share=True)
    routes = {"state_dict": lambda: via_sd.load_state_dict(params), "host_entry": via_host.sync_weights, "device": via_dev.sync_weights}
    for f in routes.values():
        for _ in range(10):
            f()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(100):
            via_dev.sync_weights()
    graph.replay()
    torch.cuda.synchronize()
    wall = {k: [] for k in routes}
    kernel = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(rounds):
        for name, f in routes.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(calls):
                f()
            t1 = time.perf_counter()          # the device route's enqueue time: it returns without waiting
            torch.cuda.synchronize()
            wall[name].append((t1 - t0) / calls * 1e6)
        e0.record()
        graph.replay()
        e1.record()
        e1.synchronize()
        kernel.append(e0.elapsed_time(e1) * 1e3 / 100)
    out = {k + "_us_per_call": statistics.median(v) for k, v in wall.items()}
    out["device_pack_kernel_us"] = statistics.median(kernel)
    return out


def collection_loop(torch, precision, dev, n, T, rounds):
    from marinevehiclereinforcementlearning_b200 import BlueROV2Heavy6DoFVecEnv, SquashedGaussianPolicy
    env = BlueROV2Heavy6DoFVecEnv(n, action_mode="setpoint", dtype=torch.float32, device=dev, seed=3, auto_reset=True,
                                  record_terminal_obs=False)
    env.reset()
    params = learner_params(torch, 9, 6, dev)
    plist = list(params.values())
    pol_sd = SquashedGaussianPolicy(9, 6, device=dev, seed=1, action_noise_std=0.1, precision=precision)
    pol = SquashedGaussianPolicy(9, 6, device=dev, seed=1, action_noise_std=0.1, precision=precision).load_state_dict(params, share=True)

    def update():          # stands in for optimizer.step(): one in-place update of every parameter
        torch._foreach_mul_(plist, 1.0)

    def loop(sync):
        for t in range(T):
            (pol if sync != "state_dict" else pol_sd).act(env, step=t)
            env.step_async()
            if sync == "state_dict":
                update()
                pol_sd.load_state_dict(params)
            elif sync == "device":
                update()
                pol.sync_weights()

    variants = {"state_dict": lambda: loop("state_dict"), "device": lambda: loop("device"), "no_sync": lambda: loop(None)}
    for f in variants.values():
        f()
    torch.cuda.synchronize()
    graphs = {}
    for name, sync in (("device_graph", "device"), ("no_sync_graph", None)):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            loop(sync)
        g.replay()
        graphs[name] = g
    torch.cuda.synchronize()
    for name, g in graphs.items():
        variants[name] = g.replay
    times = {k: [] for k in variants}
    for _ in range(rounds):
        for name, f in variants.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            f()
            torch.cuda.synchronize()
            times[name].append(time.perf_counter() - t0)
    return {name + "_env_steps_per_s": n * T / statistics.median(v) for name, v in times.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--device", default="cuda:0")
    ap.add_argument("--rounds", type=int, default=15)
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--n", type=int, default=131072)
    ap.add_argument("--steps", type=int, default=128)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("policy_sync_bench needs a CUDA device")
    dev = torch.device(args.device)
    res = {"what": "squashed-head weight sync, 6DoF shapes (9 -> 6)", "device": gpu_info(dev.index or 0), "torch": torch.__version__,
           "rounds": args.rounds, "calls_per_round": args.calls, "loop": {"num_envs": args.n, "T": args.steps}}
    for precision in ("bf16", "fp32"):
        res[precision] = {"per_call": per_call(torch, precision, dev, args.rounds, args.calls),
                          "collection_loop": collection_loop(torch, precision, dev, args.n, args.steps, args.rounds)}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
