"""Developer tool: search over the placement of the playout kernels' device functions.

ptxas lays the device functions of a kernel out in the order of their mangled names, and the playout kernels are bound by the SM's
instruction cache (profiles/README.md), so WHERE the per-step functions sit relative to each other is worth +-5 %.  This script
writes renaming headers (the format of csrc/ctd_layout_classic.h: `#define ctd_x ctd_hNN_...`) for a set of orders, builds one library per order
(only the playout units are recompiled) under citadels_self_play_b200/variants/, and prints the command that times them on the GPU box:

    python tools/layout_search.py build N SEED [parent.json ...]   # N random orders, or N mutations of the given plans
    gpurun -- 'python tools/layout_search.py run'                  # times every variants/layout_<target>_*.so next to the shipped library
    python tools/layout_search.py pick                             # reads gpurun_out/layout_search_<target>.json, prints the best orders
LAYOUT_TARGET=playout (default: the preset / classic playout units) or search (the preset cfr_train / cfr_pred units).
"""
import os, sys, json, random, subprocess, glob
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "citadels_self_play_b200", "csrc")
VAR = os.path.join(ROOT, "citadels_self_play_b200", "variants")
TARGETS = {
    "playout": {
        "units": ("ctd_preset_playout.cu", "ctd_classic_playout.cu"),
        "functions": ["philox", "has", "append", "draw", "take_like", "count_type", "count_suit", "player_from_rank", "setup_next_player",
                      "refresh_used_roles", "apply_finish", "apply_build", "move_crown", "check_game_ending", "setup_round", "shuffle_bytes",
                      "reshuffle_if_empty", "apply", "warp_choose",
                      # once-per-game and fallback code: part of the order too, so that the search can place it
                      "unpack", "enumerate", "deal_preset", "count_points", "character_options", "main_round_options", "wizard_take_options",
                      "pack"],
        "lengths": [34, 34, 34, 10],
        "bench": [(("playout_perf.py", "1048576", "0"), {"steps_per_s": "preset"}), (("playout_perf.py", "1048576", "1"), {"steps_per_s": "classic"})],
    },
    "search": {   # the preset search kernels: cfr_train (pure) and cfr_pred (deep, fused)
        "units": ("ctd_preset_search.cu", "ctd_preset_pred.cu"),
        "functions": ["append", "expand", "philox", "unpack", "new_node", "node_far", "cfr_train", "enumerate", "kn_add_hk", "take_like", "tree_init",
                      "count_suit", "count_type", "move_crown", "tree_alloc", "apply_build", "encode_game", "live_choice", "setup_round",
                      "apply_finish", "count_points", "kn_hk_remove", "action_choice", "backpropagate", "kn_setup_round", "sample_private",
                      "update_strategy", "cfr_pred_advance", "player_from_rank", "character_options", "check_game_ending", "setup_next_player",
                      "skip_false_choice", "main_round_options", "refresh_used_roles", "reshuffle_if_empty", "wizard_take_options", "has", "draw",
                      "apply"],
        "lengths": [34],
        "bench": [(("mccfr_perf.py", "4096", "200", "both"), {"pure_it_per_s": "pure", "deep_it_per_s": "deep"})],
    },
}
TARGET = os.environ.get("LAYOUT_TARGET", "playout")
HOT = TARGETS[TARGET]["functions"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "--extended-lambda", "-Xcompiler", "-fPIC"]


def header(order, length):
    lines = ["#pragma once"]
    for i, h in enumerate(order):
        new = f"ctd_h{i:02d}_{h}"
        new = (new + "_" * length)[:length] if length > len(f"ctd_h{i:02d}_") + 1 else new
        lines.append(f"#define ctd_{h} {new}")
    return "\n".join(lines) + "\n"


def build(n, seed):
    os.makedirs(VAR, exist_ok=True)
    base = "/tmp/ctd_layout_base"
    os.makedirs(base, exist_ok=True)
    units = ["ctd_kernels.cu"] + sorted(f for f in os.listdir(CSRC) if f.startswith(("ctd_generic_", "ctd_preset_", "ctd_classic_")) and f.endswith(".cu"))
    fixed = [u for u in units if u not in TARGETS[TARGET]["units"]]
    procs = [subprocess.Popen([NVCC] + FLAGS + ["-c", "-o", os.path.join(base, u[:-3] + ".o"), u], cwd=CSRC) for u in fixed]
    assert all(p.wait() == 0 for p in procs)
    rng = random.Random(seed)
    plans = []
    parents = [json.load(open(f)) for f in sys.argv[4:]]   # optional: mutate these plans instead of drawing fresh orders
    for k in range(n):
        if parents:
            par = parents[k % len(parents)]
            order = par["order"][:]
            for _ in range(rng.choice([1, 1, 2, 3])):   # move one function somewhere else
                x = order.pop(rng.randrange(len(order)))
                order.insert(rng.randrange(len(order) + 1), x)
            plans.append({"name": f"layout_{TARGET}_s{seed}_{k:02d}", "order": order, "length": par["length"], "parent": par["name"]})
        else:
            order = HOT[:]
            rng.shuffle(order)
            plans.append({"name": f"layout_{TARGET}_s{seed}_{k:02d}", "order": order, "length": rng.choice(TARGETS[TARGET]["lengths"])})
    for p in plans:
        hp = os.path.join(base, p["name"] + ".h")
        open(hp, "w").write(header(p["order"], p["length"]))
        objs = []
        procs = []
        for u in TARGETS[TARGET]["units"]:
            o = os.path.join(base, p["name"] + "_" + u[:-3] + ".o")
            objs.append(o)
            procs.append(subprocess.Popen([NVCC] + FLAGS + [f'-DCTD_LAYOUT_HEADER="{hp}"',
                                                             "-c", "-o", o, u], cwd=CSRC, stderr=subprocess.DEVNULL))
        assert all(q.wait() == 0 for q in procs)
        subprocess.check_call([NVCC, "-shared", "-o", os.path.join(VAR, p["name"] + ".so")] + objs + [os.path.join(base, u[:-3] + ".o") for u in fixed])
        json.dump(p, open(os.path.join(VAR, p["name"] + ".json"), "w"))
        print("built", p["name"], p["length"], flush=True)


def run():
    out = []
    libs = [None] + sorted(glob.glob(os.path.join(VAR, f"layout_{TARGET}_*.so")))
    for lib in libs:
        row = {"lib": os.path.basename(lib) if lib else "shipped"}
        for cmd, keys in TARGETS[TARGET]["bench"]:
            env = dict(os.environ)
            if lib: env["CTD_LIB"] = lib
            r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", cmd[0])] + list(cmd[1:]), env=env, capture_output=True, text=True)
            try:
                d = json.loads(r.stdout.strip().splitlines()[-1])
                for k, name in keys.items(): row[name] = d[k]
            except Exception:
                for name in keys.values(): row[name] = None
        out.append(row)
        print(json.dumps(row), flush=True)
    json.dump(out, open(os.path.join(ROOT, "gpurun_out", f"layout_search_{TARGET}.json"), "w"))


def pick():
    rows = json.load(open(os.path.join(ROOT, "gpurun_out", f"layout_search_{TARGET}.json")))
    keys = [name for _, ks in TARGETS[TARGET]["bench"] for name in ks.values()]
    for key in keys:
        rows2 = sorted([r for r in rows if r.get(key)], key=lambda r: -r[key])
        print(key, [(r["lib"], f"{r[key]:.4g}") for r in rows2[:5]], "shipped", [f"{r[key]:.4g}" for r in rows if r["lib"] == "shipped"])


def best_to(prefix):
    """write the plan of the best variant per benchmark key to <prefix><key>.json when it beats the shipped library of the same run"""
    rows = json.load(open(os.path.join(ROOT, "gpurun_out", f"layout_search_{TARGET}.json")))
    keys = [name for _, ks in TARGETS[TARGET]["bench"] for name in ks.values()]
    ship = {k: [r[k] for r in rows if r["lib"] == "shipped"][0] for k in keys}
    for key in keys:
        cand = sorted([r for r in rows if r.get(key) and r["lib"] != "shipped"], key=lambda r: -r[key])
        if cand and cand[0][key] > ship[key] * 1.002:   # (the shipped library of the SAME run: boxes differ by ~0.5 %)
            plan = json.load(open(os.path.join(VAR, cand[0]["lib"][:-3] + ".json")))
            plan["measured"] = {key: cand[0][key], "shipped_same_run": ship[key]}
            json.dump(plan, open(prefix + key + ".json", "w"))
            print("new best", key, cand[0]["lib"], f"{cand[0][key]:.5g}", "shipped", f"{ship[key]:.5g}")
        else:
            print("no improvement", key, f"{ship[key]:.5g}")


if __name__ == "__main__":
    if sys.argv[1] == "build": build(int(sys.argv[2]), int(sys.argv[3]))
    elif sys.argv[1] == "run": run()
    elif sys.argv[1] == "best": best_to(sys.argv[2])
    else: pick()
