"""The packed-sweep schedule the kinematics kernel runs: no base quaternion direction (their Hessian columns are
closed-form in kino_kin.cu), checked on the CPU through hb_debug_sweep_schedule_n_base.  Same execution rules as
test_sweep_schedule_cpu.py: every (joint direction, relevant body) step once, chains on one lane in increasing rounds,
slots read after every flush into them, no two flushes into one slot in a round, light rounds hold propagation only."""
import ctypes

import numpy as np

KT = dict(L=0, P=5, D=10, VALID=1 << 15, START=1 << 16, IN_L=1 << 17, IN_P=1 << 18, LOAD=19, FLUSH=25, STORE=1 << 31)


def schedule(lib, parent, feet, chest, n_base):
    tasks = np.zeros(32 * 32, dtype=np.int32)
    info = np.zeros(40, dtype=np.int32)
    par = np.asarray(parent, dtype=np.int32)
    i32p = ctypes.POINTER(ctypes.c_int32)
    rc = lib.hb_debug_sweep_schedule_n_base(len(parent), par.ctypes.data_as(i32p), feet[0], feet[1], chest, 1, n_base,
                                            tasks.ctypes.data_as(i32p), info.ctypes.data_as(i32p))
    assert rc == 0
    return tasks.view(np.uint32).reshape(32, 32), info


def expected_tasks(parent, feet, n_base):
    nb = len(parent)
    anc = lambda b: ([] if parent[b] < 0 else [parent[b]] + anc(parent[b]))  # noqa: E731
    sub = [{l for l in range(nb) if b == l or b in anc(l)} for b in range(nb)]
    out = {}
    for d in range(4 + nb - 1):
        if d < 4 and d >= n_base:
            continue
        ld = 0 if d < 4 else d - 3
        rel = set(sub[ld]) | set(anc(ld))
        for f in range(2):
            if feet[f] in sub[ld]:
                rel |= {feet[1 - f]} | set(anc(feet[1 - f]))
        for l in rel:
            out[(d, l)] = l in sub[ld]
    return out


def test_kernel_schedule_without_base_directions(model, built_library):
    parent = [int(v) for v in model.parent]
    feet = (model.frames["l_sole"][0], model.frames["r_sole"][0])
    chest = model.frames["chest"][0]
    tasks, info = schedule(built_library, parent, feet, chest, 0)
    n_rounds, n_tasks, n_heavy, heavy_mask = int(info[0]), int(info[2]), int(info[3]), int(np.uint32(info[4]))
    want = expected_tasks(parent, feet, 0)
    assert n_tasks == len(want) == 256 and n_heavy == sum(want.values()) == 92  # DESIGN.md 3.1
    assert 0 < n_rounds <= 13 and int(info[1]) * 12 <= 474
    seen, flushed_at, loads, root_store, running = {}, {}, [], {}, {}
    for r in range(n_rounds):
        kinds, flush_slots = set(), []
        for lane in range(32):
            t = int(tasks[r, lane])
            if not t & KT["VALID"]:
                continue
            l, p, d = (t >> KT["L"]) & 31, (t >> KT["P"]) & 31, (t >> KT["D"]) & 31
            assert d >= 4 and (d, l) in want and (d, l) not in seen
            seen[(d, l)] = (r, lane)
            assert bool(t & KT["IN_L"]) == want[(d, l)]
            if l != 0:
                assert p == parent[l] and bool(t & KT["IN_P"]) == want.get((d, p), False)
            kinds.add(bool(t & KT["IN_L"]))
            if t & KT["START"]:
                assert lane not in running
            else:
                pd, pl, pr = running[lane]
                assert pd == d and parent[pl] == l and pr < r
            running[lane] = (d, l, r)
            ls, fs = (t >> KT["LOAD"]) & 63, (t >> KT["FLUSH"]) & 63
            if ls:
                loads.append((ls - 1, r, d))
            if fs:
                flush_slots.append(fs - 1)
                if t & KT["STORE"]:
                    root_store[fs - 1] = (r, d)
                else:
                    flushed_at.setdefault(fs - 1, []).append((r, d))
                del running[lane]
        assert len(flush_slots) == len(set(flush_slots)), f"two flushes into one slot in round {r}"
        if kinds:
            assert bool((heavy_mask >> r) & 1) == (True in kinds), f"round {r}: heavy bit does not match its tasks"
    assert not running and set(seen) == set(want)
    for slot, r, d in loads:
        assert slot in flushed_at and all(fr < r and fd == d for fr, fd in flushed_at[slot])
    for d in range(27):
        rs = int(info[6 + d])
        if d < 4:
            assert rs == -1  # no root slot: the kernel reads its closed form instead
        else:
            assert root_store[rs][1] == d and all(fr < root_store[rs][0] for fr, _ in flushed_at.get(rs, []))
    light = [r for r in range(n_rounds) if not (heavy_mask >> r) & 1]
    assert n_rounds - len(light) <= 7 and len(light) >= 6


def test_base_direction_count(model, built_library):
    """tasks and heavy tasks by the number of base directions kept (4: what hb_debug_sweep_schedule builds)"""
    parent = [int(v) for v in model.parent]
    feet = (model.frames["l_sole"][0], model.frames["r_sole"][0])
    chest = model.frames["chest"][0]
    for n_base, n_tasks, n_heavy in ((4, 352, 188), (3, 328, 164), (0, 256, 92)):
        _, info = schedule(built_library, parent, feet, chest, n_base)
        assert (int(info[2]), int(info[3])) == (n_tasks, n_heavy)
