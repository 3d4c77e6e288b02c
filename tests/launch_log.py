"""Which CUDA kernels a piece of host code launched: CUPTI activity records through torch.profiler, and the
template arguments of a kernel in a demangled name."""
import re


def _template_args(name, kernel):
    """top-level template arguments of `kernel<...>` in a demangled name, whitespace and namespaces removed"""
    m = re.search(r"\b" + kernel + "<", name)
    if not m:
        return None
    i, depth, cur, args = m.end(), 1, "", []
    while depth:
        ch = name[i]
        i += 1
        if ch == "<":
            depth += 1
        elif ch == ">":
            depth -= 1
            if depth == 0:
                break
        if ch == "," and depth == 1:
            args.append(cur)
            cur = ""
        else:
            cur += ch
    args.append(cur)
    norm = []
    for a in args:
        a = re.sub(r"\s+|pb::|\(int\)", "", a)
        norm.append({"(bool)1": "true", "(bool)0": "false"}.get(a, a))
    return tuple(norm)


def launch_log(run):
    """Demangled names of every CUDA kernel `run()` launches, and run()'s result."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = run()
        torch.cuda.synchronize()
    names = {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
    return names, out
