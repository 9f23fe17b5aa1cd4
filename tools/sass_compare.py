"""Compares the SASS instruction sequence (cuobjdump -sass, addresses and encodings stripped) of every kernel of OLD
with the same kernel of NEW; exit status 1 if one is missing or differs.  Kernel names are matched after renamings
that do not change code: anonymous namespaces (named from a hash of their translation unit), rollout_kernel's SCREEN
argument turning from bool into ScreenMode with a second, empty kernel argument, and the rollout kernels' MODELS
argument (model-set mode) with, for the lane-split kernels, that same empty second argument.  screen_mask_kernel
gained a model count M: it is matched to its new name, and its code differs by that loop.
usage: python tools/sass_compare.py OLD NEW   (objects or shared libraries, e.g. a parent commit's libswimmer_ars.so)"""
import re, subprocess, sys

def kernels(path):
    out = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    ks, name = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = m.group(1); ks[name] = []
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;", line)
        if name and m:
            ks[name].append(m.group(1))
    return ks

def anon(k):
    # a translation unit's anonymous namespace is named from a hash of its source
    return re.sub(r"_GLOBAL__N__[0-9a-f]+_\d+_(\w+?_cu)_[0-9a-f]+", r"_GLOBAL__N__\1", k)

def rename(k):
    # rollout_kernel<..., bool SCREEN>(RolloutArgs) became rollout_kernel<..., int SCREEN>(RolloutArgs, ScreenForms<SCREEN>::type)
    k = re.sub(r"^(_ZN3swm14rollout_kernelI.*)Lb([01])EEEvNS_11RolloutArgsE$",
               r"\1Li\2EEEvNS_11RolloutArgsENS_11ScreenFormsIXT4_EE4typeE", k)
    # ... then rollout_kernel<..., int SCREEN, bool MODELS>(RolloutArgs, ScreenForms<SCREEN, MODELS>::type)
    k = re.sub(r"^(_ZN3swm14rollout_kernelI.*)EEvNS_11RolloutArgsENS_11ScreenFormsIXT4_EE4typeE$",
               r"\1Lb0EEEvNS_11RolloutArgsENS_11ScreenFormsIXT4_EXT5_EE4typeE", k)
    # lane_rollout_kernel<N, LINEAR, NORM, STATS, bool MODELS>(RolloutArgs, ScreenForms<SCREEN_NONE, MODELS>::type)
    k = re.sub(r"^(_ZN3swm19lane_rollout_kernelI.*)EEvNS_11RolloutArgsE$",
               r"\1Lb0EEEvNS_11RolloutArgsENS_11ScreenFormsILi0EXT3_EE4typeE", k)
    # lane2_rollout_kernel<N, LINEAR, NORM, STATS, NF, SCREEN, bool MODELS>(RolloutArgs, ScreenForms<..>::type)
    k = re.sub(r"^(_ZN3swm20lane2_rollout_kernelI.*)EEvNS_11RolloutArgsE$",
               r"\1Lb0EEEvNS_11RolloutArgsENS_11ScreenFormsILi0EXT5_EE4typeE", k)
    # screen_mask_kernel(sim_returns, N, ...) -> screen_mask_kernel(sim_returns, M, N, ...)
    return k.replace("_ZN3swm18screen_mask_kernelEPKdidPiS2_Px", "_ZN3swm18screen_mask_kernelEPKdiidPiS2_Px")

old = {anon(rename(k)): v for k, v in kernels(sys.argv[1]).items()}
new = {anon(k): v for k, v in kernels(sys.argv[2]).items()}
missing = [k for k in old if k not in new]
diff = [k for k in old if k in new and old[k] != new[k]]
print("kernels in old: %d, in new: %d, new-only: %d" % (len(old), len(new), len([k for k in new if k not in old])))
print("missing in new: %d, differing: %d, identical: %d" % (len(missing), len(diff), len(old) - len(missing) - len(diff)))
for k in missing[:10] + diff[:10]:
    print("  ", k)
sys.exit(1 if missing or diff else 0)
