"""Compare the SASS of the plain scan kernels of two builds of blmx_scan.cu.

    python tools/sass_compare.py OLD.so NEW.so

Every scan_kernel<J, GROUP, FAR> of OLD (the kernel before it took the SURF flag) is compared, instruction
listing for instruction listing (cuobjdump -sass), with scan_kernel<J, GROUP, FAR, SURF = false> of NEW, and every
scan_kernel<J, GROUP, FAR, SURF> of OLD (before the SPLIT flag) with scan_kernel<J, GROUP, FAR, SURF, SPLIT = false>;
a kernel OLD already has with the SPLIT flag is compared with the same instantiation in NEW.  Build both with the
same nvcc flags.  bound_kernel, which the scan runs before scan_kernel, and reduce_kernel, which runs after it, are
compared as well; a bound_kernel of OLD without the SLABS flag is compared with bound_kernel<SLABS = 0> of NEW.  Exit status 1 if any listing differs.
"""
import re
import subprocess
import sys

CUDA_BIN = '/usr/local/cuda/bin'


def scan_kernels(so, prefix='scan_kernel<'):
    """{'scan_kernel<J, GROUP, FAR[, SURF]>': SASS listing} of a library (prefix 'bound_kernel(': that kernel)."""
    out = subprocess.run([f'{CUDA_BIN}/cuobjdump', '-sass', so], capture_output=True, text=True, check=True).stdout
    parts = re.split(r'\n\s*Function : (\S+)\n', out)
    names = subprocess.run([f'{CUDA_BIN}/cu++filt'], input='\n'.join(parts[1::2]), capture_output=True, text=True,
                           check=True).stdout.splitlines()
    res = {}
    for name, body in zip(names, parts[2::2]):
        name = name.replace('<unnamed>::', '').replace('(int)', '').replace('(bool)', '')
        name = name[len('void '):] if name.startswith('void ') else name      # templates carry their return type
        if name.startswith(prefix):
            res[name[:name.index('>' if prefix.endswith('<') else '(') + 1]] = body
    return res


def main():
    old, new = scan_kernels(sys.argv[1]), scan_kernels(sys.argv[2])
    same = 0
    for name in sorted(old):
        twin = name[:-1] + ', 0' * (4 - name.count(',')) + '>'
        ok = old[name] == new.get(twin)
        same += ok
        print(f'{"identical" if ok else "DIFFERENT"}  {name} -> {twin}  ({len(old[name].splitlines())} lines)')
    print(f'{same}/{len(old)} identical')
    old_b, new_b = ({**scan_kernels(so, 'bound_kernel('), **scan_kernels(so, 'bound_kernel<'),
                     **scan_kernels(so, 'reduce_kernel(')} for so in sys.argv[1:3])
    if 'bound_kernel<0>' in new_b:
        new_b.setdefault('bound_kernel(', new_b['bound_kernel<0>'])
    same_b = sum(old_b[k] == new_b.get(k) for k in old_b)
    for k in sorted(old_b):
        print(f'{"identical" if old_b[k] == new_b.get(k) else "DIFFERENT"}  {k}  ({len(old_b[k].splitlines())} lines)')
    return 0 if same == len(old) and same_b == len(old_b) else 1


if __name__ == '__main__':
    sys.exit(main())
