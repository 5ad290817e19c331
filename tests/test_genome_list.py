"""--inputList on the CPU: the input list, early refusal of bad outputs, the genome sharding over gloo (world sizes 2
and 3, the C oracle standing in for the per-rank CUDA scan) and the helper files of a list of inputs."""
import os
import shutil
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import genome_data
import util
from ballermixplus_b200 import cli, scan, sharding

D = os.path.join(util.GOLD, 'data')


# ------------------------------------------------------------------------------------------- the list
def _write(path, text):
    with open(path, 'w') as fh:
        fh.write(text)
    return str(path)


def test_list_paths_are_relative_to_the_list_and_skip_comments(tmp_path):
    (tmp_path / 'sub').mkdir()
    a = _write(tmp_path / 'sub' / 'a.txt', 'x\n')
    b = _write(tmp_path / 'b.txt', 'x\n')
    lst = _write(tmp_path / 'sub' / 'list.txt', f'# genome\n\na.txt\n  \n#b.txt\n{b}\n')
    assert scan.input_list(lst) == [a, b]


def test_list_errors(tmp_path):
    with pytest.raises(FileNotFoundError, match='--inputList: input list .* not found'):
        scan.input_list(str(tmp_path / 'absent.txt'))
    with pytest.raises(ValueError, match='names no input'):
        scan.input_list(_write(tmp_path / 'empty.txt', '# nothing\n\n'))
    with pytest.raises(FileNotFoundError, match='--inputList: input .*missing.txt .* not found'):
        scan.input_list(_write(tmp_path / 'bad.txt', 'missing.txt\n'))
    (tmp_path / 'p').mkdir()
    (tmp_path / 'q').mkdir()
    _write(tmp_path / 'p' / 'chr1.txt', 'x\n')
    _write(tmp_path / 'q' / 'chr1.txt', 'x\n')
    with pytest.raises(ValueError, match='same file name chr1.txt'):
        scan.input_list(_write(tmp_path / 'dup.txt', 'p/chr1.txt\nq/chr1.txt\n'))


def test_null_list_messages_are_unchanged(tmp_path):
    from ballermixplus_b200 import null
    with pytest.raises(FileNotFoundError, match='^--null: replicate list .* not found$'):
        null.read_list(str(tmp_path / 'absent.txt'))


class _Read(Exception):
    pass


@pytest.fixture
def no_input_reads(monkeypatch):
    """InputData that fails the test's way if it is ever constructed; records the output files present then."""
    seen = []

    def fake(path, *a, **k):
        seen.append(path)
        raise _Read(path)
    monkeypatch.setattr(cli, 'InputData', fake)
    return seen


def _genome(tmp_path):
    lst, paths = genome_data.make_genome(str(tmp_path), chroms=genome_data.CHROMS[:2])
    return lst, paths


@pytest.mark.parametrize('which', ['-o', '--support', '--pvalues', '--refine'])
def test_bad_output_directory_fails_before_any_input_is_read(which, tmp_path, no_input_reads, capsys):
    lst, _ = _genome(tmp_path)
    null = genome_data.make_replicates(str(tmp_path), n_reps=1)
    dirs = {k: str(tmp_path / k.strip('-')) for k in ('-o', '--support', '--pvalues', '--refine')}
    for d in dirs.values():
        os.makedirs(d)
    dirs[which] = str(tmp_path / 'absent')
    argv = ['--inputList', '-i', lst, '--spect', genome_data.SPECT, '--null', null]
    for k, d in dirs.items():
        argv += [k, d]
    with pytest.raises(SystemExit) as exc:
        cli.main(argv)
    assert exc.value.code == 2
    assert f'{which} {dirs[which]} is not an existing directory' in capsys.readouterr().err
    assert no_input_reads == []


def test_output_that_is_an_input_or_a_shared_directory_is_refused(tmp_path, no_input_reads, capsys):
    lst, paths = _genome(tmp_path)
    in_dir = os.path.dirname(paths[0])
    base = ['--inputList', '-i', lst, '--spect', genome_data.SPECT]
    with pytest.raises(SystemExit):
        cli.main(base + ['-o', in_dir])
    assert 'would overwrite an input' in capsys.readouterr().err
    os.makedirs(tmp_path / 'out')
    with pytest.raises(SystemExit):
        cli.main(base + ['-o', str(tmp_path / 'out'), '--support', str(tmp_path / 'out')])
    assert 'name the same directory' in capsys.readouterr().err
    with pytest.raises(SystemExit):
        cli.main(base)
    assert '--inputList needs -o DIR' in capsys.readouterr().err
    assert no_input_reads == []
    with open(paths[0]) as fh:
        assert fh.readline() == 'physPos\tgenPos\tx\tn\n'


def test_bad_list_fails_before_any_input_is_read(tmp_path, no_input_reads, capsys):
    os.makedirs(tmp_path / 'out')
    with pytest.raises(SystemExit):
        cli.main(['--inputList', '-i', _write(tmp_path / 'l.txt', 'nope.txt\n'), '--spect', genome_data.SPECT,
                  '-o', str(tmp_path / 'out')])
    assert 'nope.txt' in capsys.readouterr().err and no_input_reads == []


def test_every_output_file_is_opened_before_the_first_input_is_read(tmp_path, monkeypatch):
    lst, paths = _genome(tmp_path)
    null = genome_data.make_replicates(str(tmp_path), n_reps=1)
    dirs = {k: str(tmp_path / k) for k in ('out', 'support', 'pvalues', 'refine')}
    for d in dirs.values():
        os.makedirs(d)
    stale = os.path.join(dirs['out'], 'chr2.txt')
    _write(stale, 'old contents\n')
    files = [os.path.join(d, os.path.basename(p)) for d in dirs.values() for p in paths]

    def fake(path, *a, **k):
        assert all(os.path.isfile(f) and os.path.getsize(f) == 0 for f in files)
        raise _Read(path)
    monkeypatch.setattr(cli, 'InputData', fake)
    with pytest.raises(_Read):
        cli.main(['--inputList', '-i', lst, '--spect', genome_data.SPECT, '-o', dirs['out'], '--support',
                  dirs['support'], '--pvalues', dirs['pvalues'], '--refine', dirs['refine'], '--null', null])


@pytest.mark.parametrize('flag', ['--support', '--refine'])
def test_torchrun_refuses_support_and_refine_before_any_input_is_read(flag, tmp_path, monkeypatch, no_input_reads,
                                                                      capsys):
    lst, _ = _genome(tmp_path)
    os.makedirs(tmp_path / 'out')
    os.makedirs(tmp_path / 'extra')
    monkeypatch.setenv('WORLD_SIZE', '2')
    with pytest.raises(SystemExit) as exc:
        cli.main(['--inputList', '-i', lst, '--spect', genome_data.SPECT, '-o', str(tmp_path / 'out'), flag,
                  str(tmp_path / 'extra')])
    assert exc.value.code == 2
    assert f'{flag} runs on one GPU; launch without torchrun (WORLD_SIZE > 1)' in capsys.readouterr().err
    assert no_input_reads == []
    assert os.listdir(tmp_path / 'out') == []


# ---------------------------------------------------------------------------------- genome sharding (gloo)
def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


#: chromosome sizes (sites) cut from one golden problem: very different, one far smaller than a rank's share
SIZES = (301, 7, 58, 190, 23)


def _genome_problems():
    from ballermixplus_b200.native import ScanProblem
    from ballermixplus_b200.problem import build_problem
    argv, _ = util.scan_cases()['ex1_B2_w15_s7p5']
    opt, data, neutral, grid, sel = util.host_objects(argv)
    prob, _ = build_problem(data, neutral, sel, grid)
    assert sum(SIZES) <= len(prob.genpos)
    probs, seqs, b = [], [], 0
    for k, n in enumerate(SIZES):
        p = ScanProblem(prob.genpos[b:b + n], prob.cls[b:b + n], prob.G, prob.SP, prob.A, prob.n_x, prob.n_a)
        c = np.arange(0, n, 1 + k % 2)
        lo, hi = np.maximum(0, c - 30), np.minimum(n - 1, c + 20)
        probs.append(p)
        seqs.append((p.genpos, p.A, p.genpos[c], lo, hi, None))
        b += n
    return probs, seqs


def _oracle_rows(p, t, lo, hi):
    from oracle import oracle_c
    T, iA, ixa, ns, _ = oracle_c.scan(p.genpos, p.cls, p.G, p.SP, p.A, t, lo, hi, n_threads=1)
    ix = np.where(ixa >= 0, ixa // p.n_a, -1).astype(np.int32)
    ia = np.where(ixa >= 0, ixa % p.n_a, -1).astype(np.int32)
    return tuple(torch.from_numpy(np.ascontiguousarray(a)) for a in (T, iA, ix, ia, ns))


def _worker(rank, world, port, out_dir):
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        probs, seqs = _genome_problems()
        loads, scanned = [], []

        def scan_fn(i, t, lo, hi):         # a fake loader: records which chromosome this rank loads
            loads.append(i)
            scanned.append(len(t))
            return _oracle_rows(probs[i], t, lo, hi)
        got = sharding.scan_sharded_seqs(seqs, rank, world, scan_fn, dist, torch)
        torch.save({'loads': loads, 'scanned': scanned, 'rows': None if got is None else [g.clone() for g in got]},
                   os.path.join(out_dir, f'rank{rank}.pt'))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize('world', [2, 3])
def test_genome_sharding_equals_per_chromosome_scans(world, tmp_path):
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    res = [torch.load(str(tmp_path / f'rank{r}.pt')) for r in range(world)]
    probs, seqs = _genome_problems()
    # gathered rows = the per-chromosome scans laid end to end
    ref = [_oracle_rows(p, *s[2:5]) for p, s in zip(probs, seqs)]
    for k, got in enumerate(res[0]['rows']):
        assert torch.equal(got, torch.cat([r[k] for r in ref]))
    assert all(r['rows'] is None for r in res[1:])
    # ranges cover every centre once, in order; each rank loaded exactly the chromosomes its range touches
    costs, offs = sharding.genome_costs(seqs)
    parts = sharding.partition(costs, world)
    assert parts[0][0] == 0 and parts[-1][1] == offs[-1]
    assert all(parts[r][1] == parts[r + 1][0] for r in range(world - 1))
    assert sum(sum(r['scanned']) for r in res) == offs[-1]
    for r, (b, e) in enumerate(parts):
        touched = [i for i in range(len(seqs)) if offs[i] < e and offs[i + 1] > b]
        assert res[r]['loads'] == touched
        assert sum(res[r]['scanned']) == e - b
    # the genome is sharded, not each chromosome: some chromosome lies wholly within one rank's range, and the
    # smallest is far below a rank's share
    assert any(len(r['loads']) > 1 for r in res)
    assert len(seqs[1][2]) < offs[-1] / world / 10


def test_pieces_and_genome_costs():
    offs = np.array([0, 5, 5, 12, 20])
    assert sharding.pieces(offs, 0, 20) == [(0, 0, 5), (2, 0, 7), (3, 0, 8)]
    assert sharding.pieces(offs, 3, 14) == [(0, 3, 5), (2, 0, 7), (3, 0, 2)]
    assert sharding.pieces(offs, 7, 7) == []
    _, seqs = _genome_problems()
    costs, o = sharding.genome_costs(seqs)
    assert list(np.diff(o)) == [len(s[2]) for s in seqs]
    for i, s in enumerate(seqs):
        assert np.array_equal(costs[o[i]:o[i + 1]], sharding.centre_costs(s[0], s[2], s[3], s[4], s[1]))


# ------------------------------------------------------------------------------------- helper files
HELPER_CASES = {
    'DAF': (['Example1_fullSweep_200kya_DAF.txt', 'Example2_balancing_10MYA_DAF.txt'], ['--getSpect']),
    'MAF': (['Example1_fullSweep_200kya_MAF.txt', 'Example2_balancing_10MYA_MAF.txt'], ['--getSpect', '--MAF']),
    'MAF_from_DAF': (['Example2_balancing_10MYA_DAF.txt', 'Example1_fullSweep_200kya_DAF.txt'],
                     ['--getSpect', '--MAF']),
    'noSub': (['Example2_balancing_10MYA_DAF.txt', 'Example2_balancing_10MYA_DAF_nosub.txt',
               'Example1_fullSweep_200kya_DAF.txt'], ['--getSpect', '--noSub']),
    'noSub_MAF': (['Example2_balancing_10MYA_MAF_nosub.txt', 'Example1_fullSweep_200kya_MAF.txt'],
                  ['--getSpect', '--noSub', '--MAF']),
    'B1': (['Example1_fullSweep_200kya_DAF.txt', 'Example2_balancing_10MYA_DAF.txt', 'synth_mixed_n.txt'],
           ['--getConfig']),
}


@pytest.mark.parametrize('case', sorted(HELPER_CASES))
def test_helper_files_of_a_list_equal_the_concatenation(case, tmp_path):
    names, flags = HELPER_CASES[case]
    for k, n in enumerate(names):                   # under distinct names: a list may not repeat a file name
        shutil.copy(os.path.join(D, n), tmp_path / f'{k}_{n}')
    files = [f'{k}_{n}' for k, n in enumerate(names)]
    lst = _write(tmp_path / 'list.txt', '# inputs\n' + '\n'.join(files) + '\n')
    cat = tmp_path / 'cat.txt'
    with open(cat, 'w') as out:
        for k, f in enumerate(files):
            with open(tmp_path / f) as fh:
                lines = fh.readlines()
            out.writelines(lines if k == 0 else lines[1:])
    got, ref = str(tmp_path / 'got.txt'), str(tmp_path / 'ref.txt')
    with util.quiet(), pytest.raises(SystemExit):
        cli.main(['--inputList', '-i', lst, '--spect', got] + flags)
    with util.quiet(), pytest.raises(SystemExit):
        cli.main(['-i', str(cat), '--spect', ref] + flags)
    with open(got, 'rb') as a, open(ref, 'rb') as b:
        ref_bytes = b.read()
        assert a.read() == ref_bytes and len(ref_bytes) > 0
