"""BASELINE config 1 plumbing on the CPU: the reference's UNMODIFIED bin/speedseq with a private config whose $BWA / $SAMBLASTER are the
oracle CLI (argv-identical to the shims) — once with the reference's sambamba, once with `SAMBAMBA=` the repo's sambamba shim, which
has to hand every call of the script (view / sort of plain SAM and BAM, index) through to the real one.  Same three BAMs both ways.
The script, the binary and the example data are the reference's own and are not part of this repository: the test runs where build()
staged them under oracle/_ref/stage (tools/stage_config1.sh) and skips elsewhere; the GPU-side runs are profiles/r02_config1_unmodified_speedseq.log."""
import os
import subprocess

import pytest

import ssq_testlib as T

REF = os.path.join(T.ROOT, "oracle", "_ref", "stage")
pytestmark = pytest.mark.skipif(not (os.path.exists(REF + "/bin/speedseq") and os.access(REF + "/src/sambamba", os.X_OK)), reason="the reference's speedseq script and sambamba are not staged under oracle/_ref/stage")


def test_unmodified_speedseq_runs_with_the_sambamba_shim_in_front_of_the_real_one(tmp_path):
    sb = REF + "/src/sambamba"
    w1, w2 = str(tmp_path / "plain"), str(tmp_path / "shim")
    subprocess.run(["bash", os.path.join(T.ROOT, "tools", "run_config1.sh"), "oracle", REF, w1], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, timeout=300)
    os.makedirs(w2)
    cfg = open(os.path.join(w1, "speedseq.b200.config")).read().replace(w1, w2)
    cfg = "\n".join(l for l in cfg.splitlines() if not l.startswith("SAMBAMBA=")) + "\nSAMBAMBA=%s\nexport SSQ_SAMBAMBA_REAL=%s\n" % (os.path.join(T.ROOT, "speedseq_b200", "bin", "sambamba"), sb)
    open(os.path.join(w2, "cfg"), "w").write(cfg)
    for f in os.listdir(w1):
        if f.startswith("ref.fa"):
            os.symlink(os.path.join(w1, f), os.path.join(w2, f))
    os.symlink(os.path.join(w1, "bin"), os.path.join(w2, "bin"))
    env = dict(os.environ, PATH=os.path.join(w2, "bin") + ":" + os.environ["PATH"])
    subprocess.run(["bash", REF + "/bin/speedseq", "align", "-o", "example", "-M", "3", "-p", "-t", "4", "-K", os.path.join(w2, "cfg"), "-R", r"@RG\tID:NA12878\tSM:NA12878\tLB:lib1", "ref.fa",
                    REF + "/example/data/NA12878.20slice.30X.fastq.gz"], cwd=w2, check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, env=env, timeout=300)
    for f, n in (("example.bam", 95890), ("example.splitters.bam", 82), ("example.discordants.bam", 220)):
        a = subprocess.run([sb, "view", os.path.join(w1, f)], stdout=subprocess.PIPE, check=True).stdout
        b = subprocess.run([sb, "view", os.path.join(w2, f)], stdout=subprocess.PIPE, check=True).stdout
        assert a == b and a.count(b"\n") == n, f
        assert os.path.exists(os.path.join(w2, f + ".bai"))
