"""Host-pipeline probe (GPU box): extract_all on 2048 JPEG files of 480x480 under a few thread settings, with the
main-thread time breakdown. Usage: python tools/io_probe.py [n_images]"""
import importlib.util, json, os, shutil, sys, tempfile, time
from pathlib import Path
ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "tests"))
from conftest import load_pkg  # noqa: E402
import numpy as np, cv2, torch  # noqa: E402

run = 0


def main():
    global run
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 2048
    ex = load_pkg("extract"); iop = load_pkg("io_pipeline"); synth = load_pkg("synth")
    tmp = Path(tempfile.mkdtemp())
    root = tmp / "images"; root.mkdir()
    imgs = synth.blobs_batch(64, 480, 480, seed0=0).numpy()
    names = []
    for i in range(n):
        name = f"im{i:05d}.jpg"
        if i < 64:
            cv2.imwrite(str(root / name), cv2.cvtColor(imgs[i], cv2.COLOR_RGB2BGR), [cv2.IMWRITE_JPEG_QUALITY, 90])
        else:
            shutil.copyfile(root / names[i % 64], root / name)
        names.append(name)
    (tmp / "list.txt").write_text("\n".join(names) + "\n")
    (tmp / "warm.txt").write_text("\n".join(names[:128]) + "\n")
    ex.extract_all(str(tmp / "warm.txt"), str(root), "dino_vits16", None, str(tmp / "warm"), K=5, batch_size=128, seed=0)
    def go(label, batch=128, wout=4, **env):
        global run
        run += 1
        old = {k: os.environ.get(k) for k in env}
        os.environ.update({k: str(v) for k, v in env.items()})
        si = float(env.get("SWITCH", 0.005)); sys.setswitchinterval(si)
        st = ex.extract_all(str(tmp / "list.txt"), str(root), "dino_vits16", None, str(tmp / f"eigs{run}"), K=5, batch_size=batch, seed=0, num_workers_out=wout)
        sys.setswitchinterval(0.005)
        for k, v in old.items():
            if v is None: os.environ.pop(k, None)
            else: os.environ[k] = v
        print("PROBE", label, round(st["images_per_s"]), {k: round(v, 3) for k, v in st["main_thread_seconds"].items()}, st.get("decode_thread_seconds_summed"), flush=True)
        shutil.rmtree(tmp / f"eigs{run}", ignore_errors=True)

    # what one .pth costs on this box's file systems (torch.save + rename, like the writers): serial and 4 processes
    import subprocess
    code = ("import torch, os, sys, time\n"
            "d = sys.argv[1]; n = int(sys.argv[2]); tag = sys.argv[3]\n"
            "obj = {'eigenvalues': torch.randn(5), 'eigenvectors': torch.randn(5, 900)}\n"
            "t = time.perf_counter()\n"
            "for i in range(n):\n"
            "    torch.save(obj, f'{d}/{tag}{i}.tmp'); os.replace(f'{d}/{tag}{i}.tmp', f'{d}/{tag}{i}.pth')\n"
            "print((time.perf_counter() - t) / n * 1e6)\n")
    for label, base in (("tmpdir", tempfile.gettempdir()), ("devshm", "/dev/shm")):
        if not os.path.isdir(base):
            continue
        d = tempfile.mkdtemp(dir=base)
        one = subprocess.run([sys.executable, "-c", code, d, "500", "a"], capture_output=True, text=True).stdout.strip()
        ps = [subprocess.Popen([sys.executable, "-c", code, d, "500", f"p{k}_"], stdout=subprocess.PIPE, text=True) for k in range(4)]
        four = [p_.communicate()[0].strip() for p_ in ps]
        print("PROBE fs", label, base, "us_per_file serial", one, "4procs_same_dir", four, flush=True)
        shutil.rmtree(d, ignore_errors=True)
    shm = Path(tempfile.mkdtemp(dir="/dev/shm")) if os.path.isdir("/dev/shm") else None

    def go_shm(label, **kw):
        nonlocal tmp
        if shm is None:
            return
        keep = tmp
        # only the outputs move to tmpfs; the JPEGs stay where they are
        global run
        run += 1
        st = ex.extract_all(str(keep / "list.txt"), str(root), "dino_vits16", None, str(shm / f"eigs{run}"), K=5, batch_size=128, seed=0, **kw)
        print("PROBE", label, round(st["images_per_s"]), {k: round(v, 3) for k, v in st["main_thread_seconds"].items()}, st.get("decode_thread_seconds_summed"), flush=True)
        shutil.rmtree(shm / f"eigs{run}", ignore_errors=True)

    os.environ["DSS_IO_TRACE"] = "1"
    for rep in range(1):
        run += 1
        st = ex.extract_all(str(tmp / "list.txt"), str(root), "dino_vits16", None, str(shm / f"eigs{run}"), K=5, batch_size=128, seed=0)
        tr = st["decode_thread_seconds_summed"].pop("trace")
        ids = {}
        print("PROBE trace run", rep, round(st["images_per_s"]), st["main_thread_seconds"], st["decode_thread_seconds_summed"], flush=True)
        for t_, ev_, d_ in tr:
            if ev_ in ("opened", "closed", "ready", "consumer_got", "released"):
                d_ = ids.setdefault(d_, len(ids))
            print("PROBE   ", f"{t_:8.4f}", ev_, d_, flush=True)
        shutil.rmtree(shm / f"eigs{run}", ignore_errors=True)
    os.environ.pop("DSS_IO_TRACE")
    for rep in range(3):
        go("default")
        go_shm("out_on_devshm")
        go_shm("out_on_devshm_8thr", num_workers=8)
        go_shm("out_on_devshm_16thr", num_workers=16)
    for rep in range(0):
        go("default")
        go_shm("out_on_devshm")
        go_shm("out_on_devshm_16thr", num_workers=16)
        go_shm("out_on_devshm_48thr", num_workers=48)
    if shm is not None:
        shutil.rmtree(shm, ignore_errors=True)
    for rep in range(0):
        go("default")
        go("decode16", DSS_IO_DECODE_THREADS=16)
        go("decode48", DSS_IO_DECODE_THREADS=48)
        go("decode64", DSS_IO_DECODE_THREADS=64)
        go("decode24", DSS_IO_DECODE_THREADS=24)
        go("decode96", DSS_IO_DECODE_THREADS=96)
        go("writers8", wout=8)
        go("writers2", wout=2)
        go("switch0.5ms", SWITCH=0.0005)
        go("switch0.1ms", SWITCH=0.0001)
        go("batch256", batch=256)
        go("batch64", batch=64)
    # decode only
    ds = ex.utils.ImagesDataset(names, str(root))
    for w in (16, 32, 64):
        t0 = time.perf_counter(); c = sum(1 for _ in iop.ImagePrefetcher(ds.load_raw, range(len(ds)), num_workers=w)); dt = time.perf_counter() - t0
        print("PROBE decode_only_raw", w, round(c / dt))
        t0 = time.perf_counter(); c = sum(1 for _ in iop.ImagePrefetcher(ds.__getitem__, range(len(ds)), num_workers=w)); dt = time.perf_counter() - t0
        print("PROBE decode_only_rgb", w, round(c / dt))
    shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":   # the writer pool uses the 'spawn' start method: children re-import this module
    main()
