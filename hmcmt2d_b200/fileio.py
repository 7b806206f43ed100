"""Readers / writers for the reference's model (.mod), data (.dat) and startup files
(HMCMT/src/HMCFileIO/*.jl, HMCMT/src/HMCSampler/readstartupFile.jl) — host-side, run once."""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List

import numpy as np


@dataclass
class TensorMesh2D:
    """Mirror of `TensorMesh2D` (HMCFileIO.jl:46-60); zLen / sigma include the air layers.
    The sparse operators of the reference struct are not needed: assembly is fused in the CUDA kernels."""
    yLen: np.ndarray
    zLen: np.ndarray
    airLayer: np.ndarray
    gridSize: tuple
    origin: np.ndarray
    sigma: np.ndarray
    setup: bool = True


@dataclass
class MTData:
    """Mirror of `MTData` (HMCFileIO.jl:26-41); rxID/freqID/dtID stay 1-based as in the file."""
    rxLoc: np.ndarray
    freqs: np.ndarray
    dataType: str
    dataComp: List[str]
    rxID: np.ndarray
    freqID: np.ndarray
    dtID: np.ndarray
    dataID: np.ndarray
    compTE: bool
    compTM: bool


@dataclass
class HMCPrior:
    """Mirror of `HMCPrior` (HMCStruct.jl:18-38) with `initHMCPrior` defaults (:129-140)."""
    burninsamples: int = 100
    totalsamples: int = 500
    sigBounds: list = field(default_factory=lambda: [0.01, 10.0])
    sigmastd: float = 0.05
    dt: float = 0.01
    timestep: list = field(default_factory=lambda: [10, 15])
    linearSolver: str = "b200"
    massType: str = "diagonal"
    regParam: float = 1.0
    nfevals: int = 0


class _Tokens:
    """Line cursor that skips blank lines and '#' comments (readEMModel2D.jl:31-37)."""

    def __init__(self, path):
        with open(path, "r") as fh:
            self.lines = [ln.strip() for ln in fh]
        self.lines = [ln for ln in self.lines if ln and not ln.startswith("#")]
        self.i = 0

    def more(self):
        return self.i < len(self.lines)

    def next(self):
        ln = self.lines[self.i]
        self.i += 1
        return ln

    def numbers(self, count):
        out = []
        while len(out) < count:
            out += [float(tok) for tok in self.next().split()]
        return np.asarray(out[:count], dtype=np.float64)


def readEMModel2D(modelfile: str) -> TensorMesh2D:
    """`readEMModel2D` (readEMModel2D.jl:11-154): substring keywords, air layers listed bottom-up."""
    tk = _Tokens(modelfile)
    ny = nz = 0
    ylen = zlen = sig = None
    air = np.zeros(0)
    origin = np.zeros(2)
    res_type = ""
    while tk.more():
        ln = tk.next()
        last = ln.split()[-1]
        if "NY" in ln:
            ny = int(last)
            ylen = tk.numbers(ny)
        elif "NZ" in ln:
            nz = int(last)
            zlen = tk.numbers(nz)
        elif "NAIR" in ln:
            air = tk.numbers(int(last))
        elif "Resistivity Type" in ln:
            res_type = last
        elif "Model Type" in ln:
            sig = tk.numbers(ny * nz)
            if res_type == "Resistivity":
                sig = 1.0 / sig
            if last == "log":
                raise ValueError("Model Type 'log' is unusable in the reference (readEMModel2D.jl:117-119)")
        elif "Origin" in ln:
            parts = ln.split()
            origin = np.array([float(parts[-2]), float(parts[-1])])
    if air.size:
        zlen = np.concatenate([air[::-1], zlen])
        origin = np.array([origin[0], origin[1] + air.sum()])
        sig = np.concatenate([np.full(ny * air.size, 1e-8), sig])
    return TensorMesh2D(ylen, zlen, air, (ny, len(zlen)), origin, sig)


def readMT2DData(datafile: str):
    """`readMT2DData` (readMT2DData.jl:14-179) -> (MTData, obsData, dataErr)."""
    tk = _Tokens(datafile)
    rx = freqs = None
    dtype_name, comps, is_cplx = "", [], False
    fid = rid = did = obs = err = None
    while tk.more():
        ln = tk.next()
        if "Format" in ln:
            continue
        if "Receiver Location" in ln:
            n = int(ln.split()[-1])
            rx = np.array([[float(v) for v in tk.next().split()[:2]] for _ in range(n)])
        elif "Frequencies" in ln:
            n = int(ln.split()[-1])
            freqs = np.array([float(tk.next()) for _ in range(n)])
        elif "DataType" in ln:
            dtype_name = ln.split()[-1]
            if dtype_name not in ("Impedance", "Rho_Pha"):
                raise ValueError(f"{dtype_name} is not supported.")
            is_cplx = dtype_name == "Impedance"
        elif "DataComp" in ln:
            comps = [tk.next().strip() for _ in range(int(ln.split()[-1]))]
        elif "Data Block" in ln:
            n = int(ln.split()[-1])
            rows = [tk.next().split() for _ in range(n)]
            fid = np.array([int(r[0]) for r in rows], dtype=np.int64)
            rid = np.array([int(r[1]) for r in rows], dtype=np.int64)
            did = np.array([int(r[2]) for r in rows], dtype=np.int64)
            if is_cplx:
                obs = np.array([float(r[3]) + 1j * float(r[4]) for r in rows], dtype=np.complex128)
                err = np.array([float(r[5]) for r in rows])
            else:
                obs = np.array([float(r[3]) for r in rows])
                err = np.array([float(r[4]) for r in rows])
    te = any("XY" in c or c == "TZY" for c in comps)            # the tipper TZY = Hz/Hy is a TE response
    tm = any("YX" in c for c in comps)
    mask = np.zeros((len(freqs), rx.shape[0], len(comps)), dtype=bool)      # vec(Bool[nDt,nRx,nFreq]) :165-172
    mask[fid - 1, rid - 1, did - 1] = True
    return MTData(rx, freqs, dtype_name, comps, rid, fid, did, mask.reshape(-1), te, tm), obs, err


def writeEMModel2D(modelfile: str, mesh: TensorMesh2D, stamp: str = "") -> None:
    """`writeEMModel2D` (writeEMModel2D.jl:11-82)."""
    ny, nz, nair = len(mesh.yLen), len(mesh.zLen), len(mesh.airLayer)

    def block(fh, vals, fmt):
        for i, v in enumerate(vals, 1):
            fh.write(fmt % v)
            if i % 8 == 0:
                fh.write("\n")
        if len(vals) % 8:
            fh.write("\n")

    with open(modelfile, "w") as fh:
        fh.write("%-18s %s\n" % ("#Format:", "EMModel2DFile"))
        fh.write("%-18s %s\n" % ("#Description:", "file generated in " + stamp))
        fh.write("%-6s %4d\n" % ("NY:", ny))
        block(fh, mesh.yLen, "%10.2f")
        if nair:
            fh.write("%-6s %4d\n" % ("NAIR:", nair))
            block(fh, mesh.airLayer, "%12.2f")
        fh.write("%-6s %4d\n" % ("NZ:", nz - nair))
        block(fh, mesh.zLen[nair:], "%10.2f")
        fh.write("%-18s %s\n" % ("Resistivity Type:", "Conductivity"))
        fh.write("%-18s %s\n" % ("Model Type:", "Linear"))
        earth = np.asarray(mesh.sigma)[ny * nair:].reshape(nz - nair, ny)
        for row in earth:
            fh.write("".join("%4.2e " % v for v in row) + "\n")
        oz = mesh.origin[1] - (np.sum(mesh.airLayer) if nair else 0.0)
        fh.write("%-15s %4.2e %4.2e" % ("Origin (m):", mesh.origin[0], oz))


def writeMT2DData(datafile: str, info: MTData, predData, dataErr=None, stamp: str = "") -> None:
    """`writeMT2DData` (writeMT2DData.jl:12-86)."""
    pred = np.asarray(predData)
    if dataErr is None or len(dataErr) == 0:
        dataErr = np.abs(pred) * 0.03
    elif len(dataErr) == 1:
        dataErr = np.abs(pred) * dataErr[0]
    with open(datafile, "w") as fh:
        fh.write("%-20s%s\n" % ("Format:", "MT2DData_1.0"))
        fh.write("# %s\n" % ("file generated in " + stamp))
        fh.write("%-25s %4d\n" % ("Receiver Location (m):", info.rxLoc.shape[0]))
        fh.write("# %5s %5s\n" % ("Y", "Z"))
        for y, z in info.rxLoc:
            fh.write("%12.2f %12.2f\n" % (y, z))
        fh.write("%-20s%3d\n" % ("Frequencies (Hz):", len(info.freqs)))
        for f in info.freqs:
            fh.write("%8.4e\n" % f)
        fh.write("%-12s %12s\n" % ("DataType:", info.dataType))
        fh.write("%-15s %d\n" % ("DataComp:", len(info.dataComp)))
        for c in info.dataComp:
            fh.write("%4s\n" % c)
        fh.write("%-15s %d\n" % ("Data Block:", len(pred)))
        if np.iscomplexobj(pred):
            fh.write("# %6s %6s %10s %10s %15s %12s\n" % ("FreqNo.", "RxNo.", "dataComp", "RealValue", "ImagValue", "Error"))
            for i, v in enumerate(pred):
                fh.write("%5d %6d %8d %15.6e %15.6e %15.6e\n" % (info.freqID[i], info.rxID[i], info.dtID[i], v.real, v.imag, dataErr[i]))
        else:
            fh.write("# %6s %6s %10s %10s %12s\n" % ("FreqNo.", "RxNo.", "dataComp", "RealValue", "Error"))
            for i, v in enumerate(pred):
                fh.write("%5d %6d %8d %15.6e %15.6e\n" % (info.freqID[i], info.rxID[i], info.dtID[i], v, dataErr[i]))


def parseStartup(startupfile: str):
    """Key/value part of `readstartupFile` (readstartupFile.jl:28-81), branch order preserved: a
    `fixedresistivity:` line contains `resistivity:` and is taken by that earlier branch, as in the reference."""
    prior = HMCPrior()
    prior.linearSolver = ""
    datafile = modelfile = None
    sigmin = sigmax = 0.0
    sigfix = [1e-8]
    tk = _Tokens(startupfile)
    while tk.more():
        ln = tk.next()
        w = ln.split()
        if "datafile:" in ln:
            datafile = w[-1]
        elif "modelfile:" in ln:
            modelfile = w[-1]
        elif "burninsamples:" in ln:
            prior.burninsamples = int(w[-1])
        elif "totalsamples:" in ln:
            prior.totalsamples = int(w[-1])
        elif "resistivity:" in ln:
            rmin, rmax = float(w[-3]), float(w[-2])
            float(w[-1])
            sigmin, sigmax = 1.0 / rmax, 1.0 / rmin
            prior.sigBounds = [sigmin, sigmax]
            prior.sigmastd = (np.log(sigmax) - np.log(sigmin)) * 0.05
        elif "fixedresistivity:" in ln:
            sigfix.append(float(w[-1]))
        elif "timeinterval:" in ln:
            prior.dt = float(w[-1])
        elif "timestep:" in ln:
            prior.timestep = [int(w[-2]), int(w[-1])]
        elif "linearsolver:" in ln:
            prior.linearSolver = w[-1]
        elif "masstype:" in ln:
            prior.massType = w[-1]
        elif "smoothparameter:" in ln:
            prior.regParam = float(w[-1])
    return datafile, modelfile, sigmin, sigmax, sigfix, prior
