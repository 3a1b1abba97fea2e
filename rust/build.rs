// build.rs -- compiles the CUDA library with nvcc for sm_100a and links it.
// (Authored, not compiled in this image: there is no Rust toolchain here.)
use std::env;
use std::path::PathBuf;
use std::process::Command;

fn main() {
    let out = PathBuf::from(env::var("OUT_DIR").unwrap());
    let root = PathBuf::from(env::var("CARGO_MANIFEST_DIR").unwrap()).join("..");
    let lib = out.join("libpairing_b200.a");
    let nvcc = env::var("NVCC").unwrap_or_else(|_| "/usr/local/cuda/bin/nvcc".into());
    // every .cu of the source directory is a translation unit of its own (pairing_b200/csrc/abi_common.cuh)
    let csrc = root.join("pairing_b200/csrc");
    let mut srcs: Vec<PathBuf> = std::fs::read_dir(&csrc)
        .expect("pairing_b200/csrc")
        .map(|e| e.expect("pairing_b200/csrc").path())
        .filter(|p| p.extension().map_or(false, |x| x == "cu"))
        .collect();
    srcs.sort();
    let mut objs = Vec::new();
    for src in &srcs {
        let obj = out.join(src.file_stem().unwrap()).with_extension("o");
        let status = Command::new(&nvcc)
            .args(&["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
                    "-Xcompiler", "-fPIC", "-c", "-o"])
            .arg(&obj)
            .arg(&src)
            .status()
            .expect("nvcc not found: set NVCC");
        assert!(status.success(), "nvcc failed");
        objs.push(obj);
    }
    let status = Command::new("ar").args(&["crs"]).arg(&lib).args(&objs).status().expect("ar");
    assert!(status.success());
    println!("cargo:rustc-link-search=native={}", out.display());
    println!("cargo:rustc-link-lib=static=pairing_b200");
    println!("cargo:rustc-link-search=native=/usr/local/cuda/lib64");
    println!("cargo:rustc-link-lib=dylib=cudart");
    println!("cargo:rustc-link-lib=dylib=stdc++");
    println!("cargo:rustc-link-lib=dylib=pthread");
    println!("cargo:rerun-if-changed={}", csrc.display());
    println!("cargo:rerun-if-changed={}", root.join("include/pairing_b200.h").display());
}
