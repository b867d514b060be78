// build.rs -- builds libblu_consensus.so with nvcc for sm_100a (no other arch, no CPU fallback) and links it.
use std::{env, path::PathBuf, process::Command};

fn main() {
    let root = PathBuf::from(env::var("CARGO_MANIFEST_DIR").unwrap()).join("../..");
    let csrc = root.join("blutils_b200/csrc");
    let status = Command::new("make").arg("-C").arg(&csrc).arg("../libblu_consensus.so").status().expect("make (nvcc) failed to start");
    assert!(status.success(), "building libblu_consensus.so failed (needs nvcc with sm_100a support)");
    println!("cargo:rustc-link-search=native={}", root.join("blutils_b200").display());
    println!("cargo:rustc-link-lib=dylib=blu_consensus");
    for f in ["blu_kernels.cu", "blu_regroup.cu", "blu_sort.cu", "blu_sort.h", "blu_api.cpp", "blu_taxonomy.cpp", "blu_core.cuh", "blu_decode.h"] {
        println!("cargo:rerun-if-changed={}", csrc.join(f).display());
    }
    println!("cargo:rerun-if-changed={}", root.join("include/blu_consensus.h").display());
}
