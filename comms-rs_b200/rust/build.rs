// build.rs -- compiles comms-rs_b200/csrc/*.cu with nvcc for sm_100a into libcomms_b200.so and
// tells cargo to link it.  With `--features prebuilt` (or COMMS_B200_LIB_DIR set) it only links.
use std::env;
use std::path::PathBuf;
use std::process::Command;

fn main() {
    let manifest = PathBuf::from(env::var("CARGO_MANIFEST_DIR").unwrap());
    let pkg = manifest.parent().unwrap().to_path_buf(); // comms-rs_b200/
    let csrc = pkg.join("csrc");
    let out = PathBuf::from(env::var("OUT_DIR").unwrap());

    if let Ok(dir) = env::var("COMMS_B200_LIB_DIR") {
        println!("cargo:rustc-link-search=native={}", dir);
    } else if cfg!(feature = "prebuilt") {
        println!("cargo:rustc-link-search=native={}", pkg.display());
    } else {
        let nvcc = env::var("NVCC").unwrap_or_else(|_| "/usr/local/cuda/bin/nvcc".into());
        let lib = out.join("libcomms_b200.so");
        let mut cmd = Command::new(nvcc);
        cmd.args(["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17"])
            .args(["-Xcompiler", "-fPIC,-fvisibility=hidden", "-shared", "-cudart", "static", "-o"])
            .arg(&lib);
        // the same list as comms-rs_b200/build.py (SOURCES)
        for f in ["api.cu", "comm.cu", "fir_kernels.cu", "fir_tc_kernel.cu", "fir_ptc_kernel.cu", "fir_real_kernel.cu", "fft_kernels.cu",
                  "fft_cluster_kernel.cu", "fft_cpipe_kernel.cu", "fft_rows_kernel.cu", "fft_big_kernel.cu", "chain_kernels.cu", "chain_tc_kernel.cu", "misc_kernels.cu",
                  "estimator_kernels.cu", "nco_kernel.cu", "fir_f64_kernels.cu", "fft_f64_kernels.cu"] {
            let p = csrc.join(f);
            println!("cargo:rerun-if-changed={}", p.display());
            cmd.arg(p);
        }
        cmd.args(["-DCB_BUILD", "-ldl"]); // comm.cu binds NCCL with dlopen
        let st = cmd.status().expect("failed to run nvcc");
        assert!(st.success(), "nvcc failed");
        println!("cargo:rustc-link-search=native={}", out.display());
    }
    println!("cargo:rustc-link-lib=dylib=comms_b200");
    println!("cargo:rerun-if-changed={}", pkg.parent().unwrap().join("include/comms_b200.h").display());
}
