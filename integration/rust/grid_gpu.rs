//! Replacement bodies for `grid::run` and `grid::solve` (src/grid.rs:31-246).  UNTESTED here (no Rust toolchain).
//! `compute_observables`, `normalise_wavefunction`, `orthogonalise_wavefunction`, `get_norm_squared` and `evolve`
//! (grid.rs:303-492, 544-687) are no longer called; `get_work_area` stays for the I/O modules.
use config;
use config::{Config, InitialCondition};
use errors::*;
use ffi::Gpu;
use input;
use ndarray::Array3;
use noisy_float::prelude::*;
use output;
use potential;
use slog::Logger;
use std::f64::MAX;

pub fn run(config: &Config, log: &Logger, debug_level: usize) -> Result<()> {
    let potentials = potential::load_arrays(config, log)?;
    let num = &config.grid.size;
    let gpu = Gpu::new((num.x, num.y, num.z), config.central_difference.ext(), config.grid.dn, config.grid.dt,
                       config.mass, config.wavemax)?;
    gpu.set_potential(&potentials.v)?;
    gpu.set_pot_sub(&potentials.pot_sub)?;

    let mut w_store: Vec<Array3<R64>> = Vec::new();
    if config.wavenum > 0 {
        input::load_wavefunctions(config, log, &mut w_store)?;
        for w in &w_store {
            gpu.push_lower(w)?;
        }
    }
    info!(log, "Starting calculation");
    for wnum in config.wavenum..config.wavemax + 1 {
        solve(config, log, debug_level, &gpu, wnum)?;
    }
    Ok(())
}

fn solve(config: &Config, log: &Logger, debug_level: usize, gpu: &Gpu, wnum: u8) -> Result<()> {
    let num = &config.grid.size;
    let bb = config.central_difference.bb();
    let init_size: [usize; 3] = [num.x + bb, num.y + bb, num.z + bb];
    if wnum > 0 {
        // grid.rs:60-96: a file in ./input wins; otherwise start from the previous state (deterministic seed instead
        // of the reference's noise-seeded clone, see DESIGN.md §2)
        if let Ok(wfn) = input::wavefunction(wnum, init_size, bb, &config.output.file_type, log) {
            if config.init_condition != InitialCondition::FromFile && wnum > config.wavenum {
                warn!(log, "Loaded a higher order wavefunction from disk although Initial conditions are set to '{}'.",
                      config.init_condition);
            }
            gpu.set_phi(&wfn)?;
        } else {
            gpu.phi_seed_from_lower(wnum as u32 - 1)?;
        }
    } else {
        let phi = config::set_initial_conditions(config, log).chain_err(|| ErrorKind::SetInitialConditions)?;
        gpu.set_phi(&phi)?;
    }
    output::print_observable_header(wnum);

    let mut step = 0;
    let mut converged = false;
    let mut last_energy = MAX;
    let mut host_phi = Array3::<R64>::zeros((init_size[0], init_size[1], init_size[2]));
    gpu.pin(&mut host_phi)?; // snapshots and the final save copy through this buffer
    loop {
        let o = gpu.check_state(wnum)?; // grid.rs:127-135 in one call
        let observables = ::grid::Observables {
            energy: r64(o.energy), norm2: r64(o.norm2), v_infinity: r64(o.v_infinity), r2: r64(o.r2),
        };
        let norm_energy = o.energy / o.norm2;
        let tau = r64(step as f64) * config.grid.dt;
        if config.output.snap_update.is_some() && step % config.output.snap_update.unwrap() == 0 {
            gpu.symmetrise(config.init_symmetry as i32)?; // grid.rs:137-139: symmetrise, normalise, write
            gpu.normalise(o.norm2)?;
            gpu.get_phi(&mut host_phi)?;
            let work = ::grid::get_work_area(&host_phi, config.central_difference.ext());
            if let Err(err) = output::wavefunction(&work, wnum, false, &config.project_name, &config.output.file_type) {
                warn!(log, "Could not output partial wavefunction per snap_update request: {}", err);
            }
        }
        let diff = (norm_energy - last_energy).abs();
        if diff < config.tolerance.raw() {
            // grid.rs:162-167: the row is printed at convergence only; between checks it goes to the progress bar
            println!("{}", output::print_measurements(tau, r64(diff), &observables));
            output::finalise_measurement(&observables, wnum, r64(num.x as f64), &config.project_name,
                                         &config.output.file_type)?;
            if config.output.snap_update.is_some() {
                let _ = output::remove_partial(wnum, &config.project_name, &config.output.file_type);
            }
            converged = true;
            break;
        } else {
            last_energy = norm_energy;
        }
        if debug_level == 3 {
            // grid.rs:198-209 (the ETA estimate of grid.rs:254-283 is unchanged and omitted here)
            info!(log, "{}", output::print_measurements(tau, r64(diff), &observables));
        }
        if config.max_steps.is_some() && step > config.max_steps.unwrap() {
            break;
        }
        gpu.evolve(wnum, config.output.screen_update)?; // grid.rs:216; asynchronous, the next check synchronises
        step += config.output.screen_update;
    }
    if config.output.save_wavefns {
        gpu.get_phi(&mut host_phi)?;
        let work = ::grid::get_work_area(&host_phi, config.central_difference.ext());
        if let Err(err) = output::wavefunction(&work, wnum, converged, &config.project_name, &config.output.file_type) {
            warn!(log, "Could not write wavefunction to disk: {}", err);
        }
    }
    gpu.unpin(&mut host_phi);
    if converged {
        gpu.push_lower_from_phi()?; // grid.rs:241
        Ok(())
    } else {
        Err(ErrorKind::MaxStep.into())
    }
}
